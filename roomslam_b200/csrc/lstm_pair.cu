// bf16 tensor-core LSTM recurrence at H = 128 (the shipped BiLSTM at d_model 256): forward and backward through time on a
// CTA PAIR (thread-block cluster of 2, tcgen05 cta_group::2), after the GRU pair kernels of rec_pair.cu.  Same operands and
// results as rs_lstm_fwd_f32 / rs_lstm_bwd_f32 (lstm_f32.cu); only W_hh h_{t-1} (forward) and dG_t W_hh (backward) run on
// the tensor core, with bf16 operands and fp32 accumulation.  The cell state, the dc carry, P, out, saved and dG stay fp32.
//
//   * A pair owns a 128-trace tile of one direction, 64 traces per CTA.  One thread of the even CTA issues M = 128 MMAs that
//     span both SMs; the accumulator of a CTA then uses all 128 TMEM lanes for its 64 rows: lane = row + 64 * (hidden-unit
//     half), so each CTA needs only the weight rows of its own 64 hidden units in shared memory.
//   * Forward, per step: G = h_{t-1} W_hh^T, N = 4H = 512 as two N = 256 MMAs (i | f, g | o), K = 128.  Per lane half the
//     accumulator holds columns [0, 64) i, [64, 128) f, [128, 192) g, [192, 256) o of the half's 64 units.  The 16
//     epilogue warps add P_t, apply the gates, keep c in registers for the whole sequence, write h_t (bf16) straight into
//     their own CTA's A tile (all 128 units of a row are produced in the row's CTA: h never crosses the pair), and store
//     out and saved.  Only mbarrier arrivals and the multicast tcgen05.commit cross the pair.
//   * Backward, per step: the epilogue forms dG_t from d_out_t, dh (the accumulator of the previous reverse step), the dc
//     carry (registers) and saved; it stores fp32 dG and writes the bf16 copy into the A tile; then dh_{t-1} = dG_t W_hh
//     runs with K = 512 and N = 128.
//   * 16 warps per CTA, all of them epilogue warps (16 hidden units of one row per thread); warp 0 of the even CTA also
//     issues the MMAs of the pair once its own share of the step is done.  Without a dedicated issuer / loader warp the
//     register cap is 128, not the 96 of 18 warps (which spilled).  P (forward) and saved / d_out (backward) of live rows
//     are pulled into L2 a few steps ahead; each thread requests its first group of operands before it waits for the
//     accumulator and the next group while it works on the current one.
//   * Rows past B read and write nothing (their A rows stay zero); the pad rows of out and dG are never written; no atomics.
#include "common.cuh"
#include "rec_common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

using namespace rs;

constexpr int H = 128;
constexpr int ROWS = 64;                        // traces of a tile held by one CTA of the pair
constexpr int CHUNK_S = ROWS * 16;              // shared: one 16-byte chunk column over this CTA's 64 rows
constexpr int W_CHUNK_F = 256 * 16;             // shared: one chunk column of this CTA's i | f | g | o rows (64 units each)
constexpr int UPT = 16;                         // hidden units per epilogue thread (4 warps per lane quadrant)
constexpr int GU = 4;                           // units per group (operands of the next group are loaded under this one)
constexpr int NUM_THREADS = 512;                // 16 epilogue warps; warp 0 of the even CTA also issues the MMAs of the pair
constexpr int PF = 4;                           // L2 prefetch distance in steps

struct Seq {
    float* p;
    long long ld, rows, row0;
    __device__ __forceinline__ float* at(long long b, long long t) const { return p + (b * rows + row0 + t) * ld; }
};

__device__ __forceinline__ float sigm_fast(float x) { return fmaf(0.5f, tanh_fast(0.5f * x), 0.5f); }
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, const float (&v)[4]) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ uint2 pack4(const float (&v)[4]) { return make_uint2(f2_to_bf2(v[0], v[1]), f2_to_bf2(v[2], v[3])); }
__device__ __forceinline__ void f4(const float4& x, float (&v)[4]) { v[0] = x.x; v[1] = x.y; v[2] = x.z; v[3] = x.w; }
// TMEM -> registers: this warp's 32 lanes x 4 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld_32x32b_x4(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}

struct FwdParams {
    Seq P, out;
    const uint8_t* w;                           // forward image [2][16 (x2 split)][512][8] bf16
    float* saved;                               // [2][B][T][5][H] or NULL
    int B, T, split;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) lstm_fwd_bf16_kernel(const FwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int nck = 16 * (1 + p.split);
    uint8_t* w_s = smem;                                   // [nck][256 rows: i | f | g | o of this CTA's 64 units][16 B]
    uint8_t* a_s = w_s + nck * W_CHUNK_F;                  // [16 chunks][64 rows][16 B]  h_{t-1} (bf16)
    uint64_t* bars = reinterpret_cast<uint64_t*>(a_s + 16 * CHUNK_S);
    uint64_t* w_full = bars;
    uint64_t* h_ready = bars + 1;               // even CTA: h_t of both CTAs written (32 epilogue warps)
    uint64_t* acc_full = bars + 2;              // both: the step's MMAs retired (multicast commit)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);

    const uint32_t rank = cluster_ctarank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y, tile = blockIdx.x >> 1, T = p.T;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        mbar_init(h_ready, 2 * 16);
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc_pair<256>(tmem_slot);
        if (lane == 0) {
            mbar_expect_tx(w_full, nck * W_CHUNK_F);
            const uint8_t* src = p.w + (long long)dir * nck * (512 * 16);
            for (int c = 0; c < nck; ++c)
                for (int g = 0; g < 4; ++g)
                    bulk_load(w_s + c * W_CHUNK_F + g * 1024, src + (long long)c * (512 * 16) + (g * 128 + rank * 64) * 16, 1024, w_full);
        }
    }
    for (int i = threadIdx.x; i < 16 * CHUNK_S / 16; i += blockDim.x) reinterpret_cast<uint4*>(a_s)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
    if (warp == 0) mbar_wait(w_full, 0);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();             // both CTAs: barriers initialised, TMEM allocated, W and h_{-1} = 0 in place
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // MMAs of one step, issued by warp 0 of the even CTA once both CTAs' h_{t-1} is in their A tiles
    auto issue = [&]() {
        constexpr uint32_t idesc = umma_idesc_bf16(128, 256, 0, 0);
        const uint32_t w_addr = smem_u32(w_s), a_addr = smem_u32(a_s);
        if (elect_one()) {
            for (int part = 0; part <= p.split; ++part) {      // split weights: h W_hi^T + h W_lo^T, same A tile
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    const uint64_t da = umma_desc_noswz(a_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                    const uint32_t wk = w_addr + (part * 16 + k * 2) * W_CHUNK_F;
                    tc_mma_bf16_pair(tmem_base, da, umma_desc_noswz(wk, W_CHUNK_F, 128), idesc, (k | part) != 0);
                    tc_mma_bf16_pair(tmem_base + 128, da, umma_desc_noswz(wk + 128 * 16, W_CHUNK_F, 128), idesc, (k | part) != 0);
                }
            }
            tc_commit_pair(acc_full);
        }
        __syncwarp();
    };
    const bool issuer = rank == 0 && warp == 0;
    if (issuer) issue();
    {
        const int q = warp & 3;                            // TMEM lane quadrant of this warp
        const int wg = warp >> 2;                          // which 16 of this lane half's 64 hidden units
        const int uh = q >> 1;                             // lane half = hidden-unit half
        const int rl = (q & 1) * 32 + lane;                // row within this CTA
        const long long b = (long long)tile * 128 + rank * ROWS + rl;
        const bool live = b < p.B;
        const int ub = uh * 64 + wg * UPT;                 // first hidden unit of this thread
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + wg * UPT;
        uint8_t* a_row = a_s + rl * 16;
        const uint32_t hr_remote = mapa_cluster(smem_u32(h_ready), 0);
        float c[UPT];
#pragma unroll
        for (int j = 0; j < UPT; ++j) c[j] = 0.0f;
        float4 pv[4];                                      // P of one group of GU units, gate g at pv[g]
        auto load_p = [&](const float* pp, int grp) {
#pragma unroll
            for (int g = 0; g < 4; ++g) pv[g] = ld4(pp + g * H + grp * GU);
        };
        for (int step = 0; step < T; ++step) {
            const int t = dir ? (T - 1 - step) : step;
            const float* pp = live ? p.P.at(b, t) + dir * 4 * H + ub : nullptr;
            float* op = live ? p.out.at(b, t) + dir * H + ub : nullptr;
            float* sp = (live && p.saved) ? p.saved + ((((long long)dir * p.B + b) * T + t) * 5) * H + ub : nullptr;
            if (live) load_p(pp, 0);
            if (live && ub == 0 && step + PF < T)           // the whole row of this direction (2 KB) into L2, PF steps ahead
                l2_prefetch(p.P.at(b, dir ? t - PF : t + PF) + dir * 4 * H, 4 * H * 4);
            mbar_wait(acc_full, step & 1);
            tc_fence_after();
#pragma unroll
            for (int grp = 0; grp < UPT / GU; ++grp) {
                uint32_t ai[GU], af[GU], ag[GU], ao[GU];
                tmem_ld_32x32b_x4(taddr + grp * GU, ai);
                tmem_ld_32x32b_x4(taddr + 64 + grp * GU, af);
                tmem_ld_32x32b_x4(taddr + 128 + grp * GU, ag);
                tmem_ld_32x32b_x4(taddr + 192 + grp * GU, ao);
                float px[4][GU];
#pragma unroll
                for (int g = 0; g < 4; ++g) f4(live ? pv[g] : make_float4(0.f, 0.f, 0.f, 0.f), px[g]);
                if (live && grp + 1 < UPT / GU) load_p(pp, grp + 1);
                tmem_ld_wait();
                float gi[GU], gf[GU], gg[GU], go[GU], hv[GU], cv[GU];
#pragma unroll
                for (int j = 0; j < GU; ++j) {
                    gi[j] = sigm_fast(__uint_as_float(ai[j]) + px[0][j]);
                    gf[j] = sigm_fast(__uint_as_float(af[j]) + px[1][j]);
                    gg[j] = tanh_fast(__uint_as_float(ag[j]) + px[2][j]);
                    go[j] = sigm_fast(__uint_as_float(ao[j]) + px[3][j]);
                    c[grp * GU + j] = live ? fmaf(gf[j], c[grp * GU + j], gi[j] * gg[j]) : 0.0f;
                    cv[j] = c[grp * GU + j];
                    hv[j] = live ? go[j] * tanh_fast(cv[j]) : 0.0f;
                }
                // next step's A operand, in place (8 bytes: GU bf16 of chunk (ub + grp GU) / 8)
                *reinterpret_cast<uint2*>(a_row + ((ub + grp * GU) / 8) * CHUNK_S + (grp & 1) * 8) = pack4(hv);
                if (live) {
                    st4(op + grp * GU, hv);
                    if (sp) {
                        st4(sp + grp * GU, gi); st4(sp + H + grp * GU, gf); st4(sp + 2 * H + grp * GU, gg);
                        st4(sp + 3 * H + grp * GU, go); st4(sp + 4 * H + grp * GU, cv);
                    }
                }
            }
            fence_proxy_async();        // h_t written with ordinary stores -> visible to the tensor core
            tc_fence_before();          // TMEM reads done before the next MMA overwrites the accumulator
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(hr_remote);
            if (issuer && step + 1 < T) {
                mbar_wait_cluster(h_ready, step & 1);
                tc_fence_after();
                issue();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the peer's tensor core reads this CTA's W half until its last MMA retired
    if (warp == 0) tmem_dealloc_pair<256>(tmem_base);
}

struct BwdParams {
    Seq d_out, dG;
    const float* saved;                         // [2][B][T][5][H]
    const uint8_t* w;                           // backward image [2][64 (x2 split)][128][8] bf16: W_hh^T, K = the 4H gate rows
    int B, T, split;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) lstm_bwd_bf16_kernel(const BwdParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int nck = 64 * (1 + p.split);
    uint8_t* w_s = smem;                                   // [nck][64 rows = this CTA's hidden units][16 B]
    uint8_t* a_s = w_s + nck * CHUNK_S;                    // [64 chunks: i | f | g | o][64 rows][16 B]  dG_t (bf16)
    uint64_t* bars = reinterpret_cast<uint64_t*>(a_s + 64 * CHUNK_S);
    uint64_t* w_full = bars;
    uint64_t* a_ready = bars + 1;               // even CTA: dG_t of both CTAs written (32 epilogue warps)
    uint64_t* acc_full = bars + 2;              // both: the dh MMAs retired (multicast commit)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3);

    const uint32_t rank = cluster_ctarank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y, tile = blockIdx.x >> 1, T = p.T;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        mbar_init(a_ready, 2 * 16);
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc_pair<64>(tmem_slot);
        if (lane == 0) {
            mbar_expect_tx(w_full, nck * CHUNK_S);
            const uint8_t* src = p.w + (long long)dir * nck * (128 * 16) + rank * 1024;
            for (int c = 0; c < nck; ++c) bulk_load(w_s + c * CHUNK_S, src + (long long)c * (128 * 16), 1024, w_full);
        }
    }
    for (int i = threadIdx.x; i < 64 * CHUNK_S / 16; i += blockDim.x) reinterpret_cast<uint4*>(a_s)[i] = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
    if (warp == 0) mbar_wait(w_full, 0);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // dh MMAs of one step, issued by warp 0 of the even CTA once both CTAs' dG_t is in their A tiles
    auto issue = [&]() {
        constexpr uint32_t idesc = umma_idesc_bf16(128, 128, 0, 0);
        const uint32_t w_addr = smem_u32(w_s), a_addr = smem_u32(a_s);
        if (elect_one()) {
            for (int part = 0; part <= p.split; ++part) {
#pragma unroll 4
                for (int k = 0; k < 32; ++k) {
                    const uint64_t da = umma_desc_noswz(a_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                    const uint64_t db = umma_desc_noswz(w_addr + (part * 64 + k * 2) * CHUNK_S, CHUNK_S, 128);
                    tc_mma_bf16_pair(tmem_base, da, db, idesc, (k | part) != 0);
                }
            }
            tc_commit_pair(acc_full);
        }
        __syncwarp();
    };
    const bool issuer = rank == 0 && warp == 0;
    {
        const int q = warp & 3;
        const int wg = warp >> 2;
        const int uh = q >> 1;
        const int rl = (q & 1) * 32 + lane;
        const long long b = (long long)tile * 128 + rank * ROWS + rl;
        const bool live = b < p.B;
        const int ub = uh * 64 + wg * UPT;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + wg * UPT;
        uint8_t* a_row = a_s + rl * 16;
        const uint32_t ar_remote = mapa_cluster(smem_u32(a_ready), 0);
        float dc[UPT];
#pragma unroll
        for (int j = 0; j < UPT; ++j) dc[j] = 0.0f;
        // one group of GU units: d_out, i, f, g, o, c_t, c_{t-1}
        float4 rv[7];
        auto load_grp = [&](const float* sp, const float* dp, bool has_prev, int grp) {
            const int o = grp * GU;
            rv[0] = ld4(dp + o);
#pragma unroll
            for (int k = 0; k < 5; ++k) rv[1 + k] = ld4(sp + k * H + o);
            const long long pstep = dir ? 5LL * H : -5LL * H;                  // c_{t-1}: the previous step in this direction
            rv[6] = has_prev ? ld4(sp + pstep + 4 * H + o) : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        for (int sidx = 0; sidx < T; ++sidx) {             // sidx-th reverse step = forward position T-1-sidx (dir 0)
            const int t = dir ? sidx : (T - 1 - sidx);
            const bool has_prev = sidx + 1 < T;
            const float* sp = live ? p.saved + ((((long long)dir * p.B + b) * T + t) * 5) * H + ub : nullptr;
            const float* dp = live ? p.d_out.at(b, t) + dir * H + ub : nullptr;
            float* gp = live ? p.dG.at(b, t) + dir * 4 * H + ub : nullptr;
            if (live) load_grp(sp, dp, has_prev, 0);
            if (live && ub == 0 && sidx + PF < T) {         // saved (2.5 KB) and d_out (512 B) of the row into L2, PF steps ahead
                const int tp = dir ? t + PF : t - PF;
                l2_prefetch(p.saved + ((((long long)dir * p.B + b) * T + tp) * 5) * H, 5 * H * 4);
                l2_prefetch(p.d_out.at(b, tp) + dir * H, H * 4);
            }
            if (sidx > 0) {
                mbar_wait(acc_full, (sidx - 1) & 1);       // dh of this step (dG_{t+1} W_hh) is in TMEM; the A tile is free
                tc_fence_after();
            }
#pragma unroll
            for (int grp = 0; grp < UPT / GU; ++grp) {
                uint32_t ah[GU] = {0u, 0u, 0u, 0u};
                if (sidx > 0) tmem_ld_32x32b_x4(taddr + grp * GU, ah);
                float v[7][GU];
#pragma unroll
                for (int k = 0; k < 7; ++k) f4(live ? rv[k] : make_float4(0.f, 0.f, 0.f, 0.f), v[k]);
                if (live && grp + 1 < UPT / GU) load_grp(sp, dp, has_prev, grp + 1);
                if (sidx > 0) tmem_ld_wait();
                float di[GU], df[GU], dg[GU], dq[GU];
#pragma unroll
                for (int j = 0; j < GU; ++j) {
                    const float d = __uint_as_float(ah[j]) + v[0][j];
                    const float gi = v[1][j], gf = v[2][j], gg = v[3][j], go = v[4][j], cc = v[5][j], cp = v[6][j];
                    const float tc = tanh_fast(cc);
                    const float dcell = fmaf(d * go, fmaf(-tc, tc, 1.0f), dc[grp * GU + j]);
                    dq[j] = live ? d * tc * go * (1.0f - go) : 0.0f;
                    di[j] = live ? dcell * gg * gi * (1.0f - gi) : 0.0f;
                    df[j] = live ? dcell * cp * gf * (1.0f - gf) : 0.0f;
                    dg[j] = live ? dcell * gi * fmaf(-gg, gg, 1.0f) : 0.0f;
                    dc[grp * GU + j] = live ? dcell * gf : 0.0f;
                }
                // A operand of the dh matvec: K order i | f | g | o (the gate rows of W_hh)
                const int ch = (ub + grp * GU) / 8, half = (grp & 1) * 8;
                *reinterpret_cast<uint2*>(a_row + (0 * 16 + ch) * CHUNK_S + half) = pack4(di);
                *reinterpret_cast<uint2*>(a_row + (1 * 16 + ch) * CHUNK_S + half) = pack4(df);
                *reinterpret_cast<uint2*>(a_row + (2 * 16 + ch) * CHUNK_S + half) = pack4(dg);
                *reinterpret_cast<uint2*>(a_row + (3 * 16 + ch) * CHUNK_S + half) = pack4(dq);
                if (live) {
                    st4(gp + grp * GU, di); st4(gp + H + grp * GU, df); st4(gp + 2 * H + grp * GU, dg); st4(gp + 3 * H + grp * GU, dq);
                }
            }
            fence_proxy_async();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(ar_remote);
            if (issuer && sidx + 1 < T) {                  // the dh of the last reverse step is unused
                mbar_wait_cluster(a_ready, sidx & 1);
                tc_fence_after();
                issue();
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_pair<64>(tmem_base);
}

// Both weight images of one layer from W_hh of the two directions ([4H][H] fp32 each), hi parts then (split) lo parts,
// lo = bf16(w - hi):
//   fwd [2][16 (x2)][4H = 512 rows][8]: element (d, part * 16 + c, n, e) = W_d[n][8 c + e]     (B operand of h W_hh^T)
//   bwd [2][64 (x2)][H = 128 rows][8]:  element (d, part * 64 + c, u, e) = W_d[8 c + e][u]     (B operand of dG W_hh)
__global__ void lstm_pack_kernel(const float* __restrict__ w0, const float* __restrict__ w1, int split, uint4* __restrict__ fwd,
                                 uint4* __restrict__ bwd, long long n_f, long long n_total) {
    const int nf = 16 * (1 + split), nb = 64 * (1 + split);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_total; e += (long long)gridDim.x * blockDim.x) {
        float v[8];
        int part;
        if (e < n_f) {
            const int d = (int)(e / (nf * 512)), rem = (int)(e % (nf * 512));
            const int c = rem / 512, n = rem % 512;
            part = c / 16;
            const float* w = (d ? w1 : w0) + (long long)n * H + (c % 16) * 8;
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __ldg(w + i);
        } else {
            const long long f = e - n_f;
            const int d = (int)(f / (nb * 128)), rem = (int)(f % (nb * 128));
            const int c = rem / 128, u = rem % 128;
            part = c / 64;
            const float* w = (d ? w1 : w0) + (long long)((c % 64) * 8) * H + u;
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = __ldg(w + (long long)i * H);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float hi = __bfloat162float(__float2bfloat16_rn(v[i]));
            v[i] = part ? v[i] - hi : hi;
        }
        (e < n_f ? fwd[e] : bwd[e - n_f]) = pack8(v);
    }
}

Seq mk(const float* p, int64_t ld, int64_t rows, int64_t row0) {
    Seq s;
    s.p = const_cast<float*>(p);
    s.ld = ld; s.rows = rows; s.row0 = row0;
    return s;
}

}  // namespace

extern "C" int rs_lstm_pack_weights_bf16(const float* w_hh, const float* w_hh_r, int H_, int split, void* fwd_img, void* bwd_img,
                                         void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(H_ == H, "rs_lstm_pack_weights_bf16: hidden size %d: the bf16 LSTM recurrence exists for H = 128 (d_model 256) only", H_);
    RS_REQUIRE(w_hh && w_hh_r && fwd_img && bwd_img, "rs_lstm_pack_weights_bf16: bad arguments");
    split = split ? 1 : 0;
    const long long n_f = 2LL * 16 * (1 + split) * 512, n_total = n_f + 2LL * 64 * (1 + split) * 128;
    lstm_pack_kernel<<<(int)((n_total + 255) / 256), 256, 0, stream>>>(w_hh, w_hh_r, split, static_cast<uint4*>(fwd_img),
                                                                      static_cast<uint4*>(bwd_img), n_f, n_total);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_lstm_fwd_bf16(const float* P, int64_t p_ld, int64_t p_rows, int64_t p_row0, const void* w_img, float* out,
                                int64_t o_ld, int64_t o_rows, int64_t o_row0, float* saved, int B, int T, int H_, int split,
                                void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(H_ == H, "rs_lstm_fwd_bf16: hidden size %d: the bf16 LSTM recurrence exists for H = 128 (d_model 256) only", H_);
    if (B == 0 || T == 0) return 0;
    RS_REQUIRE(P && w_img && out && B > 0 && T > 0, "rs_lstm_fwd_bf16: bad arguments");
    RS_REQUIRE(p_ld % 4 == 0 && o_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(P) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0
               && (reinterpret_cast<uintptr_t>(saved) & 15) == 0,
               "rs_lstm_fwd_bf16: P, out and saved must be 16-byte aligned with row strides a multiple of 4 floats");
    FwdParams p = {};
    p.P = mk(P, p_ld, p_rows, p_row0); p.out = mk(out, o_ld, o_rows, o_row0);
    p.w = static_cast<const uint8_t*>(w_img); p.saved = saved;
    p.B = B; p.T = T; p.split = split ? 1 : 0;
    const int smem = 16 * (1 + p.split) * W_CHUNK_F + 16 * CHUNK_S + 64;
    const dim3 grid(2 * ((B + 127) / 128), 2);
    RS_CUDA_OK(cudaFuncSetAttribute(lstm_fwd_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    lstm_fwd_bf16_kernel<<<grid, NUM_THREADS, smem, stream>>>(p);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_lstm_bwd_bf16(const float* d_out, int64_t do_ld, int64_t do_rows, int64_t do_row0, const float* saved,
                                const void* w_img, float* dG, int64_t g_ld, int64_t g_rows, int64_t g_row0, int B, int T, int H_,
                                int split, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(H_ == H, "rs_lstm_bwd_bf16: hidden size %d: the bf16 LSTM recurrence exists for H = 128 (d_model 256) only", H_);
    if (B == 0 || T == 0) return 0;
    RS_REQUIRE(d_out && saved && w_img && dG && B > 0 && T > 0, "rs_lstm_bwd_bf16: bad arguments");
    RS_REQUIRE(do_ld % 4 == 0 && g_ld % 4 == 0 && (reinterpret_cast<uintptr_t>(d_out) & 15) == 0 && (reinterpret_cast<uintptr_t>(dG) & 15) == 0
               && (reinterpret_cast<uintptr_t>(saved) & 15) == 0,
               "rs_lstm_bwd_bf16: d_out, saved and dG must be 16-byte aligned with row strides a multiple of 4 floats");
    BwdParams p = {};
    p.d_out = mk(d_out, do_ld, do_rows, do_row0); p.dG = mk(dG, g_ld, g_rows, g_row0);
    p.saved = saved; p.w = static_cast<const uint8_t*>(w_img);
    p.B = B; p.T = T; p.split = split ? 1 : 0;
    const int smem = 64 * (1 + p.split) * CHUNK_S + 64 * CHUNK_S + 64;
    const dim3 grid(2 * ((B + 127) / 128), 2);
    RS_CUDA_OK(cudaFuncSetAttribute(lstm_bwd_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    lstm_bwd_bf16_kernel<<<grid, NUM_THREADS, smem, stream>>>(p);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
