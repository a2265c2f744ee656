// Persistent tensor-core GRU recurrence for H = 256 (BASELINE config 4: H 256, T 4000), forward and backward through time.
// Same CTA-pair structure as rec_pair.cu (tcgen05 cta_group::2, M = 128: 64 traces per CTA, every TMEM lane busy, lane half
// = half of the hidden units), same tile-major operands -- but W_hh (3H x H bf16 = 384 KB) no longer fits: half of it per
// CTA would be 192 KB next to the h tile and the fp32 master state.  So W is NOT resident: each CTA streams its half
// (the gate rows of its 128 hidden units) from L2 through a ring of 24 KB bulk copies (cp.async.bulk, mbarrier full /
// empty pairs; RING_STAGES = 4 stages), once per time step, while the tensor core consumes it K = 16 step by K = 16 step.  The ring
// runs ahead of the recurrence: most of step t+1's weights land during the epilogue of step t, the rest under the MMA
// itself.  The whole of W_hh for both directions is 768 KB and stays L2-resident; 32 CTAs at batch 1024 pull ~2 TB/s from
// L2, nothing from HBM.  (An odd CTA's stage arrival is relayed to the issuing CTA by its otherwise idle warp 0.)
//   forward : G[64 x 768 per CTA] = h_{t-1}[64 x 256] . W_hh^T, 3 MMAs (N = 256: r, z, hn) per K step, 16 (+1) K steps
//   backward: dh[64 x 256] = z (.) dh + dGh[64 x 768] . W_hh,   1 MMA (N = 256) per K step, 48 K steps
// The epilogues are those of rec_pair.cu with 32 hidden units per thread (16 warps per CTA).

#include "common.cuh"
#include "rec_common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

using namespace rs;

constexpr int HW = 256;
constexpr int ROWS = 64;
constexpr int CHUNK_G = 2048;
constexpr int CHUNK_S = ROWS * 16;
constexpr int WSTAGE = 24576;                   // one ring stage: fwd 2 K steps x [2 chunks][384 rows][16 B], bwd 6 x [2][128][16 B]
constexpr int NSTAGE_MAX = 7;                  // ring depth: 5 stages next to the fp32 master state in shared memory, 7 when it lives in TMEM
constexpr int A_FWD_BYTES = (HW / 8 + 2) * CHUNK_S;     // 34 KB: h tile + the layer-0 input chunks of one K step
constexpr int H32_BYTES = (HW / 4) * CHUNK_S;           // 64 KB: fp32 master copy of h
constexpr int A_BWD_BYTES = (3 * HW / 8) * CHUNK_S;     // 96 KB: dGh tile
constexpr int NUM_THREADS = 64 + 512;                   // warp 0: MMA issuer (even CTA) / ring relay (odd CTA), warp 1: ring producer
constexpr int UPT = 32, NGRP = 4;                       // hidden units / 16-byte chunks per epilogue thread and step

struct FwdWideParams {
    const float* x; int I;
    const uint8_t* P; long long p_block_bytes;
    const uint8_t* Wst;                     // [2 dirs][2 ranks][stages per step][WSTAGE] streaming image (see rs_rec_fwd_bf16_wide)
    const float* b_hn;                      // [2][256]
    uint8_t* out; long long out_block_bytes;
    uint8_t* gates;                         // [tiles][T][2][128 chunks][128][8] fp16 or NULL
    float* h_n;
    const int* lengths;
    const uint8_t* drop_bits; const float* drop_scale; uint8_t* out_drop;
    int B, T, n_tiles;
    int nstage;                             // ring depth (2 .. NSTAGE_MAX)
};

struct RingBars {
    uint64_t full[NSTAGE_MAX];       // this CTA's stage landed (bulk-copy transaction bytes)
    uint64_t peer_full[NSTAGE_MAX];  // even CTA only: the odd CTA's stage landed (relayed)
    uint64_t empty[NSTAGE_MAX];      // the MMAs that read the stage retired (multicast commit)
};

// Ring producer: one thread per CTA streams this CTA's weight stages, `sps` stages per time step, T steps.
// `prefetch(step)` is called once per time step, before that step's first stage: the producer is the one thread of the CTA
// that runs ahead of the recurrence, so it also pulls the activations of a later step from HBM into L2.
template <class Prefetch>
__device__ __forceinline__ void ring_produce(RingBars* rb, uint8_t* ring, const uint8_t* wimg, int sps, long long total, int NSTAGE,
                                             Prefetch prefetch) {
    for (long long it = 0; it < total; ++it) {
        const int st = it % NSTAGE;
        if (it % sps == 0) prefetch(static_cast<int>(it / sps));
        if (it >= NSTAGE) mbar_wait(&rb->empty[st], ((it / NSTAGE) - 1) & 1);
        mbar_expect_tx(&rb->full[st], WSTAGE);
        bulk_load(ring + st * WSTAGE, wimg + (it % sps) * (long long)WSTAGE, WSTAGE, &rb->full[st]);
    }
}
// Odd CTA: tells the issuing CTA that its stage landed.
__device__ __forceinline__ void ring_relay(RingBars* rb, long long total, int NSTAGE) {
    uint32_t remote[NSTAGE_MAX];
    for (int i = 0; i < NSTAGE_MAX; ++i) remote[i] = mapa_cluster(smem_u32(&rb->peer_full[i]), 0);
    for (long long it = 0; it < total; ++it) {
        const int st = it % NSTAGE;
        mbar_wait(&rb->full[st], (it / NSTAGE) & 1);
        mbar_arrive_cluster(remote[st]);
    }
}

// kVarLen / kDrop: packed variable-length traces / inter-layer dropout as template parameters (their selects, mask tests and the
// masked copy cost instructions in the epilogue chain that bounds a time step even when unused)
// kXC (layer 0): the 16-byte input chunks per row of the (kXC + 1) / 2 input K steps (rec_common.cuh has the column map): 1
// for I <= 2 (the one K step's second chunk stays zero), else x_chunks(I); the chunk ch is loaded and packed by the row's
// thread ch (8 per row) before the wait for the accumulator and stored into the A tile after the epilogue.
template <bool kFusedX, bool kVarLen, bool kDrop, int kXC = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) rec_fwd_wide_kernel(const FwdWideParams p) {
    static_assert(kXC == 1 || (kFusedX && kXC % 2 == 0 && kXC <= 2 * x_steps(kMaxXInputs)), "input chunks per row");
    constexpr int kXS = (kXC + 1) / 2;                     // input K steps
    constexpr int A_BYTES = (HW / 8 + 2 * kXS) * CHUNK_S;  // h tile + the input chunks
    constexpr int kXCW = kXC < x_col(kMaxXInputs - 1, 2) / 8 + 1 ? kXC : x_col(kMaxXInputs - 1, 2) / 8 + 1;  // chunks that can be nonzero
    // fp32 master copy of h: layer 0 needs all 512 TMEM columns for its accumulators (r | z | W_hn h | W_in x), so the state
    // lives in shared memory; deeper layers keep it in the 128 spare TMEM columns (64 KB of shared memory less: the L1 cache
    // that backs the epilogue's global loads grows by as much)
    constexpr bool kTmemState = !kFusedX;
    const int NSTAGE = p.nstage;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* ring = smem;                                  // [NSTAGE][WSTAGE]
    uint8_t* a_s = ring + NSTAGE * WSTAGE;                 // [32 + 2 kXS chunks][64 rows][16 B]
    uint8_t* h32_s = a_s + A_BYTES;                        // [64 chunks of 4 floats][64 rows][16 B]  (layer 0 only)
    float* bhn_s = reinterpret_cast<float*>(h32_s + (kTmemState ? 0 : H32_BYTES));
    RingBars* rb = reinterpret_cast<RingBars*>(bhn_s + HW);
    uint64_t* h_ready = reinterpret_cast<uint64_t*>(rb + 1);
    uint64_t* acc_full = h_ready + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    constexpr int KS = HW / 16 + (kFusedX ? kXS : 0);      // K = 16 steps per time step
    constexpr int SPS = (KS + 1) / 2;                      // ring stages per time step (2 K steps each)
    const uint32_t rank = cluster_ctarank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y;
    const int tile = blockIdx.x >> 1;
    const int T = p.T;
    const long long total_stages = (long long)T * SPS;

    if (threadIdx.x == 0) {
        for (int i = 0; i < NSTAGE_MAX; ++i) { mbar_init(&rb->full[i], 1); mbar_init(&rb->peer_full[i], 1); mbar_init(&rb->empty[i], 1); }
        mbar_init(h_ready, 2 * 16);
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc_pair<512>(tmem_slot);
    for (int i = threadIdx.x; i < HW; i += blockDim.x) bhn_s[i] = p.b_hn[dir * HW + i];
    for (int i = threadIdx.x; i < (A_BYTES + (kTmemState ? 0 : H32_BYTES)) / 16; i += blockDim.x)
        reinterpret_cast<uint4*>(a_s)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (kXC == 1) {
        if (kFusedX && threadIdx.x < ROWS) {
            const long long b = (long long)tile * 128 + rank * ROWS + threadIdx.x;
            *reinterpret_cast<uint4*>(a_s + (HW / 8) * CHUNK_S + threadIdx.x * 16) =
                pack_x(b < p.B ? p.x + (b * T + (dir ? T - 1 : 0)) * p.I : nullptr, p.I);
        }
    } else {
        for (int i = threadIdx.x; i < kXCW * ROWS; i += blockDim.x) {
            const int rl = i % ROWS, ch = i / ROWS;
            const long long b = (long long)tile * 128 + rank * ROWS + rl;
            *reinterpret_cast<uint4*>(a_s + (HW / 8 + ch) * CHUNK_S + rl * 16) =
                pack_x_chunk(b < p.B ? p.x + (b * T + (dir ? T - 1 : 0)) * p.I : nullptr, p.I, ch);
        }
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    for (int i = threadIdx.x; i < 2 * (HW / 8) * ROWS; i += blockDim.x) {      // pad rows t' = 0, T + 1 of this CTA's rows
        const int rl = i % ROWS, c = (i / ROWS) % (HW / 8), pad = i / (ROWS * (HW / 8));
        const long long off = ((long long)tile * (T + 2) + (pad ? T + 1 : 0)) * p.out_block_bytes
                              + (long long)(dir * (HW / 8) + c) * CHUNK_G + (rank * ROWS + rl) * 16;
        stg16(p.out + off, make_uint4(0, 0, 0, 0));
        if (kDrop) stg16(p.out_drop + off, make_uint4(0, 0, 0, 0));
    }

    if (warp == 1) {
        if (elect_one()) {      // (elect.sync, not lane == 0: ptxas then issues the bulk copies without a per-instruction ELECT loop)
            // the producer runs about one time step ahead of the epilogue: prefetching step + 2 puts ~2 steps between the
            // HBM read and its use (this CTA's half of the projection block: 48 of the 96 chunks of its direction)
            auto prefetch = [&](int step) {
                const int s2 = step + 2;
                if (kFusedX || s2 >= T) return;
                const int t = dir ? (T - 1 - s2) : s2;
                const long long blk = (long long)tile * (T + 2) + t + 1;
                l2_prefetch(p.P + blk * p.p_block_bytes + (long long)(dir * 96 + rank * 48) * CHUNK_G, 48 * CHUNK_G);
            };
            ring_produce(rb, ring, p.Wst + ((long long)dir * 2 + rank) * SPS * WSTAGE, SPS, total_stages, NSTAGE, prefetch);
        }
    } else if (warp == 0) {
        if (rank == 1) {
            if (lane == 0) ring_relay(rb, total_stages, NSTAGE);
        } else {
            // ===================== MMA issuer for the pair =====================
            constexpr uint32_t idesc = umma_idesc_bf16(128, 256, 0, 0);
            const uint32_t a_addr = smem_u32(a_s), r_addr = smem_u32(ring);
            long long it = 0;
            for (int step = 0; step < T; ++step) {
                if (step > 0) {
                    mbar_wait(h_ready, (step - 1) & 1);
                    tc_fence_after();
                }
                for (int sidx = 0; sidx < SPS; ++sidx, ++it) {
                    const int st = it % NSTAGE;
                    const uint32_t ph = (it / NSTAGE) & 1;
                    mbar_wait(&rb->full[st], ph);
                    mbar_wait(&rb->peer_full[st], ph);
                    tc_fence_after();
                    if (elect_one()) {      // back-to-back UTCHMMA (a lane == 0 guard costs an ELECT loop of ~13 instructions per MMA)
#pragma unroll
                        for (int kk = 0; kk < 2; ++kk) {
                            const int ks = sidx * 2 + kk;
                            if (ks >= KS) break;
                            const uint32_t wb = r_addr + st * WSTAGE + kk * (WSTAGE / 2);
                            const uint64_t da = umma_desc_noswz(a_addr + ks * 2 * CHUNK_S, CHUNK_S, 128);
                            const uint64_t db_r = umma_desc_noswz(wb, 384 * 16, 128);
                            const uint64_t db_z = umma_desc_noswz(wb + 128 * 16, 384 * 16, 128);
                            const uint64_t db_n = umma_desc_noswz(wb + 256 * 16, 384 * 16, 128);
                            if (!kFusedX || ks < HW / 16) {
                                tc_mma_bf16_pair(tmem_base, da, db_r, idesc, ks != 0);           // r    -> columns [0, 128) of each lane half
                                tc_mma_bf16_pair(tmem_base + 128, da, db_z, idesc, ks != 0);     // z    -> [128, 256)
                                tc_mma_bf16_pair(tmem_base + 256, da, db_n, idesc, ks != 0);     // W_hn h -> [256, 384)
                            } else {        // layer 0: the input chunks (hi / lo split x and bias against hi / lo split W_ih)
                                tc_mma_bf16_pair(tmem_base, da, db_r, idesc, 1u);
                                tc_mma_bf16_pair(tmem_base + 128, da, db_z, idesc, 1u);
                                tc_mma_bf16_pair(tmem_base + 384, da, db_n, idesc, kXS == 1 ? 0u : (ks != HW / 16));   // W_in x + b_in -> [384, 512)
                            }
                        }
                        tc_commit_pair(&rb->empty[st]);
                        if (sidx == SPS - 1) tc_commit_pair(acc_full);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        // ===================== epilogue =====================
        const int wg = (warp - 2) >> 2;                    // which 32 of this lane half's 128 hidden units
        const int q = warp & 3;
        const int uh = q >> 1;
        const int rl = (q & 1) * 32 + lane;
        const int row = rank * ROWS + rl;
        const long long b = (long long)tile * 128 + row;
        const bool live = b < p.B;
        const int ub = uh * 128 + wg * UPT;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + wg * UPT;
        uint8_t* a_row = a_s + rl * 16;
        uint8_t* h32_row = h32_s + rl * 16;
        const uint32_t hr_remote = mapa_cluster(smem_u32(h_ready), 0);
        const float* xrow = p.x ? p.x + b * T * p.I : nullptr;
        const int len = (kVarLen && live) ? p.lengths[b] : T;
        const float dscale = kDrop ? __ldg(p.drop_scale) : 1.0f;
        if (kTmemState) {                                  // h_0 = 0 in the TMEM-resident master state
            uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
            for (int grp = 0; grp < NGRP; ++grp) tmem_st_32x32b_x8(taddr + 384 + grp * 8, zero);
            tmem_st_wait();
        }
        // running pointers of this thread's pieces: one signed stride per time step instead of 64-bit index arithmetic
        const int t_first = dir ? T - 1 : 0;
        const long long blk_first = (long long)tile * (T + 2) + t_first + 1;
        uint8_t* o_cur = p.out + blk_first * p.out_block_bytes + (long long)(dir * (HW / 8) + ub / 8) * CHUNK_G + row * 16;
        const long long o_step = dir ? -p.out_block_bytes : p.out_block_bytes;
        const long long od_delta = kDrop ? p.out_drop - p.out : 0;
        const uint8_t* p_cur = kFusedX ? nullptr : p.P + blk_first * p.p_block_bytes + (long long)(dir * (3 * HW / 8) + ub / 8) * CHUNK_G + row * 16;
        const long long p_step = dir ? -p.p_block_bytes : p.p_block_bytes;
        uint8_t* g_cur = p.gates ? p.gates + (((long long)tile * T + t_first) * 2 + dir) * ((long long)(4 * HW / 8) * CHUNK_G)
                                             + (long long)(ub / 8) * CHUNK_G + row * 16 : nullptr;
        const long long g_step = (dir ? -2 : 2) * ((long long)(4 * HW / 8) * CHUNK_G);
        const uint8_t* db_cur = kDrop ? p.drop_bits + (((long long)tile * T + t_first) * 128 + row) * (2 * HW / 8) + dir * (HW / 8) + ub / 8 : nullptr;
        const long long db_step = dir ? -128 * (2 * HW / 8) : 128 * (2 * HW / 8);

        for (int step = 0; step < T; ++step) {
            const int t = dir ? (T - 1 - step) : step;
            const bool active = !kVarLen || t < len;
            const uint8_t* pblk = p_cur;
            uint8_t* const o_ptr = o_cur;
            uint8_t* const od_ptr = o_cur + od_delta;
            uint8_t* gblk = g_cur;
            uint32_t dbits = 0;
            if (kDrop) {
                dbits = __ldg(reinterpret_cast<const uint32_t*>(db_cur));
                db_cur += db_step;
            }
            o_cur += o_step;
            if (!kFusedX) p_cur += p_step;
            if (g_cur) g_cur += g_step;
            uint4 xnext = make_uint4(0, 0, 0, 0);
            const int x_ui = ub / UPT;                     // this thread's place among the 8 of its row
            const bool write_x = kFusedX && (kXC == 1 ? ub == 0 : x_ui < kXCW) && step + 1 < T;
            if (write_x) {
                const float* xp = live ? xrow + (long long)(dir ? t - 1 : t + 1) * p.I : nullptr;
                if (kXC == 1) xnext = pack_x(xp, p.I);
                else {              // chunk x_ui (a warp-uniform switch: the column map of each case is a compile-time constant)
#define RS_PACK_X(U) case U: if (U < kXCW) xnext = pack_x_chunk(xp, p.I, U); break
                    switch (x_ui) { RS_PACK_X(0); RS_PACK_X(1); RS_PACK_X(2); RS_PACK_X(3); RS_PACK_X(4); RS_PACK_X(5); RS_PACK_X(6); }
#undef RS_PACK_X
                }
            }
            uint4 pv[3];
            auto load_p = [&](int grp) {
#pragma unroll
                for (int g = 0; g < 3; ++g) pv[g] = ldg16(pblk + (long long)(g * (HW / 8) + grp) * CHUNK_G);
            };
            if (!kFusedX) load_p(0);
            mbar_wait(acc_full, step & 1);
            tc_fence_after();
            uint4 last_o, last_d = make_uint4(0, 0, 0, 0), last_r, last_z, last_n, last_h;
#pragma unroll
            for (int grp = 0; grp < NGRP; ++grp) {
                const int u0 = ub + grp * 8;
                uint32_t ar[8], az[8], an[8], ax[8];            // ax: layer 0 W_in x + b_in; deeper layers: the fp32 master state
                tmem_ld_32x32b_x8(taddr + grp * 8, ar);
                tmem_ld_32x32b_x8(taddr + 128 + grp * 8, az);
                tmem_ld_32x32b_x8(taddr + 256 + grp * 8, an);
                tmem_ld_32x32b_x8(taddr + 384 + grp * 8, ax);
                uint32_t hnew[8];
                uint4 pc[3];
                if (!kFusedX) {
                    pc[0] = pv[0]; pc[1] = pv[1]; pc[2] = pv[2];
                    if (grp < NGRP - 1) load_p(grp + 1);
                }
                tmem_ld_wait();
                uint32_t wo[4], wd[4], wr[4], wz[4], wn[4], wh[4];
#pragma unroll
                for (int jp = 0; jp < 4; ++jp) {
                    float hv2[2], rv2[2], zv2[2], nv2[2], hnv2[2], od2[2];
                    const float2 ho2 = kTmemState ? make_float2(__uint_as_float(ax[2 * jp]), __uint_as_float(ax[2 * jp + 1]))
                                                  : *reinterpret_cast<const float2*>(h32_row + (u0 / 4 + jp / 2) * CHUNK_S + (jp & 1) * 8);
                    const float2 bh2 = *reinterpret_cast<const float2*>(bhn_s + u0 + 2 * jp);
                    float2 pr2 = make_float2(0.f, 0.f), pz2 = pr2, pn2 = pr2;
                    if (!kFusedX) {
                        const uint32_t* w0 = reinterpret_cast<const uint32_t*>(&pc[0]);
                        const uint32_t* w1 = reinterpret_cast<const uint32_t*>(&pc[1]);
                        const uint32_t* w2 = reinterpret_cast<const uint32_t*>(&pc[2]);
                        pr2 = bf2_to_f2(w0[jp]); pz2 = bf2_to_f2(w1[jp]); pn2 = bf2_to_f2(w2[jp]);
                    } else {
                        pn2 = make_float2(__uint_as_float(ax[2 * jp]), __uint_as_float(ax[2 * jp + 1]));
                    }
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int j = 2 * jp + e;
                        const float ho = e ? ho2.y : ho2.x;
                        const float ar_ = kFusedX ? __uint_as_float(ar[j]) : __uint_as_float(ar[j]) + (e ? pr2.y : pr2.x);
                        const float az_ = kFusedX ? __uint_as_float(az[j]) : __uint_as_float(az[j]) + (e ? pz2.y : pz2.x);
                        const float r = fmaf(0.5f, tanh_fast(ar_), 0.5f);
                        const float z = active ? fmaf(0.5f, tanh_fast(az_), 0.5f) : 1.0f;
                        const float hn = __uint_as_float(an[j]) + (e ? bh2.y : bh2.x);
                        const float n = tanh_fast(fmaf(r, hn, e ? pn2.y : pn2.x));
                        const float h = active ? fmaf(z, ho - n, n) : ho;
                        hv2[e] = h; rv2[e] = r; zv2[e] = z; nv2[e] = n; hnv2[e] = hn;
                        if (kDrop) od2[e] = (active && ((dbits >> (grp * 8 + j)) & 1u)) ? h * dscale : 0.0f;
                    }
                    if (kTmemState) { hnew[2 * jp] = __float_as_uint(hv2[0]); hnew[2 * jp + 1] = __float_as_uint(hv2[1]); }
                    else *reinterpret_cast<float2*>(h32_row + (u0 / 4 + jp / 2) * CHUNK_S + (jp & 1) * 8) = make_float2(hv2[0], hv2[1]);
                    wo[jp] = f2_to_bf2(hv2[0], hv2[1]);
                    if (kDrop) wd[jp] = f2_to_bf2(od2[0], od2[1]);
                    wr[jp] = f2_to_h2(rv2[0], rv2[1]); wz[jp] = f2_to_h2(zv2[0], zv2[1]);
                    wn[jp] = f2_to_h2(nv2[0], nv2[1]); wh[jp] = f2_to_h2(hnv2[0], hnv2[1]);
                }
                if (kTmemState) tmem_st_32x32b_x8(taddr + 384 + grp * 8, hnew);
                const uint4 o0 = make_uint4(wo[0], wo[1], wo[2], wo[3]);
                *reinterpret_cast<uint4*>(a_row + (u0 / 8) * CHUNK_S) = o0;
                const uint4 so = active ? o0 : make_uint4(0, 0, 0, 0), sd = make_uint4(wd[0], wd[1], wd[2], wd[3]);
                const uint4 sr = make_uint4(wr[0], wr[1], wr[2], wr[3]), sz = make_uint4(wz[0], wz[1], wz[2], wz[3]);
                const uint4 sn = make_uint4(wn[0], wn[1], wn[2], wn[3]), sh = make_uint4(wh[0], wh[1], wh[2], wh[3]);
                if (grp < NGRP - 1) {
                    stg16(o_ptr + (long long)grp * CHUNK_G, so);
                    if (kDrop) stg16(od_ptr + (long long)grp * CHUNK_G, sd);
                    if (gblk) {
                        stg16(gblk + (long long)(0 * (HW / 8) + grp) * CHUNK_G, sr);
                        stg16(gblk + (long long)(1 * (HW / 8) + grp) * CHUNK_G, sz);
                        stg16(gblk + (long long)(2 * (HW / 8) + grp) * CHUNK_G, sn);
                        stg16(gblk + (long long)(3 * (HW / 8) + grp) * CHUNK_G, sh);
                    }
                } else {                // the last chunk's global stores wait until after the arrival (below)
                    last_o = so; last_d = sd; last_r = sr; last_z = sz; last_n = sn; last_h = sh;
                }
            }
            if (write_x) *reinterpret_cast<uint4*>(a_row + (HW / 8 + (kXC == 1 ? 0 : x_ui)) * CHUNK_S) = xnext;
            if (kTmemState) tmem_st_wait();
            fence_proxy_async();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(hr_remote);
            // the MEMBAR inside fence.proxy.async waits for the thread's global stores still in flight: the last chunk's are
            // issued only now, under the wait for the next MMA (rec_pair.cu has the measurement)
            stg16(o_ptr + (long long)(NGRP - 1) * CHUNK_G, last_o);
            if (kDrop) stg16(od_ptr + (long long)(NGRP - 1) * CHUNK_G, last_d);
            if (gblk) {
                stg16(gblk + (long long)(0 * (HW / 8) + NGRP - 1) * CHUNK_G, last_r);
                stg16(gblk + (long long)(1 * (HW / 8) + NGRP - 1) * CHUNK_G, last_z);
                stg16(gblk + (long long)(2 * (HW / 8) + NGRP - 1) * CHUNK_G, last_n);
                stg16(gblk + (long long)(3 * (HW / 8) + NGRP - 1) * CHUNK_G, last_h);
            }
        }
        // h_n: the fp32 master state after the last step (kept out of the step loop)
#pragma unroll
        for (int grp = 0; grp < NGRP; ++grp) {
            uint32_t hv[8];
            if (kTmemState) {
                tmem_ld_32x32b_x8(taddr + 384 + grp * 8, hv);
                tmem_ld_wait();
            } else {
#pragma unroll
                for (int i = 0; i < 8; i += 2) {
                    const float2 v = *reinterpret_cast<const float2*>(h32_row + ((ub + grp * 8 + i) / 4) * CHUNK_S + ((i >> 1) & 1) * 8);
                    hv[i] = __float_as_uint(v.x); hv[i + 1] = __float_as_uint(v.y);
                }
            }
            if (live) {
                float* dst = p.h_n + ((long long)dir * p.B + b) * HW + ub + grp * 8;
                *reinterpret_cast<uint4*>(dst) = make_uint4(hv[0], hv[1], hv[2], hv[3]);
                *reinterpret_cast<uint4*>(dst + 4) = make_uint4(hv[4], hv[5], hv[6], hv[7]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_pair<512>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------------
struct BwdWideParams {
    const uint8_t* d_out; long long dout_block_bytes;
    const float* d_h_n;
    const uint8_t* gates;
    const uint8_t* out; long long out_block_bytes;
    const uint8_t* WTst;                                 // [2 dirs][2 ranks][8 stages][WSTAGE]
    uint8_t* dG; long long dg_block_bytes;
    const int* lengths;
    const uint8_t* drop_bits; const float* drop_scale;
    int B, T, n_tiles;
    int nstage;
};

template <bool kVarLen, bool kDrop>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) rec_bwd_wide_kernel(const BwdWideParams p) {
    const int NSTAGE = p.nstage;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* ring = smem;
    uint8_t* a_s = ring + NSTAGE * WSTAGE;                 // [96 chunks][64 rows][16 B]  dGh_t
    RingBars* rb = reinterpret_cast<RingBars*>(a_s + A_BWD_BYTES);
    uint64_t* a_ready = reinterpret_cast<uint64_t*>(rb + 1);
    uint64_t* acc_full = a_ready + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_full + 1);

    constexpr int SPS = 8;                                 // 48 K steps per time step, 6 per ring stage
    const uint32_t rank = cluster_ctarank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y;
    const int tile = blockIdx.x >> 1;
    const int T = p.T;
    const long long total_stages = (long long)(T - 1) * SPS;   // the result of the last reverse step is unused

    if (threadIdx.x == 0) {
        for (int i = 0; i < NSTAGE_MAX; ++i) { mbar_init(&rb->full[i], 1); mbar_init(&rb->peer_full[i], 1); mbar_init(&rb->empty[i], 1); }
        mbar_init(a_ready, 2 * 16);
        mbar_init(acc_full, 1);
        fence_mbar_init();
    }
    if (warp == 0) tmem_alloc_pair<128>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    for (int i = threadIdx.x; i < 2 * (8 * HW / 16) * ROWS; i += blockDim.x) {     // pad rows of dG: this direction's 128 chunks
        const int rl = i % ROWS, c = (i / ROWS) % (8 * HW / 16), pad = i / (ROWS * (8 * HW / 16));
        const long long off = ((long long)tile * (T + 2) + (pad ? T + 1 : 0)) * p.dg_block_bytes
                              + (long long)(dir * (8 * HW / 16) + c) * CHUNK_G + (rank * ROWS + rl) * 16;
        stg16(p.dG + off, make_uint4(0, 0, 0, 0));
    }

    if (warp == 1) {
        if (elect_one()) {
            // saved gates (4 x 32 chunks), h_{t-1} and d_out (32 chunks each) of the reverse step two ahead: this CTA's half
            auto prefetch = [&](int sidx) {
                const int s2 = sidx + 2;
                if (s2 >= T) return;
                const int t = dir ? s2 : (T - 1 - s2);
                const int t_prev = dir ? t + 1 : t - 1;
                const long long blk = (long long)tile * (T + 2) + t + 1, blk_prev = (long long)tile * (T + 2) + t_prev + 1;
                l2_prefetch(p.gates + (((long long)tile * T + t) * 2 + dir) * (128LL * CHUNK_G) + (long long)(rank * 64) * CHUNK_G, 64 * CHUNK_G);
                l2_prefetch(p.out + blk_prev * p.out_block_bytes + (long long)(dir * 32 + rank * 16) * CHUNK_G, 16 * CHUNK_G);
                if (p.d_out) l2_prefetch(p.d_out + blk * p.dout_block_bytes + (long long)(dir * 32 + rank * 16) * CHUNK_G, 16 * CHUNK_G);
            };
            ring_produce(rb, ring, p.WTst + ((long long)dir * 2 + rank) * SPS * WSTAGE, SPS, total_stages, NSTAGE, prefetch);
        }
    } else if (warp == 0) {
        if (rank == 1) {
            if (lane == 0) ring_relay(rb, total_stages, NSTAGE);
        } else {
            constexpr uint32_t idesc = umma_idesc_bf16(128, 256, 0, 0);
            const uint32_t a_addr = smem_u32(a_s), r_addr = smem_u32(ring);
            long long it = 0;
            for (int sidx = 0; sidx < T - 1; ++sidx) {
                mbar_wait(a_ready, sidx & 1);
                tc_fence_after();
                for (int sg = 0; sg < SPS; ++sg, ++it) {
                    const int st = it % NSTAGE;
                    const uint32_t ph = (it / NSTAGE) & 1;
                    mbar_wait(&rb->full[st], ph);
                    mbar_wait(&rb->peer_full[st], ph);
                    tc_fence_after();
                    if (elect_one()) {
#pragma unroll
                        for (int kk = 0; kk < 6; ++kk) {
                            const int ks = sg * 6 + kk;
                            const uint64_t da = umma_desc_noswz(a_addr + ks * 2 * CHUNK_S, CHUNK_S, 128);
                            const uint64_t db = umma_desc_noswz(r_addr + st * WSTAGE + kk * 4096, 128 * 16, 128);
                            tc_mma_bf16_pair(tmem_base, da, db, idesc, 1u);     // accumulates onto the z (.) dh carry in TMEM
                        }
                        tc_commit_pair(&rb->empty[st]);
                        if (sg == SPS - 1) tc_commit_pair(acc_full);
                    }
                    __syncwarp();
                }
            }
        }
    } else {
        const int wg = (warp - 2) >> 2;
        const int q = warp & 3;
        const int uh = q >> 1;
        const int rl = (q & 1) * 32 + lane;
        const int row = rank * ROWS + rl;
        const long long b = (long long)tile * 128 + row;
        const bool live = b < p.B;
        const int ub = uh * 128 + wg * UPT;
        const int cb = ub / 8;
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + wg * UPT;
        uint8_t* a_row = a_s + rl * 16;
        const uint32_t ar_remote = mapa_cluster(smem_u32(a_ready), 0);
        const int len = (kVarLen && live) ? p.lengths[b] : T;
        const float dscale = kDrop ? __ldg(p.drop_scale) : 1.0f;
        constexpr int HC = HW / 8;                         // chunks per H columns
#pragma unroll
        for (int sc = 0; sc < NGRP; ++sc) {
            uint32_t init[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) init[j] = 0u;
            if (p.d_h_n && live) {
                const float* src = p.d_h_n + ((long long)dir * p.B + b) * HW + ub + sc * 8;
                const float4 v0 = __ldg(reinterpret_cast<const float4*>(src));
                const float4 v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
                init[0] = __float_as_uint(v0.x); init[1] = __float_as_uint(v0.y); init[2] = __float_as_uint(v0.z); init[3] = __float_as_uint(v0.w);
                init[4] = __float_as_uint(v1.x); init[5] = __float_as_uint(v1.y); init[6] = __float_as_uint(v1.z); init[7] = __float_as_uint(v1.w);
            }
            tmem_st_32x32b_x8(taddr + sc * 8, init);
        }
        tmem_st_wait();

        uint4 raw[6];
        uint32_t dbits_next = 0;
        // running pointers of this thread's pieces (one signed stride per time step instead of 64-bit index arithmetic)
        const int t_first = dir ? 0 : T - 1;
        const long long g_step = (dir ? 2 : -2) * ((long long)(4 * HC) * CHUNK_G);
        const long long o_step = dir ? p.out_block_bytes : -p.out_block_bytes;
        const long long do_step = dir ? p.dout_block_bytes : -p.dout_block_bytes;
        const long long dg_step = dir ? p.dg_block_bytes : -p.dg_block_bytes;
        const uint8_t* g_ptr = p.gates + (((long long)tile * T + t_first) * 2 + dir) * ((long long)(4 * HC) * CHUNK_G) + (long long)cb * CHUNK_G + row * 16;
        // h_{t-1}: the block of the step before in forward time (t - 1 for the forward direction, t + 1 for the reverse one)
        const uint8_t* hp_ptr = p.out + ((long long)tile * (T + 2) + t_first + (dir ? 1 : -1) + 1) * p.out_block_bytes
                                + (long long)(dir * HC + cb) * CHUNK_G + row * 16;
        const uint8_t* do_ptr = p.d_out ? p.d_out + ((long long)tile * (T + 2) + t_first + 1) * p.dout_block_bytes
                                          + (long long)(dir * HC + cb) * CHUNK_G + row * 16 : nullptr;
        const uint8_t* db_next = kDrop ? p.drop_bits + (((long long)tile * T + t_first) * 128 + row) * (2 * HC) + dir * HC + cb : nullptr;
        const long long db_step = dir ? 128 * (2 * HC) : -128 * (2 * HC);
        uint8_t* dg_cur = p.dG + ((long long)tile * (T + 2) + t_first + 1) * p.dg_block_bytes + (long long)(dir * 4 * HC + cb) * CHUNK_G + row * 16;
        auto load_raw = [&](int sc) {                      // chunk sc of the step the pointers stand at
#pragma unroll
            for (int g = 0; g < 4; ++g) raw[g] = ldg16(g_ptr + (long long)(g * HC + sc) * CHUNK_G);
            raw[4] = ldg16(hp_ptr + (long long)sc * CHUNK_G);
            raw[5] = do_ptr ? ldg16(do_ptr + (long long)sc * CHUNK_G) : make_uint4(0, 0, 0, 0);
        };
        load_raw(0);
        if (kDrop) dbits_next = __ldg(reinterpret_cast<const uint32_t*>(db_next));
        for (int sidx = 0; sidx < T; ++sidx) {
            const int t = dir ? sidx : (T - 1 - sidx);
            const bool active = !kVarLen || t < len;
            uint8_t* dgblk = dg_cur;
            dg_cur += dg_step;
            const uint32_t dbits = dbits_next;
            if (kDrop && sidx + 1 < T) {                   // next step's mask word: requested a whole step ahead
                db_next += db_step;
                dbits_next = __ldg(reinterpret_cast<const uint32_t*>(db_next));
            }
            if (sidx > 0) {
                mbar_wait(acc_full, (sidx - 1) & 1);
                tc_fence_after();
            }
#pragma unroll
            for (int sc = 0; sc < NGRP; ++sc) {
                uint32_t acc[8];
                tmem_ld_32x32b_x8(taddr + sc * 8, acc);
                uint4 cur[6];
#pragma unroll
                for (int i = 0; i < 6; ++i) cur[i] = raw[i];
                if (sc < NGRP - 1) load_raw(sc + 1);
                float r[8], z[8], n[8], hn[8], hp[8], dout[8];
                unpack8h(cur[0], r); unpack8h(cur[1], z); unpack8h(cur[2], n); unpack8h(cur[3], hn);
                unpack8(cur[4], hp); unpack8(cur[5], dout);
                tmem_ld_wait();
                float gr[8], gz[8], gn[8], ghn[8];
                uint32_t carry[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float dov = active ? dout[j] : 0.0f;
                    if (kDrop) dov = ((dbits >> (sc * 8 + j)) & 1u) ? dov * dscale : 0.0f;
                    const float dh = __uint_as_float(acc[j]) + dov;
                    const float omz = 1.0f - z[j];
                    gn[j] = dh * omz * fmaf(-n[j], n[j], 1.0f);
                    gz[j] = dh * (hp[j] - n[j]) * (z[j] * omz);
                    ghn[j] = gn[j] * r[j];
                    gr[j] = ghn[j] * (hn[j] * (1.0f - r[j]));
                    carry[j] = __float_as_uint(dh * z[j]);
                }
                const uint4 vr = pack8(gr), vz = pack8(gz), vn = pack8(gn), vh = pack8(ghn);
                *reinterpret_cast<uint4*>(a_row + (0 * HC + cb + sc) * CHUNK_S) = vr;       // K order r | z | hn
                *reinterpret_cast<uint4*>(a_row + (1 * HC + cb + sc) * CHUNK_S) = vz;
                *reinterpret_cast<uint4*>(a_row + (2 * HC + cb + sc) * CHUNK_S) = vh;
                stg16(dgblk + (long long)(0 * HC + sc) * CHUNK_G, vr);
                stg16(dgblk + (long long)(1 * HC + sc) * CHUNK_G, vz);
                stg16(dgblk + (long long)(2 * HC + sc) * CHUNK_G, vn);
                stg16(dgblk + (long long)(3 * HC + sc) * CHUNK_G, vh);
                tmem_st_32x32b_x8(taddr + sc * 8, carry);
            }
            tmem_st_wait();
            fence_proxy_async();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(ar_remote);
            // the next step's first chunk is requested after the arrival: no load in flight at the MEMBAR of fence.proxy.async
            if (sidx + 1 < T) {
                g_ptr += g_step; hp_ptr += o_step;
                if (do_ptr) do_ptr += do_step;
                load_raw(0);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_pair<128>(tmem_base);
}

// Ring depth of the weight stream, the same in all three launches (layer 0 forward, deeper forward, backward).  More stages
// hide more of the L2 latency of the weight stream but every 24 KB of shared memory is taken from the L1 cache that backs
// the epilogue's global loads (measured, tools/c4_probe.py: see DESIGN.md 4.4).
constexpr int RING_STAGES = 4;

}  // namespace

/* Forward for H = 256.  Wst: [2 dirs][2 ranks][8 + (x_steps(I) + 1) / 2 or 8 stages][2 K steps][2 chunks][384 rows][8] bf16,
 * rows = r | z | n gate rows of hidden units [128 rank, 128 rank + 128) (r, z scaled by 1/2), K step k = hidden units
 * [16 k, 16 k + 16); layer 0: K steps 16 .. 15 + x_steps(I) = the input columns (rec_common.cuh: W_ih hi, hi, lo per input,
 * b_hi, b_lo), zero K steps up to the whole stage. */
extern "C" int rs_rec_fwd_bf16_wide(const float* x, int I, const void* P, const void* Wst, const float* b_hn, void* out,
                                    void* gates, float* h_n, const int* lengths, const void* drop_bits,
                                    const float* drop_scale, void* out_drop, int B, int T, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;
    RS_REQUIRE((x != nullptr) != (P != nullptr), "rs_rec_fwd_bf16_wide: exactly one of x (layer 0) and P (deeper layers) must be given");
    RS_REQUIRE(!x || (I >= 1 && I <= rs::kMaxXInputs), "rs_rec_fwd_bf16_wide: the MMA-fused input projection takes 1 to %d input columns (got %d)",
               rs::kMaxXInputs, I);
    RS_REQUIRE(Wst && b_hn && out && h_n && B >= 0 && T >= 0, "rs_rec_fwd_bf16_wide: bad arguments");
    RS_REQUIRE((drop_bits != nullptr) == (out_drop != nullptr) && (!drop_bits || drop_scale), "rs_rec_fwd_bf16_wide: drop_bits, drop_scale and out_drop go together");
    if (T == 0) {
        RS_CUDA_OK(cudaMemsetAsync(h_n, 0, sizeof(float) * 2 * (size_t)B * HW, stream));
        return 0;
    }
    FwdWideParams p = {};
    p.x = x; p.I = I;
    p.P = static_cast<const uint8_t*>(P); p.p_block_bytes = 6LL * HW * 256;
    p.Wst = static_cast<const uint8_t*>(Wst); p.b_hn = b_hn;
    p.out = static_cast<uint8_t*>(out); p.out_block_bytes = 2LL * HW * 256;
    p.gates = static_cast<uint8_t*>(gates); p.h_n = h_n; p.lengths = lengths;
    p.drop_bits = static_cast<const uint8_t*>(drop_bits); p.drop_scale = drop_scale; p.out_drop = static_cast<uint8_t*>(out_drop);
    p.B = B; p.T = T; p.n_tiles = (B + 127) / 128;
    p.nstage = RING_STAGES;
    const int xc = x ? rs::x_chunks(I) : 1;         // layer 0: 16-byte input chunks per row (kXC of the kernel)
    const int smem = p.nstage * WSTAGE + (x ? H32_BYTES : 0) + (HW / 8 + 2 * ((xc + 1) / 2)) * CHUNK_S + HW * 4 + (int)sizeof(RingBars) + 64;
    const dim3 grid(2 * p.n_tiles, 2);
#define RS_LAUNCH_FWDW(FX_, VL_, DROP_, XC_)                                                                            \
    do {                                                                                                                \
        RS_CUDA_OK(cudaFuncSetAttribute(rec_fwd_wide_kernel<FX_, VL_, DROP_, XC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        rec_fwd_wide_kernel<FX_, VL_, DROP_, XC_><<<grid, NUM_THREADS, smem, stream>>>(p);                              \
    } while (0)
#define RS_LAUNCH_FWDW_V(FX_, XC_)                                                                                      \
    do {                                                                                                                \
        if (lengths) { if (drop_bits) RS_LAUNCH_FWDW(FX_, true, true, XC_); else RS_LAUNCH_FWDW(FX_, true, false, XC_); } \
        else { if (drop_bits) RS_LAUNCH_FWDW(FX_, false, true, XC_); else RS_LAUNCH_FWDW(FX_, false, false, XC_); }     \
    } while (0)
    if (!x) RS_LAUNCH_FWDW_V(false, 1);
    else if (xc == 1) RS_LAUNCH_FWDW_V(true, 1);
    else if (xc == 2) RS_LAUNCH_FWDW_V(true, 2);
    else if (xc == 4) RS_LAUNCH_FWDW_V(true, 4);
    else if (xc == 6) RS_LAUNCH_FWDW_V(true, 6);
    else RS_LAUNCH_FWDW_V(true, 8);
#undef RS_LAUNCH_FWDW_V
#undef RS_LAUNCH_FWDW
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

/* Backward through time for H = 256.  WTst: [2 dirs][2 ranks][8 stages][6 K steps][2 chunks][128 rows][8] bf16 = W_hh^T, rows =
 * hidden units [128 rank, 128 rank + 128), K = the 768 gate rows in r | z | n order; dG tile-major with 8H = 2048 columns. */
extern "C" int rs_rec_bwd_bf16_wide(const void* d_out, const float* d_h_n, const void* gates, const void* out, const void* WTst,
                                    void* dG, const int* lengths, const void* drop_bits, const float* drop_scale, int B, int T,
                                    void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0 || T == 0) return 0;
    RS_REQUIRE(gates && out && WTst && dG && B >= 0 && T >= 0, "rs_rec_bwd_bf16_wide: bad arguments");
    RS_REQUIRE(!drop_bits || drop_scale, "rs_rec_bwd_bf16_wide: drop_bits needs drop_scale");
    BwdWideParams p = {};
    p.d_out = static_cast<const uint8_t*>(d_out); p.dout_block_bytes = 2LL * HW * 256;
    p.d_h_n = d_h_n; p.gates = static_cast<const uint8_t*>(gates);
    p.out = static_cast<const uint8_t*>(out); p.out_block_bytes = 2LL * HW * 256;
    p.WTst = static_cast<const uint8_t*>(WTst);
    p.dG = static_cast<uint8_t*>(dG); p.dg_block_bytes = 8LL * HW * 256;
    p.lengths = lengths;
    p.drop_bits = static_cast<const uint8_t*>(drop_bits); p.drop_scale = drop_scale;
    p.B = B; p.T = T; p.n_tiles = (B + 127) / 128;
    p.nstage = RING_STAGES;
    const int smem = p.nstage * WSTAGE + A_BWD_BYTES + (int)sizeof(RingBars) + 64;
#define RS_LAUNCH_BWDW(VL_, DROP_)                                                                                      \
    do {                                                                                                                \
        RS_CUDA_OK(cudaFuncSetAttribute(rec_bwd_wide_kernel<VL_, DROP_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        rec_bwd_wide_kernel<VL_, DROP_><<<dim3(2 * p.n_tiles, 2), NUM_THREADS, smem, stream>>>(p);                      \
    } while (0)
    if (lengths) { if (drop_bits) RS_LAUNCH_BWDW(true, true); else RS_LAUNCH_BWDW(true, false); }
    else { if (drop_bits) RS_LAUNCH_BWDW(false, true); else RS_LAUNCH_BWDW(false, false); }
#undef RS_LAUNCH_BWDW
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
