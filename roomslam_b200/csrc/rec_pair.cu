// Persistent tensor-core GRU recurrence on a CTA PAIR (thread-block cluster of 2, tcgen05 cta_group::2), H = 128:
// forward and backward through time (SURVEY.md 8(a) rows a3, a4).  Same operands, layouts and results as rec_bf16.cu
// (one CTA per 128-trace tile); what changes is how a tile is spread over the chip:
//
//   * A pair of CTAs on one TPC owns a 128-trace tile of one direction; each CTA holds 64 of its traces.  One thread of
//     the even CTA issues M = 128 MMAs that span both SMs.  In that mode the accumulator of a CTA uses ALL 128 TMEM lanes
//     for its 64 rows: lane = row + 64 * (column half), so the epilogue of a tile runs on 2 x 128 lanes instead of 128 --
//     half the serial epilogue chain per step -- and each CTA needs only HALF of W_hh in shared memory (the tensor core
//     fetches the other half from the peer): the gate rows of hidden units [64 rank, 64 rank + 64).
//   * No activation crosses the pair in software: the two lane halves of a CTA produce all 128 hidden units of its 64
//     rows, written straight into its own A-operand tile.  Only mbarrier arrivals (epilogue warps -> the issuing CTA)
//     and the multicast tcgen05.commit cross the pair.
//   * With half the footprint per tile a pair carries NT = 2 tiles in flight (2 x 256 TMEM columns, 16 epilogue warps):
//     the MMA of one tile runs under the epilogue of the other, and every scheduler has 4 epilogue warps to pick from.
//     Small batches run NT = 1 on twice as many SMs (the latency-bound regime of strong scaling, BASELINE config 3).
//   * Inter-layer dropout (README.md:114) is applied here from a bit-packed mask: the forward kernel of a layer also writes
//     out (.) mask as the next layer's input, the backward kernel masks the incoming d_out.
#include <stdlib.h>

#include "common.cuh"
#include "rec_common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

using namespace rs;

constexpr int H = 128;
constexpr int ROWS = 64;                        // traces of a tile held by one CTA of the pair
constexpr int CHUNK_G = 2048;                   // global: one 16-byte chunk column over the 128 rows of a tile
constexpr int CHUNK_S = ROWS * 16;              // shared: the same over this CTA's 64 rows
constexpr int W_CHUNK = 192 * 16;               // shared: one chunk column of this CTA's W_hh rows (r | z | hn of 64 units)
constexpr int A_FWD_BYTES = 18 * CHUNK_S;       // 18 KB per tile in flight (16 hidden chunks + one K step of input chunks)
constexpr int H32_BYTES = (H / 4) * CHUNK_S;    // 32 KB per tile in flight (fp32 master copy of h)
constexpr int W_BWD_BYTES = 48 * CHUNK_S;       // 48 KB: W_hh^T rows of this CTA's 64 hidden units, K = 384 gate rows
constexpr int A_BWD_BYTES = 48 * CHUNK_S;       // 48 KB per tile in flight (dGh)
// Epilogue warps: always 16 per CTA.  NT = 2: 8 per tile in flight (4 TMEM lane quadrants x 2 groups of 32 hidden units);
// NT = 1: all 16 on the one tile (4 groups of 16 hidden units): the serial chain per step halves once more.
template <int NT> struct EpiShape {
    static constexpr int WG = (NT == 1) ? 4 : 2;        // warp groups per lane quadrant and tile
    static constexpr int SLOT_WARPS = 4 * WG;           // epilogue warps per tile in flight
    static constexpr int UPT = 64 / WG;                 // hidden units per thread
    static constexpr int NGRP = UPT / 8;                // 16-byte chunks (8 units) per thread and step
};
constexpr int NUM_THREADS = 64 + 512;
constexpr int X_CHUNKS_USED = x_col(kMaxXInputs - 1, 2) / 8 + 1;   // 7 of the 8 chunks of 4 input K steps (the last is padding)

struct FwdPairParams {
    const float* x; int I;
    const uint8_t* P; long long p_block_bytes;
    const uint8_t* Whh;                     // [2][16 or 18][384][8] bf16 (the image rs_rec_fwd_bf16 documents)
    const float* b_hn;
    uint8_t* out; long long out_block_bytes;
    uint8_t* gates;
    float* h_n;
    const int* lengths;
    const uint8_t* drop_bits;               // [tiles][T][128 rows][32] one bit per (trace, step, output column) or NULL
    const float* drop_scale;                // device scalar 1 / keep
    uint8_t* out_drop;                      // tile-major like out: out (.) mask, the next layer's input (with drop_bits)
    int B, T, n_tiles;
    int pf_dist;
    int split;                              // 1: Whh holds hi chunks then lo chunks (bf16 pairs per weight), K loop runs over both
    const uint8_t* X; long long x_block_bytes;   // fused projection (kMode 2): this layer's INPUT, tile-major, 2H columns
    const uint8_t* Wih;                          // [2][32][384][8] bf16: W_ih (r, z rows scaled by 1/2) as a resident B operand
};

// kMode 0: the input-side pre-activations come from HBM (P, written by the projection GEMM).
// kMode 1: layer 0, the K = I input projection rides on the recurrence MMA as (kXC + 1) / 2 more K = 16 steps of hi / lo
//   split operands (rec_common.cuh has the column map).  kXC = the 16-byte input chunks per row the epilogue writes each step:
//   1 (I <= 2: the one K step's second chunk stays zero; written after the epilogue from registers loaded before the wait
//   for the accumulator), else x_chunks(I), spread over the threads of a row and double-buffered in the A tile: the chunks
//   of step t+1 go into the buffer the MMA of step t does not read, BEFORE the wait, so no packed input is held in
//   registers across it (the 96-register cap left no room for that without spills).
// kMode 2 (NT = 1): the K = 256 input projection of a deeper layer is FUSED: W_ih's rows of this CTA's hidden units stay in
//   shared memory next to W_hh (96 + 54 KB; the master state is in registers in this mode), warp 1 bulk-copies the layer
//   input X_t of the CTA's 64 rows one step ahead (32 KB, one buffer), and the issuer runs X_{t+1} . W_ih^T (+ the bias via the
//   input chunk: a constant (1, 1) column against (b_hi, b_lo)) into the OTHER of two accumulator buffers while the epilogue
//   of step t is still reading its own: the projection is off the recurrence's critical path, P (6 H bf16 per trace and step:
//   6.3 GB written + read at the benchmark shape) and the projection GEMM launch disappear, and the epilogue has no global
//   loads left at all.
// kDrop: inter-layer dropout on this layer's output (drop_bits / out_drop given).  A template parameter, not a run-time
// flag: the mask test, the scaled copy and its bf16 pack are ~3.5 of the epilogue's 24 instructions per (row, hidden unit).
template <int NT, bool kVarLen, int kMode, bool kDrop, int kXC = 1>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) rec_fwd_pair_kernel(const FwdPairParams p) {
    constexpr bool kFusedX = (kMode != 0);                 // the n gate's input part arrives in its own accumulator columns
    constexpr bool kProj = (kMode == 2);
    static_assert(!kProj || NT == 1, "the fused projection needs the double-buffered accumulator of the one-tile mode");
    static_assert(kXC == 1 || (kMode == 1 && kXC % 2 == 0 && kXC <= 2 * x_steps(kMaxXInputs)), "input chunks per row");
    constexpr int kXS = (kXC + 1) / 2;                     // input K steps
    constexpr int kXB = kXC == 1 ? 1 : 2;                  // input column buffers
    constexpr int kXCW = kXC < X_CHUNKS_USED ? kXC : X_CHUNKS_USED;   // chunks that can hold a nonzero column
    constexpr int A_BYTES = (16 + 2 * kXS * kXB) * CHUNK_S;     // A tile per tile in flight: h_{t-1} | input columns
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* w_s = smem;                                   // [16 (x2 split) + 2 kXS chunks][192 rows][16 B]
    const int n_hid = 16 * (1 + p.split);                  // hidden-state chunks of W: hi parts, then (split) lo parts
    const int n_chunks = n_hid + (kFusedX ? 2 * kXS : 0);
    uint8_t* wih_s = w_s + n_chunks * W_CHUNK;             // [32 chunks][192 rows][16 B]   (kProj)
    uint8_t* a_s = wih_s + (kProj ? 32 * W_CHUNK : 0);     // [NT][16 + 2 kXS kXB chunks][64 rows][16 B]  h_{t-1} | input columns
    uint8_t* h32_s = a_s + NT * A_BYTES;                   // [NT][32 chunks of 4 floats][64 rows][16 B]   (NT = 2 only)
    uint8_t* x_s = h32_s + (NT == 1 ? 0 : NT * H32_BYTES); // [32 chunks][64 rows][16 B]  X_t of this CTA's rows (kProj)
    float* bhn_s = reinterpret_cast<float*>(x_s + (kProj ? 32 * CHUNK_S : 0));
    uint64_t* bars = reinterpret_cast<uint64_t*>(bhn_s + H);
    uint64_t* w_full = bars;
    uint64_t* h_ready = bars + 1;               // [NT], the even CTA's copies collect the arrivals of BOTH CTAs
    uint64_t* acc_full = bars + 1 + NT;         // [NT], one per CTA (multicast commit)
    uint64_t* x_full = bars + 1 + 2 * NT;       // kProj: this CTA's X tile landed (bulk-copy bytes)
    uint64_t* x_rdy = x_full + 1;               // kProj, even CTA: both CTAs' X tiles landed (2 arrivals)
    uint64_t* x_free = x_full + 2;              // kProj: the projection MMAs that read the X tile retired (multicast commit)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(x_full + 3);

    using ES = EpiShape<NT>;
    constexpr int EPI_WARPS = ES::SLOT_WARPS, UPT = ES::UPT, NGRP = ES::NGRP;
    // fp32 master copy of h (the blend must not re-round the state every step).  NT = 1: a thread owns 16 hidden units of
    // one row for the whole sequence, so the master state is 16 REGISTERS and the 32 KB of shared memory go back to L1;
    // NT = 2 (32 units per thread at the 96-register cap): shared memory.
    constexpr bool kRegState = (NT == 1);
    const uint32_t rank = cluster_ctarank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y;
    const int tile0 = (blockIdx.x >> 1) * NT;
    const int n_slots = min(NT, p.n_tiles - tile0);
    const int T = p.T;
    constexpr bool fused_x = kFusedX;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        for (int s = 0; s < NT; ++s) {
            mbar_init(&h_ready[s], 2 * EPI_WARPS);
            mbar_init(&acc_full[s], 1);
        }
        mbar_init(x_full, 1); mbar_init(x_rdy, 2); mbar_init(x_free, 1);
        fence_mbar_init();
    }
    if (warp == 0) {
        tmem_alloc_pair<(kProj ? 512 : 256 * NT)>(tmem_slot);
        if (lane == 0) {            // this CTA's half of W_hh: per chunk the r, z, n rows of its 64 hidden units
            mbar_expect_tx(w_full, (n_chunks + (kProj ? 32 : 0)) * W_CHUNK);
            const uint8_t* src = p.Whh + (long long)dir * n_chunks * (384 * 16);
            for (int c = 0; c < n_chunks; ++c)
                for (int g = 0; g < 3; ++g)
                    bulk_load(w_s + c * W_CHUNK + g * 1024, src + (long long)c * (384 * 16) + (g * 128 + rank * 64) * 16, 1024, w_full);
            if (kProj) {
                const uint8_t* srci = p.Wih + (long long)dir * 32 * (384 * 16);
                for (int c = 0; c < 32; ++c)
                    for (int g = 0; g < 3; ++g)
                        bulk_load(wih_s + c * W_CHUNK + g * 1024, srci + (long long)c * (384 * 16) + (g * 128 + rank * 64) * 16, 1024, w_full);
            }
        }
    }
    for (int i = threadIdx.x; i < H; i += blockDim.x) bhn_s[i] = p.b_hn[dir * H + i];
    for (int i = threadIdx.x; i < NT * (A_BYTES + (NT == 1 ? 0 : H32_BYTES)) / 16; i += blockDim.x)
        reinterpret_cast<uint4*>(a_s)[i] = make_uint4(0, 0, 0, 0);
    __syncthreads();
    if (kXC == 1) {
        if (fused_x && threadIdx.x < ROWS * NT) {       // input columns of the first step
            const int s = threadIdx.x / ROWS, rl = threadIdx.x % ROWS;
            const long long b = (long long)(tile0 + s) * 128 + rank * ROWS + rl;
            *reinterpret_cast<uint4*>(a_s + s * A_BYTES + 16 * CHUNK_S + rl * 16) =      // kProj: the constant (1, 1) bias column only
                pack_x((!kProj && s < n_slots && b < p.B) ? p.x + (b * T + (dir ? T - 1 : 0)) * p.I : nullptr, p.I);
        }
    } else {
        for (int i = threadIdx.x; i < NT * kXCW * ROWS; i += blockDim.x) {      // buffer 0: the input columns of the first step
            const int rl = i % ROWS, ch = (i / ROWS) % kXCW, s = i / (ROWS * kXCW);
            const long long b = (long long)(tile0 + s) * 128 + rank * ROWS + rl;
            *reinterpret_cast<uint4*>(a_s + s * A_BYTES + (16 + ch) * CHUNK_S + rl * 16) =
                pack_x_chunk((s < n_slots && b < p.B) ? p.x + (b * T + (dir ? T - 1 : 0)) * p.I : nullptr, p.I, ch);
        }
    }
    fence_proxy_async();
    if (warp == 0) mbar_wait(w_full, 0);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();             // both CTAs: barriers initialised, TMEM allocated, W and the first A tiles in place
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // pad rows t' = 0 and T + 1 of this CTA's rows: the time-shifted weight-gradient GEMM reads them as h = 0
    for (int i = threadIdx.x; i < n_slots * 2 * 16 * ROWS; i += blockDim.x) {
        const int rl = i % ROWS, c = (i / ROWS) % 16, pad = (i / (ROWS * 16)) % 2, s = i / (ROWS * 32);
        const long long off = ((long long)(tile0 + s) * (T + 2) + (pad ? T + 1 : 0)) * p.out_block_bytes
                              + (long long)(dir * 16 + c) * CHUNK_G + (rank * ROWS + rl) * 16;
        stg16(p.out + off, make_uint4(0, 0, 0, 0));
        if (kDrop) stg16(p.out_drop + off, make_uint4(0, 0, 0, 0));
    }

    if (warp == 0) {
        if (rank == 0) {
            // ===================== MMA issuer for the pair =====================
            constexpr uint32_t idesc256 = umma_idesc_bf16(128, 256, 0, 0);
            constexpr uint32_t idesc128 = umma_idesc_bf16(128, 128, 0, 0);
            const uint32_t w_addr = smem_u32(w_s);
            if (kProj) {
                const uint32_t a_addr = smem_u32(a_s), x_addr = smem_u32(x_s), wih_addr = smem_u32(wih_s);
                // X_t . W_ih^T + bias into accumulator buffer `buf`: r | z -> [0, 128), the n gate's input part -> [192, 256)
                auto issue_proj = [&](int step_x, uint32_t buf) {
                    mbar_wait(x_rdy, step_x & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        const uint32_t d = tmem_base + buf * 256;
#pragma unroll
                        for (int k = 0; k < 16; ++k) {
                            const uint64_t da = umma_desc_noswz(x_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                            const uint32_t wk = wih_addr + k * 2 * W_CHUNK;
                            tc_mma_bf16_pair(d, da, umma_desc_noswz(wk, W_CHUNK, 128), idesc256, k != 0);
                            tc_mma_bf16_pair(d + 192, da, umma_desc_noswz(wk + 128 * 16, W_CHUNK, 128), idesc128, k != 0);
                        }
                        const uint64_t db = umma_desc_noswz(a_addr + 16 * CHUNK_S, CHUNK_S, 128);       // the (1, 1) column
                        tc_mma_bf16_pair(d, db, umma_desc_noswz(w_addr + n_hid * W_CHUNK, W_CHUNK, 128), idesc256, 1u);
                        tc_mma_bf16_pair(d + 192, db, umma_desc_noswz(w_addr + n_hid * W_CHUNK + 128 * 16, W_CHUNK, 128), idesc128, 1u);
                        tc_commit_pair(x_free);             // the X tile may be refilled in both CTAs
                    }
                    __syncwarp();
                };
                issue_proj(0, 0);
                for (int step = 0; step < T; ++step) {
                    if (step > 0) {
                        mbar_wait_cluster(&h_ready[0], (step - 1) & 1);
                        tc_fence_after();
                    }
                    if (elect_one()) {                      // hidden part of step `step`, onto the projection already in the buffer
                        const uint32_t d = tmem_base + (step & 1) * 256;
#pragma unroll
                        for (int k = 0; k < 8; ++k) {
                            const uint64_t da = umma_desc_noswz(a_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                            const uint32_t wk = w_addr + k * 2 * W_CHUNK;
                            tc_mma_bf16_pair(d, da, umma_desc_noswz(wk, W_CHUNK, 128), idesc256, 1u);
                            tc_mma_bf16_pair(d + 128, da, umma_desc_noswz(wk + 128 * 16, W_CHUNK, 128), idesc128, k != 0);
                        }
                        tc_commit_pair(&acc_full[0]);
                    }
                    __syncwarp();
                    // the other buffer was last read by the epilogue of step - 1, which the h_ready wait above has seen finish
                    if (step + 1 < T) issue_proj(step + 1, (step + 1) & 1);
                }
            } else
            for (int step = 0; step < T; ++step) {
                for (int s = 0; s < n_slots; ++s) {
                    if (step > 0) {
                        mbar_wait_cluster(&h_ready[s], (step - 1) & 1);
                        tc_fence_after();
                    }
                    if (elect_one()) {
                        const uint32_t a_addr = smem_u32(a_s + s * A_BYTES);
                        const uint32_t d = tmem_base + s * 256;
                        for (int part = 0; part <= p.split; ++part) {     // split weights: h . W_hi^T + h . W_lo^T, same A tile
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                const uint64_t da = umma_desc_noswz(a_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                                const uint32_t wk = w_addr + (part * 16 + k * 2) * W_CHUNK;
                                const uint64_t db0 = umma_desc_noswz(wk, W_CHUNK, 128);
                                const uint64_t db1 = umma_desc_noswz(wk + 128 * 16, W_CHUNK, 128);
                                tc_mma_bf16_pair(d, da, db0, idesc256, (k | part) != 0);           // r | z  -> columns [0, 128) of each lane half
                                tc_mma_bf16_pair(d + 128, da, db1, idesc128, (k | part) != 0);     // W_hn h -> columns [128, 192)
                            }
                        }
                        if (fused_x) {      // layer 0: W_ih x + b as kXS more K = 16 steps of hi / lo split operands
#pragma unroll
                            for (int k = 0; k < kXS; ++k) {
                                const uint64_t da = umma_desc_noswz(a_addr + (16 + 2 * kXS * (kXB == 2 ? (step & 1) : 0) + 2 * k) * CHUNK_S, CHUNK_S, 128);
                                const uint64_t db0 = umma_desc_noswz(w_addr + (n_hid + 2 * k) * W_CHUNK, W_CHUNK, 128);
                                const uint64_t db1 = umma_desc_noswz(w_addr + (n_hid + 2 * k) * W_CHUNK + 128 * 16, W_CHUNK, 128);
                                tc_mma_bf16_pair(d, da, db0, idesc256, 1u);
                                tc_mma_bf16_pair(d + 192, da, db1, idesc128, k != 0);     // W_in x + b_in -> columns [192, 256)
                            }
                        }
                        tc_commit_pair(&acc_full[s]);
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1 && kProj) {
        // ===================== X tile producer (both CTAs): the layer input of the CTA's 64 rows, one step ahead ==========
        // 32 pieces of 1 KB (one per 16-byte chunk column), all issued by ONE elected thread: under elect.sync ptxas emits the
        // copies back to back with uniform-register addresses (~3 instructions each).  One copy per lane -- what a lane == 0
        // guard forces, because it costs an ELECT loop of ~13 instructions per copy -- took 0.9 us per time step (ncu: 27 % of
        // this warp's samples), and that sits on the path X_{t+1} landed -> projection MMAs -> hidden MMAs of the next step.
        const uint32_t rdy_remote = mapa_cluster(smem_u32(x_rdy), 0);
        if (elect_one()) {
            for (int step = 0; step < T; ++step) {
                const int t = dir ? (T - 1 - step) : step;
                if (step > 0) mbar_wait(x_free, (step - 1) & 1);
                mbar_expect_tx(x_full, 32 * CHUNK_S);
                const uint8_t* src = p.X + ((long long)tile0 * (T + 2) + t + 1) * p.x_block_bytes + rank * 1024;
#pragma unroll
                for (int c = 0; c < 32; ++c) bulk_load(x_s + c * CHUNK_S, src + (long long)c * CHUNK_G, 1024, x_full);
                if (step + 3 < T) {                        // L2 prefetch three steps ahead: the copies above then come from L2
                    const int t3 = dir ? (T - 1 - step - 3) : step + 3;
                    l2_prefetch(p.X + ((long long)tile0 * (T + 2) + t3 + 1) * p.x_block_bytes + (long long)(rank * 16) * CHUNK_G, 16 * CHUNK_G);
                }
                mbar_wait(x_full, step & 1);
                mbar_arrive_cluster(rdy_remote);
            }
        }
    } else if (warp == 1) {
        // ===================== L2 prefetcher: this CTA pulls half of the next projection block =====================
        if (lane == 0 && !kFusedX && p.pf_dist > 0) {
            for (int step = 0; step < T; ++step) {
                const int t = dir ? (T - 1 - step) : step;
                for (int s = 0; s < n_slots; ++s) {
                    const long long blk = (long long)(tile0 + s) * (T + 2) + t + 1;
                    l2_prefetch(p.P + blk * p.p_block_bytes + (long long)(dir * 48 + rank * 24) * CHUNK_G, 24 * CHUNK_G);
                }
                if (step >= p.pf_dist) mbar_wait(&acc_full[0], (step - p.pf_dist) & 1);
            }
        }
    } else if ((warp - 2) / EPI_WARPS < n_slots) {
        // ===================== epilogue: gates, blend, stores =====================
        const int s = (warp - 2) / EPI_WARPS;
        const int wg = ((warp - 2) % EPI_WARPS) >> 2;      // which UPT of this lane half's 64 hidden units
        const int q = warp & 3;                            // TMEM lane quadrant of this warp
        const int uh = q >> 1;                             // lane half = hidden-unit half
        const int rl = (q & 1) * 32 + lane;                // row within this CTA
        const int row = rank * ROWS + rl;                  // row within the 128-trace tile
        const int tile = tile0 + s;
        const long long b = (long long)tile * 128 + row;
        const bool live = b < p.B;
        const int ub = uh * 64 + wg * UPT;                 // first hidden unit of this thread
        const uint32_t taddr0 = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + s * 256 + wg * UPT;
        uint8_t* a_row = a_s + s * A_BYTES + rl * 16;
        uint8_t* h32_row = h32_s + s * H32_BYTES + rl * 16;
        const uint32_t hr_remote = mapa_cluster(smem_u32(&h_ready[s]), 0);
        const float* xrow = (kMode == 1 && p.x) ? p.x + b * T * p.I : nullptr;
        constexpr int X_NTH = 128 / UPT;                   // threads per row (both lane halves)
        const int x_ui = ub / UPT;                         // this thread's place among them
        const int len = (kVarLen && live) ? p.lengths[b] : T;
        const float dscale = kDrop ? __ldg(p.drop_scale) : 1.0f;
        float hreg[kRegState ? UPT : 1];
#pragma unroll
        for (int i = 0; i < (kRegState ? UPT : 1); ++i) hreg[i] = 0.0f;

        // running pointers of this thread's pieces: one signed stride per time step instead of 64-bit index arithmetic
        const int t_first = dir ? T - 1 : 0;
        const long long blk_first = (long long)tile * (T + 2) + t_first + 1;
        const long long o_first = blk_first * p.out_block_bytes + (long long)(dir * 16 + ub / 8) * CHUNK_G + row * 16;
        const long long o_step = dir ? -p.out_block_bytes : p.out_block_bytes;
        uint8_t* o_cur = p.out + o_first;
        const long long od_delta = kDrop ? p.out_drop - p.out : 0;     // warp-uniform: the masked copy sits at the same offsets
        const uint8_t* p_cur = kFusedX ? nullptr : p.P + blk_first * p.p_block_bytes + (long long)(dir * 48 + ub / 8) * CHUNK_G + row * 16;
        const long long p_step = dir ? -p.p_block_bytes : p.p_block_bytes;
        uint8_t* g_cur = p.gates ? p.gates + (((long long)tile * T + t_first) * 2 + dir) * (48LL * CHUNK_G) + (long long)(ub / 8) * CHUNK_G + row * 16 : nullptr;
        const long long g_step = (dir ? -2 : 2) * (48LL * CHUNK_G);
        const uint8_t* db_cur = kDrop ? p.drop_bits + (((long long)tile * T + t_first) * 128 + row) * 32 + dir * 16 + ((ub / 8) & ~3) : nullptr;
        const long long db_step = dir ? -128 * 32 : 128 * 32;

        // kMode 0: the projection block's pieces of this thread by per-thread loads, requested one chunk ahead of their use
        uint4 pv[3];
        auto load_p = [&](const uint8_t* base, int grp) {
#pragma unroll
            for (int g = 0; g < 3; ++g) pv[g] = ldg16(base + (long long)(g * 16 + grp) * CHUNK_G);
        };
        for (int step = 0; step < T; ++step) {
            const int t = dir ? (T - 1 - step) : step;
            const bool active = !kVarLen || t < len;
            const uint8_t* pblk = p_cur;
            uint8_t* const o_ptr = o_cur;
            uint8_t* const od_ptr = o_cur + od_delta;
            uint8_t* gblk = g_cur;
            uint32_t dbits = 0;
            if (kDrop) {            // the mask bytes of this thread's units sit in one aligned 32-bit word
                dbits = __ldg(reinterpret_cast<const uint32_t*>(db_cur)) >> (((ub / 8) & 3) * 8);
                db_cur += db_step;
            }
            o_cur += o_step;
            if (!kFusedX) p_cur += p_step;
            if (g_cur) g_cur += g_step;
            // input columns of step t+1, loaded and packed before the wait.  I <= 2: one chunk, by the row's thread of units
            // 0.., stored after the epilogue; else chunk ch by the row's thread ch % X_NTH (a warp-uniform test: every chunk
            // index stays a compile-time constant, and so does its column map), stored at once into the other buffer
            uint4 xnext = make_uint4(0, 0, 0, 0);
            const bool write_x = kMode == 1 && ub == 0 && step + 1 < T;
            const uint32_t taddr = taddr0 + (kProj ? (step & 1) * 256 : 0);
            if (kXC == 1) {
                if (write_x) xnext = pack_x(live ? xrow + (long long)(dir ? t - 1 : t + 1) * p.I : nullptr, p.I);
            } else if (step + 1 < T) {
                const float* xp = live ? xrow + (long long)(dir ? t - 1 : t + 1) * p.I : nullptr;
                uint8_t* xbuf = a_row + (16 + 2 * kXS * ((step + 1) & 1)) * CHUNK_S;
#define RS_PUT_X(U)                                                                                                     \
    case U:                                                                                                             \
        if (U < kXCW) *reinterpret_cast<uint4*>(xbuf + (U) * CHUNK_S) = pack_x_chunk(xp, p.I, U);                      \
        if (U + X_NTH < kXCW) *reinterpret_cast<uint4*>(xbuf + (U + X_NTH) * CHUNK_S) = pack_x_chunk(xp, p.I, U + X_NTH); \
        break
                switch (x_ui) { RS_PUT_X(0); RS_PUT_X(1); RS_PUT_X(2); RS_PUT_X(3); RS_PUT_X(4); RS_PUT_X(5); RS_PUT_X(6); RS_PUT_X(7); }
#undef RS_PUT_X
            }
            if (!kFusedX) load_p(pblk, 0);
            mbar_wait(&acc_full[s], step & 1);
            tc_fence_after();
            // first chunk whose global stores wait for the arrival: the last one (deferring both chunks of the one-tile mode
            // costs 16 more live registers and is 14 % slower)
            constexpr int kDefer0 = NGRP - 1;
            constexpr int ND = NGRP - kDefer0;
            uint4 last_o[ND], last_d[ND], last_r[ND], last_z[ND], last_n[ND];
#pragma unroll
            for (int grp = 0; grp < NGRP; ++grp) {
                const int u0 = ub + grp * 8;
                uint32_t ar[8], az[8], an[8], ax[8];
                tmem_ld_32x32b_x8(taddr + grp * 8, ar);
                tmem_ld_32x32b_x8(taddr + 64 + grp * 8, az);
                tmem_ld_32x32b_x8(taddr + 128 + grp * 8, an);
                if (kFusedX) tmem_ld_32x32b_x8(taddr + 192 + grp * 8, ax);
                uint4 pc[3];
                if (!kFusedX) {
                    pc[0] = pv[0]; pc[1] = pv[1]; pc[2] = pv[2];
                    if (grp < NGRP - 1) load_p(pblk, grp + 1);
                }
                tmem_ld_wait();
                uint32_t wo[4], wd[4], wr[4], wz[4], wn[4];             // packed outputs: h, h (.) mask, r, z, n
#pragma unroll
                for (int jp = 0; jp < 4; ++jp) {                        // two hidden units at a time keeps the live set small
                    float hv2[2], rv2[2], zv2[2], nv2[2], od2[2];
                    const float2 ho2 = kRegState ? make_float2(hreg[grp * 8 + 2 * jp], hreg[grp * 8 + 2 * jp + 1])
                                                 : *reinterpret_cast<const float2*>(h32_row + (u0 / 4 + jp / 2) * CHUNK_S + (jp & 1) * 8);
                    const float2 bh2 = *reinterpret_cast<const float2*>(bhn_s + u0 + 2 * jp);
                    float2 pr2 = make_float2(0.f, 0.f), pz2 = pr2, pn2 = pr2;
                    if (!kFusedX) {
                        const uint32_t* w0 = reinterpret_cast<const uint32_t*>(&pc[0]);
                        const uint32_t* w1 = reinterpret_cast<const uint32_t*>(&pc[1]);
                        const uint32_t* w2 = reinterpret_cast<const uint32_t*>(&pc[2]);
                        pr2 = bf2_to_f2(w0[jp]); pz2 = bf2_to_f2(w1[jp]); pn2 = bf2_to_f2(w2[jp]);
                    } else {            // layer 0: the tensor core already added W_ih x + b to r and z
                        pn2 = make_float2(__uint_as_float(ax[2 * jp]), __uint_as_float(ax[2 * jp + 1]));
                    }
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int j = 2 * jp + e;
                        const float ho = e ? ho2.y : ho2.x;
                        // the 1/2 of sigma(a) = 1/2 tanh(a/2) + 1/2 is folded into the r and z rows of the weights and biases
                        // (fused input columns: the accumulator already holds the whole pre-activation -- no `+ 0` left behind)
                        const float ar_ = kFusedX ? __uint_as_float(ar[j]) : __uint_as_float(ar[j]) + (e ? pr2.y : pr2.x);
                        const float az_ = kFusedX ? __uint_as_float(az[j]) : __uint_as_float(az[j]) + (e ? pz2.y : pz2.x);
                        const float r = fmaf(0.5f, tanh_fast(ar_), 0.5f);
                        const float z = active ? fmaf(0.5f, tanh_fast(az_), 0.5f) : 1.0f;
                        const float hn = __uint_as_float(an[j]) + (e ? bh2.y : bh2.x);
                        const float n = tanh_fast(fmaf(r, hn, e ? pn2.y : pn2.x));
                        const float h = active ? fmaf(z, ho - n, n) : ho;
                        hv2[e] = h; rv2[e] = r; zv2[e] = z; nv2[e] = n;
                        if (kDrop) od2[e] = (active && ((dbits >> (grp * 8 + j)) & 1u)) ? h * dscale : 0.0f;
                    }
                    if (kRegState) { hreg[grp * 8 + 2 * jp] = hv2[0]; hreg[grp * 8 + 2 * jp + 1] = hv2[1]; }
                    else *reinterpret_cast<float2*>(h32_row + (u0 / 4 + jp / 2) * CHUNK_S + (jp & 1) * 8) = make_float2(hv2[0], hv2[1]);
                    wo[jp] = f2_to_bf2(hv2[0], hv2[1]);
                    if (kDrop) wd[jp] = f2_to_bf2(od2[0], od2[1]);
                    wr[jp] = f2_to_h2(rv2[0], rv2[1]); wz[jp] = f2_to_h2(zv2[0], zv2[1]);
                    wn[jp] = f2_to_h2(nv2[0], nv2[1]);
                }
                const uint4 o0 = make_uint4(wo[0], wo[1], wo[2], wo[3]);
                *reinterpret_cast<uint4*>(a_row + (u0 / 8) * CHUNK_S) = o0;      // next step's A operand, in place
                const uint4 so = active ? o0 : make_uint4(0, 0, 0, 0), sd = make_uint4(wd[0], wd[1], wd[2], wd[3]);
                const uint4 sr = make_uint4(wr[0], wr[1], wr[2], wr[3]), sz = make_uint4(wz[0], wz[1], wz[2], wz[3]);
                const uint4 sn = make_uint4(wn[0], wn[1], wn[2], wn[3]);
                if (grp < kDefer0) {
                    stg16(o_ptr + (long long)grp * CHUNK_G, so);
                    if (kDrop) stg16(od_ptr + (long long)grp * CHUNK_G, sd);
                    if (gblk) {
                        stg16(gblk + (long long)(0 * 16 + grp) * CHUNK_G, sr);
                        stg16(gblk + (long long)(1 * 16 + grp) * CHUNK_G, sz);
                        stg16(gblk + (long long)(2 * 16 + grp) * CHUNK_G, sn);
                    }   // W_hn h + b_hn is not saved: the backward kernel recomputes it on the tensor core
                } else {                // the last chunk's global stores wait until after the arrival (below)
                    last_o[grp - kDefer0] = so; last_d[grp - kDefer0] = sd; last_r[grp - kDefer0] = sr; last_z[grp - kDefer0] = sz;
                    last_n[grp - kDefer0] = sn;
                }
            }
            if (kXC == 1 && write_x) *reinterpret_cast<uint4*>(a_row + 16 * CHUNK_S) = xnext;
            fence_proxy_async();        // h_t written with ordinary stores -> visible to the tensor core of this SM
            tc_fence_before();          // TMEM reads done before the next MMA overwrites the accumulator
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(hr_remote);
            // The MEMBAR inside fence.proxy.async waits for every global store of the thread still in flight (ncu: ~0.2 us of
            // a 2.3 us step).  The stores of the earlier chunks are long acknowledged by then; the last chunk's are issued only
            // now, under the wait for the next MMA.
#pragma unroll
            for (int g = kDefer0; g < NGRP; ++g) {
                stg16(o_ptr + (long long)g * CHUNK_G, last_o[g - kDefer0]);
                if (kDrop) stg16(od_ptr + (long long)g * CHUNK_G, last_d[g - kDefer0]);
                if (gblk) {
                    stg16(gblk + (long long)(0 * 16 + g) * CHUNK_G, last_r[g - kDefer0]);
                    stg16(gblk + (long long)(1 * 16 + g) * CHUNK_G, last_z[g - kDefer0]);
                    stg16(gblk + (long long)(2 * 16 + g) * CHUNK_G, last_n[g - kDefer0]);
                }
            }
        }
        if (live) {                     // h_n: the fp32 master state after the last step (kept out of the step loop)
            float* hn_row = p.h_n + ((long long)dir * p.B + b) * H + ub;
#pragma unroll
            for (int i = 0; i < UPT; i += 2)
                *reinterpret_cast<float2*>(hn_row + i) =
                    kRegState ? make_float2(hreg[i], hreg[i + 1])
                              : *reinterpret_cast<const float2*>(h32_row + ((ub + i) / 4) * CHUNK_S + ((i >> 1) & 1) * 8);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the peer's tensor core reads this CTA's W half until its last MMA retired
    if (warp == 0) tmem_dealloc_pair<(kProj ? 512 : 256 * NT)>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------------
// Backward through time: one 128-trace tile per CTA pair (16 epilogue warps per CTA, 16 hidden units per thread).
//   dh_{t-1} = z (.) dh_t + dGh_t . W_hh   one MMA chain (K = 384) accumulating onto the carry that lives in TMEM.
// W_hn h_{t-1} + b_hn is NOT saved by the forward pass (it would be a fourth 16-bit gate block: 2.1 GB written and 2.1 GB
// read per layer at the benchmark shape): with W_hh halved per CTA there is room for the h_{t-1} tile and the W_hn rows, so
// the kernel recomputes it on the tensor core -- warp 1 bulk-copies the h_{t-1} block of the tile two steps ahead (two
// stages; it is the `out` block the epilogue used to read with per-thread loads), the even CTA's warp 1 issues
// hn = h_{t-1} . W_hn^T (N = 128, K = 128) into one of two 64-column TMEM buffers as soon as both CTAs' tiles landed, and
// the epilogue reads hn from TMEM and h_{t-1} from shared memory.  Same bf16 operands and K order as the forward MMA: the
// recomputed value is the forward's fp32 accumulator, not its fp16 rounding.
//
// kRecompute (layer 0, unsplit weights, I <= 2): r, z and n are not saved by the forward pass either (6.3 GB written and
// 6.3 GB read per step at the benchmark shape).  The even CTA's warp 1 replays the forward's whole layer-0 MMA -- the same
// A bytes (the h_{t-1} tile, which is what the forward's A tile held, plus the packed input chunk of step t, bulk-copied
// next to it), the same B image (the r | z | n rows of whh_img with its input chunk), the same instruction shapes and the
// same K order -- into one of two 256-column TMEM buffers (r | z | hn | the input part of n), and the epilogue forms r, z
// and n exactly as the forward epilogue does: the gate gradients are bit-identical to those from saved gates.  TMEM holds
// two such buffers and nothing else (512 columns), so the z (.) dh carry lives in the r columns of the buffer of the step
// that wrote it: the epilogue of step s reads r there, writes the carry over it, the dh MMA of step s + 1 accumulates onto
// it, the epilogue of step s + 1 reads dh from it first and then hands the buffer to the recompute of step s + 2, which runs
// under the rest of that epilogue.
struct BwdPairParams {
    const uint8_t* d_out; long long dout_block_bytes;
    const float* d_h_n;
    const uint8_t* gates;                                // [tiles][T][2][48 chunks: r | z | n][128][8] fp16 (NULL: kRecompute)
    const uint8_t* xpack;                                // kRecompute: [tiles][T][128][8] bf16, pack_x of each trace row and step
    const uint8_t* out; long long out_block_bytes;
    const uint8_t* WhhT;                                 // [2][48 (x2 split)][128][8] bf16
    const uint8_t* Whh;                                  // forward image [2][16 (x2 split) (+2)][384][8]: its n rows are W_hn
    int whh_chunks;                                      // chunks per direction of the forward image
    const float* b_hn;                                   // [2][H]
    uint8_t* dG; long long dg_block_bytes;
    const int* lengths;
    const uint8_t* drop_bits;                            // mask of THIS layer's output (applied to d_out) or NULL
    const float* drop_scale;
    int B, T, n_tiles;
    int split;                                           // 1: weight images hold hi chunks then lo chunks
    int pf_dist;                                         // L2 prefetch distance of the gate / d_out blocks in steps (0 = off)
};

constexpr int HP_BYTES = 16 * CHUNK_S;                   // 16 KB: the h_{t-1} tile of this CTA's 64 rows (K-major A operand)
constexpr int WF_BYTES = 18 * W_CHUNK;                   // kRecompute: 54 KB, r | z | n rows of whh_img (16 hidden + 2 input chunks)
template <bool kVarLen, bool kDrop, bool kRecompute>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1) rec_bwd_pair_kernel(const BwdPairParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr int STAGE = kRecompute ? HP_BYTES + 2 * CHUNK_S : HP_BYTES;   // + the input chunk of step t and a zero chunk
    constexpr uint32_t TMEM_COLS = kRecompute ? 512 : 256;
    const int w_chunks = 48 * (1 + p.split), n_hid = 16 * (1 + p.split);
    uint8_t* w_s = smem;                                   // [48 chunks][64 rows = hidden units of this CTA][16 B]   W_hh^T
    uint8_t* a_s = w_s + w_chunks * CHUNK_S;               // [48 chunks][64 rows][16 B]  dGh_t
    uint8_t* wn_s = a_s + A_BWD_BYTES;                     // [16 chunks][64 rows = hidden units of this CTA][16 B]   W_hn
                                                           // kRecompute: [18 chunks][192 rows][16 B] as the forward's w_s
    uint8_t* hp_s = wn_s + (kRecompute ? WF_BYTES : n_hid * CHUNK_S);   // [2 stages][16 (+2) chunks][64 rows][16 B]  h_{t-1} (| x_t)
    float* bhn_s = reinterpret_cast<float*>(hp_s + 2 * STAGE);
    uint64_t* bars = reinterpret_cast<uint64_t*>(bhn_s + H);
    uint64_t* w_full = bars;
    uint64_t* a_ready = bars + 1;               // even CTA: dGh_t of both CTAs written (32 warps)
    uint64_t* acc_full = bars + 2;              // both: the dh MMA chain retired (multicast commit)
    uint64_t* hp_full = bars + 3;               // [2] this CTA's h_{t-1} tile landed (bulk-copy bytes)
    uint64_t* hp_rdy = bars + 5;                // [2] even CTA: both CTAs' tiles landed (2 arrivals)
    uint64_t* hn_full = bars + 7;               // [2] both: the hn MMA (kRecompute: the gate MMAs) retired (multicast commit)
    uint64_t* hp_free = bars + 9;               // [2] this CTA's 16 epilogue warps are done with the stage (tile and TMEM buffer)
    uint64_t* tm_free = bars + 11;              // [2] kRecompute, even CTA: both CTAs' epilogues have read dh out of the buffer
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);

    constexpr int UPT = 16, NGRP = 2;
    const uint32_t rank = cluster_ctarank();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int dir = blockIdx.y;
    const int tile = blockIdx.x >> 1;
    const int T = p.T;

    if (threadIdx.x == 0) {
        mbar_init(w_full, 1);
        mbar_init(a_ready, 2 * 16);
        mbar_init(acc_full, 1);
        for (int i = 0; i < 2; ++i) {
            mbar_init(&hp_full[i], 1); mbar_init(&hp_rdy[i], 2); mbar_init(&hn_full[i], 1); mbar_init(&hp_free[i], 16);
            mbar_init(&tm_free[i], 2 * 16);
        }
        fence_mbar_init();
    }
    if (warp == 0) {
        // dh accumulator [0, 64), hn buffers [64, 128) and [128, 192); kRecompute: two gate buffers [0, 256), [256, 512)
        tmem_alloc_pair<TMEM_COLS>(tmem_slot);
        if (lane == 0) {
            mbar_expect_tx(w_full, w_chunks * CHUNK_S + (kRecompute ? WF_BYTES : n_hid * CHUNK_S));
            const uint8_t* src = p.WhhT + (long long)dir * w_chunks * CHUNK_G + rank * 1024;
            for (int c = 0; c < w_chunks; ++c) bulk_load(w_s + c * CHUNK_S, src + (long long)c * CHUNK_G, 1024, w_full);
            if (kRecompute) {           // the forward kernel's copy of its W half (rec_fwd_pair_kernel, layer 0, kXC = 1)
                const uint8_t* srcf = p.Whh + (long long)dir * p.whh_chunks * (384 * 16);
                for (int c = 0; c < 18; ++c)
                    for (int g = 0; g < 3; ++g)
                        bulk_load(wn_s + c * W_CHUNK + g * 1024, srcf + (long long)c * (384 * 16) + (g * 128 + rank * 64) * 16, 1024, w_full);
            } else {
                const uint8_t* srcn = p.Whh + (long long)dir * p.whh_chunks * (384 * 16) + (256 + rank * 64) * 16;
                for (int c = 0; c < n_hid; ++c) bulk_load(wn_s + c * CHUNK_S, srcn + (long long)c * (384 * 16), 1024, w_full);
            }
        }
        mbar_wait(w_full, 0);
    }
    for (int i = threadIdx.x; i < H; i += blockDim.x) bhn_s[i] = p.b_hn[dir * H + i];
    if (kRecompute) {                   // the second input chunk of the one input K step stays zero, as in the forward's A tile
        for (int i = threadIdx.x; i < 2 * CHUNK_S / 16; i += blockDim.x)
            reinterpret_cast<uint4*>(hp_s + (i / (CHUNK_S / 16)) * STAGE + 17 * CHUNK_S)[i % (CHUNK_S / 16)] = make_uint4(0, 0, 0, 0);
        fence_proxy_async();
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // pad rows of dG (the weight / data gradient GEMMs run over all T + 2 rows of a tile)
    for (int i = threadIdx.x; i < 2 * 64 * ROWS; i += blockDim.x) {
        const int rl = i % ROWS, c = (i / ROWS) % 64, pad = i / (ROWS * 64);
        const long long off = ((long long)tile * (T + 2) + (pad ? T + 1 : 0)) * p.dg_block_bytes
                              + (long long)(dir * 64 + c) * CHUNK_G + (rank * ROWS + rl) * 16;
        stg16(p.dG + off, make_uint4(0, 0, 0, 0));
    }

    if (warp == 0) {
        if (rank == 0) {
            // ===================== dh matvec issuer =====================
            constexpr uint32_t idesc = umma_idesc_bf16(128, 128, 0, 0);
            const uint32_t w_addr = smem_u32(w_s), a_addr = smem_u32(a_s);
            for (int sidx = 0; sidx < T - 1; ++sidx) {     // the result of the last reverse step is unused
                mbar_wait_cluster(a_ready, sidx & 1);
                tc_fence_after();
                const uint32_t d = tmem_base + (kRecompute ? (sidx & 1) * 256 : 0);    // kRecompute: the carry of step sidx
                if (elect_one()) {
                    for (int part = 0; part <= p.split; ++part) {
#pragma unroll
                        for (int k = 0; k < 24; ++k) {
                            const uint64_t da = umma_desc_noswz(a_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                            const uint64_t db = umma_desc_noswz(w_addr + (part * 48 + k * 2) * CHUNK_S, CHUNK_S, 128);
                            tc_mma_bf16_pair(d, da, db, idesc, 1u);           // accumulates onto the z (.) dh carry in TMEM
                        }
                    }
                    tc_commit_pair(acc_full);
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===================== h_{t-1} tile producer (both CTAs) + hn issuer (even CTA) =====================
        {
            constexpr uint32_t idesc = umma_idesc_bf16(128, 128, 0, 0);
            const uint32_t wn_addr = smem_u32(wn_s);
            const uint32_t rdy_remote[2] = {mapa_cluster(smem_u32(&hp_rdy[0]), 0), mapa_cluster(smem_u32(&hp_rdy[1]), 0)};
            for (int sidx = 0; sidx < T; ++sidx) {
                const int st = sidx & 1;
                const uint32_t ph = (sidx >> 1) & 1;
                const int t = dir ? sidx : (T - 1 - sidx);
                const int t_prev = dir ? t + 1 : t - 1;
                if (elect_one()) {
                    if (sidx >= 2) mbar_wait(&hp_free[st], ph ^ 1);    // the epilogue of step sidx - 2 is done with this stage
                    mbar_expect_tx(&hp_full[st], HP_BYTES + (kRecompute ? CHUNK_S : 0));
                    const uint8_t* src = p.out + ((long long)tile * (T + 2) + t_prev + 1) * p.out_block_bytes + (long long)(dir * 16) * CHUNK_G + rank * 1024;
#pragma unroll
                    for (int c = 0; c < 16; ++c)                       // 16 pieces of 1 KB, back to back (see the X tile producer)
                        bulk_load(hp_s + st * STAGE + c * CHUNK_S, src + (long long)c * CHUNK_G, 1024, &hp_full[st]);
                    if (kRecompute)                                    // the input chunk of step t: the A tile's chunk 16 in the forward
                        bulk_load(hp_s + st * STAGE + 16 * CHUNK_S, p.xpack + ((long long)tile * T + t) * CHUNK_G + rank * 1024, 1024, &hp_full[st]);
                    if (p.pf_dist > 0 && sidx + p.pf_dist < T) {       // optional L2 prefetch of a later step's gate / d_out blocks
                        const int t2 = dir ? sidx + p.pf_dist : (T - 1 - sidx - p.pf_dist);
                        if (!kRecompute)
                            l2_prefetch(p.gates + (((long long)tile * T + t2) * 2 + dir) * (48LL * CHUNK_G) + (long long)(rank * 24) * CHUNK_G, 24 * CHUNK_G);
                        if (p.d_out) l2_prefetch(p.d_out + ((long long)tile * (T + 2) + t2 + 1) * p.dout_block_bytes + (long long)(dir * 16 + rank * 8) * CHUNK_G, 8 * CHUNK_G);
                    }
                    mbar_wait(&hp_full[st], ph);
                    mbar_arrive_cluster(rdy_remote[st]);
                    if (rank == 0) {
                        mbar_wait(&hp_rdy[st], ph);
                        // kRecompute: buffer st last held the carry of step sidx - 2, read as dh by the epilogue of step sidx - 1
                        if (kRecompute && sidx >= 1) mbar_wait(&tm_free[st], ((sidx - 1) >> 1) & 1);
                        tc_fence_after();
                        const uint32_t hp_addr = smem_u32(hp_s + st * STAGE);
                        if (kRecompute) {       // rec_fwd_pair_kernel's layer-0 MMAs (split = 0, kXC = 1), operand for operand
                            constexpr uint32_t idesc256 = umma_idesc_bf16(128, 256, 0, 0);
                            const uint32_t d = tmem_base + st * 256;
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                const uint64_t da = umma_desc_noswz(hp_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                                const uint32_t wk = wn_addr + k * 2 * W_CHUNK;
                                tc_mma_bf16_pair(d, da, umma_desc_noswz(wk, W_CHUNK, 128), idesc256, k != 0);             // r | z
                                tc_mma_bf16_pair(d + 128, da, umma_desc_noswz(wk + 128 * 16, W_CHUNK, 128), idesc, k != 0);   // W_hn h
                            }
                            const uint64_t da = umma_desc_noswz(hp_addr + 16 * CHUNK_S, CHUNK_S, 128);
                            const uint32_t wx = wn_addr + 16 * W_CHUNK;
                            tc_mma_bf16_pair(d, da, umma_desc_noswz(wx, W_CHUNK, 128), idesc256, 1u);
                            tc_mma_bf16_pair(d + 192, da, umma_desc_noswz(wx + 128 * 16, W_CHUNK, 128), idesc, 0u);     // W_in x + b_in
                        } else {
                            for (int part = 0; part <= p.split; ++part) {
#pragma unroll
                                for (int k = 0; k < 8; ++k) {
                                    const uint64_t da = umma_desc_noswz(hp_addr + k * 2 * CHUNK_S, CHUNK_S, 128);
                                    const uint64_t db = umma_desc_noswz(wn_addr + (part * 16 + k * 2) * CHUNK_S, CHUNK_S, 128);
                                    tc_mma_bf16_pair(tmem_base + 64 + st * 64, da, db, idesc, (k | part) != 0);
                                }
                            }
                        }
                        tc_commit_pair(&hn_full[st]);
                    }
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== epilogue =====================
        const int wg = (warp - 2) >> 2;                    // which 16 of this lane half's 64 hidden units
        const int q = warp & 3;
        const int uh = q >> 1;
        const int rl = (q & 1) * 32 + lane;
        const int row = rank * ROWS + rl;
        const long long b = (long long)tile * 128 + row;
        const bool live = b < p.B;
        const int ub = uh * 64 + wg * UPT;
        const int cb = ub / 8;                             // first of this thread's 2 chunks within the H columns
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + wg * UPT;
        uint8_t* a_row = a_s + rl * 16;
        const uint32_t ar_remote = mapa_cluster(smem_u32(a_ready), 0);
        const int len = (kVarLen && live) ? p.lengths[b] : T;
        const float dscale = kDrop ? __ldg(p.drop_scale) : 1.0f;
        // the carry z (.) dh lives in the TMEM accumulator (kRecompute: the r columns of buffer 1); it starts as d_h_n
#pragma unroll
        for (int sc = 0; sc < NGRP; ++sc) {
            uint32_t init[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) init[j] = 0u;
            if (p.d_h_n && live) {
                const float* src = p.d_h_n + ((long long)dir * p.B + b) * H + ub + sc * 8;
                const float4 v0 = __ldg(reinterpret_cast<const float4*>(src));
                const float4 v1 = __ldg(reinterpret_cast<const float4*>(src + 4));
                init[0] = __float_as_uint(v0.x); init[1] = __float_as_uint(v0.y); init[2] = __float_as_uint(v0.z); init[3] = __float_as_uint(v0.w);
                init[4] = __float_as_uint(v1.x); init[5] = __float_as_uint(v1.y); init[6] = __float_as_uint(v1.z); init[7] = __float_as_uint(v1.w);
            }
            tmem_st_32x32b_x8(taddr + (kRecompute ? 256 : 0) + sc * 8, init);
        }
        tmem_st_wait();

        // r, z, n (fp16; not with kRecompute) and d_out (bf16) of the thread's two chunks (8 units each): per-thread global
        // loads, requested one chunk ahead of their use
        uint4 raw[4];
        uint32_t dbits_next = 0;
        // running pointers of this thread's pieces (one signed stride per time step instead of 64-bit index arithmetic)
        const int t_first = dir ? 0 : T - 1;
        const long long g_step = (dir ? 2 : -2) * (48LL * CHUNK_G);
        const long long do_step = dir ? p.dout_block_bytes : -p.dout_block_bytes;
        const long long dg_step = dir ? p.dg_block_bytes : -p.dg_block_bytes;
        const uint8_t* g_ptr = kRecompute ? nullptr : p.gates + (((long long)tile * T + t_first) * 2 + dir) * (48LL * CHUNK_G) + (long long)cb * CHUNK_G + row * 16;
        const uint8_t* do_ptr = p.d_out ? p.d_out + ((long long)tile * (T + 2) + t_first + 1) * p.dout_block_bytes
                                                                   + (long long)(dir * 16 + cb) * CHUNK_G + row * 16 : nullptr;
        const uint8_t* db_next = kDrop ? p.drop_bits + (((long long)tile * T + t_first) * 128 + row) * 32 + dir * 16 + (cb & ~3) : nullptr;
        const long long db_step = dir ? 128 * 32 : -128 * 32;
        uint8_t* dg_cur = p.dG + ((long long)tile * (T + 2) + t_first + 1) * p.dg_block_bytes + (long long)(dir * 64 + cb) * CHUNK_G + row * 16;
        auto load_raw = [&](int sc) {                      // chunk sc of the step g_ptr / do_ptr stand at
#pragma unroll
            for (int g = 0; g < 3; ++g) raw[g] = kRecompute ? make_uint4(0, 0, 0, 0) : ldg16(g_ptr + (long long)(g * 16 + sc) * CHUNK_G);
            raw[3] = do_ptr ? ldg16(do_ptr + (long long)sc * CHUNK_G) : make_uint4(0, 0, 0, 0);
        };
        load_raw(0);
        if (kDrop) dbits_next = __ldg(reinterpret_cast<const uint32_t*>(db_next)) >> ((cb & 3) * 8);
        for (int sidx = 0; sidx < T; ++sidx) {             // sidx-th reverse step = forward position T-1-sidx (dir 0)
            const int t = dir ? sidx : (T - 1 - sidx);
            const int st = sidx & 1;
            const bool active = !kVarLen || t < len;
            uint8_t* dgblk = dg_cur;
            dg_cur += dg_step;
            const uint8_t* hp_row = hp_s + st * STAGE + rl * 16;
            const uint32_t dbits = dbits_next;
            if (kDrop && sidx + 1 < T) {                   // next step's mask word: requested a whole step ahead
                db_next += db_step;
                dbits_next = __ldg(reinterpret_cast<const uint32_t*>(db_next)) >> ((cb & 3) * 8);
            }
            mbar_wait(&hn_full[st], (sidx >> 1) & 1);      // W_hn h_{t-1} of this step is in TMEM, the h_{t-1} tile in shared memory
            if (sidx > 0) mbar_wait(acc_full, (sidx - 1) & 1);
            tc_fence_after();
            uint32_t dh16[16];
            if (kRecompute) {                              // dh out of the other buffer first, then that buffer is free
                tmem_ld_32x32b_x16(taddr + (st ^ 1) * 256, dh16);
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive_cluster(mapa_cluster(smem_u32(&tm_free[st ^ 1]), 0));
            }
#pragma unroll
            for (int sc = 0; sc < NGRP; ++sc) {
                uint32_t acc[8], ahn[8], ar[8], az[8], ax[8];
                if (kRecompute) {
                    const uint32_t tb = taddr + st * 256 + sc * 8;
                    tmem_ld_32x32b_x8(tb, ar);
                    tmem_ld_32x32b_x8(tb + 128, ahn);
                    tmem_ld_32x32b_x8(tb + 192, ax);
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[j] = dh16[sc * 8 + j];
                } else {
                    tmem_ld_32x32b_x8(taddr + sc * 8, acc);
                    tmem_ld_32x32b_x8(taddr + 64 + st * 64 + sc * 8, ahn);
                }
                uint4 cur[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) cur[i] = raw[i];
                if (sc < NGRP - 1) load_raw(sc + 1);
                float r[8], z[8], n[8], hp[8], dout[8], bh[8];
                if (!kRecompute) { unpack8h(cur[0], r); unpack8h(cur[1], z); unpack8h(cur[2], n); }
                unpack8(cur[3], dout);
                auto load_hp_bh = [&]() {
                    unpack8(*reinterpret_cast<const uint4*>(hp_row + (cb + sc) * CHUNK_S), hp);
                    const float4 b0 = *reinterpret_cast<const float4*>(bhn_s + ub + sc * 8);
                    const float4 b1 = *reinterpret_cast<const float4*>(bhn_s + ub + sc * 8 + 4);
                    bh[0] = b0.x; bh[1] = b0.y; bh[2] = b0.z; bh[3] = b0.w; bh[4] = b1.x; bh[5] = b1.y; bh[6] = b1.z; bh[7] = b1.w;
                };
                if (!kRecompute) load_hp_bh();
                tmem_ld_wait();
                if (kRecompute) {               // rec_fwd_pair_kernel's gate math, then the fp16 rounding of the saved gates
                    tmem_ld_32x32b_x8(taddr + st * 256 + sc * 8 + 64, az);     // (z after r and n: 8 registers fewer at the peak)
                    load_hp_bh();
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float rf = fmaf(0.5f, tanh_fast(__uint_as_float(ar[j])), 0.5f);
                        const float nf = tanh_fast(fmaf(rf, __uint_as_float(ahn[j]) + bh[j], __uint_as_float(ax[j])));
                        r[j] = round_h(rf); n[j] = round_h(nf);
                    }
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j) z[j] = round_h(active ? fmaf(0.5f, tanh_fast(__uint_as_float(az[j])), 0.5f) : 1.0f);
                }
                float gr[8], gz[8], gn[8], ghn[8];
                uint32_t carry[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    float dov = active ? dout[j] : 0.0f;
                    if (kDrop) dov = ((dbits >> (sc * 8 + j)) & 1u) ? dov * dscale : 0.0f;
                    const float dh = __uint_as_float(acc[j]) + dov;
                    const float hn = __uint_as_float(ahn[j]) + bh[j];
                    const float omz = 1.0f - z[j];
                    gn[j] = dh * omz * fmaf(-n[j], n[j], 1.0f);
                    gz[j] = dh * (hp[j] - n[j]) * (z[j] * omz);
                    ghn[j] = gn[j] * r[j];
                    gr[j] = ghn[j] * (hn * (1.0f - r[j]));
                    carry[j] = __float_as_uint(dh * z[j]);
                    // past a trace's end (z = 1) every gate gradient is zero; written as +0: the r and n a forward step past
                    // the end saw are not those of the recorded h_{t-1}, and only the sign of that zero could tell them apart
                    if (kVarLen && !active) gr[j] = gz[j] = gn[j] = ghn[j] = 0.0f;
                }
                const uint4 vr = pack8(gr), vz = pack8(gz), vn = pack8(gn), vh = pack8(ghn);
                // A operand of the dh matvec: K order r | z | hn
                *reinterpret_cast<uint4*>(a_row + (0 * 16 + cb + sc) * CHUNK_S) = vr;
                *reinterpret_cast<uint4*>(a_row + (1 * 16 + cb + sc) * CHUNK_S) = vz;
                *reinterpret_cast<uint4*>(a_row + (2 * 16 + cb + sc) * CHUNK_S) = vh;
                stg16(dgblk + (long long)(0 * 16 + sc) * CHUNK_G, vr);
                stg16(dgblk + (long long)(1 * 16 + sc) * CHUNK_G, vz);
                stg16(dgblk + (long long)(2 * 16 + sc) * CHUNK_G, vn);
                stg16(dgblk + (long long)(3 * 16 + sc) * CHUNK_G, vh);
                tmem_st_32x32b_x8(taddr + (kRecompute ? st * 256 : 0) + sc * 8, carry);   // kRecompute: over r, read above
            }
            tmem_st_wait();
            fence_proxy_async();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(&hp_free[st]);                 // this warp is done with the stage's h_{t-1} tile and hn buffer
                mbar_arrive_cluster(ar_remote);
            }
            // The MEMBAR inside fence.proxy.async waits for every global load of the thread still in flight (ncu: 7 % of the
            // step), so the next step's first chunk is requested only AFTER the arrival: it flies under the wait for the dh MMA.
            // (Deferring the last chunk's four stores the same way, which pays in the forward kernel, costs 17 % here.)
            if (sidx + 1 < T) {
                if (!kRecompute) g_ptr += g_step;
                if (do_ptr) do_ptr += do_step;
                load_raw(0);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 0) tmem_dealloc_pair<TMEM_COLS>(tmem_base);
}

// (B, T, C) fp32 mask (0 or 1/keep) -> one bit per element in the order the recurrence kernels read them,
// [tile][T][128 rows][C/8 bytes]; *scale = the non-zero value of the mask (max over all elements).
__global__ void pack_drop_mask_kernel(const float* __restrict__ mask, int B, int T, int C, uint8_t* __restrict__ bits,
                                      unsigned int* __restrict__ scale_bits, long long n_bytes) {
    float mx = 0.0f;
    const int cb = C / 8;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_bytes; e += (long long)gridDim.x * blockDim.x) {
        const int c = e % cb;
        const long long rt = e / cb;
        const int row = rt & 127;
        const long long tt = rt >> 7;
        const int t = tt % T;
        const long long b = (tt / T) * 128 + row;
        unsigned int v = 0;
        if (b < B) {
            const float4* src = reinterpret_cast<const float4*>(mask + ((long long)b * T + t) * C + c * 8);
            const float4 m0 = __ldg(src), m1 = __ldg(src + 1);
            const float m[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (m[j] != 0.0f) v |= 1u << j;
                mx = fmaxf(mx, m[j]);
            }
        }
        bits[e] = static_cast<uint8_t>(v);
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    if ((threadIdx.x & 31) == 0 && mx > 0.0f) atomicMax(scale_bits, __float_as_uint(mx));   // positive floats order like their bits
}

// Bernoulli(keep) bits straight from a counter-based generator (no (B, T, C) float mask in HBM): the training default.
__device__ __forceinline__ uint64_t mix64(uint64_t x) {       // splitmix64 finaliser
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL; x ^= x >> 27; x *= 0x94d049bb133111ebULL; x ^= x >> 31;
    return x;
}
__global__ void gen_drop_bits_kernel(uint8_t* __restrict__ bits, long long n_bytes, unsigned long long seed, uint32_t keep_thr16,
                                     float* __restrict__ scale) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *scale = 65536.0f / static_cast<float>(keep_thr16);   // 1 / (probability actually used)
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_bytes / 4; e += (long long)gridDim.x * blockDim.x) {
        uint32_t word = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {                      // four 16-bit uniforms per 64-bit hash
            const uint64_t h = mix64(seed + (static_cast<uint64_t>(e) << 3) + k + 0x9e3779b97f4a7c15ULL * (k + 1));
#pragma unroll
            for (int q = 0; q < 4; ++q) word |= (((h >> (16 * q)) & 0xffffu) < keep_thr16 ? 1u : 0u) << (4 * k + q);
        }
        reinterpret_cast<uint32_t*>(bits)[e] = word;
    }
}

// x (B, T, I <= 2) fp32 -> [tiles][T][128 rows][8] bf16: the input chunk the layer-0 forward kernel packs into its A tile, for
// every trace row and step (pad traces: the bias columns only, as there).  The A operand of the backward's gate recompute.
__global__ void pack_x_steps_kernel(const float* __restrict__ x, int B, int T, int I, uint4* __restrict__ out, long long n_rows) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_rows; e += (long long)gridDim.x * blockDim.x) {
        const long long bt = e >> 7;                   // e = (tile * T + t) * 128 + row
        const long long b = (bt / T) * 128 + (e & 127);
        out[e] = pack_x(b < B ? x + (b * T + bt % T) * I : nullptr, I);
    }
}

int rec_mode() {            // RS_REC_MODE: 0 = automatic, 2 = NT = 1, 3 = NT = 2
    const char* e = getenv("RS_REC_MODE");
    return e ? atoi(e) : 0;
}

}  // namespace

namespace rs {

// Tiles in flight per CTA pair of the forward kernel.  Measured on B200 (ms per 500-step launch pair at 1024 / 8192 traces;
// "one CTA per tile" = round 1's kernels, retired):
//   forward : one CTA per tile 5.1 / 6.3   pair NT=1 2.7 / 6.3   pair NT=2 4.1 / 5.8
//   backward: one CTA per tile 5.5 / 7.4   pair NT=1 2.9 / 6.9   pair NT=2 5.8 / 8.0
// Forward: NT = 1 while every tile can have its own pair of SMs in both directions (<= 37 tiles), else NT = 2 (the MMA of one
// tile runs under the epilogue of the other).  The backward kernel is built for one tile per pair only: its epilogue is bound
// by the latency of its gate / d_out loads, which two waves of half-size CTAs hide better than two tiles on one
// register-capped CTA.  RS_REC_MODE=2 / 3 forces NT = 1 / 2 (tests/test_rec_kernels_gpu.py runs both).
int rec_fwd_nt(int B) {
    const int mode = rec_mode();
    if (mode == 2) return 1;
    if (mode == 3) return 2;
    const int n_tiles = (B + 127) / 128;
    return (n_tiles * 4 <= 148) ? 1 : 2;
}

int rec_fwd_pair(const float* x, int I, const void* P, const void* X, const void* Wih, const void* Whh, const float* b_hn, void* out,
                 void* gates, float* h_n, const int* lengths, const void* drop_bits, const float* drop_scale, void* out_drop, int split,
                 int B, int T, int nt, int pf_dist, cudaStream_t stream) {
    FwdPairParams p = {};
    p.x = x; p.I = I;
    p.P = static_cast<const uint8_t*>(P); p.p_block_bytes = 6LL * H * 256;
    p.X = static_cast<const uint8_t*>(X); p.x_block_bytes = 2LL * H * 256; p.Wih = static_cast<const uint8_t*>(Wih);
    p.Whh = static_cast<const uint8_t*>(Whh); p.b_hn = b_hn;
    p.out = static_cast<uint8_t*>(out); p.out_block_bytes = 2LL * H * 256;
    p.gates = static_cast<uint8_t*>(gates); p.h_n = h_n; p.lengths = lengths;
    p.drop_bits = static_cast<const uint8_t*>(drop_bits); p.drop_scale = drop_scale; p.out_drop = static_cast<uint8_t*>(out_drop);
    p.B = B; p.T = T; p.n_tiles = (B + 127) / 128; p.pf_dist = pf_dist; p.split = split ? 1 : 0;
    const int mode = X ? 2 : (x ? 1 : 0);
    if (mode == 2) nt = 1;                  // the fused projection runs one tile per pair (two waves above 37 tiles)
    const int xc = mode == 1 ? x_chunks(I) : 1;     // layer 0: 16-byte input chunks per row (kXC of the kernel)
    const int xs = (xc + 1) / 2;                    // input K steps
    auto smem_of = [&](int nt_) {
        return (16 * (1 + p.split) + (mode ? 2 * xs : 0)) * W_CHUNK + (mode == 2 ? 32 * W_CHUNK + 32 * CHUNK_S : 0)
               + nt_ * (16 + 2 * xs * (xc == 1 ? 1 : 2)) * CHUNK_S + (nt_ == 1 ? 0 : nt_ * H32_BYTES) + H * 4 + 256;
    };
    // split weights with 3 or 4 input K steps (I >= 11) and two tiles in flight need 235 / 245 KB: one tile per pair then
    if (nt == 2 && smem_of(2) > 227 * 1024) nt = 1;
    const int pairs = (p.n_tiles + nt - 1) / nt;
    const int smem = smem_of(nt);
    const dim3 grid(2 * pairs, 2);
#define RS_LAUNCH_FWD_D(NT_, VL_, MODE_, DROP_, XC_)                                                                    \
    do {                                                                                                                \
        RS_CUDA_OK(cudaFuncSetAttribute(rec_fwd_pair_kernel<NT_, VL_, MODE_, DROP_, XC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        rec_fwd_pair_kernel<NT_, VL_, MODE_, DROP_, XC_><<<grid, NUM_THREADS, smem, stream>>>(p);                       \
    } while (0)
#define RS_LAUNCH_FWD_X(NT_, VL_, MODE_, XC_)                                                                           \
    do {                                                                                                                \
        if (p.drop_bits) RS_LAUNCH_FWD_D(NT_, VL_, MODE_, true, XC_); else RS_LAUNCH_FWD_D(NT_, VL_, MODE_, false, XC_); \
    } while (0)
#define RS_LAUNCH_FWD(NT_, VL_, MODE_) RS_LAUNCH_FWD_X(NT_, VL_, MODE_, 1)
#define RS_LAUNCH_FWD_M(NT_, VL_)                                                                                       \
    do {                                                                                                                \
        if (mode != 1) RS_LAUNCH_FWD(NT_, VL_, 0);                                                                      \
        else if (xc == 1) RS_LAUNCH_FWD(NT_, VL_, 1);                                                                   \
        else if (xc == 2) RS_LAUNCH_FWD_X(NT_, VL_, 1, 2);                                                              \
        else if (xc == 4) RS_LAUNCH_FWD_X(NT_, VL_, 1, 4);                                                              \
        else if (xc == 6) RS_LAUNCH_FWD_X(NT_, VL_, 1, 6);                                                              \
        else RS_LAUNCH_FWD_X(NT_, VL_, 1, 8);                                                                           \
    } while (0)
    if (mode == 2) { if (lengths) RS_LAUNCH_FWD(1, true, 2); else RS_LAUNCH_FWD(1, false, 2); }
    else if (nt == 1) { if (lengths) RS_LAUNCH_FWD_M(1, true); else RS_LAUNCH_FWD_M(1, false); }
    else { if (lengths) RS_LAUNCH_FWD_M(2, true); else RS_LAUNCH_FWD_M(2, false); }
#undef RS_LAUNCH_FWD_M
#undef RS_LAUNCH_FWD
#undef RS_LAUNCH_FWD_X
#undef RS_LAUNCH_FWD_D
    count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

int rec_bwd_pair(const void* d_out, const float* d_h_n, const void* gates, const float* x, int I, void* xpack, const void* out,
                 const void* WhhT, const void* Whh, int whh_chunks, const float* b_hn, void* dG, const int* lengths,
                 const void* drop_bits, const float* drop_scale, int split, int B, int T, int pf_dist, cudaStream_t stream) {
    const bool recompute = x != nullptr;
    if (recompute) {
        const long long n_rows = (long long)((B + 127) / 128) * T * 128;
        long long blocks = (n_rows + 255) / 256;
        if (blocks > 148 * 16) blocks = 148 * 16;
        pack_x_steps_kernel<<<(int)blocks, 256, 0, stream>>>(x, B, T, I, static_cast<uint4*>(xpack), n_rows);
        count_launch();
        RS_CUDA_OK(cudaGetLastError());
    }
    BwdPairParams p = {};
    p.d_out = static_cast<const uint8_t*>(d_out); p.dout_block_bytes = 2LL * H * 256;
    p.d_h_n = d_h_n; p.gates = static_cast<const uint8_t*>(gates); p.xpack = static_cast<const uint8_t*>(xpack);
    p.out = static_cast<const uint8_t*>(out); p.out_block_bytes = 2LL * H * 256;
    p.WhhT = static_cast<const uint8_t*>(WhhT);
    p.Whh = static_cast<const uint8_t*>(Whh); p.whh_chunks = whh_chunks; p.b_hn = b_hn;
    p.dG = static_cast<uint8_t*>(dG); p.dg_block_bytes = 8LL * H * 256;
    p.lengths = lengths;
    p.drop_bits = static_cast<const uint8_t*>(drop_bits); p.drop_scale = drop_scale;
    p.B = B; p.T = T; p.n_tiles = (B + 127) / 128; p.split = split ? 1 : 0; p.pf_dist = pf_dist;
    const int smem = recompute ? W_BWD_BYTES + A_BWD_BYTES + WF_BYTES + 2 * (HP_BYTES + 2 * CHUNK_S) + H * 4 + 256
                               : (1 + p.split) * (W_BWD_BYTES + 16 * CHUNK_S) + A_BWD_BYTES + 2 * HP_BYTES + H * 4 + 256;
    const dim3 grid(2 * p.n_tiles, 2);
#define RS_LAUNCH_BWD_R(VL_, DROP_, RC_)                                                                                \
    do {                                                                                                                \
        RS_CUDA_OK(cudaFuncSetAttribute(rec_bwd_pair_kernel<VL_, DROP_, RC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
        rec_bwd_pair_kernel<VL_, DROP_, RC_><<<grid, NUM_THREADS, smem, stream>>>(p);                                   \
    } while (0)
#define RS_LAUNCH_BWD(VL_, DROP_)                                                                                       \
    do {                                                                                                                \
        if (recompute) RS_LAUNCH_BWD_R(VL_, DROP_, true); else RS_LAUNCH_BWD_R(VL_, DROP_, false);                       \
    } while (0)
    if (lengths) { if (p.drop_bits) RS_LAUNCH_BWD(true, true); else RS_LAUNCH_BWD(true, false); }
    else { if (p.drop_bits) RS_LAUNCH_BWD(false, true); else RS_LAUNCH_BWD(false, false); }
#undef RS_LAUNCH_BWD
#undef RS_LAUNCH_BWD_R
    count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

}  // namespace rs

extern "C" int rs_pack_drop_mask(const float* mask, int B, int T, int C, void* bits, float* scale, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(mask && bits && scale && B >= 0 && T >= 0 && C > 0 && C % 32 == 0, "rs_pack_drop_mask: bad arguments (C must be a multiple of 32)");
    RS_CUDA_OK(cudaMemsetAsync(scale, 0, sizeof(float), stream));
    const long long n_bytes = (long long)((B + 127) / 128) * T * 128 * (C / 8);
    if (n_bytes == 0) return 0;
    long long blocks = (n_bytes + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pack_drop_mask_kernel<<<(int)blocks, 256, 0, stream>>>(mask, B, T, C, static_cast<uint8_t*>(bits),
                                                          reinterpret_cast<unsigned int*>(scale), n_bytes);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_gen_drop_bits(void* bits, int B, int T, int C, float keep, uint64_t seed, float* scale, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(bits && scale && B >= 0 && T >= 0 && C > 0 && C % 32 == 0 && keep > 0.0f && keep <= 1.0f, "rs_gen_drop_bits: bad arguments");
    const long long n_bytes = (long long)((B + 127) / 128) * T * 128 * (C / 8);
    if (n_bytes == 0) return 0;
    // keep is quantised to 16 bits; the scale is the reciprocal of the probability actually used
    uint32_t thr = static_cast<uint32_t>(keep * 65536.0f + 0.5f);
    if (thr > 65536u) thr = 65536u;
    if (thr == 0u) thr = 1u;
    long long blocks = (n_bytes / 4 + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    gen_drop_bits_kernel<<<(int)blocks, 256, 0, stream>>>(static_cast<uint8_t*>(bits), n_bytes, seed, thr, scale);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
