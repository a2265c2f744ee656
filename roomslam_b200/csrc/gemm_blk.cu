// bf16 tensor-core GEMMs over the library's TILE-MAJOR activation layout (bf16 mode, SURVEY.md 8(a) rows a2, a4).
//
// Tile-major layout of a per-timestep activation with C columns: blocks indexed by (trace tile of 128, time row t'),
// each block = [C/8 chunks][128 traces][8 bf16] = C*256 contiguous bytes.  Every block (and every run of chunks in
// it) is ONE contiguous piece, so operands move with 1-D bulk copies (cp.async.bulk, mbarrier completion) and land in
// shared memory already in tcgen05's no-swizzle core-matrix form (8 rows x 16 bytes = 128 contiguous bytes):
//   as a K-major  operand (rows = traces,  K = columns): lbo = 2048 (next 16-byte K chunk), sbo = 128
//   as an MN-major operand (M/N = columns, K = traces ): lbo = 128 (next 8 traces),        sbo = 2048
// and the recurrence kernels read / write the same blocks with perfectly coalesced 16-byte accesses per thread.
//
//   blk_gemm_nt : per block m:  C_blk[:, n] = A_blk[:, kchunks] . W[n, :]^T + bias      (bf16 out, direct stores)
//                 -> input projection P = X W_ih^T + b  and  dX = dG W_ih
//   blk_wgrad   : C[M, N] += sum over blocks  A_blk[:, mchunks]^T . B_blk'[:, nchunks]   (fp32 out, split over blocks)
//                 (the split reductions end in fp32 atomics; deterministic mode stores per-split partials into a workspace
//                 and rs::slot_sum adds them in split order)
//                 -> dW_ih, dW_hh (block of dG at t' paired with the block of h at t' -/+ 1), bias gradients (ones column)
//
// Warp roles: warp 0 = bulk-copy producer, warp 1 = tcgen05.mma issuer (one lane), warps 2..5 = TMEM epilogue.
#include <stdlib.h>

#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

constexpr int CHUNK_BYTES = 2048;          // one 16-byte column chunk of a 128-trace block
constexpr int PIECE_BYTES = 8 * CHUNK_BYTES;   // 64 columns x 128 traces = 16 KB
constexpr int NT_STAGES = 6;               // ring depth: look-ahead that covers the L2 latency of the W pieces
constexpr int NT_MAX_KB = 24;             // 12 K blocks of the data gradient, twice with split (hi + lo) weights
constexpr int NUM_THREADS = 192;

struct NtParams {
    const uint8_t* A;  long long a_block_bytes;  int a_kchunk[NT_MAX_KB];   // chunk offset of each 64-column K block
    const uint8_t* W;                                                        // [n_tiles][k_blocks][8][128][8] bf16
    uint8_t* C;        long long c_block_bytes;  int c_chunk0;
    const float* bias;
    int n_blocks, n_tiles, k_blocks;
    // optional dropout mask on C (the data gradient of a layer whose INPUT went through inter-layer dropout): one bit per
    // element, [tile][T][128 rows][c_cols / 8 bytes] as the recurrence kernels read it; block m = tile * (T + 2) + t + 1
    const uint8_t* drop_bits; const float* drop_scale; int drop_T; int drop_row_bytes;
};

constexpr int NT_THREADS = 320;            // warp 0 producer, warp 1 MMA issuer, warps 2..9 epilogue (2 per TMEM lane quadrant)
constexpr int NT_MAX_N = 1024;             // bias staged in shared memory

__global__ void __launch_bounds__(NT_THREADS, 1) blk_gemm_nt_kernel(const NtParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    // ring of (A piece | W piece) stages (32 KB each)
    constexpr int kStageBytes = 2 * PIECE_BYTES;
    uint8_t* stages = smem;
    float* bias_s = reinterpret_cast<float*>(stages + NT_STAGES * kStageBytes);
    uint64_t* bars = reinterpret_cast<uint64_t*>(bias_s + NT_MAX_N);
    uint64_t* full_bar = bars;                       // [NT_STAGES]
    uint64_t* empty_bar = bars + NT_STAGES;          // [NT_STAGES]
    uint64_t* acc_full = bars + 2 * NT_STAGES;       // [2]
    uint64_t* acc_empty = bars + 2 * NT_STAGES + 2;  // [2]
    // [4] unused barriers, still initialised: removing them changes this kernel's machine code, a change to measure on its own
    uint64_t* spare = bars + 2 * NT_STAGES + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NT_STAGES + 8);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < NT_STAGES; ++s) { rs::mbar_init(&full_bar[s], 1); rs::mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) {
            rs::mbar_init(&acc_full[s], 1); rs::mbar_init(&acc_empty[s], 8);
            rs::mbar_init(&spare[s], 1);    rs::mbar_init(&spare[2 + s], 1);
        }
        rs::fence_mbar_init();
    }
    if (warp == 1) rs::tmem_alloc<256>(tmem_slot);
    for (int i = threadIdx.x; i < p.n_tiles * 128; i += NT_THREADS) bias_s[i] = p.bias ? p.bias[i] : 0.0f;
    rs::tc_fence_before();
    __syncthreads();
    rs::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (rs::elect_one()) {
            int stage = 0; uint32_t phase = 0;
            for (int m = blockIdx.x; m < p.n_blocks; m += gridDim.x) {
                const uint8_t* ablk = p.A + (long long)m * p.a_block_bytes;
                for (int n = 0; n < p.n_tiles; ++n) {
                    for (int kb = 0; kb < p.k_blocks; ++kb) {
                        rs::mbar_wait(&empty_bar[stage], phase ^ 1);
                        uint8_t* ss = stages + stage * kStageBytes;
                        rs::mbar_expect_tx(&full_bar[stage], kStageBytes);
                        rs::bulk_load(ss, ablk + (long long)p.a_kchunk[kb] * CHUNK_BYTES, PIECE_BYTES, &full_bar[stage]);
                        rs::bulk_load(ss + PIECE_BYTES, p.W + ((long long)n * p.k_blocks + kb) * PIECE_BYTES, PIECE_BYTES,
                                      &full_bar[stage]);
                        if (++stage == NT_STAGES) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc = rs::umma_idesc_bf16(128, 128, 0, 0);
        int stage = 0; uint32_t phase = 0; int acc = 0; uint32_t acc_phase = 0;
        for (int m = blockIdx.x; m < p.n_blocks; m += gridDim.x) {
            for (int n = 0; n < p.n_tiles; ++n) {
                rs::mbar_wait(&acc_empty[acc], acc_phase ^ 1);
                rs::tc_fence_after();
                const uint32_t tmem_d = tmem_base + acc * 128;
                for (int kb = 0; kb < p.k_blocks; ++kb) {
                    rs::mbar_wait(&full_bar[stage], phase);
                    rs::tc_fence_after();
                    if (rs::elect_one()) {
                        const uint32_t sa = rs::smem_u32(stages + stage * kStageBytes);
                        const uint32_t sb = sa + PIECE_BYTES;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            const uint64_t da = rs::umma_desc_noswz(sa + k * 2 * CHUNK_BYTES, CHUNK_BYTES, 128);
                            const uint64_t db = rs::umma_desc_noswz(sb + k * 2 * CHUNK_BYTES, CHUNK_BYTES, 128);
                            rs::tc_mma_bf16(tmem_d, da, db, idesc, (kb | k) != 0);
                        }
                        rs::tc_commit(&empty_bar[stage]);
                        if (kb == p.k_blocks - 1) rs::tc_commit(&acc_full[acc]);
                    }
                    __syncwarp();
                    if (++stage == NT_STAGES) { stage = 0; phase ^= 1; }
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3, row = q * 32 + lane;
        const int chalf = (warp - 2) >> 2;              // which 64 of the 128 tile columns this warp converts
        int acc = 0; uint32_t acc_phase = 0;
        const float dscale = p.drop_bits ? __ldg(p.drop_scale) : 1.0f;
        for (int m = blockIdx.x; m < p.n_blocks; m += gridDim.x) {
            uint8_t* cblk = p.C + (long long)m * p.c_block_bytes + row * 16;
            const uint8_t* drow = nullptr;                  // this row's mask bytes of the block (pad rows t' = 0, T + 1: none)
            if (p.drop_bits) {
                const int tp = m % (p.drop_T + 2);
                if (tp >= 1 && tp <= p.drop_T)
                    drow = p.drop_bits + (((long long)(m / (p.drop_T + 2)) * p.drop_T + (tp - 1)) * 128 + row) * p.drop_row_bytes;
            }
            for (int n = 0; n < p.n_tiles; ++n) {
                rs::mbar_wait(&acc_full[acc], acc_phase);
                rs::tc_fence_after();
                const uint32_t taddr = tmem_base + acc * 128 + chalf * 64 + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll
                for (int c0 = 0; c0 < 64; c0 += 32) {
                    uint32_t r[32];
                    rs::tmem_ld_32x32b_x32(taddr + c0, r);
                    uint32_t mbits = 0xffffffffu;           // 4 chunks x 8 columns
                    if (drow) mbits = __ldg(reinterpret_cast<const uint32_t*>(drow + p.c_chunk0 + n * 16 + chalf * 8 + c0 / 8));
                    rs::tmem_ld_wait();
                    if (drow) {                             // the pad rows have no mask: left unscaled, as without dropout
#pragma unroll
                        for (int e = 0; e < 32; ++e)
                            r[e] = ((mbits >> e) & 1u) ? __float_as_uint(__uint_as_float(r[e]) * dscale) : 0u;
                    }
                    const float* bs = bias_s + n * 128 + chalf * 64 + c0;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        uint32_t pk[4];
                        const float4 b0 = *reinterpret_cast<const float4*>(bs + 8 * j);
                        const float4 b1 = *reinterpret_cast<const float4*>(bs + 8 * j + 4);
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float v0 = __uint_as_float(r[8 * j + 2 * e]) + bb[2 * e];
                            const float v1 = __uint_as_float(r[8 * j + 2 * e + 1]) + bb[2 * e + 1];
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(v0, v1);
                            pk[e] = *reinterpret_cast<uint32_t*>(&h2);
                        }
                        const int chunk = p.c_chunk0 + n * 16 + chalf * 8 + c0 / 8 + j;
                        *reinterpret_cast<uint4*>(cblk + (long long)chunk * CHUNK_BYTES) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                }
                rs::tc_fence_before();
                __syncwarp();
                if (lane == 0) rs::mbar_arrive(&acc_empty[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    }
    rs::tc_fence_before();
    __syncthreads();
    if (warp == 1) rs::tmem_dealloc<256>(tmem_base);
}

// ---------------------------------------------------------------------------------------------------------------
// Fused weight-gradient pass: ONE launch computes every dW_ih / dW_hh / bias-gradient block of a layer.
// A "role" = one 128-column block of dG (one gate of one direction) against one B source:
//     C_role[128, n_cols] += sum over blocks  dG_blk[:, role columns]^T . B_blk'[:, ...]      (B_blk' time-shifted by b_shift)
//     bias_role[128]      += sum over blocks  dG_blk[:, role columns]^T . 1                    (extra N=16 MMA on a ones tile)
// Work item = (split of the block range, role); the roles of one split sit on neighbouring CTAs and walk the same
// blocks at the same time, so a dG piece needed by two roles (and the B blocks shared by several) come from HBM once
// and from L2 afterwards: dG is streamed from DRAM exactly once per layer instead of once per consumer.
constexpr int WG_MAX_ROLES = 18;
struct WgRole {
    int a_mchunk;                       // first 16-byte chunk of the dG columns of this role
    const uint8_t* B; long long b_block_bytes; int b_chunk0; int n_cols; int b_shift;
    float* C; long long ldc;            // C rows [0,128) x n_cols of this role
    float* bias;                        // 128 floats or NULL
    const uint8_t* B2; long long b2_block_bytes;   // optional second B source: 16 columns (2 chunks), no time shift
    float* C2; long long ldc2;          // 128 x 16
};
struct WgParams {
    const uint8_t* A; long long a_block_bytes;
    const uint8_t* ones;                // [2 chunks][128][8] bf16, first column = 1
    WgRole role[WG_MAX_ROLES];
    int n_roles, tiles, T, Tp, splits, blocks_per_split, max_b_bytes;
    // paired launch (cluster of 2 CTAs = roles 2 j, 2 j + 1 of a split): bit j set = the two roles read the SAME dG block, the
    // even CTA bulk-copies it once with cluster multicast into both CTAs' stages
    int paired; unsigned int share_mask;
    long long ws_split;                 // deterministic mode: floats per split slot (role outputs point into slot 0)
};

// Paired mode.  A dG block feeds two roles (its ih role against X, its hh role against h); as single CTAs they move 96 and 64 KB
// per block, drift apart and miss each other in L2 -- layer 1 read exactly its four shared gate blocks twice (16.7 GB for
// 12.6 GB of operands, ncu).  As a cluster of two the even CTA's producer loads the block ONCE and multicasts it into both
// stages; it waits for both CTAs' MMAs to retire before it refills a stage (the odd CTA's tcgen05.commit arrives on both
// empty barriers), each CTA streams its own B operand.  The shared ring keeps the pair in lockstep by construction.
// kDet: the outputs of role r point into slot 0 of a workspace; item (split, r) stores to slot `split` (+ split * ws_split)
template <bool kDet>
__global__ void __launch_bounds__(NUM_THREADS, 1) blk_wgrad_kernel(const WgParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int stage_bytes = 2 * PIECE_BYTES + p.max_b_bytes + 2 * CHUNK_BYTES;   // A | B | B2 (16 columns)
    uint8_t* stages = smem;
    uint8_t* ones_s = smem + 2 * stage_bytes;                    // 4 KB
    uint64_t* bars = reinterpret_cast<uint64_t*>(ones_s + 2 * CHUNK_BYTES);
    uint64_t* full_bar = bars;        // [2]
    uint64_t* empty_bar = bars + 2;   // [2]
    uint64_t* acc_full = bars + 4;
    uint64_t* ones_full = bars + 5;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 6);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const uint32_t crank = p.paired ? rs::cluster_ctarank() : 0u;
    // paired launches run ONE item per CTA (host), so the role of this CTA is fixed: does its pair share the dG block?
    const bool shared_a = p.paired && ((p.share_mask >> ((static_cast<int>(blockIdx.x) % p.n_roles) >> 1)) & 1u);
    if (warp == 0 && lane == 0) {
        // shared: the even CTA's stage is free only when BOTH CTAs' MMAs on it retired (its own commit + the odd CTA's).
        // An unshared pair must NOT cross-signal: its odd CTA is not throttled by the even one and would complete the even
        // CTA's phases with arrivals of later blocks.
        for (int s = 0; s < 2; ++s) { rs::mbar_init(&full_bar[s], 1); rs::mbar_init(&empty_bar[s], (shared_a && crank == 0) ? 2 : 1); }
        rs::mbar_init(acc_full, 1);
        rs::mbar_init(ones_full, 1);
        rs::fence_mbar_init();
    }
    if (warp == 1) rs::tmem_alloc<512>(tmem_slot);
    rs::tc_fence_before();
    __syncthreads();
    if (p.paired) rs::cluster_sync_all();       // the peer's barriers exist before anything is multicast into them
    rs::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int total_blocks = p.tiles * p.T;
    const int items = p.n_roles * p.splits;
    int stage = 0; uint32_t phase = 0, acc_phase = 0;
    if (warp == 0 && lane == 0) {
        rs::mbar_expect_tx(ones_full, 2 * CHUNK_BYTES);
        rs::bulk_load(ones_s, p.ones, 2 * CHUNK_BYTES, ones_full);
    }
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const WgRole& R = p.role[item % p.n_roles];
        const int split = item / p.n_roles;
        const int i0 = split * p.blocks_per_split;
        const int i1 = min(total_blocks, i0 + p.blocks_per_split);
        const int b_bytes = R.n_cols * 256;
        // shared pair: the even CTA loads the dG block for both; else every CTA loads its own
        if (warp == 0) {
            if (rs::elect_one()) {
                for (int i = i0; i < i1; ++i) {
                    const long long blk = (long long)(i / p.T) * p.Tp + 1 + (i % p.T);
                    rs::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = stages + stage * stage_bytes;
                    rs::mbar_expect_tx(&full_bar[stage], 2 * PIECE_BYTES + b_bytes + (R.B2 ? 2 * CHUNK_BYTES : 0));
                    const uint8_t* asrc = p.A + blk * p.a_block_bytes + (long long)R.a_mchunk * CHUNK_BYTES;
                    if (!shared_a) rs::bulk_load(sa, asrc, 2 * PIECE_BYTES, &full_bar[stage]);
                    else if (crank == 0) rs::bulk_load_mc(sa, asrc, 2 * PIECE_BYTES, &full_bar[stage], 3);
                    if (b_bytes)
                        rs::bulk_load(sa + 2 * PIECE_BYTES, R.B + (blk + R.b_shift) * R.b_block_bytes + (long long)R.b_chunk0 * CHUNK_BYTES,
                                      b_bytes, &full_bar[stage]);
                    if (R.B2)
                        rs::bulk_load(sa + 2 * PIECE_BYTES + p.max_b_bytes, R.B2 + blk * R.b2_block_bytes, 2 * CHUNK_BYTES, &full_bar[stage]);
                    if (++stage == 2) { stage = 0; phase ^= 1; }
                }
            }
        } else if (warp == 1) {
            const uint32_t idesc = rs::umma_idesc_bf16(128, R.n_cols ? R.n_cols : 16, 1, 1);
            const uint32_t idesc1 = rs::umma_idesc_bf16(128, 16, 1, 1);
            rs::mbar_wait(ones_full, 0);
            const uint32_t so = rs::smem_u32(ones_s);
            for (int i = i0; i < i1; ++i) {
                rs::mbar_wait(&full_bar[stage], phase);
                rs::tc_fence_after();
                if (rs::elect_one()) {
                    const uint32_t sa = rs::smem_u32(stages + stage * stage_bytes);
                    const uint32_t sb = sa + 2 * PIECE_BYTES;
#pragma unroll
                    for (int k = 0; k < 8; ++k) {       // 128 traces = 8 K-steps of 16
                        const uint64_t da = rs::umma_desc_noswz(sa + k * 256, 128, CHUNK_BYTES);
                        if (R.n_cols) {
                            const uint64_t db = rs::umma_desc_noswz(sb + k * 256, 128, CHUNK_BYTES);
                            rs::tc_mma_bf16(tmem_base, da, db, idesc, (i != i0) || (k != 0));
                        }
                        if (R.bias) {
                            const uint64_t d1 = rs::umma_desc_noswz(so + k * 256, 128, CHUNK_BYTES);
                            rs::tc_mma_bf16(tmem_base + 256, da, d1, idesc1, (i != i0) || (k != 0));
                        }
                        if (R.B2) {
                            const uint64_t d2 = rs::umma_desc_noswz(sb + p.max_b_bytes + k * 256, 128, CHUNK_BYTES);
                            rs::tc_mma_bf16(tmem_base + 272, da, d2, idesc1, (i != i0) || (k != 0));
                        }
                    }
                    if (shared_a && crank == 1) rs::tc_commit_mc(&empty_bar[stage], 3);   // own stage + the even CTA's
                    else rs::tc_commit(&empty_bar[stage]);
                    if (i == i1 - 1) rs::tc_commit(acc_full);
                }
                __syncwarp();
                if (++stage == 2) { stage = 0; phase ^= 1; }
            }
        } else if (i1 > i0) {
            const int q = warp & 3, row = q * 32 + lane;
            rs::mbar_wait(acc_full, acc_phase);
            rs::tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
            const long long slot = kDet ? split * p.ws_split : 0;
            float* crow = R.C + slot + (long long)row * R.ldc;
            for (int c0 = 0; c0 < R.n_cols; c0 += 16) {
                uint32_t r[16];
                rs::tmem_ld_32x32b_x16(taddr + c0, r);
                rs::tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    if (kDet) crow[c0 + j] = __uint_as_float(r[j]);
                    else atomicAdd(crow + c0 + j, __uint_as_float(r[j]));
                }
            }
            if (R.bias) {
                uint32_t r[8];
                rs::tmem_ld_32x32b_x8(taddr + 256, r);
                rs::tmem_ld_wait();
                if (kDet) R.bias[slot + row] = __uint_as_float(r[0]);
                else atomicAdd(R.bias + row, __uint_as_float(r[0]));
            }
            if (R.B2) {
                uint32_t r[16];
                rs::tmem_ld_32x32b_x16(taddr + 272, r);
                rs::tmem_ld_wait();
                float* c2 = R.C2 + slot + (long long)row * R.ldc2;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    if (kDet) c2[j] = __uint_as_float(r[j]);
                    else atomicAdd(c2 + j, __uint_as_float(r[j]));
                }
            }
            rs::tc_fence_before();
        }
        if (i1 > i0) acc_phase ^= 1;
        __syncthreads();
        rs::tc_fence_after();
    }
    rs::tc_fence_before();
    __syncthreads();
    if (p.paired) rs::cluster_sync_all();       // the peer's commits / multicast copies target this CTA's shared memory
    if (warp == 1) rs::tmem_dealloc<512>(tmem_base);
}

int g_sms = 0;
int num_sms() {
    if (g_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_sms, cudaDevAttrMultiProcessorCount, dev);
    }
    return g_sms;
}

}  // namespace

static int blk_gemm_nt_impl(const void* A, int64_t a_cols, const int* a_kchunk, int k_blocks, const void* W,
                            int n_tiles, void* C, int64_t c_cols, int c_chunk0, const float* bias, int64_t n_blocks,
                            const void* drop_bits, const float* drop_scale, int drop_T, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (n_blocks == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(A && W && C && a_kchunk, "rs_blk_gemm_nt: null pointer");
    RS_REQUIRE(k_blocks >= 1 && k_blocks <= NT_MAX_KB && n_tiles >= 1, "rs_blk_gemm_nt: 1 <= k_blocks <= %d", NT_MAX_KB);
    RS_REQUIRE(a_cols % 8 == 0 && c_cols % 8 == 0 && n_blocks < (1ll << 31), "rs_blk_gemm_nt: bad shape");
    NtParams p = {};
    p.A = static_cast<const uint8_t*>(A); p.a_block_bytes = a_cols * 256;
    for (int i = 0; i < k_blocks; ++i) {
        RS_REQUIRE(a_kchunk[i] >= 0 && (a_kchunk[i] + 8) * 8 <= a_cols, "rs_blk_gemm_nt: K block %d outside the A block", i);
        p.a_kchunk[i] = a_kchunk[i];
    }
    RS_REQUIRE((c_chunk0 + n_tiles * 16) * 8 <= c_cols, "rs_blk_gemm_nt: output columns outside the C block");
    p.W = static_cast<const uint8_t*>(W);
    p.C = static_cast<uint8_t*>(C); p.c_block_bytes = c_cols * 256; p.c_chunk0 = c_chunk0;
    p.bias = bias; p.n_blocks = (int)n_blocks; p.n_tiles = n_tiles; p.k_blocks = k_blocks;
    RS_REQUIRE(n_tiles * 128 <= NT_MAX_N, "rs_blk_gemm_nt: at most %d output columns", NT_MAX_N);
    if (drop_bits) {
        RS_REQUIRE(drop_scale && drop_T >= 1 && n_blocks % (drop_T + 2) == 0 && c_chunk0 % 4 == 0 && c_cols % 32 == 0 && !bias,
                   "rs_blk_gemm_nt_drop: the mask needs drop_scale, whole tiles of T + 2 blocks, 32-column alignment and no bias");
        p.drop_bits = static_cast<const uint8_t*>(drop_bits); p.drop_scale = drop_scale; p.drop_T = drop_T;
        p.drop_row_bytes = (int)(c_cols / 8);
    }
    const int grid = (int)(n_blocks < num_sms() ? n_blocks : num_sms());
    const int smem = NT_STAGES * 2 * PIECE_BYTES + NT_MAX_N * 4 + 256;
    RS_CUDA_OK(cudaFuncSetAttribute(blk_gemm_nt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    blk_gemm_nt_kernel<<<grid, NT_THREADS, smem, stream>>>(p);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_blk_gemm_nt(const void* A, int64_t a_cols, const int* a_kchunk, int k_blocks, const void* W,
                              int n_tiles, void* C, int64_t c_cols, int c_chunk0, const float* bias, int64_t n_blocks,
                              void* stream_) {
    return blk_gemm_nt_impl(A, a_cols, a_kchunk, k_blocks, W, n_tiles, C, c_cols, c_chunk0, bias, n_blocks, nullptr, nullptr, 0, stream_);
}

// rs_blk_gemm_nt without bias whose output is multiplied by an inter-layer dropout mask in the epilogue: C = (A . W^T) (.) mask.
// The data gradient of a layer whose input went through dropout -- masking it here (a throughput-bound epilogue) keeps the
// mask tests out of the serial per-time-step chain of the BPTT kernel of the layer below.
extern "C" int rs_blk_gemm_nt_drop(const void* A, int64_t a_cols, const int* a_kchunk, int k_blocks, const void* W,
                                   int n_tiles, void* C, int64_t c_cols, int c_chunk0, int64_t n_blocks, const void* drop_bits,
                                   const float* drop_scale, int T, void* stream_) {
    RS_REQUIRE(drop_bits != nullptr, "rs_blk_gemm_nt_drop: drop_bits is required");
    return blk_gemm_nt_impl(A, a_cols, a_kchunk, k_blocks, W, n_tiles, C, c_cols, c_chunk0, nullptr, n_blocks, drop_bits, drop_scale, T, stream_);
}

// One launch for all weight / bias gradients of a layer.  Per role r < n_roles (HOST arrays of length n_roles):
// a_mchunk[r], B[r] (tile-major pointer), b_cols[r], b_chunk0[r], n_cols[r] (multiple of 16, <= 256), b_shift[r] in {-1,0,1},
// C[r] (fp32, 128 x n_cols[r], leading dimension ldc[r]), bias[r] (128 floats or NULL).  Outputs are ACCUMULATED into.
extern "C" int rs_blk_wgrad(const void* dG, int64_t a_cols, const void* ones_block, int n_roles, const int* a_mchunk,
                            const void* const* B, const int64_t* b_cols, const int* b_chunk0, const int* n_cols,
                            const int* b_shift, float* const* C, const int64_t* ldc, float* const* bias,
                            const void* const* B2, float* const* C2, int tiles, int T, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(dG && ones_block && a_mchunk && B && b_cols && b_chunk0 && n_cols && b_shift && C && ldc && bias && B2 && C2,
               "rs_blk_wgrad: null pointer");
    RS_REQUIRE(n_roles >= 1 && n_roles <= WG_MAX_ROLES, "rs_blk_wgrad: 1 <= n_roles <= %d", WG_MAX_ROLES);
    const long long total = (long long)tiles * T;
    if (total == 0) return 0;
    RS_REQUIRE(total < (1ll << 31) && a_cols % 8 == 0, "rs_blk_wgrad: bad shape");
    WgParams p = {};
    p.A = static_cast<const uint8_t*>(dG); p.a_block_bytes = a_cols * 256;
    p.ones = static_cast<const uint8_t*>(ones_block);
    p.n_roles = n_roles; p.tiles = tiles; p.T = T; p.Tp = T + 2;
    int max_n = 16;
    for (int r = 0; r < n_roles; ++r) {
        RS_REQUIRE(a_mchunk[r] >= 0 && (a_mchunk[r] + 16) * 8 <= a_cols, "rs_blk_wgrad: role %d columns outside dG", r);
        RS_REQUIRE(n_cols[r] >= 0 && n_cols[r] <= 256 && n_cols[r] % 16 == 0, "rs_blk_wgrad: role %d n_cols", r);
        RS_REQUIRE(n_cols[r] == 0 || (b_chunk0[r] * 8 + n_cols[r] <= b_cols[r] && B[r] && C[r]), "rs_blk_wgrad: role %d B/C", r);
        RS_REQUIRE(n_cols[r] > 0 || B2[r] || bias[r], "rs_blk_wgrad: role %d has nothing to do", r);
        RS_REQUIRE(!B2[r] || C2[r], "rs_blk_wgrad: role %d has B2 but no C2", r);
        RS_REQUIRE(b_shift[r] >= -1 && b_shift[r] <= 1, "rs_blk_wgrad: role %d shift", r);
        WgRole& R = p.role[r];
        R.a_mchunk = a_mchunk[r]; R.B = static_cast<const uint8_t*>(B[r]); R.b_block_bytes = b_cols[r] * 256;
        R.b_chunk0 = b_chunk0[r]; R.n_cols = n_cols[r]; R.b_shift = b_shift[r]; R.C = C[r]; R.ldc = ldc[r]; R.bias = bias[r];
        R.B2 = static_cast<const uint8_t*>(B2[r]); R.b2_block_bytes = 16 * 256; R.C2 = C2[r]; R.ldc2 = 16;
        if (n_cols[r] > max_n) max_n = n_cols[r];
    }
    p.max_b_bytes = max_n * 256;
    const bool det = rs::deterministic();
    int splits = (det ? rs::kDetSplitSms : num_sms()) / n_roles;
    if (splits < 1) splits = 1;
    if (splits > total) splits = (int)total;
    p.blocks_per_split = (int)((total + splits - 1) / splits);
    p.splits = (int)((total + p.blocks_per_split - 1) / p.blocks_per_split);
    const int smem = 2 * (2 * PIECE_BYTES + p.max_b_bytes + 2 * CHUNK_BYTES) + 2 * CHUNK_BYTES + 256;
    // deterministic mode: every role output gets a dense image in each split's workspace slot; after the launch one slot_sum
    // adds the slots onto the outputs in split order
    rs::StreamScratch ws(stream);
    rs::SlotSum<float> jobs[3 * WG_MAX_ROLES];
    int n_jobs = 0;
    if (det) {
        long long off[3 * WG_MAX_ROLES];
        for (int r = 0; r < n_roles; ++r) {
            const WgRole& R = p.role[r];
            if (R.n_cols) { off[n_jobs] = p.ws_split; jobs[n_jobs++] = {nullptr, R.C, R.ldc, 128, R.n_cols}; p.ws_split += 128LL * R.n_cols; }
            if (R.bias) { off[n_jobs] = p.ws_split; jobs[n_jobs++] = {nullptr, R.bias, 1, 128, 1}; p.ws_split += 128; }
            if (R.B2) { off[n_jobs] = p.ws_split; jobs[n_jobs++] = {nullptr, R.C2, R.ldc2, 128, 16}; p.ws_split += 128 * 16; }
        }
        RS_CUDA_OK(ws.alloc(sizeof(float) * p.splits * p.ws_split));
        for (int j = 0; j < n_jobs; ++j) jobs[j].parts = ws.as<float>() + off[j];
        for (int r = 0, j = 0; r < n_roles; ++r) {
            WgRole& R = p.role[r];
            if (R.n_cols) { R.C = ws.as<float>() + off[j++]; R.ldc = R.n_cols; }
            if (R.bias) R.bias = ws.as<float>() + off[j++];
            if (R.B2) R.C2 = ws.as<float>() + off[j++];
        }
    }
    const auto kernel = det ? blk_wgrad_kernel<true> : blk_wgrad_kernel<false>;
    RS_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int items = n_roles * p.splits;
    int grid = items < num_sms() ? items : num_sms();
    // paired mode: roles 2 j and 2 j + 1 form a cluster; where they name the same dG columns the block is loaded once (multicast).
    // RS_WGRAD_PAIR=0 launches every role as a single CTA instead.  Read on every call (as RS_REC_MODE is), so one process can
    // run both modes: tests/test_grad_gemm_gpu.py requires them to give the same values.
    const bool pair_off = getenv("RS_WGRAD_PAIR") && atoi(getenv("RS_WGRAD_PAIR")) == 0;
    unsigned int share = 0;
    if (n_roles % 2 == 0 && !pair_off)
        for (int r = 0; r < n_roles; r += 2)
            if (a_mchunk[r] == a_mchunk[r + 1]) share |= 1u << (r / 2);
    if (share && items <= num_sms()) {          // one item per CTA: the pair's roles are fixed for the whole launch
        grid &= ~1;
        p.paired = 1; p.share_mask = share;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        RS_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, p));
    } else {
        kernel<<<grid, NUM_THREADS, smem, stream>>>(p);
    }
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    if (det) return rs::slot_sum(jobs, n_jobs, p.splits, p.ws_split, true, stream);
    return 0;
}
