// bf16 tensor-core GEMM for sm_100a: TMA (cp.async.bulk.tensor) -> shared memory (128-byte swizzle) ->
// tcgen05.mma with the fp32 accumulator in TMEM -> tcgen05.ld epilogue.  Used for the time-parallel work of the
// bf16 mode (SURVEY.md 8(a) row a2 and the weight-gradient half of a4):
//
//   mode NT  : C[M,N] = A[M,K] . B[N,K]^T (+ bias[N]), A and B K-major (row-major with K contiguous), C bf16
//              written with TMA stores.  M is huge (B*(T+2) rows), N and K are small multiples of 128 / 64.
//              -> layer input projection  P = X . W_ih^T + b_ih   and   dX = dG . W_ih
//   mode TN  : C[M,N] += A[Kr,M]^T . B[Kr,N], reduction over the ROWS of A and B (both "MN-major" operands),
//              split over CTAs along Kr, fp32 result added to C with red.global.add.f32 (deterministic mode: per-split
//              partials in a workspace, summed in split order by rs::slot_sum).  A rows and B rows may be
//              shifted against each other by one (dW_hh pairs dGh_t with h_{t-1}).
//              -> dW_ih = dGx^T . X,  dW_hh = dGh^T . H_prev
//
// One CTA = 192 threads: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2..5 = epilogue
// (warp w owns TMEM lanes 32*(w%4) .. +31).  4-stage smem ring, 2 accumulator stages in TMEM (epilogue of tile
// i overlaps the MMAs of tile i+1), persistent over tiles.
#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

constexpr int BM = 128, BN = 128, BK = 64, STAGES = 4;
constexpr int TILE_A_BYTES = BM * BK * 2;   // 16 KB
constexpr int TILE_B_BYTES = BN * BK * 2;   // 16 KB
constexpr int STAGE_BYTES = TILE_A_BYTES + TILE_B_BYTES;
constexpr int C_STAGE_BYTES = BM * BN * 2;  // bf16 staging for the TMA store (NT mode)
constexpr int NUM_THREADS = 192;
constexpr uint32_t TMEM_COLS = 2 * BN;      // two accumulator stages

struct GemmParams {
    int M, N, K;            // NT: C is M x N, reduction K.  TN: C is M x N, reduction over Kr = K rows
    int m_tiles, n_tiles;
    int k_blocks;           // number of BK blocks in the (per-split) reduction
    int splits;             // TN: number of K splits
    int k_rows_per_split;   // TN: rows per split (multiple of BK)
    int a_row_shift, b_row_shift;   // TN: row offsets applied to the TMA coordinates of A and B
    int a_col0, b_col0;     // TN: column offsets inside the global matrices (select a column block)
    int n_seg, kb_per_seg;  // TN: the reduction runs over n_seg passes of the same rows with different column blocks
    int a_seg[8], b_seg[8]; // TN: extra column offset of A / B in pass s (split-operand GEMMs: one launch for all partial products)
    const float* bias;      // NT: optional
    int flags;              // NT: RS_GEMM_RELU, RS_GEMM_OUT_F32
    float* c_nt_f32; long long ldc_nt;   // NT with fp32 output: direct row stores
    float* c_f32;           // TN: output
    long long ldc;          // TN: leading dimension of C (floats)
};

// kDet (TN only): the tile of split s is stored to slot s of the workspace p.c_f32 ([splits][M][ldc = N]) instead of being
// added to C with atomics
template <bool kTN, bool kDet = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
               const __grid_constant__ CUtensorMap tmap_c, const GemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* stage_base = smem;                                  // STAGES x (A | B)
    uint8_t* c_stage = smem + STAGES * STAGE_BYTES;              // NT: bf16 C tile, two 64-column halves (SW128)
    uint64_t* bars = reinterpret_cast<uint64_t*>(c_stage + C_STAGE_BYTES);
    uint64_t* full_bar = bars;                // [STAGES] TMA -> MMA
    uint64_t* empty_bar = bars + STAGES;      // [STAGES] MMA -> TMA
    uint64_t* acc_full = bars + 2 * STAGES;   // [2] MMA -> epilogue
    uint64_t* acc_empty = bars + 2 * STAGES + 2;  // [2] epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        rs::prefetch_tmap(&tmap_a);
        rs::prefetch_tmap(&tmap_b);
        if (!kTN) rs::prefetch_tmap(&tmap_c);
        for (int s = 0; s < STAGES; ++s) {
            rs::mbar_init(&full_bar[s], 1);
            rs::mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            rs::mbar_init(&acc_full[s], 1);
            rs::mbar_init(&acc_empty[s], 4);   // one arrival per epilogue warp
        }
        rs::fence_mbar_init();
    }
    if (warp == 1) rs::tmem_alloc<TMEM_COLS>(tmem_slot);
    rs::tc_fence_before();
    __syncthreads();
    rs::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int total_tiles = p.m_tiles * p.n_tiles * p.splits;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (rs::elect_one()) {
            int stage = 0;
            uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
                const int split = tile / (p.m_tiles * p.n_tiles);
                const int mn = tile % (p.m_tiles * p.n_tiles);
                const int m_blk = mn / p.n_tiles, n_blk = mn % p.n_tiles;
                for (int kb = 0; kb < p.k_blocks; ++kb) {
                    rs::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = stage_base + stage * STAGE_BYTES;
                    uint8_t* sb = sa + TILE_A_BYTES;
                    rs::mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
                    if (!kTN) {
                        rs::tma_load_2d(sa, &tmap_a, &full_bar[stage], kb * BK, m_blk * BM);
                        rs::tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * BK, n_blk * BN);
                    } else {
                        const int g = split * p.k_blocks + kb;              // k block over all passes
                        const int seg = g / p.kb_per_seg;
                        if (seg >= p.n_seg) {                                // tail of the last split: nothing left, feed zeros
                            rs::tma_load_2d(sa, &tmap_a, &full_bar[stage], 0, 0x3fffffff);
                            rs::tma_load_2d(sa + TILE_A_BYTES / 2, &tmap_a, &full_bar[stage], 0, 0x3fffffff);
                            rs::tma_load_2d(sb, &tmap_b, &full_bar[stage], 0, 0x3fffffff);
                            rs::tma_load_2d(sb + TILE_B_BYTES / 2, &tmap_b, &full_bar[stage], 0, 0x3fffffff);
                        } else {
                            const int krow = (g - seg * p.kb_per_seg) * BK;
                            const int ac = p.a_col0 + p.a_seg[seg] + m_blk * BM, bc = p.b_col0 + p.b_seg[seg] + n_blk * BN;
                            // MN-major operands: box = 64 columns (128 B) x 64 rows; two boxes cover 128 columns
                            rs::tma_load_2d(sa, &tmap_a, &full_bar[stage], ac, krow + p.a_row_shift);
                            rs::tma_load_2d(sa + TILE_A_BYTES / 2, &tmap_a, &full_bar[stage], ac + 64, krow + p.a_row_shift);
                            rs::tma_load_2d(sb, &tmap_b, &full_bar[stage], bc, krow + p.b_row_shift);
                            rs::tma_load_2d(sb + TILE_B_BYTES / 2, &tmap_b, &full_bar[stage], bc + 64, krow + p.b_row_shift);
                        }
                    }
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        constexpr uint32_t idesc = rs::umma_idesc_bf16(BM, BN, kTN ? 1u : 0u, kTN ? 1u : 0u);
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            rs::mbar_wait(&acc_empty[acc], acc_phase ^ 1);      // epilogue drained this accumulator stage
            rs::tc_fence_after();
            const uint32_t tmem_d = tmem_base + acc * BN;
            for (int kb = 0; kb < p.k_blocks; ++kb) {
                rs::mbar_wait(&full_bar[stage], phase);
                rs::tc_fence_after();
                if (rs::elect_one()) {
                    const uint32_t sa = rs::smem_u32(stage_base + stage * STAGE_BYTES);
                    const uint32_t sb = sa + TILE_A_BYTES;
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) {
                        uint64_t da, db;
                        if (!kTN) {
                            da = rs::umma_desc_k_sw128(sa + k * 32);
                            db = rs::umma_desc_k_sw128(sb + k * 32);
                        } else {
                            da = rs::umma_desc_mn_sw128(sa + k * 2048, TILE_A_BYTES / 2, 1024);
                            db = rs::umma_desc_mn_sw128(sb + k * 2048, TILE_B_BYTES / 2, 1024);
                        }
                        rs::tc_mma_bf16(tmem_d, da, db, idesc, (kb | k) != 0);
                    }
                    rs::tc_commit(&empty_bar[stage]);            // frees the smem stage when the MMAs retire
                    if (kb == p.k_blocks - 1) rs::tc_commit(&acc_full[acc]);
                }
                __syncwarp();
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int q = warp & 3;                      // TMEM lane quadrant this warp may read
        const int row = q * 32 + lane;               // row of the tile owned by this thread
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
            const int mn = tile % (p.m_tiles * p.n_tiles);
            const int m_blk = mn / p.n_tiles, n_blk = mn % p.n_tiles;
            rs::mbar_wait(&acc_full[acc], acc_phase);
            rs::tc_fence_after();
            const uint32_t taddr = tmem_base + acc * BN + (static_cast<uint32_t>(q * 32) << 16);
            if (!kTN && (p.flags & RS_GEMM_OUT_F32)) {
                // fp32 result: each thread writes its own row (small outputs only: decoder heads)
                const long long gm = (long long)m_blk * BM + row;
#pragma unroll
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    uint32_t r[32];
                    rs::tmem_ld_32x32b_x32(taddr + c0, r);
                    rs::tmem_ld_wait();
                    if (gm < p.M) {
                        float* crow = p.c_nt_f32 + gm * p.ldc_nt + n_blk * BN + c0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            float4 v;
                            v.x = __uint_as_float(r[j]); v.y = __uint_as_float(r[j + 1]); v.z = __uint_as_float(r[j + 2]); v.w = __uint_as_float(r[j + 3]);
                            if (p.bias) {
                                const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias + n_blk * BN + c0 + j));
                                v.x += bb.x; v.y += bb.y; v.z += bb.z; v.w += bb.w;
                            }
                            if (p.flags & RS_GEMM_RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
                            *reinterpret_cast<float4*>(crow + j) = v;
                        }
                    }
                }
                rs::tc_fence_before();
                if (lane == 0) rs::mbar_arrive(&acc_empty[acc]);
            } else if (!kTN) {
                // make sure the previous TMA store has finished reading the staging tile
                if (warp == 2 && lane == 0) rs::tma_store_wait_read<0>();
                asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    uint32_t r[32];
                    rs::tmem_ld_32x32b_x32(taddr + c0, r);
                    rs::tmem_ld_wait();
                    uint32_t packed[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float v0 = __uint_as_float(r[2 * j]), v1 = __uint_as_float(r[2 * j + 1]);
                        if (p.bias) {
                            v0 += __ldg(&p.bias[n_blk * BN + c0 + 2 * j]);
                            v1 += __ldg(&p.bias[n_blk * BN + c0 + 2 * j + 1]);
                        }
                        if (p.flags & RS_GEMM_RELU) { v0 = fmaxf(v0, 0.0f); v1 = fmaxf(v1, 0.0f); }
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(v0, v1);
                        packed[j] = *reinterpret_cast<uint32_t*>(&h2);
                    }
                    // staging layout: two [128 rows x 128 B] halves (64 columns each), 128-byte swizzle
                    uint8_t* half = c_stage + (c0 / 64) * (BM * 128);
                    const int chunk0 = (c0 % 64) / 8;          // first 16-byte chunk of these 32 columns
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int chunk = (chunk0 + j) ^ (row & 7);
                        *reinterpret_cast<uint4*>(half + row * 128 + chunk * 16) =
                            make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
                    }
                }
                rs::tc_fence_before();
                if (lane == 0) rs::mbar_arrive(&acc_empty[acc]);     // accumulator stage may be overwritten
                rs::fence_proxy_async();
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (warp == 2 && lane == 0) {
                    rs::tma_store_2d(&tmap_c, c_stage, n_blk * BN, m_blk * BM);
                    rs::tma_store_2d(&tmap_c, c_stage + BM * 128, n_blk * BN + 64, m_blk * BM);
                    rs::tma_store_commit();
                }
            } else {
                const int gm = m_blk * BM + row;
                float* cbase = kDet ? p.c_f32 + static_cast<long long>(tile / (p.m_tiles * p.n_tiles)) * p.M * p.ldc : p.c_f32;
#pragma unroll
                for (int c0 = 0; c0 < BN; c0 += 32) {
                    uint32_t r[32];
                    rs::tmem_ld_32x32b_x32(taddr + c0, r);
                    rs::tmem_ld_wait();
                    if (gm < p.M) {
                        float* crow = cbase + static_cast<long long>(gm) * p.ldc + n_blk * BN + c0;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            if (n_blk * BN + c0 + j >= p.N) continue;
                            if (kDet) crow[j] = __uint_as_float(r[j]);
                            else atomicAdd(crow + j, __uint_as_float(r[j]));
                        }
                    }
                }
                rs::tc_fence_before();
                if (lane == 0) rs::mbar_arrive(&acc_empty[acc]);
            }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (!kTN && !(p.flags & RS_GEMM_OUT_F32) && warp == 2 && lane == 0) rs::tma_store_wait<0>();
    }

    rs::tc_fence_before();
    __syncthreads();
    if (warp == 1) rs::tmem_dealloc<TMEM_COLS>(tmem_base);
}

constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + C_STAGE_BYTES + 256;
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

// C[M,N] (bf16, leading dimension ldc) = A[M,K] (lda) . B[N,K]^T (ldb) + bias.  K % 64 == 0, N % 128 == 0.
extern "C" int rs_gemm_bf16_nt(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc,
                               const float* bias, int64_t M, int N, int K, int flags, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (M == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(A && B && C && M >= 0 && N > 0 && K > 0, "rs_gemm_bf16_nt: bad arguments");
    RS_REQUIRE(K % BK == 0 && N % BN == 0, "rs_gemm_bf16_nt: need K %% 64 == 0 and N %% 128 == 0 (got N=%d K=%d)", N, K);
    RS_REQUIRE(lda % 8 == 0 && ldb % 8 == 0 && ldc % 8 == 0, "rs_gemm_bf16_nt: leading dimensions must be multiples of 8");
    const bool out_f32 = flags & RS_GEMM_OUT_F32;
    RS_REQUIRE(!out_f32 || ((reinterpret_cast<uintptr_t>(C) & 15) == 0 && ldc % 4 == 0 && (reinterpret_cast<uintptr_t>(bias) & 15) == 0),
               "rs_gemm_bf16_nt: with RS_GEMM_OUT_F32, C and bias are accessed as float4 and must be 16-byte aligned");
    RS_REQUIRE(M < (1ll << 31), "rs_gemm_bf16_nt: M too large");
    CUtensorMap ta, tb, tc;
    if (rs::make_tmap_2d(&ta, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, K, M, lda * 2, BK, BM, CU_TENSOR_MAP_SWIZZLE_128B)) return 2;
    if (rs::make_tmap_2d(&tb, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, K, N, ldb * 2, BK, BN, CU_TENSOR_MAP_SWIZZLE_128B)) return 2;
    if (out_f32) tc = ta;      // unused by the kernel in this mode
    else if (rs::make_tmap_2d(&tc, C, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, N, M, ldc * 2, 64, BM, CU_TENSOR_MAP_SWIZZLE_128B)) return 2;
    GemmParams p = {};
    p.M = (int)M; p.N = N; p.K = K;
    p.m_tiles = (int)((M + BM - 1) / BM);
    p.n_tiles = N / BN;
    p.k_blocks = K / BK;
    p.splits = 1;
    p.bias = bias; p.flags = flags; p.c_nt_f32 = static_cast<float*>(C); p.ldc_nt = ldc;
    RS_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    long long tiles = (long long)p.m_tiles * p.n_tiles;
    int grid = (int)(tiles < num_sms() ? tiles : num_sms());
    gemm_tc_kernel<false><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(ta, tb, tc, p);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

// C[M,N] (fp32, ldc) += sum over passes s < n_seg of  A[rows, a_col0 + a_seg[s] : +M]^T . B[rows, b_col0 + b_seg[s] : +N],
// pairing row r + a_row_shift of A with row r + b_row_shift of B for r in [0, rows).  Rows outside the matrices read as
// zero.  M % 128 == 0, N % 128 == 0.
static int tn_launch(const void* A, int64_t lda, int64_t a_rows, int a_col0, int a_row_shift, const void* B, int64_t ldb,
                     int64_t b_rows, int b_col0, int b_row_shift, int n_seg, const int* a_seg, const int* b_seg, float* C,
                     int64_t ldc, int M, int N, int64_t rows, cudaStream_t stream) {
    RS_REQUIRE(A && B && C && M > 0 && N > 0 && rows >= 0, "rs_gemm_bf16_tn_acc: bad arguments");
    RS_REQUIRE(M % BM == 0 && N % BN == 0, "rs_gemm_bf16_tn_acc: need M %% 128 == 0 and N %% 128 == 0 (got %d x %d)", M, N);
    RS_REQUIRE(lda % 8 == 0 && ldb % 8 == 0, "rs_gemm_bf16_tn_acc: leading dimensions must be multiples of 8");
    RS_REQUIRE(rows < (1ll << 31) && a_rows < (1ll << 31) && b_rows < (1ll << 31), "rs_gemm_bf16_tn_acc: too many rows");
    RS_REQUIRE(n_seg >= 1 && n_seg <= 8, "rs_gemm_bf16_tn_acc: 1 <= passes <= 8");
    if (rows == 0) return 0;
    CUtensorMap ta, tb;
    // clamp the visible rows so that nothing past the last valid pair is read (TMA returns zero out of bounds)
    const int64_t a_vis = (rows + a_row_shift < a_rows) ? rows + a_row_shift : a_rows;
    const int64_t b_vis = (rows + b_row_shift < b_rows) ? rows + b_row_shift : b_rows;
    RS_REQUIRE(a_vis > 0 && b_vis > 0, "rs_gemm_bf16_tn_acc: empty operand after the row shift");
    if (rs::make_tmap_2d(&ta, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, lda, a_vis, lda * 2, 64, BK, CU_TENSOR_MAP_SWIZZLE_128B)) return 2;
    if (rs::make_tmap_2d(&tb, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, ldb, b_vis, ldb * 2, 64, BK, CU_TENSOR_MAP_SWIZZLE_128B)) return 2;
    GemmParams p = {};
    p.M = M; p.N = N; p.K = (int)rows;
    p.m_tiles = M / BM;
    p.n_tiles = N / BN;
    const int out_tiles = p.m_tiles * p.n_tiles;
    const long long kb_per_seg = (rows + BK - 1) / BK;
    const long long kblocks_total = kb_per_seg * n_seg;
    const bool det = rs::deterministic();
    int splits = (det ? rs::kDetSplitSms : num_sms()) / out_tiles;
    if (splits < 1) splits = 1;
    if (splits > kblocks_total) splits = (int)kblocks_total;
    const long long kb_per_split = (kblocks_total + splits - 1) / splits;
    splits = (int)((kblocks_total + kb_per_split - 1) / kb_per_split);
    p.splits = splits;
    p.k_blocks = (int)kb_per_split;
    p.k_rows_per_split = (int)(kb_per_split * BK);
    p.n_seg = n_seg; p.kb_per_seg = (int)kb_per_seg;
    for (int s = 0; s < n_seg; ++s) { p.a_seg[s] = a_seg ? a_seg[s] : 0; p.b_seg[s] = b_seg ? b_seg[s] : 0; }
    p.a_row_shift = a_row_shift; p.b_row_shift = b_row_shift;
    p.a_col0 = a_col0; p.b_col0 = b_col0;
    p.c_f32 = C; p.ldc = ldc;
    const int total = out_tiles * splits;
    int grid = total < num_sms() ? total : num_sms();
    if (det && splits > 1) {
        rs::StreamScratch ws(stream);
        RS_CUDA_OK(ws.alloc(sizeof(float) * (size_t)splits * M * N));
        p.c_f32 = ws.as<float>(); p.ldc = N;
        RS_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        gemm_tc_kernel<true, true><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(ta, tb, ta, p);
        rs::count_launch();
        RS_CUDA_OK(cudaGetLastError());
        const rs::SlotSum<float> job = {ws.as<float>(), C, ldc, M, N};
        return rs::slot_sum(&job, 1, splits, (long long)M * N, true, stream);
    }
    RS_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    gemm_tc_kernel<true><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(ta, tb, ta, p);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_gemm_bf16_tn_acc(const void* A, int64_t lda, int64_t a_rows, int a_col0, int a_row_shift,
                                   const void* B, int64_t ldb, int64_t b_rows, int b_col0, int b_row_shift, float* C,
                                   int64_t ldc, int M, int N, int64_t rows, void* stream_) {
    if (rs::check_device_sm100()) return 3;
    return tn_launch(A, lda, a_rows, a_col0, a_row_shift, B, ldb, b_rows, b_col0, b_row_shift, 1, nullptr, nullptr, C, ldc, M, N,
                     rows, static_cast<cudaStream_t>(stream_));
}

extern "C" int rs_gemm_bf16_tn_seg_acc(const void* A, int64_t lda, int64_t a_rows, int a_col0, int a_row_shift, const void* B,
                                       int64_t ldb, int64_t b_rows, int b_col0, int b_row_shift, int n_seg, const int* a_seg,
                                       const int* b_seg, float* C, int64_t ldc, int M, int N, int64_t rows, void* stream_) {
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(a_seg && b_seg, "rs_gemm_bf16_tn_seg_acc: null pointer");
    return tn_launch(A, lda, a_rows, a_col0, a_row_shift, B, ldb, b_rows, b_col0, b_row_shift, n_seg, a_seg, b_seg, C, ldc, M, N,
                     rows, static_cast<cudaStream_t>(stream_));
}
