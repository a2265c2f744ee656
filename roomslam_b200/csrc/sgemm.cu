// fp32 CUDA-core GEMM with generic strides, used by the fp32 (1e-4 parity) mode for the time-parallel
// projections, weight gradients and the decoder MLP.  The bf16 mode uses the tcgen05 kernel (gemm_tc.cu).
//   C[m,n] = act( sum_k A(m,k) * B(k,n) + bias[n] ) (+ C[m,n] when accumulate)
// A(m,k) = A[m*a_sm + k*a_sk], B(k,n) = B[k*b_sk + n*b_sn], C row-major with leading dimension ldc.
// 64x64x16 tiles, 256 threads, 4x4 register micro-tiles; optional split-K over gridDim.z with fp32 atomics (deterministic
// mode: per-split partials in a workspace, summed in split order by rs::slot_sum).
#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

constexpr int BM = 64, BN = 64, BK = 16;

// kDet: split z stores its partial (bias added by split 0) to C + z * M * N, a dense [M][N] slot (ldc = N)
template <bool kDet>
__global__ void __launch_bounds__(256)
sgemm_kernel(const float* __restrict__ A, long long a_sm, long long a_sk, const float* __restrict__ B, long long b_sk,
             long long b_sn, float* __restrict__ C, long long ldc, const float* __restrict__ bias, int M, int N, int K,
             int k_per_split, int flags) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const int k_begin = blockIdx.z * k_per_split;
    const int k_end = min(K, k_begin + k_per_split);
    const bool a_k_contig = (a_sk == 1), b_n_contig = (b_sn == 1);

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

    for (int k0 = k_begin; k0 < k_end; k0 += BK) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int idx = tid + e * 256;
            int m, k;
            if (a_k_contig) { m = idx >> 4; k = idx & 15; } else { k = idx >> 6; m = idx & 63; }
            const int gm = m0 + m, gk = k0 + k;
            As[k][m] = (gm < M && gk < k_end) ? A[gm * a_sm + gk * a_sk] : 0.0f;
            int n, kb;
            if (b_n_contig) { kb = idx >> 6; n = idx & 63; } else { n = idx >> 4; kb = idx & 15; }
            const int gn = n0 + n, gkb = k0 + kb;
            Bs[kb][n] = (gn < N && gkb < k_end) ? B[gkb * b_sk + gn * b_sn] : 0.0f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }

    const bool accumulate = flags & RS_GEMM_ACCUMULATE, relu = flags & RS_GEMM_RELU, split = gridDim.z > 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            float v = acc[i][j];
            float* c = &C[gm * ldc + gn];
            if (kDet) {
                if (bias && blockIdx.z == 0) v += bias[gn];
                C[(long long)blockIdx.z * M * N + gm * ldc + gn] = v;
            } else if (split) {
                if (bias && blockIdx.z == 0) v += bias[gn];
                atomicAdd(c, v);  // C was zeroed (or holds the value to accumulate onto) before the launch
            } else {
                if (bias) v += bias[gn];
                if (accumulate) v += *c;
                if (relu) v = fmaxf(v, 0.0f);
                *c = v;
            }
        }
    }
}

// kDet: slab y stores its sums to out + y * N instead
template <bool kDet>
__global__ void colsum_kernel(const float* __restrict__ A, long long lda, int M, int N, int rows_per_block,
                              float* __restrict__ out) {
    // block = 32 columns x 8 row-lanes over a slab of rows; slabs are combined with fp32 atomics
    __shared__ float part[8][33];
    const int col = blockIdx.x * 32 + threadIdx.x;
    const int m_begin = blockIdx.y * rows_per_block, m_end = min(M, m_begin + rows_per_block);
    float s = 0.0f;
    if (col < N)
        for (int m = m_begin + threadIdx.y; m < m_end; m += 8) s += A[m * lda + col];
    part[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && col < N) {
        float t = 0.0f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += part[i][threadIdx.x];
        if (kDet) out[(long long)blockIdx.y * N + col] = t;
        else atomicAdd(&out[col], t);
    }
}

}  // namespace

extern "C" int rs_sgemm(const float* A, int64_t a_sm, int64_t a_sk, const float* B, int64_t b_sk, int64_t b_sn, float* C,
                        int64_t ldc, const float* bias, int M, int N, int K, int flags, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (M == 0 || N == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(A && B && C && M >= 0 && N >= 0 && K >= 0, "rs_sgemm: bad arguments");
    dim3 grid((N + BN - 1) / BN, (M + BM - 1) / BM, 1);
    int k_per_split = K;
    const bool relu = flags & RS_GEMM_RELU;
    const long long tiles = (long long)grid.x * grid.y;
    if (!relu && K >= 4096 && tiles < 296) {  // long reductions with few output tiles (weight gradients)
        int splits = (int)((296 + tiles - 1) / tiles);
        if (splits > K / 512) splits = K / 512;
        if (splits > 1) {
            k_per_split = ((K + splits - 1) / splits + BK - 1) / BK * BK;
            grid.z = (K + k_per_split - 1) / k_per_split;
        }
    }
    if (grid.z > 1 && rs::deterministic()) {
        rs::StreamScratch ws(stream);
        RS_CUDA_OK(ws.alloc(sizeof(float) * (size_t)grid.z * M * N));
        sgemm_kernel<true><<<grid, 256, 0, stream>>>(A, a_sm, a_sk, B, b_sk, b_sn, ws.as<float>(), N, bias, M, N, K, k_per_split,
                                                     flags);
        rs::count_launch();
        RS_CUDA_OK(cudaGetLastError());
        const rs::SlotSum<float> job = {ws.as<float>(), C, ldc, M, N};
        return rs::slot_sum(&job, 1, (int)grid.z, (long long)M * N, flags & RS_GEMM_ACCUMULATE, stream);
    }
    if (grid.z > 1 && !(flags & RS_GEMM_ACCUMULATE)) {
        if (ldc == N) {
            RS_CUDA_OK(cudaMemsetAsync(C, 0, sizeof(float) * (size_t)M * N, stream));
        } else {
            RS_CUDA_OK(cudaMemset2DAsync(C, sizeof(float) * ldc, 0, sizeof(float) * N, M, stream));
        }
    }
    sgemm_kernel<false><<<grid, 256, 0, stream>>>(A, a_sm, a_sk, B, b_sk, b_sn, C, ldc, bias, M, N, K, k_per_split, flags);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_colsum_f32(const float* A, int64_t lda, int M, int N, float* out, int accumulate, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE((A || M == 0) && out && M >= 0 && N > 0, "rs_colsum_f32: bad arguments");
    if (!accumulate) RS_CUDA_OK(cudaMemsetAsync(out, 0, sizeof(float) * N, stream));
    if (M == 0) return 0;        // the column sums of an empty matrix are zero
    int slabs = (M + 2047) / 2048;
    if (slabs > 128) slabs = 128;
    const int rows_per_block = (M + slabs - 1) / slabs;
    if (slabs > 1 && rs::deterministic()) {
        rs::StreamScratch ws(stream);
        RS_CUDA_OK(ws.alloc(sizeof(float) * (size_t)slabs * N));
        colsum_kernel<true><<<dim3((N + 31) / 32, slabs), dim3(32, 8), 0, stream>>>(A, lda, M, N, rows_per_block, ws.as<float>());
        rs::count_launch();
        RS_CUDA_OK(cudaGetLastError());
        const rs::SlotSum<float> job = {ws.as<float>(), out, N, 1, N};
        return rs::slot_sum(&job, 1, slabs, N, true, stream);     // onto the zeroed or accumulated output
    }
    colsum_kernel<false><<<dim3((N + 31) / 32, slabs), dim3(32, 8), 0, stream>>>(A, lda, M, N, rows_per_block, out);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
