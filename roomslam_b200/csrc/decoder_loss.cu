// Decoder head post-processing and the fused multi-task loss (SURVEY.md 8(a) rows a6, a7; upstream spec
// README.md:117-125; loss weights D9 after src/benchmark/train.py:433-437).  Always fp32.
//
// The decoder trunk / head GEMMs run in rs_sgemm (fp32 mode) or the tcgen05 GEMM (bf16 mode); this file holds
// the element-wise pieces around them:
//   heads_split : raw [B, N*(C+6)] -> class_logits [B,N,C], positions [B,N,2], sizes = softplus(raw)+1e-4 [B,N,2],
//                 orientations [B,N], validity_logits [B,N]      (column order class | pos | size | orient | valid)
//   heads_merge : the reverse for gradients (softplus' = sigmoid(raw))
//   loss fwd    : one thread per (trace, slot): CE over C classes, L1 position / size / orientation masked by
//                 `valid`, BCE-with-logits on validity; block-reduced sums -> 6 losses; the un-normalised
//                 per-element gradients are produced in the same pass
//   loss bwd    : scales those gradients by the incoming d(loss) coefficients (device-side, no host sync)
#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

constexpr int kMaxClasses = 16;

__global__ void heads_split_kernel(const float* __restrict__ raw, int B, int N, int C, float* __restrict__ cls,
                                   float* __restrict__ pos, float* __restrict__ size, float* __restrict__ orient,
                                   float* __restrict__ valid) {
    const int NH = N * (C + 6);
    const long long n = (long long)B * NH;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int c = e % NH;
        const long long b = e / NH;
        const float v = raw[e];
        if (c < N * C) cls[b * N * C + c] = v;
        else if (c < N * C + 2 * N) pos[b * 2 * N + (c - N * C)] = v;
        else if (c < N * C + 4 * N) {
            const float sp = (v > 20.0f) ? v : log1pf(expf(v));   // torch softplus, threshold 20
            size[b * 2 * N + (c - N * C - 2 * N)] = sp + 1e-4f;
        } else if (c < N * C + 5 * N) orient[b * N + (c - N * C - 4 * N)] = v;
        else valid[b * N + (c - N * C - 5 * N)] = v;
    }
}

__global__ void heads_merge_kernel(const float* __restrict__ raw, int B, int N, int C, const float* __restrict__ d_cls,
                                   const float* __restrict__ d_pos, const float* __restrict__ d_size,
                                   const float* __restrict__ d_orient, const float* __restrict__ d_valid,
                                   float* __restrict__ d_raw) {
    const int NH = N * (C + 6);
    const long long n = (long long)B * NH;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int c = e % NH;
        const long long b = e / NH;
        float g = 0.0f;
        if (c < N * C) g = d_cls ? d_cls[b * N * C + c] : 0.0f;
        else if (c < N * C + 2 * N) g = d_pos ? d_pos[b * 2 * N + (c - N * C)] : 0.0f;
        else if (c < N * C + 4 * N) {
            if (d_size) {
                const float v = raw[e];
                const float sg = (v > 20.0f) ? 1.0f : 1.0f / (1.0f + expf(-v));
                g = d_size[b * 2 * N + (c - N * C - 2 * N)] * sg;
            }
        } else if (c < N * C + 5 * N) g = d_orient ? d_orient[b * N + (c - N * C - 4 * N)] : 0.0f;
        else g = d_valid ? d_valid[b * N + (c - N * C - 5 * N)] : 0.0f;
        d_raw[e] = g;
    }
}

// dx may alias dy (both decoders call these in place).  Each element is read and written by the same thread in one
// iteration, and no other element is read, so __restrict__ allows no reordering that changes the result.
__global__ void relu_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ y, float* __restrict__ dx,
                                long long n) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        dx[e] = y[e] > 0.0f ? dy[e] : 0.0f;
}

__global__ void relu_bwd_bf16_kernel(const __nv_bfloat16* __restrict__ dy, const __nv_bfloat16* __restrict__ y,
                                     __nv_bfloat16* __restrict__ dx, long long n) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x)
        dx[e] = __bfloat162float(y[e]) > 0.0f ? dy[e] : __float2bfloat16(0.0f);
}

__device__ __forceinline__ float sgn(float d) { return (d > 0.0f) - (d < 0.0f); }

// sums: [0] n_valid, [1] ce, [2] |dpos|, [3] |dsize|, [4] |dorient|, [5] bce   (double accumulators)
// kDet: block b stores its six sums to sums + 6 b (summed in block order by rs::slot_sum)
template <bool kDet>
__global__ void __launch_bounds__(256)
loss_fwd_kernel(const float* __restrict__ cls, const float* __restrict__ pos, const float* __restrict__ size,
                const float* __restrict__ orient, const float* __restrict__ vlogit, const long long* __restrict__ t_cls,
                const float* __restrict__ t_pos, const float* __restrict__ t_size, const float* __restrict__ t_orient,
                const float* __restrict__ t_valid, long long slots, int C, double* __restrict__ sums,
                float* __restrict__ g_cls, float* __restrict__ g_pos, float* __restrict__ g_size,
                float* __restrict__ g_orient, float* __restrict__ g_valid) {
    float s[6] = {0, 0, 0, 0, 0, 0};
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < slots; e += (long long)gridDim.x * blockDim.x) {
        const float v = t_valid[e];
        s[0] += v;
        // cross entropy over C classes
        float lg[kMaxClasses];
        float mx = -INFINITY;
        for (int c = 0; c < C; ++c) { lg[c] = cls[e * C + c]; mx = fmaxf(mx, lg[c]); }
        float se = 0.0f;
        for (int c = 0; c < C; ++c) se += expf(lg[c] - mx);
        const float lse = mx + logf(se);
        const int tc = (int)t_cls[e];
        s[1] += v * (lse - lg[tc]);
        for (int c = 0; c < C; ++c) g_cls[e * C + c] = v * (expf(lg[c] - lse) - (c == tc ? 1.0f : 0.0f));
        // L1 terms
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float dp = pos[e * 2 + k] - t_pos[e * 2 + k];
            s[2] += v * fabsf(dp);
            g_pos[e * 2 + k] = v * sgn(dp);
            const float ds = size[e * 2 + k] - t_size[e * 2 + k];
            s[3] += v * fabsf(ds);
            g_size[e * 2 + k] = v * sgn(ds);
        }
        const float dor = orient[e] - t_orient[e];
        s[4] += v * fabsf(dor);
        g_orient[e] = v * sgn(dor);
        // BCE with logits (over every slot)
        const float l = vlogit[e];
        s[5] += fmaxf(l, 0.0f) - l * v + log1pf(expf(-fabsf(l)));
        g_valid[e] = 1.0f / (1.0f + expf(-l)) - v;
    }
    __shared__ float red[6][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const float w = rs::warp_sum(s[k]);
        if (lane == 0) red[k][warp] = w;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += (double)red[threadIdx.x][w];
        if (kDet) sums[blockIdx.x * 6 + threadIdx.x] = t;
        else atomicAdd(&sums[threadIdx.x], t);
    }
}

// losses: [total, class, position, size, orientation, validity]
__global__ void loss_finalize_kernel(const double* __restrict__ sums, long long slots, float* __restrict__ losses,
                                     float w_cls, float w_pos, float w_size, float w_orient, float w_valid) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const double nv = sums[0] < 1.0 ? 1.0 : sums[0];
        const double lc = sums[1] / nv, lp = sums[2] / (2.0 * nv), ls = sums[3] / (2.0 * nv), lo = sums[4] / nv;
        const double lv = slots > 0 ? sums[5] / (double)slots : 0.0;
        losses[1] = (float)lc; losses[2] = (float)lp; losses[3] = (float)ls; losses[4] = (float)lo; losses[5] = (float)lv;
        losses[0] = (float)(w_cls * lc + w_pos * lp + w_size * ls + w_orient * lo + w_valid * lv);
    }
}

// d_pred = unnormalised_grad * coef with coef built from the incoming d(losses) (d_losses[6], device memory)
__global__ void loss_bwd_kernel(const double* __restrict__ sums, const float* __restrict__ d_losses, long long slots,
                                int C, float w_cls, float w_pos, float w_size, float w_orient, float w_valid,
                                const float* __restrict__ g_cls, const float* __restrict__ g_pos,
                                const float* __restrict__ g_size, const float* __restrict__ g_orient,
                                const float* __restrict__ g_valid, float* __restrict__ d_cls, float* __restrict__ d_pos,
                                float* __restrict__ d_size, float* __restrict__ d_orient, float* __restrict__ d_valid) {
    const float nv = (float)(sums[0] < 1.0 ? 1.0 : sums[0]);
    const float gt = d_losses[0];
    const float k_cls = (gt * w_cls + d_losses[1]) / nv;
    const float k_pos = (gt * w_pos + d_losses[2]) / (2.0f * nv);
    const float k_size = (gt * w_size + d_losses[3]) / (2.0f * nv);
    const float k_orient = (gt * w_orient + d_losses[4]) / nv;
    const float k_valid = (gt * w_valid + d_losses[5]) / (float)slots;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < slots; e += (long long)gridDim.x * blockDim.x) {
        for (int c = 0; c < C; ++c) d_cls[e * C + c] = g_cls[e * C + c] * k_cls;
        d_pos[e * 2] = g_pos[e * 2] * k_pos;
        d_pos[e * 2 + 1] = g_pos[e * 2 + 1] * k_pos;
        d_size[e * 2] = g_size[e * 2] * k_size;
        d_size[e * 2 + 1] = g_size[e * 2 + 1] * k_size;
        d_orient[e] = g_orient[e] * k_orient;
        d_valid[e] = g_valid[e] * k_valid;
    }
}

int blocks_for(long long n, int per = 256, int cap = 148 * 8) {
    long long b = (n + per - 1) / per;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (int)b;
}

}  // namespace

extern "C" int rs_heads_split_f32(const float* raw, int B, int N, int C, float* cls, float* pos, float* size,
                                  float* orient, float* valid, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(raw && cls && pos && size && orient && valid, "rs_heads_split_f32: null pointer");
    heads_split_kernel<<<blocks_for((long long)B * N * (C + 6)), 256, 0, stream>>>(raw, B, N, C, cls, pos, size, orient, valid);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_heads_merge_bwd_f32(const float* raw, int B, int N, int C, const float* d_cls, const float* d_pos,
                                      const float* d_size, const float* d_orient, const float* d_valid, float* d_raw,
                                      void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(raw && d_raw, "rs_heads_merge_bwd_f32: null pointer");
    heads_merge_kernel<<<blocks_for((long long)B * N * (C + 6)), 256, 0, stream>>>(raw, B, N, C, d_cls, d_pos, d_size,
                                                                                  d_orient, d_valid, d_raw);
                                                                                  rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_relu_bwd_f32(const float* dy, const float* y, float* dx, int64_t n, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (n == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(dy && y && dx, "rs_relu_bwd_f32: null pointer");
    relu_bwd_kernel<<<blocks_for(n), 256, 0, stream>>>(dy, y, dx, n);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_relu_bwd_bf16(const void* dy, const void* y, void* dx, int64_t n, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (n == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(dy && y && dx, "rs_relu_bwd_bf16: null pointer");
    relu_bwd_bf16_kernel<<<blocks_for(n), 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(dy), static_cast<const __nv_bfloat16*>(y),
                                                            static_cast<__nv_bfloat16*>(dx), n);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_loss_fwd_f32(const float* cls, const float* pos, const float* size, const float* orient,
                               const float* vlogit, const int64_t* t_cls, const float* t_pos, const float* t_size,
                               const float* t_orient, const float* t_valid, int B, int N, int C, const float* weights5,
                               double* sums6, float* losses6, float* g_cls, float* g_pos, float* g_size, float* g_orient,
                               float* g_valid, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(cls && pos && size && orient && vlogit && t_cls && t_pos && t_size && t_orient && t_valid && weights5 &&
               sums6 && losses6 && g_cls && g_pos && g_size && g_orient && g_valid, "rs_loss_fwd_f32: null pointer");
    RS_REQUIRE(C >= 1 && C <= kMaxClasses, "rs_loss_fwd_f32: 1 <= num_classes <= %d", kMaxClasses);
    const long long slots = (long long)B * N;
    RS_CUDA_OK(cudaMemsetAsync(sums6, 0, 6 * sizeof(double), stream));
    rs::StreamScratch ws(stream);
    if (slots > 0 && rs::deterministic()) {
        const int blocks = blocks_for(slots);
        RS_CUDA_OK(ws.alloc(sizeof(double) * 6 * blocks));
        loss_fwd_kernel<true><<<blocks, 256, 0, stream>>>(cls, pos, size, orient, vlogit, reinterpret_cast<const long long*>(t_cls),
                                                          t_pos, t_size, t_orient, t_valid, slots, C, ws.as<double>(), g_cls,
                                                          g_pos, g_size, g_orient, g_valid);
        rs::count_launch();
        const rs::SlotSum<double> job = {ws.as<double>(), sums6, 6, 1, 6};
        if (int rc = rs::slot_sum(&job, 1, blocks, 6, false, stream)) return rc;
    } else if (slots > 0) {
        loss_fwd_kernel<false><<<blocks_for(slots), 256, 0, stream>>>(cls, pos, size, orient, vlogit,
                                                              reinterpret_cast<const long long*>(t_cls), t_pos, t_size,
                                                              t_orient, t_valid, slots, C, sums6, g_cls, g_pos, g_size,
                                                              g_orient, g_valid);
                                                              rs::count_launch();
    }
    loss_finalize_kernel<<<1, 32, 0, stream>>>(sums6, slots, losses6, weights5[0], weights5[1], weights5[2], weights5[3],
                                               weights5[4]);
                                               rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_loss_bwd_f32(const double* sums6, const float* d_losses6, int B, int N, int C, const float* weights5,
                               const float* g_cls, const float* g_pos, const float* g_size, const float* g_orient,
                               const float* g_valid, float* d_cls, float* d_pos, float* d_size, float* d_orient,
                               float* d_valid, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(sums6 && d_losses6 && weights5 && g_cls && g_pos && g_size && g_orient && g_valid && d_cls && d_pos &&
               d_size && d_orient && d_valid, "rs_loss_bwd_f32: null pointer");
    const long long slots = (long long)B * N;
    if (slots == 0) return 0;
    loss_bwd_kernel<<<blocks_for(slots), 256, 0, stream>>>(sums6, d_losses6, slots, C, weights5[0], weights5[1],
                                                           weights5[2], weights5[3], weights5[4], g_cls, g_pos, g_size,
                                                           g_orient, g_valid, d_cls, d_pos, d_size, d_orient, d_valid);
                                                           rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
