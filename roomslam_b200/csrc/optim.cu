// Fused optimizer step over the flat parameter buffer: global-norm gradient clipping (upstream train loop:
// src/benchmark/train.py:220 clip_grad_norm_(1.0)) + AdamW (train.py:440-444).  Part of the timed training step.
#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

// kDet: block b stores its sum to out[b] (summed in block order by rs::slot_sum) instead of adding it to out[0]
template <bool kDet>
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, long long n, float scale, double* out) {
    float s = 0.0f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float v = g[i] * scale;
        s = fmaf(v, v, s);
    }
    __shared__ float red[8];
    s = rs::warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += (double)red[w];
        if (kDet) out[blockIdx.x] = t;
        else atomicAdd(out, t);
    }
}

__global__ void __launch_bounds__(256)
adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
             float lr, float beta1, float beta2, float eps, float wd, float bc1, float bc2, float grad_scale,
             float max_norm, const double* __restrict__ sumsq) {
    float clip = 1.0f;
    if (max_norm > 0.0f) {
        const float norm = sqrtf((float)(*sumsq));
        clip = fminf(1.0f, max_norm / (norm + 1e-6f));
    }
    const float gs = grad_scale * clip;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i] * gs;
        float pi = p[i];
        pi *= (1.0f - lr * wd);
        const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
        const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
        p[i] = pi - (lr / bc1) * mi / denom;
    }
}

}  // namespace

extern "C" int rs_adamw_step_f32(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                                 float beta2, float eps, float weight_decay, int step, float grad_scale, float max_norm,
                                 double* sumsq_scratch, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (n == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(p && g && m && v && sumsq_scratch && n >= 0 && step >= 1, "rs_adamw_step_f32: bad arguments");
    int blocks = (int)((n + 255) / 256);
    if (blocks > 148 * 4) blocks = 148 * 4;
    rs::StreamScratch ws(stream);
    if (max_norm > 0.0f && rs::deterministic()) {
        RS_CUDA_OK(ws.alloc(sizeof(double) * blocks));
        sumsq_kernel<true><<<blocks, 256, 0, stream>>>(g, n, grad_scale, ws.as<double>());
        rs::count_launch();
        const rs::SlotSum<double> job = {ws.as<double>(), sumsq_scratch, 1, 1, 1};
        if (int rc = rs::slot_sum(&job, 1, blocks, 1, false, stream)) return rc;
    } else if (max_norm > 0.0f) {
        RS_CUDA_OK(cudaMemsetAsync(sumsq_scratch, 0, sizeof(double), stream));
        sumsq_kernel<false><<<blocks, 256, 0, stream>>>(g, n, grad_scale, sumsq_scratch);
        rs::count_launch();
    }
    const float bc1 = 1.0f - powf(beta1, (float)step), bc2 = 1.0f - powf(beta2, (float)step);
    adamw_kernel<<<blocks, 256, 0, stream>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2, grad_scale,
                                             max_norm, sumsq_scratch);
                                             rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
