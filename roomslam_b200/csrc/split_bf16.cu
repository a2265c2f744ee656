// fp32 -> split-bf16 operands for fp32-accurate GEMMs on the bf16 tensor cores ("bf16x6").
//   x = hi + mid + lo + O(2^-25 |x|),  hi = bf16(x), mid = bf16(x - hi), lo = bf16(x - hi - mid)     (3 x 8 mantissa bits)
//   a . b ~= hi hi + hi mid + mid hi + mid mid + hi lo + lo hi           (dropped terms are O(2^-24) relative)
// The six products become ONE tensor-core GEMM over a six times longer K by concatenating along K:
//   A operand rows: [lo | hi | mid | mid | hi | hi]      B operand rows: [hi | lo | mid | hi | mid | hi]
// (each sixth padded with zero columns to kpad).  bf16 x bf16 products are exact in the fp32 accumulator; the tensor
// core TRUNCATES the running sum at every K = 16 step (measured: a biased ~3e-8 relative per step), so the small
// products come first and only the last sixth (hi.hi) accumulates at full magnitude: fp32-grade results (~3e-7
// against fp64, like the CUDA-core fp32 GEMM) at tensor-core speed.  A two-term
// split (three products, ~1e-6) was measured first: accurate enough for the smooth part of the model, but behind the
// ReLU of the 3 M head pre-activations a 1e-6 perturbation flips dozens of units and moves the head weight gradients by
// 7e-3 -- outside the 1e-4 parity bar.  Used for the time-parallel GEMMs of the BiLSTM model (SURVEY.md 8(f) rank 2).
#include <cuda_bf16.h>

#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 a, __nv_bfloat16 b) {
    __nv_bfloat162 t; t.x = a; t.y = b;
    return *reinterpret_cast<uint32_t*>(&t);
}

__global__ void split_bf16x6_kernel(const float* __restrict__ x, long long ld, long long rows, int cols, int kpad, int role_b,
                                    __nv_bfloat16* __restrict__ out, long long ld_out) {
    const int groups = kpad / 8;                          // 8 columns (16 bytes of bf16) per thread
    const long long total = rows * groups;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long r = e / groups;
        const int c0 = (int)(e % groups) * 8;
        float v[8];
        if (c0 + 8 <= cols && (ld & 3) == 0) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(x + r * ld + c0));
            const float4 b = __ldg(reinterpret_cast<const float4*>(x + r * ld + c0 + 4));
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = (c0 + j < cols) ? __ldg(x + r * ld + c0 + j) : 0.0f;
        }
        uint32_t hi[4], mid[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            __nv_bfloat16 h[2], m[2], l[2];
#pragma unroll
            for (int t = 0; t < 2; ++t) {
                const float a = v[2 * j + t];
                h[t] = __float2bfloat16_rn(a);
                const float r1 = a - __bfloat162float(h[t]);               // exact
                m[t] = __float2bfloat16_rn(r1);
                l[t] = __float2bfloat16_rn(r1 - __bfloat162float(m[t]));    // exact difference, rounded once
            }
            hi[j] = pack2(h[0], h[1]); mid[j] = pack2(m[0], m[1]); lo[j] = pack2(l[0], l[1]);
        }
        const uint4 H = make_uint4(hi[0], hi[1], hi[2], hi[3]), Mi = make_uint4(mid[0], mid[1], mid[2], mid[3]),
                    Lo = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        __nv_bfloat16* o = out + r * ld_out + c0;
        // smallest products first:  lo.hi  hi.lo  mid.mid  mid.hi  hi.mid  hi.hi
        // A role: lo hi mid mid hi hi      B role: hi lo mid hi mid hi
        *reinterpret_cast<uint4*>(o) = role_b ? H : Lo;
        *reinterpret_cast<uint4*>(o + kpad) = role_b ? Lo : H;
        *reinterpret_cast<uint4*>(o + 2 * kpad) = Mi;
        *reinterpret_cast<uint4*>(o + 3 * kpad) = role_b ? H : Mi;
        *reinterpret_cast<uint4*>(o + 4 * kpad) = role_b ? Mi : H;
        *reinterpret_cast<uint4*>(o + 5 * kpad) = H;
    }
}

}  // namespace

extern "C" int rs_split_bf16x6(const float* x, int64_t ld, int64_t rows, int cols, int kpad, int role_b, void* out, int64_t ld_out,
                               void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (rows == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(x && out && rows >= 0 && cols >= 1, "rs_split_bf16x6: bad arguments");
    RS_REQUIRE(kpad % 8 == 0 && kpad >= cols && ld_out >= 6 * (int64_t)kpad && ld_out % 8 == 0,
               "rs_split_bf16x6: kpad must be a multiple of 8 >= cols and ld_out >= 6 * kpad (multiple of 8)");
    RS_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15) == 0, "rs_split_bf16x6: output must be 16-byte aligned");
    RS_REQUIRE((ld & 3) || (reinterpret_cast<uintptr_t>(x) & 15) == 0,
               "rs_split_bf16x6: with ld %% 4 == 0 the rows are read as float4, so x must be 16-byte aligned");
    const long long total = rows * (kpad / 8);
    long long blocks = (total + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    split_bf16x6_kernel<<<(int)blocks, 256, 0, stream>>>(x, ld, rows, cols, kpad, role_b, static_cast<__nv_bfloat16*>(out), ld_out);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
