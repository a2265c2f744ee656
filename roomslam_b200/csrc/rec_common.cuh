// Device helpers shared by the bf16 recurrence kernels (rec_pair.cu: H = 128, rec_wide.cu: H = 256; a CTA pair per tile on
// tcgen05 cta_group::2): fast tanh, bf16 / fp16 pack and unpack of 16-byte pieces, the layer-0 input columns.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace rs {

__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float2 bf2_to_f2(uint32_t v) {
    __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&v);
    return __bfloat1622float2(h);
}
__device__ __forceinline__ uint32_t f2_to_bf2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
    float2 a = bf2_to_f2(v.x), b = bf2_to_f2(v.y), c = bf2_to_f2(v.z), d = bf2_to_f2(v.w);
    f[0] = a.x; f[1] = a.y; f[2] = b.x; f[3] = b.y; f[4] = c.x; f[5] = c.y; f[6] = d.x; f[7] = d.y;
}
__device__ __forceinline__ uint4 pack8(const float* f) {
    return make_uint4(f2_to_bf2(f[0], f[1]), f2_to_bf2(f[2], f[3]), f2_to_bf2(f[4], f[5]), f2_to_bf2(f[6], f[7]));
}
// saved gates are private to the two recurrence kernels: fp16 (r, z, n live in [-1, 1], where fp16 is 8x finer than bf16)
__device__ __forceinline__ uint32_t f2_to_h2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float round_h(float a) { return __half2float(__float2half_rn(a)); }   // a saved gate's value
__device__ __forceinline__ uint4 pack8h(const float* f) {
    return make_uint4(f2_to_h2(f[0], f[1]), f2_to_h2(f[2], f[3]), f2_to_h2(f[4], f[5]), f2_to_h2(f[6], f[7]));
}
__device__ __forceinline__ void unpack8h(const uint4& v, float* f) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        f[2 * i] = t.x; f[2 * i + 1] = t.y;
    }
}
__device__ __forceinline__ uint4 ldg16(const uint8_t* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void stg16(uint8_t* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }

// Layer-0 input columns: W_ih x + b rides on the recurrence MMA as extra K = 16 steps of hi / lo split operands.  The column
// map (A operand = the trace row, built here; B operand = the weight image, built by pack_w.cu for H = 128 and by
// functional_bf16.py for H = 256):
//   input i < 2 : columns 3 i + k        k = 0, 1, 2:  x (hi, lo, hi)  against  W_ih (hi, hi, lo)
//   bias        : columns 6, 7                         (1, 1)          against  b (hi, lo)
//   input i >= 2: columns 8 + 3 (i - 2) + k            as inputs 0 and 1
//   every other column of the input K steps is zero.
// Inputs 0, 1 and the bias fill the first 16-byte chunk exactly as the 2-input layout always did; I inputs take 3 I + 2
// columns, so x_steps(I) = ceil((3 I + 2) / 16) K steps: 1 up to 4 inputs, 2 up to 10, 3 up to 15, 4 for 16.
constexpr int kMaxXInputs = 16;
__host__ __device__ constexpr int x_col(int i, int k) { return i < 2 ? 3 * i + k : 8 + 3 * (i - 2) + k; }
__host__ __device__ constexpr int x_col_input(int c) { return c < 6 ? c / 3 : (c < 8 ? -1 : 2 + (c - 8) / 3); }  // -1: bias
__host__ __device__ constexpr int x_col_part(int c) { return c < 6 ? c % 3 : (c < 8 ? c - 6 : (c - 8) % 3); }
__host__ __device__ constexpr int x_steps(int I) { return (3 * I + 2 + 15) / 16; }
// 16-byte chunks per row of the input columns a recurrence kernel writes: 1 for I <= 2 (the second chunk of the one K step
// stays zero), else every chunk of the x_steps(I) K steps
__host__ __device__ constexpr int x_chunks(int I) { return I <= 2 ? 1 : 2 * x_steps(I); }
constexpr bool x_map_ok() {
    for (int i = 0; i < kMaxXInputs; ++i)
        for (int k = 0; k < 3; ++k)
            if (x_col_input(x_col(i, k)) != i || x_col_part(x_col(i, k)) != k || x_col(i, k) >= 16 * x_steps(i + 1)) return false;
    return x_col_input(6) == -1 && x_col_input(7) == -1 && x_steps(2) == 1 && x_steps(kMaxXInputs) == 4;
}
static_assert(x_map_ok(), "layer-0 input column map");

// Chunk 0 of the input columns of one trace row: per input c < 2 the triple (hi, lo, hi) with hi = bf16(x_c),
// lo = bf16(x_c - hi), then (1, 1).  Everything a row with at most 2 inputs needs.
__device__ __forceinline__ uint4 pack_x(const float* xp, int I) {
    float c[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (xp) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            if (i < I) {
                const float v = __ldg(xp + i);
                const float hi = __bfloat162float(__float2bfloat16_rn(v));
                c[3 * i] = hi; c[3 * i + 1] = v - hi; c[3 * i + 2] = hi;
            }
        }
    }
    c[6] = 1.0f; c[7] = 1.0f;
    return pack8(c);
}
// Chunk ch (any of the x_chunks(I)) of the input columns of one trace row; xp = NULL (pad row): the bias columns only.
__device__ __forceinline__ uint4 pack_x_chunk(const float* xp, int I, int ch) {
    uint32_t w[4];
#pragma unroll
    for (int jp = 0; jp < 4; ++jp) {                   // two columns at a time keeps the live set small
        float v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = x_col_input(ch * 8 + 2 * jp + e), k = x_col_part(ch * 8 + 2 * jp + e);
            v[e] = i < 0 ? 1.0f : 0.0f;
            if (xp && i >= 0 && i < I) {
                const float x = __ldg(xp + i);
                const float hi = __bfloat162float(__float2bfloat16_rn(x));
                v[e] = k == 1 ? x - hi : hi;
            }
        }
        w[jp] = f2_to_bf2(v[0], v[1]);
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}



#ifdef __CUDACC__
// rec_pair.cu: the CTA-pair kernels behind rs_rec_fwd_bf16 / rs_rec_bwd_bf16 (same operands and results as rec_bf16.cu)
int rec_fwd_nt(int B);                      // tiles in flight per pair of the forward kernel (1 or 2)
int rec_fwd_pair(const float* x, int I, const void* P, const void* X, const void* Wih, const void* Whh, const float* b_hn, void* out,
                 void* gates, float* h_n, const int* lengths, const void* drop_bits, const float* drop_scale, void* out_drop, int split,
                 int B, int T, int nt, int pf_dist, cudaStream_t stream);
// x != NULL: layer 0 (I <= 2, unsplit, gates NULL) recomputes r, z, n; xpack is its [tiles][T][128][8] bf16 workspace
int rec_bwd_pair(const void* d_out, const float* d_h_n, const void* gates, const float* x, int I, void* xpack, const void* out,
                 const void* WhhT, const void* Whh, int whh_chunks, const float* b_hn, void* dG, const int* lengths,
                 const void* drop_bits, const float* drop_scale, int split, int B, int T, int pf_dist, cudaStream_t stream);
#endif

}  // namespace rs
