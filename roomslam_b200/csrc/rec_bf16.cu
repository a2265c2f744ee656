// C-ABI entry points of the persistent tensor-core GRU recurrence for the bf16 mode at H = 128 (SURVEY.md 8(a) rows a3, a4)
// and the layer-0 input packer.  The kernels themselves are in rec_pair.cu (a CTA pair per 128-trace tile, tcgen05
// cta_group::2); round 1's one-CTA-per-tile kernels lived here and were retired once the pair kernels beat them at every
// batch size (DESIGN.md 4.2 has the A/B numbers).
#include <cuda_fp16.h>
#include <stdlib.h>

#include "common.cuh"
#include "rec_common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

using namespace rs;

constexpr int H = 128;

// x (B, T, I <= 16) fp32 -> tile-major bf16 with 16 columns (the rest zero), pad rows and pad traces zero:
// the B operand that carries the layer-0 input into the fused weight-gradient pass.
__global__ void pack_x_tm_kernel(const float* __restrict__ x, int B, int T, int I, uint4* __restrict__ out, long long n_rows) {
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n_rows; e += (long long)gridDim.x * blockDim.x) {
        const int row = e & 127;                       // e = ((tile * (T+2) + t') * 128 + row)
        const long long bt = e >> 7;
        const int tp = bt % (T + 2);
        const long long b = (bt / (T + 2)) * 128 + row;
        float c[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) c[i] = 0.0f;
        if (b < B && tp >= 1 && tp <= T) {
            const float* xp = x + (b * T + (tp - 1)) * I;
#pragma unroll
            for (int i = 0; i < 16; ++i)
                if (i < I) c[i] = __ldg(xp + i);
        }
        const long long blk = bt * 256;                // 2 chunks x 128 rows of uint4 per block
        out[blk + row] = pack8(c);
        out[blk + 128 + row] = pack8(c + 8);
    }
}

int pf_dist_env(const char* name, int dflt) {
    const char* e = getenv(name);
    int v = e ? atoi(e) : dflt;
    if (v < 0) v = 0;
    if (v > 64) v = 64;
    return v;
}

}  // namespace

extern "C" int rs_rec_fwd_bf16(const float* x, int I, const void* P, int64_t p_cols, const void* X, const void* Wih, const void* Whh,
                               const float* b_hn, void* out, void* gates, float* h_n, const int* lengths,
                               const void* drop_bits, const float* drop_scale, void* out_drop, int split, int B, int T,
                               void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE((x != nullptr) + (P != nullptr) + (X != nullptr) == 1,
               "rs_rec_fwd_bf16: exactly one of x (layer 0), P (deeper layers, projected) and X (deeper layers, projection fused) must be given");
    RS_REQUIRE(!X || (Wih && !split), "rs_rec_fwd_bf16: the fused projection needs Wih and plain (unsplit) weights");
    RS_REQUIRE(!x || (I >= 1 && I <= rs::kMaxXInputs), "rs_rec_fwd_bf16: the MMA-fused input projection takes 1 to %d input columns (got %d)",
               rs::kMaxXInputs, I);
    RS_REQUIRE(!P || p_cols == 6 * H, "rs_rec_fwd_bf16: P must have 6H = %d columns", 6 * H);
    RS_REQUIRE(Whh && b_hn && out && h_n && B >= 0 && T >= 0, "rs_rec_fwd_bf16: bad arguments");
    if (T == 0) {
        RS_CUDA_OK(cudaMemsetAsync(h_n, 0, sizeof(float) * 2 * (size_t)B * H, stream));
        return 0;
    }
    RS_REQUIRE((drop_bits != nullptr) == (out_drop != nullptr) && (!drop_bits || drop_scale),
               "rs_rec_fwd_bf16: drop_bits, drop_scale and out_drop go together");
    return rs::rec_fwd_pair(x, I, P, X, Wih, Whh, b_hn, out, gates, h_n, lengths, drop_bits, drop_scale, out_drop, split, B, T,
                            rs::rec_fwd_nt(B), pf_dist_env("RS_PF_DIST_FWD", 1), stream);
}

extern "C" int rs_rec_bwd_bf16(const void* d_out, const float* d_h_n, const void* gates, const void* out, const void* WhhT,
                               const void* Whh, int whh_chunks, const float* b_hn, void* dG, const int* lengths,
                               const void* drop_bits, const float* drop_scale, int split, int B, int T, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0 || T == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(gates && out && WhhT && Whh && b_hn && dG && B >= 0 && T >= 0, "rs_rec_bwd_bf16: bad arguments");
    RS_REQUIRE(whh_chunks >= 16 * (split ? 2 : 1), "rs_rec_bwd_bf16: Whh is the forward image (16 hidden chunks, twice with split)");
    RS_REQUIRE(!drop_bits || drop_scale, "rs_rec_bwd_bf16: drop_bits needs drop_scale");
    // L2 prefetch of the gate / d_out blocks RS_PF_DIST_BWD steps ahead (default 1; issued by the thread that also issues the
    // h_{t-1} tile copies).  Measured once single-thread issue had become cheap (elect.sync): BPTT at 8192 traces 3.14 / 3.30 ms
    // per layer without, 2.94 / 3.21 with distance 1, 3.11 / 3.53 with 2, 3.43 / 3.94 with 4 (evicted before use); at 1024
    // traces 1.16 / 1.18 -> 1.13 / 1.14 ms.
    return rs::rec_bwd_pair(d_out, d_h_n, gates, out, WhhT, Whh, whh_chunks, b_hn, dG, lengths, drop_bits, drop_scale, split, B, T,
                            pf_dist_env("RS_PF_DIST_BWD", 1), stream);
}

extern "C" int rs_pack_x_tm(const float* x, int B, int T, int I, void* out, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(x && out && B >= 0 && T >= 0 && I >= 1 && I <= 16, "rs_pack_x_tm: bad arguments");
    const long long n_rows = (long long)((B + 127) / 128) * (T + 2) * 128;
    if (n_rows == 0) return 0;
    long long blocks = (n_rows + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pack_x_tm_kernel<<<(int)blocks, 256, 0, stream>>>(x, B, T, I, static_cast<uint4*>(out), n_rows);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
