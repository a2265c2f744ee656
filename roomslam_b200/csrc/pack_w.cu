// One launch builds every bf16 operand image a bidirectional GRU layer needs from its fp32 master weights
// (torch.nn.GRU's weight_ih / weight_hh / bias_ih / bias_hh and their _reverse twins, rnn.py:1290-1297 gate order r|z|n):
//   whh_img   [2][16 (+2 s)][3H][8]  B operand of the recurrence forward (r, z rows scaled by 1/2: sigma(a) = tanh(a/2)/2 + 1/2);
//                                  layer 0 (I <= 16): chunks 16 .. 15 + 2 s, s = x_steps(I) = the input columns: per gate row
//                                  (w_hi, w_hi, w_lo) per input and (b_hi, b_lo) at the columns of rec_common.cuh's map
//   b_hn      [2][H]               bias of the hidden side of the n gate
//   bias_x    [2][3H]              b_ih (+ b_hh for r, z), scaled like the rows: folded into the projection / the input chunk
//   wt_proj   [6H/128][I/64][8][128][8]   W_ih (scaled) as B pieces of the projection GEMM            (deeper layers)
//   whhT_img  [2][3H/8][H][8]      W_hh^T: B operand of the BPTT matvec dh = dGh . W_hh
//   wt_dgrad  [I/128][6H/64][8][128][8]   W_ih^T as B pieces of the data-gradient GEMM dX = dG . W_ih (deeper layers)
//   wih_img   [2][I/8][3H][8]      W_ih (scaled) as a RESIDENT B operand: projection fused into the recurrence (rec_pair.cu);
//                                  whh_img then carries the bias in its input chunk (b_hi, b_lo against a constant (1, 1))
// With split = 1 every weight operand is a PAIR of bf16 images, hi = bf16(w) and lo = bf16(w - hi), stacked along K (the
// kernels run their K loops over both against the same activations): the weights then enter the tensor core with
// ~16 mantissa bits.  Rounding the weights to bf16 alone moves the fp32 oracle's gradients by 2.3 % at batch 32 -- a
// coherent perturbation that does not average out over the batch -- so small batches run with split weights.
// It replaces ~30 torch cat / stack / permute / cast launches per layer and step (VERDICT r1, weak item 7).
#include "common.cuh"
#include "rec_common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

using namespace rs;

struct PackWParams {
    const float* w_ih[2];
    const float* w_hh[2];
    const float* b_ih[2];
    const float* b_hh[2];
    int H, I, nck, split;                      // split: every weight as a bf16 pair hi + lo (see rs_gru_pack_weights_bf16)
    uint4* whh_img; float* b_hn; float* bias_x; uint4* wt_proj; uint4* whhT_img; uint4* wt_dgrad; uint4* wih_img;
    int layer0;                                // whh_img's input chunks hold the input weights and the bias (else: the bias only)
    long long n_a, n_e, n_d, n_f, n_g, n_b;    // pieces per region
};

// part 0: the value itself (rounded to bf16 by the caller's pack8); part 1: what that rounding lost
__device__ __forceinline__ float hi_lo(float w, int part) {
    return part == 0 ? w : w - __bfloat162float(__float2bfloat16_rn(w));
}

__device__ __forceinline__ float bias_x_of(const PackWParams& p, int d, int row) {
    const float s = row < 2 * p.H ? 0.5f : 1.0f;
    const float b = __ldg(p.b_ih[d] + row) + (row < 2 * p.H ? __ldg(p.b_hh[d] + row) : 0.0f);
    return b * s;
}

__global__ void pack_w_kernel(const PackWParams p) {
    const int H = p.H, I = p.I, H3 = 3 * p.H;
    const long long total = p.n_a + p.n_e + p.n_d + p.n_f + p.n_g + p.n_b;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        float v[8];
        long long e = i;
        if (e < p.n_a) {                                   // ---- whh_img
            const int row = e % H3;
            const int c = (e / H3) % p.nck;
            const int d = e / ((long long)H3 * p.nck);
            const float s = row < 2 * H ? 0.5f : 1.0f;
            const int nh = (H / 8) * (1 + p.split);         // hidden chunks: hi parts, then (split) lo parts
            if (c < nh) {
                const int part = c / (H / 8), cc = c % (H / 8);
                const float4* src = reinterpret_cast<const float4*>(p.w_hh[d] + (long long)row * H + cc * 8);
                const float4 a = __ldg(src), b = __ldg(src + 1);
                const float w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = hi_lo(w[j] * s, part);
            } else {
#pragma unroll
                for (int j = 0; j < 8; ++j) v[j] = 0.0f;
                // input chunks (rec_common.cuh's column map): layer-0 input weights (hi, hi, lo) and the bias (hi, lo);
                // with the fused projection the bias only
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = (c - nh) * 8 + j, i = x_col_input(col), k = x_col_part(col);
                    if (i < 0) {
                        const float b = bias_x_of(p, d, row);
                        const float bhi = __bfloat162float(__float2bfloat16_rn(b));
                        v[j] = k == 0 ? bhi : b - bhi;
                    } else if (p.layer0 && i < I) {
                        const float w = __ldg(p.w_ih[d] + (long long)row * I + i) * s;
                        const float hi = __bfloat162float(__float2bfloat16_rn(w));
                        v[j] = k == 2 ? w - hi : hi;
                    }
                }
            }
            p.whh_img[e] = pack8(v);
            continue;
        }
        e -= p.n_a;
        if (e < p.n_e) {                                   // ---- whhT_img [2][3H/8][H][8]
            const int nc = (H3 / 8) * (1 + p.split);
            const int u = e % H;
            const int c = (e / H) % nc;
            const int d = e / ((long long)H * nc);
            const int part = c / (H3 / 8), cc = c % (H3 / 8);
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = hi_lo(__ldg(p.w_hh[d] + (long long)(cc * 8 + j) * H + u), part);
            p.whhT_img[e] = pack8(v);
            continue;
        }
        e -= p.n_e;
        if (e < p.n_d) {                                   // ---- wt_proj [6H/128][I/64][8][128][8]
            const int r = e & 127;
            const int c8 = (e >> 7) & 7;
            const int nk = (I / 64) * (1 + p.split);
            const int kk = (e >> 10) % nk;
            const int n = (e >> 10) / nk;
            const int part = kk / (I / 64), k = kk % (I / 64);
            const int grow = n * 128 + r;
            const int d = grow / H3, row = grow % H3;
            const float s = row < 2 * H ? 0.5f : 1.0f;
            const float4* src = reinterpret_cast<const float4*>(p.w_ih[d] + (long long)row * I + k * 64 + c8 * 8);
            const float4 a = __ldg(src), b = __ldg(src + 1);
            const float w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = hi_lo(w[j] * s, part);
            p.wt_proj[e] = pack8(v);
            continue;
        }
        e -= p.n_d;
        if (e < p.n_f) {                                   // ---- wt_dgrad [I/128][6H/64][8][128][8]
            const int r = e & 127;
            const int c8 = (e >> 7) & 7;
            const int nk = (2 * H3 / 64) * (1 + p.split);
            const int kk = (e >> 10) % nk;
            const int n = (e >> 10) / nk;
            const int part = kk / (2 * H3 / 64), k = kk % (2 * H3 / 64);
            const int col = n * 128 + r;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int grow = k * 64 + c8 * 8 + j;
                v[j] = hi_lo(__ldg(p.w_ih[grow / H3] + (long long)(grow % H3) * I + col), part);
            }
            p.wt_dgrad[e] = pack8(v);
            continue;
        }
        e -= p.n_f;
        if (e < p.n_g) {                                   // ---- wih_img [2][I/8][3H][8]: W_ih as a resident B operand (fused projection)
            const int row = e % H3;
            const int c = (e / H3) % (I / 8);
            const int d = e / ((long long)H3 * (I / 8));
            const float s = row < 2 * H ? 0.5f : 1.0f;
            const float4* src = reinterpret_cast<const float4*>(p.w_ih[d] + (long long)row * I + c * 8);
            const float4 a = __ldg(src), b = __ldg(src + 1);
            v[0] = a.x * s; v[1] = a.y * s; v[2] = a.z * s; v[3] = a.w * s; v[4] = b.x * s; v[5] = b.y * s; v[6] = b.z * s; v[7] = b.w * s;
            p.wih_img[e] = pack8(v);
            continue;
        }
        e -= p.n_g;
        if (e < 2 * H) {                                   // ---- b_hn
            const int d = e / H, u = e % H;
            p.b_hn[e] = __ldg(p.b_hh[d] + 2 * H + u);
        } else {                                           // ---- bias_x
            const long long f = e - 2 * H;
            p.bias_x[f] = bias_x_of(p, f / H3, f % H3);
        }
    }
}

}  // namespace

extern "C" int rs_gru_pack_weights_bf16(const float* const* w, int H, int I, int split, void* whh_img, float* b_hn, float* bias_x,
                                        void* wt_proj, void* whhT_img, void* wt_dgrad, void* wih_img, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    RS_REQUIRE(w && whh_img && b_hn && bias_x && whhT_img, "rs_gru_pack_weights_bf16: bad arguments");
    RS_REQUIRE(H % 128 == 0 && H >= 128, "rs_gru_pack_weights_bf16: H must be a multiple of 128");
    const bool layer0 = (I <= rs::kMaxXInputs);            // deeper layers take a multiple of 128: unambiguous
    RS_REQUIRE(layer0 ? (I >= 1 && !wt_dgrad && !wt_proj && !wih_img) : (I % 128 == 0 && (wt_proj || wih_img)),
               "rs_gru_pack_weights_bf16: layer 0 takes 1-16 input columns (no projection images); deeper layers a multiple of 128 "
               "and wt_proj (projection GEMM) or wih_img (projection fused into the recurrence)");
    RS_REQUIRE(!(wih_img && split), "rs_gru_pack_weights_bf16: the fused projection takes plain (unsplit) weights");
    PackWParams p = {};
    for (int d = 0; d < 2; ++d) {
        p.w_ih[d] = w[4 * d]; p.w_hh[d] = w[4 * d + 1]; p.b_ih[d] = w[4 * d + 2]; p.b_hh[d] = w[4 * d + 3];
        RS_REQUIRE(p.w_ih[d] && p.w_hh[d] && p.b_ih[d] && p.b_hh[d], "rs_gru_pack_weights_bf16: null weight pointer");
    }
    split = split ? 1 : 0;
    p.layer0 = layer0 ? 1 : 0;
    p.H = H; p.I = I; p.split = split; p.nck = (H / 8) * (1 + split) + (layer0 ? 2 * rs::x_steps(I) : (wih_img ? 2 : 0));
    p.whh_img = static_cast<uint4*>(whh_img); p.b_hn = b_hn; p.bias_x = bias_x;
    p.wt_proj = static_cast<uint4*>(wt_proj); p.whhT_img = static_cast<uint4*>(whhT_img); p.wt_dgrad = static_cast<uint4*>(wt_dgrad);
    p.wih_img = static_cast<uint4*>(wih_img);
    p.n_a = 2LL * p.nck * 3 * H;
    p.n_e = 2LL * (3 * H / 8) * H * (1 + split);
    p.n_d = wt_proj ? 6LL * H * I / 8 * (1 + split) : 0;
    p.n_g = wih_img ? 6LL * H * I / 8 : 0;
    p.n_f = wt_dgrad ? 6LL * H * I / 8 * (1 + split) : 0;
    p.n_b = 2LL * H + 2LL * 3 * H;
    const long long total = p.n_a + p.n_e + p.n_d + p.n_f + p.n_g + p.n_b;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 148 * 8) blocks = 148 * 8;
    pack_w_kernel<<<blocks, 256, 0, stream>>>(p);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
