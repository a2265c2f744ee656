// fp32 LSTM recurrence, forward and backward-through-time, for the model the upstream repository trains
// (SURVEY.md 8(f) rank 2; src/benchmark/model.py:16-23 nn.LSTM(d_model, d_model/2, 2 layers, bidirectional)).
// Generic in the hidden size H (multiple of 32, <= 256).  Tolerance 1e-4 against torch.nn.LSTM on the CPU.
//
// Gate equations (torch.nn.LSTM, weight rows ordered i | f | g | o):
//   i = sigma(P_i + Wh_i h)  f = sigma(P_f + Wh_f h)  g = tanh(P_g + Wh_g h)  o = sigma(P_o + Wh_o h)
//   c' = f * c + i * g        h' = o * tanh(c')                  P = W_ih x + b_ih + b_hh   (time-parallel GEMM)
//
// One CTA owns Bt = S*R traces of ONE direction for all T steps.  blockDim = (H, S): thread (u, y) owns hidden unit u
// of traces y*R .. y*R+R-1 and keeps their cell state in registers.  W_hh^T (H x 4H fp32) stays resident in shared
// memory when it fits (H <= 64: 64 KB), otherwise it streams from L2; since H <= 64 always takes the register-resident
// kernels further down, these run with W streamed (S = 2 at H <= 128, S = 1 above; R = 1, or 4 when B > 296).  h is
// double-buffered in shared memory: one __syncthreads() per step.  Sequence buffers use the (rows, row0, ld) addressing
// of roomslam_b200.h.
#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

struct SeqF {
    float* p;
    long long ld, trace_rows, row0;
    __device__ __forceinline__ float* at(long long b, long long t) const { return p + ((b * trace_rows + row0 + t) * ld); }
};

__device__ __forceinline__ float sigm(float x) { return 1.0f / (1.0f + expf(-x)); }
// (ex2.approx-based __expf forms were measured: their ~2e-6 relative error grows to 6e-4 in the weight gradients of a
// 300-trace batch, outside the 1e-4 parity tolerance; the accurate expf / tanhf stay.)
__device__ __forceinline__ float sigm_q(float x) { return __fdividef(1.0f, 1.0f + expf(-x)); }
__device__ __forceinline__ float tanh_q(float x) { return tanhf(x); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
constexpr int PF_STEPS = 8;                 // L2 prefetch distance of the register-resident kernels, in time steps

template <int R, bool WSMEM>
__global__ void __launch_bounds__(256)
lstm_fwd_f32_kernel(SeqF P, const float* __restrict__ w_hh_t, SeqF out, float* __restrict__ saved, int B, int T, int H) {
    extern __shared__ __align__(16) float lsm[];
    const int u = threadIdx.x, y = threadIdx.y, S = blockDim.y, Bt = S * R;
    const int dir = blockIdx.y, H4 = 4 * H;
    float* Ws = lsm;                                   // [H][4H]
    float* hs = lsm + (WSMEM ? H * H4 : 0);            // [2][Bt][H]
    const float* Wg = w_hh_t + (size_t)dir * H * H4;
    const int tid = y * blockDim.x + u, nthr = blockDim.x * blockDim.y;
    if (WSMEM) for (int e = tid; e < H * H4; e += nthr) Ws[e] = Wg[e];
    for (int e = tid; e < 2 * Bt * H; e += nthr) hs[e] = 0.0f;
    __syncthreads();

    const long long b0 = (long long)blockIdx.x * Bt + y * R;
    float c[R];
#pragma unroll
    for (int rr = 0; rr < R; ++rr) c[rr] = 0.0f;
    int cur = 0;
    for (int step = 0; step < T; ++step) {
        const int t = dir ? (T - 1 - step) : step;
        float acc[R][4];
#pragma unroll
        for (int rr = 0; rr < R; ++rr)
#pragma unroll
            for (int g = 0; g < 4; ++g) acc[rr][g] = 0.0f;
        // issue this step's projection loads before the matvec so their latency hides behind it
        float px[R][4];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const long long b = b0 + rr;
            if (b < B) {
                const float* pp = P.at(b, t) + dir * H4 + u;
#pragma unroll
                for (int g = 0; g < 4; ++g) px[rr][g] = __ldg(pp + g * H);
            } else {
#pragma unroll
                for (int g = 0; g < 4; ++g) px[rr][g] = 0.0f;
            }
        }
        const float* hcur = hs + (size_t)cur * Bt * H + (size_t)y * R * H;
#pragma unroll 2
        for (int k = 0; k < H; k += 4) {
            float w[4][4];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                for (int g = 0; g < 4; ++g)
                    w[kk][g] = WSMEM ? Ws[(k + kk) * H4 + g * H + u] : __ldg(&Wg[(size_t)(k + kk) * H4 + g * H + u]);
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                const float4 hv = *reinterpret_cast<const float4*>(hcur + rr * H + k);
                const float h4[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
                for (int kk = 0; kk < 4; ++kk)
#pragma unroll
                    for (int g = 0; g < 4; ++g) acc[rr][g] = fmaf(w[kk][g], h4[kk], acc[rr][g]);
            }
        }
        float* hnxt = hs + (size_t)(cur ^ 1) * Bt * H + (size_t)y * R * H;
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const long long b = b0 + rr;
            if (b < B) {
                const float gi = sigm(px[rr][0] + acc[rr][0]);
                const float gf = sigm(px[rr][1] + acc[rr][1]);
                const float gg = tanhf(px[rr][2] + acc[rr][2]);
                const float go = sigm(px[rr][3] + acc[rr][3]);
                c[rr] = gf * c[rr] + gi * gg;
                const float hnew = go * tanhf(c[rr]);
                hnxt[rr * H + u] = hnew;
                out.at(b, t)[dir * H + u] = hnew;
                if (saved) {
                    float* sp = saved + ((((size_t)dir * B + b) * T + t) * 5) * H + u;
                    sp[0] = gi; sp[H] = gf; sp[2 * H] = gg; sp[3 * H] = go; sp[4 * H] = c[rr];
                }
            }
        }
        __syncthreads();
        cur ^= 1;
    }
}

// Backward through time: dG[b, t, dir*4H + {i,f,g,o}] = gradient w.r.t. the gate pre-activations (the same tensor
// feeds dW_ih, dW_hh, the biases and dX); the carries dh_{t-1} = dG . W_hh and dc_{t-1} = dc * f stay on chip.
template <int R, bool WSMEM>
__global__ void __launch_bounds__(256)
lstm_bwd_f32_kernel(SeqF d_out, const float* __restrict__ saved, const float* __restrict__ w_hh, SeqF dG, int B, int T, int H) {
    extern __shared__ __align__(16) float lsm[];
    const int u = threadIdx.x, y = threadIdx.y, S = blockDim.y, Bt = S * R;
    const int dir = blockIdx.y, H4 = 4 * H;
    float* Ws = lsm;                                   // [4H][H] (the original row-major layout)
    float* dgs = lsm + (WSMEM ? H * H4 : 0);           // [Bt][4H]
    const float* Wg = w_hh + (size_t)dir * H4 * H;
    const int tid = y * blockDim.x + u, nthr = blockDim.x * blockDim.y;
    if (WSMEM) for (int e = tid; e < H * H4; e += nthr) Ws[e] = Wg[e];
    const long long b0 = (long long)blockIdx.x * Bt + y * R;
    float dh[R], dc[R];
#pragma unroll
    for (int rr = 0; rr < R; ++rr) { dh[rr] = 0.0f; dc[rr] = 0.0f; }
    __syncthreads();

    for (int step = T - 1; step >= 0; --step) {
        const int t = dir ? (T - 1 - step) : step;
        const int t_prev = dir ? (t + 1) : (t - 1);
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const long long b = b0 + rr;
            float g_i = 0.0f, g_f = 0.0f, g_g = 0.0f, g_o = 0.0f;
            if (b < B) {
                const float d = dh[rr] + d_out.at(b, t)[dir * H + u];
                const float* sp = saved + ((((size_t)dir * B + b) * T + t) * 5) * H + u;
                const float gi = sp[0], gf = sp[H], gg = sp[2 * H], go = sp[3 * H], cc = sp[4 * H];
                const float cprev = (step == 0) ? 0.0f : saved[((((size_t)dir * B + b) * T + t_prev) * 5 + 4) * H + u];
                const float tc = tanhf(cc);
                const float dcell = dc[rr] + d * go * (1.0f - tc * tc);
                g_o = d * tc * go * (1.0f - go);
                g_i = dcell * gg * gi * (1.0f - gi);
                g_f = dcell * cprev * gf * (1.0f - gf);
                g_g = dcell * gi * (1.0f - gg * gg);
                dc[rr] = dcell * gf;
                float* gp = dG.at(b, t) + dir * H4 + u;
                gp[0] = g_i; gp[H] = g_f; gp[2 * H] = g_g; gp[3 * H] = g_o;
            }
            float* ds = dgs + (size_t)(y * R + rr) * H4;
            ds[u] = g_i; ds[H + u] = g_f; ds[2 * H + u] = g_g; ds[3 * H + u] = g_o;
        }
        __syncthreads();
        float acc[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) acc[rr] = 0.0f;
        const float* dsy = dgs + (size_t)y * R * H4;
#pragma unroll 2
        for (int j = 0; j < H4; j += 4) {
            float w[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) w[jj] = WSMEM ? Ws[(j + jj) * H + u] : __ldg(&Wg[(size_t)(j + jj) * H + u]);
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                const float4 gv = *reinterpret_cast<const float4*>(dsy + rr * H4 + j);
                acc[rr] = fmaf(w[0], gv.x, acc[rr]);
                acc[rr] = fmaf(w[1], gv.y, acc[rr]);
                acc[rr] = fmaf(w[2], gv.z, acc[rr]);
                acc[rr] = fmaf(w[3], gv.w, acc[rr]);
            }
        }
#pragma unroll
        for (int rr = 0; rr < R; ++rr) dh[rr] = acc[rr];
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Register-resident variant for H <= 64 (the trained configuration: d_model 128 -> H = 64).  The serial chain of
// T = 3000 steps is latency bound, and in the kernels above every FMA costs a shared-memory load of W.  Here the
// CTA has one thread per GATE ROW (4H threads); thread j keeps row j of W_hh (H floats) in registers for the whole
// sequence, h_{t-1} of the CTA's R traces is broadcast from shared memory (one LDS.128 feeds 4 FMAs x R traces), and
// the cell update runs on one thread per (trace, unit).  Two __syncthreads() per step.
template <int HH, int R>
__global__ void __launch_bounds__(4 * HH)
lstm_reg_fwd_kernel(SeqF P, const float* __restrict__ w_hh, SeqF out, float* __restrict__ saved, int B, int T) {
    constexpr int H4 = 4 * HH, CPT = (R * HH + H4 - 1) / H4, NACC = (R <= 2) ? 4 : 1;
    __shared__ __align__(16) float h_s[R * HH];
    __shared__ float g_s[R * H4];
    const int j = threadIdx.x, dir = blockIdx.y, gate = j / HH;
    const long long b0 = (long long)blockIdx.x * R;
    float w[HH];
    {
        const float* wr = w_hh + ((size_t)dir * H4 + j) * HH;
#pragma unroll
        for (int k = 0; k < HH; ++k) w[k] = wr[k];
    }
    float c[CPT];
#pragma unroll
    for (int m = 0; m < CPT; ++m) c[m] = 0.0f;
    for (int e = j; e < R * HH; e += H4) h_s[e] = 0.0f;
    float px_next[R];                       // the projection is fetched one step ahead: its latency is off the serial chain
#pragma unroll
    for (int r = 0; r < R; ++r) px_next[r] = (b0 + r < B) ? __ldg(P.at(b0 + r, dir ? T - 1 : 0) + dir * H4 + j) : 0.0f;
    __syncthreads();
    for (int step = 0; step < T; ++step) {
        const int t = dir ? (T - 1 - step) : step;
        float px[R];
#pragma unroll
        for (int r = 0; r < R; ++r) px[r] = px_next[r];
        if (step + 1 < T) {
            const int tn = dir ? (t - 1) : (t + 1);
#pragma unroll
            for (int r = 0; r < R; ++r) px_next[r] = (b0 + r < B) ? __ldg(P.at(b0 + r, tn) + dir * H4 + j) : 0.0f;
        }
        if ((j & 31) == 0 && step + PF_STEPS < T) {          // one DRAM round trip per step would otherwise bound the step time
            const int tp = dir ? (t - PF_STEPS) : (t + PF_STEPS);
#pragma unroll
            for (int r = 0; r < R; ++r) if (b0 + r < B) prefetch_l2(P.at(b0 + r, tp) + dir * H4 + j);
        }
        float acc[R][4];                    // R <= 2: four partial sums per trace (FMA chain 16 deep, not 64)
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.0f;
#pragma unroll
        for (int k = 0; k < HH; k += 4) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const float4 hv = *reinterpret_cast<const float4*>(h_s + r * HH + k);
                acc[r][0] = fmaf(w[k], hv.x, acc[r][0]);
                acc[r][1 % NACC] = fmaf(w[k + 1], hv.y, acc[r][1 % NACC]);
                acc[r][2 % NACC] = fmaf(w[k + 2], hv.z, acc[r][2 % NACC]);
                acc[r][3 % NACC] = fmaf(w[k + 3], hv.w, acc[r][3 % NACC]);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float a = px[r] + ((acc[r][0] + acc[r][1]) + (acc[r][2] + acc[r][3]));
            const float v = (gate == 2) ? tanh_q(a) : sigm_q(a);
            g_s[r * H4 + j] = v;
            if (saved && b0 + r < B) saved[((((size_t)dir * B + b0 + r) * T + t) * 5) * HH + j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int m = 0; m < CPT; ++m) {
            const int idx = j + m * H4;
            if (idx < R * HH) {
                const int r = idx / HH, u = idx % HH;
                const float* g = g_s + r * H4 + u;
                c[m] = g[HH] * c[m] + g[0] * g[2 * HH];
                const float hnew = g[3 * HH] * tanh_q(c[m]);
                h_s[r * HH + u] = hnew;
                if (b0 + r < B) {
                    out.at(b0 + r, t)[dir * HH + u] = hnew;
                    if (saved) saved[((((size_t)dir * B + b0 + r) * T + t) * 5 + 4) * HH + u] = c[m];
                }
            }
        }
        __syncthreads();
    }
}

// backward: thread j = (part p, unit u) keeps W_hh[p*H .. p*H+H)[u] in registers; dh_{t-1}[u] = sum_p partial_p[u].
template <int HH, int R>
__global__ void __launch_bounds__(4 * HH)
lstm_reg_bwd_kernel(SeqF d_out, const float* __restrict__ saved, const float* __restrict__ w_hh, SeqF dG, int B, int T) {
    constexpr int H4 = 4 * HH, CPT = (R * HH + H4 - 1) / H4, NACC = (R <= 2) ? 4 : 1;
    __shared__ __align__(16) float dg_s[R * H4];
    __shared__ float part_s[4 * R * HH];
    const int j = threadIdx.x, dir = blockIdx.y, p = j / HH, u0 = j % HH;
    const long long b0 = (long long)blockIdx.x * R;
    float w[HH];
#pragma unroll
    for (int k = 0; k < HH; ++k) w[k] = w_hh[((size_t)dir * H4 + p * HH + k) * HH + u0];
    float dc[CPT];
#pragma unroll
    for (int m = 0; m < CPT; ++m) dc[m] = 0.0f;
    for (int e = j; e < 4 * R * HH; e += H4) part_s[e] = 0.0f;
    // operands of a step (d_out, i, f, g, o, c) are fetched one step ahead; c_{prev} of a step is c of the next one
    float nx[CPT][6];
    auto fetch = [&](int step, float (*dst)[6]) {
        const int t = dir ? (T - 1 - step) : step;
#pragma unroll
        for (int m = 0; m < CPT; ++m) {
            const int idx = j + m * H4;
            const int r = idx / HH, u = idx % HH;
            if (idx < R * HH && b0 + r < B) {
                const long long b = b0 + r;
                const float* sp = saved + ((((size_t)dir * B + b) * T + t) * 5) * HH + u;
                dst[m][0] = __ldg(d_out.at(b, t) + dir * HH + u);
                dst[m][1] = __ldg(sp); dst[m][2] = __ldg(sp + HH); dst[m][3] = __ldg(sp + 2 * HH);
                dst[m][4] = __ldg(sp + 3 * HH); dst[m][5] = __ldg(sp + 4 * HH);
            } else {
#pragma unroll
                for (int q = 0; q < 6; ++q) dst[m][q] = 0.0f;
            }
        }
    };
    fetch(T - 1, nx);
    __syncthreads();
    for (int step = T - 1; step >= 0; --step) {
        const int t = dir ? (T - 1 - step) : step;
        float cur[CPT][6];
#pragma unroll
        for (int m = 0; m < CPT; ++m)
#pragma unroll
            for (int q = 0; q < 6; ++q) cur[m][q] = nx[m][q];
        if (step > 0) fetch(step - 1, nx);
        if ((j & 31) == 0 && step >= PF_STEPS) {
            const int tp = dir ? (T - 1 - (step - PF_STEPS)) : (step - PF_STEPS);
#pragma unroll
            for (int m = 0; m < CPT; ++m) {
                const int idx = j + m * H4;
                const int r = idx / HH, u = idx % HH;
                if (idx < R * HH && b0 + r < B) {
                    const float* sp = saved + ((((size_t)dir * B + b0 + r) * T + tp) * 5) * HH + u;
#pragma unroll
                    for (int q = 0; q < 5; ++q) prefetch_l2(sp + q * HH);
                    prefetch_l2(d_out.at(b0 + r, tp) + dir * HH + u);
                }
            }
        }
#pragma unroll
        for (int m = 0; m < CPT; ++m) {
            const int idx = j + m * H4;
            if (idx < R * HH) {
                const int r = idx / HH, u = idx % HH;
                float g_i = 0.0f, g_f = 0.0f, g_g = 0.0f, g_o = 0.0f;
                if (b0 + r < B) {
                    const long long b = b0 + r;
                    const float dh = part_s[(0 * R + r) * HH + u] + part_s[(1 * R + r) * HH + u] +
                                     part_s[(2 * R + r) * HH + u] + part_s[(3 * R + r) * HH + u];
                    const float d = dh + cur[m][0];
                    const float gi = cur[m][1], gf = cur[m][2], gg = cur[m][3], go = cur[m][4], cc = cur[m][5];
                    const float cprev = (step == 0) ? 0.0f : nx[m][5];
                    const float tc = tanh_q(cc);
                    const float dcell = dc[m] + d * go * (1.0f - tc * tc);
                    g_o = d * tc * go * (1.0f - go);
                    g_i = dcell * gg * gi * (1.0f - gi);
                    g_f = dcell * cprev * gf * (1.0f - gf);
                    g_g = dcell * gi * (1.0f - gg * gg);
                    dc[m] = dcell * gf;
                    float* gp = dG.at(b, t) + dir * H4 + u;
                    gp[0] = g_i; gp[HH] = g_f; gp[2 * HH] = g_g; gp[3 * HH] = g_o;
                }
                float* ds = dg_s + r * H4 + u;
                ds[0] = g_i; ds[HH] = g_f; ds[2 * HH] = g_g; ds[3 * HH] = g_o;
            }
        }
        __syncthreads();
        float acc[R][4];
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.0f;
#pragma unroll
        for (int k = 0; k < HH; k += 4) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const float4 gv = *reinterpret_cast<const float4*>(dg_s + r * H4 + p * HH + k);
                acc[r][0] = fmaf(w[k], gv.x, acc[r][0]);
                acc[r][1 % NACC] = fmaf(w[k + 1], gv.y, acc[r][1 % NACC]);
                acc[r][2 % NACC] = fmaf(w[k + 2], gv.z, acc[r][2 % NACC]);
                acc[r][3 % NACC] = fmaf(w[k + 3], gv.w, acc[r][3 % NACC]);
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r) part_s[(p * R + r) * HH + u0] = (acc[r][0] + acc[r][1]) + (acc[r][2] + acc[r][3]);
        __syncthreads();
    }
}

// traces per CTA: the smallest R whose grid is co-resident in one wave (several small CTAs per SM overlap each other's
// barrier and latency stalls; resident CTAs per SM follow the register footprint of each variant).  What it returns:
// R = 1 for B <= 148, 2 for B <= 296, 4 for B <= 592, 16 above.  R = 8 is never returned: R = 4 already covers every
// B <= 592, and R = 8's own condition (2 ceil(B / 8) <= 148) also ends at 592.  The <HH, 8> launches below are kept
// so that a change of the occupancy table needs no new instantiation; tests/test_bilstm_kernels_gpu.py reaches every
// other one.
int pick_r(int B) {
    const int rs[5] = {1, 2, 4, 8, 16}, occ[5] = {2, 2, 2, 1, 1};
    for (int i = 0; i < 5; ++i)
        if (2LL * ((B + rs[i] - 1) / rs[i]) <= 148LL * occ[i]) return rs[i];
    return 16;
}

template <int HH>
int launch_reg_fwd(const SeqF& sp, const float* w_hh, const SeqF& so, float* saved, int B, int T, cudaStream_t stream) {
    const int R = pick_r(B);
#define RS_REG_FWD(RR) lstm_reg_fwd_kernel<HH, RR><<<dim3((B + RR - 1) / RR, 2), 4 * HH, 0, stream>>>(sp, w_hh, so, saved, B, T)
    switch (R) {
        case 16: RS_REG_FWD(16); break;
        case 8: RS_REG_FWD(8); break;
        case 4: RS_REG_FWD(4); break;
        case 2: RS_REG_FWD(2); break;
        default: RS_REG_FWD(1); break;
    }
#undef RS_REG_FWD
    return 0;
}

template <int HH>
int launch_reg_bwd(const SeqF& sdo, const float* saved, const float* w_hh, const SeqF& sg, int B, int T, cudaStream_t stream) {
    const int R = pick_r(B);
#define RS_REG_BWD(RR) lstm_reg_bwd_kernel<HH, RR><<<dim3((B + RR - 1) / RR, 2), 4 * HH, 0, stream>>>(sdo, saved, w_hh, sg, B, T)
    switch (R) {
        case 16: RS_REG_BWD(16); break;
        case 8: RS_REG_BWD(8); break;
        case 4: RS_REG_BWD(4); break;
        case 2: RS_REG_BWD(2); break;
        default: RS_REG_BWD(1); break;
    }
#undef RS_REG_BWD
    return 0;
}

SeqF mkf(const float* p, int64_t ld, int64_t trace_rows, int64_t row0) {
    SeqF s;
    s.p = const_cast<float*>(p);
    s.ld = ld; s.trace_rows = trace_rows; s.row0 = row0;
    return s;
}

// The general kernels run at H = 96 .. 256 only (H = 32 and 64 take the register kernels above), so wsmem, which needs
// H <= 64, is always false here: the <R, true> instantiations cannot be reached.
struct Shape { int S, R; bool wsmem; };
Shape pick(int B, int H) {
    Shape s;
    s.wsmem = (size_t)H * 4 * H * 4 <= 96 * 1024;          // H <= 64 keeps two CTAs per SM with W resident
    s.S = (H <= 64) ? 4 : (H <= 128 ? 2 : 1);
    s.R = (B > 148 * 2) ? 4 : 1;                          // few traces: one per thread row, more CTAs, lower step latency
    return s;
}

}  // namespace

extern "C" int rs_lstm_fwd_f32(const float* P, int64_t p_ld, int64_t p_rows, int64_t p_row0, const float* w_hh,
                               const float* w_hh_t, float* out, int64_t o_ld, int64_t o_rows, int64_t o_row0, float* saved, int B, int T, int H,
                               void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0 || T == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(H >= 32 && H % 32 == 0 && H <= 256, "rs_lstm_fwd_f32: hidden size %d must be a multiple of 32 in [32,256]", H);
    RS_REQUIRE(P && w_hh && w_hh_t && out && B >= 0 && T >= 0, "rs_lstm_fwd_f32: bad arguments");
    if (H == 32 || H == 64) {                               // weights in registers
        SeqF rp = mkf(P, p_ld, p_rows, p_row0), ro = mkf(out, o_ld, o_rows, o_row0);
        if (H == 64) launch_reg_fwd<64>(rp, w_hh, ro, saved, B, T, stream);
        else launch_reg_fwd<32>(rp, w_hh, ro, saved, B, T, stream);
        rs::count_launch();
        RS_CUDA_OK(cudaGetLastError());
        return 0;
    }
    const Shape s = pick(B, H);
    const int Bt = s.S * s.R;
    const size_t smem = ((s.wsmem ? (size_t)H * 4 * H : 0) + 2 * (size_t)Bt * H) * sizeof(float);
    dim3 grid((B + Bt - 1) / Bt, 2), block(H, s.S);
    SeqF sp = mkf(P, p_ld, p_rows, p_row0), so = mkf(out, o_ld, o_rows, o_row0);
#define RS_LSTM_FWD(RR, WS)                                                                                            \
    do {                                                                                                               \
        RS_CUDA_OK(cudaFuncSetAttribute(lstm_fwd_f32_kernel<RR, WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        lstm_fwd_f32_kernel<RR, WS><<<grid, block, smem, stream>>>(sp, w_hh_t, so, saved, B, T, H);                    \
    } while (0)
    if (s.R == 4) { if (s.wsmem) RS_LSTM_FWD(4, true); else RS_LSTM_FWD(4, false); }
    else          { if (s.wsmem) RS_LSTM_FWD(1, true); else RS_LSTM_FWD(1, false); }
#undef RS_LSTM_FWD
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_lstm_bwd_f32(const float* d_out, int64_t do_ld, int64_t do_rows, int64_t do_row0, const float* saved,
                               const float* w_hh, float* dG, int64_t g_ld, int64_t g_rows, int64_t g_row0, int B, int T,
                               int H, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0 || T == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(H >= 32 && H % 32 == 0 && H <= 256, "rs_lstm_bwd_f32: hidden size %d must be a multiple of 32 in [32,256]", H);
    RS_REQUIRE(d_out && saved && w_hh && dG && B >= 0 && T >= 0, "rs_lstm_bwd_f32: bad arguments");
    if (H == 32 || H == 64) {
        SeqF rdo = mkf(d_out, do_ld, do_rows, do_row0), rg = mkf(dG, g_ld, g_rows, g_row0);
        if (H == 64) launch_reg_bwd<64>(rdo, saved, w_hh, rg, B, T, stream);
        else launch_reg_bwd<32>(rdo, saved, w_hh, rg, B, T, stream);
        rs::count_launch();
        RS_CUDA_OK(cudaGetLastError());
        return 0;
    }
    const Shape s = pick(B, H);
    const int Bt = s.S * s.R;
    const size_t smem = ((s.wsmem ? (size_t)H * 4 * H : 0) + (size_t)Bt * 4 * H) * sizeof(float);
    dim3 grid((B + Bt - 1) / Bt, 2), block(H, s.S);
    SeqF sdo = mkf(d_out, do_ld, do_rows, do_row0), sg = mkf(dG, g_ld, g_rows, g_row0);
#define RS_LSTM_BWD(RR, WS)                                                                                            \
    do {                                                                                                               \
        RS_CUDA_OK(cudaFuncSetAttribute(lstm_bwd_f32_kernel<RR, WS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        lstm_bwd_f32_kernel<RR, WS><<<grid, block, smem, stream>>>(sdo, saved, w_hh, sg, B, T, H);                     \
    } while (0)
    if (s.R == 4) { if (s.wsmem) RS_LSTM_BWD(4, true); else RS_LSTM_BWD(4, false); }
    else          { if (s.wsmem) RS_LSTM_BWD(1, true); else RS_LSTM_BWD(1, false); }
#undef RS_LSTM_BWD
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
