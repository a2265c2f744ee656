// Query decoder of the shipped model (SURVEY.md 8(f) rank 2; src/benchmark/model.py:60-137 SimpleQueryDecoder) as ONE
// streaming pass over the encoder memory per direction of autograd, plus the per-trace normaliser (model.py:38-46).
//
// The queries are parameters, not data: q = q_proj(query_embed) is the same for every trace.  The key and value
// projections therefore fold into the query side,
//     scores[b,q,n] = tau * (q_q . (W_k m_n + b_k))   = (tau q W_k)_q . m_n + tau q_q . b_k      =: qk_q . m_n + qb_q
//     attn . (W_v m + b_v)                             = W_v (attn . m) + b_v                     (rows of attn sum to 1)
// so neither K nor V (2 x B x N x D floats) is ever materialised: the kernel reads each memory row once, keeps a running
// softmax (max, sum) per query, and accumulates ctx[b,q,:] = sum_n attn m_n, anchor[b,q,:] = sum_n attn (xyz_n - mean)/rms
// and the masked mean of the memory (the FiLM summary, model.py:98-104).  Long traces are split over several CTAs
// (flash-decoding style) and merged by a small combine kernel.  The backward pass recomputes the probabilities from
// the saved (max, sum) and produces d_memory, d_qk, d_qb in one more pass.
//
// Tiling: 256 threads = 32 queries x 8 lanes; 32 tokens per chunk staged in shared memory with rows padded to D+1
// floats (conflict-free for both the score dot products and the ctx update).
#include <math.h>

#include "common.cuh"
#include "../../include/roomslam_b200.h"

namespace {

constexpr int QT = 32;        // queries per tile
constexpr int TC = 32;        // tokens per chunk
constexpr int NT = 256;
constexpr int MAXJ = 32;      // D / 8 <= 32  (D <= 256)

struct SeqC {
    const float* p;
    long long ld, trace_rows, row0;
    __device__ __forceinline__ const float* at(long long b, long long t) const { return p + ((b * trace_rows + row0 + t) * ld); }
};

// ---- per-trace statistics: masked mean of (x, y, z), RMS of the centred (x, z) with floor 1e-3, valid count ----
__global__ void __launch_bounds__(256)
trace_stats_kernel(const float* __restrict__ traces, int F, const unsigned char* __restrict__ mask, int N,
                   float* __restrict__ mean, float* __restrict__ rms, float* __restrict__ count) {
    __shared__ double red[4][8];
    __shared__ float mu[3];
    const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* tr = traces + (long long)b * N * F;
    const unsigned char* mk = mask ? mask + (long long)b * N : nullptr;
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int n = threadIdx.x; n < N; n += 256) {
        if (!mk || mk[n]) { s[0] += tr[(long long)n * F]; s[1] += tr[(long long)n * F + 1]; s[2] += tr[(long long)n * F + 2]; s[3] += 1.0; }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
        if (lane == 0) red[k][warp] = s[k];
    }
    __syncthreads();
    double cnt = 0.0;
    for (int w = 0; w < 8; ++w) cnt += red[3][w];
    const double denom = cnt < 1.0 ? 1.0 : cnt;
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[threadIdx.x][w];
        mu[threadIdx.x] = (float)(t / denom);
        mean[b * 3 + threadIdx.x] = mu[threadIdx.x];
    }
    __syncthreads();
    double q = 0.0;
    for (int n = threadIdx.x; n < N; n += 256) {
        if (!mk || mk[n]) {
            const float dx = tr[(long long)n * F] - mu[0], dz = tr[(long long)n * F + 2] - mu[2];
            q += (double)dx * dx + (double)dz * dz;
        }
    }
    for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
    __syncthreads();
    if (lane == 0) red[0][warp] = q;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += red[0][w];
        const float r = sqrtf((float)(t / denom));
        rms[b] = r < 1e-3f ? 1e-3f : r;
        count[b] = (float)denom;
    }
}

// stage TC tokens of the memory (rows n0 .. n0+TC) and their normalised coordinates / validity into shared memory
__device__ __forceinline__ void stage_chunk(const SeqC& mem, const float* __restrict__ traces, int F,
                                            const unsigned char* __restrict__ mask, const float* mu, float inv_rms,
                                            long long b, int N, int n0, int n_end, int D, float* m_s, float* nc_s) {
    const int Dp = D + 1;
    const float* src = mem.at(b, n0);
    for (int e = threadIdx.x; e < TC * (D / 4); e += NT) {
        const int tok = e / (D / 4), k4 = e % (D / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (n0 + tok < n_end) v = __ldg(reinterpret_cast<const float4*>(src + (long long)tok * mem.ld) + k4);
        float* d = m_s + tok * Dp + k4 * 4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    if (threadIdx.x < TC) {
        const int n = n0 + threadIdx.x;
        const bool ok = n < n_end && (!mask || mask[b * N + n]);
        float c0 = 0.f, c1 = 0.f, c2 = 0.f;
        if (n < n_end) {
            const float* tp = traces + (b * N + n) * F;
            c0 = (tp[0] - mu[0]) * inv_rms; c1 = (tp[1] - mu[1]) * inv_rms; c2 = (tp[2] - mu[2]) * inv_rms;
        }
        nc_s[threadIdx.x * 4 + 0] = c0; nc_s[threadIdx.x * 4 + 1] = c1; nc_s[threadIdx.x * 4 + 2] = c2;
        nc_s[threadIdx.x * 4 + 3] = ok ? 1.0f : 0.0f;
    }
}

// partial record per (b, split, q): [max, sum, anchor x3, ctx D];  one extra row per (b, split): [count, -, -, -, -, sum_m D]
__global__ void __launch_bounds__(NT)
query_attn_fwd_kernel(SeqC mem, const float* __restrict__ traces, int F, const unsigned char* __restrict__ mask,
                      const float* __restrict__ mean, const float* __restrict__ rms, const float* __restrict__ qk,
                      const float* __restrict__ qb, int N, int Q, int D, int tokens_per_split, float* __restrict__ part) {
    extern __shared__ __align__(16) float sm[];
    const int Dp = D + 1, J = D / 8;
    float* qk_s = sm;                       // [QT][Dp]
    float* m_s = qk_s + QT * Dp;            // [TC][Dp]
    float* p_s = m_s + TC * Dp;             // [QT][TC+1]
    float* nc_s = p_s + QT * (TC + 1);      // [TC][4]
    float* qb_s = nc_s + TC * 4;            // [QT]
    __shared__ float mu[3];
    const long long b = blockIdx.x;
    const int split = blockIdx.y, qt = blockIdx.z, splits = gridDim.y;
    const int q = threadIdx.x >> 3, g8 = threadIdx.x & 7;
    const int qg = qt * QT + q;
    for (int e = threadIdx.x; e < QT * D; e += NT) {
        const int qq = e / D, k = e % D;
        qk_s[qq * Dp + k] = (qt * QT + qq < Q) ? qk[(long long)(qt * QT + qq) * D + k] : 0.0f;
    }
    if (threadIdx.x < QT) qb_s[threadIdx.x] = (qt * QT + threadIdx.x < Q) ? qb[qt * QT + threadIdx.x] : 0.0f;
    if (threadIdx.x < 3) mu[threadIdx.x] = mean[b * 3 + threadIdx.x];
    const float inv_rms = 1.0f / rms[b];
    const int n_begin = split * tokens_per_split;
    const int n_end = min(N, n_begin + tokens_per_split);
    float m_run = -INFINITY, l_run = 0.0f, anc = 0.0f;
    float acc[MAXJ];
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) acc[j] = 0.0f;
    float msum = 0.0f, mcnt = 0.0f;         // FiLM summary: thread d < D sums memory[., d] over the valid tokens (q tile 0 only)
    __syncthreads();
    for (int n0 = n_begin; n0 < n_end; n0 += TC) {
        stage_chunk(mem, traces, F, mask, mu, inv_rms, b, N, n0, n_end, D, m_s, nc_s);
        __syncthreads();
        float s[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) s[j] = 0.0f;
        const float* qrow = qk_s + q * Dp;
        for (int k = 0; k < D; ++k) {
            const float w = qrow[k];
#pragma unroll
            for (int j = 0; j < 4; ++j) s[j] = fmaf(w, m_s[(g8 + 8 * j) * Dp + k], s[j]);
        }
        float cmax = -INFINITY;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            s[j] = nc_s[(g8 + 8 * j) * 4 + 3] != 0.0f ? s[j] + qb_s[q] : -INFINITY;
            cmax = fmaxf(cmax, s[j]);
        }
        for (int o = 1; o < 8; o <<= 1) cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        const float m_new = fmaxf(m_run, cmax);
        float alpha = 1.0f, psum = 0.0f;
        if (m_new != -INFINITY) {
            alpha = __expf(m_run - m_new);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float pj = __expf(s[j] - m_new);
                p_s[q * (TC + 1) + g8 + 8 * j] = pj;
                psum += pj;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) p_s[q * (TC + 1) + g8 + 8 * j] = 0.0f;
        }
        for (int o = 1; o < 8; o <<= 1) psum += __shfl_xor_sync(0xffffffffu, psum, o);
        l_run = l_run * alpha + psum;
        m_run = m_new;
        __syncwarp();                       // the 8 lanes of a query share one warp: p_s row complete
        const float* prow = p_s + q * (TC + 1);
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) if (j < J) acc[j] *= alpha;
        anc *= alpha;
        for (int tok = 0; tok < TC; ++tok) {
            const float pj = prow[tok];
            const float* mrow = m_s + tok * Dp + g8;
#pragma unroll
            for (int j = 0; j < MAXJ; ++j) if (j < J) acc[j] = fmaf(pj, mrow[8 * j], acc[j]);
            anc = fmaf(pj, nc_s[tok * 4 + (g8 & 3)], anc);
        }
        if (qt == 0 && threadIdx.x < D) {
            for (int tok = 0; tok < TC; ++tok) {
                const float v = nc_s[tok * 4 + 3];
                msum = fmaf(v, m_s[tok * Dp + threadIdx.x], msum);
                mcnt += v;
            }
        }
        __syncthreads();
    }
    const long long rec = D + 5;
    float* base = part + ((b * splits + split) * (long long)(Q + 1)) * rec;
    if (qg < Q) {
        float* r = base + (long long)qg * rec;
        if (g8 == 0) { r[0] = m_run; r[1] = l_run; }
        if (g8 < 3) r[2 + g8] = anc;
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) if (j < J) r[5 + g8 + 8 * j] = acc[j];
    }
    if (qt == 0 && threadIdx.x < D) {
        float* r = base + (long long)Q * rec;
        if (threadIdx.x == 0) r[0] = mcnt;
        r[5 + threadIdx.x] = msum;
    }
}

// merges the per-split partials: ctx, anchor, softmax stats (max, sum) and the FiLM summary
__global__ void query_attn_combine_kernel(const float* __restrict__ part, int Q, int D, int splits, float* __restrict__ ctx,
                                          float* __restrict__ anchor, float* __restrict__ summary, float* __restrict__ stats) {
    const long long b = blockIdx.x;
    const int qg = blockIdx.y;              // Q = the summary row
    const long long rec = D + 5;
    const float* base = part + (b * splits * (long long)(Q + 1)) * rec + (long long)qg * rec;
    const long long sstride = (long long)(Q + 1) * rec;
    if (qg == Q) {
        float cnt = 0.0f;
        for (int s = 0; s < splits; ++s) cnt += base[s * sstride];
        const float inv = 1.0f / fmaxf(cnt, 1.0f);
        for (int d = threadIdx.x; d < D; d += blockDim.x) {
            float t = 0.0f;
            for (int s = 0; s < splits; ++s) t += base[s * sstride + 5 + d];
            summary[b * D + d] = t * inv;
        }
        return;
    }
    float M = -INFINITY;
    for (int s = 0; s < splits; ++s) M = fmaxf(M, base[s * sstride]);
    float L = 0.0f;
    for (int s = 0; s < splits; ++s) {
        const float ms = base[s * sstride];
        if (ms != -INFINITY) L += base[s * sstride + 1] * __expf(ms - M);
    }
    const float invL = 1.0f / L;            // a trace without a single valid token gives NaN, like the reference softmax
    for (int d = threadIdx.x; d < D + 3; d += blockDim.x) {
        float t = 0.0f;
        for (int s = 0; s < splits; ++s) {
            const float ms = base[s * sstride];
            if (ms != -INFINITY) t += base[s * sstride + (d < D ? 5 + d : 2 + d - D)] * __expf(ms - M);
        }
        if (d < D) ctx[(b * Q + qg) * D + d] = t * invL;
        else anchor[(b * Q + qg) * 3 + d - D] = t * invL;
    }
    if (threadIdx.x == 0) { stats[(b * Q + qg) * 2] = M; stats[(b * Q + qg) * 2 + 1] = L; }
}

// backward: recompute p from (max, sum); dP = d_ctx . m + d_anchor . nc; dS = p (dP - delta);
//   d_memory[n] (+)= sum_q p d_ctx_q + dS qk_q  (+ d_summary / count on valid tokens)
//   dqk partial[b, split][q] = sum_n dS m_n ; dqb partial = sum_n dS
// Several query tiles add into the same d_memory rows: with atomics (atomic_dm) in one launch, or (kDet) one launch per
// tile, qt = qt_det, each adding onto what the launches of the tiles before it wrote -- a fixed order, one writer per element
// and launch.  A launch per tile was chosen over per-tile partial buffers: no workspace (B N D floats per tile) and no
// extra reduction kernel.
template <bool kDet>
__global__ void __launch_bounds__(NT)
query_attn_bwd_kernel(SeqC mem, const float* __restrict__ traces, int F, const unsigned char* __restrict__ mask,
                      const float* __restrict__ mean, const float* __restrict__ rms, const float* __restrict__ count,
                      const float* __restrict__ qk, const float* __restrict__ qb, const float* __restrict__ ctx,
                      const float* __restrict__ anchor, const float* __restrict__ stats, const float* __restrict__ d_ctx,
                      const float* __restrict__ d_anchor, const float* __restrict__ d_summary, int N, int Q, int D,
                      int tokens_per_split, float* __restrict__ d_mem, long long dm_ld, long long dm_rows, long long dm_row0,
                      int atomic_dm, float* __restrict__ dq_part, int qt_det) {
    extern __shared__ __align__(16) float sm[];
    const int Dp = D + 1, J = D / 8;
    float* qk_s = sm;                       // [QT][Dp]
    float* dc_s = qk_s + QT * Dp;           // [QT][Dp]   d_ctx rows
    float* m_s = dc_s + QT * Dp;            // [TC][Dp]
    float* p_s = m_s + TC * Dp;             // [QT][TC+1]
    float* ds_s = p_s + QT * (TC + 1);      // [QT][TC+1]
    float* nc_s = ds_s + QT * (TC + 1);     // [TC][4]
    float* qv_s = nc_s + TC * 4;            // [QT][8]: qb, max, 1/sum, delta, d_anchor x3, -
    __shared__ float mu[3];
    const long long b = blockIdx.x;
    const int split = blockIdx.y, qt = kDet ? qt_det : blockIdx.z, splits = gridDim.y;
    const int q = threadIdx.x >> 3, g8 = threadIdx.x & 7;
    const int qg = qt * QT + q;
    for (int e = threadIdx.x; e < QT * D; e += NT) {
        const int qq = e / D, k = e % D;
        const bool ok = qt * QT + qq < Q;
        qk_s[qq * Dp + k] = ok ? qk[(long long)(qt * QT + qq) * D + k] : 0.0f;
        dc_s[qq * Dp + k] = ok ? d_ctx[(b * Q + qt * QT + qq) * D + k] : 0.0f;
    }
    if (threadIdx.x < 3) mu[threadIdx.x] = mean[b * 3 + threadIdx.x];
    {   // delta_q = d_ctx_q . ctx_q + d_anchor_q . anchor_q   (= sum_n p dP)
        float part = 0.0f;
        if (qg < Q) {
            for (int d = g8; d < D; d += 8) part = fmaf(d_ctx[(b * Q + qg) * D + d], ctx[(b * Q + qg) * D + d], part);
            if (g8 < 3) part = fmaf(d_anchor[(b * Q + qg) * 3 + g8], anchor[(b * Q + qg) * 3 + g8], part);
        }
        for (int o = 1; o < 8; o <<= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (g8 == 0) {
            float* v = qv_s + q * 8;
            const bool ok = qg < Q;
            v[0] = ok ? qb[qg] : 0.0f;
            v[1] = ok ? stats[(b * Q + qg) * 2] : 0.0f;
            v[2] = ok ? 1.0f / stats[(b * Q + qg) * 2 + 1] : 0.0f;
            v[3] = part;
            v[4] = ok ? d_anchor[(b * Q + qg) * 3] : 0.0f;
            v[5] = ok ? d_anchor[(b * Q + qg) * 3 + 1] : 0.0f;
            v[6] = ok ? d_anchor[(b * Q + qg) * 3 + 2] : 0.0f;
        }
    }
    const float inv_rms = 1.0f / rms[b];
    const float inv_cnt = 1.0f / count[b];
    const int n_begin = split * tokens_per_split;
    const int n_end = min(N, n_begin + tokens_per_split);
    float dqk[MAXJ];
#pragma unroll
    for (int j = 0; j < MAXJ; ++j) dqk[j] = 0.0f;
    float dqb = 0.0f;
    __syncthreads();
    const float* qv = qv_s + q * 8;
    for (int n0 = n_begin; n0 < n_end; n0 += TC) {
        stage_chunk(mem, traces, F, mask, mu, inv_rms, b, N, n0, n_end, D, m_s, nc_s);
        __syncthreads();
        float s[4], dp[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { s[j] = 0.0f; dp[j] = 0.0f; }
        const float* qrow = qk_s + q * Dp;
        const float* drow = dc_s + q * Dp;
        for (int k = 0; k < D; ++k) {
            const float w = qrow[k], g = drow[k];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float mv = m_s[(g8 + 8 * j) * Dp + k];
                s[j] = fmaf(w, mv, s[j]);
                dp[j] = fmaf(g, mv, dp[j]);
            }
        }
        float dsum = 0.0f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int tok = g8 + 8 * j;
            float p = 0.0f, dS = 0.0f;
            if (nc_s[tok * 4 + 3] != 0.0f && qg < Q) {
                p = __expf(s[j] + qv[0] - qv[1]) * qv[2];
                const float dP = dp[j] + qv[4] * nc_s[tok * 4] + qv[5] * nc_s[tok * 4 + 1] + qv[6] * nc_s[tok * 4 + 2];
                dS = p * (dP - qv[3]);
            }
            p_s[q * (TC + 1) + tok] = p;
            ds_s[q * (TC + 1) + tok] = dS;
            dsum += dS;
        }
        for (int o = 1; o < 8; o <<= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
        dqb += dsum;
        __syncwarp();
        {   // dqk_q += sum_tok dS m_tok
            const float* dsrow = ds_s + q * (TC + 1);
            for (int tok = 0; tok < TC; ++tok) {
                const float w = dsrow[tok];
                const float* mrow = m_s + tok * Dp + g8;
#pragma unroll
                for (int j = 0; j < MAXJ; ++j) if (j < J) dqk[j] = fmaf(w, mrow[8 * j], dqk[j]);
            }
        }
        __syncthreads();                    // p_s / ds_s of all queries complete
        {   // d_memory: thread (tok = q, g8) owns columns g8 + 8 j of token n0 + tok
            const int tok = q;
            const int n = n0 + tok;
            float dm[MAXJ];
            const float add = (qt == 0 && d_summary) ? nc_s[tok * 4 + 3] * inv_cnt : 0.0f;
#pragma unroll
            for (int j = 0; j < MAXJ; ++j) if (j < J) dm[j] = (add != 0.0f) ? add * d_summary[b * D + g8 + 8 * j] : 0.0f;
            for (int qq = 0; qq < QT; ++qq) {
                const float p = p_s[qq * (TC + 1) + tok], dS = ds_s[qq * (TC + 1) + tok];
                const float* c = dc_s + qq * Dp + g8;
                const float* w = qk_s + qq * Dp + g8;
#pragma unroll
                for (int j = 0; j < MAXJ; ++j) if (j < J) dm[j] = fmaf(p, c[8 * j], fmaf(dS, w[8 * j], dm[j]));
            }
            if (n < n_end) {
                float* dst = d_mem + ((b * dm_rows + dm_row0 + n) * dm_ld) + g8;
#pragma unroll
                for (int j = 0; j < MAXJ; ++j) {
                    if (j < J) {
                        if (kDet) dst[8 * j] = qt == 0 ? dm[j] : dst[8 * j] + dm[j];
                        else if (atomic_dm) atomicAdd(dst + 8 * j, dm[j]);
                        else dst[8 * j] = dm[j];
                    }
                }
            }
        }
        __syncthreads();
    }
    if (qg < Q) {
        float* r = dq_part + ((b * splits + split) * (long long)Q + qg) * (D + 1);
#pragma unroll
        for (int j = 0; j < MAXJ; ++j) if (j < J) r[g8 + 8 * j] = dqk[j];
        if (g8 == 0) r[D] = dqb;
    }
}

SeqC mkc(const float* p, int64_t ld, int64_t rows, int64_t row0) {
    SeqC s; s.p = p; s.ld = ld; s.trace_rows = rows; s.row0 = row0;
    return s;
}

}  // namespace

extern "C" int rs_trace_stats_f32(const float* traces, int F, const unsigned char* mask, int B, int N, float* mean, float* rms,
                                  float* count, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(traces && mean && rms && count && F >= 3 && B >= 0 && N >= 1, "rs_trace_stats_f32: bad arguments");
    trace_stats_kernel<<<B, 256, 0, stream>>>(traces, F, mask, N, mean, rms, count);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int64_t rs_query_attn_workspace(int B, int Q, int D, int splits) {
    return (int64_t)B * splits * (Q + 1) * (D + 5);
}

extern "C" int rs_query_attn_fwd_f32(const float* memory, int64_t m_ld, int64_t m_rows, int64_t m_row0, const float* traces,
                                     int F, const unsigned char* mask, const float* mean, const float* rms, const float* qk,
                                     const float* qb, int B, int N, int Q, int D, int splits, float* workspace, float* ctx,
                                     float* anchor, float* summary, float* stats, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(memory && traces && mean && rms && qk && qb && workspace && ctx && anchor && summary && stats,
               "rs_query_attn_fwd_f32: null pointer");
    RS_REQUIRE(D >= 32 && D % 32 == 0 && D <= 256, "rs_query_attn_fwd_f32: d_model %d must be a multiple of 32 in [32,256]", D);
    RS_REQUIRE(Q >= 1 && N >= 1 && splits >= 1 && F >= 3 && m_ld % 4 == 0, "rs_query_attn_fwd_f32: bad sizes");
    const int chunks = (N + TC - 1) / TC;
    const int tps = ((chunks + splits - 1) / splits) * TC;
    const int qtiles = (Q + QT - 1) / QT;
    const size_t smem = ((size_t)2 * QT * (D + 1) + QT * (TC + 1) + TC * 4 + QT) * sizeof(float);
    RS_CUDA_OK(cudaFuncSetAttribute(query_attn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    query_attn_fwd_kernel<<<dim3(B, splits, qtiles), NT, smem, stream>>>(mkc(memory, m_ld, m_rows, m_row0), traces, F, mask, mean,
                                                                        rms, qk, qb, N, Q, D, tps, workspace);
    rs::count_launch();
    query_attn_combine_kernel<<<dim3(B, Q + 1), 128, 0, stream>>>(workspace, Q, D, splits, ctx, anchor, summary, stats);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}

extern "C" int rs_query_attn_bwd_f32(const float* memory, int64_t m_ld, int64_t m_rows, int64_t m_row0, const float* traces,
                                     int F, const unsigned char* mask, const float* mean, const float* rms, const float* count,
                                     const float* qk, const float* qb, const float* ctx, const float* anchor,
                                     const float* stats, const float* d_ctx, const float* d_anchor, const float* d_summary,
                                     int B, int N, int Q, int D, int splits, float* d_memory, int64_t dm_ld, int64_t dm_rows,
                                     int64_t dm_row0, float* dq_part, void* stream_) {
    cudaStream_t stream = static_cast<cudaStream_t>(stream_);
    if (rs::check_device_sm100()) return 3;
    if (B == 0) return 0;        // nothing to do: empty tensors carry null pointers
    RS_REQUIRE(memory && traces && mean && rms && count && qk && qb && ctx && anchor && stats && d_ctx && d_anchor && d_memory &&
                   dq_part, "rs_query_attn_bwd_f32: null pointer");
    RS_REQUIRE(D >= 32 && D % 32 == 0 && D <= 256, "rs_query_attn_bwd_f32: d_model %d must be a multiple of 32 in [32,256]", D);
    RS_REQUIRE(Q >= 1 && N >= 1 && splits >= 1 && F >= 3 && m_ld % 4 == 0, "rs_query_attn_bwd_f32: bad sizes");
    const int chunks = (N + TC - 1) / TC;
    const int tps = ((chunks + splits - 1) / splits) * TC;
    const int qtiles = (Q + QT - 1) / QT;
    const size_t smem = ((size_t)3 * QT * (D + 1) + 2 * QT * (TC + 1) + TC * 4 + QT * 8) * sizeof(float);
    if (qtiles > 1 && rs::deterministic()) {
        RS_CUDA_OK(cudaFuncSetAttribute(query_attn_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        for (int qt = 0; qt < qtiles; ++qt) {
            query_attn_bwd_kernel<true><<<dim3(B, splits, 1), NT, smem, stream>>>(
                mkc(memory, m_ld, m_rows, m_row0), traces, F, mask, mean, rms, count, qk, qb, ctx, anchor, stats, d_ctx, d_anchor,
                d_summary, N, Q, D, tps, d_memory, dm_ld, dm_rows, dm_row0, 0, dq_part, qt);
            rs::count_launch();
        }
        RS_CUDA_OK(cudaGetLastError());
        return 0;
    }
    RS_CUDA_OK(cudaFuncSetAttribute(query_attn_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    query_attn_bwd_kernel<false><<<dim3(B, splits, qtiles), NT, smem, stream>>>(
        mkc(memory, m_ld, m_rows, m_row0), traces, F, mask, mean, rms, count, qk, qb, ctx, anchor, stats, d_ctx, d_anchor,
        d_summary, N, Q, D, tps, d_memory, dm_ld, dm_rows, dm_row0, qtiles > 1 ? 1 : 0, dq_part, 0);
    rs::count_launch();
    RS_CUDA_OK(cudaGetLastError());
    return 0;
}
