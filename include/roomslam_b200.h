/* roomslam_b200 C ABI: the drop-in boundary for Room-SLAM's data-parallel hot path on B200 (sm_100a).
 *
 * Upstream (Ex10si0n/room-slam) is pure Python and has no FFI; the seam it exposes is
 *   model(traces) -> dict of tensors            src/benchmark/model.py:150-153, built by build_model :406-443
 *   criterion(outputs, targets) -> dict          src/benchmark/train.py:109-135
 * and the README-specified GRU model / heatmap baseline (README.md:110-125, :15, :163-164) that this library
 * implements.  A Python caller binds these symbols with ctypes (roomslam_b200/_lib.py; INTEGRATION.md shows the
 * stub a maintainer would add upstream).  Conventions for every entry point:
 *   - plain pointers and sizes only; pointers are DEVICE pointers unless the name ends in _host;
 *   - tensors are dense, row-major, with the shapes given per function; nothing is copied or re-laid out silently;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); calls are asynchronous on it
 *     unless documented as blocking;
 *   - return 0 on success; non-zero on error (1 bad argument, 2 CUDA error, 3 no sm_100 device) with the text
 *     available from rs_last_error().  There is no CPU fallback anywhere.
 */
#ifndef ROOMSLAM_B200_H
#define ROOMSLAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library ------------------------------------------------------------------------------------------- */
const char* rs_last_error(void);       /* thread-local message of the last failing call */
int rs_abi_version(void);              /* bumped on any signature change */
int rs_device_ok(void);                /* 1 when the current CUDA device is sm_100 (B200), else 0 */
int64_t rs_launch_count(void);         /* kernels launched by this library so far (process-wide) */
/* Deterministic mode (process-wide, default off).  On: every reduction the library splits over CTAs stores per-split
 * partials into a workspace allocated in stream order on the call's stream (cudaMallocAsync) and adds them onto the output
 * in a fixed order, and the split depends on the shape only, so repeated calls on the same inputs give the same bits.
 * Off: split reductions end in floating-point atomics.  The Python binding follows torch.use_deterministic_algorithms. */
int rs_set_deterministic(int on);      /* returns 0 */
int rs_deterministic(void);            /* 1 when deterministic mode is on, else 0 */

/* ---- occupancy heatmap + stationary time (replaces README.md:15,163-164 `src/models/baseline.py`) ------- */
/* points: float32 [n_traces, seq_len, 2].  occ, stat: int32 [gy, gx].  n_dropped: one uint64.
 * Binning rules: SURVEY.md 8(a) D10/D11 (bit-exact with oracle/baseline_ref.py).  accumulate != 0 adds to
 * the existing contents of occ/stat/n_dropped instead of zeroing them first (used when sharding by trace). */
int rs_heatmap_bin(const float* points, int64_t n_traces, int64_t seq_len, float x_min, float y_min, float res,
                   int gx, int gy, float thr2, int32_t* occ, int32_t* stat, unsigned long long* n_dropped,
                   int accumulate, void* stream);
/* Same, forcing a kernel variant: 0 auto (5 when the TMA path applies, else 3); TMA variants are
 * warps x points-per-chunk x stages: 1 = 16x8x2, 2 = 8x16x2, 4 = 32x8x1, 5 = 24x8x1; 3 = generic global-atomic
 * kernel (odd seq_len, unaligned pointers, grids above 40960 cells).  For tests and tuning. */
int rs_heatmap_bin_variant(const float* points, int64_t n_traces, int64_t seq_len, float x_min, float y_min,
                           float res, int gx, int gy, float thr2, int32_t* occ, int32_t* stat,
                           unsigned long long* n_dropped, int accumulate, int variant, void* stream);
/* HOST pointers in and out; blocking; overlaps the host->device copy with binning. */
int rs_heatmap_bin_host(const float* host_points, int64_t n_traces, int64_t seq_len, float x_min, float y_min,
                        float res, int gx, int gy, float thr2, int32_t* host_occ, int32_t* host_stat,
                        unsigned long long* host_dropped);

/* ---- fp32 building blocks of the RoomSLAM model (replace torch.nn.GRU / nn.Linear / losses on the hot path) --- */
/* Sequence buffers are addressed as element(b, t, c) = p[((b*rows + row0 + t) * ld) + c]: plain (B, T, C) tensors
 * use rows = T, row0 = 0; the library's padded activation layout uses rows = T + 2, row0 = 1 with zero pad rows. */
#define RS_GEMM_ACCUMULATE 1
#define RS_GEMM_RELU 2
#define RS_GEMM_OUT_F32 4
/* C[m,n] = act(sum_k A[m*a_sm + k*a_sk] * B[k*b_sk + n*b_sn] + bias[n]) (+ C).  fp32 CUDA-core GEMM. */
int rs_sgemm(const float* A, int64_t a_sm, int64_t a_sk, const float* B, int64_t b_sk, int64_t b_sn, float* C,
             int64_t ldc, const float* bias, int M, int N, int K, int flags, void* stream);
/* out[n] (+)= sum_m A[m*lda + n] */
int rs_colsum_f32(const float* A, int64_t lda, int M, int N, float* out, int accumulate, void* stream);
/* One bidirectional GRU layer, forward (torch.nn.GRU semantics, rnn.py:1221-1224; zero initial state).
 * Either x (input size I <= 4, projection fused; w_ih [2][3H][I]) or P ([., 6H] = x W_ih^T + b_ih for both
 * directions) feeds the layer.  w_hh_t [2][H][3H] (transposed), b_ih/b_hh [2][3H], out [., 2H], h_n [2][B][H],
 * gates [2][B][T][4][H] (r, z, n, W_hn h + b_hn; NULL to skip saving for inference). */
int rs_gru_fwd_f32(const float* x, int64_t x_ld, int64_t x_rows, int64_t x_row0, int I, const float* w_ih,
                   const float* b_ih, const float* P, int64_t p_ld, int64_t p_rows, int64_t p_row0,
                   const float* w_hh_t, const float* b_hh, float* out, int64_t o_ld, int64_t o_rows, int64_t o_row0,
                   float* h_n, float* gates, const int* lengths, int B, int T, int H, void* stream);
/* lengths (all recurrence entry points): int32 [B] valid steps per trace or NULL.  Packed-sequence semantics of
 * torch.nn.utils.rnn.pack_padded_sequence: past its length a trace keeps its state (h_n = state at the last valid step),
 * emits zero outputs, and its padded outputs carry no gradient.
 * Backward through time of the same layer.  d_out [., 2H] and d_h_n [2][B][H] may be NULL (zero).  w_hh [2][3H][H].
 * Writes dGx, dGh [., 6H]: gradients w.r.t. the input-side / hidden-side gate pre-activations. */
int rs_gru_bwd_f32(const float* d_out, int64_t do_ld, int64_t do_rows, int64_t do_row0, const float* d_h_n,
                   const float* gates, const float* out, int64_t o_ld, int64_t o_rows, int64_t o_row0,
                   const float* w_hh, float* dGx, float* dGh, int64_t g_ld, int64_t g_rows, int64_t g_row0,
                   const int* lengths, int B, int T, int H, void* stream);
/* o = a * m element-wise over sequence buffers (m NULL: copy).  Inter-layer dropout mask (decision D4). */
int rs_seq_mul_f32(const float* a, int64_t a_ld, int64_t a_rows, int64_t a_row0, const float* m, int64_t m_ld,
                   int64_t m_rows, int64_t m_row0, float* o, int64_t o_ld, int64_t o_rows, int64_t o_row0, int B, int T,
                   int C, void* stream);
/* Decoder heads: raw [B, N*(C+6)] (columns class | pos | size | orient | valid) -> the five prediction tensors;
 * sizes = softplus(raw) + 1e-4 (analogue src/benchmark/model.py:129). */
int rs_heads_split_f32(const float* raw, int B, int N, int C, float* cls, float* pos, float* size, float* orient,
                       float* valid, void* stream);
int rs_heads_merge_bwd_f32(const float* raw, int B, int N, int C, const float* d_cls, const float* d_pos,
                           const float* d_size, const float* d_orient, const float* d_valid, float* d_raw, void* stream);
int rs_relu_bwd_f32(const float* dy, const float* y, float* dx, int64_t n, void* stream);
int rs_relu_bwd_bf16(const void* dy, const void* y, void* dx, int64_t n, void* stream);   /* bf16 tensors */
/* Multi-task loss (README.md:122-125): weights5 is a HOST array {class, position, size, orientation, validity}.
 * losses6 = {total, class, position, size, orientation, validity}; sums6 (double) and g_* keep what backward needs. */
int rs_loss_fwd_f32(const float* cls, const float* pos, const float* size, const float* orient, const float* vlogit,
                    const int64_t* t_cls, const float* t_pos, const float* t_size, const float* t_orient,
                    const float* t_valid, int B, int N, int C, const float* weights5, double* sums6, float* losses6,
                    float* g_cls, float* g_pos, float* g_size, float* g_orient, float* g_valid, void* stream);
int rs_loss_bwd_f32(const double* sums6, const float* d_losses6, int B, int N, int C, const float* weights5,
                    const float* g_cls, const float* g_pos, const float* g_size, const float* g_orient,
                    const float* g_valid, float* d_cls, float* d_pos, float* d_size, float* d_orient, float* d_valid,
                    void* stream);

/* ---- bf16 tensor-core GEMMs (tcgen05 + TMEM accumulators, TMA-fed): the time-parallel work of the bf16 mode ---- */
/* C[M,N] (ldc) = act(A[M,K] (bf16, lda) . B[N,K]^T (bf16, ldb) + bias[N] (fp32, optional)).  K % 64 == 0, N % 128 == 0,
 * leading dimensions in elements and multiples of 8.  flags: RS_GEMM_RELU, RS_GEMM_OUT_F32 (C is fp32 and written
 * with direct row stores; default: bf16 through TMA stores).  TMA-fed tcgen05: the decoder MLP of the bf16 mode.
 * With RS_GEMM_OUT_F32, C and bias are accessed as float4: both 16-byte aligned, ldc % 4 == 0. */
int rs_gemm_bf16_nt(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, const float* bias,
                    int64_t M, int N, int K, int flags, void* stream);
/* C[M,N] (fp32, ldc) += A[:, a_col0:a_col0+M]^T . B[:, b_col0:b_col0+N], reduction over `rows` row pairs
 * (row r + a_row_shift of A with row r + b_row_shift of B; rows outside a matrix count as zero).  M, N % 128 == 0.
 * Weight gradients dW_ih = dGx^T X and dW_hh = dGh^T H_prev (one-row shift between the operands). */
int rs_gemm_bf16_tn_acc(const void* A, int64_t lda, int64_t a_rows, int a_col0, int a_row_shift, const void* B,
                        int64_t ldb, int64_t b_rows, int b_col0, int b_row_shift, float* C, int64_t ldc, int M, int N,
                        int64_t rows, void* stream);

/* fp32 [rows, cols] (ld) -> bf16 [rows, 6 * kpad] (ld_out): sixths [lo | hi | mid | mid | hi | hi] (role_b = 0, A operand) or
 * [hi | lo | mid | hi | mid | hi] (role_b = 1, B operand; smallest partial products first); hi + mid + lo = x to 24 mantissa bits, zero padded to kpad columns.
 * One rs_gemm_bf16_nt over K = 6 * kpad then yields A . B^T at fp32 accuracy ("bf16x6") at tensor-core speed.
 * With ld % 4 == 0 the rows are read as float4: x must then be 16-byte aligned. */
int rs_split_bf16x6(const float* x, int64_t ld, int64_t rows, int cols, int kpad, int role_b, void* out, int64_t ld_out,
                    void* stream);

/* The same with the reduction running over n_seg (<= 8) passes of the same rows, pass s reading the column blocks
 * a_col0 + a_seg[s] of A and b_col0 + b_seg[s] of B (host int arrays): all partial products of a split-operand ("bf16x6")
 * weight gradient in ONE launch. */
int rs_gemm_bf16_tn_seg_acc(const void* A, int64_t lda, int64_t a_rows, int a_col0, int a_row_shift, const void* B,
                            int64_t ldb, int64_t b_rows, int b_col0, int b_row_shift, int n_seg, const int* a_seg,
                            const int* b_seg, float* C, int64_t ldc, int M, int N, int64_t rows, void* stream);

/* ---- optimizer: global-norm clipping + AdamW over one flat fp32 buffer (upstream train.py:220, :440-444) ------- */
/* g is first scaled by grad_scale (1/world_size after a sum all-reduce), then clipped to max_norm (<= 0: off). */
int rs_adamw_step_f32(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                      float eps, float weight_decay, int step, float grad_scale, float max_norm, double* sumsq_scratch,
                      void* stream);

/* ---- bf16 mode: GEMMs over the TILE-MAJOR activation layout ----------------------------------------------------
 * A per-timestep activation with C columns is stored as blocks (trace tile of 128, time row t' in [0, T+2)), each
 * block = [C/8][128][8] bf16 (C*256 contiguous bytes); rows t' = 0 and T+1 are zero padding (h before the first /
 * after the last step).  csrc/gemm_blk.cu explains why (1-D bulk copies, no-swizzle tcgen05 operands, coalesced
 * per-thread access in the recurrence kernels). */
/* For every block m < n_blocks: C_blk[:, c_chunk0*8 + n*128 ...] = A_blk[:, K blocks] . W^T + bias, K block kb =
 * the 64 columns starting at chunk a_kchunk[kb] (HOST array); W is pre-tiled [n_tiles][k_blocks][8][128][8] bf16. */
int rs_blk_gemm_nt(const void* A, int64_t a_cols, const int* a_kchunk, int k_blocks, const void* W, int n_tiles, void* C,
                   int64_t c_cols, int c_chunk0, const float* bias, int64_t n_blocks, void* stream);
/* The same without bias, the result multiplied by an inter-layer dropout mask in the epilogue: C = (A . W^T) (.) mask, mask =
 * drop_bits ([tiles][T][128][c_cols / 8] bytes, one bit per element: rs_pack_drop_mask / rs_gen_drop_bits) x *drop_scale;
 * n_blocks = tiles * (T + 2).  The data gradient dX of a layer whose INPUT went through dropout (README.md:114). */
int rs_blk_gemm_nt_drop(const void* A, int64_t a_cols, const int* a_kchunk, int k_blocks, const void* W, int n_tiles, void* C,
                        int64_t c_cols, int c_chunk0, int64_t n_blocks, const void* drop_bits, const float* drop_scale, int T,
                        void* stream);
/* Fused weight-gradient pass of one layer: every role r < n_roles (<= 18) accumulates C[r][128, n_cols[r]] += sum over
 * blocks dG_blk[:, a_mchunk[r]*8 .. +128]^T . B[r]_blk'[:, b_chunk0[r]*8 .. + n_cols[r]] (time shift b_shift[r]; n_cols
 * may be 0), when bias[r] != NULL bias[r][128] += column sums of the same dG columns, and when B2[r] != NULL
 * C2[r][128, 16] += the same dG columns ^T . B2[r]_blk (a 16-column tile-major tensor, e.g. the layer-0 input).
 * All arrays are HOST arrays of length n_roles.  Roles should do equal work per block (they share operands through
 * L2 only while they advance in lockstep).  With an even n_roles, roles 2 j and 2 j + 1 that name the same dG columns
 * (a_mchunk) run as a CTA pair: the block is read once and multicast into both CTAs -- order the roles accordingly. */
int rs_blk_wgrad(const void* dG, int64_t a_cols, const void* ones_block, int n_roles, const int* a_mchunk,
                 const void* const* B, const int64_t* b_cols, const int* b_chunk0, const int* n_cols, const int* b_shift,
                 float* const* C, const int64_t* ldc, float* const* bias, const void* const* B2, float* const* C2,
                 int tiles, int T, void* stream);
/* ---- bf16 mode: every bf16 operand image of one bidirectional layer from its fp32 master weights, one launch -------
 * w: HOST array of 8 DEVICE pointers (weight_ih, weight_hh, bias_ih, bias_hh, then the _reverse twins; torch.nn.GRU's
 * names, shapes and r|z|n gate order).  I <= 16 is layer 0, deeper layers take a multiple of 128.  Outputs (device):
 * whh_img [2][H/8 (+2 x_steps(I) for layer 0, +2 with wih_img)][3H][8] bf16 (the image rs_rec_fwd_bf16 documents), b_hn
 * [2][H], bias_x [2][3H] (b_ih + b_hh of r, z; scaled like the rows), wt_proj [6H/128][I/64][8][128][8] bf16 (B pieces of
 * rs_blk_gemm_nt for P = X W_ih^T; NULL for layer 0 whose I <= 16 columns ride in whh_img), whhT_img [2][3H/8][H][8] bf16 (rs_rec_bwd_bf16), wt_dgrad [I/128][6H/64][8][128][8] bf16 (dX = dG W_ih) or
 * NULL.
 * split = 1: every weight image holds a bf16 PAIR per weight, hi = bf16(w) then lo = bf16(w - hi), stacked along K
 * (whh_img: chunks [0, H/8) hi, [H/8, H/4) lo, then the layer-0 input chunks; whhT_img, wt_proj, wt_dgrad: K blocks hi
 * then lo); rs_rec_fwd_bf16 / rs_rec_bwd_bf16 take the same flag, rs_blk_gemm_nt simply runs the longer K.
 * wih_img [2][I/8][3H][8] bf16 (or NULL): W_ih as a resident B operand for the projection fused into the recurrence kernel
 * (rs_rec_fwd_bf16 with X); whh_img then also carries the two input chunks, holding the folded bias only. */
int rs_gru_pack_weights_bf16(const float* const* w, int H, int I, int split, void* whh_img, float* b_hn, float* bias_x,
                             void* wt_proj, void* whhT_img, void* wt_dgrad, void* wih_img, void* stream);
/* ---- bf16 mode: persistent tcgen05 GRU recurrence (H = 128), tile-major activations --------------------------- */
/* Forward of one bidirectional layer.  Layer 0: x (B, T, 1 <= I <= 16) fp32, its projection rides on the tensor core as
 * s = x_steps(I) = ceil((3 I + 2) / 16) more K = 16 steps: Whh is then [2][16 + 2 s][384][8] bf16 whose chunks 16 .. 15 + 2 s
 * hold the input columns: input i at columns 3 i + k (i < 2) or 8 + 3 (i - 2) + k (i >= 2), k = 0, 1, 2 = per gate row
 * (w_hi, w_hi, w_lo); the bias (b_hi, b_lo) at columns 6, 7; every other column 0 (I <= 2: chunk 16 as always, chunk
 * 17 = 0).  Any other I is rejected with an error.  Deeper layers, either: P tile-major (6H columns, bias folded in) and Whh [2][16][384][8]; or, with the
 * projection FUSED into the recurrence (unsplit weights): X = the layer's tile-major input (2H columns), Wih
 * [2][32][384][8] and Whh [2][18][384][8] whose chunk 16 holds only the bias (rs_gru_pack_weights_bf16 with wih_img) --
 * P and the projection GEMM are then not needed at all.  The r and z rows of all
 * weights / biases carry the factor 1/2 of sigma(a) = tanh(a/2)/2 + 1/2.  b_hn [2][H], out tile-major (2H columns,
 * zero pad rows), gates [tiles][T][2][48][128][8] fp16 = r | z | n (NULL for inference, and for a layer 0 whose backward
 * recomputes them: rs_rec_bwd_bf16_recompute; W_hn h + b_hn is NOT saved, the backward kernel recomputes it), h_n [2][B][H]
 * fp32. */
int rs_rec_fwd_bf16(const float* x, int I, const void* P, int64_t p_cols, const void* X, const void* Wih, const void* Whh,
                    const float* b_hn, void* out,
                    void* gates, float* h_n, const int* lengths, const void* drop_bits, const float* drop_scale,
                    void* out_drop, int split, int B, int T, void* stream);
/* x (B, T, I <= 16) fp32 -> tile-major bf16 with 16 columns (zero padded): layer-0 input for rs_blk_wgrad. */
int rs_pack_x_tm(const float* x, int B, int T, int I, void* out, void* stream);
/* Backward through time.  d_out tile-major (2H) or NULL, d_h_n [2][B][H] or NULL, WhhT [2][48][128][8] bf16,
 * dG tile-major (8H columns: per direction r | z | n | hn gate-gradient blocks).  Whh (the forward image, whh_chunks chunks
 * per direction) and b_hn: the kernel recomputes W_hn h_{t-1} + b_hn on the tensor core from the bulk-copied h_{t-1} tile. */
int rs_rec_bwd_bf16(const void* d_out, const float* d_h_n, const void* gates, const void* out, const void* WhhT,
                    const void* Whh, int whh_chunks, const float* b_hn, void* dG, const int* lengths, const void* drop_bits,
                    const float* drop_scale, int split, int B, int T, void* stream);
/* rs_rec_bwd_bf16 for layer 0 with unsplit weights and 1 <= I <= 2 inputs, WITHOUT saved gates: the forward ran with
 * gates = NULL, and the kernel recomputes r, z and n by replaying the forward's MMA on the tensor core (same operands, shapes
 * and K order) and its gate math; dG is bit-identical to rs_rec_bwd_bf16's from the saved gates.  x (B, T, I) fp32 is the
 * layer input the forward took, xpack a [tiles][T][128][8] bf16 workspace (its packed input chunks, written here), Whh the
 * forward image with its 18 chunks per direction; the other arguments as for rs_rec_bwd_bf16. */
int rs_rec_bwd_bf16_recompute(const void* d_out, const float* d_h_n, const float* x, int I, void* xpack, const void* out,
                              const void* WhhT, const void* Whh, int whh_chunks, const float* b_hn, void* dG, const int* lengths,
                              const void* drop_bits, const float* drop_scale, int B, int T, void* stream);
/* The same two kernels for hidden_size = 256 (BASELINE config 4: H 256, T 4000), where W_hh no longer fits in shared memory:
 * each CTA of the pair streams its half of the weights from L2 through a ring of bulk copies once per time step
 * (csrc/rec_wide.cu).  Tile-major operands as above with H = 256 (P 6H, out 2H, dG 8H columns; gates
 * [tiles][T][2][128][128][8] fp16).  Wst: [2 dirs][2 ranks][8 + ceil(s / 2) (layer 0, s = x_steps(I), 1 <= I <= 16) or 8
 * stages][2 K steps][2 chunks][384 rows][8] bf16, rows = r | z | n gate rows of hidden units [128 rank, 128 rank + 128) (r, z
 * scaled by 1/2), K step k = hidden units [16 k, 16 k + 16); layer 0: K steps 16 .. 15 + s = the input columns of
 * rs_rec_fwd_bf16's Whh (same column map), then zero K steps up to the whole stage.  WTst: [2][2][8 stages][6 K steps][2 chunks][128 rows][8] bf16 = W_hh^T with rows = hidden units
 * [128 rank, +128) and K = the 768 gate rows in r | z | n order. */
int rs_rec_fwd_bf16_wide(const float* x, int I, const void* P, const void* Wst, const float* b_hn, void* out, void* gates,
                         float* h_n, const int* lengths, const void* drop_bits, const float* drop_scale, void* out_drop,
                         int B, int T, void* stream);
int rs_rec_bwd_bf16_wide(const void* d_out, const float* d_h_n, const void* gates, const void* out, const void* WTst, void* dG,
                         const int* lengths, const void* drop_bits, const float* drop_scale, int B, int T, void* stream);
/* Inter-layer dropout (README.md:114; analogue src/benchmark/model.py:13,20) without a (B, T, 2H) multiply in HBM: the
 * mask travels as ONE BIT per element, [tiles][T][128 rows][C/8 bytes] (C = 2H), plus a device scalar scale = 1/keep.
 * rs_rec_fwd_bf16 with drop_bits writes out_drop = out (.) mask * scale next to out (the next layer's input);
 * rs_rec_bwd_bf16 with drop_bits multiplies the incoming d_out by the same mask.  rs_pack_drop_mask packs an explicit
 * (B, T, C) fp32 mask (decision D4: values 0 or 1/keep; scale = its maximum); rs_gen_drop_bits draws Bernoulli(keep)
 * bits from a counter-based hash of (seed, position) directly on the device. */
int rs_pack_drop_mask(const float* mask, int B, int T, int C, void* bits, float* scale, void* stream);
int rs_gen_drop_bits(void* bits, int B, int T, int C, float keep, uint64_t seed, float* scale, void* stream);

/* ---- on-GPU trace preprocessing (SURVEY.md 8(f) rank 1; replaces src/benchmark/dataloader.py:410-457 _process_traces
 *      = src/benchmark/inference.py:24-57 process_traces, plus the padding of collate_fn dataloader.py:510-559) ------ */
/* pts: [total, 4] fp32 rows (x, y, z, timestamp), the B traces back to back, each sorted by timestamp; offsets: [B+1]
 * int64 (device).  feats: [B, out_len, 11] = x, y, z, t - t0, vx, vy, vz, ax, ay, az, speed; rows past a trace's length
 * are zero; traces longer than max_len are down-sampled with numpy's linspace indices; mask: [B, out_len] uint8;
 * lengths: [B] int64; unsorted_flag: one int set to 1 if a timestamp decreases.  Bit-identical to the numpy reference. */
int rs_trace_features(const float* pts, const int64_t* offsets, int B, int max_len, int out_len, float* feats,
                      unsigned char* mask, int64_t* lengths, int* unsorted_flag, void* stream);

/* Uniform-rate resampling + windowing of recorded traces into the GRU's (W, seq_len, 2) input (floor plane x, z).
 * pts: [total, 4] fp64 rows (x, y, z, timestamp), time-sorted per trace; offsets [B+1]; window w covers samples
 * win_start[w] .. win_start[w]+seq_len-1 of trace win_trace[w] on the grid numpy.arange(t_first, t_last, step);
 * values = numpy.interp in fp64, rounded to fp32: bit-identical to the numpy procedure (oracle/resample_ref.py). */
int rs_resample_windows_f64(const double* pts, const int64_t* offsets, const int64_t* win_trace, const int64_t* win_start,
                            int64_t n_windows, int seq_len, double step, float* out, void* stream);

/* ---- the shipped BiLSTM + query-decoder model (SURVEY.md 8(f) rank 2; src/benchmark/model.py:6-153), fp32 ------------ */
/* One bidirectional LSTM layer (replaces torch.nn.LSTM, model.py:16-23,49).  P: [.., 2*4H] = W_ih x + b_ih + b_hh for both
 * directions (gate rows i|f|g|o); w_hh: [2][4H][H] and its transpose w_hh_t: [2][H][4H]; out: [.., 2H]; saved: [2][B][T][5][H] (i, f, g, o, c) or NULL. */
int rs_lstm_fwd_f32(const float* P, int64_t p_ld, int64_t p_rows, int64_t p_row0, const float* w_hh, const float* w_hh_t,
                    float* out, int64_t o_ld, int64_t o_rows, int64_t o_row0, float* saved, int B, int T, int H,
                    void* stream);
/* w_hh: [2][4H][H]; dG: [.., 2*4H] gradient w.r.t. the gate pre-activations. */
int rs_lstm_bwd_f32(const float* d_out, int64_t do_ld, int64_t do_rows, int64_t do_row0, const float* saved,
                    const float* w_hh, float* dG, int64_t g_ld, int64_t g_rows, int64_t g_row0, int B, int T, int H,
                    void* stream);
/* bf16 tensor-core recurrence of the same layer, H = 128 only (d_model 256): any other H returns 1 and rs_last_error names the
 * limit.  Same P / out / saved / d_out / dG operands as the fp32 pair above; W_hh h_{t-1} and dG_t W_hh run with bf16 operands
 * and fp32 accumulation, everything else (gates, cell state, carries, stores) in fp32.  Pad rows of out and dG are not written;
 * no atomics (reruns are bit-identical).
 * rs_lstm_pack_weights_bf16 builds both weight images of a layer in one launch from W_hh of the forward (w_hh) and reverse
 * (w_hh_r) direction, [4H][H] fp32 each.  split = 0: one bf16 part per weight; split = 1: hi = bf16(w) then lo = bf16(w - hi),
 * which doubles K (the hi chunks come first, the lo chunks after them):
 *   fwd_img [2][16 (x2)][4H][8] bf16: element (d, part * 16 + c, n, e) = part of W_d[n][8 c + e]   (2 * 128 KB unsplit)
 *   bwd_img [2][64 (x2)][H][8]  bf16: element (d, part * 64 + c, u, e) = part of W_d[8 c + e][u]   (2 * 128 KB unsplit)
 * rs_lstm_fwd_bf16 reads fwd_img and rs_lstm_bwd_bf16 bwd_img, with the split flag they were packed with.  P, out, saved,
 * d_out and dG must be 16-byte aligned with row strides a multiple of 4 floats. */
int rs_lstm_pack_weights_bf16(const float* w_hh, const float* w_hh_r, int H, int split, void* fwd_img, void* bwd_img, void* stream);
int rs_lstm_fwd_bf16(const float* P, int64_t p_ld, int64_t p_rows, int64_t p_row0, const void* fwd_img, float* out,
                     int64_t o_ld, int64_t o_rows, int64_t o_row0, float* saved, int B, int T, int H, int split, void* stream);
int rs_lstm_bwd_bf16(const float* d_out, int64_t do_ld, int64_t do_rows, int64_t do_row0, const float* saved,
                     const void* bwd_img, float* dG, int64_t g_ld, int64_t g_rows, int64_t g_row0, int B, int T, int H, int split,
                     void* stream);
/* Per-trace normaliser (model.py:38-46): mean [B,3] of the valid (x, y, z), rms [B] of the centred (x, z) (floor 1e-3),
 * count [B] = max(valid tokens, 1).  traces: [B, N, F]; mask: [B, N] uint8 or NULL. */
int rs_trace_stats_f32(const float* traces, int F, const unsigned char* mask, int B, int N, float* mean, float* rms,
                       float* count, void* stream);
/* Query attention of SimpleQueryDecoder.forward (model.py:86-127) with the k/v projections folded into the query side:
 * scores = qk . m + qb (qk: [Q, D], qb: [Q], temperature and 1/sqrt(D) already applied), softmax over the valid tokens,
 * ctx [B,Q,D] = attn . memory, anchor [B,Q,3] = attn . (xyz - mean) / rms, summary [B,D] = masked mean of memory,
 * stats [B,Q,2] = softmax (max, sum).  workspace: rs_query_attn_workspace(B, Q, D, splits) floats. */
int64_t rs_query_attn_workspace(int B, int Q, int D, int splits);
int rs_query_attn_fwd_f32(const float* memory, int64_t m_ld, int64_t m_rows, int64_t m_row0, const float* traces, int F,
                          const unsigned char* mask, const float* mean, const float* rms, const float* qk, const float* qb,
                          int B, int N, int Q, int D, int splits, float* workspace, float* ctx, float* anchor,
                          float* summary, float* stats, void* stream);
/* d_memory: written ([.., D] rows; must be zero-filled when Q > 32); dq_part: [B*splits][Q][D+1] partial gradients of
 * (qk | qb), to be summed over the first axis. */
int rs_query_attn_bwd_f32(const float* memory, int64_t m_ld, int64_t m_rows, int64_t m_row0, const float* traces, int F,
                          const unsigned char* mask, const float* mean, const float* rms, const float* count,
                          const float* qk, const float* qb, const float* ctx, const float* anchor, const float* stats,
                          const float* d_ctx, const float* d_anchor, const float* d_summary, int B, int N, int Q, int D,
                          int splits, float* d_memory, int64_t dm_ld, int64_t dm_rows, int64_t dm_row0, float* dq_part,
                          void* stream);

/* ---- batched Hungarian matching + set loss (SURVEY.md 8(f) rank 3; src/benchmark/train.py:14-187) ------------------- */
/* pred_boxes [B,Q,6], pred_logits [B,Q,4], gt_boxes [B,M,6], gt_labels [B,M] int64, gt_valid [B,M] uint8 (Q <= 128,
 * M <= 64).  cost = w_class * (-softmax(logits)[label]) + w_box * L1(box) over the valid colliders (train.py:44-53);
 * optimal assignment per sample (= scipy.optimize.linear_sum_assignment, train.py:57).  Outputs, K = min(Q, M) per
 * sample, pairs ordered by query index, -1 padded: match_pred [B,K] query index, match_slot [B,K] collider slot,
 * match_rank [B,K] index among the sample's valid colliders (the reference's gt_idx), n_match [B]. */
int rs_hungarian_match(const float* pred_boxes, const float* pred_logits, const float* gt_boxes, const int64_t* gt_labels,
                       const unsigned char* gt_valid, int B, int Q, int M, float w_class, float w_box, int* match_pred,
                       int* match_slot, int* match_rank, int* n_match, void* stream);
/* SetCriterion.forward (train.py:109-187) on the matched pairs: losses[4] = cross-entropy, L1, 1 - GIoU (each a mean over
 * the batch-wide pairs) and the weighted total; g_logits [B,Q,4], g_l1 [B,Q,6], g_giou [B,Q,6] = gradients of the three
 * unweighted losses w.r.t. the predictions (zero for unmatched queries).  workspace: 1 + 3*B floats. */
int rs_set_loss_f32(const float* pred_boxes, const float* pred_logits, const float* gt_boxes, const int64_t* gt_labels, int B,
                    int Q, int M, const int* match_pred, const int* match_slot, const int* n_match, float w_class, float w_l1,
                    float w_giou, float* workspace, float* losses, float* g_logits, float* g_l1, float* g_giou, void* stream);

/* ---- batched evaluation (SURVEY.md 8(f) rank 4; src/benchmark/train.py:234-328, src/benchmark/inference.py:60-170) ---- */
/* counts[7] (double, device) += [sum of matched IoUs, matched pairs, TP (IoU >= thr), FP, FN (valid colliders without a
 * match), class hits, class total] of this batch; matches from rs_hungarian_match.  workspace: 7*B doubles. */
int rs_eval_pairs(const float* pred_boxes, const float* pred_logits, const float* gt_boxes, const int64_t* gt_labels,
                  const unsigned char* gt_valid, int B, int Q, int M, const int* match_pred, const int* match_slot,
                  const int* n_match, float iou_thresh, double* workspace, double* counts, void* stream);
/* post_process_predictions (inference.py:130-170): confidence = max softmax > conf_thr, then per-class greedy NMS (a box
 * is dropped when its IoU with a kept, more confident box of its class is >= nms_thr).  keep_idx [B,Q]: kept query
 * indices in the reference's output order (class 0..3, descending confidence), -1 padded; n_keep [B]; conf, label [B,Q]. */
int rs_nms_3d(const float* pred_boxes, const float* pred_logits, int B, int Q, float conf_thr, float nms_thr, int* keep_idx,
              int* n_keep, float* conf, int* label, void* stream);
/* True-positive flags for mAP: per scene, predictions in descending confidence claim the best-IoU unclaimed valid collider
 * of their predicted class; flag = 1 when that IoU >= iou_thr.  n_gt[4] += colliders per class. */
int rs_ap_flags(const float* pred_boxes, const float* pred_logits, const float* gt_boxes, const int64_t* gt_labels,
                const unsigned char* gt_valid, int B, int Q, int M, float iou_thr, int* flags, float* conf, int* label, int* n_gt,
                void* stream);

/* Evaluation of the README GRU model's slot outputs (README.md:93-132; BASELINE config 5), n_slots = B * max_objects:
 * 2-D axis-aligned IoU per slot, predicted class, conf = sigmoid(validity) * max class probability, flag = target slot
 * valid && class right && IoU >= iou_thr, n_gt[C] += valid target slots per class; counts[6] (double, device) +=
 * [IoU sum over valid slots, valid slots, class hits, validity hits, TP, predicted-valid].  workspace: 6 * 1184 doubles. */
int rs_slot_eval(const float* class_logits, const float* positions, const float* sizes, const float* validity_logits,
                 const int64_t* t_classes, const float* t_positions, const float* t_sizes, const float* t_valid,
                 int64_t n_slots, int C, float iou_thr, float* conf, int* label, int* flag, int* n_gt, double* workspace,
                 double* counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ROOMSLAM_B200_H */
