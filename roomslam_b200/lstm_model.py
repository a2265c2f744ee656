"""The model the upstream repository actually trains -- BiLSTM trace encoder + learnable-query attention decoder --
on the library's CUDA kernels (SURVEY.md 8(f) rank 2).

Drop-in for ``build_model(model_type='lstm')`` (src/benchmark/model.py:406-443): same constructor arguments, the same
``state_dict`` keys (src/benchmark/model.py:6-153), ``model(traces, mask) -> {'pred_boxes': [B,Q,6], 'pred_classes':
[B,Q,4]}``.  torch modules are used as parameter holders only; every FLOP that scales with the number of trace points
(input projection, LSTM projections and recurrence, output projection, attention over the memory) runs in
libroomslam_b200.so.  The per-query tail ([B, Q, D] tensors, ~1 % of the work) chains the library GEMM with torch
element-wise ops.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from . import functional as _F
from .functional import (_need_cuda, _p, _stream, _tc_ok, colsum, ktime, linear_nt, matmul_nn, matmul_tn, nt_tc, padded, split3,
                         tn_tc)



class LinearFn(torch.autograd.Function):
    """y[M, N] = x[M, K] @ w[N, K]^T + b.  Large M: bf16x6 tensor-core GEMMs; otherwise rs_sgemm.  Bias gradient: rs_colsum_f32."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, x, w, b, allow_tc=False):
        _need_cuda(x, w, b)
        x, w = x.contiguous().float(), w.contiguous().float()
        bias = b.contiguous().float() if b is not None else None
        y = torch.empty(x.shape[0], w.shape[0], device=x.device)
        ctx.tc = allow_tc and _tc_ok(x.shape[0], w.shape[0])
        if ctx.tc:
            x3, kp = split3(x)
            with ktime("gemm_tc_kernel(linear bf16x6)", 12.0 * x.shape[0] * w.shape[0] * kp):
                nt_tc(x3, split3(w, role_b=True)[0], bias, y)
            ctx.kp = kp
            ctx.save_for_backward(x3, w)
        else:
            with ktime("sgemm_kernel(linear)", 2.0 * x.shape[0] * w.shape[0] * w.shape[1]):
                linear_nt(x, w, bias, y)
            ctx.save_for_backward(x, w)
        ctx.has_bias = b is not None
        return y

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        dy = dy.contiguous().float()
        N, K = w.shape
        dx = dw = db = None
        if ctx.tc:
            dy3, kpy = split3(dy)
            if ctx.needs_input_grad[0]:
                dx = torch.empty(dy.shape[0], K, device=w.device)
                if K % 128 == 0:
                    with ktime("gemm_tc_kernel(linear bf16x6)", 12.0 * dy.shape[0] * K * kpy):
                        nt_tc(dy3, split3(w.t(), role_b=True)[0], None, dx)
                else:
                    matmul_nn(dy, w, dx)
            if ctx.needs_input_grad[1]:
                full = torch.zeros(N, ctx.kp, device=w.device)
                with ktime("gemm_tc_kernel(linear bf16x6)", 12.0 * dy.shape[0] * N * ctx.kp):
                    tn_tc(dy3, kpy, 0, N, x, ctx.kp, ctx.kp, full)
                dw = full[:, :K].contiguous()
        else:
            if ctx.needs_input_grad[0]:
                dx = torch.empty_like(x)
                matmul_nn(dy, w, dx)
            if ctx.needs_input_grad[1]:
                dw = torch.empty_like(w)
                matmul_tn(dy, x, dw)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = torch.empty(N, device=w.device)
            colsum(dy, db)
        return dx, dw, db, None


def linear(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor], allow_tc: bool = False) -> torch.Tensor:
    """allow_tc: the per-token projections (millions of rows) may use the bf16x6 tensor-core GEMM; the per-query tail
    ([B*Q, D] rows, ~1 % of the work) stays on the CUDA-core GEMM."""
    lead = x.shape[:-1]
    return LinearFn.apply(x.reshape(-1, x.shape[-1]), w, b, allow_tc).view(*lead, w.shape[0])


PRECISIONS = ("fp32", "bf16")
# Weight form of the bf16 recurrence: False = W_hh rounded to bf16 once, True = hi + lo bf16 parts (K doubles).  The
# cheapest form that keeps the model within 2e-2 of fp32 at 20 x 3000 (DESIGN.md section 7.2).
LSTM_BF16_SPLIT = False


def check_precision(precision: str, H: int) -> None:
    """ValueError for an unknown precision; RoomSlamError for "bf16" at a hidden size without a tensor-core kernel."""
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {PRECISIONS}, got {precision!r}")
    if precision == "bf16" and H != 128:
        raise _lib.RoomSlamError(f"precision='bf16': the tensor-core LSTM recurrence exists for d_model 256 (hidden size 128) "
                                 f"only, not d_model {2 * H}; use precision='fp32'")


def lstm_pack_bf16(w_hh, w_hh_r, split=None):
    """(fwd_img, bwd_img): the bf16 weight images rs_lstm_fwd_bf16 / rs_lstm_bwd_bf16 read (layouts in roomslam_b200.h),
    built from W_hh of both directions in one launch.  split None: LSTM_BF16_SPLIT."""
    split = LSTM_BF16_SPLIT if split is None else split
    w_hh, w_hh_r = w_hh.contiguous().float(), w_hh_r.contiguous().float()
    H = w_hh.shape[1]
    n = 2 * (1 + int(split)) * 4 * H * H
    fwd = torch.empty(n, dtype=torch.bfloat16, device=w_hh.device)
    bwd = torch.empty(n, dtype=torch.bfloat16, device=w_hh.device)
    _lib.call("rs_lstm_pack_weights_bf16", _p(w_hh), _p(w_hh_r), H, int(split), _p(fwd), _p(bwd), _stream(w_hh))
    return fwd, bwd


def lstm_layer_fwd(xin, mask, weights, need_grad=True, precision="fp32", images=None, split=None):
    """Forward of ONE bidirectional LSTM layer (the body of LSTMLayerFn.forward).

    xin (B, T+2, I) padded; mask (B, T, I) inter-layer dropout multiplier or None; weights = (w_ih, w_hh, b_ih, b_hh,
    w_ih_r, w_hh_r, b_ih_r, b_hh_r).  Returns (out (B, T+2, 2H) padded with zero pad rows, saved [2][B][T][5][H] (i, f,
    g, o, c; None unless need_grad), xin_saved, w_ih_cat [8H, I], w_hh_cat [2][4H][H], tc): xin_saved is the masked input
    the projection read, as its bf16x6 split when tc (the tensor-core path) is taken.
    precision "bf16" (H = 128 only) runs the recurrence on rs_lstm_fwd_bf16 with the weight images `images` (packed here
    with `split` when None; split None: LSTM_BF16_SPLIT); everything else is the same."""
    w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r = weights
    check_precision(precision, w_hh.shape[1])
    xin = xin.contiguous().float()
    B, Tp, I = xin.shape
    T, H = Tp - 2, w_hh.shape[1]
    dev, st = xin.device, _stream(xin)
    if mask is not None:
        xm = padded(B, T, I, dev)
        m = mask.contiguous().float()
        _lib.call("rs_seq_mul_f32", _p(xin), I, Tp, 1, _p(m), I, T, 0, _p(xm), I, Tp, 1, B, T, I, st)
        xin = xm
    w_ih_cat = torch.cat([w_ih, w_ih_r], 0).contiguous().float()              # [8H, I]
    w_hh_cat = torch.stack([w_hh, w_hh_r], 0).contiguous().float()            # [2, 4H, H]
    w_hh_t = w_hh_cat.transpose(1, 2).contiguous() if precision == "fp32" else None   # [2, H, 4H]
    bias = (torch.cat([b_ih, b_ih_r], 0) + torch.cat([b_hh, b_hh_r], 0)).contiguous().float()
    P = torch.empty(B, Tp, 8 * H, device=dev)
    tc = _tc_ok(B * Tp, I, 2 * H)
    if tc:
        xin3, kpi = split3(xin.view(B * Tp, I))
        with ktime("gemm_tc_kernel(lstm projection bf16x6)", 12.0 * B * Tp * 8 * H * kpi):
            nt_tc(xin3, split3(w_ih_cat, role_b=True)[0], bias, P.view(B * Tp, 8 * H))
    else:
        with ktime("sgemm_kernel(lstm projection)", 2.0 * B * Tp * 8 * H * I):
            linear_nt(xin.view(B * Tp, I), w_ih_cat, bias, P.view(B * Tp, 8 * H))
    out = padded(B, T, 2 * H, dev)
    saved = torch.empty(2, B, T, 5, H, device=dev) if need_grad else None
    if precision == "bf16":
        split = LSTM_BF16_SPLIT if split is None else split
        if images is None:
            images = lstm_pack_bf16(w_hh_cat[0], w_hh_cat[1], split)
        with ktime("lstm_fwd_bf16_kernel", 2.0 * B * T * 2 * 4 * H * H):
            _lib.call("rs_lstm_fwd_bf16", _p(P), 8 * H, Tp, 1, _p(images[0]), _p(out), 2 * H, Tp, 1, _p(saved), B, T, H, int(split), st)
    else:
        with ktime("lstm_fwd_f32_kernel", 2.0 * B * T * 2 * 4 * H * H):
            _lib.call("rs_lstm_fwd_f32", _p(P), 8 * H, Tp, 1, _p(w_hh_cat), _p(w_hh_t), _p(out), 2 * H, Tp, 1, _p(saved), B, T, H, st)
    del P
    return out, saved, (xin3 if tc else xin), w_ih_cat, w_hh_cat, tc


def lstm_bptt(d_out, saved, w_hh_cat, precision="fp32", w_img=None, split=None):
    """Backward through time of one layer: d_out (B, T+2, 2H) padded -> dG (B, T+2, 8H) padded (pad rows zero), the
    gradient w.r.t. the gate pre-activations, columns [forward i | f | g | o, reverse i | f | g | o].  precision "bf16":
    rs_lstm_bwd_bf16 with the backward weight image w_img (packed from w_hh_cat with `split` when None; split None:
    LSTM_BF16_SPLIT)."""
    _, B, T, _, H = saved.shape
    check_precision(precision, H)
    Tp = T + 2
    d_out = d_out.contiguous().float()
    dG = padded(B, T, 8 * H, d_out.device)
    if precision == "bf16":
        split = LSTM_BF16_SPLIT if split is None else split
        if w_img is None:
            w_img = lstm_pack_bf16(w_hh_cat[0], w_hh_cat[1], split)[1]
        with ktime("lstm_bwd_bf16_kernel", 2.0 * B * T * 2 * 4 * H * H):
            _lib.call("rs_lstm_bwd_bf16", _p(d_out), 2 * H, Tp, 1, _p(saved), _p(w_img), _p(dG), 8 * H, Tp, 1, B, T, H, int(split),
                      _stream(d_out))
        return dG
    with ktime("lstm_bwd_f32_kernel", 2.0 * B * T * 2 * 4 * H * H):
        _lib.call("rs_lstm_bwd_f32", _p(d_out), 2 * H, Tp, 1, _p(saved), _p(w_hh_cat), _p(dG), 8 * H, Tp, 1, B, T, H, _stream(d_out))
    return dG


def lstm_grads_from_dG(dG, out, xin_saved, w_ih_cat, mask, tc, need_dx=True):
    """Everything LSTMLayerFn.backward does after the BPTT: (dW_ih [8H, I], dW_hh [2][4H][H], db [8H], d_xin (B, T+2, I)
    or None).  db is the gradient of b_ih and of b_hh alike; d_xin is multiplied by the dropout mask at rows 1..T."""
    B, Tp, H8 = dG.shape
    T, H, I, M = Tp - 2, H8 // 8, w_ih_cat.shape[1], B * Tp
    dev, st = dG.device, _stream(dG)
    dG2, out2 = dG.view(M, 8 * H), out.view(M, 2 * H)
    # h_{t-1} of a step is the row before (forward) / after (reverse); the zero pad rows close the boundary
    if tc:
        dG3, kpg = split3(dG2)
        out3, kpo = split3(out2)
        kpi = xin_saved.shape[1] // 6
        dW_ih = torch.zeros(8 * H, I, device=dev)
        hh = torch.zeros(2, 4 * H, 2 * H, device=dev)
        with ktime("gemm_tc_kernel(lstm wgrad bf16x6)", 12.0 * M * 8 * H * (I + 2 * H)):
            tn_tc(dG3, kpg, 0, 8 * H, xin_saved, kpi, I, dW_ih)
            tn_tc(dG3, kpg, 0, 4 * H, out3, kpo, 2 * H, hh[0], a_shift=1, b_shift=0)
            tn_tc(dG3, kpg, 4 * H, 4 * H, out3, kpo, 2 * H, hh[1], a_shift=0, b_shift=1)
        dW_hh = torch.stack([hh[0, :, 0:H], hh[1, :, H:2 * H]], 0)
        del out3
    else:
        dW_ih = torch.empty(8 * H, I, device=dev)
        with ktime("sgemm_kernel(lstm wgrad)", 2.0 * M * 8 * H * (I + H)):
            matmul_tn(dG2, xin_saved.view(M, I), dW_ih)
            dW_hh = torch.empty(2, 4 * H, H, device=dev)
            matmul_tn(dG2[1:, 0:4 * H], out2[:M - 1, 0:H], dW_hh[0])
            matmul_tn(dG2[:M - 1, 4 * H:8 * H], out2[1:, H:2 * H], dW_hh[1])
    db = torch.empty(8 * H, device=dev)
    colsum(dG2, db)
    d_xin = None
    if need_dx:
        d_xin = torch.empty(B, Tp, I, device=dev)
        if tc:
            with ktime("gemm_tc_kernel(lstm dgrad bf16x6)", 12.0 * M * I * kpg):
                nt_tc(dG3, split3(w_ih_cat.t(), role_b=True)[0], None, d_xin.view(M, I))
        else:
            with ktime("sgemm_kernel(lstm dgrad)", 2.0 * M * 8 * H * I):
                matmul_nn(dG2, w_ih_cat, d_xin.view(M, I))
        if mask is not None:
            m = mask.contiguous().float()
            _lib.call("rs_seq_mul_f32", _p(d_xin), I, Tp, 1, _p(m), I, T, 0, _p(d_xin), I, Tp, 1, B, T, I, st)
    return dW_ih, dW_hh, db, d_xin


class LSTMLayerFn(torch.autograd.Function):
    """ONE bidirectional LSTM layer over the padded activation layout.

    apply(xin (B, T+2, I) padded, mask (B, T, I) or None, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r
          [, precision "fp32" | "bf16"])
        -> out (B, T+2, 2H) padded (pad rows zero).  Replaces one layer of torch.nn.LSTM (model.py:16-23).  With "bf16" the
    weight images are packed once per forward and kept for the backward pass."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, xin, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, precision="fp32"):
        _need_cuda(xin, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r)
        check_precision(precision, w_hh.shape[1])
        split = LSTM_BF16_SPLIT
        images = lstm_pack_bf16(w_hh, w_hh_r, split) if precision == "bf16" else None
        out, saved, xin_saved, w_ih_cat, w_hh_cat, tc = lstm_layer_fwd(
            xin, mask, (w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r), need_grad=any(ctx.needs_input_grad),
            precision=precision, images=images, split=split)
        ctx.split = split
        ctx.mask = mask
        ctx.tc = tc
        ctx.precision, ctx.w_img = precision, (images[1] if images is not None else None)
        ctx.save_for_backward(out, saved, xin_saved, w_ih_cat, w_hh_cat)
        return out

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_out):
        out, saved, xin_saved, w_ih_cat, w_hh_cat = ctx.saved_tensors
        if saved is None:
            raise RuntimeError("LSTMLayerFn: forward ran without saving activations (nothing required grad)")
        dG = lstm_bptt(d_out, saved, w_hh_cat, ctx.precision, ctx.w_img, ctx.split)
        dW_ih, dW_hh, db, d_xin = lstm_grads_from_dG(dG, out, xin_saved, w_ih_cat, ctx.mask, ctx.tc, ctx.needs_input_grad[0])
        H = w_hh_cat.shape[2]
        return (d_xin, None, dW_ih[:4 * H], dW_hh[0], db[:4 * H], db[:4 * H], dW_ih[4 * H:], dW_hh[1], db[4 * H:], db[4 * H:], None)


def _splits(B: int, N: int, Q: int) -> int:
    """Enough CTAs to fill 148 SMs twice when the batch is small (long traces are split flash-decoding style)."""
    qtiles = (Q + 31) // 32
    want = -(-2 * 148 // max(1, B * qtiles))
    return max(1, min(want, (N + 31) // 32))


def query_attn_fwd(memory, qk, qb, traces, mask_u8, mean, rms, splits=None):
    """Forward of the query attention (the body of QueryAttnFn.forward): memory padded (B, N+2, D), qk (Q, D), qb (Q,),
    traces (B, N, F), mask_u8 (B, N) or None, mean (B, 3), rms (B,) -> (ctx (B, Q, D), anchor (B, Q, 3), summary (B, D),
    stats (B, Q, 2) = per-query softmax (max, sum), splits).  splits defaults to what _splits picks for the shape."""
    memory, qk, qb = memory.contiguous().float(), qk.contiguous().float(), qb.contiguous().float()
    B, Np, D = memory.shape
    N, Q, Fdim = Np - 2, qk.shape[0], traces.shape[2]
    dev, st = memory.device, _stream(memory)
    splits = _splits(B, N, Q) if splits is None else splits
    ws = torch.empty(_lib.load().rs_query_attn_workspace(B, Q, D, splits), device=dev)
    ctx = torch.empty(B, Q, D, device=dev)
    anchor = torch.empty(B, Q, 3, device=dev)
    summary = torch.empty(B, D, device=dev)
    stats = torch.empty(B, Q, 2, device=dev)
    with ktime("query_attn_fwd_kernel", 4.0 * B * N * Q * D):
        _lib.call("rs_query_attn_fwd_f32", _p(memory), D, Np, 1, _p(traces), Fdim, _p(mask_u8), _p(mean), _p(rms), _p(qk),
                  _p(qb), B, N, Q, D, splits, _p(ws), _p(ctx), _p(anchor), _p(summary), _p(stats), st)
    return ctx, anchor, summary, stats, splits


def query_attn_bwd(memory, qk, qb, traces, mask_u8, mean, rms, count, ctx, anchor, stats, d_ctx, d_anchor, d_summary, splits):
    """Backward of the query attention (the body of QueryAttnFn.backward) -> (d_memory (B, N+2, D) padded with zero pad
    rows, dqk (Q, D), dqb (Q,)).  The kernel leaves per-(trace, split) partials of [dqk | dqb]; their column sum is the
    gradient.  d_ctx / d_anchor None stand for zeros, d_summary None for no summary gradient."""
    B, Np, D = memory.shape
    N, Q, Fdim = Np - 2, qk.shape[0], traces.shape[2]
    dev, st = memory.device, _stream(memory)
    d_ctx = d_ctx.contiguous().float() if d_ctx is not None else torch.zeros_like(ctx)
    d_anchor = d_anchor.contiguous().float() if d_anchor is not None else torch.zeros_like(anchor)
    d_summary = d_summary.contiguous().float() if d_summary is not None else None
    d_mem = torch.zeros(B, Np, D, device=dev) if Q > 32 else padded(B, N, D, dev)
    dq_part = torch.empty(B * splits, Q * (D + 1), device=dev)
    with ktime("query_attn_bwd_kernel", 10.0 * B * N * Q * D):
        _lib.call("rs_query_attn_bwd_f32", _p(memory), D, Np, 1, _p(traces), Fdim, _p(mask_u8), _p(mean), _p(rms), _p(count),
                  _p(qk), _p(qb), _p(ctx), _p(anchor), _p(stats), _p(d_ctx), _p(d_anchor), _p(d_summary), B, N, Q, D,
                  splits, _p(d_mem), D, Np, 1, _p(dq_part), st)
    dq = torch.empty(Q * (D + 1), device=dev)
    colsum(dq_part, dq)
    dq = dq.view(Q, D + 1)
    return d_mem, dq[:, :D].contiguous(), dq[:, D].contiguous()


class QueryAttnFn(torch.autograd.Function):
    """(memory padded (B, N+2, D), qk (Q, D), qb (Q,)) -> ctx (B, Q, D), anchor (B, Q, 3), summary (B, D).
    traces / mask / mean / rms / count are data (no gradient)."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx_, memory, qk, qb, traces, mask_u8, mean, rms, count):
        _need_cuda(memory, qk, qb, traces, mask_u8, mean, rms, count)
        memory, qk, qb = memory.contiguous().float(), qk.contiguous().float(), qb.contiguous().float()
        ctx, anchor, summary, stats, splits = query_attn_fwd(memory, qk, qb, traces, mask_u8, mean, rms)
        ctx_.save_for_backward(memory, qk, qb, traces, mask_u8, mean, rms, count, ctx, anchor, stats)
        ctx_.splits = splits
        return ctx, anchor, summary

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx_, d_ctx, d_anchor, d_summary):
        d_mem, dqk, dqb = query_attn_bwd(*ctx_.saved_tensors, d_ctx, d_anchor, d_summary, ctx_.splits)
        return d_mem, dqk, dqb, None, None, None, None, None


@_lib.on_tensor_device
def trace_stats(traces: torch.Tensor, mask_u8: Optional[torch.Tensor]):
    """Per-trace (mean (B,3), rms (B,), count (B,)) of model.py:38-46 in one launch."""
    B, N, Fdim = traces.shape
    mean = torch.empty(B, 3, device=traces.device)
    rms = torch.empty(B, device=traces.device)
    count = torch.empty(B, device=traces.device)
    _lib.call("rs_trace_stats_f32", _p(traces), Fdim, _p(mask_u8), B, N, _p(mean), _p(rms), _p(count), _stream(traces))
    return mean, rms, count


class _MLP2(nn.Module):
    """Parameter holder with the reference MLP's key names (layers.0 / layers.2; model.py:351-369)."""

    def __init__(self, d_in, d_hidden, d_out):
        super().__init__()
        self.layers = nn.Sequential(nn.Linear(d_in, d_hidden), nn.ReLU(), nn.Linear(d_hidden, d_out))

    def forward(self, x):
        return linear(torch.relu(linear(x, self.layers[0].weight, self.layers[0].bias)), self.layers[2].weight, self.layers[2].bias)


def _seq2(seq: nn.Sequential, x):
    return linear(torch.relu(linear(x, seq[0].weight, seq[0].bias)), seq[2].weight, seq[2].bias)


class LSTMTraceEncoder(nn.Module):
    """src/benchmark/model.py:6-57.  forward -> (memory padded (B, N+2, D), mean (B,3), rms (B,), count (B,)).
    precision "bf16" runs the LSTM recurrence on the tensor core (d_model 256 only); the parameters are the same."""

    def __init__(self, input_dim: int = 11, d_model: int = 128, num_layers: int = 2, dropout: float = 0.1, precision: str = "fp32"):
        super().__init__()
        if (d_model // 2) % 32 != 0 or d_model > 256:
            raise ValueError("d_model must be a multiple of 64, at most 256 (LSTM hidden size = d_model / 2 is a multiple of 32)")
        check_precision(precision, d_model // 2)
        self.precision = precision
        self.input_proj = nn.Linear(input_dim, d_model)
        self.lstm = nn.LSTM(input_size=d_model, hidden_size=d_model // 2, num_layers=num_layers,
                            dropout=dropout if num_layers > 1 else 0.0, batch_first=True, bidirectional=True)
        self.out_proj = nn.Linear(d_model, d_model)
        self.num_layers, self.dropout, self.d_model = num_layers, (dropout if num_layers > 1 else 0.0), d_model

    def forward(self, traces, mask_u8, dropout_mask=None):
        B, N, Fdim = traces.shape
        mean, rms, count = trace_stats(traces, mask_u8)
        xp = padded(B, N, Fdim, traces.device)
        xp[:, 1:N + 1] = traces
        cur = linear(xp, self.input_proj.weight, self.input_proj.bias, allow_tc=True)
        for l in range(self.num_layers):
            m = None
            if l > 0:
                if dropout_mask is not None:
                    m = dropout_mask[l - 1]
                elif self.training and self.dropout > 0:
                    keep = 1.0 - self.dropout
                    m = torch.bernoulli(torch.full((B, N, self.d_model), keep, device=traces.device)) / keep
            w = [getattr(self.lstm, f"{n}_l{l}{sfx}") for sfx in ("", "_reverse") for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")]
            cur = LSTMLayerFn.apply(cur, m, *w, self.precision)
        memory = linear(cur, self.out_proj.weight, self.out_proj.bias, allow_tc=True)          # pad rows hold the bias; never read as tokens
        return memory, mean, rms, count


class SimpleQueryDecoder(nn.Module):
    """src/benchmark/model.py:60-137 with the k/v projections folded into the query side (see csrc/query_attn.cu)."""

    def __init__(self, d_model: int = 128, num_queries: int = 30):
        super().__init__()
        self.num_queries = num_queries
        self.query_embed = nn.Embedding(num_queries, d_model)
        self.q_proj = nn.Linear(d_model, d_model)
        self.k_proj = nn.Linear(d_model, d_model)
        self.v_proj = nn.Linear(d_model, d_model)
        self.scale = d_model ** 0.5
        self.center_delta_head = _MLP2(d_model, d_model, 3)
        self.size_head = _MLP2(d_model, d_model, 3)
        self.class_head = nn.Linear(d_model, 4)
        self.gamma_mlp = nn.Sequential(nn.Linear(d_model, d_model), nn.ReLU(), nn.Linear(d_model, d_model))
        self.beta_mlp = nn.Sequential(nn.Linear(d_model, d_model), nn.ReLU(), nn.Linear(d_model, d_model))
        self.inv_temp = nn.Parameter(torch.tensor(1.0))

    def forward(self, memory, traces, mask_u8, mean, rms, count):
        q = linear(self.query_embed.weight, self.q_proj.weight, self.q_proj.bias)                 # (Q, D), batch independent
        tau = self.inv_temp / self.scale
        qk = linear(q, self.k_proj.weight.t().contiguous(), None) * tau                           # (q W_k) tau
        qb = (q * self.k_proj.bias).sum(-1) * tau
        ctx, anchor, summary = QueryAttnFn.apply(memory, qk, qb, traces, mask_u8, mean, rms, count)
        qfeat = linear(ctx, self.v_proj.weight, self.v_proj.bias)                                  # W_v (attn . m) + b_v
        gamma, beta = _seq2(self.gamma_mlp, summary), _seq2(self.beta_mlp, summary)
        decoded = qfeat * (1.0 + gamma.unsqueeze(1)) + beta.unsqueeze(1)
        scale, centre0 = rms.view(-1, 1, 1), mean.view(-1, 1, 3)
        centre = (anchor + self.center_delta_head(decoded)) * scale + centre0
        size = (F.softplus(self.size_head(decoded)) + 1e-4) * scale
        return torch.cat([centre, size], -1), linear(decoded, self.class_head.weight, self.class_head.bias)


class TraceToColliderLSTM(nn.Module):
    """src/benchmark/model.py:140-153.  ``forward(traces [B,N,11], mask [B,N] bool or None)``.  precision: "fp32" (default)
    or "bf16" (tensor-core LSTM recurrence, d_model 256 only); state_dicts interchange between the two."""

    def __init__(self, d_model: int = 128, num_queries: int = 30, lstm_layers: int = 2, dropout: float = 0.1, precision: str = "fp32"):
        super().__init__()
        self.encoder = LSTMTraceEncoder(11, d_model, lstm_layers, dropout, precision)
        self.decoder = SimpleQueryDecoder(d_model, num_queries)

    def forward(self, traces: torch.Tensor, mask: Optional[torch.Tensor] = None, dropout_mask=None) -> Dict[str, torch.Tensor]:
        if not traces.is_cuda:
            raise _lib.RoomSlamError("TraceToColliderLSTM runs on CUDA tensors only (no CPU fallback)")
        if traces.dim() != 3 or traces.shape[2] != 11:
            raise ValueError(f"expected traces of shape (B, N, 11), got {tuple(traces.shape)}")
        traces = traces.contiguous().float()
        mask_u8 = mask.to(torch.uint8).contiguous() if mask is not None else None
        memory, mean, rms, count = self.encoder(traces, mask_u8, dropout_mask)
        boxes, classes = self.decoder(memory, traces, mask_u8, mean, rms, count)
        return {"pred_boxes": boxes, "pred_classes": classes}


def build_model(num_queries: int = 80, d_model: int = 256, model_type: str = "lstm", lstm_layers: int = 2,
                dropout: float = 0.1, precision: str = "fp32", **unused):
    """Signature of src/benchmark/model.py:406-443; only the 'lstm' variant is on this library's path.  precision "bf16"
    (d_model 256) runs the LSTM recurrence on the tensor core."""
    if model_type.lower() != "lstm":
        raise ValueError("roomslam_b200.build_model implements model_type='lstm' only (the transformer variant is out of scope)")
    return TraceToColliderLSTM(d_model=d_model, num_queries=num_queries, lstm_layers=lstm_layers, dropout=dropout, precision=precision)
