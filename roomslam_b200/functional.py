"""autograd.Function wrappers that orchestrate the C-ABI kernels for the RoomSLAM model.

Host-side mirror of what torch.nn.GRU / nn.Linear / the loss functions do in the CPU reference
(oracle/room_slam_ref.py): same tensors in and out, but every FLOP runs in libroomslam_b200.so.
torch is used for device memory, streams and autograd bookkeeping only.

Activation layout ("padded"): every per-timestep activation lives in a (B, T+2, C) buffer whose rows 0 and T+1
of each trace are zero.  h_{t-1} of step t is then simply "the row before" (forward direction) or "the row
after" (reverse direction) for every t including the boundary, which lets dW_hh = sum_t dGh_t^T h_{t-1} run as
ONE time-parallel GEMM with a one-row pointer shift.
"""
from __future__ import annotations

import ctypes
import os
from typing import List, Optional, Tuple

import torch

from . import _lib

ACC, RELU = 1, 2
LOSS_WEIGHTS = (2.0, 5.0, 5.0, 1.0, 1.0)   # class, position, size, orientation, validity (decision D9)
_W5 = (ctypes.c_float * 5)(*LOSS_WEIGHTS)


# ---- optional per-kernel timing (CUDA events on the launch stream; used by bench.py for the roofline object) ----
_KT = {"on": False, "events": []}


class ktime:
    """with ktime("kernel name", algorithmic_flops): <one C-ABI call>"""

    def __init__(self, name: str, flops: float = 0.0):
        self.name, self.flops = name, flops

    def __enter__(self):
        if _KT["on"]:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _KT["on"]:
            self.e1.record()
            _KT["events"].append((self.name, self.e0, self.e1, self.flops))
        return False


def enable_kernel_timing(flag: bool):
    _KT["on"] = bool(flag)
    _KT["events"] = []
    return True


def collect_kernel_timing():
    """{kernel: [total ms, launches, total algorithmic flops]} since enable_kernel_timing(True)."""
    torch.cuda.synchronize()
    out = {}
    for name, e0, e1, fl in _KT["events"]:
        rec = out.setdefault(name, [0.0, 0, 0.0])
        rec[0] += e0.elapsed_time(e1)
        rec[1] += 1
        rec[2] += fl
    _KT["events"] = []
    return out


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _p(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.RoomSlamError("roomslam_b200 ops need CUDA tensors: there is no CPU fallback")


def sgemm(A, a_sm, a_sk, Bm, b_sk, b_sn, C, ldc, bias, M, N, K, flags=0):
    _lib.call("rs_sgemm", _p(A), a_sm, a_sk, _p(Bm), b_sk, b_sn, _p(C), ldc, _p(bias), M, N, K, flags, _stream(C))


def linear_nt(x2d: torch.Tensor, w: torch.Tensor, bias, out: torch.Tensor, flags=0):
    """out[M,N] = x2d[M,K] @ w[N,K]^T + bias."""
    M, K = x2d.shape
    N = w.shape[0]
    sgemm(x2d, x2d.stride(0), 1, w, 1, w.stride(0), out, out.stride(0), bias, M, N, K, flags)


def matmul_nn(a2d: torch.Tensor, w: torch.Tensor, out: torch.Tensor, flags=0):
    """out[M,N] = a2d[M,K] @ w[K,N]."""
    M, K = a2d.shape
    N = w.shape[1]
    sgemm(a2d, a2d.stride(0), 1, w, w.stride(0), 1, out, out.stride(0), None, M, N, K, flags)


def matmul_tn(a2d: torch.Tensor, b2d: torch.Tensor, out: torch.Tensor, flags=0):
    """out[M,N] = a2d[K,M]^T @ b2d[K,N]  (weight gradients: reduction over rows)."""
    K, M = a2d.shape
    N = b2d.shape[1]
    sgemm(a2d, 1, a2d.stride(0), b2d, b2d.stride(0), 1, out, out.stride(0), None, M, N, K, flags)


def colsum(a2d: torch.Tensor, out: torch.Tensor, accumulate=False):
    _lib.call("rs_colsum_f32", _p(a2d), a2d.stride(0), a2d.shape[0], a2d.shape[1], _p(out), int(accumulate), _stream(out))


# ---- fp32-accurate GEMMs on the bf16 tensor cores ("bf16x6", csrc/split_bf16.cu + csrc/gemm_tc.cu) -------------------
# Operands are split into bf16 (hi, mid, lo) triples; the six significant partial products run as ONE tcgen05 GEMM over a
# six times longer K (weight gradients: six accumulating passes over the thirds).  bf16 products are exact in the fp32
# accumulator, so the result is fp32-grade -- at tensor-core instead of CUDA-core speed.  Used when the row count is
# large enough to matter.
TC_MIN_ROWS = 4096
TC_ENABLED = os.environ.get("RS_TC_GEMM", "1") != "0"
OUT_F32 = 4
_HI, _MID, _LO = 5, 2, 0            # column sixths of an A-role buffer that hold hi, mid, lo


def _kpad(cols: int) -> int:
    return (cols + 127) // 128 * 128


def split3(x2d: torch.Tensor, role_b: bool = False):
    """fp32 [rows, cols] -> (bf16 [rows, 6*kpad], kpad) in the A-role or B-role layout of rs_split_bf16x6."""
    x2d = x2d.float()
    if x2d.stride(1) != 1:
        x2d = x2d.contiguous()
    if x2d.data_ptr() % 16:             # rows are read as float4; a parameter may be a view at any offset of a flat buffer
        x2d = x2d.clone()
    rows, cols = x2d.shape
    kp = _kpad(cols)
    out = torch.empty(rows, 6 * kp, dtype=torch.bfloat16, device=x2d.device)
    _lib.call("rs_split_bf16x6", _p(x2d), x2d.stride(0), rows, cols, kp, int(role_b), _p(out), 6 * kp, _stream(x2d))
    return out, kp


def nt_tc(a3: torch.Tensor, b3: torch.Tensor, bias, out: torch.Tensor):
    """out[M, N] (fp32) = A . B^T + bias from split operands (a3: [M, 6kp] A role, b3: [N, 6kp] B role); N % 128 == 0."""
    if bias is not None and bias.data_ptr() % 16:    # read as float4 (FlatParams views sit at any offset)
        bias = bias.clone()
    _lib.call("rs_gemm_bf16_nt", _p(a3), a3.stride(0), _p(b3), b3.stride(0), _p(out), out.stride(0), _p(bias), a3.shape[0],
              b3.shape[0], a3.shape[1], OUT_F32, _stream(out))


def tn_tc(a3, kpa, a_col0, m_out, b3, kpb, n_out, out, a_shift=0, b_shift=0):
    """out[m_out, n_out] (fp32, zero-initialised by the caller) += A[:, a_col0:a_col0+m_out]^T . B[:, :n_out], row r + a_shift
    of A paired with row r + b_shift of B; both operands in the A-role split layout."""
    rows = a3.shape[0] - max(a_shift, b_shift)
    order = ((_LO, _HI), (_HI, _LO), (_MID, _MID), (_MID, _HI), (_HI, _MID), (_HI, _HI))      # smallest products first
    a_seg = (ctypes.c_int * 6)(*[ta * kpa for ta, _ in order])
    b_seg = (ctypes.c_int * 6)(*[tb * kpb for _, tb in order])
    _lib.call("rs_gemm_bf16_tn_seg_acc", _p(a3), a3.stride(0), a3.shape[0], a_col0, a_shift, _p(b3), b3.stride(0), b3.shape[0], 0,
              b_shift, 6, ctypes.addressof(a_seg), ctypes.addressof(b_seg), _p(out), out.stride(0), m_out, n_out, rows, _stream(out))


def _tc_ok(rows: int, *dims128) -> bool:
    return TC_ENABLED and rows >= TC_MIN_ROWS and all(d % 128 == 0 for d in dims128)



def padded(B: int, T: int, C: int, device, dtype=torch.float32) -> torch.Tensor:
    buf = torch.empty(B, T + 2, C, device=device, dtype=dtype)
    buf[:, 0].zero_()
    buf[:, T + 1].zero_()
    return buf


class GRULayerFn(torch.autograd.Function):
    """ONE bidirectional GRU layer, fp32 kernels.

    apply(xin, meta, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r)
        -> (out_padded (B, T+2, 2H), h_n (2, B, H))
    meta = (padded_in, B, T[, lengths]); lengths: int32 (B,) valid steps per trace (packed-sequence semantics) or None.
    xin : padded_in False: the traces (B, T, I);  True: the padded output (B, T+2, I) of the layer below.
    mask: None or (B, T, I) dropout keep-mask (scaled by 1/(1-p)) applied to xin (decision D4).
    One Function per layer, so a layer's weight gradients are final (and can be all-reduced) while the
    backward-through-time of the layer below is still running."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, xin, meta, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r):
        # unused outputs (the top layer's sequence output feeds nothing: only h_n reaches the decoder) must arrive in
        # backward as None, not as a materialised 2 GB tensor of zeros that is then filled, converted and read back
        ctx.set_materialize_grads(False)
        _need_cuda(xin, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r)
        padded_in = meta[0]
        lengths = meta[3] if len(meta) > 3 else None
        xin = xin.contiguous().float()
        ctx.padded_in_orig = bool(padded_in)
        B, Il = xin.shape[0], xin.shape[2]
        T = xin.shape[1] - 2 if padded_in else xin.shape[1]
        H = w_hh.shape[1]
        dev = xin.device
        st = _stream(xin)
        need_grad = any(ctx.needs_input_grad)
        w_ih_cat = torch.cat([w_ih, w_ih_r], 0).contiguous()                # [6H, I_l]
        w_hh_cat = torch.stack([w_hh, w_hh_r], 0).contiguous()              # [2, 3H, H]
        w_hh_t = w_hh_cat.transpose(1, 2).contiguous()                      # [2, H, 3H]
        b_ih_cat = torch.cat([b_ih, b_ih_r], 0).contiguous()
        b_hh_cat = torch.cat([b_hh, b_hh_r], 0).contiguous()
        out = padded(B, T, 2 * H, dev)
        h_n = torch.empty(2, B, H, device=dev)
        gates = torch.empty(2, B, T, 4, H, device=dev) if need_grad else None
        if mask is not None:
            xm = padded(B, T, Il, dev)
            m = mask.contiguous().float()
            _lib.call("rs_seq_mul_f32", _p(xin), Il, xin.shape[1], 1 if padded_in else 0, _p(m), Il, T, 0, _p(xm), Il,
                      T + 2, 1, B, T, Il, st)
            xin, padded_in = xm, True
        rec_flops = 2.0 * B * T * 2 * 3 * H * H
        if Il <= 4:
            with ktime("gru_fwd_f32_kernel", rec_flops + 2.0 * B * T * 6 * H * Il):
                _lib.call("rs_gru_fwd_f32", _p(xin), Il, xin.shape[1], 1 if padded_in else 0, Il, _p(w_ih_cat),
                          _p(b_ih_cat), 0, 0, 0, 0, _p(w_hh_t), _p(b_hh_cat), _p(out), 2 * H, T + 2, 1, _p(h_n),
                          _p(gates), _p(lengths), B, T, H, st)
        else:
            if not padded_in:
                xp = padded(B, T, Il, dev)
                xp[:, 1:T + 1] = xin
                xin, padded_in = xp, True
            P = torch.empty(B, T + 2, 6 * H, device=dev)
            tc = _tc_ok(B * (T + 2), Il, H)
            if tc:      # fp32-grade GEMM on the bf16 tensor cores (split operands, see csrc/split_bf16.cu)
                xin3, kpi = split3(xin.view(B * (T + 2), Il))
                with ktime("gemm_tc_kernel(projection bf16x6)", 12.0 * B * (T + 2) * 6 * H * kpi):
                    nt_tc(xin3, split3(w_ih_cat, role_b=True)[0], b_ih_cat, P.view(B * (T + 2), 6 * H))
                del xin3
            else:
                with ktime("sgemm_kernel(projection)", 2.0 * B * (T + 2) * 6 * H * Il):
                    linear_nt(xin.view(B * (T + 2), Il), w_ih_cat, b_ih_cat, P.view(B * (T + 2), 6 * H))
            with ktime("gru_fwd_f32_kernel", rec_flops):
                _lib.call("rs_gru_fwd_f32", 0, 0, 0, 0, Il, 0, _p(b_ih_cat), _p(P), 6 * H, T + 2, 1, _p(w_hh_t),
                          _p(b_hh_cat), _p(out), 2 * H, T + 2, 1, _p(h_n), _p(gates), _p(lengths), B, T, H, st)
            del P
        ctx.dims = (B, T, Il, H)
        ctx.mask = mask
        ctx.lengths = lengths
        ctx.padded_in_saved = bool(padded_in)
        ctx.save_for_backward(out, gates, xin, w_ih_cat, w_hh_cat)   # outputs must go through save_for_backward (no ref cycle)
        return out, h_n

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_out, d_h_n):
        B, T, Il, H = ctx.dims
        out, gates, xin, w_ih_cat, w_hh_cat = ctx.saved_tensors
        padded_in = ctx.padded_in_saved
        if gates is None:
            raise RuntimeError("GRULayerFn: forward ran without saving activations (nothing required grad)")
        dev = out.device
        st = torch.cuda.current_stream(dev).cuda_stream
        Tp = T + 2
        M = B * Tp
        d_out = d_out.contiguous().float() if d_out is not None else None          # padded (B, T+2, 2H)
        d_h_n = d_h_n.contiguous().float() if d_h_n is not None else None
        dGx = padded(B, T, 6 * H, dev)
        dGh = padded(B, T, 6 * H, dev)
        with ktime("gru_bwd_f32_kernel", 2.0 * B * T * 2 * 3 * H * H):
            _lib.call("rs_gru_bwd_f32", _p(d_out), 2 * H, Tp, 1, _p(d_h_n), _p(gates), _p(out), 2 * H, Tp, 1,
                      _p(w_hh_cat), _p(dGx), _p(dGh), 6 * H, Tp, 1, _p(ctx.lengths), B, T, H, st)
        dGx2, dGh2, out2 = dGx.view(M, 6 * H), dGh.view(M, 6 * H), out.view(M, 2 * H)
        if not padded_in:                                # layer 0 with the fused projection: x is not padded
            xp = padded(B, T, Il, dev)
            xp[:, 1:T + 1] = xin
            xin = xp
        db_ih = torch.empty(6 * H, device=dev)
        colsum(dGx2, db_ih)
        db_hh = torch.empty(6 * H, device=dev)
        colsum(dGh2, db_hh)
        # hidden-side weight gradients: pair row r of dGh with row r-1 (forward) / r+1 (reverse) of out;
        # the zero pad rows make the boundary steps (h_prev = 0) come out right
        tc_hh = _tc_ok(M, H)                    # hidden-side GEMM shapes: 3H x 2H per direction
        tc_ih = tc_hh and Il % 128 == 0         # input-side: 6H x Il (layer 0 has Il = 2: CUDA cores)
        d_xin = dX = None
        if ctx.needs_input_grad[0]:
            dX = torch.empty(B, Tp, Il, device=dev)
        # fp32-grade GEMMs on the bf16 tensor cores where the shapes allow; the split copies are transient, one at a time
        if tc_ih:
            dGx3, kpg = split3(dGx2)
            x3, kpi = split3(xin.view(M, Il))
            dW_ih = torch.zeros(6 * H, Il, device=dev)
            with ktime("gemm_tc_kernel(wgrad bf16x6)", 12.0 * M * 6 * H * Il):
                tn_tc(dGx3, kpg, 0, 6 * H, x3, kpi, Il, dW_ih)
            del x3
            if dX is not None:
                with ktime("gemm_tc_kernel(dgrad bf16x6)", 12.0 * M * Il * kpg):
                    nt_tc(dGx3, split3(w_ih_cat.t(), role_b=True)[0], None, dX.view(M, Il))
            del dGx3
        else:
            dW_ih = torch.empty(6 * H, Il, device=dev)
            with ktime("sgemm_kernel(wgrad)", 2.0 * M * 6 * H * Il):
                matmul_tn(dGx2, xin.view(M, Il), dW_ih)      # both directions at once
            if dX is not None:
                with ktime("sgemm_kernel(dgrad)", 2.0 * M * 6 * H * Il):
                    matmul_nn(dGx2, w_ih_cat, dX.view(M, Il))    # pad rows of dGx are zero -> pad rows of dX are zero
        if tc_hh:
            dGh3, kph = split3(dGh2)
            out3, kpo = split3(out2)
            hh = torch.zeros(2, 3 * H, 2 * H, device=dev)
            with ktime("gemm_tc_kernel(wgrad bf16x6)", 12.0 * M * 6 * H * 2 * H):
                tn_tc(dGh3, kph, 0, 3 * H, out3, kpo, 2 * H, hh[0], a_shift=1, b_shift=0)
                tn_tc(dGh3, kph, 3 * H, 3 * H, out3, kpo, 2 * H, hh[1], a_shift=0, b_shift=1)
            dW_hh = torch.stack([hh[0, :, 0:H], hh[1, :, H:2 * H]], 0)
            del dGh3, out3
        else:
            dW_hh = torch.empty(2, 3 * H, H, device=dev)
            with ktime("sgemm_kernel(wgrad)", 2.0 * M * 6 * H * H):
                matmul_tn(dGh2[1:, 0:3 * H], out2[:M - 1, 0:H], dW_hh[0])
                matmul_tn(dGh2[:M - 1, 3 * H:6 * H], out2[1:, H:2 * H], dW_hh[1])
        if dX is not None:
            if ctx.mask is not None:
                m = ctx.mask.contiguous().float()
                _lib.call("rs_seq_mul_f32", _p(dX), Il, Tp, 1, _p(m), Il, T, 0, _p(dX), Il, Tp, 1, B, T, Il, st)
            d_xin = dX if ctx.padded_in_orig else dX[:, 1:T + 1, :]
        return (d_xin, None, None, dW_ih[:3 * H], dW_hh[0], db_ih[:3 * H], db_hh[:3 * H],
                dW_ih[3 * H:], dW_hh[1], db_ih[3 * H:], db_hh[3 * H:])


def gru_encoder(x, mask, num_layers, weights, layer_fn=None, lengths=None, split_weights=False, mask_in_bptt=False):
    """Stack of bidirectional layers -> (out (B,T,2H) of the top layer, h_n (2L,B,H)), torch.nn.GRU semantics
    (with `lengths`: those of a packed sequence).  mask_in_bptt (bf16 layers): the backward half of inter-layer dropout runs
    inside the BPTT kernel of the producing layer instead of the dgrad epilogue of the consuming one (tests)."""
    layer_fn = layer_fn or GRULayerFn
    B, T = x.shape[0], x.shape[1]
    cur, padded_in, h_all = x, False, []
    if lengths is not None:
        lengths = lengths.to(device=x.device, dtype=torch.int32).contiguous()
    # bf16 layers take dropout as packed bits on the PRODUCING layer (the recurrence kernel writes out (.) mask itself);
    # the fp32 layers multiply their input by the float mask.  `mask` is either a float tensor (L-1, B, T, 2H) or, for the
    # bf16 path, a list of (bits, scale) pairs per layer boundary.
    bits_mode = isinstance(mask, (list, tuple))
    if layer_fn is not GRULayerFn and not bits_mode:
        from .functional_bf16 import drop_bits_from_mask
        mask = [drop_bits_from_mask(mask[l]) for l in range(num_layers - 1)] if mask is not None else [None] * num_layers
        bits_mode = True
    for l in range(num_layers):
        if bits_mode:
            drop = mask[l] if l < num_layers - 1 else None
            in_drop = mask[l - 1] if (l > 0 and not mask_in_bptt) else None   # the consumer masks its data gradient
            cur, h_n = layer_fn.apply(cur, (padded_in, B, T, lengths, drop, split_weights, in_drop, mask_in_bptt), None,
                                      *weights[8 * l: 8 * l + 8])
            padded_in = True
            h_all.append(h_n)
            continue
        m = mask[l - 1] if (mask is not None and l > 0) else None
        cur, h_n = layer_fn.apply(cur, (padded_in, B, T, lengths), m, *weights[8 * l: 8 * l + 8])
        padded_in = True
        h_all.append(h_n)
    h_n = torch.cat(h_all, 0) if num_layers > 1 else h_all[0]
    if cur.dim() == 5:                       # bf16 mode: tile-major -> (B, T, 2H); only materialised when it is used
        from . import layout
        return _LazyOut(cur, B, T), h_n
    return cur[:, 1:T + 1, :], h_n


class _LazyOut:
    """Top-layer output of the bf16 mode, kept tile-major until somebody asks for the (B, T, 2H) tensor."""

    def __init__(self, tm, B, T):
        self.tm, self.B, self.T = tm, B, T

    def materialize(self) -> torch.Tensor:
        from . import layout
        return layout.from_tile_major(self.tm, self.B, self.T).float()


def heads_split(raw: torch.Tensor, N: int, C: int):
    """raw [B, N*(C+6)] fp32 (columns class | pos | size | orient | valid) -> (cls, pos, size, orient, valid):
    rs_heads_split_f32, sizes = softplus(raw) + 1e-4."""
    B, dev = raw.shape[0], raw.device
    out = (torch.empty(B, N, C, device=dev), torch.empty(B, N, 2, device=dev), torch.empty(B, N, 2, device=dev),
           torch.empty(B, N, device=dev), torch.empty(B, N, device=dev))
    _lib.call("rs_heads_split_f32", _p(raw), B, N, C, *[_p(t) for t in out], _stream(raw))
    return out


def heads_merge(raw: torch.Tensor, N: int, C: int, d_cls, d_pos, d_size, d_orient, d_valid) -> torch.Tensor:
    """The gradients of the five prediction tensors (None: zero) -> d_raw [B, N*(C+6)]: rs_heads_merge_bwd_f32."""
    c = lambda t: t.contiguous().float() if t is not None else None  # noqa: E731
    d_raw = torch.empty_like(raw)
    _lib.call("rs_heads_merge_bwd_f32", _p(raw), raw.shape[0], N, C, _p(c(d_cls)), _p(c(d_pos)), _p(c(d_size)),
              _p(c(d_orient)), _p(c(d_valid)), _p(d_raw), _stream(raw))
    return d_raw


def decoder_fwd(latent, N, C, W1, b1, W2, b2, heads):
    """Forward of DecoderFn.  Returns a dict: the saved operands latent, W1, W2, Wh, the intermediates f1, f2, raw and
    heads = (cls, pos, size, orient, valid)."""
    latent = latent.contiguous().float()
    B = latent.shape[0]
    dev = latent.device
    Wh = torch.cat(heads[0::2], 0).contiguous()      # [N*(C+6), D]
    bh = torch.cat(heads[1::2], 0).contiguous()
    D1, D2, NH = W1.shape[0], W2.shape[0], Wh.shape[0]
    f1 = torch.empty(B, D1, device=dev)
    f2 = torch.empty(B, D2, device=dev)
    raw = torch.empty(B, NH, device=dev)
    with ktime("decoder_fwd(sgemm x3)", 2.0 * B * (latent.shape[1] * D1 + D1 * D2 + D2 * NH)):
        linear_nt(latent, W1.contiguous(), b1, f1, RELU)
        linear_nt(f1, W2.contiguous(), b2, f2, RELU)
        linear_nt(f2, Wh, bh, raw)
    return dict(latent=latent, W1=W1, W2=W2, Wh=Wh, f1=f1, f2=f2, raw=raw, heads=heads_split(raw, N, C))


def decoder_bwd(latent, W1, W2, Wh, f1, f2, d_raw):
    """Backward of DecoderFn from d_raw [B, NH].  Returns a dict of dWh, dbh, df2 (after the ReLU mask), dW2, db2, df1,
    dW1, db1, dlat."""
    dev = latent.device
    st = _stream(latent)
    kt = ktime("decoder_bwd(sgemm x6)", 4.0 * latent.shape[0] * (latent.shape[1] * W1.shape[0] + W1.shape[0] * W2.shape[0] + W2.shape[0] * Wh.shape[0]))
    kt.__enter__()
    dWh = torch.empty_like(Wh)
    matmul_tn(d_raw, f2, dWh)
    dbh = torch.empty(Wh.shape[0], device=dev)
    colsum(d_raw, dbh)
    df2 = torch.empty_like(f2)
    matmul_nn(d_raw, Wh, df2)
    _lib.call("rs_relu_bwd_f32", _p(df2), _p(f2), _p(df2), df2.numel(), st)
    dW2 = torch.empty_like(W2)
    matmul_tn(df2, f1, dW2)
    db2 = torch.empty(W2.shape[0], device=dev)
    colsum(df2, db2)
    df1 = torch.empty_like(f1)
    matmul_nn(df2, W2.contiguous(), df1)
    _lib.call("rs_relu_bwd_f32", _p(df1), _p(f1), _p(df1), df1.numel(), st)
    dW1 = torch.empty_like(W1)
    matmul_tn(df1, latent, dW1)
    db1 = torch.empty(W1.shape[0], device=dev)
    colsum(df1, db1)
    dlat = torch.empty_like(latent)
    matmul_nn(df1, W1.contiguous(), dlat)
    kt.__exit__(None, None, None)
    return dict(dWh=dWh, dbh=dbh, df2=df2, dW2=dW2, db2=db2, df1=df1, dW1=dW1, db1=db1, dlat=dlat)


def split_head_grads(dWh, dbh, head_rows):
    """Row blocks of the stacked head gradients, one (dW, db) pair per head."""
    out, r0 = [], 0
    for rows in head_rows:
        out += [dWh[r0:r0 + rows], dbh[r0:r0 + rows]]
        r0 += rows
    return out


class DecoderFn(torch.autograd.Function):
    """MLP trunk (2 x Linear+ReLU) + five heads, fp32.
    apply(latent, N, C, W1, b1, W2, b2, Wc, bc, Wp, bp, Ws, bs, Wo, bo, Wv, bv) -> 5 prediction tensors."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, latent, N, C, W1, b1, W2, b2, *heads):
        _need_cuda(latent, W1, W2, *heads)
        r = decoder_fwd(latent, N, C, W1, b1, W2, b2, heads)
        ctx.save_for_backward(r["latent"], W1, W2, r["Wh"], r["f1"], r["f2"], r["raw"])
        ctx.dims = (N, C)
        ctx.head_rows = [h.shape[0] for h in heads[0::2]]
        return r["heads"]

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_cls, d_pos, d_size, d_orient, d_valid):
        latent, W1, W2, Wh, f1, f2, raw = ctx.saved_tensors
        N, C = ctx.dims
        d_raw = heads_merge(raw, N, C, d_cls, d_pos, d_size, d_orient, d_valid)
        g = decoder_bwd(latent, W1, W2, Wh, f1, f2, d_raw)
        return (g["dlat"], None, None, g["dW1"], g["db1"], g["dW2"], g["db2"], *split_head_grads(g["dWh"], g["dbh"], ctx.head_rows))


def loss_fwd(cls, pos, size, orient, vlogit, t_cls, t_pos, t_size, t_orient, t_valid):
    """rs_loss_fwd_f32.  Returns (losses[6] fp32, sums[6] fp64, g = [g_cls, g_pos, g_size, g_orient, g_valid]): the six
    un-normalised sums and the per-element gradients that loss_bwd scales."""
    B, N, C = cls.shape
    dev = cls.device
    f = lambda t: t.contiguous().float()  # noqa: E731
    cls, pos, size, orient, vlogit = f(cls), f(pos), f(size), f(orient), f(vlogit)
    t_cls = t_cls.contiguous().long()
    t_pos, t_size, t_orient, t_valid = f(t_pos), f(t_size), f(t_orient), f(t_valid)
    sums = torch.empty(6, dtype=torch.float64, device=dev)
    losses = torch.empty(6, device=dev)
    g = [torch.empty_like(t) for t in (cls, pos, size, orient, vlogit)]
    _lib.call("rs_loss_fwd_f32", _p(cls), _p(pos), _p(size), _p(orient), _p(vlogit), _p(t_cls), _p(t_pos),
              _p(t_size), _p(t_orient), _p(t_valid), B, N, C, ctypes.addressof(_W5), _p(sums), _p(losses),
              *[_p(t) for t in g], _stream(cls))
    return losses, sums, g


def loss_bwd(sums, g, d_losses):
    """rs_loss_bwd_f32: the gradients of the five prediction tensors for the incoming d(losses)[6]."""
    B, N, C = g[0].shape
    d_losses = d_losses.contiguous().float()
    d = [torch.empty_like(t) for t in g]
    _lib.call("rs_loss_bwd_f32", _p(sums), _p(d_losses), B, N, C, ctypes.addressof(_W5), *[_p(t) for t in g],
              *[_p(t) for t in d], _stream(sums))
    return d


class MultiTaskLossFn(torch.autograd.Function):
    """apply(cls, pos, size, orient, valid_logits, t_cls, t_pos, t_size, t_orient, t_valid) -> losses[6]
    = [total, class, position, size, orientation, validity] (README.md:122-125, weights D9)."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, cls, pos, size, orient, vlogit, t_cls, t_pos, t_size, t_orient, t_valid):
        _need_cuda(cls, pos, size, orient, vlogit, t_cls, t_pos, t_size, t_orient, t_valid)
        losses, sums, g = loss_fwd(cls, pos, size, orient, vlogit, t_cls, t_pos, t_size, t_orient, t_valid)
        ctx.save_for_backward(sums, *g)
        return losses

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_losses):
        sums, *g = ctx.saved_tensors
        return (*loss_bwd(sums, g, d_losses), None, None, None, None, None)
