"""bf16 tensor-core mode of the GRU encoder: orchestration of the tcgen05 kernels (hidden_size = 128; 256: GRULayerBF16WideFn).

Per layer:   layer 0: fused K=2 input projection inside the recurrence kernel
             deeper : input projection fused into the recurrence kernel (W_ih resident, X_t bulk-copied one step ahead);
                      with split (hi + lo) weights below 1024 traces: P = X W_ih^T + b by rs_blk_gemm_nt, then the recurrence
             recurrence forward                  rs_rec_fwd_bf16  (persistent CTA pairs, W_hh resident in shared memory)
backward:    recurrence backward (BPTT)          rs_rec_bwd_bf16  -> dG (r | z | n | hn gate gradients); W_hn h recomputed
             dW_ih, dW_hh, bias gradients        rs_blk_wgrad     (one launch per layer, 12 roles over dG)
             dX     = dG[r,z,n] W_ih             rs_blk_gemm_nt / rs_blk_gemm_nt_drop (x the dropout mask of the layer input)
All per-timestep activations stay in the tile-major bf16 layout (roomslam_b200/layout.py); master weights and
weight gradients are fp32.  Tolerance against the fp32 CPU oracle: 2e-2 relative (BASELINE.json north_star).
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

from . import _lib
from . import functional as F_
from . import layout as L
from .functional import _need_cuda, _p, _stream, ktime

H = 128

# Layer-0 input columns (csrc/rec_common.cuh): W_ih x + b rides on the recurrence MMA as x_steps(I) extra K = 16 steps.
# Input i takes the 3 columns x_col(i, 0..2) (x hi, lo, hi against W_ih hi, hi, lo), the bias columns 6 and 7 (1, 1 against
# b hi, lo); every other column is zero.  Inputs 0, 1 and the bias fill the first 8 columns exactly as with 2 inputs.
MAX_X_INPUTS = 16


def x_col(i: int, k: int) -> int:
    return 3 * i + k if i < 2 else 8 + 3 * (i - 2) + k


def x_steps(I: int) -> int:
    return (3 * I + 2 + 15) // 16


def _check_x_inputs(I: int):
    if I > MAX_X_INPUTS:
        raise _lib.RoomSlamError(f"bf16 mode fuses the layer-0 projection into the recurrence for input_size <= {MAX_X_INPUTS} "
                                 f"(got {I}); use precision='fp32'")


def _nt(A, a_cols, kchunks, W_tiled, n_tiles, C, c_cols, c_chunk0, bias, n_blocks, st, drop=None, T=0):
    """drop = (bits, scale): the result is multiplied by that dropout mask in the epilogue (data gradient of a layer whose
    input went through inter-layer dropout; no bias then)."""
    kch = L.int_array(kchunks)
    if drop is not None:
        _lib.call("rs_blk_gemm_nt_drop", _p(A), a_cols, ctypes.addressof(kch), len(kchunks), _p(W_tiled), n_tiles, _p(C), c_cols,
                  c_chunk0, n_blocks, _p(drop[0]), _p(drop[1]), T, st)
        return
    _lib.call("rs_blk_gemm_nt", _p(A), a_cols, ctypes.addressof(kch), len(kchunks), _p(W_tiled), n_tiles, _p(C), c_cols,
              c_chunk0, _p(bias), n_blocks, st)


def _tn(A, a_cols, mchunks, rows, Bm, b_cols, b_chunk0, n_cols, shift, bcast, C, ldc, tiles, T, st):
    mch, r0 = L.int_array(mchunks), L.int_array(rows)
    _lib.call("rs_blk_gemm_tn_acc", _p(A), a_cols, ctypes.addressof(mch), ctypes.addressof(r0), len(mchunks), _p(Bm), b_cols,
              b_chunk0, n_cols, shift, int(bcast), _p(C), ldc, tiles, T, st)


def _wgrad(dG, a_cols, ones, roles, tiles, T, st):
    """roles: list of (a_mchunk, B tensor or None, b_cols, b_chunk0, n_cols, b_shift, C view or None, ldc, bias view or None,
    B2 tensor or None, C2 view or None)."""
    n = len(roles)
    vp = ctypes.c_void_p * n
    i64 = ctypes.c_int64 * n
    a_m = L.int_array([r[0] for r in roles])
    ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
    Bp = vp(*[ptr(r[1]) for r in roles])
    b_cols = i64(*[r[2] for r in roles])
    b_c0 = L.int_array([r[3] for r in roles])
    n_cols = L.int_array([r[4] for r in roles])
    shift = L.int_array([r[5] for r in roles])
    Cp = vp(*[ptr(r[6]) for r in roles])
    ldc = i64(*[r[7] for r in roles])
    bias = vp(*[ptr(r[8]) for r in roles])
    B2p = vp(*[ptr(r[9]) for r in roles])
    C2p = vp(*[ptr(r[10]) for r in roles])
    adr = ctypes.addressof
    _lib.call("rs_blk_wgrad", _p(dG), a_cols, _p(ones), n, adr(a_m), adr(Bp), adr(b_cols), adr(b_c0), adr(n_cols), adr(shift),
              adr(Cp), adr(ldc), adr(bias), adr(B2p), adr(C2p), tiles, T, st)


_ONES = {}


def _ones_block(device):
    """One tile-major block with 16 columns whose first column is 1: B operand that turns a TN GEMM into column sums."""
    key = str(device)
    if key not in _ONES:
        blk = torch.zeros(2, L.TILE, 8, device=device, dtype=torch.bfloat16)
        blk[0, :, 0] = 1.0
        _ONES[key] = blk
    return _ONES[key]


@_lib.on_tensor_device
def drop_bits_from_mask(mask: torch.Tensor):
    """(B, T, C) fp32 dropout mask (0 or 1/keep, decision D4) -> (bits uint8 [tiles][T][128][C/8], scale (1,) fp32)."""
    B, T, C = mask.shape
    m = mask.contiguous().float()
    bits = torch.empty(L.n_tiles(B), T, L.TILE, C // 8, device=m.device, dtype=torch.uint8)
    scale = torch.empty(1, device=m.device)
    _lib.call("rs_pack_drop_mask", _p(m), B, T, C, _p(bits), _p(scale), _stream(m))
    return bits, scale


def gen_drop_bits(B: int, T: int, C: int, keep: float, seed: int, device):
    """Bernoulli(keep) dropout bits drawn on the device (no (B, T, C) float mask ever exists) -> (bits, scale)."""
    bits = torch.empty(L.n_tiles(B), T, L.TILE, C // 8, device=device, dtype=torch.uint8)
    scale = torch.empty(1, device=device)
    with torch.cuda.device(bits.device):
        _lib.call("rs_gen_drop_bits", _p(bits), B, T, C, float(keep), int(seed), _p(scale), _stream(bits))
    return bits, scale


def unpack_drop_bits(bits: torch.Tensor, scale: torch.Tensor, B: int) -> torch.Tensor:
    """The (B, T, C) float mask a (bits, scale) pair stands for (tests; the oracle takes the float mask)."""
    tiles, T, _, cb = bits.shape
    b = bits.to(torch.int32).unsqueeze(-1) >> torch.arange(8, device=bits.device, dtype=torch.int32)
    m = (b & 1).to(torch.float32).reshape(tiles, T, L.TILE, cb * 8) * scale
    return m.permute(0, 2, 1, 3).reshape(tiles * L.TILE, T, cb * 8)[:B].contiguous()


class GRULayerBF16Fn(torch.autograd.Function):
    """apply(xin, meta, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r) -> (out tile-major bf16, h_n (2,B,H) fp32)
    meta = (padded_in, B, T, lengths, drop, split, in_drop).  padded_in False: xin is the raw trace batch (B, T, I) fp32
    (layer 0); True: xin is the tile-major bf16 output of the layer below.  drop = None or (bits, scale) from
    `drop_bits_from_mask` / `gen_drop_bits`: inter-layer dropout on THIS layer's output -- the returned sequence is then
    out (.) mask (written by the recurrence kernel next to out).  Its backward half belongs to the CONSUMER: the layer above
    gets the same pair as in_drop and multiplies its data gradient dX by the mask in the epilogue of the dgrad GEMM (a
    throughput-bound kernel), so the gradient arriving here is already masked and the mask tests stay out of the serial
    per-time-step chain of the BPTT kernel (-0.5 ms per step at 8192 traces).  meta[7] = True restores in-kernel masking of
    the incoming gradient (a caller that feeds this layer's output to something else than the next layer).  `mask` (the
    fp32 path's float mask on the layer INPUT) must be None here."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, xin, meta, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r):
        # unused outputs (the top layer's sequence output feeds nothing: only h_n reaches the decoder) must arrive in
        # backward as None, not as a materialised 2 GB tensor of zeros that is then filled, converted and read back
        ctx.set_materialize_grads(False)
        _need_cuda(xin, mask, w_ih, w_hh)
        padded_in, B, T = meta[:3]
        lengths = meta[3] if len(meta) > 3 else None
        drop = meta[4] if len(meta) > 4 else None
        split = 1 if (len(meta) > 5 and meta[5]) else 0      # weights as bf16 pairs hi + lo (small batches; csrc/pack_w.cu)
        ctx.in_drop = meta[6] if len(meta) > 6 else None     # mask on this layer's INPUT: applied to dX in backward
        ctx.mask_d_out = bool(meta[7]) if len(meta) > 7 else False
        if mask is not None:
            raise _lib.RoomSlamError("GRULayerBF16Fn: pass dropout as packed bits on the producing layer (meta[4]), not as a float mask")
        if w_hh.shape[1] != H:
            raise _lib.RoomSlamError(f"bf16 mode is built for hidden_size = {H} (got {w_hh.shape[1]}); use precision='fp32'")
        dev = xin.device
        st = _stream(xin)
        need_grad = any(ctx.needs_input_grad)
        tiles = L.n_tiles(B)
        Il = w_ih.shape[1]
        with torch.no_grad():
            # every bf16 operand image of the layer (forward AND backward) in one launch, from the fp32 master weights
            ws = [t.detach().float().contiguous() for t in (w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r)]
            bf = torch.bfloat16
            need_dx = padded_in and ctx.needs_input_grad[0]
            # deeper layers: the input projection is fused into the recurrence kernel (W_ih resident next to W_hh, no P in HBM,
            # no projection GEMM) whenever the weights are not split into hi + lo pairs (W_ih hi + lo would not fit).  Since the
            # X tile copies are issued by one elected thread the fused kernel is within 6 % of the plain one per time step, and
            # the projection launch it replaces costs more than that at every batch size (training step at 1024 / 2048 / 4096 /
            # 8192 traces: 5.85 -> 5.72, 6.83 -> 6.52, 9.55 -> 8.93, 19.6 -> 18.3 ms).  RS_FUSE_PROJ=0/1 forces.
            fuse_env = os.environ.get("RS_FUSE_PROJ")
            fuse_proj = padded_in and not split and (fuse_env == "1" if fuse_env in ("0", "1") else True)
            if not padded_in:
                _check_x_inputs(Il)
            x_chunks = 2 * x_steps(Il) if not padded_in else (2 if fuse_proj else 0)   # input columns (layer 0) / bias (fused)
            whh_img = torch.empty(2, (H // 8) * (1 + split) + x_chunks, 3 * H, 8, device=dev, dtype=bf)
            b_hn = torch.empty(2, H, device=dev)
            bias_x = torch.empty(2, 3 * H, device=dev)
            wt = torch.empty(6 * H // 128, (Il // 64) * (1 + split), 8, L.TILE, 8, device=dev, dtype=bf) if (padded_in and not fuse_proj) else None
            wih_img = torch.empty(2, Il // 8, 3 * H, 8, device=dev, dtype=bf) if fuse_proj else None
            whhT_img = torch.empty(2, (3 * H // 8) * (1 + split), H, 8, device=dev, dtype=bf)
            wt_dgrad = torch.empty(Il // 128, (6 * H // 64) * (1 + split), 8, L.TILE, 8, device=dev, dtype=bf) if need_dx else None
            if padded_in and Il != 2 * H:
                raise _lib.RoomSlamError("bf16 mode: deeper layers take the 2H-column output of the layer below")
            wp = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in ws])
            _lib.call("rs_gru_pack_weights_bf16", ctypes.addressof(wp), H, Il, split, _p(whh_img), _p(b_hn), _p(bias_x), _p(wt), _p(whhT_img),
                      _p(wt_dgrad), _p(wih_img), st)
            # (the recurrence kernels zero the pad rows t' = 0, T + 1 of what they write)
            out = L.empty_tm(B, T, 2 * H, dev, zero_pads=False)
            out_drop = L.empty_tm(B, T, 2 * H, dev, zero_pads=False) if drop is not None else None
            d_bits, d_scale = drop if drop is not None else (None, None)
            h_n = torch.empty(2, B, H, device=dev)
            gates = torch.empty(tiles, T, 2, 48, L.TILE, 8, device=dev, dtype=torch.bfloat16) if need_grad else None   # r | z | n
            rec_flops = 2.0 * B * T * 2 * 3 * H * H
            X = None
            if not padded_in:
                x = xin.contiguous().float()
                with ktime("rec_fwd_pair_kernel", rec_flops + 2.0 * B * T * 6 * H * Il):
                    _lib.call("rs_rec_fwd_bf16", _p(x), Il, 0, 0, 0, 0, _p(whh_img), _p(b_hn), _p(out), _p(gates), _p(h_n), _p(lengths),
                              _p(d_bits), _p(d_scale), _p(out_drop), split, B, T, st)
                saved_in = x
            elif fuse_proj:
                X = xin
                with ktime("rec_fwd_pair_kernel", rec_flops + 2.0 * B * T * 6 * H * Il):
                    _lib.call("rs_rec_fwd_bf16", 0, 0, 0, 0, _p(X), _p(wih_img), _p(whh_img), _p(b_hn), _p(out), _p(gates), _p(h_n),
                              _p(lengths), _p(d_bits), _p(d_scale), _p(out_drop), 0, B, T, st)
                saved_in = X
            else:
                X = xin
                P = torch.empty(tiles, T + 2, 6 * H // 8, L.TILE, 8, device=dev, dtype=torch.bfloat16)
                with ktime("blk_gemm_nt_kernel(projection)", 2.0 * tiles * L.TILE * (T + 2) * 6 * H * Il):
                    _nt(X, Il, [8 * k for k in range(Il // 64)] * (1 + split), wt, 6, P, 6 * H, 0, bias_x.reshape(-1).contiguous(),
                        tiles * (T + 2), st)
                with ktime("rec_fwd_pair_kernel", rec_flops):
                    _lib.call("rs_rec_fwd_bf16", 0, 0, _p(P), 6 * H, 0, 0, _p(whh_img), _p(b_hn), _p(out), _p(gates), _p(h_n), _p(lengths),
                              _p(d_bits), _p(d_scale), _p(out_drop), split, B, T, st)
                del P
                saved_in = X
        ctx.meta = (padded_in, B, T, Il, split)
        ctx.drop = drop
        ctx.lengths = lengths
        # save_for_backward (not ctx attributes): `out` is an OUTPUT of this node; holding it in a plain attribute
        # would create a reference cycle node -> out -> grad_fn -> node and keep gigabytes alive until the cycle GC runs
        ctx.save_for_backward(out, gates, saved_in, whhT_img, wt_dgrad, whh_img, b_hn)
        if out_drop is not None:
            return out_drop, h_n
        return out, h_n

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_out, d_h_n):
        padded_in, B, T, Il, split = ctx.meta
        out, gates, saved_in, whhT_img, wt_dgrad, whh_img, b_hn = ctx.saved_tensors
        if gates is None:
            raise RuntimeError("GRULayerBF16Fn: forward ran without saving activations (nothing required grad)")
        dev = out.device
        st = torch.cuda.current_stream(dev).cuda_stream
        tiles = L.n_tiles(B)
        with torch.no_grad():
            d_out = d_out.contiguous().to(torch.bfloat16) if d_out is not None else None
            d_h_n = d_h_n.contiguous().float() if d_h_n is not None else None
            dG = torch.empty(tiles, T + 2, 8 * H // 8, L.TILE, 8, device=dev, dtype=torch.bfloat16)
            with ktime("rec_bwd_pair_kernel", 2.0 * B * T * 2 * 3 * H * H):
                d_bits, d_scale = ctx.drop if (ctx.drop is not None and ctx.mask_d_out) else (None, None)
                _lib.call("rs_rec_bwd_bf16", _p(d_out), _p(d_h_n), _p(gates), _p(out), _p(whhT_img), _p(whh_img), whh_img.shape[1],
                          _p(b_hn), _p(dG), _p(ctx.lengths), _p(d_bits), _p(d_scale), split, B, T, st)
            dW_ih, dW_hh, db_ih, db_hh, d_xin = grads_from_dG_128(dG, out, saved_in, padded_in, B, T, Il, split, wt_dgrad,
                                                                  ctx.in_drop, padded_in and ctx.needs_input_grad[0])
            dW_ih = dW_ih[:, :Il].contiguous() if not padded_in else dW_ih
        return (d_xin, None, None, dW_ih[:3 * H], dW_hh[0], db_ih[0], db_hh[0], dW_ih[3 * H:], dW_hh[1], db_ih[1], db_hh[1])


def grads_from_dG_128(dG, out, saved_in, padded_in, B, T, Il, split, wt_dgrad, in_drop, need_dx):
    """Everything GRULayerBF16Fn's backward computes from the BPTT's dG [tiles][T + 2][8H / 8][128][8] (per direction
    r | z | n | hn): -> (dW_ih (6H, Il; layer 0: (6H, 16), the columns >= Il zero), dW_hh (2, 3H, H), db_ih (2, 3H), db_hh (2, 3H), dX tile-major or None), each
    direction's rows in torch.nn.GRU's r | z | n order.  out: the layer's tile-major output; saved_in: the raw (B, T, Il)
    fp32 input (layer 0, padded_in False) or the tile-major input X; wt_dgrad: the dgrad image of rs_gru_pack_weights_bf16
    (used when need_dx); in_drop: (bits, scale) of the dropout on the layer input, applied to dX, or None."""
    dev = dG.device
    st = torch.cuda.current_stream(dev).cuda_stream
    tiles = L.n_tiles(B)
    # ALL weight / bias gradients of the layer in one fused pass over dG (12 roles, see csrc/gemm_blk.cu):
    #   ih roles (dir, g in r,z,n): dG block ^T . X            -> dW_ih rows, bias sums of r, z, n
    #   hh roles (dir, g in r,z,hn): dG block ^T . h(t' -/+ 1) -> dW_hh rows, bias sum of hn
    dW_hh = torch.zeros(2, 3 * H, H, device=dev)
    sums = torch.zeros(2, 4, H, device=dev)              # per direction: r | z | n | hn column sums of dG
    roles = []
    if not padded_in:
        # layer 0: the input has <= 16 columns -> it rides along as the 16-column second B source of the r, z and n roles
        xa_tm = torch.empty(tiles, T + 2, 2, L.TILE, 8, device=dev, dtype=torch.bfloat16)
        _lib.call("rs_pack_x_tm", _p(saved_in), B, T, Il, _p(xa_tm), st)
        dW_ih_buf = torch.zeros(6 * H, 16, device=dev)
        for d in (0, 1):
            sh = -1 if d == 0 else 1
            for g in (0, 1):                               # r, z: hidden-side block + input-side columns + bias sum
                roles.append((d * 64 + g * 16, out, 2 * H, d * 16, H, sh, dW_hh[d, g * H:], H, sums[d, g],
                              xa_tm, dW_ih_buf[(d * 3 + g) * H:]))
            roles.append((d * 64 + 48, out, 2 * H, d * 16, H, sh, dW_hh[d, 2 * H:], H, sums[d, 3], None, None))   # hn
            roles.append((d * 64 + 32, None, 0, 0, 0, 0, None, 0, sums[d, 2], xa_tm, dW_ih_buf[(d * 3 + 2) * H:]))  # n
        flops = 2.0 * tiles * L.TILE * T * (6 * H * 16 + 6 * H * H + 8 * H * 16)
    else:
        # deeper layers: 12 roles: ih (N = 2H) and hh (N = H) per gate block.  (18 equal-weight N = H roles were
        # tried to keep the roles in lockstep for L2 sharing: slower, 6.1 ms vs 5.5 ms - more L2->SM traffic.)
        # Roles 2 j, 2 j + 1 run as a CTA pair; where both name the same dG block (r, z) it is loaded once and
        # multicast into both CTAs (csrc/gemm_blk.cu, paired mode).
        dW_ih_buf = torch.zeros(6 * H, Il, device=dev)
        for d in (0, 1):
            sh = -1 if d == 0 else 1
            ih = lambda g: (d * 64 + g * 16, saved_in, Il, 0, Il, 0, dW_ih_buf[(d * 3 + g) * H:], Il, sums[d, g], None, None)  # noqa: E731
            hh = lambda gi, g: (d * 64 + g * 16, out, 2 * H, d * 16, H, sh, dW_hh[d, gi * H:], H,                           # noqa: E731
                                sums[d, 3] if g == 3 else None, None, None)
            roles += [ih(0), hh(0, 0), ih(1), hh(1, 1), ih(2), hh(2, 3)]   # (r, X) (r, h) | (z, X) (z, h) | (n, X) (hn, h)
        flops = 2.0 * tiles * L.TILE * T * (6 * H * Il + 6 * H * H + 8 * H * 16)
    with ktime("blk_wgrad_kernel", flops):
        _wgrad(dG, 8 * H, _ones_block(dev), roles, tiles, T, st)
    db_ih = sums[:, :3].reshape(2, 3 * H)
    db_hh = torch.cat([sums[:, :2].reshape(2, 2 * H), sums[:, 3]], 1)
    dX = None
    if need_dx:
        dX = torch.empty(tiles, T + 2, Il // 8, L.TILE, 8, device=dev, dtype=torch.bfloat16)
        kch = [d * 64 + g * 16 + hf * 8 for d in (0, 1) for g in (0, 1, 2) for hf in (0, 1)]   # wt_dgrad: [Il/128][12][8][128][8]
        with ktime("blk_gemm_nt_kernel(dgrad)", 2.0 * tiles * L.TILE * (T + 2) * 6 * H * Il):
            _nt(dG, 8 * H, kch * (1 + split), wt_dgrad, Il // 128, dX, Il, 0, None, tiles * (T + 2), st, in_drop, T)
    return dW_ih_buf, dW_hh, db_ih, db_hh, dX


def wide_fwd_image(w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r, layer0: bool):
    """The forward operands of GRULayerBF16WideFn from the fp32 master weights (torch.nn.GRU layout, both directions):
    -> (wst, b_hn, bias_x, w_ih_fwd, w_ih_cat, w_hh_cat).  wst is the streaming W_hh image of rs_rec_fwd_bf16_wide
    [2 dirs][2 ranks][K steps][2][384][8] bf16 (r, z rows scaled by 1/2; layer 0: then the input columns of x_col, hi / lo
    split, and a zero K step up to whole stages); b_hn [2][H]; bias_x [2][3H] (b_ih + b_hh on r, z, b_ih on n, scaled like
    the rows); w_ih_fwd [2][3H][I] the scaled W_ih of the projection GEMM; w_ih_cat [6H][I] and w_hh_cat [2][3H][H] unscaled."""
    HW = w_hh.shape[1]
    dev, bf = w_hh.device, torch.bfloat16
    Il = w_ih.shape[1]
    half = torch.ones(3 * HW, device=dev)
    half[:2 * HW] = 0.5
    w_hh_cat = torch.stack([w_hh, w_hh_r], 0).float()                      # [2, 3H, H]
    w_ih_cat = torch.cat([w_ih, w_ih_r], 0).float()                        # [6H, Il]
    b_hn = torch.stack([b_hh[2 * HW:], b_hh_r[2 * HW:]], 0).float().contiguous()
    bias_x = torch.stack([b_ih, b_ih_r], 0).float().clone()
    bias_x[0, :2 * HW] += b_hh[:2 * HW]
    bias_x[1, :2 * HW] += b_hh_r[:2 * HW]
    bias_x *= half[None, :]
    whs = w_hh_cat * half[None, :, None]
    w_ih_fwd = (w_ih_cat.view(2, 3 * HW, Il) * half[None, :, None])
    rows = lambda t, r: torch.cat([t[:, g * HW + 128 * r: g * HW + 128 * r + 128] for g in range(3)], 1)   # noqa: E731
    per_rank = []
    for r in (0, 1):
        img = rows(whs, r).view(2, 384, HW // 16, 2, 8).permute(0, 2, 3, 1, 4)          # [2][16 K steps][2 chunks][384][8]
        if layer0:
            xs = x_steps(Il)
            w_hi = w_ih_fwd.to(bf).float()
            b_hi = bias_x.to(bf).float()
            xcols = torch.zeros(2, 3 * HW, 16 * xs, device=dev)           # the input columns (see x_col)
            for c in range(Il):
                xcols[:, :, x_col(c, 0)] = w_hi[:, :, c]
                xcols[:, :, x_col(c, 1)] = w_hi[:, :, c]
                xcols[:, :, x_col(c, 2)] = w_ih_fwd[:, :, c] - w_hi[:, :, c]
            xcols[:, :, 6] = b_hi
            xcols[:, :, 7] = bias_x - b_hi
            xstep = rows(xcols, r).view(2, 384, xs, 2, 8).permute(0, 2, 3, 1, 4)        # the input K steps
            pad = torch.zeros(2, xs % 2, 2, 384, 8, device=dev)                          # + a zero K step: full stages
            img = torch.cat([img, xstep, pad], 1)
        per_rank.append(img)
    wst = torch.stack(per_rank, 1).to(bf).contiguous()                     # [2 dirs][2 ranks][K steps][2][384][8]
    return wst, b_hn, bias_x, w_ih_fwd, w_ih_cat, w_hh_cat


def wide_bwd_image(w_hh_cat):
    """W_hh^T as rs_rec_bwd_bf16_wide streams it: [2 dirs][2 ranks][48 K steps][2 chunks][128 rows][8] bf16, rows = hidden
    units [128 rank, 128 rank + 128), K = the 3H gate rows r | z | n (unscaled)."""
    HW = w_hh_cat.shape[2]
    whhT = w_hh_cat.transpose(1, 2)                                        # [2, H, 3H]
    return torch.stack([whhT[:, 128 * r: 128 * r + 128].reshape(2, 128, 3 * HW // 16, 2, 8).permute(0, 2, 3, 1, 4)
                        for r in (0, 1)], 1).to(torch.bfloat16).contiguous()   # [2][2][48 K steps][2][128][8]


class GRULayerBF16WideFn(torch.autograd.Function):
    """GRULayerBF16Fn for hidden_size = 256 (BASELINE config 4).  Same tile-major operands and the same GEMM kernels; the
    recurrence runs on csrc/rec_wide.cu, which streams W_hh from L2 (it no longer fits in shared memory).  The GEMM calls are
    cut to the kernels' limits (<= 1024 output columns per projection launch, <= 18 weight-gradient roles of <= 256 columns
    per launch).  The weight images are laid out with torch ops here: a step of this configuration takes ~100 ms."""

    HW = 256

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, xin, meta, mask, w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r):
        ctx.set_materialize_grads(False)
        _need_cuda(xin, w_ih, w_hh)
        HW = GRULayerBF16WideFn.HW
        padded_in, B, T = meta[:3]
        lengths = meta[3] if len(meta) > 3 else None
        drop = meta[4] if len(meta) > 4 else None
        ctx.in_drop = meta[6] if len(meta) > 6 else None     # see GRULayerBF16Fn
        ctx.mask_d_out = bool(meta[7]) if len(meta) > 7 else False
        if mask is not None:
            raise _lib.RoomSlamError("GRULayerBF16WideFn: pass dropout as packed bits on the producing layer (meta[4])")
        if w_hh.shape[1] != HW:
            raise _lib.RoomSlamError(f"GRULayerBF16WideFn is built for hidden_size = {HW}")
        dev, st, bf = xin.device, _stream(xin), torch.bfloat16
        need_grad = any(ctx.needs_input_grad)
        tiles, Il = L.n_tiles(B), w_ih.shape[1]
        with torch.no_grad():
            if not padded_in:
                _check_x_inputs(Il)
            wst, b_hn, bias_x, w_ih_fwd, w_ih_cat, w_hh_cat = wide_fwd_image(w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r,
                                                                             not padded_in)
            out = L.empty_tm(B, T, 2 * HW, dev, zero_pads=False)
            out_drop = L.empty_tm(B, T, 2 * HW, dev, zero_pads=False) if drop is not None else None
            d_bits, d_scale = drop if drop is not None else (None, None)
            h_n = torch.empty(2, B, HW, device=dev)
            gates = torch.empty(tiles, T, 2, 4 * HW // 8, L.TILE, 8, device=dev, dtype=bf) if need_grad else None
            rec_flops = 2.0 * B * T * 2 * 3 * HW * HW
            if not padded_in:
                x = xin.contiguous().float()
                with ktime("rec_fwd_wide_kernel", rec_flops + 2.0 * B * T * 6 * HW * Il):
                    _lib.call("rs_rec_fwd_bf16_wide", _p(x), Il, 0, _p(wst), _p(b_hn), _p(out), _p(gates), _p(h_n), _p(lengths),
                              _p(d_bits), _p(d_scale), _p(out_drop), B, T, st)
                saved_in = x
            else:
                if Il != 2 * HW:
                    raise _lib.RoomSlamError("bf16 mode: deeper layers take the 2H-column output of the layer below")
                P = wide_projection(xin, w_ih_fwd, bias_x, B, T)
                with ktime("rec_fwd_wide_kernel", rec_flops):
                    _lib.call("rs_rec_fwd_bf16_wide", 0, 0, _p(P), _p(wst), _p(b_hn), _p(out), _p(gates), _p(h_n), _p(lengths),
                              _p(d_bits), _p(d_scale), _p(out_drop), B, T, st)
                del P
                saved_in = xin
        ctx.meta = (padded_in, B, T, Il)
        ctx.drop, ctx.lengths = drop, lengths
        ctx.save_for_backward(out, gates, saved_in, w_ih_cat, w_hh_cat)
        return (out_drop if out_drop is not None else out), h_n

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_out, d_h_n):
        HW = GRULayerBF16WideFn.HW
        padded_in, B, T, Il = ctx.meta
        out, gates, saved_in, w_ih_cat, w_hh_cat = ctx.saved_tensors
        if gates is None:
            raise RuntimeError("GRULayerBF16WideFn: forward ran without saving activations (nothing required grad)")
        dev, bf = out.device, torch.bfloat16
        st = torch.cuda.current_stream(dev).cuda_stream
        tiles, HC = L.n_tiles(B), HW // 8
        with torch.no_grad():
            d_out = d_out.contiguous().to(bf) if d_out is not None else None
            d_h_n = d_h_n.contiguous().float() if d_h_n is not None else None
            wtst = wide_bwd_image(w_hh_cat)
            dG = torch.empty(tiles, T + 2, 8 * HC, L.TILE, 8, device=dev, dtype=bf)
            d_bits, d_scale = ctx.drop if (ctx.drop is not None and ctx.mask_d_out) else (None, None)
            with ktime("rec_bwd_wide_kernel", 2.0 * B * T * 2 * 3 * HW * HW):
                _lib.call("rs_rec_bwd_bf16_wide", _p(d_out), _p(d_h_n), _p(gates), _p(out), _p(wtst), _p(dG), _p(ctx.lengths),
                          _p(d_bits), _p(d_scale), B, T, st)
            dW_ih, dW_hh, db_ih, db_hh, d_xin = grads_from_dG_256(dG, out, saved_in, padded_in, B, T, Il, w_ih_cat, ctx.in_drop,
                                                                  padded_in and ctx.needs_input_grad[0])
            dW_ih = dW_ih[:, :Il].contiguous() if not padded_in else dW_ih
        return (d_xin, None, None, dW_ih[:3 * HW], dW_hh[0], db_ih[0], db_hh[0], dW_ih[3 * HW:], dW_hh[1], db_ih[1], db_hh[1])


def wide_projection(X, w_ih_fwd, bias_x, B, T):
    """The input projection of a deeper H = 256 layer: P = X W_ih^T + b over all T + 2 rows of the tile-major X (Il
    columns), tile-major bf16 with 6H columns.  w_ih_fwd (2, 3H, Il) and bias_x (2, 3H) as wide_fwd_image returns them;
    the 1536 output columns take two launches of 768 (the second writes from chunk 96 on)."""
    HW, Il = GRULayerBF16WideFn.HW, X.shape[2] * 8
    tiles = L.n_tiles(B)
    P = torch.empty(tiles, T + 2, 6 * HW // 8, L.TILE, 8, device=X.device, dtype=torch.bfloat16)
    wt = L.tile_weight_nt(w_ih_fwd.reshape(6 * HW, Il))                # [12][Il/64][8][128][8]
    bias_flat = bias_x.reshape(-1).contiguous()
    with ktime("blk_gemm_nt_kernel(projection)", 2.0 * tiles * L.TILE * (T + 2) * 6 * HW * Il):
        for part in (0, 1):
            _nt(X, Il, [8 * k for k in range(Il // 64)], wt[6 * part: 6 * part + 6].contiguous(), 6, P, 6 * HW,
                96 * part, bias_flat[768 * part: 768 * part + 768].contiguous(), tiles * (T + 2), _stream(X))
    return P


def grads_from_dG_256(dG, out, saved_in, padded_in, B, T, Il, w_ih_cat, in_drop, need_dx):
    """grads_from_dG_128 for GRULayerBF16WideFn: the same outputs at H = 256.  w_ih_cat (6H, Il): the unscaled fp32 W_ih
    of both directions (wide_fwd_image), whose bf16 image the dgrad multiplies."""
    HW = GRULayerBF16WideFn.HW
    dev, bf = dG.device, torch.bfloat16
    st = torch.cuda.current_stream(dev).cuda_stream
    tiles, HC = L.n_tiles(B), HW // 8
    dW_hh = torch.zeros(2, 3 * HW, HW, device=dev)
    sums = torch.zeros(2, 4, HW, device=dev)             # per direction: r | z | n | hn column sums of dG
    ones = _ones_block(dev)
    if not padded_in:
        xa_tm = torch.empty(tiles, T + 2, 2, L.TILE, 8, device=dev, dtype=bf)
        _lib.call("rs_pack_x_tm", _p(saved_in), B, T, Il, _p(xa_tm), st)
        dW_ih_buf = torch.zeros(6 * HW, 16, device=dev)
    else:
        dW_ih_buf = torch.zeros(6 * HW, Il, device=dev)
    flops = 2.0 * tiles * L.TILE * T * (6 * HW * (Il if padded_in else 16) + 6 * HW * HW + 8 * HW * 16)
    with ktime("blk_wgrad_kernel", flops):
        for d in (0, 1):                                 # one launch per direction: <= 18 roles of one 128-row gate block
            sh = -1 if d == 0 else 1
            roles, hh_roles = [], []
            for mb in (0, 1):                            # the two 128-row halves of a 256-row gate block
                m0 = mb * 128
                if not padded_in:
                    for g in (0, 1):
                        roles.append((d * 4 * HC + g * HC + mb * 16, out, 2 * HW, d * HC, HW, sh, dW_hh[d, g * HW + m0:], HW,
                                      sums[d, g, m0:], xa_tm, dW_ih_buf[(d * 3 + g) * HW + m0:]))
                    roles.append((d * 4 * HC + 3 * HC + mb * 16, out, 2 * HW, d * HC, HW, sh, dW_hh[d, 2 * HW + m0:], HW,
                                  sums[d, 3, m0:], None, None))
                    roles.append((d * 4 * HC + 2 * HC + mb * 16, None, 0, 0, 0, 0, None, 0, sums[d, 2, m0:], xa_tm,
                                  dW_ih_buf[(d * 3 + 2) * HW + m0:]))
                else:
                    for g in (0, 1, 2):                  # r, z, n against the layer input, 256 columns at a time: the two
                        for nb in range(Il // 256):      # halves of Il are adjacent roles = one CTA pair sharing its dG block
                            roles.append((d * 4 * HC + g * HC + mb * 16, saved_in, Il, nb * 32, 256, 0,
                                          dW_ih_buf[(d * 3 + g) * HW + m0:, nb * 256:], Il, sums[d, g, m0:] if nb == 0 else None,
                                          None, None))
                    for gi, g in enumerate((0, 1, 3)):   # r, z, hn against the shifted hidden state
                        hh_roles.append((d * 4 * HC + g * HC + mb * 16, out, 2 * HW, d * HC, HW, sh, dW_hh[d, gi * HW + m0:], HW,
                                         sums[d, 3, m0:] if g == 3 else None, None, None))
            _wgrad(dG, 8 * HW, ones, roles + hh_roles, tiles, T, st)
    db_ih = sums[:, :3].reshape(2, 3 * HW)
    db_hh = torch.cat([sums[:, :2].reshape(2, 2 * HW), sums[:, 3]], 1)
    dX = None
    if need_dx:
        dX = torch.empty(tiles, T + 2, Il // 8, L.TILE, 8, device=dev, dtype=bf)
        wt = L.tile_weight_nt(w_ih_cat.t().contiguous())                   # [Il/128][6H/64][8][128][8]
        kch = [d * 4 * HC + g * HC + hf * 8 for d in (0, 1) for g in (0, 1, 2) for hf in range(HW // 64)]
        with ktime("blk_gemm_nt_kernel(dgrad)", 2.0 * tiles * L.TILE * (T + 2) * 6 * HW * Il):
            _nt(dG, 8 * HW, kch, wt, Il // 128, dX, Il, 0, None, tiles * (T + 2), st, in_drop, T)
    return dW_ih_buf, dW_hh, db_ih, db_hh, dX


def _gemm_nt(A, Bw, C, bias, flags=0):
    """C[M,N] = act(A[M,K] . Bw[N,K]^T + bias): TMA-fed tcgen05 GEMM (csrc/gemm_tc.cu)."""
    M, K = A.shape
    N = Bw.shape[0]
    _lib.call("rs_gemm_bf16_nt", _p(A), A.stride(0), _p(Bw), Bw.stride(0), _p(C), C.stride(0), _p(bias), M, N, K, flags, _stream(C))


def _gemm_tn(A, Bm, C):
    """C[M,N] (fp32) += A[rows,M]^T . Bm[rows,N]."""
    rows, M = A.shape
    N = Bm.shape[1]
    _lib.call("rs_gemm_bf16_tn_acc", _p(A), A.stride(0), rows, 0, 0, _p(Bm), Bm.stride(0), rows, 0, 0, _p(C), C.stride(0), M, N,
              rows, _stream(C))


RELU, OUT_F32 = 2, 4


def decoder_bf16_fwd(latent, N, C, W1, b1, W2, b2, heads):
    """Forward of DecoderBF16Fn.  The head rows are stacked into Wh [NHp, D2] (bf16) and bh [NHp] with zero rows up to
    NHp = ceil(N (C + 6) / 128) 128.  Returns a dict: the GEMM operands lat, W1b, W2b (bf16), Wh, bh, the intermediates
    f1, f2 (bf16), rawp [B, NHp] and raw = rawp[:, :NH] (fp32), and heads = (cls, pos, size, orient, valid)."""
    dev = latent.device
    bf = torch.bfloat16
    NH = sum(h.shape[0] for h in heads[0::2])
    NHp = (NH + 127) // 128 * 128
    Wh = torch.zeros(NHp, W2.shape[0], device=dev, dtype=bf)
    Wh[:NH] = torch.cat(heads[0::2], 0)
    bh = torch.zeros(NHp, device=dev)
    bh[:NH] = torch.cat(heads[1::2], 0)
    lat = latent.to(bf).contiguous()
    W1b, W2b = W1.to(bf).contiguous(), W2.to(bf).contiguous()
    B = lat.shape[0]
    f1 = torch.empty(B, W1.shape[0], device=dev, dtype=bf)
    f2 = torch.empty(B, W2.shape[0], device=dev, dtype=bf)
    rawp = torch.empty(B, NHp, device=dev)
    flops = 2.0 * B * (lat.shape[1] * W1.shape[0] + W1.shape[0] * W2.shape[0] + W2.shape[0] * NHp)
    with ktime("gemm_tc_kernel(decoder fwd)", flops):
        _gemm_nt(lat, W1b, f1, b1.float().contiguous(), RELU)
        _gemm_nt(f1, W2b, f2, b2.float().contiguous(), RELU)
        _gemm_nt(f2, Wh, rawp, bh, OUT_F32)
    raw = rawp[:, :NH].contiguous()
    return dict(lat=lat, W1b=W1b, W2b=W2b, Wh=Wh, bh=bh, f1=f1, f2=f2, rawp=rawp, raw=raw, heads=F_.heads_split(raw, N, C))


def decoder_bf16_bwd(lat, W1b, W2b, Wh, f1, f2, d_raw):
    """Backward of DecoderBF16Fn from d_raw [B, NH] (fp32).  Returns a dict of d_rawp [B, NHp] (bf16, zero columns from NH
    on), dWh [NHp, D2], dbh [NH], df2 (after the ReLU mask), dW2, db2, df1, dW1, db1 and dlat."""
    B, NH = d_raw.shape
    NHp = Wh.shape[0]
    dev = lat.device
    bf = torch.bfloat16
    st = _stream(lat)
    d_rawp = torch.zeros(B, NHp, device=dev, dtype=bf)
    d_rawp[:, :NH] = d_raw
    D1, D2, DL = W1b.shape[0], W2b.shape[0], lat.shape[1]
    flops = 4.0 * B * (DL * D1 + D1 * D2 + D2 * NHp)
    kt = ktime("gemm_tc_kernel(decoder bwd)", flops)
    kt.__enter__()
    dWh = torch.zeros(NHp, D2, device=dev)
    _gemm_tn(d_rawp, f2, dWh)
    dbh = d_raw.sum(0)
    df2 = torch.empty(B, D2, device=dev, dtype=bf)
    _gemm_nt(d_rawp, Wh.t().contiguous(), df2, None)
    _lib.call("rs_relu_bwd_bf16", _p(df2), _p(f2), _p(df2), df2.numel(), st)
    dW2 = torch.zeros(D2, D1, device=dev)
    _gemm_tn(df2, f1, dW2)
    db2 = df2.float().sum(0)
    df1 = torch.empty(B, D1, device=dev, dtype=bf)
    _gemm_nt(df2, W2b.t().contiguous(), df1, None)
    _lib.call("rs_relu_bwd_bf16", _p(df1), _p(f1), _p(df1), df1.numel(), st)
    dW1 = torch.zeros(D1, DL, device=dev)
    _gemm_tn(df1, lat, dW1)
    db1 = df1.float().sum(0)
    dlat = torch.empty(B, DL, device=dev)
    _gemm_nt(df1, W1b.t().contiguous(), dlat, None, OUT_F32)
    kt.__exit__(None, None, None)
    return dict(d_rawp=d_rawp, dWh=dWh, dbh=dbh, df2=df2, dW2=dW2, db2=db2, df1=df1, dW1=dW1, db1=db1, dlat=dlat)


class DecoderBF16Fn(torch.autograd.Function):
    """MLP trunk + heads of the bf16 mode on the TMA-fed tcgen05 GEMM: bf16 operands, fp32 accumulate, the head
    outputs (logits, positions, ...) leave the last GEMM in fp32.  Same signature as functional.DecoderFn."""

    @staticmethod
    @_lib.on_tensor_device
    def forward(ctx, latent, N, C, W1, b1, W2, b2, *heads):
        _need_cuda(latent, W1, W2, *heads)
        with torch.no_grad():
            r = decoder_bf16_fwd(latent, N, C, W1, b1, W2, b2, heads)
        ctx.save_for_backward(r["lat"], r["W1b"], r["W2b"], r["Wh"], r["f1"], r["f2"], r["raw"])
        ctx.dims = (N, C)
        ctx.head_rows = [h.shape[0] for h in heads[0::2]]
        return r["heads"]

    @staticmethod
    @_lib.on_tensor_device
    def backward(ctx, d_cls, d_pos, d_size, d_orient, d_valid):
        lat, W1b, W2b, Wh, f1, f2, raw = ctx.saved_tensors
        N, C = ctx.dims
        with torch.no_grad():
            d_raw = F_.heads_merge(raw, N, C, d_cls, d_pos, d_size, d_orient, d_valid)
            g = decoder_bf16_bwd(lat, W1b, W2b, Wh, f1, f2, d_raw)
        return (g["dlat"], None, None, g["dW1"], g["db1"], g["dW2"], g["db2"],
                *F_.split_head_grads(g["dWh"], g["dbh"], ctx.head_rows))
