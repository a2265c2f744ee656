"""float64 reference of what the bf16 GRU recurrence kernels compute, on the operands they actually see.

The kernels are rec_fwd_pair_kernel / rec_bwd_pair_kernel (csrc/rec_pair.cu, H = 128) and rec_fwd_wide_kernel /
rec_bwd_wide_kernel (csrc/rec_wide.cu, H = 256), fed by rs_gru_pack_weights_bf16 (csrc/pack_w.cu) at H = 128 and by
functional_bf16.wide_fwd_image / wide_bwd_image at H = 256.  Nothing in the product imports this module.

Three parts:
  * decoders of the raw layouts that keep the pad rows t' = 0, T + 1 and the pad traces b >= B of the last tile
    (layout.from_tile_major drops both): tile-major `out` / `dG`, the fp16 `gates` buffer;
  * the weights as the tensor core sees them: r, z rows bf16(w / 2), n rows bf16(w), with split = 1 each weight the pair
    hi + lo of pack_w.cu::hi_lo, the layer-0 input columns of rec_common.cuh (x hi, lo, hi against W_ih hi, hi, lo; the
    bias as b_hi + b_lo), all in the fp32 operation order of pack_w.cu;
  * a teacher-forced forward step (h_{t-1} = the kernel's own bf16 `out` of the step before, the MMA's A operand) and the
    backward recursion of rec_pair.cu's epilogue over the kernel's saved gates and `out`.

Every function takes torch tensors and works on their device: the GPU tests run it in float64 on the GPU, the self-check
(tests/test_rec_bf16_ref.py) on the CPU.  quant=False builds the exact (unquantised) float64 weights instead, so the same
code can be checked against torch.nn.GRU.

Conventions: per direction d, time t is the trace's own time (0 .. T-1); direction 0 runs t = 0 .. T-1, direction 1
t = T-1 .. 0.  Gates are those of torch.nn.GRU (r | z | n); the r and z pre-activations a are carried HALVED, as the
kernels fold the 1/2 of sigma(a) = 1/2 tanh(a/2) + 1/2 into the r and z rows: r = 1/2 tanh(a_r) + 1/2 here.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import torch

TILE = 128
F64 = torch.float64


# ----------------------------------------------------------------------------------------------------------- decoders
def tm_full(xt: torch.Tensor) -> torch.Tensor:
    """Tile-major (tiles, T + 2, C / 8, 128, 8) -> (tiles * 128, T + 2, C) float64, pad rows and pad traces kept."""
    nt, tp, c8 = xt.shape[:3]
    return xt.permute(0, 3, 1, 2, 4).reshape(nt * TILE, tp, c8 * 8).to(F64)


def to_tm(x: torch.Tensor, dtype=torch.bfloat16) -> torch.Tensor:
    """(tiles * 128, T + 2, C) -> tile-major (tiles, T + 2, C / 8, 128, 8): the inverse of tm_full (no padding added)."""
    bp, tp, c = x.shape
    return x.to(dtype).reshape(bp // TILE, TILE, tp, c // 8, 8).permute(0, 2, 3, 1, 4).contiguous()


def out_full(out: torch.Tensor, H: int) -> torch.Tensor:
    """`out` / `out_drop` ([fwd H | bwd H] columns) -> (2, tiles * 128, T + 2, H)."""
    o = tm_full(out)
    return torch.stack([o[..., :H], o[..., H:]], 0)


def dG_full(dG: torch.Tensor, H: int) -> torch.Tensor:
    """`dG` (8H columns, per direction r | z | n | hn) -> (2, tiles * 128, T + 2, 4, H)."""
    g = tm_full(dG)
    bp, tp = g.shape[:2]
    return g.reshape(bp, tp, 2, 4, H).permute(2, 0, 1, 3, 4)


def gates_full(gates: torch.Tensor, H: int) -> torch.Tensor:
    """`gates` [tiles][T][2][NG H / 8][128][8] -> (2, tiles * 128, T, NG, H), NG = 3 (r | z | n, H = 128) or 4 (| hn,
    H = 256).  The buffer is allocated as bfloat16 but holds fp16 bits."""
    nt, T, _, nch = gates.shape[:4]
    g = gates.view(torch.float16).permute(2, 0, 4, 1, 3, 5).reshape(2, nt * TILE, T, nch * 8 // H, H)
    return g.to(F64)


def drop_full(bits: torch.Tensor, scale: torch.Tensor, H: int) -> torch.Tensor:
    """Dropout bits [tiles][T][128][2H / 8] and their scale -> the multiplier (2, tiles * 128, T, H) (0 or scale)."""
    nt, T = bits.shape[:2]
    b = (bits.to(torch.int32).unsqueeze(-1) >> torch.arange(8, device=bits.device, dtype=torch.int32)) & 1
    m = b.reshape(nt, T, TILE, 2, H).permute(3, 0, 2, 1, 4).reshape(2, nt * TILE, T, H)
    return m.to(F64) * scale.to(F64)


def active_mask(lengths: Optional[torch.Tensor], Bp: int, T: int, device) -> torch.Tensor:
    """(Bp, T) bool: step t of trace b is inside its length.  Pad traces (and lengths = None) run all T steps."""
    act = torch.ones(Bp, T, dtype=torch.bool, device=device)
    if lengths is not None:
        B = lengths.shape[0]
        act[:B] = torch.arange(T, device=device)[None, :] < lengths.to(device).long()[:, None]
    return act


def h_prev_forward(outf: torch.Tensor, lengths: Optional[torch.Tensor]) -> torch.Tensor:
    """The A operand of the forward MMA at every step: (2, Bp, T, H) from the decoded `out` (2, Bp, T + 2, H).
    Direction 0 reads row t (the step before; row 0 is the zero pad) and, past a trace's length, keeps reading its last
    valid step: the kernel stores zeros there but its A tile keeps bf16 of the held state.  Direction 1 reads row t + 2:
    the zero pad at t = T - 1, and at t = len - 1 the stored zero of step len."""
    T = outf.shape[2] - 2
    Bp = outf.shape[1]
    idx = torch.arange(T, device=outf.device)[None, :].expand(Bp, T)
    if lengths is not None:
        lim = torch.full((Bp,), T, dtype=torch.long, device=outf.device)
        lim[:lengths.shape[0]] = lengths.to(outf.device).long()
        idx = torch.minimum(idx, lim[:, None])
    f = torch.gather(outf[0], 1, idx[..., None].expand(Bp, T, outf.shape[3]))
    return torch.stack([f, outf[1, :, 2:]], 0)


def h_prev_backward(outf: torch.Tensor) -> torch.Tensor:
    """h_{t-1} as the backward kernels read it: the stored `out` of the step before in forward time, (2, Bp, T, H)."""
    return torch.stack([outf[0, :, :-2], outf[1, :, 2:]], 0)


# ------------------------------------------------------------------------------------------- weights as the MMA sees them
def bf16(w: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest-even to bf16, back in the input's dtype (w fp32, as the kernels round fp32 values)."""
    return w.to(torch.bfloat16).to(w.dtype)


def hi_lo(w32: torch.Tensor, split: int, quant: bool = True) -> torch.Tensor:
    """The value the tensor core multiplies for fp32 weight w: bf16(w), or with split = 1 the pair
    hi + lo = bf16(w) + bf16(w - bf16(w)) (pack_w.cu::hi_lo; the difference is exact in fp32)."""
    if not quant:
        return w32.to(F64)
    hi = bf16(w32)
    if not split:
        return hi.to(F64)
    return hi.to(F64) + bf16(w32 - hi).to(F64)


def gate_scale(H: int, device, dtype=torch.float32) -> torch.Tensor:
    """(3H,): 1/2 on the r and z rows, 1 on the n rows."""
    s = torch.ones(3 * H, device=device, dtype=dtype)
    s[:2 * H] = 0.5
    return s


def bias_x(b_ih: torch.Tensor, b_hh: torch.Tensor, H: int, dtype=torch.float32) -> torch.Tensor:
    """(3H,): (b_ih + b_hh) / 2 on r, z, b_ih on n -- pack_w.cu::bias_x_of's operation order (in fp32 there)."""
    s = gate_scale(H, b_ih.device, dtype)
    add = torch.cat([b_hh[:2 * H].to(dtype), torch.zeros(H, device=b_ih.device, dtype=dtype)])
    return (b_ih.to(dtype) + add) * s


@dataclass
class RefWeights:
    """Per direction (index 0 / 1): the float64 operand values of one bidirectional layer.
    whh     (2, 3H, H)  forward B operand: r, z rows of W_hh / 2, n rows W_hn (quantised as the kernel's image)
    whh_bwd (2, 3H, H)  W_hh of the BPTT matvec (unscaled; hi + lo with split at H = 128, bf16 at H = 256)
    b_hn    (2, H)      fp32 bias of the hidden side of n
    bias    (2, 3H)     the input-side bias as the kernel adds it (b_hi + b_lo), r, z halved
    wih_hi, wih_lo (2, 3H, I)   layer-0 input columns (W_ih, r, z halved, as bf16 hi and lo); quant=False: lo = 0
    wih     (2, 3H, I)  the fused projection's W_ih (r, z halved, bf16)"""
    H: int
    whh: torch.Tensor
    whh_bwd: torch.Tensor
    b_hn: torch.Tensor
    bias: torch.Tensor
    wih_hi: torch.Tensor
    wih_lo: torch.Tensor
    wih: torch.Tensor
    quant: bool


def ref_weights(w, H: int, split: int, quant: bool = True, bwd_split: Optional[int] = None) -> RefWeights:
    """w = (w_ih, w_hh, b_ih, b_hh, w_ih_r, w_hh_r, b_ih_r, b_hh_r), fp32 (torch.nn.GRU's layout, gate order r | z | n).
    split: hi + lo weights (H = 128 only).  bwd_split defaults to split (H = 256: the backward image is plain bf16)."""
    bwd_split = split if bwd_split is None else bwd_split
    per = [w[:4], w[4:]]
    dev = w[0].device
    dt = torch.float32 if quant else F64          # quant=False: exact float64 values throughout
    s = gate_scale(H, dev, dt)
    whh, whh_bwd, b_hn, bias, wih_hi, wih_lo, wih = [], [], [], [], [], [], []
    for w_ih, w_hh, b_ih, b_hh in per:
        w_ih, w_hh = w_ih.to(dt), w_hh.to(dt)
        whh.append(hi_lo(w_hh * s[:, None], split, quant))
        whh_bwd.append(hi_lo(w_hh, bwd_split, quant))
        b_hn.append(b_hh[2 * H:].to(F64))
        bx = bias_x(b_ih, b_hh, H, dt)
        wsc = w_ih * s[:, None]
        if quant:
            bhi = bf16(bx)
            bias.append(bhi.to(F64) + bf16(bx - bhi).to(F64))
            whi = bf16(wsc)
            wih_hi.append(whi.to(F64))
            wih_lo.append(bf16(wsc - whi).to(F64))
            wih.append(whi.to(F64))
        else:
            bias.append(bx.to(F64))
            wih_hi.append(wsc.to(F64))
            wih_lo.append(torch.zeros_like(wsc, dtype=F64))
            wih.append(wsc.to(F64))
    st = lambda v: torch.stack(v, 0)  # noqa: E731
    return RefWeights(H, st(whh), st(whh_bwd), st(b_hn), st(bias), st(wih_hi), st(wih_lo), st(wih), quant)


# -------------------------------------------------------------------------------------------------- input pre-activations
def input_from_x(x: torch.Tensor, W: RefWeights, Bp: int) -> torch.Tensor:
    """Layer 0: x (B, T, I) fp32 -> the input part of the pre-activations (2, Bp, T, 3H) (r, z halved, bias included):
    x_hi W_hi + x_lo W_hi + x_hi W_lo + b_hi + b_lo per rec_common.cuh's columns.  Pad traces get the bias only."""
    B, T, I = x.shape
    xp = torch.zeros(Bp, T, I, device=x.device, dtype=torch.float32 if W.quant else F64)
    xp[:B] = x
    if W.quant:
        xhi = bf16(xp)
        xlo = bf16(xp - xhi)
        xhi, xlo = xhi.to(F64), xlo.to(F64)
    else:
        xhi, xlo = xp.to(F64), torch.zeros(Bp, T, I, device=x.device, dtype=F64)
    res = []
    for d in (0, 1):
        wh, wl = W.wih_hi[d], W.wih_lo[d]
        res.append(xhi @ wh.T + xlo @ wh.T + xhi @ wl.T + W.bias[d])
    return torch.stack(res, 0)


def input_from_P(P: torch.Tensor, H: int) -> torch.Tensor:
    """Deeper layers, projection GEMM: the tile-major bf16 P (6H columns, per direction r | z | n) -> (2, Bp, T, 3H)."""
    p = tm_full(P)[:, 1:-1]
    return torch.stack([p[..., :3 * H], p[..., 3 * H:]], 0)


def input_from_X(X: torch.Tensor, W: RefWeights) -> torch.Tensor:
    """Deeper layers, fused projection: tile-major bf16 X (the layer input) -> X W_ih^T + b_hi + b_lo, (2, Bp, T, 3H)."""
    xf = tm_full(X)[:, 1:-1]
    return torch.stack([xf @ W.wih[d].T + W.bias[d] for d in (0, 1)], 0)


# ---------------------------------------------------------------------------------------------------- forward, one step
def forward_step(h_prev: torch.Tensor, inp: torch.Tensor, W: RefWeights, active: torch.Tensor) -> dict:
    """Every step at once, teacher-forced: h_prev (2, Bp, T, H) is the MMA's A operand (h_prev_forward), inp the input
    pre-activations (2, Bp, T, 3H).  Returns r, z, n, hn = W_hn h + b_hn and the blend h = z h_prev + (1 - z) n, each
    (2, Bp, T, H).  Past a trace's length z = 1 (the state is held)."""
    H = W.H
    a = torch.einsum("dbtk,dgk->dbtg", h_prev, W.whh)
    r = 0.5 * torch.tanh(a[..., :H] + inp[..., :H]) + 0.5
    z = 0.5 * torch.tanh(a[..., H:2 * H] + inp[..., H:2 * H]) + 0.5
    z = torch.where(active[None, :, :, None], z, torch.ones_like(z))
    hn = a[..., 2 * H:] + W.b_hn[:, None, None, :]
    n = torch.tanh(inp[..., 2 * H:] + r * hn)
    return {"r": r, "z": z, "n": n, "hn": hn, "h": z * h_prev + (1.0 - z) * n}


def recompute_hn(h_prev_bwd: torch.Tensor, W: RefWeights) -> torch.Tensor:
    """H = 128 backward: hn = W_hn h_{t-1} + b_hn recomputed from the stored bf16 `out` (what rec_bwd_pair_kernel does)."""
    H = W.H
    return torch.einsum("dbtk,dgk->dbtg", h_prev_bwd, W.whh[:, 2 * H:]) + W.b_hn[:, None, None, :]


# ------------------------------------------------------------------------------------------------------------- backward
def backward(r, z, n, hn, h_prev, W: RefWeights, active, d_out=None, d_h_n=None, drop=None, feedback=None) -> torch.Tensor:
    """Backward through time of both directions, rec_pair.cu's epilogue in float64.  r, z, n, hn, h_prev: (2, Bp, T, H);
    d_out (2, Bp, T, H) or None; d_h_n (2, Bp, H) or None; drop: the multiplier of d_out (drop_full) or None.
        dh = carry + d_out;  gn = dh (1 - z)(1 - n^2);  gz = dh (h_prev - n) z (1 - z);  ghn = gn r;  gr = ghn hn (1 - r)
        carry = z dh + [gr | gz | ghn] W_hh
    Past a trace's length z = 1 and d_out = 0, so the gradients there are 0 and the carry passes through.
    feedback (2, Bp, T, 3, H) or None: the [gr | gz | ghn] to feed into the matvec instead of this recursion's own --
    the kernel's bf16 dG blocks r, z, hn, which are exactly its MMA's A operand (a teacher-forced backward).
    Returns dG (2, Bp, T, 4, H): r | z | n | hn."""
    _, Bp, T, H = r.shape
    dG = torch.zeros(2, Bp, T, 4, H, dtype=F64, device=r.device)
    act = active[..., None].to(F64)
    for d in (0, 1):
        carry = d_h_n[d].to(F64).clone() if d_h_n is not None else torch.zeros(Bp, H, dtype=F64, device=r.device)
        steps = range(T - 1, -1, -1) if d == 0 else range(T)
        for t in steps:
            dov = d_out[d][:, t] * act[:, t] if d_out is not None else 0.0
            if drop is not None:
                dov = dov * drop[d][:, t]
            zt = torch.where(active[:, t, None], z[d][:, t], torch.ones_like(z[d][:, t]))
            rt, nt, hnt, hp = r[d][:, t], n[d][:, t], hn[d][:, t], h_prev[d][:, t]
            dh = carry + dov
            gn = dh * (1.0 - zt) * (1.0 - nt * nt)
            gz = dh * (hp - nt) * (zt * (1.0 - zt))
            ghn = gn * rt
            gr = ghn * (hnt * (1.0 - rt))
            dG[d, :, t] = torch.stack([gr, gz, gn, ghn], 1)
            fb = feedback[d][:, t] if feedback is not None else torch.stack([gr, gz, ghn], 1)
            carry = zt * dh + fb.reshape(Bp, 3 * H) @ W.whh_bwd[d]
    return dG


def weight_grads(dG, x_seq, h_prev) -> dict:
    """The weight and bias gradients a dG stands for (what rs_blk_wgrad assembles), per direction:
    dW_ih = sum dG_{r,z,n}^T x, dW_hh = sum dG_{r,z,hn}^T h_{t-1}, db_ih = sum dG_{r,z,n}, db_hh = sum dG_{r,z,hn}.
    dG (2, Bp, T, 4, H), x_seq (2, Bp, T, I) (the layer input as each direction sees it), h_prev (2, Bp, T, H)."""
    ih = dG[:, :, :, [0, 1, 2]].flatten(3)          # (2, Bp, T, 3H)
    hh = dG[:, :, :, [0, 1, 3]].flatten(3)
    return {"w_ih": torch.einsum("dbtg,dbti->dgi", ih, x_seq), "w_hh": torch.einsum("dbtg,dbtk->dgk", hh, h_prev),
            "b_ih": ih.sum((1, 2)), "b_hh": hh.sum((1, 2))}


# ---------------------------------------------------------------------------------- operands and outputs of the GEMMs
def x_operand(x: torch.Tensor, Bp: int, T: int) -> torch.Tensor:
    """What rs_pack_x_tm writes for the layer-0 input x (B, T, I <= 16) fp32, decoded: (Bp, T + 2, 16) float64 holding
    bf16(x) in columns < I, and zeros in the columns >= I, the pad rows t' = 0, T + 1 and the pad traces b >= B."""
    B, _, I = x.shape
    xo = torch.zeros(Bp, T + 2, 16, dtype=F64, device=x.device)
    xo[:B, 1:T + 1, :I] = bf16(x.float()).to(F64)
    return xo


def data_grad(dG_full: torch.Tensor, w_ih: torch.Tensor, drop: Optional[torch.Tensor] = None) -> torch.Tensor:
    """dX of a deeper layer over all T + 2 rows, what rs_blk_gemm_nt(_drop) computes from dG before its bf16 rounding:
    sum over both directions and the r, z, n blocks of dG W_ih.  dG_full (2, Bp, T + 2, 4, H) (dG_full, pad rows kept);
    w_ih (2, 3H, I): W_ih as the dgrad image holds it (unscaled; bf16, or hi + lo with split); drop (Bp, T, I) or None:
    the multiplier (0 or scale) of the dropout on the layer input, applied at rows 1 .. T only.  -> (Bp, T + 2, I).
    With an exact fp32 sum the kernel's result is bf16(fp32(this)): the product of the fp32 sum and the fp32 scale is exact
    in float64, so one rounding to fp32 is the kernel's fp32 multiply."""
    dx = sum(dG_full[d, :, :, :3].flatten(2) @ w_ih[d] for d in (0, 1))
    if drop is not None:
        dx[:, 1:-1] = dx[:, 1:-1] * drop
    return dx


def projection(X_full: torch.Tensor, w_ih: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """P = X W_ih^T + b over all rows, what rs_blk_gemm_nt computes for the input projection before its bf16 rounding.
    X_full (Bp, T + 2, I) (tm_full of the layer input, pad rows kept); w_ih (2, 3H, I): the weights as the projection
    image holds them (r, z rows halved; bf16, or hi + lo with split); bias (2, 3H): the fp32 bias the epilogue adds
    (bias_x).  -> (Bp, T + 2, 6H), per direction r | z | n."""
    return torch.cat([X_full @ w_ih[d].T + bias[d] for d in (0, 1)], -1)
