"""float64 reference of the decoder, the multi-task loss and the AdamW step, one kernel stage at a time.  TEST
INFRASTRUCTURE ONLY (tests/test_decoder_ref.py checks it against float64 autograd of oracle.room_slam_ref and
torch.optim.AdamW; tests/test_decoder_loss_gpu.py checks the kernels against it).

Every function takes the operands a kernel actually sees (bf16-rounded activations and weights, fp32 biases, the kernel's
own intermediates when a stage is teacher-forced) as tensors of any dtype and computes in float64 on their device.

  heads_split / heads_merge   rs_heads_split_f32 / rs_heads_merge_bwd_f32: columns class | pos | size | orient | valid,
                              sizes = softplus (threshold 20) + 1e-4, d size = d_size * sigmoid (1 above the threshold)
  decoder_fwd / decoder_bwd   the three GEMM stages forward (ReLU on the first two) and the backward chain, with the
                              head rows zero-padded to NHp; each stage may take the kernel's own input (teacher forcing)
  loss_terms / loss_finalize  rs_loss_fwd_f32: the six sums and the un-normalised per-element gradients g_*
  loss_bwd                    rs_loss_bwd_f32: g_* scaled for an arbitrary d(losses)[6]
  adamw_step                  rs_adamw_step_f32: global-norm clip (+ 1e-6), decoupled decay, bias correction
"""
from __future__ import annotations

import math

import numpy as np
import torch

F64 = torch.float64
LOSS_WEIGHTS = (2.0, 5.0, 5.0, 1.0, 1.0)      # class, position, size, orientation, validity (room_slam_ref.LOSS_WEIGHTS)
SOFTPLUS_THRESHOLD = 20.0


def _d(t):
    return None if t is None else t.to(F64)


def head_blocks(N: int, C: int):
    """(name, first column, columns) of the five head blocks of raw [B, N (C + 6)]."""
    return (("cls", 0, N * C), ("pos", N * C, 2 * N), ("size", N * C + 2 * N, 2 * N), ("orient", N * C + 4 * N, N),
            ("valid", N * C + 5 * N, N))


def softplus(v, threshold=SOFTPLUS_THRESHOLD):
    v = _d(v)
    return torch.where(v > threshold, v, torch.log1p(torch.exp(torch.clamp(v, max=threshold))))


def heads_split(raw, N: int, C: int, threshold=SOFTPLUS_THRESHOLD):
    raw = _d(raw)
    B = raw.shape[0]
    cls, pos, size, orient, valid = (raw[:, c0:c0 + n] for _, c0, n in head_blocks(N, C))
    return (cls.reshape(B, N, C), pos.reshape(B, N, 2), (softplus(size, threshold) + 1e-4).reshape(B, N, 2), orient.clone(),
            valid.clone())


def heads_merge(raw, N: int, C: int, d_cls, d_pos, d_size, d_orient, d_valid, threshold=SOFTPLUS_THRESHOLD):
    raw = _d(raw)
    B = raw.shape[0]
    out = torch.zeros_like(raw)
    for (name, c0, n), d in zip(head_blocks(N, C), (d_cls, d_pos, d_size, d_orient, d_valid)):
        if d is None:
            continue
        d = _d(d).reshape(B, n)
        if name == "size":
            v = raw[:, c0:c0 + n]
            d = d * torch.where(v > threshold, torch.ones_like(v), torch.sigmoid(v))
        out[:, c0:c0 + n] = d
    return out


# ---- decoder stages ---------------------------------------------------------------------------------------------------
def linear(a, w, b=None, relu=False):
    """a [M, K] . w [N, K]^T + b, optional ReLU; and the error scale sum_k |a||w| + |b| of every output."""
    a, w = _d(a), _d(w)
    y = a @ w.t()
    s = a.abs() @ w.abs().t()
    if b is not None:
        y = y + _d(b)
        s = s + _d(b).abs()
    return (y.clamp_min(0.0) if relu else y), s


def pad_heads(heads, NHp=None):
    """Stack the five (weight, bias) head pairs into Wh [NHp, D], bh [NHp] with zero rows from NH on."""
    Wh, bh = torch.cat([_d(w) for w in heads[0::2]]), torch.cat([_d(b) for b in heads[1::2]])
    NH = Wh.shape[0]
    NHp = NHp or (NH + 127) // 128 * 128
    return torch.cat([Wh, Wh.new_zeros(NHp - NH, Wh.shape[1])]), torch.cat([bh, bh.new_zeros(NHp - NH)])


def decoder_fwd(lat, W1, b1, W2, b2, Wh, bh, f1=None, f2=None):
    """Returns dict f1, f2, rawp and their error scales s1, s2, s3.  f1 / f2 given: the next stage reads them (teacher
    forcing); otherwise it reads this function's own float64 result."""
    r = {}
    r["f1"], r["s1"] = linear(lat, W1, b1, relu=True)
    r["f2"], r["s2"] = linear(r["f1"] if f1 is None else f1, W2, b2, relu=True)
    r["rawp"], r["s3"] = linear(r["f2"] if f2 is None else f2, Wh, bh)
    return r


def decoder_bwd(lat, W1, W2, Wh, f1, f2, d_rawp, d_raw=None, df2=None, df1=None, mask2=None, mask1=None):
    """The backward chain from d_rawp [B, NHp] (what the GEMMs read; d_raw [B, NH], default d_rawp, feeds the bias sum).
    df2 / df1 given: the later stages read them (teacher forcing).  mask2 / mask1 override the ReLU masks f2 > 0 and
    f1 > 0.  Returns dict dWh, dbh, df2, dW2, db2, df1, dW1, db1, dlat and the error scales s_* of the GEMM stages."""
    lat, W1, W2, Wh, f1, f2, d_rawp = (_d(t) for t in (lat, W1, W2, Wh, f1, f2, d_rawp))
    d_raw = d_rawp if d_raw is None else _d(d_raw)
    mask2 = (f2 > 0) if mask2 is None else mask2
    mask1 = (f1 > 0) if mask1 is None else mask1
    r = {"dWh": d_rawp.t() @ f2, "s_dWh": d_rawp.abs().t() @ f2.abs(), "dbh": d_raw.sum(0)}
    r["df2"] = (d_rawp @ Wh) * mask2
    r["s_df2"] = (d_rawp.abs() @ Wh.abs()) * mask2
    g2 = r["df2"] if df2 is None else _d(df2)
    r["dW2"], r["s_dW2"], r["db2"] = g2.t() @ f1, g2.abs().t() @ f1.abs(), g2.sum(0)
    r["df1"] = (g2 @ W2) * mask1
    r["s_df1"] = (g2.abs() @ W2.abs()) * mask1
    g1 = r["df1"] if df1 is None else _d(df1)
    r["dW1"], r["s_dW1"], r["db1"] = g1.t() @ lat, g1.abs().t() @ lat.abs(), g1.sum(0)
    r["dlat"], r["s_dlat"] = g1 @ W1, g1.abs() @ W1.abs()
    return r


# ---- loss ---------------------------------------------------------------------------------------------------------------
def loss_terms(cls, pos, size, orient, vlogit, t_cls, t_pos, t_size, t_orient, t_valid):
    """Returns (sums[6] = n_valid, sum v ce, sum v |dpos|, sum v |dsize|, sum v |dorient|, sum bce;
    g = [g_cls, g_pos, g_size, g_orient, g_valid]) of loss_fwd_kernel, un-normalised."""
    cls, pos, size, orient, vlogit, t_pos, t_size, t_orient, v = (
        _d(t) for t in (cls, pos, size, orient, vlogit, t_pos, t_size, t_orient, t_valid))
    t_cls = t_cls.long()
    lse = torch.logsumexp(cls, -1)
    ce = lse - cls.gather(-1, t_cls.unsqueeze(-1)).squeeze(-1)
    onehot = torch.nn.functional.one_hot(t_cls, cls.shape[-1]).to(F64)
    dp, ds, do = pos - t_pos, size - t_size, orient - t_orient
    l = vlogit
    sums = torch.stack([v.sum(), (v * ce).sum(), (v[..., None] * dp.abs()).sum(), (v[..., None] * ds.abs()).sum(),
                        (v * do.abs()).sum(), (l.clamp_min(0) - l * v + torch.log1p(torch.exp(-l.abs()))).sum()])
    g = [v[..., None] * (torch.exp(cls - lse[..., None]) - onehot), v[..., None] * torch.sign(dp),
         v[..., None] * torch.sign(ds), v * torch.sign(do), torch.sigmoid(l) - v]
    return sums, g


def _nv(sums):
    return max(float(sums[0]), 1.0)


def loss_finalize(sums, slots: int, weights=LOSS_WEIGHTS):
    """losses[6] = [total, class, position, size, orientation, validity] from the six sums."""
    nv = _nv(sums)
    parts = [float(sums[1]) / nv, float(sums[2]) / (2 * nv), float(sums[3]) / (2 * nv), float(sums[4]) / nv,
             float(sums[5]) / slots if slots > 0 else 0.0]
    return torch.tensor([sum(w * p for w, p in zip(weights, parts))] + parts, dtype=F64)


def loss_coefs(sums, slots: int, d_losses, weights=LOSS_WEIGHTS):
    """The factors loss_bwd_kernel multiplies g_cls, g_pos, g_size, g_orient, g_valid by."""
    nv = _nv(sums)
    d = [float(x) for x in d_losses]
    return [(d[0] * weights[0] + d[1]) / nv, (d[0] * weights[1] + d[2]) / (2 * nv), (d[0] * weights[2] + d[3]) / (2 * nv),
            (d[0] * weights[3] + d[4]) / nv, (d[0] * weights[4] + d[5]) / slots]


def loss_bwd(sums, g, d_losses, weights=LOSS_WEIGHTS):
    slots = g[4].numel()
    return [_d(t) * k for t, k in zip(g, loss_coefs(sums, slots, d_losses, weights))]


# ---- AdamW --------------------------------------------------------------------------------------------------------------
CLIP_EPS = float(np.float32(1e-6))


def bias_corrections(beta1, beta2, step: int, f32: bool):
    """1 - beta^step.  f32: as rs_adamw_step_f32 computes them on the host (float32 powf of the float32 beta), otherwise in
    float64 of the float32 beta."""
    b1, b2 = np.float32(beta1), np.float32(beta2)
    if f32:
        one = np.float32(1.0)
        return float(one - np.power(b1, np.float32(step))), float(one - np.power(b2, np.float32(step)))
    return 1.0 - float(b1) ** step, 1.0 - float(b2) ** step


def adamw_step(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step: int, grad_scale=1.0, max_norm=0.0, f32_args=True,
               f32_bias_correction=False, decay_after=False, sqrt_bc2=True):
    """One rs_adamw_step_f32 in float64.  Returns (p, m, v, sumsq); sumsq = ||g grad_scale||^2 (0 with max_norm <= 0).
    f32_args: every hyperparameter rounded to float32 first, as the C ABI passes it (False: the given doubles, as
    torch.optim.AdamW uses them).  decay_after / sqrt_bc2 = False build the faulty variants of the sensitivity test."""
    r = (lambda x: float(np.float32(x))) if f32_args else float
    lr, b1, b2, eps, wd, gsc, mn = (r(x) for x in (lr, beta1, beta2, eps, weight_decay, grad_scale, max_norm))
    if f32_args:
        bc1, bc2 = bias_corrections(beta1, beta2, step, f32_bias_correction)
    else:
        bc1, bc2 = 1.0 - b1 ** step, 1.0 - b2 ** step
    p, g, m, v = (_d(t) for t in (p, g, m, v))
    g = g * gsc
    sumsq = float(g.square().sum()) if mn > 0 else 0.0
    if mn > 0:
        g = g * min(1.0, mn / (math.sqrt(sumsq) + CLIP_EPS))
    if not decay_after:
        p = p * (1.0 - lr * wd)
    m = b1 * m + (1.0 - b1) * g
    v = b2 * v + (1.0 - b2) * g * g
    p = p - (lr / bc1) * m / (v.sqrt() / (math.sqrt(bc2) if sqrt_bc2 else bc2) + eps)
    if decay_after:
        p = p * (1.0 - lr * wd)
    return p, m, v, sumsq
