"""TEST INFRASTRUCTURE ONLY.  Float64 reference of what the BiLSTM + query-decoder kernels compute, on the operands they
actually see (csrc/lstm_f32.cu, csrc/query_attn.cu, lstm_model.lstm_grads_from_dG).  Self-checked against float64
torch.nn.LSTM and autograd of oracle/lstm_ref.py by tests/test_bilstm_ref.py; used per step by
tests/test_bilstm_kernels_gpu.py.

Layouts (those of the C ABI):
  * sequence buffers are padded (B, T + 2, C): rows 1..T hold the steps, rows 0 and T + 1 are zero pad rows;
  * P (B, T + 2, 8H): the input projection with b_ih + b_hh folded in, columns [forward i | f | g | o, reverse i | f | g | o];
  * w_hh [2][4H][H] (rows i | f | g | o per direction); saved [2][B][T][5][H] = (i, f, g, o, c) per step;
  * out (B, T + 2, 2H) = [forward h | reverse h]; dG (B, T + 2, 8H) has P's columns.
Inside this module a direction-major form (2, B, T, ...) is used, and `proc` turns it into processing order (the
reverse direction's time axis flipped), in which both directions run step s = 0 .. T - 1 together.
"""
from __future__ import annotations

from typing import Optional

import torch

F64 = torch.float64
U32 = 2.0 ** -24             # unit roundoff of float32


# ------------------------------------------------------------------------------------------------------------ layouts
def dirs(x: torch.Tensor, per: int) -> torch.Tensor:
    """(B, T, 2 per H) -> (2, B, T, per, H) float64 (per = 4: gate blocks; per = 1: hidden states)."""
    B, T, C = x.shape
    return x.to(F64).reshape(B, T, 2, per, C // (2 * per)).permute(2, 0, 1, 3, 4)


def undirs(x: torch.Tensor) -> torch.Tensor:
    """(2, B, T, per, H) -> (B, T, 2 per H): the inverse of dirs."""
    _, B, T, per, H = x.shape
    return x.permute(1, 2, 0, 3, 4).reshape(B, T, 2 * per * H)


def proc(x: torch.Tensor) -> torch.Tensor:
    """(2, B, T, ...) time order <-> processing order (reverse direction flipped in time).  Its own inverse."""
    return torch.stack([x[0], x[1].flip(1)])


def prev_step(x: torch.Tensor) -> torch.Tensor:
    """(2, B, T, ...): the value at the step processed before (t - 1 forward, t + 1 reverse); zero at each first step."""
    p = torch.zeros_like(x)
    p[0, :, 1:] = x[0, :, :-1]
    p[1, :, :-1] = x[1, :, 1:]
    return p


def saved_split(saved: torch.Tensor):
    """saved [2][B][T][5][H] -> (gates (2, B, T, 4, H), c (2, B, T, H)) float64."""
    s = saved.to(F64)
    return s[:, :, :, :4], s[:, :, :, 4]


# ------------------------------------------------------------------------------------------------------- LSTM forward
def _act(a: torch.Tensor):
    """Pre-activations (..., 4, H) -> (activated gates, derivative of the activation), tanh on the g block."""
    g = torch.sigmoid(a)
    g[..., 2, :] = torch.tanh(a[..., 2, :])
    d = g * (1 - g)
    d[..., 2, :] = 1 - g[..., 2, :] ** 2
    return g, d


def matvec(w_hh: torch.Tensor, h: torch.Tensor) -> torch.Tensor:
    """w_hh [2][4H][H], h (2, B, T, H) -> (2, B, T, 4, H)."""
    H = w_hh.shape[2]
    return torch.einsum("dgk,dbtk->dbtg", w_hh.to(F64), h).unflatten(-1, (4, H))


def forward_step(Pd: torch.Tensor, w_hh: torch.Tensor, h_prev: torch.Tensor) -> dict:
    """Every step at once, teacher-forced: Pd (2, B, T, 4, H) (dirs of P rows 1..T), h_prev (2, B, T, H) the kernel's own
    h of the step before (prev_step of its `out`).  Returns the activated gates and `bound` = act'(a) (|P| + sum |W||h|),
    the size of an fp32 evaluation's error in units of U32."""
    a = Pd + matvec(w_hh, h_prev)
    g, d = _act(a)
    S = Pd.abs() + matvec(w_hh.abs(), h_prev.abs())
    return {"a": a, "gates": g, "bound": d * S}


def cell(gates: torch.Tensor, c_prev: torch.Tensor):
    """c = f c_prev + i g and h = o tanh(c) from given gates (2, B, T, 4, H) and c_prev (2, B, T, H); with the bounds of
    their fp32 evaluation (units of U32)."""
    i, f, g, o = gates.unbind(3)
    c = f * c_prev + i * g
    return c, (f * c_prev).abs() + (i * g).abs()


def h_of(o: torch.Tensor, c: torch.Tensor):
    th = torch.tanh(c)
    return o * th, o.abs() * (th.abs() + (1 - th ** 2) * c.abs())


def forward_free(Pd: torch.Tensor, w_hh: torch.Tensor) -> dict:
    """The float64 recursion from zero states: gates (2, B, T, 4, H), c and h (2, B, T, H)."""
    Pp = proc(Pd)
    _, B, T, _, H = Pp.shape
    w = w_hh.to(F64)
    h = torch.zeros(2, B, H, dtype=F64, device=Pd.device)
    c = torch.zeros_like(h)
    G, C, Hs = torch.empty_like(Pp), torch.empty(2, B, T, H, dtype=F64, device=Pd.device), torch.empty(2, B, T, H, dtype=F64, device=Pd.device)
    for s in range(T):
        a = Pp[:, :, s] + torch.einsum("dgk,dbk->dbg", w, h).unflatten(-1, (4, H))
        g, _ = _act(a)
        c = g[:, :, 1] * c + g[:, :, 0] * g[:, :, 2]
        h = g[:, :, 3] * torch.tanh(c)
        G[:, :, s], C[:, :, s], Hs[:, :, s] = g, c, h
    return {"gates": proc(G), "c": proc(C), "h": proc(Hs)}


# ------------------------------------------------------------------------------------------------------ LSTM backward
def backward(gates: torch.Tensor, c: torch.Tensor, w_hh: torch.Tensor, d_out: torch.Tensor,
             feedback: Optional[torch.Tensor] = None, dc_no_f: bool = False) -> dict:
    """Backward through time of both directions, lstm_{reg_,}bwd kernels' epilogue in float64.

    gates (2, B, T, 4, H), c (2, B, T, H): the kernel's saved values; d_out (2, B, T, H).  Without feedback the recursion
    runs free; with feedback (2, B, T, 4, H) = the kernel's own dG, dh at a step is W_hh^T times the kernel's dG of the
    step processed before it, and the carry dc stays in float64 -- an error then shows at the step where it happens.
    dc_no_f carries dc without the x f (a deliberately wrong reference).  Returns dG (2, B, T, 4, H) and `bound` (units of
    U32): the size of an fp32 evaluation's error given the operands."""
    gp, cp, dop = proc(gates.to(F64)), proc(c.to(F64)), proc(d_out.to(F64))
    fb = proc(feedback.to(F64)) if feedback is not None else None
    _, B, T, _, H = gp.shape
    w = w_hh.to(F64).reshape(2, 4 * H, H)
    wa = w.abs()
    dh = torch.zeros(2, B, H, dtype=F64, device=gp.device)
    dh_b = torch.zeros_like(dh)
    dc = torch.zeros_like(dh)
    dG, bound = torch.empty_like(gp), torch.empty_like(gp)
    for s in reversed(range(T)):
        i, f, g, o = gp[:, :, s].unbind(2)
        cc = cp[:, :, s]
        cprev = cp[:, :, s - 1] if s > 0 else torch.zeros_like(cc)
        d = dh + dop[:, :, s]
        d_b = dh_b + dop[:, :, s].abs()
        tc = torch.tanh(cc)
        dcell = dc + d * o * (1 - tc * tc)
        dcell_b = dc.abs() + d_b * (o * (1 - tc * tc)).abs()
        G = torch.stack([dcell * g * i * (1 - i), dcell * cprev * f * (1 - f), dcell * i * (1 - g * g), d * tc * o * (1 - o)], 2)
        bound[:, :, s] = torch.stack([dcell_b * (g * i * (1 - i)).abs(), dcell_b * (cprev * f * (1 - f)).abs(),
                                      dcell_b * (i * (1 - g * g)).abs(), d_b * (tc * o * (1 - o)).abs()], 2)
        dc = dcell if dc_no_f else dcell * f
        dG[:, :, s] = G
        Gin = (fb[:, :, s] if fb is not None else G).reshape(2, B, 4 * H)
        dh = torch.einsum("dgk,dbg->dbk", w, Gin)
        dh_b = torch.einsum("dgk,dbg->dbk", wa, Gin.abs())
    return {"dG": proc(dG), "bound": proc(bound)}


# ------------------------------------------------------------------------------------------------------ layer assembly
def masked_input(xin: torch.Tensor, mask: Optional[torch.Tensor]) -> torch.Tensor:
    """What the projection reads: xin (B, T + 2, I) times the dropout mask (B, T, I) at rows 1..T, zero pad rows (the
    masked copy is a fresh padded buffer); without a mask, xin itself."""
    x = xin.to(F64)
    if mask is None:
        return x
    xm = torch.zeros_like(x)
    xm[:, 1:-1] = x[:, 1:-1] * mask.to(F64)
    return xm


def lstm_weight_grads(dG: torch.Tensor, out: torch.Tensor, xin: torch.Tensor, mask: Optional[torch.Tensor] = None):
    """(dW_ih [8H, I], dW_hh [2][4H][H], db [8H]) of one layer from dG (B, T + 2, 8H), out (B, T + 2, 2H) and the layer
    input xin (B, T + 2, I), per trace: h_{t-1} of the forward direction is the row before, of the reverse the row after
    (pad rows of out and dG zero, as the kernels write them).  db is the gradient of b_ih and of b_hh alike."""
    dG, out = dG.to(F64), out.to(F64)
    H = out.shape[2] // 2
    x = masked_input(xin, mask)
    dW_ih = torch.einsum("btg,bti->gi", dG, x)
    dW_hh = torch.stack([torch.einsum("btg,btk->gk", dG[:, 1:, :4 * H], out[:, :-1, :H]),
                         torch.einsum("btg,btk->gk", dG[:, :-1, 4 * H:], out[:, 1:, H:])])
    return dW_ih, dW_hh, dG.sum((0, 1))


def data_grad(dG: torch.Tensor, w_ih_cat: torch.Tensor, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """d_xin over all T + 2 rows: dG w_ih_cat, times the dropout mask at rows 1..T."""
    d = dG.to(F64) @ w_ih_cat.to(F64)
    if mask is not None:
        d[:, 1:-1] = d[:, 1:-1] * mask.to(F64)
    return d


# --------------------------------------------------------------------------------------------------------- trace stats
def trace_stats(traces: torch.Tensor, mask: Optional[torch.Tensor], fp32: bool = True):
    """(mean (B, 3), rms (B,), count (B,)) of rs_trace_stats_f32.  With fp32 the kernel's roundings are reproduced: sums
    in float64, mean = float32(sum / max(count, 1)), dx = float32(x - mean), squares summed in float64,
    rms = max(float32(sqrt(float32(q / count))), float32(1e-3)), count = max(count, 1).  fp32=False stays in float64
    (TraceEncoderRef.stats)."""
    x = traces[..., :3].to(F64)
    v = torch.ones(x.shape[:2], dtype=F64, device=x.device) if mask is None else mask.to(F64)
    denom = v.sum(1).clamp_min(1.0)
    mean = (x * v[..., None]).sum(1) / denom[:, None]
    if fp32:
        mean = mean.float().to(F64)
    dev = x - mean[:, None]
    if fp32:
        dev = dev.float().to(F64)
    q = ((dev[..., 0] ** 2 + dev[..., 2] ** 2) * v).sum(1) / denom
    if fp32:
        rms = torch.sqrt(q.float()).clamp_min(torch.tensor(1e-3, dtype=torch.float32, device=q.device)).to(F64)
    else:
        rms = torch.sqrt(q).clamp_min(1e-3)
    return mean, rms, denom


# ----------------------------------------------------------------------------------------------------- query attention
def _valid(memory, mask):
    B, N, _ = memory.shape
    return torch.ones(B, N, dtype=torch.bool, device=memory.device) if mask is None else mask.bool()


def attn_fwd(memory, qk, qb, traces, mask, mean, rms, skip_alpha_split=None, tokens_per_split=None, summary_by_n=False,
             ignore_mask_at=None, anchor_y_for_z=False) -> dict:
    """The query attention forward in float64.  memory (B, N, D) (rows 1..N of the padded buffer), qk (Q, D), qb (Q,),
    traces (B, N, F), mask (B, N) or None, mean (B, 3), rms (B,) as the kernel is given them.

    scores = m qk^T + qb over the valid tokens; attn = masked softmax; ctx = attn m; anchor = attn (xyz - mean) / rms;
    summary = sum of the valid m / max(count, 1); stats = (max, sum of exp(score - max)).  A trace without a valid token
    gives NaN ctx and anchor, summary 0 and stats (-inf, 0).  The keyword arguments build deliberately wrong references
    (a split whose running max is not rescaled, summary over N, one token's mask ignored, anchor with y for z).
    Also returns `S` (B, Q, N) = 1 + |qb| + sum |qk||m|, the score's size, for the error bounds."""
    m = memory.to(F64)
    B, N, D = m.shape
    valid = _valid(m, mask).clone()
    if ignore_mask_at is not None:
        valid[ignore_mask_at] = True
    nc = (traces[..., :3].to(F64) - mean.to(F64)[:, None]) / rms.to(F64)[:, None, None]
    if anchor_y_for_z:
        nc = nc[..., [0, 1, 1]]
    s = torch.einsum("bnd,qd->bqn", m, qk.to(F64)) + qb.to(F64)[None, :, None]
    s = s.masked_fill(~valid[:, None, :], float("-inf"))
    M = s.amax(-1, keepdim=True)
    e = torch.exp(s - torch.where(torch.isfinite(M), M, torch.zeros_like(M)))
    e = torch.where(valid[:, None, :], e, torch.zeros_like(e))
    if skip_alpha_split is not None:
        # the split's partials keep the scale of its own running max: weight it by exp(M_split - M) once more
        lo, hi = skip_alpha_split * tokens_per_split, min(N, (skip_alpha_split + 1) * tokens_per_split)
        ms = s[..., lo:hi].amax(-1, keepdim=True)
        e[..., lo:hi] = e[..., lo:hi] * torch.exp(M - torch.where(torch.isfinite(ms), ms, M))
    L = e.sum(-1, keepdim=True)
    p = e / L
    cnt = valid.to(F64).sum(1)
    summary = (m * valid[..., None]).sum(1) / (float(N) if summary_by_n else cnt.clamp_min(1.0)[:, None])
    S = 1.0 + qb.to(F64).abs()[None, :, None] + torch.einsum("bnd,qd->bqn", m.abs(), qk.to(F64).abs())
    pz = torch.nan_to_num(p, nan=0.0)
    return {"p": p, "ctx": p @ m, "anchor": p @ nc, "summary": summary, "stats": torch.cat([M, L], -1), "nc": nc,
            "valid": valid, "S": S, "ctx_bound": (pz * S) @ m.abs(), "anchor_bound": (pz * S) @ nc.abs(),
            "summary_bound": (m.abs() * valid[..., None]).sum(1) / cnt.clamp_min(1.0)[:, None]}


def attn_bwd(memory, qk, fwd: dict, count, d_ctx, d_anchor, d_summary=None) -> dict:
    """The query attention backward in float64 from attn_fwd's result (its p, ctx, anchor).  count (B,) is the count the
    kernel is given (trace_stats' max(count, 1)).  dP = d_ctx m + d_anchor nc; dS = p (dP - delta), delta = d_ctx ctx +
    d_anchor anchor; d_memory = sum_q p d_ctx + dS qk (+ d_summary / count on valid tokens); dqk = sum_{b,n} dS m;
    dqb = sum dS.  A trace without a valid token contributes nothing.  Bounds (the size of an fp32 evaluation's error,
    dimensionless) in *_bound."""
    m, qk = memory.to(F64), qk.to(F64)
    p = torch.nan_to_num(fwd["p"], nan=0.0)
    dead = ~fwd["valid"].any(1)
    ctx, anchor = torch.nan_to_num(fwd["ctx"]), torch.nan_to_num(fwd["anchor"])
    dc, da = d_ctx.to(F64), d_anchor.to(F64)
    nc = fwd["nc"]
    dP = torch.einsum("bqd,bnd->bqn", dc, m) + torch.einsum("bqk,bnk->bqn", da, nc)
    delta = (dc * ctx).sum(-1) + (da * anchor).sum(-1)
    dS = p * (dP - delta[..., None])
    dS[dead] = 0
    dm = torch.einsum("bqn,bqd->bnd", p, dc) + torch.einsum("bqn,qd->bnd", dS, qk)
    dPa = torch.einsum("bqd,bnd->bqn", dc.abs(), m.abs()) + torch.einsum("bqk,bnk->bqn", da.abs(), nc.abs())
    dela = (dc * ctx).abs().sum(-1) + (da * anchor).abs().sum(-1)
    dS_b = p * fwd["S"] * (dPa + dela[..., None])
    dm_b = torch.einsum("bqn,bqd->bnd", p * fwd["S"], dc.abs()) + torch.einsum("bqn,qd->bnd", dS_b, qk.abs())
    if d_summary is not None:
        add = fwd["valid"].to(F64)[..., None] * d_summary.to(F64)[:, None, :] / count.to(F64)[:, None, None]
        dm = dm + add
        dm_b = dm_b + add.abs()
    return {"d_memory": dm, "dqk": torch.einsum("bqn,bnd->qd", dS, m), "dqb": dS.sum((0, 2)), "dS": dS,
            "d_memory_bound": dm_b, "dqk_bound": torch.einsum("bqn,bnd->qd", dS_b, m.abs()), "dqb_bound": dS_b.sum((0, 2))}
