"""The BiLSTM recurrence, the query attention and the trace statistics kernels called through their C entry points and
checked per direction, trace, step and gate block (LSTM) or per trace, query and token row (attention) against the
float64 reference of oracle/bilstm_ref.py (itself checked against torch.nn.LSTM and autograd by test_bilstm_ref.py).

Entry points: rs_lstm_fwd_f32 / rs_lstm_bwd_f32 (csrc/lstm_f32.cu), rs_trace_stats_f32, rs_query_attn_fwd_f32 (split
kernel + combine kernel) and rs_query_attn_bwd_f32 (atomic and per-query-tile deterministic variants) of
csrc/query_attn.cu, and the layer assembly lstm_model.lstm_grads_from_dG.  Every case runs in the default and the
deterministic mode (torch.use_deterministic_algorithms).

Sentinels.  Every output is NaN-filled before a call, inside a frame of SENT values that must survive: the pad rows 0 and
T + 1 of `out`, `dG` and `d_memory`, and extra columns (ld > width).  The inputs carry NaN wherever a kernel must not
read: the pad rows and extra columns of P, d_out and `memory`, and `traces` columns 3 and up.

LSTM instantiations (host logic restated in lstm_path; test_lstm_matrix_reaches_every_instantiation asserts it):
    register  lstm_reg_{fwd,bwd}_kernel<HH, R>, HH = 32, 64     R = 1: B 1, 148   R = 2: B 149, 296   R = 4: B 297, 592
                                                                R = 16: B 593, 601 (partial last CTA)
    general   lstm_{fwd,bwd}_f32_kernel<R, false>               H 96, 128 (S = 2): R = 1 at B 1, 3, 296; R = 4 at B 297, 301
                                                                H 160, 256 (S = 1): R = 1 at B 3; R = 4 at B 301
    unreachable: lstm_reg_*<HH, 8> (pick_r returns 4 for every B <= 592, and R = 8's condition also ends at 592) and
                 lstm_*_f32_kernel<R, true> (WSMEM needs H <= 64, which always takes the register kernels).
T runs over 1, 2, 8, 9 and 200: the register kernels prefetch PF_STEPS = 8 steps ahead, so the first and last 8 steps
take the other prefetch branch.

LSTM checks, each error normalised by the size of an fp32 evaluation's error given the kernel's own operands (units
of float32 ulps, U32 = 2^-24):
    gates i | f | g | o   teacher-forced step on the kernel's own h_{t-1}: |dg| / (act'(a) (|P| + sum |W||h|) + |g|)
    c                     f c_prev + i g of the kernel's own gates and c_prev: |dc| / (|f c_prev| + |i g| + |c|)
    out                   o tanh(c) of the kernel's own o and c: |dh| / (|o| (|tanh c| + sech^2(c) |c|))
    dG (teacher-forced)   dh = W^T (the kernel's dG of the step processed before), dc carried in float64:
                          |ddG| / (the same bound propagated through the epilogue + |dG|)
    out (free-running)    absolute error against the float64 recursion from P
    dG (free-running)     against the float64 recursion over the kernel's saved gates and c, relative to the largest
                          reference value of the (direction, gate block)
Attention checks, dimensionless: ctx and anchor per (trace, query) by sum_n p_n |m_n| (1 + S_n), S_n = |qb| +
sum |qk||m_n| (the score's size carries the rounding of the score into p); summary by the mean |m|; stats as
max + log(sum) against the float64 log-sum-exp, by 1 + max S_n; d_memory per token row by sum_q p (1 + S)|d_ctx| +
|dS| |qk| + |d_summary| / count; dqk / dqb after the column sum by sum |dS||m| and sum |dS|.

Bars (BARS), each about 4x the largest value measured over the matrices below, default and deterministic mode, on a
B200 at a 1000 W power limit:
    gates        20 ulps     measured 4.9 (H 256, B 301, T 200)     dG teacher-forced  72 ulps   measured 17.7 (same case;
    c             4 ulps     measured 0.98                                             the W_hh^T dG sum has 4H = 1024 terms)
    out          10 ulps     measured 2.3                           out free-running   1.6e-6    measured 3.9e-7
                                                                    dG free-running    1.8e-6    measured 4.3e-7
    ctx          1.8e-6      measured 4.4e-7                        stats              1e-6      measured 2.6e-7
    anchor       8e-7        measured 2.1e-7                        d_memory           1.6e-6    measured 3.8e-7
    summary      2.6e-6      measured 6.5e-7                        dqk / dqb          1e-7 / 6e-8  measured 2.5e-8 / 1.4e-8
"""
import contextlib
import math
from dataclasses import dataclass

import pytest
import torch

from oracle import bilstm_ref as R
from roomslam_b200 import _lib
from roomslam_b200 import functional as F_
from roomslam_b200 import lstm_model as LM

pytestmark = pytest.mark.gpu

MODES = ("default", "deterministic")
SENT = -77.0
F64 = torch.float64
X = 3                        # extra columns of every LSTM sequence buffer (ld = width + 3)
XM = 4                       # extra columns of `memory` / d_memory (the kernels read memory as float4: ld % 4 == 0)

BARS = {
    # LSTM, units of float32 ulps of the bound
    "gates": 20.0, "c": 4.0, "out": 10.0, "dG_tf": 72.0,
    # LSTM, looser: absolute (out) and relative to the block's largest value (dG)
    "out_free": 1.6e-6, "dG_free": 1.8e-6,
    # attention, dimensionless
    "ctx": 1.8e-6, "anchor": 8e-7, "summary": 2.6e-6, "stats": 1e-6, "d_memory": 1.6e-6, "dqk": 1e-7, "dqb": 6e-8,
}


@contextlib.contextmanager
def mode(name):
    det = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(name == "deterministic")
        yield
    finally:
        torch.use_deterministic_algorithms(det)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def framed(B, rows, width, extra, inner=float("nan")):
    """(B, rows + 2, width + extra) filled with SENT; rows 1..rows of the first `width` columns hold `inner`."""
    buf = torch.full((B, rows + 2, width + extra), SENT, device="cuda")
    buf[:, 1:-1, :width] = inner
    return buf


def frame_intact(buf, width):
    """The pad rows and the extra columns still hold SENT (bit for bit)."""
    m = torch.ones(buf.shape, dtype=torch.bool, device="cuda")
    m[:, 1:-1, :width] = False
    return bool((buf[m] == SENT).all())


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def norm_err(got, want, bound):
    """|got - want| / bound with NaN (an unwritten or non-finite output) reported as inf."""
    e = (got.to(F64) - want).abs() / bound.clamp_min(1e-300)
    return torch.nan_to_num(e, nan=math.inf, posinf=math.inf)


# ====================================================================================================== LSTM recurrence
def pick_r(B):
    """lstm_f32.cu::pick_r."""
    for r, occ in ((1, 2), (2, 2), (4, 2), (8, 1), (16, 1)):
        if 2 * ((B + r - 1) // r) <= 148 * occ:
            return r
    return 16


def lstm_path(H, B):
    """(path, R, S) of rs_lstm_{fwd,bwd}_f32 for hidden size H and batch B (lstm_f32.cu's host logic restated)."""
    if H in (32, 64):
        return ("register", pick_r(B), None)
    return ("general", 4 if B > 296 else 1, 2 if H <= 128 else 1)


@dataclass(frozen=True)
class LCase:
    H: int
    B: int
    T: int
    expect: tuple             # (path, R, S) the case must reach

    def __str__(self):
        return f"H{self.H}-B{self.B}-T{self.T}"


_REG = [(1, 1), (148, 1), (149, 2), (296, 2), (297, 4), (592, 4), (593, 16), (601, 16)]
_TS = (1, 2, 8, 9, 200)
LSTM_MATRIX = [LCase(H, B, _TS[(j + hi) % 5], ("register", r, None)) for hi, H in enumerate((32, 64)) for j, (B, r) in enumerate(_REG)]
LSTM_MATRIX += [LCase(H, B, _TS[(j + hi + 2) % 5], ("general", r, 2))
                for hi, H in enumerate((96, 128)) for j, (B, r) in enumerate([(1, 1), (3, 1), (296, 1), (297, 4), (301, 4)])]
LSTM_MATRIX += [LCase(160, 3, 200, ("general", 1, 1)), LCase(160, 301, 9, ("general", 4, 1)),
                LCase(256, 3, 8, ("general", 1, 1)), LCase(256, 301, 200, ("general", 4, 1)),
                LCase(64, 601, 200, ("register", 16, None)), LCase(128, 301, 200, ("general", 4, 2))]


def lstm_inputs(c: LCase, seed=0):
    g = torch.Generator(device="cuda").manual_seed(1000 * c.H + c.B + 7 * c.T + seed)
    H, B, T = c.H, c.B, c.T
    w_hh = (torch.rand(2, 4 * H, H, generator=g, device="cuda") * 2 - 1) * (2.0 / math.sqrt(H))
    P = torch.full((B, T + 2, 8 * H + X), float("nan"), device="cuda")
    P[:, 1:-1, :8 * H] = torch.randn(B, T, 8 * H, generator=g, device="cuda") * 0.8
    d_out = torch.full((B, T + 2, 2 * H + X), float("nan"), device="cuda")
    d_out[:, 1:-1, :2 * H] = torch.randn(B, T, 2 * H, generator=g, device="cuda")
    return {"w_hh": w_hh.contiguous(), "w_hh_t": w_hh.transpose(1, 2).contiguous(), "P": P, "d_out": d_out}


def run_lstm(c: LCase, inp, save=True, backward=True):
    H, B, T = c.H, c.B, c.T
    k = {"out": framed(B, T, 2 * H, X), "saved": torch.full((2, B, T, 5, H), float("nan"), device="cuda") if save else None}
    _lib.call("rs_lstm_fwd_f32", _p(inp["P"]), 8 * H + X, T + 2, 1, _p(inp["w_hh"]), _p(inp["w_hh_t"]), _p(k["out"]),
              2 * H + X, T + 2, 1, _p(k["saved"]), B, T, H, _st())
    if backward:
        k["dG"] = framed(B, T, 8 * H, X)
        _lib.call("rs_lstm_bwd_f32", _p(inp["d_out"]), 2 * H + X, T + 2, 1, _p(k["saved"]), _p(inp["w_hh"]), _p(k["dG"]),
                  8 * H + X, T + 2, 1, B, T, H, _st())
    torch.cuda.synchronize()
    return k


def lstm_reference(c: LCase, inp, k, swap_if=False, rev_from_before=False, c0=0.0, drop_last=False, dc_no_f=False,
                   swap_dout=False):
    """The float64 references around the kernel outputs k.  The keyword arguments each inject one fault."""
    H, B, T = c.H, c.B, c.T
    Pd = R.dirs(inp["P"][:, 1:-1, :8 * H], 4)
    w = inp["w_hh"].to(F64)
    if swap_if:
        Pd, w = Pd[:, :, :, [1, 0, 2, 3]], w.view(2, 4, H, H)[:, [1, 0, 2, 3]].reshape(2, 4 * H, H)
    if drop_last:
        Pd = Pd.clone()
        Pd[:, B - 1] = 0
    hk = R.dirs(k["out"][:, 1:-1, :2 * H], 1)[:, :, :, 0]
    gk, ck = R.saved_split(k["saved"])
    h_prev = R.prev_step(hk)
    if rev_from_before:
        h_prev[1] = R.prev_step(torch.stack([hk[1], hk[1]]))[0]
    c_prev = R.prev_step(ck)
    if c0:
        c_prev[0, :, 0] += c0
        c_prev[1, :, T - 1] += c0
    ref = {"tf": R.forward_step(Pd, w, h_prev), "hk": hk, "gk": gk, "ck": ck, "free": R.forward_free(Pd, w)}
    ref["c"], ref["c_bound"] = R.cell(gk, c_prev)
    ref["h"], ref["h_bound"] = R.h_of(gk[:, :, :, 3], ck)
    if "dG" in k:
        do = R.dirs(inp["d_out"][:, 1:-1, :2 * H], 1)[:, :, :, 0]
        if swap_dout:
            do = do.flip(0)
        dGk = R.dirs(k["dG"][:, 1:-1, :8 * H], 4)
        ref["dGk"] = dGk
        ref["bw_tf"] = R.backward(gk, ck, w, do, feedback=dGk, dc_no_f=dc_no_f)
        ref["bw_free"] = R.backward(gk, ck, w, do, dc_no_f=dc_no_f)
    return ref


def lstm_measure(c: LCase, k, ref):
    """Normalised errors per check: name -> (2, B, T, blocks) tensor; plus the exact violations (a list)."""
    H, U = c.H, R.U32
    m, exact = {}, []
    if not frame_intact(k["out"], 2 * H):
        exact.append("out_frame")
    if not bool(torch.isfinite(k["saved"]).all()):
        exact.append("saved_unwritten")
    tf = ref["tf"]
    m["gates"] = norm_err(ref["gk"], tf["gates"], U * (tf["bound"] + tf["gates"].abs()))
    m["c"] = norm_err(ref["ck"], ref["c"], U * (ref["c_bound"] + ref["c"].abs())).amax(-1, keepdim=True)
    m["out"] = norm_err(ref["hk"], ref["h"], U * ref["h_bound"]).amax(-1, keepdim=True)
    m["out_free"] = norm_err(ref["hk"], ref["free"]["h"], torch.ones_like(ref["hk"])).amax(-1, keepdim=True)
    if "dGk" in ref:
        if not frame_intact(k["dG"], 8 * H):
            exact.append("dG_frame")
        bt, bf = ref["bw_tf"], ref["bw_free"]
        m["dG_tf"] = norm_err(ref["dGk"], bt["dG"], U * (bt["bound"] + bt["dG"].abs()))
        scale = bf["dG"].abs().amax(dim=(1, 2, 4), keepdim=True).clamp_min(1e-30)
        m["dG_free"] = norm_err(ref["dGk"], bf["dG"], scale.expand_as(bf["dG"])).amax(-1)
    for n in ("gates", "dG_tf"):
        if n in m:
            m[n] = m[n].amax(-1)                # (2, B, T, 4): worst unit of each gate block
    return m, exact


def violations(m: dict) -> dict:
    """name -> (n, 4) tensor of [direction, trace, step, block] (LSTM) or the flagged indices (attention) over its bar."""
    return {n: (e > BARS[n]).nonzero() for n, e in m.items() if bool((e > BARS[n]).any())}


def worst(m: dict) -> dict:
    return {n: float(e.max()) for n, e in m.items()}


def test_lstm_matrix_reaches_every_instantiation():
    reached = {(c.H if c.expect[0] == "register" else c.expect[2], c.expect[1]) for c in LSTM_MATRIX}
    for c in LSTM_MATRIX:
        assert lstm_path(c.H, c.B) == c.expect, c
    assert {(32, 1), (32, 2), (32, 4), (32, 16), (64, 1), (64, 2), (64, 4), (64, 16)} <= reached
    assert {(2, 1), (2, 4), (1, 1), (1, 4)} <= reached           # (S, R) of the general kernels
    assert not any(pick_r(B) == 8 for B in range(1, 5000))       # lstm_reg_*<HH, 8> cannot be reached
    for c in LSTM_MATRIX:                                       # a partial last CTA where the table says so
        if c.B in (593, 601, 301):
            R_, S_ = c.expect[1], c.expect[2] or 1
            assert c.B % (R_ * S_) != 0
    assert {c.T for c in LSTM_MATRIX} == set(_TS)


@pytest.mark.parametrize("m_", MODES)
@pytest.mark.parametrize("c", LSTM_MATRIX, ids=str)
def test_lstm_per_step(c, m_):
    inp = lstm_inputs(c)
    with mode(m_):
        k = run_lstm(c, inp)
        inf = run_lstm(c, inp, save=False, backward=False)
    assert same_bits(inf["out"], k["out"]), "inference (saved = NULL) changed out"
    m, exact = lstm_measure(c, k, lstm_reference(c, inp, k))
    assert exact == [] and violations(m) == {}, (worst(m), exact, {n: v[:8].tolist() for n, v in violations(m).items()})


@pytest.mark.parametrize("c", [LCase(32, 601, 9, None), LCase(64, 297, 8, None), LCase(64, 149, 2, None),
                               LCase(128, 301, 9, None), LCase(96, 3, 9, None), LCase(256, 301, 2, None)], ids=str)
def test_lstm_trace_permutation(c):
    """Permuting the traces of a batch (same B, so the same R) permutes every output bit for bit."""
    inp = lstm_inputs(c)
    k = run_lstm(c, inp)
    perm = torch.randperm(c.B, generator=torch.Generator().manual_seed(c.B)).cuda()
    pin = dict(inp, P=inp["P"][perm].contiguous(), d_out=inp["d_out"][perm].contiguous())
    kp = run_lstm(c, pin)
    assert same_bits(kp["out"], k["out"][perm])
    assert same_bits(kp["saved"], k["saved"][:, perm])
    assert same_bits(kp["dG"], k["dG"][perm])


# ------------------------------------------------------------------------------------------- layer assembly, exact family
def ints(shape, g, lo, hi, density=1.0):
    v = torch.randint(lo, hi + 1, shape, generator=g, device="cuda").float()
    return v * (torch.rand(shape, generator=g, device="cuda") < density)


ASM_CASES = [(128, 1, 30), (128, 40, 110), (256, 1, 4200), (256, 3, 20), (192, 40, 110), (192, 1, 9)]


@pytest.mark.parametrize("m_", MODES)
@pytest.mark.parametrize("drop", [False, True])
@pytest.mark.parametrize("d_model,B,T", ASM_CASES)
def test_layer_assembly_exact(d_model, B, T, drop, m_):
    """Small-integer dG, out and xin: every fp32 sum is exact and the bf16x6 split holds each integer in its hi term, so
    lstm_grads_from_dG must equal the float64 reference bit for bit -- on rs_sgemm below TC_MIN_ROWS and at d_model 192,
    on tn_tc / nt_tc from TC_MIN_ROWS at d_model 128 and 256."""
    H, I = d_model // 2, d_model
    g = torch.Generator(device="cuda").manual_seed(d_model + B + T + drop)
    xin = ints((B, T + 2, I), g, -2, 2)
    mask = ints((B, T, I), g, 0, 1) * 2.0 if drop else None
    w = [ints(s, g, -2, 2, 0.3) for s in ((4 * H, I), (4 * H, H), (4 * H,), (4 * H,))] * 2
    with mode(m_):
        _, _, xin_saved, w_ih_cat, _, tc = LM.lstm_layer_fwd(xin, mask, w)
        assert tc == (B * (T + 2) >= F_.TC_MIN_ROWS and d_model != 192)
        dG = torch.zeros(B, T + 2, 8 * H, device="cuda")
        dG[:, 1:-1] = ints((B, T, 8 * H), g, -3, 3, 0.5)
        out = torch.zeros(B, T + 2, 2 * H, device="cuda")
        out[:, 1:-1] = ints((B, T, 2 * H), g, -3, 3, 0.5)
        dW_ih, dW_hh, db, d_xin = LM.lstm_grads_from_dG(dG, out, xin_saved, w_ih_cat, mask, tc)
    want = R.lstm_weight_grads(dG, out, xin, mask) + (R.data_grad(dG, w_ih_cat, mask),)
    for name, got, ref in zip(("dW_ih", "dW_hh", "db", "d_xin"), (dW_ih, dW_hh, db, d_xin), want):
        assert torch.equal(ref.float().double(), ref), name       # representable: the comparison is exact
        assert torch.equal(got.double(), ref), (name, float((got.double() - ref).abs().max()))


# ------------------------------------------------------------------------------------------------------- autograd tie
@pytest.mark.parametrize("d_model,B,T", [(128, 3, 50), (128, 40, 110), (192, 5, 20)])
def test_lstm_autograd_equals_module_functions(d_model, B, T):
    H, I = d_model // 2, d_model
    g = torch.Generator(device="cuda").manual_seed(B + T)
    xin = torch.zeros(B, T + 2, I, device="cuda")
    xin[:, 1:-1] = torch.randn(B, T, I, generator=g, device="cuda")
    mask = (torch.rand(B, T, I, generator=g, device="cuda") < 0.9).float() / 0.9
    w = [((torch.rand(*s, generator=g, device="cuda") * 2 - 1) / math.sqrt(H)) for s in ((4 * H, I), (4 * H, H), (4 * H,), (4 * H,))] * 2
    d_out = torch.randn(B, T + 2, 2 * H, generator=g, device="cuda")
    with mode("deterministic"):
        x = xin.clone().requires_grad_(True)
        wa = [t.clone().requires_grad_(True) for t in w]
        out_a = LM.LSTMLayerFn.apply(x, mask, *wa)
        out_a.backward(d_out)
        out, saved, xs, w_ih_cat, w_hh_cat, tc = LM.lstm_layer_fwd(xin, mask, w)
        dW_ih, dW_hh, db, d_xin = LM.lstm_grads_from_dG(LM.lstm_bptt(d_out, saved, w_hh_cat), out, xs, w_ih_cat, mask, tc)
    assert same_bits(out_a.detach(), out)
    assert same_bits(x.grad, d_xin)
    want = (dW_ih[:4 * H], dW_hh[0], db[:4 * H], db[:4 * H], dW_ih[4 * H:], dW_hh[1], db[4 * H:], db[4 * H:])
    for i, (a, b) in enumerate(zip(wa, want)):
        assert same_bits(a.grad, b), i


def test_query_attn_autograd_equals_module_functions():
    B, N, D, Q = 3, 500, 128, 80
    a = attn_inputs(ACase(D, Q, N, B, 11, "p90", 3.0))
    mem = a["memory"][:, :, :D].contiguous()
    mem[:, 0] = 0
    mem[:, -1] = 0
    tr = a["traces"].clone()
    tr[..., 3:] = 0
    with mode("deterministic"):
        mean, rms, count = LM.trace_stats(tr, a["mask"])
        m_ = mem.clone().requires_grad_(True)
        qk, qb = a["qk"].clone().requires_grad_(True), a["qb"].clone().requires_grad_(True)
        ctx, anc, summ = LM.QueryAttnFn.apply(m_, qk, qb, tr, a["mask"], mean, rms, count)
        (ctx * a["d_ctx"]).sum().add_((anc * a["d_anchor"]).sum()).add_((summ * a["d_summary"]).sum()).backward()
        c2, a2, s2, st2, splits = LM.query_attn_fwd(mem, a["qk"], a["qb"], tr, a["mask"], mean, rms)
        dm, dqk, dqb = LM.query_attn_bwd(mem, a["qk"], a["qb"], tr, a["mask"], mean, rms, count, c2, a2, st2, a["d_ctx"],
                                          a["d_anchor"], a["d_summary"], splits)
    for x, y in ((ctx, c2), (anc, a2), (summ, s2), (m_.grad, dm), (qk.grad, dqk), (qb.grad, dqb)):
        assert same_bits(x.detach(), y)


# ====================================================================================================== query attention
@dataclass(frozen=True)
class ACase:
    D: int
    Q: int
    N: int
    B: int
    F: int
    mask: str                 # "none" | "p90" | "first_chunk" | "last_only" | "dead" (one trace without a valid token)
    scale: float

    def __str__(self):
        return f"D{self.D}-Q{self.Q}-N{self.N}-B{self.B}-F{self.F}-{self.mask}-s{self.scale:g}"

    def splits(self):
        ch = (self.N + 31) // 32
        return sorted({1, 2, 4, ch, ch + 2, LM._splits(self.B, self.N, self.Q)})


A = ACase
ATTN_MATRIX = [
    A(32, 1, 1, 2, 3, "none", 0.1), A(32, 7, 31, 3, 11, "p90", 30.0), A(64, 32, 32, 2, 11, "first_chunk", 30.0),
    A(64, 33, 33, 3, 3, "dead", 0.1), A(96, 64, 160, 2, 11, "last_only", 30.0), A(96, 80, 3000, 2, 11, "p90", 30.0),
    A(128, 80, 3000, 3, 11, "dead", 30.0), A(128, 30, 3000, 20, 11, "p90", 0.1), A(192, 7, 160, 2, 3, "first_chunk", 30.0),
    A(192, 33, 33, 4, 11, "none", 30.0), A(256, 1, 3000, 2, 11, "last_only", 0.1), A(256, 64, 31, 3, 3, "dead", 30.0),
    A(256, 32, 160, 2, 11, "p90", 30.0), A(32, 80, 160, 2, 11, "first_chunk", 0.1), A(128, 7, 1, 3, 11, "none", 30.0),
]


def attn_inputs(c: ACase, seed=0):
    """memory rises along n in the direction u, and every qk row has a positive component along u: the scores rise
    along the trace, so the running max moves in every chunk.  scale sets the size of the scores."""
    g = torch.Generator(device="cuda").manual_seed(c.D + 100 * c.Q + c.N + seed)
    B, N, D, Q = c.B, c.N, c.D, c.Q
    u = torch.ones(D, device="cuda") / math.sqrt(D)
    inner = torch.randn(B, N, D, generator=g, device="cuda") * 0.5 + (2.0 * torch.arange(N, device="cuda") / max(N, 1))[None, :, None] * u
    memory = torch.full((B, N + 2, D + XM), float("nan"), device="cuda")
    memory[:, 1:-1, :D] = inner
    qk = (c.scale * (0.3 * torch.randn(Q, D, generator=g, device="cuda") / math.sqrt(D) + u)).contiguous()
    qb = 0.1 * torch.randn(Q, generator=g, device="cuda")
    traces = torch.full((B, N, c.F), float("nan"), device="cuda")
    traces[..., :3] = torch.randn(B, N, 3, generator=g, device="cuda") * 2 + 1
    mask = None
    if c.mask != "none":
        mk = torch.ones(B, N, dtype=torch.bool, device="cuda")
        if c.mask in ("p90", "dead"):
            mk = torch.rand(B, N, generator=g, device="cuda") < 0.9
            mk[:, 0] = True
        elif c.mask == "first_chunk":
            mk[:, 32:] = False
        elif c.mask == "last_only":
            mk[:] = False
            mk[:, N - 1] = True
        if c.mask == "dead":
            mk[B // 2] = False
        mask = mk.to(torch.uint8)
    return {"memory": memory, "qk": qk, "qb": qb, "traces": traces, "mask": mask,
            "d_ctx": torch.randn(B, Q, D, generator=g, device="cuda"), "d_anchor": torch.randn(B, Q, 3, generator=g, device="cuda"),
            "d_summary": torch.randn(B, D, generator=g, device="cuda")}


def run_stats(traces, mask):
    B, N, F = traces.shape
    out = [torch.full(s, float("nan"), device="cuda") for s in ((B, 3), (B,), (B,))]
    _lib.call("rs_trace_stats_f32", _p(traces), F, _p(mask), B, N, *[_p(t) for t in out], _st())
    return out


def run_attn(c: ACase, a, splits, stats3, fwd=None):
    """Forward and backward through the C entry points; the backward reads `fwd`'s ctx / anchor / stats when given
    (another run's forward), else this run's own."""
    B, N, D, Q = c.B, c.N, c.D, c.Q
    mean, rms, count = stats3
    k = {n: torch.full(s, float("nan"), device="cuda") for n, s in (("ctx", (B, Q, D)), ("anchor", (B, Q, 3)), ("summary", (B, D)),
                                                                 ("stats", (B, Q, 2)))}
    ws = torch.full((_lib.load().rs_query_attn_workspace(B, Q, D, splits),), float("nan"), device="cuda")
    mem = a["memory"]
    _lib.call("rs_query_attn_fwd_f32", _p(mem), D + XM, N + 2, 1, _p(a["traces"]), c.F, _p(a["mask"]), _p(mean), _p(rms),
              _p(a["qk"]), _p(a["qb"]), B, N, Q, D, splits, _p(ws), _p(k["ctx"]), _p(k["anchor"]), _p(k["summary"]), _p(k["stats"]), _st())
    f = fwd if fwd is not None else k
    atomic = Q > 32 and not torch.are_deterministic_algorithms_enabled()      # the atomic variant adds onto zeros
    k["d_memory"] = framed(B, N, D, XM, inner=0.0 if atomic else float("nan"))
    dq_part = torch.full((B * splits, Q * (D + 1)), float("nan"), device="cuda")
    _lib.call("rs_query_attn_bwd_f32", _p(mem), D + XM, N + 2, 1, _p(a["traces"]), c.F, _p(a["mask"]), _p(mean), _p(rms),
              _p(count), _p(a["qk"]), _p(a["qb"]), _p(f["ctx"]), _p(f["anchor"]), _p(f["stats"]), _p(a["d_ctx"]), _p(a["d_anchor"]),
              _p(a["d_summary"]), B, N, Q, D, splits, _p(k["d_memory"]), D + XM, N + 2, 1, _p(dq_part), _st())
    dq = torch.empty(Q * (D + 1), device="cuda")
    F_.colsum(dq_part, dq)
    k["dqk"], k["dqb"] = dq.view(Q, D + 1)[:, :D], dq.view(Q, D + 1)[:, D]
    k["dq_part_finite"] = bool(torch.isfinite(dq_part).all())
    torch.cuda.synchronize()
    return k


def attn_reference(c: ACase, a, stats3, **fault):
    mean, rms, count = stats3
    mem = a["memory"][:, 1:-1, :c.D]
    mask = a["mask"].bool() if a["mask"] is not None else None
    fw = R.attn_fwd(mem, a["qk"], a["qb"], a["traces"], mask, mean, rms, **fault)
    bw = R.attn_bwd(mem, a["qk"], fw, count, a["d_ctx"], a["d_anchor"], a["d_summary"])
    return fw, bw


def attn_measure(c: ACase, k, fw, bw):
    live = fw["valid"].any(1)
    m, exact = {}, []
    if not frame_intact(k["d_memory"], c.D):
        exact.append("d_memory_frame")
    if not k["dq_part_finite"]:
        exact.append("dq_part_unwritten")
    # a trace without a valid token: NaN ctx / anchor, summary 0, stats (-inf, 0), zero d_memory (documented)
    dead = ~live
    if bool(dead.any()):
        if not bool(torch.isnan(k["ctx"][dead]).all() and torch.isnan(k["anchor"][dead]).all()):
            exact.append("dead_ctx")
        if not bool((k["summary"][dead] == 0).all()):
            exact.append("dead_summary")
        if not bool((k["stats"][dead][..., 0] == -math.inf).all() and (k["stats"][dead][..., 1] == 0).all()):
            exact.append("dead_stats")
        if not bool((k["d_memory"][dead][:, 1:-1, :c.D] == 0).all()):
            exact.append("dead_d_memory")
    z = lambda t: torch.where(live.view(-1, *([1] * (t.dim() - 1))), t, torch.zeros_like(t))      # noqa: E731
    m["ctx"] = z(norm_err(k["ctx"], torch.nan_to_num(fw["ctx"]), fw["ctx_bound"])).amax(-1)             # (B, Q)
    m["anchor"] = z(norm_err(k["anchor"], torch.nan_to_num(fw["anchor"]), fw["anchor_bound"])).amax(-1)
    m["summary"] = norm_err(k["summary"], fw["summary"], fw["summary_bound"].amax(-1, keepdim=True) + 1e-30).amax(-1)   # (B,)
    st = k["stats"].to(F64)
    lse = fw["stats"][..., 0] + torch.log(fw["stats"][..., 1])
    m["stats"] = z(norm_err(st[..., 0] + torch.log(st[..., 1]), torch.nan_to_num(lse, neginf=0.0), 1.0 + fw["S"].amax(-1)))
    m["d_memory"] = norm_err(k["d_memory"][:, 1:-1, :c.D], bw["d_memory"], bw["d_memory_bound"] + 1e-300).amax(-1)  # (B, N)
    m["dqk"] = norm_err(k["dqk"], bw["dqk"], bw["dqk_bound"]).amax(-1)                                  # (Q,)
    m["dqb"] = norm_err(k["dqb"], bw["dqb"], bw["dqb_bound"])
    return m, exact


def test_attn_matrix_covers_the_issue_values():
    assert {c.D for c in ATTN_MATRIX} == {32, 64, 96, 128, 192, 256}
    assert {c.Q for c in ATTN_MATRIX} >= {1, 7, 32, 33, 64, 80}
    assert {c.N for c in ATTN_MATRIX} == {1, 31, 32, 33, 160, 3000}
    assert {c.F for c in ATTN_MATRIX} == {3, 11}
    assert {c.mask for c in ATTN_MATRIX} == {"none", "p90", "first_chunk", "last_only", "dead"}
    assert {c.scale for c in ATTN_MATRIX} == {0.1, 30.0}
    assert any(c.splits()[-1] > (c.N + 31) // 32 for c in ATTN_MATRIX)
    # the reference batch of the benchmark (20 x 3000, Q 30) picks 15 splits of 224 tokens: split 14 starts past N
    assert LM._splits(20, 3000, 30) == 15 and 14 * 7 * 32 >= 3000


@pytest.mark.parametrize("m_", MODES)
@pytest.mark.parametrize("c", ATTN_MATRIX, ids=str)
def test_query_attention(c, m_):
    a = attn_inputs(c)
    with mode(m_):
        stats3 = run_stats(a["traces"], a["mask"])
        fw, bw = attn_reference(c, a, stats3)
        runs = {}
        for s in c.splits():
            k = run_attn(c, a, s, stats3)
            m, exact = attn_measure(c, k, fw, bw)
            assert exact == [] and violations(m) == {}, (s, worst(m), exact, {n: v[:8].tolist() for n, v in violations(m).items()})
            runs[s] = k
        if c.Q > 32 and m_ == "deterministic":
            again = run_attn(c, a, c.splits()[0], stats3)
            for n in ("ctx", "anchor", "summary", "stats", "d_memory", "dqk", "dqb"):
                assert same_bits(again[n], runs[c.splits()[0]][n]), n
        if c.Q <= 32:   # the chunk boundaries do not move and no atomics are involved: with the same forward outputs,
            first = runs[c.splits()[0]]                 # d_memory does not depend on the split count
            for s in c.splits():
                assert same_bits(run_attn(c, a, s, stats3, fwd=first)["d_memory"], first["d_memory"]), s


# ------------------------------------------------------------------------------------------------------- trace stats
def stats_traces(B, N, F, kind, g):
    """Values on a 2^-12 grid below 2^11 in magnitude: every float64 sum of them is exact in any order."""
    t = torch.full((B, N, F), float("nan"), device="cuda")
    x = torch.randn(B, N, 3, generator=g, device="cuda") * 3 + 5
    if kind == "offset":
        x = 1000.0 + torch.randn(B, N, 3, generator=g, device="cuda") * 0.01
    t[..., :3] = torch.round(x * 4096) / 4096
    return t


@pytest.mark.parametrize("m_", MODES)
@pytest.mark.parametrize("kind", ["none", "rand", "all_masked", "one_valid", "offset"])
@pytest.mark.parametrize("N", [1, 257, 5000])
def test_trace_stats(N, kind, m_):
    g = torch.Generator(device="cuda").manual_seed(N)
    B = 5
    t = stats_traces(B, N, 11 if N != 257 else 3, kind, g)
    mask = None
    if kind in ("rand", "offset"):
        mask = torch.rand(B, N, generator=g, device="cuda") < 0.7
    elif kind == "all_masked":
        mask = torch.zeros(B, N, dtype=torch.bool, device="cuda")
    elif kind == "one_valid":
        mask = torch.zeros(B, N, dtype=torch.bool, device="cuda")
        mask[torch.arange(B), torch.arange(B) * 37 % N] = True
    mu8 = mask.to(torch.uint8) if mask is not None else None
    with mode(m_):
        mean, rms, count = run_stats(t, mu8)
    wm, wr, wc = R.trace_stats(t, mask)
    assert torch.equal(mean.double(), wm), (mean, wm)
    assert torch.equal(count.double(), wc)
    ulp = torch.abs(torch.nextafter(wr.float(), torch.full_like(wr.float(), math.inf)).double() - wr)
    assert bool(((rms.double() - wr).abs() <= ulp).all()), (rms, wr)
    if kind in ("all_masked", "one_valid"):
        assert bool((rms == torch.tensor(1e-3, dtype=torch.float32)).all())


# ============================================================================================================ sensitivity
SENS_L = LCase(64, 601, 20, ("register", 16, None))
SENS_A = ACase(128, 33, 3000, 3, 11, "p90", 3.0)


@pytest.fixture(scope="module")
def lstm_sens():
    inp = lstm_inputs(SENS_L)
    k = run_lstm(SENS_L, inp)
    m, exact = lstm_measure(SENS_L, k, lstm_reference(SENS_L, inp, k))
    assert exact == [] and violations(m) == {}, worst(m)
    return inp, k


def _flagged(v, names):
    """Rows [direction, trace, step, block] of the named checks' violations."""
    rows = [v[n] for n in names if n in v]
    return torch.cat(rows) if rows else torch.zeros(0, 4, dtype=torch.long, device="cuda")


@pytest.mark.parametrize("fault", ["swap_if", "rev_from_before", "c0", "drop_last", "dc_no_f", "swap_dout"])
def test_lstm_checkers_locate_injected_faults(lstm_sens, fault):
    """The kernel runs once; the reference is then built with one fault.  Each must be reported where it is."""
    inp, k = lstm_sens
    c, T, B = SENS_L, SENS_L.T, SENS_L.B
    m, _ = lstm_measure(c, k, lstm_reference(c, inp, k, **{fault: 0.25 if fault == "c0" else True}))
    v = violations(m)
    assert v, fault
    if fault == "swap_if":
        f = _flagged(v, ["gates"])
        assert set(f[:, 3].tolist()) == {0, 1} and set(f[:, 0].tolist()) == {0, 1}
    elif fault == "rev_from_before":
        f = _flagged(v, ["gates"])
        assert len(f) and set(f[:, 0].tolist()) == {1}
        assert "c" not in v and "out" not in v
    elif fault == "c0":
        f = _flagged(v, ["c"])
        assert set(map(tuple, f[:, [0, 2]].tolist())) <= {(0, 0), (1, T - 1)} and len(f)
        assert set(v) == {"c"}
    elif fault == "drop_last":
        f = _flagged(v, ["gates", "out_free"])
        assert len(f) and set(f[:, 1].tolist()) == {B - 1}
    elif fault == "dc_no_f":
        assert "dG_tf" in v and not {"gates", "c", "out"} & set(v)
        f = _flagged(v, ["dG_tf"])
        assert (f[f[:, 0] == 0][:, 2] < T - 1).all() and (f[f[:, 0] == 1][:, 2] > 0).all()     # never a direction's first step
    else:
        f = _flagged(v, ["dG_tf"])
        assert set(f[:, 0].tolist()) == {0, 1} and not {"gates", "c", "out"} & set(v)


@pytest.fixture(scope="module")
def attn_sens():
    c = SENS_A
    a = attn_inputs(c)
    stats3 = run_stats(a["traces"], a["mask"])
    splits = 8
    k = run_attn(c, a, splits, stats3)
    m, exact = attn_measure(c, k, *attn_reference(c, a, stats3))
    assert exact == [] and violations(m) == {}, worst(m)
    return a, stats3, k, splits


@pytest.mark.parametrize("fault", ["skip_alpha", "summary_by_n", "ignore_mask", "anchor_y_for_z"])
def test_attention_checkers_locate_injected_faults(attn_sens, fault):
    a, stats3, k, splits = attn_sens
    c = SENS_A
    tps = (((c.N + 31) // 32 + splits - 1) // splits) * 32
    if fault == "skip_alpha":
        kw = {"skip_alpha_split": 2, "tokens_per_split": tps}
    elif fault == "ignore_mask":
        n0 = int((a["mask"][1] == 0).nonzero()[len((a["mask"][1] == 0).nonzero()) // 2])
        kw = {"ignore_mask_at": (1, n0)}
    else:
        kw = {fault: True}
    fw, bw = attn_reference(c, a, stats3, **kw)
    if fault == "skip_alpha":   # one split of every trace: every query's ctx is off, and the d_memory rows of that split
        v = violations(attn_measure(c, k, fw, bw)[0])
        assert "ctx" in v and "d_memory" in v
        rows = v["d_memory"][:, 1]
        assert bool(((rows >= 2 * tps) & (rows < 3 * tps)).any())
    elif fault == "summary_by_n":
        v = violations(attn_measure(c, k, fw, bw)[0])
        assert set(v) == {"summary"} or set(v) <= {"summary", "d_memory"}
        assert "summary" in v
    elif fault == "ignore_mask":
        v = violations(attn_measure(c, k, fw, bw)[0])
        assert [1, n0] in v["d_memory"].tolist()          # the token's own row, in its trace, and nothing in the others
        assert all(set(x[:, 0].tolist()) == {1} for n, x in v.items() if n in ("ctx", "anchor", "summary", "stats", "d_memory"))
    else:
        v = violations(attn_measure(c, k, fw, bw)[0])
        assert set(v) == {"anchor"} or set(v) <= {"anchor", "d_memory", "dqk", "dqb"}
        assert "anchor" in v and "ctx" not in v
