"""The bf16 GRU recurrence kernels called through their C entry points and checked step by step against the float64
reference of oracle/rec_bf16_ref.py (itself checked against torch.nn.GRU by test_rec_bf16_ref.py).

rs_rec_fwd_bf16 / rs_rec_bwd_bf16 (csrc/rec_pair.cu, H = 128), rs_rec_fwd_bf16_wide / rs_rec_bwd_bf16_wide (csrc/rec_wide.cu,
H = 256) and the weight images of rs_gru_pack_weights_bf16 (csrc/pack_w.cu) and functional_bf16.wide_fwd_image /
wide_bwd_image.  Every output buffer is filled with NaN before a call, so an element a kernel fails to write cannot pass.

What is checked, per case of the matrix below:
  * weight images: bit for bit against the same images built here with torch from the documented layouts;
  * forward, teacher-forced: the saved gates against the reference step computed from the kernel's own bf16 `out` of
    the step before (the MMA's A operand), per (direction, gate block, step); `out` against the blend
    z h_{t-1} + (1 - z) n of the saved gates; `out_drop` against out * scale; bf16(h_n) against `out` at each trace's
    last valid step (bit for bit);
  * exact zeros the weight- and data-gradient GEMMs rely on: `out` and `dG` at the pad rows t' = 0, T + 1, past each
    trace's length, and `dG` at the pad traces b >= B of the last tile (d_out is zero there, as to_tile_major writes it);
    z = 1 past a trace's length;
  * backward: dG per (direction, gate block, step), normalised by that block's largest reference value, against
      - the teacher-forced recursion, which feeds the kernel's own bf16 dG r | z | hn (its MMA's A operand) into
        [gr | gz | ghn] W_hh: the error stays at the bf16 rounding of the stored dG, so a fault shows at its step;
      - the free-running float64 recursion over the kernel's saved gates and `out`, which also carries the effect of
        feeding bf16 gradients into the matvec step after step;
  * bit-exact equivalences: one against two tiles in flight per CTA pair (RS_REC_MODE = 2 / 3, read on every call), an
    odd tile count included; lengths = None against lengths all T; gates = NULL (inference) against training.
The sensitivity test runs the checkers against references built from a deliberately wrong operand and requires each
fault to be reported at its direction, gate block and steps.

Bars (absolute for gates and out; hn and dG relative to their block's largest reference value), each about 4x the largest
error measured over the whole matrix on a B200 (1000 W power limit):
    gates r | z | n          GATE_BAR  = 1e-3      measured 2.5e-4   (tanh.approx.f32 and fp16 storage)
    gates hn (H = 256)       HN_BAR    = 1.6e-3    measured 4.4e-4
    out vs blend             BLEND_BAR = 1.6e-2    measured 4.2e-3   (one bf16 ulp at |h| in [0.5, 1) is 3.9e-3)
    dG, teacher-forced       DG_TF_BAR = 1.4e-2    measured 3.7e-3   (the bf16 rounding of the stored dG)
    dG, free-running         DG_BAR    = 1.6e-2    measured 4.0e-3
"""
import ctypes
import math
from dataclasses import dataclass, replace
from typing import Optional

import pytest
import torch

from oracle import rec_bf16_ref as R
from roomslam_b200 import _lib
from roomslam_b200 import functional_bf16 as FB
from roomslam_b200 import layout as L

pytestmark = pytest.mark.gpu

GATE_BAR = 1e-3
HN_BAR = 1.6e-3
BLEND_BAR = 1.6e-2
DG_TF_BAR = 1.4e-2
DG_BAR = 1.6e-2
KEEP = 0.75
BF, F16 = torch.bfloat16, torch.float16


GIVEN = object()             # keyword default: the operand of the case itself


def _p(t):
    return 0 if t is None else t.data_ptr()


def _st():
    return torch.cuda.current_stream().cuda_stream


def nan_like(shape, dtype):
    return torch.full(shape, float("nan"), device="cuda", dtype=dtype)


def bits16(t):
    return t.contiguous().view(torch.int16)


# ------------------------------------------------------------------------------------------------------- cases, inputs
@dataclass(frozen=True)
class Case:
    H: int
    B: int
    T: int
    mode: str                 # "x": layer 0 with I inputs; "P": deeper layer, projection given; "X": deeper, fused projection
    I: int = 2
    split: int = 0
    lengths: str = "none"     # "none" | "full" | "rand" (contains 1 and T)
    drop: bool = False        # dropout bits in the forward (out_drop) and on d_out in the backward
    d_out: bool = True
    d_h_n: bool = True
    nt: Optional[str] = None  # RS_REC_MODE: "2" forces one tile in flight per pair, "3" two
    seed: int = 0

    def __str__(self):
        s = f"H{self.H}-B{self.B}-T{self.T}-{self.mode}{self.I if self.mode == 'x' else ''}-s{self.split}-len_{self.lengths}"
        s += ("-drop" if self.drop else "") + ("" if self.d_out else "-no_dout") + ("" if self.d_h_n else "-no_dhn")
        return s + (f"-mode{self.nt}" if self.nt else "")


def make_inputs(c: Case) -> dict:
    g = torch.Generator().manual_seed(1000 + c.seed)
    H, B, T = c.H, c.B, c.T
    Bp = L.n_tiles(B) * L.TILE
    Il = c.I if c.mode == "x" else 2 * H
    k = 1.0 / math.sqrt(H)
    u = lambda *s: ((torch.rand(*s, generator=g) * 2 - 1) * k).cuda()  # noqa: E731
    w = [u(3 * H, Il), u(3 * H, H) * 3.0, u(3 * H), u(3 * H)] + [u(3 * H, Il), u(3 * H, H) * 3.0, u(3 * H), u(3 * H)]
    inp = {"w": [t.contiguous() for t in w]}
    if c.mode == "x":
        inp["x"] = torch.randn(B, T, c.I, generator=g).cuda()
    elif c.mode == "P":
        P = torch.zeros(Bp, T + 2, 6 * H)
        P[:, 1:-1] = torch.randn(Bp, T, 6 * H, generator=g) * 0.7
        inp["P"] = R.to_tm(P.cuda())
    else:
        X = torch.zeros(Bp, T + 2, 2 * H)
        X[:B, 1:-1] = torch.rand(B, T, 2 * H, generator=g) * 2 - 1
        inp["X"] = R.to_tm(X.cuda())
    if c.lengths == "full":
        inp["lengths"] = torch.full((B,), T, dtype=torch.int32).cuda()
    elif c.lengths == "rand":
        ln = torch.randint(1, T + 1, (B,), generator=g, dtype=torch.int32)
        ln[0] = 1
        ln[-1] = T
        inp["lengths"] = ln.cuda()
    else:
        inp["lengths"] = None
    if c.drop:
        keep = torch.rand(L.n_tiles(B), T, L.TILE, 2 * H, generator=g) < KEEP
        bits = (keep.view(*keep.shape[:3], 2 * H // 8, 8).to(torch.int32) << torch.arange(8, dtype=torch.int32)).sum(-1)
        inp["drop"] = (bits.to(torch.uint8).cuda(), torch.tensor([1.0 / KEEP], dtype=torch.float32).cuda())
    else:
        inp["drop"] = None
    if c.d_out:
        d = torch.zeros(Bp, T + 2, 2 * H)
        d[:B, 1:-1] = torch.randn(B, T, 2 * H, generator=g)     # zero at the pad rows and pad traces, as to_tile_major
        inp["d_out"] = R.to_tm(d.cuda())
    else:
        inp["d_out"] = None
    inp["d_h_n"] = torch.randn(2, B, H, generator=g).cuda() if c.d_h_n else None
    return inp


# ------------------------------------------------------------------------------------------------------------ images
def ref_images_128(w, I, split, layer0, fused):
    """Every output of rs_gru_pack_weights_bf16, built with torch from the layouts pack_w.cu documents."""
    H = 128
    s = R.gate_scale(H, "cuda")
    parts = lambda v: [v] if not split else [R.bf16(v), v - R.bf16(v)]      # noqa: E731  (pack8 rounds each part to bf16)
    per = [w[:4], w[4:]]
    whh, bhn, bx, whhT = [], [], [], []
    for w_ih, w_hh, b_ih, b_hh in per:
        ws = w_hh * s[:, None]
        cols = torch.cat(parts(ws), 1)                                             # [3H][16 hi (+16 lo) chunks of 8]
        b = R.bias_x(b_ih, b_hh, H)
        if layer0 or fused:
            nx = 16 * FB.x_steps(I) if layer0 else 16
            xc = torch.zeros(3 * H, nx, device="cuda")
            bhi = R.bf16(b)
            xc[:, 6], xc[:, 7] = bhi, b - bhi
            if layer0:
                wsc = w_ih * s[:, None]
                whi = R.bf16(wsc)
                for i in range(I):
                    xc[:, FB.x_col(i, 0)] = whi[:, i]
                    xc[:, FB.x_col(i, 1)] = whi[:, i]
                    xc[:, FB.x_col(i, 2)] = wsc[:, i] - whi[:, i]
            cols = torch.cat([cols, xc], 1)
        whh.append(cols.view(3 * H, -1, 8).permute(1, 0, 2))
        bhn.append(b_hh[2 * H:])
        bx.append(b)
        whhT.append(torch.cat(parts(w_hh.t()), 1).view(H, -1, 8).permute(1, 0, 2))
    img = {"whh_img": torch.stack(whh).to(BF), "b_hn": torch.stack(bhn), "bias_x": torch.stack(bx), "whhT_img": torch.stack(whhT).to(BF)}
    if not layer0:
        w_all = torch.cat([w[0], w[4]], 0)                                         # [6H][I]
        sc = torch.cat([s, s])[:, None]
        img["wt_dgrad"] = L.tile_weight_nt(torch.cat(parts(w_all.t().contiguous()), 1))
        if fused:
            img["wih_img"] = (w_all * sc).view(2, 3 * H, I // 8, 8).permute(0, 2, 1, 3).to(BF)
        else:
            img["wt_proj"] = L.tile_weight_nt(torch.cat(parts(w_all * sc), 1))
    return img


def pack_128(w, I, split, layer0, fused):
    """rs_gru_pack_weights_bf16 into NaN-filled buffers (the shapes GRULayerBF16Fn allocates)."""
    H = 128
    xch = 2 * FB.x_steps(I) if layer0 else (2 if fused else 0)
    o = {"whh_img": nan_like((2, 16 * (1 + split) + xch, 3 * H, 8), BF), "b_hn": nan_like((2, H), torch.float32),
         "bias_x": nan_like((2, 3 * H), torch.float32), "whhT_img": nan_like((2, 48 * (1 + split), H, 8), BF)}
    if not layer0:
        o["wt_dgrad"] = nan_like((I // 128, 12 * (1 + split), 8, 128, 8), BF)
        if fused:
            o["wih_img"] = nan_like((2, I // 8, 3 * H, 8), BF)
        else:
            o["wt_proj"] = nan_like((6, (I // 64) * (1 + split), 8, 128, 8), BF)
    wp = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in w])
    _lib.call("rs_gru_pack_weights_bf16", ctypes.addressof(wp), H, I, split, _p(o["whh_img"]), _p(o["b_hn"]), _p(o["bias_x"]),
              _p(o.get("wt_proj")), _p(o["whhT_img"]), _p(o.get("wt_dgrad")), _p(o.get("wih_img")), _st())
    return o


def wide_images(w, layer0):
    wst, b_hn, _, _, _, w_hh_cat = FB.wide_fwd_image(*w, layer0)
    return wst, b_hn, FB.wide_bwd_image(w_hh_cat)


# ------------------------------------------------------------------------------------------------------ kernel calls
def run_kernels(c: Case, inp: dict, save_gates=True, backward=True, lengths=GIVEN) -> dict:
    """One forward and (optionally) one backward through the C entry points; every output NaN-filled first."""
    H, B, T = c.H, c.B, c.T
    tiles = L.n_tiles(B)
    w = inp["w"]
    ln = inp["lengths"] if lengths is GIVEN else lengths
    bits, scale = inp["drop"] if inp["drop"] is not None else (None, None)
    k = {"out": nan_like((tiles, T + 2, 2 * H // 8, 128, 8), BF), "h_n": nan_like((2, B, H), torch.float32)}
    k["out_drop"] = nan_like(k["out"].shape, BF) if bits is not None else None
    k["gates"] = nan_like((tiles, T, 2, (3 if H == 128 else 4) * H // 8, 128, 8), BF) if save_gates else None
    x = inp.get("x")
    if H == 128:
        layer0, fused = c.mode == "x", c.mode == "X"
        img = pack_128(w, c.I if layer0 else 2 * H, c.split, layer0, fused)
        k["img"] = img
        _lib.call("rs_rec_fwd_bf16", _p(x), c.I if layer0 else 0, _p(inp.get("P")), 6 * H if c.mode == "P" else 0, _p(inp.get("X")),
                  _p(img.get("wih_img")) if fused else 0, _p(img["whh_img"]), _p(img["b_hn"]), _p(k["out"]), _p(k["gates"]),
                  _p(k["h_n"]), _p(ln), _p(bits), _p(scale), _p(k["out_drop"]), c.split, B, T, _st())
    else:
        wst, b_hn, wtst = wide_images(w, c.mode == "x")
        _lib.call("rs_rec_fwd_bf16_wide", _p(x), c.I if x is not None else 0, _p(inp.get("P")), _p(wst), _p(b_hn), _p(k["out"]),
                  _p(k["gates"]), _p(k["h_n"]), _p(ln), _p(bits), _p(scale), _p(k["out_drop"]), B, T, _st())
    if backward:
        k["dG"] = nan_like((tiles, T + 2, H, 128, 8), BF)
        if H == 128:
            _lib.call("rs_rec_bwd_bf16", _p(inp["d_out"]), _p(inp["d_h_n"]), _p(k["gates"]), _p(k["out"]), _p(img["whhT_img"]),
                      _p(img["whh_img"]), img["whh_img"].shape[1], _p(img["b_hn"]), _p(k["dG"]), _p(ln), _p(bits), _p(scale),
                      c.split, B, T, _st())
        else:
            _lib.call("rs_rec_bwd_bf16_wide", _p(inp["d_out"]), _p(inp["d_h_n"]), _p(k["gates"]), _p(k["out"]), _p(wtst), _p(k["dG"]),
                      _p(ln), _p(bits), _p(scale), B, T, _st())
    torch.cuda.synchronize()
    return k


def run_with_mode(monkeypatch, c: Case, inp: dict, **kw) -> dict:
    if c.nt:
        monkeypatch.setenv("RS_REC_MODE", c.nt)
    else:
        monkeypatch.delenv("RS_REC_MODE", raising=False)
    return run_kernels(c, inp, **kw)


# ----------------------------------------------------------------------------------------------------- reference, checks
def reference(c: Case, inp: dict, k: dict, w=None, lengths=GIVEN, d_h_n=GIVEN, rev_shift=False) -> dict:
    """The float64 reference around the kernel outputs k.  The keyword arguments replace one operand (sensitivity test)."""
    H, B, T = c.H, c.B, c.T
    w = inp["w"] if w is None else w
    ln = inp["lengths"] if lengths is GIVEN else lengths
    dhn = inp["d_h_n"] if d_h_n is GIVEN else d_h_n
    W = R.ref_weights(w, H, c.split)
    outf = R.out_full(k["out"], H)
    Bp = outf.shape[1]
    act = R.active_mask(ln, Bp, T, "cuda")
    hp = R.h_prev_forward(outf, ln)
    hpb = R.h_prev_backward(outf)
    if rev_shift:                       # the reverse direction reading the step itself instead of the one before
        hp[1] = outf[1, :, 1:-1]
        hpb[1] = outf[1, :, 1:-1]
    if c.mode == "x":
        u = R.input_from_x(inp["x"], W, Bp)
    elif c.mode == "P":
        u = R.input_from_P(inp["P"], H)
    else:
        u = R.input_from_X(inp["X"], W)
    ref = {"W": W, "outf": outf, "act": act, "hp": hp, "hpb": hpb, "lengths": ln}
    ref["fwd"] = R.forward_step(hp, u, W, act)
    if k.get("gates") is None:
        return ref
    g = R.gates_full(k["gates"], H)
    ref["g"] = g
    if "dG" not in k:
        return ref
    hn = g[..., 3, :] if H == 256 else R.recompute_hn(hpb, W)
    d_out = R.out_full(inp["d_out"], H)[:, :, 1:-1] if inp["d_out"] is not None else None
    dh = None
    if dhn is not None:
        dh = torch.zeros(2, Bp, H, dtype=torch.float64, device="cuda")
        dh[:, :B] = dhn.double()
    drop = R.drop_full(*inp["drop"], H) if inp["drop"] is not None else None
    dGk = R.dG_full(k["dG"], H)
    ref["dGk"] = dGk
    args = (g[..., 0, :], g[..., 1, :], g[..., 2, :], hn, hpb, W, act)
    ref["dG_tf"] = R.backward(*args, d_out=d_out, d_h_n=dh, drop=drop, feedback=dGk[:, :, 1:-1][:, :, :, [0, 1, 3]])
    ref["dG_free"] = R.backward(*args, d_out=d_out, d_h_n=dh, drop=drop)
    return ref


def bf16_ulp(v):
    """The spacing of bf16 numbers at |v| (0 at v = 0: a zero must be exact)."""
    return torch.where(v != 0, 2.0 ** (torch.floor(torch.log2(v.abs().clamp_min(1e-30))) - 7), torch.zeros_like(v))


def per_step(err):
    """(2, Bp, T, ..., H) -> max over traces and units: (2, T, ...)."""
    return err.abs().amax(dim=-1).amax(dim=1)


def measure(c: Case, inp: dict, k: dict, ref: dict) -> dict:
    """Per (direction, block, step) errors of each check, and the located violations of the exact ones."""
    H, B, T = c.H, c.B, c.T
    act, outf = ref["act"], ref["outf"]
    m, exact = {}, []

    def located(name, bad):             # bad: (2, Bp, T) bool -> [(name, d, -1, t)] for each offending (direction, step)
        dt = bad.any(1).nonzero().tolist()
        exact.extend((name, d, -1, t) for d, t in dt)

    finite = {n: k[n] for n in ("out", "out_drop", "gates", "h_n", "dG") if k.get(n) is not None}
    for n, t in finite.items():
        v = t.view(F16) if n == "gates" else t
        if not bool(torch.isfinite(v).all()):
            exact.append(("unwritten_" + n, -1, -1, -1))
    # out: pad rows zero, zero past the length, bf16(h_n) = out at the last valid step
    located("out_pad", torch.stack([(outf[:, :, 0] != 0).any(-1), (outf[:, :, -1] != 0).any(-1)], 2))
    located("out_past_len", ((outf[:, :, 1:-1] != 0).any(-1)) & ~act[None])
    ln = ref["lengths"].long() if ref["lengths"] is not None else torch.full((B,), T, device="cuda", dtype=torch.long)
    hn_bf = k["h_n"].to(BF).double()
    last0 = outf[0, torch.arange(B, device="cuda"), ln]
    if not torch.equal(hn_bf[0], last0):
        exact.append(("h_n", 0, -1, -1))
    if not torch.equal(hn_bf[1], outf[1, :B, 1]):
        exact.append(("h_n", 1, -1, -1))
    # out_drop: exactly 0 where the bit is clear or past the length; elsewhere bf16(h scale) with out = bf16(h): within
    # half an ulp of itself plus scale times half an ulp of out of out * scale
    if k.get("out_drop") is not None:
        od = R.out_full(k["out_drop"], H)[:, :, 1:-1]
        mult = R.drop_full(*inp["drop"], H) * act[None, :, :, None]
        want = outf[:, :, 1:-1] * mult
        tol = 0.5 * bf16_ulp(od) + 0.5 * mult * bf16_ulp(outf[:, :, 1:-1])
        located("out_drop", ((od - want).abs() > tol).any(-1))
        located("out_drop_pad", torch.stack([(R.out_full(k["out_drop"], H)[:, :, p] != 0).any(-1) for p in (0, -1)], 2))
    if "g" in ref:
        g, f = ref["g"], ref["fwd"]
        m["gates"] = torch.stack([per_step(g[..., i, :] - f[n]) for i, n in enumerate("rzn")], 2)    # (2, T, 3)
        if H == 256:
            m["hn"] = per_step(g[..., 3, :] - f["hn"]) / f["hn"].abs().amax(dim=(1, 2, 3))[:, None]
        located("z_past_len", ((g[..., 1, :] != 1).any(-1)) & ~act[None])
        blend = g[..., 1, :] * ref["hp"] + (1 - g[..., 1, :]) * g[..., 2, :]
        m["blend"] = per_step((outf[:, :, 1:-1] - blend) * act[None, :, :, None])
    if "dG_tf" in ref:
        dGk = ref["dGk"]
        located("dG_pad", torch.stack([(dGk[:, :, p] != 0).flatten(2).any(-1) for p in (0, -1)], 2))
        inner = dGk[:, :, 1:-1]
        located("dG_past_len", (inner != 0).flatten(3).any(-1) & ~act[None])
        if inner.shape[1] > B:
            located("dG_pad_traces", (inner[:, B:] != 0).flatten(3).any(-1))
        for name, r in (("dG_tf", ref["dG_tf"]), ("dG", ref["dG_free"])):
            scale = r.abs().amax(dim=(1, 2, 4)).clamp_min(1e-30)                                      # (2, 4)
            m[name] = (inner - r).abs().amax(dim=(1, 4)) / scale[:, None, :]                           # (2, T, 4)
    m["exact"] = exact
    return m


BARS = {"gates": GATE_BAR, "hn": HN_BAR, "blend": BLEND_BAR, "dG_tf": DG_TF_BAR, "dG": DG_BAR}


def failures(m: dict) -> list:
    """[(check, direction, block, step)] of every bar exceeded, then the exact violations (block / step -1: not applicable)."""
    out = []
    for name, bar in BARS.items():
        if name not in m:
            continue
        e = m[name]
        e = e[..., None] if e.dim() == 2 else e                     # (2, T, blocks)
        for d, t, b in (e > bar).nonzero().tolist():
            out.append((name, d, b, t))
        if bool(torch.isnan(e).any()):
            out.append((name + "_nan", -1, -1, -1))
    return out + m["exact"]


def summary(m: dict) -> dict:
    return {n: float(v.max()) for n, v in m.items() if n != "exact"}


# ---------------------------------------------------------------------------------------------------------- the matrix
C = Case
MATRIX = [
    C(128, 1, 1, "x", I=1, split=1),
    C(128, 127, 2, "x", I=2, lengths="full", drop=True, d_h_n=False),
    C(128, 128, 3, "x", I=3, split=1, lengths="rand", d_out=False),
    C(128, 129, 37, "x", I=4, lengths="rand", drop=True),
    C(128, 300, 37, "x", I=5, lengths="rand", nt="3"),                        # 3 tiles, two in flight: the last pair has one
    C(128, 300, 200, "x", I=10, split=1, lengths="rand", drop=True, nt="3"),
    C(128, 4987, 37, "x", I=11, lengths="rand", drop=True),                   # 39 tiles: automatically two in flight, odd count
    C(128, 129, 37, "x", I=15, split=1, nt="3"),                              # split + 3 input K steps: the host runs one tile
    C(128, 300, 37, "x", I=16, split=1, lengths="rand", drop=True, nt="3"),   # split + 4 input K steps: likewise
    C(128, 129, 37, "x", I=16, lengths="rand", drop=True),
    C(128, 300, 37, "P", lengths="rand", drop=True, nt="3"),
    C(128, 127, 37, "P", split=1, d_h_n=False),
    C(128, 4987, 37, "P", lengths="rand"),
    C(128, 129, 37, "X", lengths="rand", drop=True),
    C(128, 300, 200, "X", d_out=False),
    C(256, 1, 1, "x", I=2),
    C(256, 128, 2, "x", I=2, d_h_n=False),
    C(256, 129, 37, "x", I=11, lengths="rand", drop=True),
    C(256, 300, 200, "x", I=16, lengths="rand"),
    C(256, 127, 37, "P", lengths="full", drop=True, d_out=False),
    C(256, 300, 3, "P", lengths="rand"),
]


@pytest.mark.parametrize("c", MATRIX, ids=str)
def test_forward_backward_per_step(monkeypatch, c):
    inp = make_inputs(c)
    k = run_with_mode(monkeypatch, c, inp)
    m = measure(c, inp, k, reference(c, inp, k))
    assert failures(m) == [], (summary(m), failures(m)[:20])


# ------------------------------------------------------------------------------------------------------ weight images
PACK_CASES = [(I, s, True, False) for I in (1, 2, 3, 4, 5, 10, 11, 15, 16) for s in (0, 1)] + \
             [(256, 0, False, False), (256, 1, False, False), (256, 0, False, True)]


@pytest.mark.parametrize("I,split,layer0,fused", PACK_CASES)
def test_pack_weights_bit_exact(I, split, layer0, fused):
    inp = make_inputs(Case(128, 1, 1, "x" if layer0 else "P", I=I if layer0 else 2))
    got = pack_128(inp["w"], I, split, layer0, fused)
    want = ref_images_128(inp["w"], I, split, layer0, fused)
    assert sorted(got) == sorted(want)
    for n in got:
        a, b = got[n], want[n]
        assert a.shape == b.shape, n
        if a.dtype == BF:
            assert torch.equal(bits16(a), bits16(b)), n
        else:
            assert torch.equal(a.view(torch.int32), b.contiguous().view(torch.int32)), n


@pytest.mark.parametrize("I", [2, 11, 16, 512])
def test_wide_images_follow_documented_layout(I):
    """H = 256: Wst [2 dirs][2 ranks][K steps][2 chunks][384 rows][8], rows = r | z | n rows of hidden units
    [128 rank, 128 rank + 128), K = bf16(W_hh) (r, z / 2) then (layer 0) the input columns and a zero K step up to whole
    stages of two; WTst [2][2][48][2][128][8] = bf16(W_hh)^T."""
    H, layer0 = 256, I <= 16
    inp = make_inputs(Case(H, 1, 1, "x" if layer0 else "P", I=I if layer0 else 2))
    w = inp["w"]
    wst, b_hn, wtst = wide_images(w, layer0)
    s = R.gate_scale(H, "cuda")
    for d in (0, 1):
        w_ih, w_hh, b_ih, b_hh = w[4 * d: 4 * d + 4]
        K = [w_hh * s[:, None]]
        if layer0:
            xs = FB.x_steps(I)
            xc = torch.zeros(3 * H, 16 * (xs + xs % 2), device="cuda")
            b = R.bias_x(b_ih, b_hh, H)
            wsc = w_ih * s[:, None]
            whi = R.bf16(wsc)
            for i in range(I):
                xc[:, FB.x_col(i, 0)] = whi[:, i]
                xc[:, FB.x_col(i, 1)] = whi[:, i]
                xc[:, FB.x_col(i, 2)] = wsc[:, i] - whi[:, i]
            xc[:, 6], xc[:, 7] = R.bf16(b), b - R.bf16(b)
            K.append(xc)
        wk = torch.cat(K, 1).to(BF)                                          # [3H][K]
        ks = wk.shape[1] // 16
        want = wk.view(3, 2, 128, ks, 2, 8).permute(1, 3, 4, 0, 2, 5).reshape(2, ks, 2, 384, 8)
        assert torch.equal(bits16(wst[d]), bits16(want)), d
        assert torch.equal(b_hn[d], b_hh[2 * H:])
        wt = w_hh.t().to(BF).reshape(2, 128, 48, 2, 8).permute(0, 2, 3, 1, 4)
        assert torch.equal(bits16(wtst[d]), bits16(wt)), d


# ------------------------------------------------------------------------------------------------ bit-exact equivalences
def assert_same(a: dict, b: dict, names):
    for n in names:
        if a.get(n) is None and b.get(n) is None:
            continue
        x, y = a[n], b[n]
        eq = torch.equal(bits16(x), bits16(y)) if x.dtype in (BF, F16) else torch.equal(x.view(torch.int32), y.view(torch.int32))
        assert eq, n


@pytest.mark.parametrize("c", [
    C(128, 300, 37, "x", I=2, lengths="rand", drop=True),                     # 3 tiles: the second pair carries one
    C(128, 300, 37, "x", I=11, lengths="rand"),
    C(128, 300, 37, "x", I=16, drop=True),
    C(128, 300, 37, "P", split=1, lengths="rand", drop=True),
    C(128, 4987, 5, "x", I=2, lengths="rand", drop=True),                     # 39 tiles
], ids=str)
def test_one_against_two_tiles_in_flight(monkeypatch, c):
    inp = make_inputs(c)
    one = run_with_mode(monkeypatch, replace(c, nt="2"), inp, backward=False)
    two = run_with_mode(monkeypatch, replace(c, nt="3"), inp, backward=False)
    assert_same(one, two, ("out", "gates", "h_n", "out_drop"))
    if c.B > 37 * 128:                  # the automatic choice at 39 tiles is two in flight
        auto = run_with_mode(monkeypatch, replace(c, nt=None), inp, backward=False)
        assert_same(two, auto, ("out", "gates", "h_n", "out_drop"))


@pytest.mark.parametrize("c", [
    C(128, 129, 37, "x", I=2, drop=True), C(128, 300, 37, "x", I=11, split=1), C(128, 129, 37, "P"), C(128, 129, 37, "X"),
    C(256, 129, 37, "x", I=2, drop=True), C(256, 129, 37, "P"),
], ids=str)
def test_lengths_none_equals_all_full(c):
    inp = make_inputs(c)
    a = run_kernels(c, inp, lengths=None)
    b = run_kernels(c, inp, lengths=torch.full((c.B,), c.T, dtype=torch.int32, device="cuda"))
    assert_same(a, b, ("out", "gates", "h_n", "dG", "out_drop"))


@pytest.mark.parametrize("c", [
    C(128, 300, 37, "x", I=2, lengths="rand", drop=True), C(128, 129, 37, "x", I=16, split=1), C(128, 129, 37, "X", lengths="rand"),
    C(128, 4987, 5, "P"), C(256, 129, 37, "x", I=11, lengths="rand", drop=True), C(256, 129, 37, "P"),
], ids=str)
def test_inference_equals_training_forward(c):
    inp = make_inputs(c)
    a = run_kernels(c, inp, save_gates=False, backward=False)
    b = run_kernels(c, inp, backward=False)
    assert_same(a, b, ("out", "h_n", "out_drop"))


# ------------------------------------------------------------------------------------------------ tests of the tests
SENS = C(128, 300, 37, "x", I=2, lengths="rand", drop=True, nt="3")


@pytest.fixture(scope="module")
def sens_run():
    inp = make_inputs(SENS)
    with pytest.MonkeyPatch.context() as mp:
        k = run_with_mode(mp, SENS, inp)
    m = measure(SENS, inp, k, reference(SENS, inp, k))
    assert failures(m) == [], summary(m)
    return inp, k


@pytest.mark.parametrize("fault", ["w_hh", "length", "d_h_n", "rev_shift"])
def test_checkers_locate_injected_faults(sens_run, fault):
    """The kernel runs once; the reference is then built from one wrong operand.  Each fault must be reported, at the
    direction, gate block and steps it touches -- a checker reading kernel outputs at the wrong place would miss it."""
    inp, k = sens_run
    c, T, H = SENS, SENS.T, SENS.H
    if fault == "w_hh":
        # one W_hn element of the reverse direction moved by 2^-5, on the hidden unit with the largest mean |h|: the
        # forward n gate of that direction is off at every step.  (In the backward the same element moves one term of a
        # K = 384 sum against a single gradient: below the dG bars, which sit at the bf16 rounding of dG.)
        outf = R.out_full(k["out"], H)
        col = int(outf[1, :c.B].abs().mean((0, 1)).argmax())
        w = [t.clone() for t in inp["w"]]
        w[5][2 * H + 7, col] += 2.0 ** -5
        f = failures(measure(c, inp, k, reference(c, inp, k, w=w)))
        steps = {t for n, d, b, t in f if n == "gates" and d == 1 and b == 2}
        assert len(steps) > T // 2, f
        assert not any(d == 0 or (n == "gates" and b != 2) for n, d, b, _ in f), f
    elif fault == "length":
        ln = inp["lengths"].clone()
        b0 = int(((ln > 2) & (ln < T)).nonzero()[0])
        L0 = int(ln[b0])
        ln[b0] = L0 - 1
        f = failures(measure(c, inp, k, reference(c, inp, k, lengths=ln)))
        for d in (0, 1):
            assert any(n in ("out_past_len", "gates") and dd == d and t == L0 - 1 for n, dd, _, t in f), (d, f)
    elif fault == "d_h_n":
        dhn = inp["d_h_n"].clone()
        dhn[:, 128:256] = 0                                              # tile 1
        f = failures(measure(c, inp, k, reference(c, inp, k, d_h_n=dhn)))
        assert any(n == "dG_tf" and d == 0 and t == T - 1 for n, d, _, t in f), f
        assert any(n == "dG_tf" and d == 1 and t == 0 for n, d, _, t in f), f
        assert not any(n in ("gates", "blend") for n, *_ in f), f
    else:
        f = failures(measure(c, inp, k, reference(c, inp, k, rev_shift=True)))
        assert any(n == "gates" and d == 1 for n, d, _, _ in f), f
        assert not any(d == 0 for n, d, _, _ in f), f
