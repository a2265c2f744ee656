"""The bf16 GRU gradient and projection GEMMs called through the functions the autograd layers use, against the float64
reference of oracle/rec_bf16_ref.py (weight_grads, data_grad, projection, x_operand; self-checked against torch.nn.GRU by
test_rec_bf16_ref.py).

Entry points: rs_blk_wgrad (every dW_ih / dW_hh / bias gradient of a layer, with the production role tables of
functional_bf16.grads_from_dG_128 / grads_from_dG_256), rs_blk_gemm_nt_drop / rs_blk_gemm_nt (the data gradient dX and
the input projection P, functional_bf16.wide_projection at H = 256) and rs_pack_x_tm (the layer-0 input as the 16-column
second B source of the weight gradient).

A. Exact arithmetic, no tolerance.  dG in {-2 .. 2} (about half zeros), `out`, X and x in {-1, 0, 1}, weights a + b 2^-10
   (a in {+-1/2, +-1}, b in {-1, 0, 1}: bf16 hi = a and lo = b 2^-10 exact, still dyadic after the 1/2 of the r, z rows),
   biases multiples of 2^-4.  Every product and every partial sum is then an fp32 number (asserted per output element:
   sum |products| < 2^20 units of the product grid), so the kernels' fp32 sums are exact in any order, and the outputs
   equal the float64 reference bit for bit: independent of the split count, the atomic order, paired or unpaired mode
   (RS_WGRAD_PAIR = 0) and deterministic mode, which all three run.  The pad rows and pad traces of dG, `out` and X hold
   non-zero values: the reference reads them at the documented places, so a kernel that reads a wrong row, sums a pad row
   of dG or skips a row of a tile differs.  Every non-accumulating output is NaN-filled (deterministic mode fills
   torch.empty with NaN; the other modes must match it bit for bit), and dX and P are checked at all T + 2 rows.
B. Realistic operands: the recurrence kernels' own dG and `out` (test_rec_kernels_gpu.py's cases) through the same
   functions.  Weight-gradient errors are normalised entry by entry by sum |a||b| of that entry (the condition-free bound
   of an fp32 sum in any order) and reported per (direction, gate, 128-row block); dX is held elementwise to
   1/2 ulp_bf16 + c sum |dG||W|, its pad rows exactly 0.  In deterministic mode the gradients of GRULayerBF16Fn /
   GRULayerBF16WideFn equal these functions on the dG of a rerun of the BPTT, bit for bit.
C. Sensitivity: references built with one injected fault each must differ from the kernel outputs (A), and the first
   three must be located at their direction and gate block (B).

Bars of family B, each about 4x the largest value measured over B_CASES in three runs on a B200 (1000 W power limit);
the maxima were the same in all three runs:
    weight gradients, |err| / sum |a||b|     WG_BAR = 2e-6    measured 4.9e-7 (dW_ih, H = 256 P case; dW_hh 4.7e-7,
                                                              the bias sums 8.7e-8)
    dX, c in 1/2 ulp + c sum |dG||W|         DX_BAR = 2e-6    measured 4.4e-7 (H = 256 P and H = 128 P split cases)
"""
import contextlib
import ctypes
import os
import zlib

import pytest
import torch

from oracle import rec_bf16_ref as R
from roomslam_b200 import _lib
from roomslam_b200 import functional_bf16 as FB
from roomslam_b200 import layout as L
from test_rec_kernels_gpu import KEEP, Case, make_inputs, nan_like, run_kernels

pytestmark = pytest.mark.gpu

WG_BAR = 2e-6
DX_BAR = 2e-6
BF, F64 = torch.bfloat16, torch.float64
MODES = ("default", "deterministic", "unpaired")


def _st():
    return torch.cuda.current_stream().cuda_stream


@contextlib.contextmanager
def mode(name):
    """default | deterministic (torch.use_deterministic_algorithms, restored after) | unpaired (RS_WGRAD_PAIR=0)."""
    det, pair = torch.are_deterministic_algorithms_enabled(), os.environ.get("RS_WGRAD_PAIR")
    try:
        torch.use_deterministic_algorithms(name == "deterministic")
        if name == "unpaired":
            os.environ["RS_WGRAD_PAIR"] = "0"
        else:
            os.environ.pop("RS_WGRAD_PAIR", None)
        yield
    finally:
        torch.use_deterministic_algorithms(det)
        if pair is None:
            os.environ.pop("RS_WGRAD_PAIR", None)
        else:
            os.environ["RS_WGRAD_PAIR"] = pair


def n_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def last_block_of_split0(n_roles, tiles, T):
    """(tile, t) of the last block of split 0 by rs_blk_wgrad's split formula.  The host divides the SM count in default
    mode and kDetSplitSms = 148 in deterministic mode; the two agree on a B200 (148 SMs)."""
    total = tiles * T
    splits = min(max(n_sms() // n_roles, 1), total)
    bps = (total + splits - 1) // splits
    return (bps - 1) // T, (bps - 1) % T


def bf16_round(v):
    """float64 -> fp32 (round to nearest even) -> bf16, back in float64: the kernels' epilogue rounding."""
    return v.float().to(BF).to(F64)


def drop_cols(bits, scale):
    """Dropout bits [tiles][T][128][C / 8] -> the multiplier (tiles * 128, T, C) float64 (0 or scale)."""
    nt, T, _, cb = bits.shape
    b = (bits.to(torch.int32).unsqueeze(-1) >> torch.arange(8, device=bits.device, dtype=torch.int32)) & 1
    return b.reshape(nt, T, 128, cb * 8).permute(0, 2, 1, 3).reshape(nt * 128, T, cb * 8).to(F64) * scale.to(F64)


def rand_bits(tiles, T, C, g):
    keep = torch.rand(tiles, T, 128, C, generator=g) < KEEP
    bits = (keep.view(tiles, T, 128, C // 8, 8).to(torch.int32) << torch.arange(8, dtype=torch.int32)).sum(-1)
    return bits.to(torch.uint8).cuda(), torch.tensor([1.0 / KEEP], dtype=torch.float32).cuda()


# --------------------------------------------------------------------------------------------- the layers' functions
def pack_deeper_128(w, split):
    """rs_gru_pack_weights_bf16 for a deeper H = 128 layer with the projection GEMM -> (wt_proj, bias_x, wt_dgrad)."""
    H, Il = 128, 256
    wt = torch.empty(6, (Il // 64) * (1 + split), 8, 128, 8, device="cuda", dtype=BF)
    wt_dgrad = torch.empty(Il // 128, 12 * (1 + split), 8, 128, 8, device="cuda", dtype=BF)
    whh = torch.empty(2, 16 * (1 + split), 3 * H, 8, device="cuda", dtype=BF)
    whhT = torch.empty(2, 48 * (1 + split), H, 8, device="cuda", dtype=BF)
    bhn, bx = torch.empty(2, H, device="cuda"), torch.empty(2, 3 * H, device="cuda")
    arr = (ctypes.c_void_p * 8)(*[t.data_ptr() for t in w])
    _lib.call("rs_gru_pack_weights_bf16", ctypes.addressof(arr), H, Il, split, whh.data_ptr(), bhn.data_ptr(), bx.data_ptr(),
              wt.data_ptr(), whhT.data_ptr(), wt_dgrad.data_ptr(), 0, _st())
    return wt, bx, wt_dgrad


def run_grads(H, dG, out, saved_in, layer0, B, T, Il, split=0, w=None, in_drop=None, need_dx=False):
    """grads_from_dG_128 / _256 -> dict.  w: the 8 fp32 master weights (the dgrad image is built from them)."""
    if H == 128:
        wt_dgrad = pack_deeper_128(w, split)[2] if need_dx else None
        r = FB.grads_from_dG_128(dG, out, saved_in, not layer0, B, T, Il, split, wt_dgrad, in_drop, need_dx)
    else:
        w_ih_cat = torch.cat([w[0], w[4]], 0).float() if w is not None else None
        r = FB.grads_from_dG_256(dG, out, saved_in, not layer0, B, T, Il, w_ih_cat, in_drop, need_dx)
    torch.cuda.synchronize()
    return dict(zip(("w_ih", "w_hh", "b_ih", "b_hh", "dX"), r))


def ref_grads(H, dGf, outf, x_seq):
    """weight_grads in the kernels' output shapes: w_ih (6H, I), w_hh (2, 3H, H), b_ih / b_hh (2, 3H)."""
    gw = R.weight_grads(dGf[:, :, 1:-1], torch.stack([x_seq, x_seq], 0), R.h_prev_backward(outf))
    gw["w_ih"] = gw["w_ih"].flatten(0, 1)
    return gw


def w_ih_operand(w, split, H):
    """W_ih of both directions (2, 3H, I) as the dgrad image holds it: unscaled, bf16 or hi + lo."""
    return torch.stack([R.hi_lo(w[0].float(), split), R.hi_lo(w[4].float(), split)], 0)


# ----------------------------------------------------------------------------------------- A. exact-arithmetic family
def ints(shape, lo, hi, g, zero_frac=0.0):
    """Integers in [lo, hi] as fp32 on the GPU, about zero_frac of them (additionally) zero."""
    v = torch.randint(lo, hi + 1, shape, generator=g, device="cuda").float()
    if zero_frac:
        v *= torch.rand(shape, generator=g, device="cuda") >= zero_frac
    return v


def exact_weights(H, Il, g):
    """The 8 fp32 master weights: a + b 2^-10 (a in {+-1/2, +-1}, b in {-1, 0, 1}); biases k / 16, |k| <= 8."""
    def wt(*s):
        a = torch.tensor([-1.0, -0.5, 0.5, 1.0], device="cuda")[torch.randint(0, 4, s, generator=g, device="cuda")]
        return a + ints(s, -1, 1, g) * 2.0 ** -10

    def bias():
        return ints((3 * H,), -8, 8, g) / 16.0
    return [wt(3 * H, Il), wt(3 * H, H), bias(), bias(), wt(3 * H, Il), wt(3 * H, H), bias(), bias()]


def exact_operands(H, B, T, layer0, I, g):
    """dG and `out` (non-zero at pad rows and pad traces too), and x (layer 0) or the tile-major X."""
    Bp = L.n_tiles(B) * 128
    op = {"dG": R.to_tm(ints((Bp, T + 2, 8 * H), -2, 2, g, 0.5)), "out": R.to_tm(ints((Bp, T + 2, 2 * H), -1, 1, g))}
    if layer0:
        op["x"] = ints((B, T, I), -1, 1, g)
    else:
        op["X"] = R.to_tm(ints((Bp, T + 2, 2 * H), -1, 1, g))
    return op


def assert_exactly(got, want, name):
    got = got.to(F64)
    bad = got != want
    assert not bool(bad.any()), (name, int(bad.sum()), bad.nonzero()[:5].tolist())


def exact_sum_bound(S, unit, name):
    """sum |products| of every output element, in units of the product grid, below 2^20: every fp32 partial sum is exact."""
    assert float(S.max()) / unit < 2.0 ** 20, (name, float(S.max()) / unit)


A_WGRAD = [  # (H, B, T, layer0, I, split, in_drop)
    (128, 1, 1, True, 1, 0, False),          # 1 block: fewer blocks than splits
    (128, 2, 3, True, 2, 0, False),
    (128, 129, 37, True, 11, 0, False),      # 74 blocks over 18 splits of 5: the last split short
    (128, 4100, 142, True, 16, 0, False),    # 33 tiles (odd); rs_pack_x_tm wraps its grid stride (33 x 144 > 4736 blocks)
    (128, 1, 1, False, 0, 0, False),
    (128, 129, 37, False, 0, 1, True),       # 12 roles, paired (share mask 0b11011): 74 blocks over 11 splits of 7
    (128, 127, 3, False, 0, 0, True),
    (128, 4100, 100, False, 0, 1, False),
    (256, 1, 1, True, 2, 0, False),
    (256, 129, 37, True, 11, 0, False),
    (256, 1300, 40, True, 16, 0, False),     # 11 tiles: 440 blocks over 18 splits of 25
    (256, 2, 3, False, 0, 0, True),
    (256, 129, 37, False, 0, 0, False),      # 18 roles, paired: 74 blocks over 8 splits of 10
    (256, 1300, 40, False, 0, 0, True),      # Il = 512: 64 mask bytes per row
]


def a_id(c):
    H, B, T, layer0, I, split, drop = c
    return f"H{H}-B{B}-T{T}-" + (f"x{I}" if layer0 else "X") + f"-s{split}" + ("-drop" if drop else "")


def run_exact_case(c, modes=MODES):
    H, B, T, layer0, I, split, drop = c
    g = torch.Generator(device="cuda").manual_seed(zlib.crc32(a_id(c).encode()))
    Il = I if layer0 else 2 * H
    tiles = L.n_tiles(B)
    op = exact_operands(H, B, T, layer0, I, g)
    w = exact_weights(H, Il, g)
    in_drop = rand_bits(tiles, T, Il, torch.Generator().manual_seed(T)) if drop else None
    saved_in = op["x"] if layer0 else op["X"]
    res = {}
    for m in modes:
        with mode(m):
            res[m] = run_grads(H, op["dG"], op["out"], saved_in, layer0, B, T, Il, split, w, in_drop, need_dx=not layer0)
            if not layer0:
                res[m]["P"] = project(H, op["X"], w, split, B, T)
    return op, w, in_drop, res


def project(H, X, w, split, B, T):
    """The production projection: rs_blk_gemm_nt with GRULayerBF16Fn's arguments (H = 128, split weights) or
    wide_projection (H = 256).  None where the layer has no projection GEMM (H = 128 without split: fused)."""
    if H == 256:
        _, _, bias_x, w_ih_fwd, _, _ = FB.wide_fwd_image(*w, False)
        P = FB.wide_projection(X, w_ih_fwd, bias_x, B, T)
        torch.cuda.synchronize()
        return P
    if not split:
        return None
    Il, tiles = 2 * H, L.n_tiles(B)
    wt, bx, _ = pack_deeper_128(w, 1)
    P = nan_like((tiles, T + 2, 6 * H // 8, 128, 8), BF)
    FB._nt(X, Il, [8 * k for k in range(Il // 64)] * 2, wt, 6, P, 6 * H, 0, bx.reshape(-1).contiguous(), tiles * (T + 2), _st())
    torch.cuda.synchronize()
    return P


def proj_operand(H, w, split):
    """The projection's W_ih (2, 3H, I) (r, z rows halved; hi + lo at H = 128 split, bf16 at H = 256) and fp32 bias_x."""
    s = R.gate_scale(H, "cuda")
    wih = torch.stack([R.hi_lo(w[4 * d].float() * s[:, None], split) for d in (0, 1)], 0)
    bias = torch.stack([R.bias_x(w[4 * d + 2], w[4 * d + 3], H) for d in (0, 1)], 0).to(F64)
    return wih, bias


def check_exact(c, op, w, in_drop, res):
    """Every output of every mode in res against the float64 reference, bit for bit."""
    H, B, T, layer0, I, split, drop = c
    dGf, outf = R.dG_full(op["dG"], H), R.out_full(op["out"], H)
    Bp = dGf.shape[1]
    x_seq = R.x_operand(op["x"], Bp, T)[:, 1:-1] if layer0 else R.tm_full(op["X"])[:, 1:-1]
    ref = ref_grads(H, dGf, outf, x_seq)
    absr = ref_grads(H, dGf.abs(), outf.abs(), x_seq.abs())
    for n in ("w_ih", "w_hh", "b_ih", "b_hh"):
        exact_sum_bound(absr[n], 1.0, n)
    out = {}
    if not layer0:
        wop = w_ih_operand(w, split if H == 128 else 0, H)
        mult = drop_cols(*in_drop) if in_drop is not None else None
        out["dX"] = bf16_round(R.data_grad(dGf, wop, mult))
        exact_sum_bound(R.data_grad(dGf.abs(), wop.abs(), None), 2.0 ** -10 if split else 0.5, "dX")
        if res["default"].get("P") is not None:
            wih, bias = proj_operand(H, w, split)
            Xf = R.tm_full(op["X"])
            out["P"] = bf16_round(R.projection(Xf, wih, bias))
            exact_sum_bound(R.projection(Xf.abs(), wih.abs(), bias.abs()), 2.0 ** -11, "P")
    for m, k in res.items():
        for n in ("w_ih", "w_hh", "b_ih", "b_hh"):
            assert_exactly(k[n], ref[n], (m, n))
        for n, want in out.items():
            assert_exactly(R.tm_full(k[n]), want, (m, n))
    return ref, out


@pytest.mark.parametrize("c", A_WGRAD, ids=a_id)
def test_exact_gradients_in_every_mode(c):
    op, w, in_drop, res = run_exact_case(c)
    check_exact(c, op, w, in_drop, res)
    H, B, T, layer0, I, split, drop = c
    if layer0:                          # rs_pack_x_tm bit for bit; the dW_ih columns >= I of the 16-column buffer are 0
        tiles = L.n_tiles(B)
        xa = nan_like((tiles, T + 2, 2, 128, 8), BF)
        _lib.call("rs_pack_x_tm", op["x"].data_ptr(), B, T, I, xa.data_ptr(), _st())
        torch.cuda.synchronize()
        assert_exactly(R.tm_full(xa), R.x_operand(op["x"], tiles * 128, T), "x_operand")
        for m in MODES:
            assert res[m]["w_ih"].shape == (6 * H, 16)
            assert_exactly(res[m]["w_ih"][:, I:], torch.zeros(6 * H, 16 - I, dtype=F64, device="cuda"), (m, "w_ih cols >= I"))


# ------------------------------------------------------------------------------------------------- C, on family A
SENS_A = [(128, 129, 37, True, 11, 0, False), (128, 129, 37, False, 0, 1, True), (256, 129, 37, False, 0, 0, True)]


@pytest.mark.parametrize("c", SENS_A, ids=a_id)
def test_exact_checks_see_injected_faults(c):
    """Each fault in the reference must change what the exact comparison sees.  The kernels run once, in default mode (the
    modes are compared by test_exact_gradients_in_every_mode); the unfaulted reference must match them first."""
    H, B, T, layer0, I, split, drop = c
    op, w, in_drop, res = run_exact_case(c, ("default",))
    k = res["default"]
    check_exact(c, op, w, in_drop, res)
    dGf, outf = R.dG_full(op["dG"], H), R.out_full(op["out"], H)
    Bp = dGf.shape[1]
    x_seq = R.x_operand(op["x"], Bp, T)[:, 1:-1] if layer0 else R.tm_full(op["X"])[:, 1:-1]

    def differs(ref):
        return any(not torch.equal(k[n].to(F64), ref[n]) for n in ("w_ih", "w_hh", "b_ih", "b_hh"))
    n_roles = 8 if layer0 else (12 if H == 128 else 18)            # roles of one launch (H = 256: one per direction)
    tile, t = last_block_of_split0(n_roles, L.n_tiles(B), T)
    faults = {}
    d0 = dGf.clone()
    # one block dropped: the one a split loop one block short would skip.  On exact operands losing any block shows, so
    # this checks that the comparison sees one block out of all of them, not which block the split formula picks.
    d0[:, tile * 128:(tile + 1) * 128, 1 + t] = 0
    faults["block"] = ref_grads(H, d0, outf, x_seq)
    o1 = outf.clone()
    o1[1, :, 2:] = outf[1, :, :-2]                                      # reverse direction reads t' - 1
    faults["rev_shift"] = ref_grads(H, dGf, o1, x_seq)
    faults["rz_swap"] = ref_grads(H, dGf[:, :, :, [1, 0, 2, 3]], outf, x_seq)
    if layer0:
        faults["x_cols"] = ref_grads(H, dGf, outf, x_seq[..., [1, 0] + list(range(2, 16))])
    for name, ref in faults.items():
        assert differs(ref), name
    if not layer0:
        wop = w_ih_operand(w, split if H == 128 else 0, H)
        mult = drop_cols(*in_drop)
        dx = R.tm_full(k["dX"])
        # one mask byte ignored: the 8 columns of the first byte with a cleared bit where the masked-off sum is not 0
        full = R.data_grad(dGf, wop, None)[:, 1:-1]
        cand = ((mult == 0) & (full != 0)).nonzero()
        b, tt, col = cand[0].tolist()
        m1 = mult.clone()
        m1[b, tt, col // 8 * 8: col // 8 * 8 + 8] = mult.max()
        assert not torch.equal(dx, bf16_round(R.data_grad(dGf, wop, m1))), "mask_byte"
        if split:                                                       # the lo half of the split weights dropped
            hi = w_ih_operand(w, 0, H)
            assert not torch.equal(dx, bf16_round(R.data_grad(dGf, hi, mult))), "lo_dgrad"
            wih, bias = proj_operand(H, w, split)
            whi, _ = proj_operand(H, w, 0)
            Xf = R.tm_full(op["X"])
            assert not torch.equal(R.tm_full(k["P"]), bf16_round(R.projection(Xf, whi, bias))), "lo_projection"


# --------------------------------------------------------------------------------------------- B. realistic family
B_CASES = [
    Case(128, 300, 37, "x", I=16, split=1, lengths="rand", drop=True, nt="3"),
    Case(128, 129, 37, "x", I=4, lengths="rand", drop=True),
    Case(128, 127, 37, "P", split=1, d_h_n=False),
    Case(128, 129, 37, "X", lengths="rand", drop=True),
    Case(128, 4987, 37, "x", I=11, lengths="rand", drop=True),                # 39 tiles
    Case(256, 129, 37, "x", I=11, lengths="rand", drop=True),
    Case(256, 127, 37, "P", lengths="full", drop=True, d_out=False),
]


def realistic(c: Case):
    """The recurrence kernels' own dG and `out` for case c, the layer input, and the gradient functions' outputs."""
    inp = make_inputs(c)
    with pytest.MonkeyPatch.context() as mp:
        if c.nt:
            mp.setenv("RS_REC_MODE", c.nt)
        k = run_kernels(c, inp)
    H, B, T = c.H, c.B, c.T
    tiles = L.n_tiles(B)
    layer0 = c.mode == "x"
    Il = c.I if layer0 else 2 * H
    g = torch.Generator().manual_seed(77 + c.seed)
    if layer0:
        saved_in = inp["x"]
    elif c.mode == "X":
        saved_in = inp["X"]
    else:                               # the P cases were given their projection: a layer input for the weight gradient
        X = torch.zeros(tiles * 128, T + 2, Il)
        X[:B, 1:-1] = torch.rand(B, T, Il, generator=g) * 2 - 1
        saved_in = R.to_tm(X.cuda())
    in_drop = rand_bits(tiles, T, Il, g) if not layer0 else None
    got = run_grads(H, k["dG"], k["out"], saved_in, layer0, B, T, Il, c.split, inp["w"], in_drop, need_dx=not layer0)
    return {"inp": inp, "k": k, "saved_in": saved_in, "in_drop": in_drop, "got": got}


def wgrad_errors(c: Case, r, dGf=None, outf=None, x_seq=None):
    """Per output, |err| / sum |a||b| entry by entry, max per (direction, gate, 128-row block): name -> (2, 3, H / 128).
    Keyword operands replace the decoded kernel operands (sensitivity test)."""
    H, T = c.H, c.T
    k = r["k"]
    dGf = R.dG_full(k["dG"], H) if dGf is None else dGf
    outf = R.out_full(k["out"], H) if outf is None else outf
    Bp = dGf.shape[1]
    if x_seq is None:
        # layer 0: the B2 operand is bf16(x), not hi + lo
        x_seq = R.x_operand(r["inp"]["x"], Bp, T)[:, 1:-1] if c.mode == "x" else R.tm_full(r["saved_in"])[:, 1:-1]
    ref = ref_grads(H, dGf, outf, x_seq)
    S = ref_grads(H, dGf.abs(), outf.abs(), x_seq.abs())
    errs = {}
    for n in ("w_ih", "w_hh", "b_ih", "b_hh"):
        e = (r["got"][n].to(F64) - ref[n]).abs() / S[n].clamp_min(1e-300)
        e = e.reshape(2, 3, H // 128, 128, -1)
        errs[n] = e.amax(dim=(3, 4))
    return errs


def flagged(errs):
    return sorted({(n, d, gi, mb) for n, e in errs.items() for d, gi, mb in (e > WG_BAR).nonzero().tolist()})


def dx_error(c: Case, r):
    """The smallest c with |dX - ref| <= 1/2 ulp_bf16 + c sum |dG||W| at every element; the pad rows must be exactly 0."""
    H = c.H
    dGf = R.dG_full(r["k"]["dG"], H)
    wop = w_ih_operand(r["inp"]["w"], c.split if H == 128 else 0, H)
    mult = drop_cols(*r["in_drop"])
    ref = R.data_grad(dGf, wop, mult)
    S = R.data_grad(dGf.abs(), wop.abs(), mult)
    dx = R.tm_full(r["got"]["dX"])
    assert bool(torch.isfinite(dx).all())
    assert not bool((dx[:, [0, -1]] != 0).any()), "dX pad rows"
    half_ulp = 0.5 * torch.maximum(bf16_ulp(ref), bf16_ulp(dx))
    excess = ((dx - ref).abs() - half_ulp).clamp_min(0)
    return float((excess / S.clamp_min(1e-300)).max())


def bf16_ulp(v):
    """The spacing of bf16 numbers at |v| (0 at v = 0)."""
    return torch.where(v != 0, 2.0 ** (torch.floor(torch.log2(v.abs().clamp_min(1e-30))) - 7), torch.zeros_like(v))


@pytest.mark.parametrize("c", B_CASES, ids=str)
def test_realistic_gradients(c):
    r = realistic(c)
    errs = wgrad_errors(c, r)
    meas = {n: float(e.max()) for n, e in errs.items()}
    if c.mode != "x":
        meas["dX_c"] = dx_error(c, r)
    print(f"measured {c}: " + " ".join(f"{n}={v:.3e}" for n, v in meas.items()))
    assert flagged(errs) == [], meas
    assert meas.get("dX_c", 0.0) <= DX_BAR, meas


def test_realistic_checks_locate_injected_faults():
    """At few blocks (B = 129, T = 37): one dropped block, the reverse direction's hidden-side shift flipped and the r, z
    role outputs swapped must each be flagged at their direction and gate block."""
    c = Case(128, 129, 37, "x", I=4, lengths="rand", drop=True)
    r = realistic(c)
    assert flagged(wgrad_errors(c, r)) == []
    H, T = c.H, c.T
    dGf, outf = R.dG_full(r["k"]["dG"], H), R.out_full(r["k"]["out"], H)
    tile, t = last_block_of_split0(8, L.n_tiles(c.B), T)
    d0 = dGf.clone()
    d0[:, tile * 128:(tile + 1) * 128, 1 + t] = 0
    f = flagged(wgrad_errors(c, r, dGf=d0))
    assert all(("w_hh", d, gi, 0) in f for d in (0, 1) for gi in (0, 1, 2)), f
    o1 = outf.clone()
    o1[1, :, 2:] = outf[1, :, :-2]
    f = flagged(wgrad_errors(c, r, outf=o1))
    assert all(("w_hh", 1, gi, 0) in f for gi in (0, 1, 2)) and not any(d == 0 or n != "w_hh" for n, d, _, _ in f), f
    f = flagged(wgrad_errors(c, r, dGf=dGf[:, :, :, [1, 0, 2, 3]]))
    assert all((n, d, gi, 0) in f for n in ("w_ih", "w_hh", "b_ih", "b_hh") for d in (0, 1) for gi in (0, 1)), f
    assert not any(gi == 2 for _, _, gi, _ in f), f


# ------------------------------------------------------------------------------- the autograd layers use these functions
@pytest.mark.parametrize("H,layer0,split", [(128, True, 0), (128, False, 1), (256, True, 0), (256, False, 0)])
def test_autograd_layers_equal_the_tested_functions(H, layer0, split):
    """Deterministic mode: GRULayerBF16Fn / GRULayerBF16WideFn backward gives, bit for bit, grads_from_dG_* of the dG that
    the BPTT kernel computes again from the tensors the forward saved."""
    B, T = 129, 7
    c = Case(H, B, T, "x" if layer0 else "X", I=11, split=split)
    inp = make_inputs(c)
    tiles = L.n_tiles(B)
    Il = 11 if layer0 else 2 * H
    g = torch.Generator().manual_seed(3)
    in_drop = None if layer0 else rand_bits(tiles, T, Il, g)
    ws = [t.clone().requires_grad_() for t in inp["w"]]
    xin = (inp["x"] if layer0 else inp["X"]).clone().requires_grad_(not layer0)
    fn = FB.GRULayerBF16Fn if H == 128 else FB.GRULayerBF16WideFn
    d_out = inp["d_out"]
    with mode("deterministic"):
        y, h_n = fn.apply(xin, (not layer0, B, T, None, None, split, in_drop), None, *ws)
        saved = y.grad_fn.saved_tensors
        dG = nan_like((tiles, T + 2, H, 128, 8), BF)
        if H == 128:
            out, gates, saved_in, whhT, wt_dgrad, whh, b_hn = saved
            _lib.call("rs_rec_bwd_bf16", d_out.data_ptr(), inp["d_h_n"].data_ptr(), gates.data_ptr(), out.data_ptr(),
                      whhT.data_ptr(), whh.data_ptr(), whh.shape[1], b_hn.data_ptr(), dG.data_ptr(), 0, 0, 0, split, B, T, _st())
            want = FB.grads_from_dG_128(dG, out, saved_in, not layer0, B, T, Il, split, wt_dgrad, in_drop, not layer0)
        else:
            out, gates, saved_in, w_ih_cat, w_hh_cat = saved
            wtst = FB.wide_bwd_image(w_hh_cat)
            _lib.call("rs_rec_bwd_bf16_wide", d_out.data_ptr(), inp["d_h_n"].data_ptr(), gates.data_ptr(), out.data_ptr(),
                      wtst.data_ptr(), dG.data_ptr(), 0, 0, 0, B, T, _st())
            want = FB.grads_from_dG_256(dG, out, saved_in, not layer0, B, T, Il, w_ih_cat, in_drop, not layer0)
        grads = torch.autograd.grad((y, h_n), ws + ([xin] if not layer0 else []), (d_out, inp["d_h_n"]))
    torch.cuda.synchronize()
    dW_ih, dW_hh, db_ih, db_hh, dX = want
    dW_ih = dW_ih[:, :Il]
    exp = [dW_ih[:3 * H], dW_hh[0], db_ih[0], db_hh[0], dW_ih[3 * H:], dW_hh[1], db_ih[1], db_hh[1]] + ([dX] if not layer0 else [])
    bits = lambda t: t.contiguous().view(torch.int16 if t.dtype == BF else torch.int32)  # noqa: E731
    assert len(grads) == len(exp)
    for i, (a, b) in enumerate(zip(grads, exp)):
        assert a.shape == b.shape and a.dtype == b.dtype, i
        assert torch.equal(bits(a), bits(b)), i
