"""The decoder, the multi-task loss and the AdamW step, each kernel stage against the float64 reference of
oracle/decoder_ref.py (self-checked against float64 autograd and torch.optim.AdamW by test_decoder_ref.py).

Entry points: rs_gemm_bf16_nt (every flag combination), rs_gemm_bf16_tn_acc / _seg_acc, rs_sgemm (the three layouts of
functional.py), rs_colsum_f32, rs_heads_split_f32, rs_heads_merge_bwd_f32, rs_relu_bwd_*, rs_loss_fwd_f32,
rs_loss_bwd_f32, rs_adamw_step_f32, and both decoders through the functions their autograd classes call
(functional.decoder_fwd / decoder_bwd, functional_bf16.decoder_bf16_fwd / decoder_bf16_bwd).  Every case runs in the
default and the deterministic mode (torch.use_deterministic_algorithms).

A. Exact arithmetic, no tolerance.  Operands are small integers, mostly zero, biases multiples of 1/2; every product
   and partial sum is then an fp32 number and every stored output is representable in its type (asserted on the
   reference), so the kernels' sums are exact in any order and every output equals the reference bit for bit.  Outputs
   are NaN-filled before each call and sit inside canary rows and columns (ldc > N, extra rows) that must survive;
   the padding columns of the operands (lda > K) hold NaN, so reading them shows.
B. Realistic operands: model-initialised weights and the kernels' own intermediates (teacher forcing).  The error of
   every output of a stage, less 1/2 ulp of the output type, is normalised by sum |a||b| (+ |bias|) of that output and
   reported per stage and head block.  The copy stages (heads_split copies, relu_bwd, the dWh head-row slices) are
   bit-exact.
C. The heads and loss kernels directly, at their edges; AdamW against the reference per element relative to the update.
D. Sensitivity: references with one injected fault each must be told apart from the kernel outputs, and in family B
   located at their stage and head block.

Bars of family B, each about 4x the largest value measured over REAL_CASES on a B200 (1000 W power limit):
    forward stages (f1, f2 in bf16, rawp in fp32)          FWD_BAR = 1e-6   measured 2.7e-7 (rawp, class block)
    backward GEMM stages (dWh, df2, dW2, df1, dW1, dlat)   BWD_BAR = 4e-6   measured 9.5e-7 (dWh, size block; dW2 9.1e-7)
Softplus (log1pf(expf) + 1e-4) and the size gradient d_size * sigmoid are held to SP_ULPS = 4 float32 ulps of float64;
measured 3.07 and 2.14.
"""
import contextlib
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import decoder_ref as D
from roomslam_b200 import _lib
from roomslam_b200 import functional as F_
from roomslam_b200 import functional_bf16 as FB

pytestmark = pytest.mark.gpu

FWD_BAR = 1e-6
BWD_BAR = 4e-6
SP_ULPS = 4
BF, F32, F64 = torch.bfloat16, torch.float32, torch.float64
MODES = ("default", "deterministic")
ORDER = ((5, 0), (0, 5), (2, 2), (2, 5), (5, 2), (5, 5))     # functional.tn_tc: (A sixth, B sixth) of each bf16x6 pass


def _st():
    return torch.cuda.current_stream().cuda_stream


@contextlib.contextmanager
def mode(name):
    det = torch.are_deterministic_algorithms_enabled()
    try:
        torch.use_deterministic_algorithms(name == "deterministic")
        yield
    finally:
        torch.use_deterministic_algorithms(det)


def gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def sparse_int(shape, g, lo, hi, density):
    """Integers in [lo, hi] on a random `density` share of the entries, zero elsewhere (float64, on the GPU)."""
    v = torch.randint(lo, hi + 1, shape, generator=g, device="cuda").to(F64)
    return v * (torch.rand(shape, generator=g, device="cuda") < density)


def representable(ref, dtype):
    return bool(torch.equal(ref.to(dtype).to(F64), ref))


def framed(rows, cols, dtype, extra_rows=3, extra_cols=24, fill=float("nan"), canary=-77.0):
    """A [rows + extra_rows, cols + extra_cols] buffer: the view [:rows, :cols] filled with `fill`, the rest `canary`."""
    buf = torch.full((rows + extra_rows, cols + extra_cols), canary, dtype=dtype, device="cuda")
    view = buf[:rows, :cols]
    view.fill_(fill)
    return buf, view


def canary_intact(buf, rows, cols, canary=-77.0):
    mask = torch.ones(buf.shape, dtype=torch.bool, device="cuda")
    mask[:rows, :cols] = False
    return bool((buf[mask].to(F64) == canary).all())


def operand(x, dtype, pad):
    """x [rows, K] stored with leading dimension K + pad; the pad columns hold NaN."""
    buf = torch.full((x.shape[0], x.shape[1] + pad), float("nan"), dtype=dtype, device="cuda")
    buf[:, :x.shape[1]] = x.to(dtype)
    return buf[:, :x.shape[1]]


# =========================================== A. exact family ===========================================================
NT_SHAPES = [(1, 128, 64), (127, 256, 256), (129, 512, 512), (8192, 128, 64), (8192, 256, 256), (300, 128, 512),
             (16384, 512, 64)]       # the last: 512 tiles > 3 x 148 SMs, every CTA cycles through both TMEM stages


def _nt_call(A, Bw, C, bias, flags):
    M, K = A.shape
    _lib.call("rs_gemm_bf16_nt", A.data_ptr(), A.stride(0), Bw.data_ptr(), Bw.stride(0), C.data_ptr(), C.stride(0),
              0 if bias is None else bias.data_ptr(), M, Bw.shape[0], K, flags, _st())


@pytest.mark.parametrize("m", MODES)
@pytest.mark.parametrize("flags", [0, FB.RELU, FB.OUT_F32, FB.RELU | FB.OUT_F32])
@pytest.mark.parametrize("with_bias", [False, True])
def test_gemm_bf16_nt_exact(m, flags, with_bias):
    g = gen(1 + flags)
    for M, N, K in NT_SHAPES:
        a = sparse_int((M, K), g, -1, 1, 6.0 / K)
        b = sparse_int((N, K), g, -2, 2, 0.5)
        bias = (torch.randint(-8, 9, (N,), generator=g, device="cuda") * 0.5).to(F64) if with_bias else None
        ref = a @ b.t() + (bias if bias is not None else 0)
        if flags & FB.RELU:
            ref = ref.clamp_min(0)
        out_t = F32 if flags & FB.OUT_F32 else BF
        assert representable(ref, out_t)
        A, Bw = operand(a, BF, 64), operand(b, BF, 8)
        buf, C = framed(M, N, out_t)
        bias_t = None if bias is None else bias.float()
        with mode(m):
            _nt_call(A, Bw, C, bias_t, flags)
        torch.cuda.synchronize()
        assert torch.equal(C.to(F64), ref), (M, N, K)
        assert canary_intact(buf, M, N), (M, N, K)


TN_ROWS = [1, 63, 64, 65, 300, 8192, 70000]


def _tn_ref(a, a_col0, a_shift, b, b_col0, b_shift, rows, segs, M, N):
    out = torch.zeros(M, N, dtype=F64, device="cuda")
    ar = torch.zeros(rows, a.shape[1], dtype=F64, device="cuda")
    br = torch.zeros(rows, b.shape[1], dtype=F64, device="cuda")
    na, nb = max(0, min(rows, a.shape[0] - a_shift)), max(0, min(rows, b.shape[0] - b_shift))
    ar[:na], br[:nb] = a[a_shift:a_shift + na], b[b_shift:b_shift + nb]
    for sa, sb in segs:
        out += ar[:, a_col0 + sa:a_col0 + sa + M].t() @ br[:, b_col0 + sb:b_col0 + sb + N]
    return out


@pytest.mark.parametrize("m", MODES)
def test_gemm_bf16_tn_acc_exact(m):
    """C += A^T B onto a non-zero C: row shifts on either operand, column offsets, 1 to 6 passes in the bf16x6 order
    (rs_gemm_bf16_tn_seg_acc; the first pass alone also through rs_gemm_bf16_tn_acc), a short operand whose missing rows
    read as zero, and (70000 rows, 6 passes at one output tile) a last split whose tail is fed zeros."""
    g = gen(7)
    kp = 128
    for i, rows in enumerate(TN_ROWS):
        M, N = (128, 128) if rows > 8192 else ((256, 128) if i % 2 else (128, 256))
        n_seg = 1 + i % 6 if rows <= 8192 else 6
        a_shift, b_shift = (i % 3 == 1), (i % 3 == 2)
        a_col0, b_col0 = 64 * (i % 2), 128 * (i % 3 == 0)
        a_rows = rows + a_shift - (rows > 64)            # A one row short of the last pair where rows > 64
        a = sparse_int((max(a_rows, 1), a_col0 + 6 * kp + M), g, -1, 1, 0.3)
        b = sparse_int((rows + b_shift, b_col0 + 6 * kp + N), g, -2, 2, 0.5)
        segs = [(ta * kp, tb * kp) for ta, tb in ORDER[:n_seg]]
        c0 = sparse_int((M, N), g, -50, 50, 0.8)
        ref = c0 + _tn_ref(a, a_col0, a_shift, b, b_col0, b_shift, rows, segs, M, N)
        assert ref.abs().max() < 2 ** 24
        A, Bm = operand(a, BF, 8), operand(b, BF, 16)
        ref1 = c0 + _tn_ref(a, a_col0, a_shift, b, b_col0, b_shift, rows, segs[:1], M, N)
        for seg_api, want in ((True, ref), (False, ref1)):
            buf, C = framed(M, N, F32, fill=0.0)
            C.copy_(c0)
            a_seg = (ctypes.c_int * 6)(*[s for s, _ in segs] + [0] * (6 - n_seg))
            b_seg = (ctypes.c_int * 6)(*[s for _, s in segs] + [0] * (6 - n_seg))
            with mode(m):
                if seg_api:
                    _lib.call("rs_gemm_bf16_tn_seg_acc", A.data_ptr(), A.stride(0), A.shape[0], a_col0, int(a_shift), Bm.data_ptr(),
                              Bm.stride(0), Bm.shape[0], b_col0, int(b_shift), n_seg, ctypes.addressof(a_seg), ctypes.addressof(b_seg),
                              C.data_ptr(), C.stride(0), M, N, rows, _st())
                else:
                    _lib.call("rs_gemm_bf16_tn_acc", A.data_ptr(), A.stride(0), A.shape[0], a_col0 + segs[0][0], int(a_shift),
                              Bm.data_ptr(), Bm.stride(0), Bm.shape[0], b_col0 + segs[0][1], int(b_shift), C.data_ptr(), C.stride(0),
                              M, N, rows, _st())
            torch.cuda.synchronize()
            assert torch.equal(C.to(F64), want), (rows, n_seg, seg_api)
            assert canary_intact(buf, M, N), rows


SGEMM_CASES = [  # layout, M, N, K, flags, bias
    ("linear_nt", 300, 130, 100, F_.RELU, True), ("linear_nt", 1, 64, 17, 0, True), ("linear_nt", 257, 70, 4100, 0, True),
    ("matmul_nn", 129, 200, 77, 0, False), ("matmul_nn", 64, 64, 5000, F_.ACC, False), ("matmul_nn", 65, 33, 1, F_.RELU | F_.ACC, False),
    ("matmul_tn", 130, 100, 20001, 0, False), ("matmul_tn", 128, 256, 8192, F_.ACC, False), ("matmul_tn", 40, 50, 333, F_.ACC, False),
]


@pytest.mark.parametrize("m", MODES)
def test_sgemm_exact(m):
    """rs_sgemm in the three layouts of functional.py with bias, RELU and ACCUMULATE; split-K (K >= 4096 with fewer
    than 296 tiles, K not a multiple of 16 or of the split); ldc > N with canaries."""
    g = gen(11)
    for layout, M, N, K, flags, with_bias in SGEMM_CASES:
        x = sparse_int((M, K), g, -2, 2, min(1.0, 40.0 / K))
        w = sparse_int((N, K), g, -2, 2, 0.5)
        bias = (torch.randint(-8, 9, (N,), generator=g, device="cuda") * 0.5).to(F64) if with_bias else None
        c0 = sparse_int((M, N), g, -9, 9, 0.7)
        ref = x @ w.t() + (bias if bias is not None else 0) + (c0 if flags & F_.ACC else 0)
        if flags & F_.RELU:
            ref = ref.clamp_min(0)
        buf, C = framed(M, N, F32)
        if flags & F_.ACC:
            C.copy_(c0)
        bias_t = None if bias is None else bias.float()
        with mode(m):
            if layout == "linear_nt":
                F_.linear_nt(operand(x, F32, 4), operand(w, F32, 3), bias_t, C, flags)
            elif layout == "matmul_nn":
                F_.matmul_nn(operand(x, F32, 5), operand(w.t().contiguous(), F32, 2), C, flags)
            else:
                F_.matmul_tn(operand(x.t().contiguous(), F32, 7), operand(w.t().contiguous(), F32, 1), C, flags)
        torch.cuda.synchronize()
        assert torch.equal(C.to(F64), ref), (layout, M, N, K, flags)
        assert canary_intact(buf, M, N), (layout, M, N, K)


@pytest.mark.parametrize("m", MODES)
def test_colsum_exact(m):
    g = gen(13)
    for M, N in ((1, 5), (2048, 130), (2049, 33), (300000, 70)):       # one slab; many slabs (up to the cap of 128)
        a = sparse_int((M, N), g, -3, 3, 0.5)
        for acc in (False, True):
            o0 = sparse_int((N,), g, -9, 9, 1.0)
            ref = a.sum(0) + (o0 if acc else 0)
            out = torch.full((N + 4,), -77.0, device="cuda")
            out[:N] = o0 if acc else float("nan")
            A = operand(a, F32, 3)
            with mode(m):
                _lib.call("rs_colsum_f32", A.data_ptr(), A.stride(0), M, N, out.data_ptr(), int(acc), _st())
            torch.cuda.synchronize()
            assert torch.equal(out[:N].to(F64), ref) and bool((out[N:] == -77.0).all()), (M, N, acc)


def _head_params(g, N, C, D, scale_fn):
    heads = []
    for rows in (N * C, 2 * N, 2 * N, N, N):
        heads += [scale_fn((rows, D)), scale_fn((rows,))]
    return heads


@pytest.mark.parametrize("m", MODES)
@pytest.mark.parametrize("bf16", [True, False])
def test_decoder_exact(m, bf16):
    """Both decoders end to end through the seam on exact operands: every intermediate and gradient bit for bit."""
    g = gen(17)
    B, DL, D1, D2, N, C = (300, 256, 256, 128, 13, 4)          # NH = 130: two head tiles in bf16
    lat = sparse_int((B, DL), g, -1, 1, 0.03)
    W1, W2 = sparse_int((D1, DL), g, -1, 1, 0.05), sparse_int((D2, D1), g, -1, 1, 0.05)
    b1 = torch.randint(-2, 3, (D1,), generator=g, device="cuda").to(F64) * 0.5
    b2 = torch.randint(-2, 3, (D2,), generator=g, device="cuda").to(F64) * 0.5
    heads = _head_params(g, N, C, D2, lambda s: sparse_int(s, g, -1, 1, 0.05))
    d_pred = [sparse_int(s, g, -2, 2, 0.05) for s in ((B, N, C), (B, N, 2), (B, N, 2), (B, N), (B, N))]
    d_pred[2] = None                                           # the size block multiplies by a sigmoid: not exact
    with mode(m):
        args = [t.float() for t in (lat, W1, b1, W2, b2)]
        hs = [t.float() for t in heads]
        r = (FB.decoder_bf16_fwd if bf16 else F_.decoder_fwd)(args[0], N, C, *args[1:], hs)
        d_raw = F_.heads_merge(r["raw"], N, C, *[None if d is None else d.float() for d in d_pred])
        if bf16:
            gr = FB.decoder_bf16_bwd(r["lat"], r["W1b"], r["W2b"], r["Wh"], r["f1"], r["f2"], d_raw)
        else:
            gr = F_.decoder_bwd(r["latent"], W1.float(), W2.float(), r["Wh"], r["f1"], r["f2"], d_raw)
    torch.cuda.synchronize()
    Wh, bh = D.pad_heads(heads) if bf16 else D.pad_heads(heads, N * (C + 6))
    f = D.decoder_fwd(lat, W1, b1, W2, b2, Wh, bh)
    act_t = BF if bf16 else F32
    for name in ("f1", "f2"):
        assert representable(f[name], act_t) and torch.equal(r[name].to(F64), f[name]), name
    raw = f["rawp"][:, :N * (C + 6)]
    assert torch.equal(r["raw"].to(F64), raw)
    if bf16:
        assert torch.equal(r["rawp"].to(F64), f["rawp"])
    d_raw_ref = D.heads_merge(raw, N, C, *d_pred)
    assert torch.equal(d_raw.to(F64), d_raw_ref)
    d_rawp = torch.cat([d_raw_ref, d_raw_ref.new_zeros(B, Wh.shape[0] - d_raw_ref.shape[1])], 1)
    b = D.decoder_bwd(lat, W1, W2, Wh, f["f1"], f["f2"], d_rawp, d_raw_ref)
    assert representable(b["df2"], act_t) and representable(b["df1"], act_t)
    for name in ("dWh", "dbh", "df2", "dW2", "db2", "df1", "dW1", "db1", "dlat"):
        assert torch.equal(gr[name].to(F64), b[name]), name
    if bf16:
        assert torch.equal(gr["d_rawp"].to(F64), d_rawp)


# =========================================== B. realistic family =======================================================
def ulp_half(ref, dtype):
    """An upper bound of 1/2 ulp of `ref` in the output type."""
    return ref.abs() * (2.0 ** -8 if dtype == BF else 2.0 ** -24)


def stage_err(got, ref, scale, dtype, col_blocks=None, row_blocks=None):
    """max over the outputs of (|got - ref| - 1/2 ulp) / scale, overall or per named column / row block."""
    e = ((got.to(F64) - ref).abs() - ulp_half(ref, dtype)).clamp_min(0) / scale.clamp_min(1e-30)
    e = torch.where((got.to(F64) == ref), torch.zeros_like(e), e)
    if not torch.isfinite(got.to(F64)).all():
        e = torch.full_like(e, float("inf"))
    if col_blocks is not None:
        return {n: float(e[:, c0:c0 + k].max()) for n, c0, k in col_blocks}
    if row_blocks is not None:
        return {n: float(e[c0:c0 + k].max()) for n, c0, k in row_blocks}
    return float(e.max())


REAL_CASES = [  # B, H (latent 2H), decoder_hidden, N, C
    (1, 128, 256, 10, 4), (255, 256, 128, 10, 7), (256, 128, 256, 10, 4), (300, 128, 512, 13, 4),
    (8192, 128, 256, 10, 4), (20000, 256, 512, 20, 16), (256, 256, 128, 20, 16), (8192, 256, 512, 10, 7),
]


def _real_problem(B, H, DH, N, C, seed):
    from roomslam_b200.model import Decoder
    torch.manual_seed(seed)
    dec = Decoder(2 * H, DH, N, C).cuda()
    g = gen(seed)
    lat = torch.rand(B, 2 * H, generator=g, device="cuda") * 2 - 1
    heads = []
    for h in (dec.class_head, dec.pos_head, dec.size_head, dec.orient_head, dec.valid_head):
        heads += [h.weight.detach(), h.bias.detach()]
    W = [dec.trunk[0].weight.detach(), dec.trunk[0].bias.detach(), dec.trunk[2].weight.detach(), dec.trunk[2].bias.detach()]
    tgt = (torch.randint(0, C, (B, N), generator=g, device="cuda"), torch.randn(B, N, 2, generator=g, device="cuda"),
           torch.rand(B, N, 2, generator=g, device="cuda"), torch.randn(B, N, generator=g, device="cuda"),
           (torch.rand(B, N, generator=g, device="cuda") < 0.5).float())
    return lat, W, heads, tgt


def real_run(case, m, seed=5):
    B, H, DH, N, C = case
    lat, (W1, b1, W2, b2), heads, tgt = _real_problem(B, H, DH, N, C, seed)
    with mode(m):
        r = FB.decoder_bf16_fwd(lat, N, C, W1, b1, W2, b2, heads)
        losses, sums, gl = F_.loss_fwd(*r["heads"], *tgt)
        d_pred = F_.loss_bwd(sums, gl, torch.tensor([1.0, 0.3, -0.2, 0.5, 0.1, -0.4], device="cuda"))
        d_raw = F_.heads_merge(r["raw"], N, C, *d_pred)
        gr = FB.decoder_bf16_bwd(r["lat"], r["W1b"], r["W2b"], r["Wh"], r["f1"], r["f2"], d_raw)
    torch.cuda.synchronize()
    return dict(r=r, gr=gr, d_raw=d_raw, N=N, C=C, heads=heads, b1=b1, b2=b2)


def real_report(run, fault=None):
    """Per-stage (and per head block) errors of one realistic run against the reference, optionally with a fault."""
    r, gr, N, C = run["r"], run["gr"], run["N"], run["C"]
    NH = N * (C + 6)
    NHp = r["Wh"].shape[0]
    blocks = list(D.head_blocks(N, C)) + [("pad", NH, NHp - NH)]
    Wh = r["Wh"].to(F64)
    bh = r["bh"].to(F64)
    if fault == "swap_pos_size":
        Wh, bh = Wh.clone(), bh.clone()
        p0, s0 = N * C, N * C + 2 * N
        Wh[p0:p0 + 2 * N], Wh[s0:s0 + 2 * N] = Wh[s0:s0 + 2 * N].clone(), Wh[p0:p0 + 2 * N].clone()
        bh[p0:p0 + 2 * N], bh[s0:s0 + 2 * N] = bh[s0:s0 + 2 * N].clone(), bh[p0:p0 + 2 * N].clone()
    if fault == "lost_pad_column":
        Wh, bh = Wh.clone(), bh.clone()
        Wh[NH - 1] = 0
        bh[NH - 1] = 0
    f = D.decoder_fwd(r["lat"], r["W1b"], run["b1"], r["W2b"], run["b2"], Wh, bh, f1=r["f1"], f2=r["f2"])
    rep = {"f1": stage_err(r["f1"], f["f1"], f["s1"], BF), "f2": stage_err(r["f2"], f["f2"], f["s2"], BF)}
    rep.update({"rawp." + k: v for k, v in stage_err(r["rawp"], f["rawp"], f["s3"], F32, col_blocks=blocks).items()})
    mask2 = (r["f1"] > 0) if fault == "wrong_relu_mask" else None
    b = D.decoder_bwd(r["lat"], r["W1b"], r["W2b"], Wh, r["f1"], r["f2"], gr["d_rawp"], run["d_raw"], df2=gr["df2"],
                      df1=gr["df1"], mask2=mask2)
    rep.update({"dWh." + k: v for k, v in stage_err(gr["dWh"], b["dWh"], b["s_dWh"], F32, row_blocks=blocks).items()})
    for name, t in (("df2", BF), ("dW2", F32), ("df1", BF), ("dW1", F32), ("dlat", F32)):
        rep[name] = stage_err(gr[name], b[name], b["s_" + name], t)
    return rep


def _bar(stage):
    return FWD_BAR if stage.split(".")[0] in ("f1", "f2", "rawp") else BWD_BAR


@pytest.mark.parametrize("m", MODES)
@pytest.mark.parametrize("case", REAL_CASES, ids=lambda c: "B%d-H%d-D%d-N%d-C%d" % c)
def test_decoder_bf16_realistic(case, m, record_property):
    run = real_run(case, m)
    r, gr, N, C = run["r"], run["gr"], run["N"], run["C"]
    NH = N * (C + 6)
    rep = real_report(run)
    record_property("errors", rep)
    print("decoder_bf16", case, m, {k: "%.2e" % v for k, v in rep.items()})
    bad = {k: v for k, v in rep.items() if v > _bar(k)}
    assert not bad, bad
    # copy stages: bit for bit
    assert bool((r["rawp"][:, NH:] == 0).all()) and bool((gr["d_rawp"][:, NH:] == 0).all())
    assert torch.equal(gr["d_rawp"][:, :NH], run["d_raw"].to(BF))
    assert bool((gr["dWh"][NH:] == 0).all())
    cls, pos, size, orient, valid = r["heads"]
    (_, c0, _), (_, p0, _), _, (_, o0, _), (_, v0, _) = D.head_blocks(N, C)
    assert torch.equal(cls.reshape(-1, N * C), r["raw"][:, :N * C]) and torch.equal(pos.reshape(-1, 2 * N), r["raw"][:, p0:p0 + 2 * N])
    assert torch.equal(orient, r["raw"][:, o0:o0 + N]) and torch.equal(valid, r["raw"][:, v0:v0 + N])
    hg = F_.split_head_grads(gr["dWh"], gr["dbh"], [N * C, 2 * N, 2 * N, N, N])
    assert torch.equal(torch.cat(hg[0::2]), gr["dWh"][:NH]) and torch.equal(torch.cat(hg[1::2]), gr["dbh"])


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_relu_bwd_in_place_exact(dtype):
    """rs_relu_bwd_* called in place (dy == dx), as both decoders call it: dx = y > 0 ? dy : 0 bit for bit."""
    g = gen(19)
    n = 1184 * 256 * 3 + 5                                     # every thread loops
    t = BF if dtype == "bf16" else F32
    y = torch.randn(n, generator=g, device="cuda").to(t)
    y[::7] = 0
    y[1::11] = -0.0
    dy = torch.randn(n, generator=g, device="cuda").to(t)
    dy[::13] = float("nan")
    want = torch.where(y.float() > 0, dy, torch.zeros_like(dy))
    x = dy.clone()
    _lib.call("rs_relu_bwd_bf16" if dtype == "bf16" else "rs_relu_bwd_f32", x.data_ptr(), y.data_ptr(), x.data_ptr(), n, _st())
    torch.cuda.synchronize()
    assert torch.equal(x.view(torch.int16 if dtype == "bf16" else torch.int32), want.view(torch.int16 if dtype == "bf16" else torch.int32))


# =========================================== C. heads, loss, AdamW =====================================================
def ulps(got, ref):
    """max |got - ref| in units of the float32 ulp of ref; differences below the smallest normal float32 (an underflowed
    exp) count as 0."""
    ref = ref.to(F64)
    e = torch.floor(torch.log2(ref.abs().clamp_min(2.0 ** -126)))
    d = ((got.to(F64) - ref).abs() - 2.0 ** -126).clamp_min(0)
    return (d / torch.exp2(e - 23)).max().item() if ref.numel() else 0.0


HEAD_NC = [(1, 1), (10, 4), (13, 7), (37, 16), (1, 16), (37, 1)]


@pytest.mark.parametrize("m", MODES)
@pytest.mark.parametrize("N,C", HEAD_NC)
def test_heads_split_merge(N, C, m):
    g = gen(23 + N * C)
    B = 517
    NH = N * (C + 6)
    raw = torch.randn(B, NH, generator=g, device="cuda") * 8
    s0 = N * C + 2 * N
    special = torch.tensor([20.0, float(np.nextafter(np.float32(20), np.float32(30))), -100.0, 88.0, 19.99, 0.0], device="cuda")
    raw[:6, s0:s0 + 2 * N] = special[:, None].expand(6, 2 * N)
    raw[7, :N * C] = float("nan")                              # NaN passes through the copy columns
    raw[7, N * C:s0] = float("nan")
    with mode(m):
        out = F_.heads_split(raw, N, C)
    torch.cuda.synchronize()
    ref = D.heads_split(raw, N, C)
    for k, (got, want) in enumerate(zip(out, ref)):
        if k == 2:
            assert ulps(got, want) <= SP_ULPS, ulps(got, want)
        else:
            assert torch.equal(got.to(F64).nan_to_num(7.5), want.nan_to_num(7.5)), k
    assert bool(out[0][7].isnan().all()) and bool(out[1][7].isnan().all())
    # A softplus threshold moved from 20 to 21 is not observable in float32: above 20, log1p(exp(-v)) < 2^-24 v, so both
    # branches round to the same float32 size and sigmoid; the reference equality below holds for either threshold.
    assert torch.equal(D.heads_split(raw, N, C, threshold=21.0)[2].float(), ref[2].float())
    d = [torch.randn(s, generator=g, device="cuda") for s in ((B, N, C), (B, N, 2), (B, N, 2), (B, N), (B, N))]
    d[2][:3] = 1.0                                             # d_size = 1: the sigmoid itself
    for drop in (None, 0, 1, 2, 3, 4):
        dd = [None if k == drop else t for k, t in enumerate(d)]
        d_raw = torch.full_like(raw, float("nan"))
        with mode(m):
            _lib.call("rs_heads_merge_bwd_f32", raw.data_ptr(), B, N, C, *[0 if t is None else t.data_ptr() for t in dd],
                      d_raw.data_ptr(), _st())
        torch.cuda.synchronize()
        want = D.heads_merge(raw, N, C, *dd)
        for k, (name, c0, n) in enumerate(D.head_blocks(N, C)):
            if k == drop:
                assert bool((d_raw[:, c0:c0 + n] == 0).all()), name
            elif name == "size":
                assert ulps(d_raw[:, c0:c0 + n], want[:, c0:c0 + n]) <= SP_ULPS, name
            else:
                assert torch.equal(d_raw[:, c0:c0 + n].to(F64).nan_to_num(7.5), want[:, c0:c0 + n].nan_to_num(7.5)), name


def _loss_inputs(B, N, C, g, valid="binary", extreme=False):
    cls = torch.randn(B, N, C, generator=g, device="cuda") * 3
    pos, size = torch.randn(B, N, 2, generator=g, device="cuda"), torch.rand(B, N, 2, generator=g, device="cuda")
    orient, vlog = torch.randn(B, N, generator=g, device="cuda"), torch.randn(B, N, generator=g, device="cuda") * 4
    t_cls = torch.randint(0, C, (B, N), generator=g, device="cuda")
    t_pos, t_size, t_orient = torch.randn(B, N, 2, generator=g, device="cuda"), torch.rand(B, N, 2, generator=g, device="cuda"), \
        torch.randn(B, N, generator=g, device="cuda")
    if valid == "none":
        t_valid = torch.zeros(B, N, device="cuda")
    elif valid == "all":
        t_valid = torch.ones(B, N, device="cuda")
    elif valid == "fractional":
        t_valid = torch.rand(B, N, generator=g, device="cuda")
    else:
        t_valid = (torch.rand(B, N, generator=g, device="cuda") < 0.4).float()
    if extreme:
        cls[0, :, 0] += 100.0                                  # logit gap of 100
        vlog[0, 0], vlog[0, -1] = 100.0, -100.0                # BCE logits of +-100
        pos[1], size[1], orient[1] = t_pos[1], t_size[1], t_orient[1]      # exact L1 ties: zero gradient
    return [cls, pos, size, orient, vlog], [t_cls, t_pos, t_size, t_orient, t_valid]


LOSS_CASES = [  # B, N, C, valid, extreme
    (3, 10, 4, "none", True), (64, 10, 4, "all", True), (50, 13, 7, "fractional", True), (40, 37, 1, "binary", True),
    (30, 1, 16, "binary", True), (31000, 10, 4, "binary", False),   # 310000 > 1184 x 256 slots: every thread loops
]


def loss_check(pred, tgt, losses, sums, g, d, d_losses, fault=None):
    """True when the kernel outputs agree with the (optionally faulty) reference."""
    B, N, C = pred[0].shape
    slots = B * N
    rs, rg = D.loss_terms(*pred, *tgt)
    ok = abs(float(sums[0]) - float(rs[0])) <= 1e-6 * max(1.0, float(rs[0]))
    for k in range(1, 6):
        scale = {1: (tgt[4].double() * (torch.logsumexp(pred[0].double(), -1).abs() + 1)).sum(), 5: rs[5].abs() + slots}.get(k, rs[k].abs())
        ok &= abs(float(sums[k]) - float(rs[k])) <= 1e-6 * float(scale) + 1e-30
    lf = D.loss_finalize(rs, slots)
    coefs = D.loss_coefs(rs, slots, d_losses)
    if fault == "pos_by_nv":
        lf[2] *= 2
        coefs[1] *= 2
    if fault == "bce_over_valid":
        lf[5] = float(rs[5]) / max(float(rs[0]), 1.0)
        coefs[4] = (float(d_losses[0]) * D.LOSS_WEIGHTS[4] + float(d_losses[5])) / max(float(rs[0]), 1.0)
    if fault in ("pos_by_nv", "bce_over_valid"):
        lf[0] = sum(w * float(x) for w, x in zip(D.LOSS_WEIGHTS, lf[1:]))
    ok &= bool(((losses.double().cpu() - lf).abs() <= 1e-5 * lf.abs() + 1e-12).all())
    lse = torch.logsumexp(pred[0].double(), -1, keepdim=True).abs()
    v = tgt[4].double()
    for k, (got, want) in enumerate(zip(g, rg)):
        if k in (1, 2, 3):
            ok &= torch.equal(got.to(F64), want)               # exactly +-v or 0
        elif k == 0:                                           # exp(l - lse): lse carries 1/2 ulp of |lse|
            ok &= bool(((got.to(F64) - want).abs() <= 4 * 2.0 ** -24 * v[..., None] * (1 + lse)).all())
        else:
            ok &= bool(((got.to(F64) - want).abs() <= 4 * 2.0 ** -24).all())
    for got, gg, k in zip(d, g, coefs):                       # the kernel's own g times the reference coefficient
        want = gg.to(F64) * k                                  # (a product below the smallest normal may flush to 0)
        ok &= bool(((got.to(F64) - want).abs() <= 8 * 2.0 ** -24 * want.abs() + 2.0 ** -126).all())
    return ok


@pytest.mark.parametrize("m", MODES)
@pytest.mark.parametrize("case", LOSS_CASES, ids=lambda c: "B%d-N%d-C%d-%s" % c[:4])
def test_loss_kernels(case, m):
    B, N, C, valid, extreme = case
    g = gen(29 + B)
    pred, tgt = _loss_inputs(B, N, C, g, valid, extreme)
    d_losses = torch.tensor([0.7, -1.3, 2.1, 0.4, -0.9, 1.6], device="cuda")
    with mode(m):
        losses, sums, gk = F_.loss_fwd(*pred, *tgt)
        d = F_.loss_bwd(sums, gk, d_losses)
    torch.cuda.synchronize()
    assert loss_check(pred, tgt, losses, sums, gk, d, d_losses.double())
    if extreme:
        assert bool((gk[1][1] == 0).all() and (gk[2][1] == 0).all() and (gk[3][1] == 0).all())
        assert bool(torch.isfinite(losses).all())
    if valid == "none":
        assert float(sums[0]) == 0 and float(losses[1]) == 0 and float(losses[2]) == 0


def test_loss_rejects_17_classes():
    g = gen(31)
    pred, tgt = _loss_inputs(4, 2, 17, g)
    with pytest.raises(_lib.RoomSlamError):
        F_.loss_fwd(*pred, *tgt)


ADAM_CASES = [  # n, step, max_norm, grad_scale, grad magnitude, clipping active
    (1, 1, 1.0, 1.0, 3.0, True), (255, 2, 1.0, 0.125, 0.01, False), (257, 1000, 0.0, 1.0, 0.1, False),
    (592 * 256 + 1, 2, 1.0, 0.125, 1.0, True), (10 ** 6, 1000, 1.0, 1.0, 0.05, True), (10 ** 6, 1, 1e4, 0.125, 0.05, False),
]


def _adam_state(n, step, gmag, g):
    p0 = torch.randn(n, generator=g, device="cuda") * 0.1
    gr = torch.randn(n, generator=g, device="cuda") * gmag
    if step == 1:
        m0, v0 = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    else:
        m0 = torch.randn(n, generator=g, device="cuda") * gmag * 0.1
        v0 = torch.rand(n, generator=g, device="cuda") * gmag * gmag * 0.01
    return p0, gr, m0, v0


def adam_run(p0, gr, m0, v0, hp, m):
    p, mm, v = p0.clone(), m0.clone(), v0.clone()
    scratch = torch.full((1,), float("nan"), dtype=F64, device="cuda")
    with mode(m):
        _lib.call("rs_adamw_step_f32", p.data_ptr(), gr.data_ptr(), mm.data_ptr(), v.data_ptr(), p.numel(), hp["lr"], hp["b1"],
                  hp["b2"], hp["eps"], hp["wd"], hp["step"], hp["gs"], hp["max_norm"], scratch.data_ptr(), _st())
    torch.cuda.synchronize()
    return p, mm, v, scratch


def upd_scale(p0, m0, gr, hp, ref):
    """The size of each element's update before its terms cancel: lr wd |p0| + lr / bc1 (b1 |m0| + (1 - b1) |g|) / denom,
    g the scaled and clipped gradient."""
    f = lambda x: float(np.float32(x))  # noqa: E731
    lr, wd, b1, eps = f(hp["lr"]), f(hp["wd"]), f(hp["b1"]), f(hp["eps"])
    bc1, bc2 = D.bias_corrections(hp["b1"], hp["b2"], hp["step"], True)
    clip = min(1.0, hp["max_norm"] / (math.sqrt(ref[3]) + D.CLIP_EPS)) if hp["max_norm"] > 0 else 1.0
    gi = gr.double().abs() * f(hp["gs"]) * clip
    adam = (lr / bc1) * (b1 * m0.double().abs() + (1 - b1) * gi) / (ref[2].sqrt() / math.sqrt(bc2) + eps)
    return lr * wd * p0.double().abs() + adam


def adam_err(p, mm, v, p0, m0, v0, gr, hp, ref):
    """max over the elements of (|p - p_ref| - 2 ulp(p)) / update size, and the errors of m and v relative to the sizes
    of their two terms."""
    rp, rm, rv, _ = ref
    e = ((p.double() - rp).abs() - rp.abs() * 2.0 ** -22).clamp_min(0) / upd_scale(p0, m0, gr, hp, ref).clamp_min(1e-30)
    gs = gr.double().abs() * hp["gs"]
    em = ((mm.double() - rm).abs() / (m0.double().abs() + 0.1 * gs + 1e-30)).max().item()
    ev = ((v.double() - rv).abs() / (v0.double().abs() + 1e-3 * gs * gs + 1e-38)).max().item()
    return e.max().item(), em, ev


ADAM_UPDATE_BAR = 1e-6          # about 8 float32 roundings of the update, beyond 2 ulp of p (the decay product and the store)


@pytest.mark.parametrize("m", MODES)
@pytest.mark.parametrize("case", ADAM_CASES, ids=lambda c: "n%d-t%d-clip%g-gs%g" % c[:4])
def test_adamw(case, m):
    n, step, max_norm, gs, gmag, clips = case
    g = gen(37 + n)
    p0, gr, m0, v0 = _adam_state(n, step, gmag, g)
    hp = dict(lr=2.0 ** -5, b1=0.9, b2=0.999, eps=1e-8, wd=1e-2, step=step, gs=gs, max_norm=max_norm)
    p, mm, v, scratch = adam_run(p0, gr, m0, v0, hp, m)
    args = (p0, gr, m0, v0, hp["lr"], hp["b1"], hp["b2"], hp["eps"], hp["wd"], step, gs, max_norm)
    ref = D.adamw_step(*args, f32_bias_correction=True)
    ep, em, ev = adam_err(p, mm, v, p0, m0, v0, gr, hp, ref)
    assert ep < ADAM_UPDATE_BAR and em < 1e-6 and ev < 1e-6, (ep, em, ev)
    if max_norm > 0:
        assert abs(float(scratch) - ref[3]) <= 1e-6 * ref[3]
    assert (max_norm > 0 and max_norm / (math.sqrt(ref[3]) + 1e-6) < 1) == clips
    for fault in (dict(sqrt_bc2=False), dict(decay_after=True)):
        faulty = D.adamw_step(*args, f32_bias_correction=True, **fault)
        assert adam_err(p, mm, v, p0, m0, v0, gr, hp, faulty)[0] > 100 * ADAM_UPDATE_BAR, fault


def test_adamw_against_torch():
    """With float32-exact betas the step agrees with torch.optim.AdamW (clip_grad_norm_ first) at float32 rounding of
    the update.  With the default betas it deviates by what float32 beta and float32 bias corrections (the C ABI) make:
    the median update is about 1.0e-5 smaller than torch's at step 2 and 3.8e-6 at step 1000 (DESIGN.md section 8)."""
    g = gen(41)
    n = 100_000
    for betas, step, exact in (((0.875, 1 - 2.0 ** -10), 2, True), ((0.9, 0.999), 2, False), ((0.9, 0.999), 1000, False)):
        p0, gr, m0, v0 = _adam_state(n, step, 0.05, g)
        hp = dict(lr=2.0 ** -5, b1=betas[0], b2=betas[1], eps=2.0 ** -27, wd=2.0 ** -7, step=step, gs=1.0, max_norm=1.0)
        p, mm, v, _ = adam_run(p0, gr, m0, v0, hp, "default")
        pt = torch.nn.Parameter(p0.double().clone())
        opt = torch.optim.AdamW([pt], lr=hp["lr"], betas=betas, eps=hp["eps"], weight_decay=hp["wd"])
        pt.grad = gr.double().clone()
        opt.step()                                              # creates the state; then replay from the given state
        with torch.no_grad():
            pt.copy_(p0.double())
        st = opt.state[pt]
        st["exp_avg"].copy_(m0.double())
        st["exp_avg_sq"].copy_(v0.double())
        st["step"].fill_(step - 1)
        pt.grad = gr.double().clone()
        torch.nn.utils.clip_grad_norm_([pt], 1.0)
        opt.step()
        pt = pt.detach()
        ref32 = D.adamw_step(p0, gr, m0, v0, hp["lr"], betas[0], betas[1], hp["eps"], hp["wd"], step, 1.0, 1.0,
                             f32_bias_correction=True)
        if exact:
            scale = upd_scale(p0, m0, gr, hp, ref32)
            assert (((p.double() - pt).abs() - pt.abs() * 2.0 ** -22) / scale).max().item() < ADAM_UPDATE_BAR
        else:                                                   # relative to the signed update: median over the elements
            expected = ((ref32[0] - pt) / (pt - p0.double())).median().item()
            med = ((p.double() - pt) / (pt - p0.double())).median().item()
            assert abs(med - expected) < 3e-7, (med, expected)
            assert (5e-6 < -expected < 2e-5) if step == 2 else (1e-6 < -expected < 8e-6), expected


# =========================================== autograd tie and sensitivity ===============================================
def test_autograd_matches_seam_bit_for_bit():
    """Deterministic mode: DecoderBF16Fn, DecoderFn and MultiTaskLossFn give the seam functions' gradients bit for bit."""
    B, H, DH, N, C = 300, 128, 256, 13, 4
    lat, W, heads, tgt = _real_problem(B, H, DH, N, C, 3)
    d_losses = torch.tensor([1.0, 0.5, -0.25, 0.125, 2.0, -1.0], device="cuda")
    with mode("deterministic"):
        for bf16 in (True, False):
            params = [t.clone().requires_grad_(True) for t in W + heads]
            latr = lat.clone().requires_grad_(True)
            fn = FB.DecoderBF16Fn if bf16 else F_.DecoderFn
            pred = fn.apply(latr, N, C, *params)
            predr = [t.detach().clone().requires_grad_(True) for t in pred]
            losses = F_.MultiTaskLossFn.apply(*predr, *tgt)
            losses.backward(d_losses)
            torch.autograd.backward(pred, [t.grad for t in predr])
            # the seam
            fwd = FB.decoder_bf16_fwd if bf16 else F_.decoder_fwd
            r = fwd(lat, N, C, *W, heads)
            for a, b in zip(r["heads"], pred):
                assert torch.equal(a, b)
            l2, sums, gl = F_.loss_fwd(*r["heads"], *tgt)
            assert torch.equal(l2, losses)
            d_pred = F_.loss_bwd(sums, gl, d_losses)
            for a, b in zip(d_pred, predr):
                assert torch.equal(a, b.grad)
            d_raw = F_.heads_merge(r["raw"], N, C, *d_pred)
            if bf16:
                gr = FB.decoder_bf16_bwd(r["lat"], r["W1b"], r["W2b"], r["Wh"], r["f1"], r["f2"], d_raw)
            else:
                gr = F_.decoder_bwd(r["latent"], W[0], W[2], r["Wh"], r["f1"], r["f2"], d_raw)
            want = [gr["dW1"], gr["db1"], gr["dW2"], gr["db2"]] + F_.split_head_grads(gr["dWh"], gr["dbh"], [N * C, 2 * N, 2 * N, N, N])
            for p, w in zip(params, want):
                assert torch.equal(p.grad, w)
            assert torch.equal(latr.grad, gr["dlat"])


def test_sensitivity():
    """Each injected fault is told apart from the kernel outputs and, in the realistic family, located."""
    run = real_run((300, 128, 256, 10, 4), "default")
    clean = real_report(run)
    assert all(v <= _bar(k) for k, v in clean.items())
    flagged = lambda rep: {k for k, v in rep.items() if v > _bar(k)}  # noqa: E731
    fwd_flags = lambda rep: {k for k in flagged(rep) if k.startswith("rawp")}  # noqa: E731
    assert fwd_flags(real_report(run, "swap_pos_size")) == {"rawp.pos", "rawp.size"}     # (df2 reads Wh too)
    assert flagged(real_report(run, "wrong_relu_mask")) == {"df2"}
    assert fwd_flags(real_report(run, "lost_pad_column")) == {"rawp.valid"}
    g = gen(43)
    pred, tgt = _loss_inputs(200, 10, 4, g, "binary")
    d_losses = torch.tensor([0.7, -1.3, 2.1, 0.4, -0.9, 1.6], device="cuda")
    losses, sums, gk = F_.loss_fwd(*pred, *tgt)
    d = F_.loss_bwd(sums, gk, d_losses)
    torch.cuda.synchronize()
    assert loss_check(pred, tgt, losses, sums, gk, d, d_losses.double())
    for fault in ("pos_by_nv", "bce_over_valid"):
        assert not loss_check(pred, tgt, losses, sums, gk, d, d_losses.double(), fault), fault
    # the softplus threshold at 21 and the two AdamW faults: test_heads_split_merge and test_adamw
