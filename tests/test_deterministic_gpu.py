"""Deterministic mode: under torch.use_deterministic_algorithms(True) the library's split reductions sum per-split partials
in a fixed order instead of ending in floating-point atomics, so training replays bit for bit.  The mode changes the
order of the sums only: it must compute what the default path computes, to fp32 summation-order noise."""
import ctypes
import os

import pytest
import torch

from roomslam_b200 import RoomSLAM, _lib, layout as L, synth
from roomslam_b200.train_utils import FlatParams, FusedAdamW


def _set_torch_flag(on, warn_only=False):
    torch.use_deterministic_algorithms(on, warn_only=warn_only)


@pytest.fixture
def det():
    """Turns torch's deterministic flag on for the test and restores the previous state afterwards."""
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    prev_cublas = os.environ.get("CUBLAS_WORKSPACE_CONFIG")
    os.environ["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"      # torch's condition for deterministic cuBLAS calls
    _set_torch_flag(True)
    yield
    _set_torch_flag(prev, prev_warn)
    if prev_cublas is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = prev_cublas


def test_library_mode_follows_torch_flag(built_lib):
    """No GPU needed: the binding hands torch's flag (warn_only included) to rs_set_deterministic before a call."""
    lib = _lib.load()
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        for on, warn_only in ((True, False), (False, False), (True, True), (False, False)):
            _set_torch_flag(on, warn_only)
            _lib.sync_deterministic()
            assert lib.rs_deterministic() == int(on)
    finally:
        _set_torch_flag(prev, prev_warn)
        _lib.sync_deterministic()


def rel_l2(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def rel_max(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def st():
    return torch.cuda.current_stream().cuda_stream


# ---- training: RoomSLAM + multi-task loss + FusedAdamW ------------------------------------------------------------------
# fp32 at 32 x 200: split-K weight gradients and multi-slab column sums; bf16 H 128 at 1100 traces: projection fused into the
# recurrence, at 300 traces: split (hi + lo) weights and the projection GEMM; H 256: the wide kernels
TRAIN_SHAPES = [("fp32", 128, 32, 200, False), ("bf16", 128, 1100, 60, False), ("bf16", 128, 300, 40, False),
                ("bf16", 256, 260, 20, False), ("bf16", 128, 300, 40, True)]


def train_run(precision, H, B, T, use_lengths, steps):
    torch.manual_seed(0)
    model = RoomSLAM(hidden_size=H, dropout=0.1, precision=precision).cuda().train()
    flat = FlatParams(model)
    opt = FusedAdamW(flat, lr=1e-3, max_grad_norm=1.0)
    x, tgt = synth.make_sample(B, T, 10, seed=5)
    x, tgt = x.cuda(), {k: v.cuda() for k, v in tgt.items()}
    lengths = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(1)) if use_lengths else None
    for _ in range(steps):
        flat.zero_grad()
        pred = model(x, lengths=lengths)
        losses = model.compute_loss(pred, tgt)
        losses["total"].backward()
        grads = {n: p.grad.clone() for n, p in zip(flat.names, flat.params)}
        opt.step()
    torch.cuda.synchronize()
    return {"pred": {k: v.detach().clone() for k, v in pred.items()}, "loss": torch.stack([v.detach() for v in losses.values()]),
            "grad": flat.grad.clone(), "grads": grads, "param": flat.flat.clone(), "m": opt.m.clone(), "v": opt.v.clone()}


@pytest.mark.gpu
@pytest.mark.parametrize("precision,H,B,T,use_lengths", TRAIN_SHAPES)
def test_chained_training_is_bit_identical(det, precision, H, B, T, use_lengths):
    a = train_run(precision, H, B, T, use_lengths, steps=3)
    b = train_run(precision, H, B, T, use_lengths, steps=3)
    for k in a["pred"]:
        assert torch.equal(a["pred"][k], b["pred"][k]), k
    for k in ("loss", "grad", "param", "m", "v"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("precision,H,B,T,use_lengths", TRAIN_SHAPES)
def test_deterministic_step_matches_default_step(det, precision, H, B, T, use_lengths):
    """One step: the forward pass is untouched (bit-identical predictions), the gradients differ by summation order only."""
    on = train_run(precision, H, B, T, use_lengths, steps=1)
    _set_torch_flag(False)
    off = train_run(precision, H, B, T, use_lengths, steps=1)
    for k in off["pred"]:
        assert torch.equal(on["pred"][k], off["pred"][k]), k
    bad = {n: rel_l2(on["grads"][n], g) for n, g in off["grads"].items() if float(g.norm()) > 0}
    bad = {n: e for n, e in bad.items() if not e < 1e-5}
    assert not bad, bad


# ---- every changed entry point, called twice, against float64 -----------------------------------------------------------
def twice(fn):
    """fn() -> tensor; runs it twice in deterministic mode and checks the bits agree."""
    a = fn().clone()
    b = fn().clone()
    assert torch.equal(a, b)
    return a


@pytest.mark.gpu
def test_sgemm_split_k_accumulate(det):
    from roomslam_b200.functional import matmul_tn
    torch.manual_seed(0)
    K, M, N = 12000, 96, 160                    # K >= 4096 and 2 x 2 output tiles: split over K
    a, b = torch.randn(K, M, device="cuda"), torch.randn(K, N, device="cuda")
    c0 = torch.randn(M, N, device="cuda")

    def run():
        c = c0.clone()
        matmul_tn(a, b, c, flags=1)             # RS_GEMM_ACCUMULATE
        return c
    got = twice(run)
    ref = c0.double() + a.double().t() @ b.double()
    assert rel_max(got, ref) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("accumulate", [False, True])
def test_colsum_multi_slab(det, accumulate):
    from roomslam_b200.functional import colsum
    torch.manual_seed(1)
    a = torch.randn(10000, 300, device="cuda")
    o0 = torch.randn(300, device="cuda")

    def run():
        o = o0.clone()
        colsum(a, o, accumulate=accumulate)
        return o
    got = twice(run)
    ref = a.double().sum(0) + (o0.double() if accumulate else 0)
    assert rel_max(got, ref) < 1e-5


@pytest.mark.gpu
def test_gemm_bf16_tn_seg_acc(det):
    from roomslam_b200.functional import split3, tn_tc
    torch.manual_seed(2)
    M, N, K = 9000, 256, 200
    dy, a = torch.randn(M, N, device="cuda"), torch.randn(M, K, device="cuda")
    dy3, kpy = split3(dy)
    a3, kp = split3(a)

    def run():
        dw = torch.ones(N, kp, device="cuda")
        tn_tc(dy3, kpy, 0, N, a3, kp, kp, dw, a_shift=1, b_shift=0)
        return dw
    got = twice(run)
    ref = 1.0 + dy[1:].double().t() @ a[:-1].double()
    assert rel_max(got[:, :K], ref) < 5e-6


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [True, False])
def test_blk_wgrad(det, paired):
    from roomslam_b200.functional_bf16 import _ones_block, _wgrad
    torch.manual_seed(4)
    B, T, Ca, Cb = 300, 40, 256, 256
    g, h, x = torch.randn(B, T, Ca, device="cuda"), torch.randn(B, T, Cb, device="cuda"), torch.randn(B, T, 16, device="cuda")
    gt, ht, xt = L.to_tile_major(g), L.to_tile_major(h), L.to_tile_major(x)
    # (dG columns, B column 0, n_cols, time shift, bias?, B2?): paired = an even role count, each pair on the same dG columns
    spec = [(0, 0, 128, 0, True, False), (0, 128, 64, -1, False, True), (128, 64, 128, 1, True, True), (128, 0, 0, 0, True, False)]
    if not paired:
        spec = [spec[0], spec[2], spec[3]]

    def run():
        outs, roles = [], []
        for c0, b0, n, sh, has_bias, has_b2 in spec:
            C = torch.ones(128, max(n, 16), device="cuda")
            bias = torch.ones(128, device="cuda") if has_bias else None
            C2 = torch.ones(128, 16, device="cuda") if has_b2 else None
            roles.append((c0 // 8, ht if n else None, Cb, b0 // 8, n, sh, C if n else None, C.shape[1], bias, xt if has_b2 else None, C2))
            outs += [C, bias, C2]
        _wgrad(gt, Ca, _ones_block(torch.device("cuda")), roles, gt.shape[0], T, st())
        return torch.cat([o.reshape(-1) for o in outs if o is not None])
    got = twice(run)
    gd, hd, xd = g.bfloat16().double(), h.bfloat16().double(), x.bfloat16().double()
    ref = []
    for c0, b0, n, sh, has_bias, has_b2 in spec:
        ga = gd[..., c0:c0 + 128]
        hb = torch.zeros(B, T, max(n, 16), dtype=torch.float64, device="cuda")
        src = hd[..., b0:b0 + n]
        if sh == 0:
            hb[..., :n] = src
        elif sh == -1:
            hb[:, 1:, :n] = src[:, :-1]
        else:
            hb[:, :-1, :n] = src[:, 1:]
        ref.append(1.0 + torch.einsum("btm,btn->mn", ga, hb))
        if has_bias:
            ref.append(1.0 + ga.sum((0, 1)))
        if has_b2:
            ref.append(1.0 + torch.einsum("btm,btn->mn", ga, xd))
    ref = torch.cat([r.reshape(-1) for r in ref])
    assert rel_max(got, ref) < 1e-5


@pytest.mark.gpu
def test_adamw_with_clipping(det):
    torch.manual_seed(5)
    n = 400_000                                   # > 256 x 592: every block of the norm pass strides over several chunks
    p0, g = torch.randn(n, device="cuda"), torch.randn(n, device="cuda") * 0.05
    m0, v0 = torch.randn(n, device="cuda") * 0.01, torch.rand(n, device="cuda") * 1e-4
    lr, b1, b2, eps, wd, step, max_norm = 1e-3, 0.9, 0.999, 1e-8, 1e-2, 3, 1.0
    scratch = torch.zeros(1, dtype=torch.float64, device="cuda")

    def run():
        p, m, v = p0.clone(), m0.clone(), v0.clone()
        _lib.call("rs_adamw_step_f32", p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr, b1, b2, eps, wd, step, 1.0,
                  max_norm, scratch.data_ptr(), st())
        return torch.cat([p, m, v, scratch.float()])
    got = twice(run)
    gd = g.double()
    norm = float(gd.square().sum().sqrt())
    assert norm > 10 * max_norm                   # clipping is active
    assert abs(float(scratch) - norm ** 2) <= 1e-6 * norm ** 2
    gc = gd * min(1.0, max_norm / (norm + 1e-6))
    m = b1 * m0.double() + (1 - b1) * gc
    v = b2 * v0.double() + (1 - b2) * gc * gc
    p = p0.double() * (1 - lr * wd) - (lr / (1 - b1 ** step)) * m / (v.sqrt() / (1 - b2 ** step) ** 0.5 + eps)
    assert rel_max(got[:n], p) < 1e-6 and rel_max(got[n:2 * n], m) < 1e-5 and rel_max(got[2 * n:3 * n], v) < 1e-5


@pytest.mark.gpu
def test_loss_sums_over_many_blocks(det):
    torch.manual_seed(6)
    B, N, C = 20000, 10, 4                        # 200k slots: 782 blocks of partial sums
    cls, pos, size = torch.randn(B, N, C, device="cuda"), torch.randn(B, N, 2, device="cuda"), torch.rand(B, N, 2, device="cuda")
    orient, vlog = torch.randn(B, N, device="cuda"), torch.randn(B, N, device="cuda")
    t_cls, t_pos, t_size = torch.randint(0, C, (B, N), device="cuda"), torch.randn(B, N, 2, device="cuda"), torch.rand(B, N, 2, device="cuda")
    t_orient, t_valid = torch.randn(B, N, device="cuda"), (torch.rand(B, N, device="cuda") < 0.4).float()
    w5 = (ctypes.c_float * 5)(1.0, 2.0, 3.0, 4.0, 5.0)
    sums, losses = torch.empty(6, dtype=torch.float64, device="cuda"), torch.empty(6, device="cuda")
    g = [torch.empty_like(t) for t in (cls, pos, size, orient, vlog)]

    def run():
        _lib.call("rs_loss_fwd_f32", cls.data_ptr(), pos.data_ptr(), size.data_ptr(), orient.data_ptr(), vlog.data_ptr(),
                  t_cls.data_ptr(), t_pos.data_ptr(), t_size.data_ptr(), t_orient.data_ptr(), t_valid.data_ptr(), B, N, C,
                  ctypes.addressof(w5), sums.data_ptr(), losses.data_ptr(), *[t.data_ptr() for t in g], st())
        return torch.cat([sums, losses.double()])
    got = twice(run)
    v, l = t_valid.double(), vlog.double()
    ce = torch.logsumexp(cls.double(), -1) - cls.double().gather(-1, t_cls.unsqueeze(-1)).squeeze(-1)
    ref = torch.stack([v.sum(), (v * ce).sum(), (v[..., None] * (pos.double() - t_pos.double()).abs()).sum(),
                       (v[..., None] * (size.double() - t_size.double()).abs()).sum(), (v * (orient.double() - t_orient.double()).abs()).sum(),
                       (l.clamp_min(0) - l * v + torch.log1p(torch.exp(-l.abs()))).sum()])
    assert rel_max(got[:6], ref) < 1e-5
    nv = float(ref[0])
    parts = [ref[1] / nv, ref[2] / (2 * nv), ref[3] / (2 * nv), ref[4] / nv, ref[5] / (B * N)]
    total = sum(w * float(x) for w, x in zip((1.0, 2.0, 3.0, 4.0, 5.0), parts))
    assert rel_max(got[6:], torch.tensor([total] + [float(x) for x in parts], dtype=torch.float64)) < 1e-5


@pytest.mark.gpu
def test_query_attn_bwd_with_80_queries(det):
    from roomslam_b200.lstm_model import QueryAttnFn, trace_stats
    torch.manual_seed(7)
    B, N, Q, D = 4, 700, 80, 64
    traces = torch.randn(B, N, 11, device="cuda")
    valid = torch.rand(B, N, device="cuda") < 0.9
    mask = valid.to(torch.uint8)
    memory = torch.zeros(B, N + 2, D, device="cuda")
    memory[:, 1:N + 1] = torch.randn(B, N, D, device="cuda")
    qk, qb = torch.randn(Q, D, device="cuda") * 0.1, torch.randn(Q, device="cuda") * 0.1
    gc, ga, gs = torch.randn(B, Q, D, device="cuda"), torch.randn(B, Q, 3, device="cuda"), torch.randn(B, D, device="cuda")
    mean, rms, count = trace_stats(traces, mask)

    def run():
        mem, k, b = memory.clone().requires_grad_(True), qk.clone().requires_grad_(True), qb.clone().requires_grad_(True)
        ctx, anchor, summary = QueryAttnFn.apply(mem, k, b, traces, mask, mean, rms, count)
        ((ctx * gc).sum() + (anchor * ga).sum() + (summary * gs).sum()).backward()
        return torch.cat([mem.grad.reshape(-1), k.grad.reshape(-1), b.grad])
    got = twice(run)
    # float64 reference on the host, mean / rms / count as constants
    mem = memory[:, 1:N + 1].double().cpu().requires_grad_(True)
    k, b = qk.double().cpu().requires_grad_(True), qb.double().cpu().requires_grad_(True)
    vm = valid.cpu()
    nc = (traces[..., :3].double().cpu() - mean.double().cpu()[:, None]) / rms.double().cpu()[:, None, None]
    s = torch.einsum("qd,bnd->bqn", k, mem) + b[None, :, None]
    attn = torch.softmax(s.masked_fill(~vm[:, None, :], float("-inf")), -1)
    ctx, anchor = attn @ mem, attn @ nc
    summary = (mem * vm[..., None]).sum(1) / count.double().cpu()[:, None]
    ((ctx * gc.double().cpu()).sum() + (anchor * ga.double().cpu()).sum() + (summary * gs.double().cpu()).sum()).backward()
    d_mem = got[:B * (N + 2) * D].view(B, N + 2, D)
    assert float(d_mem[:, 0].abs().max()) == 0 and float(d_mem[:, N + 1].abs().max()) == 0
    assert rel_max(d_mem[:, 1:N + 1], mem.grad) < 1e-4
    dq = got[B * (N + 2) * D:]
    assert rel_max(dq[:Q * D].view(Q, D), k.grad) < 1e-4
    # d qb = sum_n p (dP - delta) is zero up to rounding (a per-query shift of all scores leaves the softmax unchanged)
    assert float((dq[Q * D:].cpu() - b.grad).abs().max()) < 1e-4 * float(k.grad.abs().max())


# ---- the shipped BiLSTM + query-decoder pipeline ----------------------------------------------------------------------
def bilstm_run(steps):
    from roomslam_b200.lstm_model import build_model
    from roomslam_b200.set_loss import SetCriterion
    torch.manual_seed(0)
    model = build_model(num_queries=80, d_model=256).cuda().train()
    flat = FlatParams(model)
    opt = FusedAdamW(flat, lr=1e-3, max_grad_norm=1.0)
    g = torch.Generator().manual_seed(1)
    B, N, M = 4, 1200, 50                         # B (N + 2) >= 4096: the tensor-core (bf16x6) GEMMs run
    x = torch.randn(B, N, 11, generator=g).cuda()
    tmask = torch.ones(B, N, dtype=torch.bool, device="cuda")
    tgt = {"boxes": torch.cat([torch.randn(B, M, 3, generator=g), torch.rand(B, M, 3, generator=g) + 0.2], -1).cuda(),
           "labels": torch.randint(0, 4, (B, M), generator=g).cuda(), "valid_mask": (torch.rand(B, M, generator=g) < 0.3).cuda()}
    crit = SetCriterion({"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0})
    for _ in range(steps):
        flat.zero_grad()
        crit(model(x, tmask), tgt)["total_loss"].backward()
        opt.step()
    torch.cuda.synchronize()
    return flat.flat.clone()


@pytest.mark.gpu
def test_bilstm_pipeline_chained_steps_are_bit_identical(det):
    assert torch.equal(bilstm_run(2), bilstm_run(2))
