"""bf16 tensor-core encoder with up to 16 input features per step: the layer-0 projection W_ih x + b rides on the recurrence
MMA as ceil((3 I + 2) / 16) extra K = 16 steps (csrc/rec_common.cuh has the column map).  Against the fp32 torch CPU oracle
with the conventions of test_bf16_gpu.py: max|a-b| / max|b| < 2e-2 on states and losses, relative L2 < 2e-2 plus a 1e-1
max-norm bound on every gradient, except the relative L2 error of the layer-0 input weights (below).  Input features at
unit scale.

The layer-0 input-weight gradient is the sum over B T steps of dG x, where dG arrives in bf16 (through the data gradient of
the layer above at L = 2) and x enters the weight-gradient pass as one bf16 value per column.  With more input columns,
each of whose gradients cancels over the batch, its relative L2 error reaches about 2 % on trajectory-like inputs and 3.4 %
on white-noise inputs (B200; 130 to 700 traces, L = 2), with the max-norm error at most 3.3 %.  The backward pass is the
one the 2-input model has always used; this bar records that accuracy rather than the 2e-2 of the other tensors."""
import ctypes

import numpy as np
import pytest
import torch

from oracle.room_slam_ref import RoomSLAM as RefRoomSLAM
from roomslam_b200 import RoomSLAM, _lib, preprocess, synth
from roomslam_b200.train_utils import FlatParams, FusedAdamW

pytestmark = pytest.mark.gpu
RTOL = 2e-2
W_IH0_L2 = 4e-2          # weight_ih_l0(_reverse): relative L2 bar (module docstring)
LOSS_KEYS = ("total", "class", "position", "size", "orientation", "validity")


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-6))


def l2_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def to_cuda(d):
    return {k: v.cuda() for k, v in d.items()}


def features(B, T, I, seed):
    """Unit-scale inputs like a trace's kinematic columns: a synthetic trajectory (x, y), then projections of it on seeded
    directions plus a slow per-trace oscillation, each column standardised.  (White-noise columns, independent of the
    trajectory and of each other from step to step, make the true layer-0 input-weight gradient pure cancellation: the bf16
    weight_ih gradients then stay within the 1e-1 max-norm bound but reach 2-3.4 % relative L2 at L = 2.)"""
    x, tgt = synth.make_sample(B, T, 10, seed=seed)
    x = (x - x.mean((0, 1))) / x.std((0, 1))
    g = torch.Generator().manual_seed(seed + 1)
    n = max(I - 2, 0)
    ang = torch.rand(n, generator=g) * 6.2832
    omega = 0.02 + 0.2 * torch.rand(n, generator=g)
    phase = torch.rand(B, 1, n, generator=g) * 6.2832
    t = torch.arange(T, dtype=torch.float32)[None, :, None]
    extra = x[..., :1] * torch.cos(ang) + x[..., 1:2] * torch.sin(ang) + 0.5 * torch.sin(omega * t + phase)
    extra = (extra - extra.mean((0, 1))) / extra.std((0, 1)).clamp_min(1e-6)
    return torch.cat([x, extra], 2)[:, :, :I].contiguous(), tgt


def check_against_oracle(ref, dev, x, tgt, mask=None, lengths=None):
    enc_ref, hn_ref = ref.encode(x, mask, lengths)
    loss_ref = ref.compute_loss(ref(x, mask, lengths), tgt)
    loss_ref["total"].backward()
    xm = mask.cuda() if mask is not None else None
    ld = lengths.cuda() if lengths is not None else None
    enc_dev, hn_dev = dev.encode(x.cuda(), xm, ld)
    loss_dev = dev.compute_loss(dev(x.cuda(), xm, ld), to_cuda(tgt))
    loss_dev["total"].backward()
    assert rel_err(enc_dev, enc_ref) < RTOL and rel_err(hn_dev, hn_ref) < RTOL
    for k in LOSS_KEYS:
        assert abs(loss_dev[k].item() - loss_ref[k].item()) <= RTOL * max(abs(loss_ref[k].item()), 1e-6), k
    ref_grads = dict(ref.named_parameters())
    errs = {pn: (l2_err(p.grad, ref_grads[pn].grad), rel_err(p.grad, ref_grads[pn].grad)) for pn, p in dev.named_parameters()}
    bad = {k: v for k, v in errs.items() if not (v[0] < (W_IH0_L2 if "weight_ih_l0" in k else RTOL) and v[1] < 1e-1)}
    assert not bad, bad


# (input_size, B, T, L, dropout mask, lengths, split weights).  Below 1024 traces the weights are split (hi + lo); from 38
# tiles (4737 traces) up a CTA pair carries two tiles (NT = 2); split weights with 3 or 4 input K steps do not fit two tiles
# in shared memory, so the host runs those with one.
H128_CASES = [(1, 130, 40, 1, False, False, None), (3, 130, 40, 2, False, False, None), (4, 256, 500, 2, False, False, None),
              (5, 130, 40, 2, True, False, None), (9, 130, 40, 1, False, False, None), (11, 256, 500, 2, False, False, None),
              (16, 130, 40, 2, False, True, None), (3, 4864, 64, 2, False, False, None), (9, 4864, 64, 2, False, False, None),
              (16, 4864, 64, 1, False, False, None), (9, 4864, 64, 1, False, False, True), (11, 4864, 64, 1, False, False, True),
              (16, 700, 64, 2, False, False, False)]


@pytest.mark.parametrize("I,B,T,L,use_mask,use_lengths,split", H128_CASES)
def test_bf16_input_features_match_oracle(I, B, T, L, use_mask, use_lengths, split):
    torch.manual_seed(I + B + T)
    ref = RefRoomSLAM(input_size=I, num_layers=L, dropout=0.1 if use_mask else 0.0)
    dev = RoomSLAM(input_size=I, num_layers=L, dropout=ref.dropout, precision="bf16", bf16_split_weights=split).cuda()
    dev.load_state_dict(ref.state_dict())
    ref.train(use_mask); dev.train(use_mask)
    x, tgt = features(B, T, I, seed=B + I)
    mask = ref.make_dropout_mask(B, T, torch.Generator().manual_seed(1)) if use_mask else None
    lengths = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(2)) if use_lengths else None
    check_against_oracle(ref, dev, x, tgt, mask, lengths)


@pytest.mark.parametrize("I,B,T,L", [(3, 130, 40, 2), (11, 130, 40, 1), (16, 130, 40, 2), (3, 200, 64, 1), (11, 200, 64, 2),
                                     (16, 200, 64, 1)])
def test_bf16_hidden_256_input_features_match_oracle(I, B, T, L):
    torch.manual_seed(I + B + T)
    ref = RefRoomSLAM(input_size=I, hidden_size=256, num_layers=L, dropout=0.0)
    dev = RoomSLAM(input_size=I, hidden_size=256, num_layers=L, dropout=0.0, precision="bf16").cuda()
    dev.load_state_dict(ref.state_dict())
    x, tgt = features(B, T, I, seed=B + I)
    check_against_oracle(ref, dev, x, tgt)


@pytest.mark.parametrize("I", [3, 4, 5, 11, 16])
def test_fp32_input_features_match_oracle(I):
    """fp32 kernels: the fused layer-0 projection (I <= 4) and the projection GEMM (I > 4), 1e-4."""
    B, T = 64, 30
    torch.manual_seed(I)
    ref = RefRoomSLAM(input_size=I, dropout=0.0)
    dev = RoomSLAM(input_size=I, dropout=0.0, precision="fp32").cuda()
    dev.load_state_dict(ref.state_dict())
    x, tgt = features(B, T, I, seed=I)
    _, hn_ref = ref.encode(x)
    loss_ref = ref.compute_loss(ref(x), tgt)
    loss_ref["total"].backward()
    _, hn_dev = dev.encode(x.cuda())
    loss_dev = dev.compute_loss(dev(x.cuda()), to_cuda(tgt))
    loss_dev["total"].backward()
    assert rel_err(hn_dev, hn_ref) < 1e-4
    assert abs(loss_dev["total"].item() - loss_ref["total"].item()) <= 1e-4 * abs(loss_ref["total"].item())
    ref_grads = dict(ref.named_parameters())
    bad = {n: l2_err(p.grad, ref_grads[n].grad) for n, p in dev.named_parameters()}
    bad = {n: e for n, e in bad.items() if not e < 1e-4}
    assert not bad, bad


@pytest.mark.parametrize("H", [128, 256])
@pytest.mark.parametrize("I", [4, 11, 16])
def test_zero_padded_inputs_reproduce_two_input_model(I, H):
    """Pins the column map against the 2-input layout: extra inputs with zero weight_ih columns change nothing."""
    B, T = 300, 50
    torch.manual_seed(7)
    m2 = RoomSLAM(input_size=2, hidden_size=H, dropout=0.0, precision="bf16").cuda()
    mk = RoomSLAM(input_size=I, hidden_size=H, dropout=0.0, precision="bf16").cuda()
    sd = m2.state_dict()
    for k in ("encoder.weight_ih_l0", "encoder.weight_ih_l0_reverse"):
        sd[k] = torch.cat([sd[k], torch.zeros(sd[k].shape[0], I - 2, device=sd[k].device)], 1)
    mk.load_state_dict(sd)
    x2, tgt = features(B, T, 2, seed=3)
    xk = torch.cat([x2, 3.0 * torch.randn(B, T, I - 2, generator=torch.Generator().manual_seed(4))], 2)
    tgt = to_cuda(tgt)
    out2, hn2 = m2.encode(x2.cuda())
    outk, hnk = mk.encode(xk.cuda())
    if I == 4:                          # the same single input K step, plus exact zeros
        assert torch.equal(out2, outk) and torch.equal(hn2, hnk)
    else:
        assert rel_err(outk, out2) <= 1e-6 and rel_err(hnk, hn2) <= 1e-6
    m2.compute_loss(m2(x2.cuda()), tgt)["total"].backward()
    mk.compute_loss(mk(xk.cuda()), tgt)["total"].backward()
    for k in ("weight_ih_l0", "weight_ih_l0_reverse"):
        g2 = getattr(m2.encoder, k).grad
        gk = getattr(mk.encoder, k).grad[:, :2]
        assert l2_err(gk, g2) <= 1e-5, (k, l2_err(gk, g2))


def golden_traces(real_traces, n, seed):
    """n recorded-trace crops of seeded start and length as (N, 4) [x, height, z, t] point arrays."""
    rng = np.random.default_rng(seed)
    w = real_traces["windows"]
    raw = []
    for _ in range(n):
        xz = w[rng.integers(len(w))]
        start = int(rng.integers(0, xz.shape[0] - 20))
        cnt = int(rng.integers(20, xz.shape[0] - start + 1))
        t = np.cumsum(rng.uniform(0.01, 0.2, cnt)) + 10.0
        hgt = rng.normal(1.6, 0.05, cnt)
        raw.append(np.stack([xz[start:start + cnt, 0], hgt, xz[start:start + cnt, 1], t], 1).astype(np.float32))
    return raw


def test_end_to_end_trace_features(real_traces):
    """preprocess.trace_features -> (B, W, 11) kinematic rows -> RoomSLAM(input_size=11, bf16) with lengths, vs the oracle."""
    B = 256
    feats = preprocess.trace_features(golden_traces(real_traces, B, seed=11), max_len=500)
    x, m, lengths = feats["traces"], feats["trace_mask"], feats["lengths"]
    assert x.shape[2] == 11
    valid = x[m]
    x = torch.where(m[..., None], (x - valid.mean(0)) / valid.std(0).clamp_min(1e-6), torch.zeros_like(x)).cpu()
    _, tgt = synth.make_sample(B, 4, 10, seed=12)
    torch.manual_seed(13)
    ref = RefRoomSLAM(input_size=11, dropout=0.0)
    dev = RoomSLAM(input_size=11, dropout=0.0, precision="bf16").cuda()
    dev.load_state_dict(ref.state_dict())
    check_against_oracle(ref, dev, x, tgt, lengths=lengths.cpu())


def train_steps(steps, I=11, B=1100, T=60):
    torch.manual_seed(0)
    model = RoomSLAM(input_size=I, dropout=0.1, precision="bf16").cuda().train()
    flat = FlatParams(model)
    opt = FusedAdamW(flat, lr=1e-3, max_grad_norm=1.0)
    x, tgt = features(B, T, I, seed=5)
    x, tgt = x.cuda(), to_cuda(tgt)
    for _ in range(steps):
        flat.zero_grad()
        pred = model(x)
        model.compute_loss(pred, tgt)["total"].backward()
        opt.step()
    torch.cuda.synchronize()
    return {k: v.detach().clone() for k, v in pred.items()}, flat.grad.clone(), flat.flat.clone()


def test_deterministic_chained_steps_are_bit_identical():
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        a, b = train_steps(2), train_steps(2)
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    for k in a[0]:
        assert torch.equal(a[0][k], b[0][k]), k
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


@pytest.mark.parametrize("H,I", [(128, 11), (128, 16), (256, 11)])
def test_inference_matches_training_forward(H, I):
    """Under no_grad the forward kernel saves no gates; the predictions must not change."""
    torch.manual_seed(1)
    dev = RoomSLAM(input_size=I, hidden_size=H, dropout=0.0, precision="bf16").cuda().eval()
    x, _ = features(300, 40, I, seed=6)
    x = x.cuda()
    with torch.no_grad():
        inf = dev(x)
    trn = dev(x)
    for k in inf:
        assert torch.equal(inf[k], trn[k].detach()), k


def test_rejects_more_than_16_inputs():
    dev = RoomSLAM(input_size=17, precision="bf16").cuda()
    with pytest.raises(_lib.RoomSlamError, match="16"):
        dev(torch.zeros(2, 4, 17, device="cuda"))
    lib = _lib.load()
    B, T, I = 4, 3, 17
    x = torch.zeros(B, T, I, device="cuda")
    whh = torch.zeros(2, 16 + 8, 384, 8, device="cuda", dtype=torch.bfloat16)
    b_hn = torch.zeros(2, 128, device="cuda")
    out = torch.zeros(1, T + 2, 32, 128, 8, device="cuda", dtype=torch.bfloat16)
    h_n = torch.zeros(2, B, 128, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = lib.rs_rec_fwd_bf16(p(x), I, None, ctypes.c_int64(0), None, None, p(whh), p(b_hn), p(out), None, p(h_n), None, None,
                             None, None, 0, B, T, st)
    assert rc != 0
    rc = lib.rs_rec_fwd_bf16_wide(p(x), I, None, p(whh), p(b_hn), p(out), None, p(h_n), None, None, None, None, B, T, st)
    assert rc != 0
    torch.cuda.synchronize()
