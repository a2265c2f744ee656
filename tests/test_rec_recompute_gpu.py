"""Layer-0 BPTT without saved gates (rs_rec_bwd_bf16_recompute): the backward kernel replays the forward's MMA and gate
math, so its dG must equal, bit for bit, the dG rs_rec_bwd_bf16 computes from the gates the forward saved.  The forward
without a gates buffer must write the same out, out_drop and h_n.  One level up, a training step whose layer 0 recomputes
its gates must predict exactly what the saved-gate step predicts, and its gradients may differ only by the order of the
fp32 atomic sums (none at all in deterministic mode)."""
import os

import pytest
import torch

from roomslam_b200 import RoomSLAM, _lib, synth
from roomslam_b200 import functional_bf16 as FB
from roomslam_b200 import layout as L
from test_rec_kernels_gpu import BF, Case, _p, _st, make_inputs, nan_like, run_kernels

pytestmark = pytest.mark.gpu

CASES = [
    Case(128, 1024, 40, "x"),
    Case(128, 8192, 12, "x"),
    Case(128, 300, 33, "x", lengths="rand"),                       # 3 tiles (odd), the last one partial
    Case(128, 300, 33, "x", I=1, lengths="rand", d_h_n=False),
    Case(128, 1000, 21, "x", drop=True),                            # layer-0 dropout bits: out_drop and the masked d_out
    Case(128, 1000, 21, "x", lengths="full", drop=True, d_h_n=False, seed=3),
]


@pytest.fixture(params=[False, True], ids=["default", "deterministic"])
def det_mode(request):
    prev, prev_warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    prev_cublas = os.environ.get("CUBLAS_WORKSPACE_CONFIG")
    os.environ["CUBLAS_WORKSPACE_CONFIG"] = ":4096:8"
    torch.use_deterministic_algorithms(request.param)
    yield request.param
    torch.use_deterministic_algorithms(prev, warn_only=prev_warn)
    if prev_cublas is None:
        os.environ.pop("CUBLAS_WORKSPACE_CONFIG", None)
    else:
        os.environ["CUBLAS_WORKSPACE_CONFIG"] = prev_cublas


def bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def run_recompute(c: Case, inp: dict, img: dict) -> dict:
    """Forward with gates = NULL, then the recompute backward; every output NaN-filled first."""
    H, B, T = c.H, c.B, c.T
    tiles = L.n_tiles(B)
    drop_bits, scale = inp["drop"] if inp["drop"] is not None else (None, None)
    k = {"out": nan_like((tiles, T + 2, 2 * H // 8, 128, 8), BF), "h_n": nan_like((2, B, H), torch.float32)}
    k["out_drop"] = nan_like(k["out"].shape, BF) if drop_bits is not None else None
    _lib.call("rs_rec_fwd_bf16", _p(inp["x"]), c.I, 0, 0, 0, 0, _p(img["whh_img"]), _p(img["b_hn"]), _p(k["out"]), 0,
              _p(k["h_n"]), _p(inp["lengths"]), _p(drop_bits), _p(scale), _p(k["out_drop"]), 0, B, T, _st())
    xpack = nan_like((tiles, T, 128, 8), BF)
    k["dG"] = nan_like((tiles, T + 2, H, 128, 8), BF)
    _lib.call("rs_rec_bwd_bf16_recompute", _p(inp["d_out"]), _p(inp["d_h_n"]), _p(inp["x"]), c.I, _p(xpack), _p(k["out"]),
              _p(img["whhT_img"]), _p(img["whh_img"]), img["whh_img"].shape[1], _p(img["b_hn"]), _p(k["dG"]), _p(inp["lengths"]),
              _p(drop_bits), _p(scale), B, T, _st())
    torch.cuda.synchronize()
    return k


@pytest.mark.parametrize("c", CASES, ids=str)
def test_recompute_dG_bit_identical(c, det_mode):
    inp = make_inputs(c)
    saved = run_kernels(c, inp)
    rec = run_recompute(c, inp, saved["img"])
    for n in ("out", "out_drop", "h_n", "dG"):
        if saved.get(n) is None:
            continue
        assert not torch.isnan(rec[n].float()).any(), n
        mism = (bits(rec[n]) != bits(saved[n])).sum().item()
        assert mism == 0, f"{n}: {mism} elements differ from the saved-gate path"


def test_recompute_rejects_what_it_does_not_cover():
    inp = make_inputs(Case(128, 256, 4, "x", I=3))
    with pytest.raises(_lib.RoomSlamError):
        _lib.call("rs_rec_bwd_bf16_recompute", 0, 0, _p(inp["x"]), 3, _p(inp["x"]), _p(inp["x"]), _p(inp["x"]), _p(inp["x"]), 18,
                  _p(inp["x"]), _p(inp["x"]), 0, 0, 0, 256, 4, _st())


def train_step(B, T, recompute, monkeypatch):
    monkeypatch.setattr(FB, "recompute_gates", (lambda padded_in, split, I: not padded_in and not split and I <= 2) if recompute
                        else (lambda padded_in, split, I: False))
    torch.manual_seed(0)
    model = RoomSLAM(hidden_size=128, num_layers=2, dropout=0.0, precision="bf16", bf16_split_weights=False).cuda().train()
    x, tgt = synth.make_sample(B, T, 10, seed=4)
    x, tgt = x.cuda(), {k: v.cuda() for k, v in tgt.items()}
    pred = model(x)
    loss = model.compute_loss(pred, tgt)
    loss["total"].backward()
    torch.cuda.synchronize()
    return {k: v.detach().clone() for k, v in pred.items()}, {n: p.grad.detach().clone() for n, p in model.named_parameters()}


@pytest.mark.parametrize("B", [1024, 8192])
def test_training_step_recompute_vs_saved_gates(B, det_mode, monkeypatch):
    T = 64
    pred_s, grad_s = train_step(B, T, False, monkeypatch)
    pred_r, grad_r = train_step(B, T, True, monkeypatch)
    for k in pred_s:
        assert torch.equal(bits(pred_r[k]) if pred_r[k].is_floating_point() else pred_r[k],
                           bits(pred_s[k]) if pred_s[k].is_floating_point() else pred_s[k]), k
    for n, g in grad_s.items():
        if det_mode:
            assert torch.equal(bits(grad_r[n]), bits(g)), n
        else:
            err = float((grad_r[n].double() - g.double()).norm() / g.double().norm().clamp_min(1e-30))
            assert err <= 1e-5, (n, err)
