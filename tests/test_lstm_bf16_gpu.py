"""GPU: the bf16 tensor-core LSTM recurrence (csrc/lstm_pair.cu, H = 128) and the shipped model's precision="bf16".

Per step, direct C-ABI calls against oracle/bilstm_ref.py, teacher-forced on the kernel's own operands: the float64 step is
fed the kernel's bf16-rounded h_{t-1} (forward) or bf16-rounded dG_{t+1} (backward) and the exact bf16 weights (hi, or
hi + lo with split).  What is left is an fp32 sum of products in some order, bounded by U32 * sum |a||b| (the oracle's
`bound`), plus the error of the tanh.approx activations (max relative error 2^-10.99 per the PTX ISA): ACT below.

    gates      |dg| <= 20 U32 (bound + |g|) + ACT                    c   |dc| <= 4 U32 (|f c_prev| + |i g| + |c|)
    out        |dh| <= 10 U32 h_bound + ACT |h|                      dG  |ddG| <= 72 U32 (bound + |dG|) + 4 ACT bound U32

The ulp factors are those of tests/test_bilstm_kernels_gpu.py for the fp32 kernels; ACT = 2^-10 covers the approximate
activations (sigma(x) = tanh(x / 2) / 2 + 1 / 2 and tanh), and in dG the approximate tanh(c) of the recomputed cell
derivative.  A fault (i / f swapped, dc carried without x f, the reverse direction reading the wrong neighbour) moves
values by O(0.1) and is told apart.

Model level, bf16 against the fp32 path (which tests/test_lstm_gpu.py holds to the CPU oracle at 1e-4): relative L2 <= 2e-2
for the predictions, every set-loss term and every parameter gradient at 20 x 3000, d_model 256, Q 80, on the recorded
traces of tests/golden/features.npz, also with ragged masks and an inter-layer dropout mask.
"""
import math

import numpy as np
import os
import pytest
import torch

from oracle import bilstm_ref as R
from roomslam_b200 import _lib
from roomslam_b200 import lstm_model as LM

pytestmark = pytest.mark.gpu

H = 128
SENT = -77.0
F64 = torch.float64
X = 4                        # extra columns of every sequence buffer (ld = width + 4: the kernels access float4)
ACT = 2.0 ** -10
BARS = {"gates": 20.0, "c": 4.0, "out": 10.0, "dG_tf": 72.0}
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


def framed(B, rows, width):
    buf = torch.full((B, rows + 2, width + X), SENT, device="cuda")
    buf[:, 1:-1, :width] = float("nan")
    return buf


def frame_intact(buf, width):
    m = torch.ones(buf.shape, dtype=torch.bool, device="cuda")
    m[:, 1:-1, :width] = False
    return bool((buf[m] == SENT).all())


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def bf16(x):
    return x.to(torch.bfloat16).to(F64)


def weights_seen(w_hh, split):
    """The weights the tensor core multiplies by: bf16(w), or bf16(w) + bf16(w - bf16(w))."""
    hi = bf16(w_hh.float())
    return hi + bf16((w_hh.double() - hi).float()) if split else hi


CASES = [(1, 1), (1, 3000), (20, 2), (20, 200), (20, 3000), (129, 9), (129, 200), (300, 1), (300, 9), (300, 200)]


def inputs(B, T, seed=0):
    g = torch.Generator(device="cuda").manual_seed(1000 * B + 7 * T + seed)
    w_hh = (torch.rand(2, 4 * H, H, generator=g, device="cuda") * 2 - 1) * (2.0 / math.sqrt(H))
    P = torch.full((B, T + 2, 8 * H + X), float("nan"), device="cuda")
    P[:, 1:-1, :8 * H] = torch.randn(B, T, 8 * H, generator=g, device="cuda") * 0.8
    d_out = torch.full((B, T + 2, 2 * H + X), float("nan"), device="cuda")
    d_out[:, 1:-1, :2 * H] = torch.randn(B, T, 2 * H, generator=g, device="cuda")
    return {"w_hh": w_hh.contiguous(), "P": P, "d_out": d_out}


def run(B, T, inp, split, save=True, backward=True):
    fwd_img, bwd_img = LM.lstm_pack_bf16(inp["w_hh"][0], inp["w_hh"][1], split)
    k = {"out": framed(B, T, 2 * H), "saved": torch.full((2, B, T, 5, H), float("nan"), device="cuda") if save else None}
    _lib.call("rs_lstm_fwd_bf16", _p(inp["P"]), 8 * H + X, T + 2, 1, _p(fwd_img), _p(k["out"]), 2 * H + X, T + 2, 1,
              _p(k["saved"]), B, T, H, int(split), _st())
    if backward:
        k["dG"] = framed(B, T, 8 * H)
        _lib.call("rs_lstm_bwd_bf16", _p(inp["d_out"]), 2 * H + X, T + 2, 1, _p(k["saved"]), _p(bwd_img), _p(k["dG"]),
                  8 * H + X, T + 2, 1, B, T, H, int(split), _st())
    torch.cuda.synchronize()
    return k


def reference(B, T, inp, k, split, swap_if=False, rev_from_before=False, dc_no_f=False):
    """Float64 teacher-forced references around the kernel outputs k; the keyword arguments each inject one fault."""
    Pd = R.dirs(inp["P"][:, 1:-1, :8 * H], 4)
    w = weights_seen(inp["w_hh"], split)
    if swap_if:
        Pd, w = Pd[:, :, :, [1, 0, 2, 3]], w.view(2, 4, H, H)[:, [1, 0, 2, 3]].reshape(2, 4 * H, H)
    hk = R.dirs(k["out"][:, 1:-1, :2 * H], 1)[:, :, :, 0]
    gk, ck = R.saved_split(k["saved"])
    h_prev = bf16(R.prev_step(hk).float())
    if rev_from_before:
        h_prev[1] = bf16(R.prev_step(torch.stack([hk[1], hk[1]]))[0].float())
    ref = {"tf": R.forward_step(Pd, w, h_prev), "hk": hk, "gk": gk, "ck": ck}
    ref["c"], ref["c_bound"] = R.cell(gk, R.prev_step(ck))
    ref["h"], ref["h_bound"] = R.h_of(gk[:, :, :, 3], ck)
    do = R.dirs(inp["d_out"][:, 1:-1, :2 * H], 1)[:, :, :, 0]
    dGk = R.dirs(k["dG"][:, 1:-1, :8 * H], 4)
    ref["dGk"] = dGk
    ref["bw"] = R.backward(gk, ck, w, do, feedback=bf16(dGk.float()), dc_no_f=dc_no_f)
    return ref


def measure(k, ref):
    U = R.U32
    m, exact = {}, []
    if not frame_intact(k["out"], 2 * H):
        exact.append("out_frame")
    if not frame_intact(k["dG"], 8 * H):
        exact.append("dG_frame")
    if not bool(torch.isfinite(k["saved"]).all()):
        exact.append("saved_unwritten")
    tf = ref["tf"]

    def err(got, want, bound):
        e = (got.to(F64) - want).abs() / bound.clamp_min(1e-300)
        return torch.nan_to_num(e, nan=math.inf, posinf=math.inf)

    m["gates"] = err(ref["gk"], tf["gates"], BARS["gates"] * U * (tf["bound"] + tf["gates"].abs()) + ACT).amax(-1)
    m["c"] = err(ref["ck"], ref["c"], BARS["c"] * U * (ref["c_bound"] + ref["c"].abs()))
    m["out"] = err(ref["hk"], ref["h"], BARS["out"] * U * ref["h_bound"] + ACT * ref["h"].abs())
    bw = ref["bw"]
    m["dG_tf"] = err(ref["dGk"], bw["dG"], (BARS["dG_tf"] + 4 * ACT / U) * U * (bw["bound"] + bw["dG"].abs())).amax(-1)
    return m, exact


def over(m):
    return {n: (e > 1.0).nonzero()[:8].tolist() for n, e in m.items() if bool((e > 1.0).any())}


def worst(m):
    return {n: float(e.max()) for n, e in m.items()}


@pytest.mark.parametrize("split", [0, 1])
@pytest.mark.parametrize("B,T", CASES, ids=lambda v: str(v))
def test_lstm_bf16_per_step(B, T, split):
    inp = inputs(B, T)
    k = run(B, T, inp, split)
    inf = run(B, T, inp, split, save=False, backward=False)
    assert same_bits(inf["out"], k["out"]), "inference (saved = NULL) changed out"
    again = run(B, T, inp, split)
    assert all(same_bits(again[n], k[n]) for n in ("out", "saved", "dG")), "a rerun is not bit-identical"
    m, exact = measure(k, reference(B, T, inp, k, split))
    assert exact == [] and over(m) == {}, (worst(m), exact, over(m))


@pytest.mark.parametrize("fault", ["swap_if", "dc_no_f", "rev_from_before"])
def test_lstm_bf16_reference_tells_faults_apart(fault):
    B, T = 20, 9
    inp = inputs(B, T)
    k = run(B, T, inp, 0)
    m, _ = measure(k, reference(B, T, inp, k, 0, **{fault: True}))
    assert max(float(e.max()) for e in m.values()) > 10.0, (fault, worst(m))


def test_lstm_bf16_trace_permutation():
    B, T = 129, 9
    inp = inputs(B, T)
    k = run(B, T, inp, 0)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(B)).cuda()
    kp = run(B, T, dict(inp, P=inp["P"][perm].contiguous(), d_out=inp["d_out"][perm].contiguous()), 0)
    assert same_bits(kp["out"], k["out"][perm])
    assert same_bits(kp["saved"], k["saved"][:, perm])
    assert same_bits(kp["dG"], k["dG"][perm])


def test_lstm_bf16_other_hidden_size_is_an_error():
    w = torch.zeros(4 * 64, 64, device="cuda")
    img = torch.empty(1 << 20, dtype=torch.bfloat16, device="cuda")
    with pytest.raises(_lib.RoomSlamError, match="H = 128"):
        _lib.call("rs_lstm_pack_weights_bf16", _p(w), _p(w), 64, 0, _p(img), _p(img), _st())


# ------------------------------------------------------------------------------------------------------------ model level
def recorded_batch(B, N, ragged, seed=0):
    """B traces of N points from the three recorded traces of tests/golden/features.npz (features at max_len N), each copy
    shifted and scaled by a seeded amount; ragged: seeded valid lengths."""
    from roomslam_b200 import preprocess
    z = np.load(os.path.join(GOLDEN, "features.npz"))
    raw = [z[f"real{i}_points"] for i in range(3)]
    rng = np.random.default_rng(seed)
    pts = []
    for b in range(B):
        r = raw[b % 3].copy()
        r[:, :3] = r[:, :3] * rng.uniform(0.8, 1.2) + rng.normal(0, 1.0, 3).astype(np.float32)
        if ragged:
            r = r[: max(2, int(len(r) * rng.uniform(0.3, 1.0)))]
        pts.append(r.astype(np.float32))
    f = preprocess.trace_features(pts, max_len=N)
    return f["traces"], f["trace_mask"]


def step_outputs(model, x, mask, tg, dropout_mask, matches=None):
    from roomslam_b200.set_loss import SetCriterion, SetLossFn
    crit = SetCriterion({"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0})
    model.zero_grad(set_to_none=True)
    out = model(x, mask, dropout_mask)
    gb, gl = tg["boxes"].float(), tg["labels"].long()
    if matches is None:
        mp, ms, _, n = crit.matcher.match(out["pred_boxes"], out["pred_classes"], gb, gl, tg["valid_mask"])
        matches = (mp, ms, n)
    losses = SetLossFn.apply(out["pred_boxes"], out["pred_classes"], gb, gl, *matches, (2.0, 5.0, 2.0))
    losses[3].backward()
    res = {"pred_boxes": out["pred_boxes"].detach(), "pred_classes": out["pred_classes"].detach()}
    res.update({f"loss/{n}": losses[i].detach().reshape(1) for i, n in enumerate(("class", "l1", "giou", "total"))})
    res.update({f"grad/{n}": p.grad.detach().clone() for n, p in model.named_parameters()})
    return res, matches


ZERO_GRAD = "grad/decoder.k_proj.bias"


def rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.mark.parametrize("ragged", [False, True])
def test_model_bf16_against_fp32(ragged):
    B, N, Q = 20, 3000, 80
    torch.manual_seed(0)
    ref = LM.build_model(num_queries=Q, d_model=256).cuda().train()
    dev = LM.build_model(num_queries=Q, d_model=256, precision="bf16").cuda().train()
    dev.load_state_dict(ref.state_dict())
    x, mask = recorded_batch(B, N, ragged)
    g = torch.Generator().manual_seed(3)
    tg = {"boxes": torch.cat([torch.randn(B, 50, 3, generator=g), torch.rand(B, 50, 3, generator=g) + 0.2], -1).cuda(),
          "labels": torch.randint(0, 4, (B, 50), generator=g).cuda(), "valid_mask": (torch.rand(B, 50, generator=g) < 0.3).cuda()}
    # the same inter-layer dropout mask on both sides (all ones: dropout off)
    dm = (torch.bernoulli(torch.full((1, B, N, 256), 0.9), generator=g) / 0.9).cuda() if ragged else torch.ones(1, B, N, 256, device="cuda")
    want, matches = step_outputs(ref, x, mask, tg, dm)
    got, _ = step_outputs(dev, x, mask, tg, dm, matches)
    errs = {n: rel_l2(got[n], want[n]) for n in want if n != ZERO_GRAD}
    bad = {n: e for n, e in errs.items() if not e <= 2e-2}
    assert not bad, (bad, max(errs.values()))
    # the one exception: b_k shifts every score of a query by the same amount, which the softmax cancels -- its gradient is 0
    # in exact arithmetic, and both paths hold rounding noise there (bf16 against fp32: relative L2 1.6, measured).  The bar:
    # the noise stays below 1e-4 of the whole gradient's norm in each path.
    total = torch.cat([want[n].flatten() for n in want if n.startswith("grad/")]).norm()
    assert float(got[ZERO_GRAD].norm()) <= 1e-4 * float(total) and float(want[ZERO_GRAD].norm()) <= 1e-4 * float(total), \
        (float(got[ZERO_GRAD].norm()), float(want[ZERO_GRAD].norm()), float(total))


def test_model_bf16_deterministic_steps_and_state_dict():
    """Two chained training steps in deterministic mode are bit-identical run to run; state_dicts interchange."""
    from roomslam_b200.set_loss import SetCriterion
    B, N = 3, 200
    x, mask = recorded_batch(B, N, True, seed=1)
    g = torch.Generator().manual_seed(4)
    tg = {"boxes": torch.cat([torch.randn(B, 50, 3, generator=g), torch.rand(B, 50, 3, generator=g) + 0.2], -1).cuda(),
          "labels": torch.randint(0, 4, (B, 50), generator=g).cuda(), "valid_mask": (torch.rand(B, 50, generator=g) < 0.3).cuda()}
    det = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        finals = []
        for _ in range(2):
            torch.manual_seed(0)
            m = LM.build_model(num_queries=30, d_model=256, precision="bf16").cuda().train()
            opt = torch.optim.AdamW(m.parameters(), lr=1e-3)
            crit = SetCriterion({"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0})
            for _ in range(2):
                opt.zero_grad()
                crit(m(x, mask), tg)["total_loss"].backward()
                opt.step()
            finals.append({k: v.detach().clone() for k, v in m.state_dict().items()})
    finally:
        torch.use_deterministic_algorithms(det)
    assert all(same_bits(finals[0][k].float(), finals[1][k].float()) for k in finals[0])
    fp = LM.build_model(num_queries=30, d_model=256).cuda()
    fp.load_state_dict(finals[0])
    back = LM.build_model(num_queries=30, d_model=256, precision="bf16").cuda()
    back.load_state_dict(fp.state_dict())
    assert set(fp.state_dict()) == set(finals[0]) and all(same_bits(back.state_dict()[k].float(), finals[0][k].float()) for k in finals[0])


def test_precision_arguments():
    with pytest.raises(_lib.RoomSlamError, match="d_model 256"):
        LM.build_model(d_model=128, precision="bf16")
    with pytest.raises(ValueError):
        LM.build_model(precision="fp16")


def test_training_recipe_lowers_the_loss():
    """features -> model -> set loss -> AdamW at d_model 256 in bf16 (the recipe of tests/test_pipeline_gpu.py)."""
    from roomslam_b200.set_loss import SetCriterion
    B, N = 8, 500
    x, mask = recorded_batch(B, N, True, seed=2)
    g = torch.Generator().manual_seed(5)
    tg = {"boxes": torch.cat([torch.randn(B, 50, 3, generator=g), torch.rand(B, 50, 3, generator=g) + 0.2], -1).cuda(),
          "labels": torch.randint(0, 4, (B, 50), generator=g).cuda(), "valid_mask": (torch.rand(B, 50, generator=g) < 0.3).cuda()}
    torch.manual_seed(0)
    m = LM.build_model(num_queries=30, d_model=256, precision="bf16").cuda().train()
    opt = torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4)
    crit = SetCriterion({"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0})
    losses = []
    for _ in range(30):
        opt.zero_grad()
        loss = crit(m(x, mask), tg)["total_loss"]
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
        opt.step()
        losses.append(float(loss.detach()))
    assert all(math.isfinite(v) for v in losses)
    assert np.mean(losses[-5:]) < 0.8 * np.mean(losses[:5]), losses


def test_train_and_inference_drivers_bf16(tmp_path):
    """train_benchmark.py --precision bf16 --d_model 256 runs an epoch on the recorded traces; config.json records the
    precision; inference_benchmark.py --precision bf16 reads the checkpoint."""
    import json
    import subprocess
    import sys
    f = np.load(os.path.join(GOLDEN, "features.npz"))
    cols = json.loads(str(np.load(os.path.join(GOLDEN, "colliders.npz"))["train_json"]))
    for split, ks in (("train", (0, 1)), ("val", (2,))):
        d = tmp_path / split
        d.mkdir()
        json.dump({"colliders": cols}, open(d / "colliders.json", "w"))
        for k in ks:
            json.dump([{"timestamp": float(p[3]), "x": float(p[0]), "y": float(p[1]), "z": float(p[2])} for p in f[f"real{k}_points"]],
                      open(d / f"human_data_{k}.json", "w"))
    root = os.path.dirname(os.path.dirname(__file__))
    out = subprocess.run([sys.executable, os.path.join(root, "train_benchmark.py"), "--data_dir", str(tmp_path / "train"),
                          "--val_dir", str(tmp_path / "val"), "--save_dir", str(tmp_path / "ckpt"), "--epochs", "1",
                          "--d_model", "256", "--num_queries", "80", "--precision", "bf16"],
                         capture_output=True, text=True, cwd=root, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert "Epoch 0:" in out.stdout and "Training completed!" in out.stdout
    assert json.load(open(tmp_path / "ckpt" / "config.json"))["precision"] == "bf16"
    res = tmp_path / "pred.json"
    out = subprocess.run([sys.executable, os.path.join(root, "inference_benchmark.py"), "--checkpoint", str(tmp_path / "ckpt" / "best_model.pth"),
                          "--input", str(tmp_path / "val" / "human_data_2.json"), "--output", str(res), "--threshold", "0.0",
                          "--precision", "bf16"], capture_output=True, text=True, cwd=root, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.load(open(res))["metadata"]["num_colliders"] >= 1
