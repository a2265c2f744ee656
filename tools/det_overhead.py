#!/usr/bin/env python
"""Cost of deterministic mode (torch.use_deterministic_algorithms(True)) on three training steps:

    BASELINE config 3 at one GPU: bf16, 8192 traces x 500 steps, H 128, 2 layers
    C1: fp32, 32 traces x 500 steps (BASELINE config 1)
    the BiLSTM + query-decoder step of the shipped pipeline: 20 traces x 3000 points, 80 queries, d_model 256, Hungarian
    set loss

Each step is forward + loss + backward + FusedAdamW (clip 1.0) and starts from the same parameters and optimizer state.
After a warm-up of every mode the modes are timed alternately, step by step, in this process (CUDA events around each
step); the line reports the medians.  A third mode keeps the flag on but turns off torch's own cost of it,
torch.utils.deterministic.fill_uninitialized_memory (every torch.empty is filled with NaN), which separates the library's
deterministic reductions from what torch adds.  It also reports whether two deterministic runs of 3 chained steps from the same
state end with bit-identical parameters, and the card's name and power limit.

    python tools/det_overhead.py [--steps 20] [--out FILE]
Prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")     # torch's condition for deterministic cuBLAS calls

import torch  # noqa: E402
import torch.utils.deterministic  # noqa: E402,F401

from roomslam_b200.train_utils import FlatParams, FusedAdamW  # noqa: E402


class Workload:
    def __init__(self, name, model, loss_fn):
        self.name, self.model, self.loss_fn = name, model, loss_fn
        self.flat = FlatParams(model)
        self.opt = FusedAdamW(self.flat, lr=1e-3, max_grad_norm=1.0)
        self.start = self.flat.flat.clone()

    def reset(self):
        self.flat.flat.copy_(self.start)
        self.opt.m.zero_()
        self.opt.v.zero_()
        self.opt.t = 0

    def step(self):
        self.flat.zero_grad()
        self.loss_fn().backward()
        self.opt.step()


def gru_workload(name, precision, batch):
    from roomslam_b200 import RoomSLAM, synth
    torch.manual_seed(0)
    model = RoomSLAM(hidden_size=128, num_layers=2, max_objects=10, dropout=0.0, precision=precision).cuda().train()
    x, tgt = synth.make_sample(batch, 500, 10, seed=0)
    x, tgt = x.cuda(), {k: v.cuda() for k, v in tgt.items()}
    return Workload(name, model, lambda: model.compute_loss(model(x), tgt)["total"])


def bilstm_workload():
    from roomslam_b200.lstm_model import build_model
    from roomslam_b200.set_loss import SetCriterion
    torch.manual_seed(0)
    model = build_model(num_queries=80, d_model=256).cuda().train()
    model.encoder.dropout = 0.0
    g = torch.Generator().manual_seed(0)
    B, N, M = 20, 3000, 50
    x = torch.randn(B, N, 11, generator=g).cuda()
    mask = torch.ones(B, N, dtype=torch.bool, device="cuda")
    tgt = {"boxes": torch.cat([torch.randn(B, M, 3, generator=g), torch.rand(B, M, 3, generator=g) + 0.2], -1).cuda(),
           "labels": torch.randint(0, 4, (B, M), generator=g).cuda(), "valid_mask": (torch.rand(B, M, generator=g) < 0.3).cuda()}
    crit = SetCriterion({"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0})
    return Workload("bilstm_20x3000_q80_d256", model, lambda: crit(model(x, mask), tgt)["total_loss"])


def timed_step(w):
    w.reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    w.step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


MODES = {"default": (False, True), "deterministic": (True, True), "deterministic_no_fill": (True, False)}


def set_mode(mode):
    on, fill = MODES[mode]
    torch.use_deterministic_algorithms(on)
    torch.utils.deterministic.fill_uninitialized_memory = fill


def measure(w, steps, warmup):
    for mode in MODES:
        set_mode(mode)
        for _ in range(warmup):
            timed_step(w)
    ms = {mode: [] for mode in MODES}
    for _ in range(steps):
        for mode in MODES:
            set_mode(mode)
            ms[mode].append(timed_step(w))
    set_mode("deterministic")
    finals = []
    for _ in range(2):
        w.reset()
        for _ in range(3):
            w.step()
        finals.append(w.flat.flat.clone())
    set_mode("default")
    med = {mode: statistics.median(v) for mode, v in ms.items()}
    out = {f"ms_{mode}": round(m, 3) for mode, m in med.items()}
    out["overhead_pct"] = round(100.0 * (med["deterministic"] / med["default"] - 1.0), 2)
    out["overhead_no_fill_pct"] = round(100.0 * (med["deterministic_no_fill"] / med["default"] - 1.0), 2)
    out["spread_ms"] = {mode: [round(min(v), 3), round(max(v), 3)] for mode, v in ms.items()}
    out["chained_3_steps_bit_identical"] = bool(torch.equal(finals[0], finals[1]))
    return out


def card():
    out = {"name": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # pragma: no cover
        out["power_limit_w"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="timed steps per mode and workload (medians reported)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.steps < 10:
        raise SystemExit("--steps must be at least 10")
    if not torch.cuda.is_available():
        raise SystemExit("det_overhead.py measures on the GPU: no CUDA device")
    line = {"tool": "det_overhead", "steps_per_mode": args.steps, "card": card(), "workloads": {}}
    for make in (lambda: gru_workload("config3_bf16_8192x500", "bf16", 8192), lambda: gru_workload("c1_fp32_32x500", "fp32", 32),
                 bilstm_workload):
        w = make()
        line["workloads"][w.name] = measure(w, args.steps, args.warmup)
        del w
        torch.cuda.empty_cache()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
