#!/usr/bin/env python
"""fp32 against bf16 LSTM recurrence in the shipped BiLSTM model at d_model 256, Q 80 (build_model's defaults).

    training step (forward + Hungarian set loss + backward + clip 1.0 + AdamW) at 20 x 3000 and 256 x 3000 points
    single-trace inference latency at 1 x 3000

After a warm-up of every workload, the fp32 and bf16 workloads of one shape are timed alternately, step by step, in this
process (CUDA events around each step; medians).  A separate pass with the library's kernel timing on gives the per-kernel
breakdown of one step and the microseconds per serial step of the recurrence kernels (kernel time / (layers x T); both
directions run concurrently).  The SM clock is sampled with nvidia-smi during the timed passes; a run whose clocks were
throttled (any active slowdown reason) is marked rejected.  Inputs are seeded (unit-scale features).

    python tools/lstm_bf16_bench.py [--steps 10] [--warmup 2] [--out FILE]
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

import torch  # noqa: E402

from bench import ClockSampler  # noqa: E402
from roomslam_b200 import functional as F_  # noqa: E402
from roomslam_b200.lstm_model import build_model  # noqa: E402
from roomslam_b200.set_loss import SetCriterion  # noqa: E402

Q, D, LAYERS = 80, 256, 2


class Workload:
    def __init__(self, precision, B, N, train=True):
        self.precision, self.B, self.N = precision, B, N
        torch.manual_seed(0)
        self.model = build_model(num_queries=Q, d_model=D, precision=precision).cuda().train(train)
        self.opt = torch.optim.AdamW(self.model.parameters(), lr=2e-4, weight_decay=1e-4)
        self.crit = SetCriterion({"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0})
        g = torch.Generator().manual_seed(1)
        self.x = torch.randn(B, N, 11, generator=g).cuda()
        self.mask = torch.ones(B, N, dtype=torch.bool, device="cuda")
        self.tg = {"boxes": torch.cat([torch.randn(B, 50, 3, generator=g), torch.rand(B, 50, 3, generator=g) + 0.2], -1).cuda(),
                   "labels": torch.randint(0, 4, (B, 50), generator=g).cuda(),
                   "valid_mask": (torch.rand(B, 50, generator=g) < 0.3).cuda()}
        self.train = train

    def step(self):
        if not self.train:
            with torch.no_grad():
                return self.model(self.x, self.mask)["pred_boxes"]
        self.opt.zero_grad()
        loss = self.crit(self.model(self.x, self.mask), self.tg)["total_loss"]
        loss.backward()
        torch.nn.utils.clip_grad_norm_(self.model.parameters(), 1.0)
        self.opt.step()
        return loss

    def timed(self):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def breakdown(self):
        F_.enable_kernel_timing(True)
        self.step()
        kt = F_.collect_kernel_timing()
        F_.enable_kernel_timing(False)
        return {k: {"ms": round(v[0], 3), "launches": v[1]} for k, v in sorted(kt.items(), key=lambda kv: -kv[1][0])}


def pair(B, N, train, steps, warmup):
    loads = [Workload(p, B, N, train) for p in ("fp32", "bf16")]
    for w in loads:
        for _ in range(warmup):
            w.step()
    torch.cuda.synchronize()
    times = {w.precision: [] for w in loads}
    for _ in range(steps):
        for w in loads:
            times[w.precision].append(w.timed())
    res = {}
    for w in loads:
        res[w.precision] = {"median_ms": round(statistics.median(times[w.precision]), 3),
                            "min_ms": round(min(times[w.precision]), 3), "max_ms": round(max(times[w.precision]), 3)}
        if train:
            bd = w.breakdown()
            res[w.precision]["kernels"] = bd
            per_step = {}
            for k in ("lstm_fwd_f32_kernel", "lstm_bwd_f32_kernel", "lstm_fwd_bf16_kernel", "lstm_bwd_bf16_kernel"):
                if k in bd:
                    per_step[k] = round(1000.0 * bd[k]["ms"] / (LAYERS * N), 3)
            res[w.precision]["us_per_serial_step"] = per_step
    res["bf16_speedup"] = round(res["fp32"]["median_ms"] / res["bf16"]["median_ms"], 2)
    del loads
    torch.cuda.empty_cache()
    return res


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # pragma: no cover
        out["power_limit_w"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lstm_bf16_bench.py needs a CUDA device")
    line = {"tool": "lstm_bf16_bench", "card": card(), "steps": a.steps, "d_model": D, "queries": Q}
    clk = ClockSampler(0)
    clk.start()
    try:
        line["train_20x3000"] = pair(20, 3000, True, a.steps, a.warmup)
        line["train_256x3000"] = pair(256, 3000, True, a.steps, a.warmup)
        line["infer_1x3000"] = pair(1, 3000, False, a.steps, a.warmup)
    finally:
        line["clocks"] = clk.stop()
    line["rejected"] = bool(line["clocks"].get("reasons"))
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
