#!/usr/bin/env python
"""Cost of input features on the bf16 tensor-core GRU encoder: what a user pays per training step for I input columns.

    bf16, H 128, 2 layers, 8192 traces x 500 steps: input_size 2, 4, 11, 16
    fp32, same shape, input_size 11 (what such a user got before bf16 took more than 2 input columns)
    bf16, H 256, 2 layers, 1024 traces x 4000 steps: input_size 2, 11

Each step is forward + multi-task loss + backward + FusedAdamW (clip 1.0) on unit-scale inputs, dropout 0.1.  After a warm-up
of every workload the workloads of one group are timed alternately, step by step, in this process (CUDA events around each
step); the line reports the medians, and for each workload the median time of the layer-0 recurrence forward kernel
(rec_fwd_pair_kernel / rec_fwd_wide_kernel / fp32: gru_fwd_f32_kernel, the first of the two per step in the library's
kernel-timing records), timed in a separate pass.  It also reports the card's name and power limit.

    python tools/input_features_bench.py [--steps 10] [--out FILE]
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

from roomslam_b200 import RoomSLAM, functional as F_, synth  # noqa: E402
from roomslam_b200.train_utils import FlatParams, FusedAdamW  # noqa: E402


class Workload:
    def __init__(self, precision, H, I, B, T):
        self.name = f"{precision}_H{H}_I{I}_{B}x{T}"
        torch.manual_seed(0)
        self.model = RoomSLAM(input_size=I, hidden_size=H, dropout=0.1, precision=precision).cuda().train()
        self.flat = FlatParams(self.model)
        self.opt = FusedAdamW(self.flat, lr=1e-3, max_grad_norm=1.0)
        x, tgt = synth.make_sample(B, T, 10, seed=1)
        x = (x - x.mean((0, 1))) / x.std((0, 1))
        g = torch.Generator().manual_seed(2)
        self.x = torch.cat([x, torch.randn(B, T, max(I - 2, 0), generator=g)], 2)[:, :, :I].contiguous().cuda()
        self.tgt = {k: v.cuda() for k, v in tgt.items()}
        self.kernel = "gru_fwd_f32_kernel" if precision == "fp32" else ("rec_fwd_pair_kernel" if H == 128 else "rec_fwd_wide_kernel")

    def step(self):
        self.flat.zero_grad()
        loss = self.model.compute_loss(self.model(self.x), self.tgt)["total"]
        loss.backward()
        self.opt.step()
        return loss

    def timed(self):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.step()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)

    def layer0_kernel_ms(self, steps):
        ms = []
        for _ in range(steps):
            F_.enable_kernel_timing(True)
            self.step()
            torch.cuda.synchronize()
            ev = [(e0, e1) for name, e0, e1, _ in F_._KT["events"] if name == self.kernel]
            ms.append(ev[0][0].elapsed_time(ev[0][1]))       # layer 0 runs first
            F_.enable_kernel_timing(False)
        return statistics.median(ms)


def card():
    out = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        out["power_limit_w"], out["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # pragma: no cover
        out["power_limit_w"] = f"unavailable: {e}"
    return out


def run_group(specs, steps, warmup):
    res = {}
    loads = [Workload(*s) for s in specs]
    for w in loads:
        for _ in range(warmup):
            w.step()
    torch.cuda.synchronize()
    times = {w.name: [] for w in loads}
    for _ in range(steps):
        for w in loads:
            times[w.name].append(w.timed())
    for w in loads:
        res[w.name] = {"step_ms": round(statistics.median(times[w.name]), 3),
                       "layer0_fwd_kernel_ms": round(w.layer0_kernel_ms(max(3, steps // 3)), 3)}
    del loads
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("input_features_bench.py needs a CUDA device")
    line = {"tool": "input_features_bench", "card": card(), "steps": a.steps}
    line["h128_8192x500"] = run_group([("bf16", 128, I, 8192, 500) for I in (2, 4, 11, 16)] + [("fp32", 128, 11, 8192, 500)],
                                      a.steps, a.warmup)
    line["h256_1024x4000"] = run_group([("bf16", 256, I, 1024, 4000) for I in (2, 11)], a.steps, a.warmup)
    base = line["h128_8192x500"]["bf16_H128_I2_8192x500"]["step_ms"]
    line["h128_step_vs_input_size_2"] = {k: round(v["step_ms"] / base, 4) for k, v in line["h128_8192x500"].items()}
    s = json.dumps(line)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
