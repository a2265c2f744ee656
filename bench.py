#!/usr/bin/env python
"""Benchmark contract:  python bench.py --gpus N --steps K --warmup W [--impl reference]

Headline metric (BASELINE.json): training traces/s of the RoomSLAM bi-GRU (seq 500, H 128, 2 layers, N=10 objects)
at a GLOBAL batch of 8192 traces (BASELINE config 3: "global batch 8192, bf16, at 1/2/4/8 B200"), plus the
occupancy-heatmap binning throughput in Gpoints/s (1M traces x 500 points in total, 0.05 m grid; config 2).
One "step" = forward + multi-task loss + backward (+ NCCL gradient all-reduce for N > 1) + clip + AdamW on one
synthetic batch.  The headline `value` is STRONG scaling: the global batch is fixed and each of the N GPUs gets 8192/N
traces; the weak-scaling figure (8192 traces PER GPU) is measured in the same run and reported under `weak`.
`--scaling weak` swaps the two.  For N > 1 the run ends with an invariance check: the all-reduced gradients and the
reduced heatmap grids of the N shards against one GPU processing the concatenated batch.

Prints ONE JSON line (rank 0).  `value` is measured with the batch already resident in HBM; `e2e` repeats the
measurement through the public API with HOST (pinned) inputs: host->device copies and the device->host read of the
loss sit inside the timed region.  `--impl reference` times the CPU reference implementation (the torch / C oracle,
all host threads) on a bounded sample of the same workload.

`--dump-outputs DIR` writes what the last timed step computed (the training step's predictions, losses, gradient and
updated parameters; the heatmap grids) as DIR/<name>.npy.  Every input is seeded, so two builds run with the same
arguments can be compared output for output.  Each timed training step starts from the same parameters and optimizer
state (TrainLeg.step_resident), so from run to run the predictions repeat and the losses, gradient and parameters differ
only by the summation order of fp32 atomics; the heatmap grids are exact.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

SEQ_LEN, HIDDEN, LAYERS, MAX_OBJECTS = 500, 128, 2, 10
TRAIN_BATCH = 8192                     # GLOBAL batch (BASELINE config 3); per GPU in the weak-scaling leg
HEATMAP_TRACES = 1_000_000             # in total (BASELINE config 2); per GPU in the weak-scaling leg
METRIC = "train traces/sec (seq500, H128) at 1/2/4/8 B200; heatmap Gpoints/s"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"], "tflops_sustained": d["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def gru_flops_per_trace(T=SEQ_LEN, H=HIDDEN, L=LAYERS, I=2):
    macs = sum(3 * H * (I if l == 0 else 2 * H) + 3 * H * H for l in range(L))
    fwd = 2.0 * 2 * T * macs
    dec = 2.0 * (2 * H * 256 + 256 * 256 + 256 * MAX_OBJECTS * 10)
    return 3.0 * (fwd + dec)           # fwd + dgrad + wgrad (SURVEY.md 8(d))


# ------------------------------------------------------------------------------------------------------------
# reference arm: the CPU oracle on the box's host cores
# ------------------------------------------------------------------------------------------------------------
def cpu_train_baseline(steps: int, warmup: int, sample_batch: int = 32, hidden: int = HIDDEN, seq_len: int = SEQ_LEN):
    from oracle.room_slam_ref import RoomSLAM as Ref
    from roomslam_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    model = Ref(hidden_size=hidden, num_layers=LAYERS, max_objects=MAX_OBJECTS, dropout=0.0).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-3)
    x, tgt = synth.make_sample(sample_batch, seq_len, MAX_OBJECTS, seed=0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        loss = model.compute_loss(model(x), tgt)["total"]
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    return {"value": sample_batch / sec, "unit": "traces/s", "cores": cores, "kind": "port",
            "sample": f"{sample_batch} traces x {seq_len} steps per step (H {hidden}), fp32 torch {torch.__version__} CPU oracle "
                      f"(fwd+loss+bwd+clip+AdamW), {steps} timed steps", "ms_per_step": sec * 1e3}


def cpu_heatmap_baseline(reps: int = 3, sample_traces: int = 40_000):
    import numpy as np
    from oracle import heatmap_ref_c
    from roomslam_b200 import synth
    cores = os.cpu_count() or 1
    pts = synth.make_traces(sample_traces, SEQ_LEN, seed=0).numpy()
    thr2 = np.float32((0.1 * 0.1) ** 2)
    heatmap_ref_c.bin_points(pts[:1000], 0, 0, 0.05, 200, 200, thr2)
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        heatmap_ref_c.bin_points(pts, 0, 0, 0.05, 200, 200, thr2, n_threads=0)
        best = min(best, time.perf_counter() - t0)
    return {"value": sample_traces * SEQ_LEN / best / 1e9, "unit": "Gpoints/s", "cores": cores, "kind": "port",
            "sample": f"{sample_traces} traces x {SEQ_LEN} points, C restatement (oracle/heatmap_ref.c), OpenMP all cores, "
                      f"best of {reps}"}


def run_reference(args):
    """The CPU reference arm: K timed + W warm-up steps of the oracle, each on a bounded sample (32 traces = BASELINE
    config 1) of the workload; `steps`, `warmup` and `ms_per_step` describe exactly what was timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    sample_batch = 32
    cb = cpu_train_baseline(args.steps, args.warmup, sample_batch)
    hb = cpu_heatmap_baseline()
    cfg = workload_config(args, precision="fp32", world=args.gpus)
    cfg["reference_sample"] = {"traces_per_step": sample_batch, "steps_timed": args.steps, "warmup_steps": args.warmup,
                               "note": "each step = one bounded sample of the workload (BASELINE config 1 batch), "
                                       "fwd+loss+bwd+clip+AdamW in fp32 on all host cores"}
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "traces/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": cb["value"], "unit": "traces/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "heatmap": {"value": hb["value"], "unit": "Gpoints/s", "cpu_baseline": hb,
                    "e2e": {"value": hb["value"], "unit": "Gpoints/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}},
        "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


def shard_sizes(args, world):
    """(train traces per GPU, heatmap traces per GPU) of the headline leg."""
    if args.scaling == "strong":
        if args.batch % world or args.heatmap_traces % world:
            raise SystemExit(f"--scaling strong: batch {args.batch} and heatmap traces {args.heatmap_traces} must divide by {world} GPUs")
        return args.batch // world, args.heatmap_traces // world
    return args.batch, args.heatmap_traces


def workload_config(args, precision, world):
    b_gpu, h_gpu = shard_sizes(args, world)
    return {"workload": f"RoomSLAM bi-GRU H={HIDDEN} L={LAYERS} seq_len={SEQ_LEN} N={MAX_OBJECTS}, fwd+loss+bwd+clip+AdamW, "
                        f"global batch {b_gpu * world} = {b_gpu}/GPU x {world} ({args.scaling} scaling); heatmap: "
                        f"{h_gpu * world} traces x {SEQ_LEN} points in total ({h_gpu}/GPU), 10 m x 10 m room, 0.05 m grid",
            "global_batch": b_gpu * world, "batch_per_gpu": b_gpu, "seq_len": SEQ_LEN, "hidden": HIDDEN, "layers": LAYERS,
            "precision": precision, "parallelism": f"dp{world}",
            "l2": "inputs larger than L2 (train activations are GBs per step; heatmap input >= 0.5 GB per GPU vs 126 MB L2)"}


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.dev = device_index
        self.proc, self.path = None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.dev)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.count(",") >= 8]
            sm = [float(r[1]) for r in rows]
            loaded = [s for s in sm if s > 0.5 * max(sm)] if sm else []
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = sorted({n for r in rows for n, v in zip(names, r[5:9]) if v.strip().lower().startswith("active")})
            out = {"sm_mhz": statistics.median(loaded) if loaded else None,
                   "sm_max_mhz": float(rows[0][2]) if rows else None, "reasons": reasons, "samples": len(rows),
                   "power_w_max": max(float(r[3]) for r in rows) if rows else None}
        except Exception as e:  # pragma: no cover
            out["error"] = str(e)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
def timed(fn, steps, warmup, dist_on):
    """W untimed + K timed calls of fn(); CUDA events, barrier + synchronize on both sides, max over ranks."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist_on:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda", dtype=torch.float64)
    if dist_on:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / steps


class TrainLeg:
    """One training configuration (model + flat buffers + optimizer + one synthetic batch resident on host and device)."""

    def __init__(self, batch, rank, world, precision, dropout=0.0, seed_base=0, hidden=HIDDEN, seq_len=SEQ_LEN):
        from roomslam_b200 import RoomSLAM, synth
        from roomslam_b200.train_utils import FlatParams, GradReducer, FusedAdamW, HostBatchPrefetcher
        torch.manual_seed(0)
        self.world, self.batch = world, batch
        self.model = RoomSLAM(hidden_size=hidden, num_layers=LAYERS, max_objects=MAX_OBJECTS, dropout=dropout,
                              precision=precision).cuda().train()
        self.flat = FlatParams(self.model)
        self.reducer = GradReducer(self.flat)
        self.opt = FusedAdamW(self.flat, lr=1e-3, max_grad_norm=1.0)
        self.start = self.flat.flat.clone()
        x_host, tgt_host = synth.make_sample(batch, seq_len, MAX_OBJECTS, seed=seed_base + rank)
        self.x_host = x_host.pin_memory()
        self.tgt_host = {k: v.pin_memory() for k, v in tgt_host.items()}
        self.x_dev = self.x_host.cuda()
        self.tgt_dev = {k: v.cuda() for k, v in self.tgt_host.items()}
        self.loss_host = torch.zeros(6).pin_memory()
        self.prefetch = HostBatchPrefetcher("cuda")
        self.h2d_bytes = self.x_host.numel() * 4 + sum(v.numel() * v.element_size() for v in self.tgt_host.values())
        self.keep_outputs = False          # True: self.last holds the predictions and losses of the latest step
        self.last = None

    def step(self, x, tgt):
        self.flat.zero_grad()
        self.reducer.prepare()
        pred = self.model(x)
        losses = self.model.compute_loss(pred, tgt)
        losses["total"].backward()
        self.reducer.finish()
        self.opt.step(grad_scale=1.0 / self.world)
        if self.keep_outputs:
            self.last = {"pred": {k: v.detach() for k, v in pred.items()}, "loss": {k: v.detach() for k, v in losses.items()}}
        return losses["total"]

    def step_resident(self):
        # Every resident step starts from the initial parameters and optimizer state: it runs a training step's kernels on
        # the same shapes, and what it computes depends on the seeded inputs alone.  Chained steps would not be reproducible:
        # the weight gradients end in fp32 atomic sums, and a few steps later the bf16 forward pass has turned that
        # summation-order noise in the parameters into visibly different predictions.
        self.flat.flat.copy_(self.start)
        self.opt.m.zero_()
        self.opt.v.zero_()
        self.opt.t = 0
        self.step(self.x_dev, self.tgt_dev)

    def step_e2e(self):
        # public-API training loop: every step copies ITS batch from pinned host memory (one copy per step, started while
        # the previous step computes) and reads its loss back to the host
        if not self.prefetch.has_pending:
            self.prefetch.submit(self.x_host, self.tgt_host)
        x, tgt = self.prefetch.get()
        self.prefetch.submit(self.x_host, self.tgt_host)                            # next step's batch: overlaps this step
        loss = self.step(x, tgt)
        self.loss_host[0:1].copy_(loss.detach().reshape(1), non_blocking=True)      # device -> host read of the loss (pinned)

    def free(self):
        if self.prefetch.has_pending:
            self.prefetch.get()
        del self.x_dev, self.tgt_dev
        torch.cuda.empty_cache()


def invariance_check(world, rank):
    """SURVEY.md 4(v) on the hardware: N shards + all-reduce against ONE GPU processing the concatenated batch.
    Gradients: every trace has the same number of valid slots, so the global masked-mean loss is exactly the mean of the
    shard losses and  sum_r grad_r / N  must equal the single-GPU gradient up to fp32 summation order.
    Heatmap: the int32 sum of the shard grids must equal the grid of all points binned by one GPU, bit for bit."""
    import torch.distributed as dist
    from roomslam_b200 import RoomSLAM, OccupancyHeatmapBaseline, synth
    from roomslam_b200.train_utils import FlatParams
    out = {}
    # Both sides run the default kernels: from 1024 traces per rank up (8192 / N for N <= 8) the shards and the concatenated
    # batch take the same path (unsplit weights, input projection of layer 1 fused into the recurrence kernel).
    for precision, per_rank, tol in (("fp32", 64, 1e-5), ("bf16", TRAIN_BATCH // world, 1e-4)):
        G = per_rank * world
        x, tgt = synth.make_sample(G, SEQ_LEN, MAX_OBJECTS, seed=4242)
        tgt["valid"] = torch.zeros_like(tgt["valid"])
        tgt["valid"][:, :5] = 1
        torch.manual_seed(0)
        model = RoomSLAM(hidden_size=HIDDEN, num_layers=LAYERS, max_objects=MAX_OBJECTS, dropout=0.0, precision=precision).cuda().train()
        flat = FlatParams(model)

        def grads(lo, hi):
            flat.zero_grad()
            loss = model.compute_loss(model(x[lo:hi].cuda()), {k: v[lo:hi].cuda() for k, v in tgt.items()})["total"]
            loss.backward()
            return flat.grad.clone()
        g = grads(rank * per_rank, (rank + 1) * per_rank)
        dist.all_reduce(g, op=dist.ReduceOp.SUM)
        g /= world
        if rank == 0:
            g1 = grads(0, G)
            err = float((g.double() - g1.double()).norm() / g1.double().norm().clamp_min(1e-30))
            out[f"grad_rel_l2_{precision}"] = err
            out[f"grad_ok_{precision}"] = bool(err <= tol)
            out[f"grad_tol_{precision}"] = tol
            out[f"grad_global_batch_{precision}"] = G
        del model, flat, g
        torch.cuda.empty_cache()
    # heatmap: HEATMAP_TRACES in total, shard r = traces [r n, (r+1) n)
    hm = OccupancyHeatmapBaseline()
    n = HEATMAP_TRACES // world
    pts = synth.make_traces(n, SEQ_LEN, seed=7000 + rank, device="cuda")
    occ, stat, dropped = hm.bin(pts)
    both = torch.cat([occ.reshape(-1), stat.reshape(-1), torch.tensor([dropped], device="cuda", dtype=torch.int64).to(torch.int32)])
    dist.all_reduce(both, op=dist.ReduceOp.SUM)
    allpts = torch.empty(world * n, SEQ_LEN, 2, device="cuda") if rank == 0 else None
    dist.gather(pts, list(allpts.view(world, n, SEQ_LEN, 2).unbind(0)) if rank == 0 else None, dst=0)
    if rank == 0:
        o1, s1, d1 = hm.bin(allpts)
        one = torch.cat([o1.reshape(-1), s1.reshape(-1), torch.tensor([d1], device="cuda", dtype=torch.int32)])
        out["heatmap_bit_identical"] = bool(torch.equal(one, both))
        out["heatmap_traces"] = world * n
        out["invariance"] = bool(out["heatmap_bit_identical"] and out["grad_ok_fp32"] and out["grad_ok_bf16"])
    return out


DUMP_MAX_BYTES = 64 << 20
DUMP_TRACES = 65536                    # per-trace outputs of a larger batch: a fixed, seeded sample of this many traces


def train_outputs(leg):
    """What the last timed training step computed, as float32 arrays: the predictions and losses its caller receives,
    the gradient it produced and the parameters after its optimizer update."""
    import numpy as np
    rows = None
    if leg.batch > DUMP_TRACES:
        rows = torch.from_numpy(np.sort(np.random.default_rng(0).choice(leg.batch, DUMP_TRACES, replace=False))).cuda()
    out = {f"train_{k}": v if rows is None else v[rows] for k, v in leg.last["pred"].items()}
    out.update({f"train_loss_{k}": v for k, v in leg.last["loss"].items()})
    out["train_grad"] = leg.flat.grad
    out["train_params"] = leg.flat.flat
    return {k: v.float().cpu().numpy() for k, v in out.items()}


def write_outputs(path, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def run_ours(args):
    import torch.distributed as dist
    from roomslam_b200 import OccupancyHeatmapBaseline, synth, _lib
    from roomslam_b200 import functional as F_

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: roomslam_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dist_on = world > 1
    if dist_on:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if world != args.gpus and rank == 0:
        print(f"[bench] note: --gpus {args.gpus} but WORLD_SIZE={world}; using {world}", file=sys.stderr)
    args.gpus = world
    pk = peaks()
    lib = _lib.load()
    precision = "bf16" if args.precision == "auto" else args.precision
    B, n_tr = shard_sizes(args, world)                     # per GPU, headline leg
    other = "weak" if args.scaling == "strong" else "strong"

    # ---- training step: headline leg -----------------------------------------------------------------------
    leg = TrainLeg(B, rank, world, precision)
    dump = {} if args.dump_outputs and rank == 0 else None
    leg.keep_outputs = dump is not None
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.rs_launch_count()
    ms_train = timed(leg.step_resident, args.steps, args.warmup, dist_on)
    launches_train = (lib.rs_launch_count() - n0) // (args.steps + args.warmup) * args.steps
    if dump is not None:
        dump.update(train_outputs(leg))
        leg.keep_outputs, leg.last = False, None
    ms_train_e2e = timed(leg.step_e2e, args.steps, max(1, args.warmup // 2), dist_on)
    h2d_train = leg.h2d_bytes
    final_loss = float(leg.loss_host[0])
    # per-kernel timing of one extra step (CUDA events on the launch stream) for the roofline object
    F_.enable_kernel_timing(True)
    leg.step_resident()
    torch.cuda.synchronize()
    kernel_ms = F_.collect_kernel_timing()
    F_.enable_kernel_timing(False)
    leg.free()
    del leg

    # ---- the other scaling mode (N > 1 only; at N = 1 the two coincide) ---------------------------------------
    other_leg = None
    if dist_on:
        args_o = argparse.Namespace(**{**vars(args), "scaling": other})
        B_o, n_tr_o = shard_sizes(args_o, world)
        leg_o = TrainLeg(B_o, rank, world, precision)
        ms_o = timed(leg_o.step_resident, args.steps, args.warmup, dist_on)
        ms_o_e2e = timed(leg_o.step_e2e, args.steps, 2, dist_on)
        leg_o.free()
        del leg_o
        other_leg = {"scaling": other, "global_batch": B_o * world, "batch_per_gpu": B_o, "value": B_o * world / (ms_o / 1e3),
                     "unit": "traces/s", "ms_per_step": ms_o, "e2e_value": B_o * world / (ms_o_e2e / 1e3)}

    # ---- single-GPU extras: BASELINE config 1 on the GPU (same config as the CPU arm), dropout = 0.1 ---------------
    c1 = drop = None
    if not dist_on:
        c1_leg = TrainLeg(32, 0, 1, "fp32")
        ms_c1 = timed(c1_leg.step_resident, args.steps, 3, False)
        c1_leg.free()
        del c1_leg
        c1 = {"workload": "BASELINE config 1: batch 32 x 500 steps, fp32 kernels (1e-4 parity mode), fwd+loss+bwd+clip+AdamW",
              "value": 32 / (ms_c1 / 1e3), "unit": "traces/s", "ms_per_step": ms_c1, "precision": "fp32", "batch": 32}
        d_leg = TrainLeg(B, 0, 1, precision, dropout=0.1)
        ms_d = timed(d_leg.step_resident, args.steps, 3, False)
        d_leg.free()
        del d_leg
        drop = {"workload": "same step with the README's inter-layer dropout p = 0.1 (bit mask drawn on the device, applied inside "
                            "the recurrence kernels)", "value": B / (ms_d / 1e3), "unit": "traces/s", "ms_per_step": ms_d,
                "slowdown_vs_p0": ms_d / ms_train - 1.0}

    # ---- single-GPU extra: BASELINE config 4 (long-trace variant: H 256, T 4000, batch 1024) on the tensor-core path ----------
    c4 = None
    if not dist_on and not args.skip_c4:
        c4_leg = TrainLeg(1024, 0, 1, "bf16", hidden=256, seq_len=4000)
        ms_c4 = timed(c4_leg.step_resident, args.steps, 2, False)
        F_.enable_kernel_timing(True)
        c4_leg.step_resident()
        torch.cuda.synchronize()
        c4_kernels = F_.collect_kernel_timing()
        F_.enable_kernel_timing(False)
        c4_leg.free()
        del c4_leg
        c4_flops = gru_flops_per_trace(T=4000, H=256)
        c4 = {"workload": "BASELINE config 4: bi-GRU H=256 L=2 seq_len=4000, batch 1024, bf16, fwd+loss+bwd+clip+AdamW "
                          "(W_hh streamed from L2 by the recurrence kernels, csrc/rec_wide.cu)",
              "value": 1024 / (ms_c4 / 1e3), "unit": "traces/s", "ms_per_step": ms_c4, "steps": args.steps, "warmup": 2,
              "algorithmic_gflop_per_trace": c4_flops / 1e9, "flop_bound_ms": c4_flops * 1024 / (pk["tflops_sustained"] * 1e12) * 1e3,
              "frac_of_flop_bound": c4_flops * 1024 / (pk["tflops_sustained"] * 1e12) * 1e3 / ms_c4,
              "kernel_ms": {k: v[0] for k, v in c4_kernels.items()}}

    # ---- heatmap -------------------------------------------------------------------------------------------
    hm = OccupancyHeatmapBaseline()
    pts = synth.make_traces(n_tr, SEQ_LEN, seed=1000 + rank, device="cuda")
    occ = torch.empty(hm.gy, hm.gx, dtype=torch.int32, device="cuda")
    stat = torch.empty_like(occ)
    dropped = torch.empty(1, dtype=torch.int64, device="cuda")
    packed = torch.empty(2 * hm.gx * hm.gy, dtype=torch.int32, device="cuda")

    def heat_resident():
        hm.bin_into(pts, occ, stat, dropped)
        if dist_on:       # sharded per trace: exact int32 sum of the two grids
            packed[: hm.gx * hm.gy].copy_(occ.reshape(-1))
            packed[hm.gx * hm.gy:].copy_(stat.reshape(-1))
            dist.all_reduce(packed, op=dist.ReduceOp.SUM)

    n1 = lib.rs_launch_count()
    ms_heat = timed(heat_resident, args.steps, args.warmup, dist_on)
    launches_heat = (lib.rs_launch_count() - n1) // (args.steps + args.warmup) * args.steps
    if dump is not None:              # int32 counts: float64 holds every value exactly
        grids = packed.view(2, hm.gy, hm.gx) if dist_on else torch.stack([occ, stat])
        dump["heatmap_occupancy"] = grids[0].double().cpu().numpy()
        dump["heatmap_stationary"] = grids[1].double().cpu().numpy()
        dump["heatmap_dropped"] = dropped.double().cpu().numpy()
    # the binning kernel alone (events around the single launch, same stream)
    ms_kernel = timed(lambda: hm.bin_into(pts, occ, stat, dropped), args.steps, 1, False)
    conserved = int(occ.sum().item()) + int(dropped.item()) == n_tr * SEQ_LEN
    pts_host = torch.empty(n_tr, SEQ_LEN, 2, dtype=torch.float32).pin_memory()
    pts_host.copy_(pts)
    del pts
    torch.cuda.empty_cache()

    def heat_e2e():
        o, s, _ = hm.bin(pts_host)               # CPU tensor in -> rs_heatmap_bin_host -> CPU tensors out
        if dist_on:
            both = torch.cat([o.reshape(-1), s.reshape(-1)]).cuda()
            dist.all_reduce(both, op=dist.ReduceOp.SUM)
            both.cpu()

    ms_heat_e2e = timed(heat_e2e, args.steps, 1, dist_on)
    del pts_host
    heat_other = None
    if dist_on:
        pts_o = synth.make_traces(n_tr_o, SEQ_LEN, seed=2000 + rank, device="cuda")
        ms_ho = timed(lambda: (hm.bin_into(pts_o, occ, stat, dropped), packed[: hm.gx * hm.gy].copy_(occ.reshape(-1)),
                               packed[hm.gx * hm.gy:].copy_(stat.reshape(-1)), dist.all_reduce(packed, op=dist.ReduceOp.SUM)),
                      args.steps, args.warmup, True)
        heat_other = {"scaling": other, "traces_per_gpu": n_tr_o, "value": n_tr_o * SEQ_LEN * world / (ms_ho / 1e3) / 1e9,
                      "unit": "Gpoints/s", "ms_per_step": ms_ho}
        del pts_o
        torch.cuda.empty_cache()
    clocks = sampler.stop() if rank == 0 else None
    inv = invariance_check(world, rank) if dist_on else None

    if rank == 0:
        traces_s = B * world / (ms_train / 1e3)
        flops = gru_flops_per_trace()
        traffic = load_traffic()
        line = {
            "metric": METRIC, "value": traces_s, "unit": "traces/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_train, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(args, precision, world),
            "e2e": {"value": B * world / (ms_train_e2e / 1e3), "unit": "traces/s", "h2d_bytes_per_step": h2d_train,
                    "d2h_bytes_per_step": 4, "ms_per_step": ms_train_e2e},
            "gpu_launches": int(launches_train + launches_heat),
            "clocks": clocks, "final_loss": final_loss,
            "train": {"algorithmic_gflop_per_trace": flops / 1e9,
                      "achieved_tflops_per_gpu": flops * B / (ms_train / 1e3) / 1e12,
                      "frac_of_sustained_bf16_peak": flops * B / (ms_train / 1e3) / 1e12 / pk["tflops_sustained"],
                      "kernel_ms": kernel_ms},
            "heatmap": {
                "value": n_tr * SEQ_LEN * world / (ms_heat / 1e3) / 1e9, "unit": "Gpoints/s", "ms_per_step": ms_heat,
                "points_per_gpu": n_tr * SEQ_LEN, "conservation_check": bool(conserved),
                "e2e": {"value": n_tr * SEQ_LEN * world / (ms_heat_e2e / 1e3) / 1e9, "unit": "Gpoints/s",
                        "h2d_bytes_per_step": n_tr * SEQ_LEN * 8, "d2h_bytes_per_step": 2 * hm.gx * hm.gy * 4 + 8,
                        "ms_per_step": ms_heat_e2e},
                "roofline": {"bound": "hbm", "achieved": n_tr * SEQ_LEN * 8 / (ms_kernel / 1e3) / 1e9, "peak": pk["hbm_gbs"],
                             "unit": "GB/s", "frac": n_tr * SEQ_LEN * 8 / (ms_kernel / 1e3) / 1e9 / pk["hbm_gbs"],
                             "traffic": (int(traffic["heatmap_bytes_per_point"] * n_tr * SEQ_LEN)
                                         if traffic and "heatmap_bytes_per_point" in traffic else None),
                             "traffic_source": traffic.get("source") if traffic else None,
                             "kernel": "heatmap_tma_kernel", "kernel_ms": ms_kernel,
                             "algorithmic_bytes_per_point": 8, "algorithmic_bytes": 8 * n_tr * SEQ_LEN,
                             "peak_source": pk["source"] + ", burst (kernel timed alone)"},
            },
        }
        line["roofline"] = train_roofline(kernel_ms, B, pk, precision, traffic) or line["heatmap"]["roofline"]
        if other_leg is not None:
            line[other] = other_leg
            line["heatmap"][other] = heat_other
        if inv is not None:
            line["invariance"] = inv.pop("invariance")
            line["invariance_detail"] = inv
        if c1 is not None:
            line["c1"] = c1
            line["dropout"] = drop
        if c4 is not None:
            line["c4"] = c4
            cb4 = cpu_train_baseline(1, 0, sample_batch=8, hidden=256, seq_len=4000)
            line["c4"]["cpu_baseline"] = {k: cb4[k] for k in ("value", "unit", "cores", "kind", "sample")}
        if world == 1:
            cb = cpu_train_baseline(2, 1)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            line["c1"]["cpu_same_config"] = {"value": cb["value"], "unit": "traces/s", "ratio": line["c1"]["value"] / cb["value"]}
            line["heatmap"]["cpu_baseline"] = cpu_heatmap_baseline()
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if dist_on:
        dist.barrier()
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------
# --suite next: the SURVEY.md 8(f) rows (preprocessing, shipped BiLSTM model, Hungarian set loss, evaluation), each
# timed on the GPU with the CPU oracle beside it.  One JSON line per row; not part of the default run.
# ------------------------------------------------------------------------------------------------------------
def _time_gpu(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def _time_cpu(fn, reps=1):
    fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps


def run_next_rows(args):
    import numpy as np
    from roomslam_b200 import _lib, preprocess
    from roomslam_b200.evaluation import MetricAccumulator, mean_average_precision, nms_batch
    from roomslam_b200.lstm_model import TraceToColliderLSTM
    from roomslam_b200.set_loss import SetCriterion
    from oracle import eval_ref, features_ref, set_loss_ref
    from oracle.lstm_ref import TraceToColliderLSTMRef
    _lib.load()
    torch.cuda.set_device(0)
    pk = peaks()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    W = {"class_loss": 2.0, "l1_loss": 5.0, "giou_loss": 2.0}

    # ---- row 1: trace preprocessing, 4096 traces x 3000 points ----
    B, N = 4096, 3000
    pts = torch.randn(B, N, 4, generator=g)
    pts[..., 3] = torch.cumsum(torch.rand(B, N, generator=g) * 0.1 + 1e-3, 1)
    flat, off = pts.reshape(-1, 4).cuda(), torch.arange(B + 1, dtype=torch.int64) * N
    dev_off = off.cuda()
    feats = torch.empty(B, N, 11, device="cuda"); mask = torch.empty(B, N, dtype=torch.uint8, device="cuda")
    lens = torch.empty(B, dtype=torch.int64, device="cuda"); flag = torch.empty(1, dtype=torch.int32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    ms_k = _time_gpu(lambda: _lib.call("rs_trace_features", flat.data_ptr(), dev_off.data_ptr(), B, 3000, N, feats.data_ptr(),
                                       mask.data_ptr(), lens.data_ptr(), flag.data_ptr(), st), args.steps * 4, 3)
    ms_api = _time_gpu(lambda: preprocess.trace_features(flat, off, max_len=3000), args.steps, 3)
    sample = [pts[b].numpy() for b in range(64)]
    t_cpu = _time_cpu(lambda: [features_ref.process_points(p) for p in sample])
    gbs = B * N * 61 / ms_k / 1e6
    print(json.dumps({"row": "8(f)1 trace preprocessing", "metric": "Gpoints/s", "value": round(B * N / ms_k / 1e6, 2),
                      "value_api": round(B * N / ms_api / 1e6, 2), "ms_kernel": round(ms_k, 4), "dtype": "f32",
                      "config": {"workload": f"{B} traces x {N} points -> (B, 3000, 11) features + mask"},
                      "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                                   "frac": round(gbs / pk["hbm_gbs"], 3), "traffic": None, "bytes_per_point": 61},
                      "cpu_baseline": {"value": round(64 * N / t_cpu / 1e9, 5), "unit": "Gpoints/s", "cores": 1, "kind": "port",
                                       "sample": "64 traces x 3000 points, numpy oracle"}}), flush=True)

    # ---- row 2 + 3: shipped BiLSTM model + Hungarian set loss, forward + backward ----
    for B in (20, 256):
        N, Q, M = 3000, 30, 50
        model = TraceToColliderLSTM(128, Q).cuda().train()
        model.encoder.dropout = 0.0
        x = torch.randn(B, N, 11, generator=g).cuda()
        tmask = torch.ones(B, N, dtype=torch.bool, device="cuda")
        tg = {"boxes": torch.cat([torch.randn(B, M, 3, generator=g), torch.rand(B, M, 3, generator=g) + 0.2], -1).cuda(),
              "labels": torch.randint(0, 4, (B, M), generator=g).cuda(), "valid_mask": (torch.rand(B, M, generator=g) < 0.3).cuda()}
        crit = SetCriterion(W)

        def step():
            model.zero_grad(set_to_none=True)
            crit(model(x, tmask), tg)["total_loss"].backward()
        ms = _time_gpu(step, args.steps, 3)
        line = {"row": "8(f)2+3 BiLSTM query-decoder model + Hungarian set loss, fwd+bwd", "metric": "train traces/s",
                "value": round(B / ms * 1e3, 1), "ms_per_step": round(ms, 2), "dtype": "f32",
                "config": {"workload": f"batch {B} x {N} points, d_model 128, 30 queries, 50 collider slots"}}
        if B == 20:
            ref = TraceToColliderLSTMRef(128, Q).train()
            ref.encoder.lstm.dropout = 0.0
            xc, mc = x[:4].cpu(), tmask[:4].cpu()
            tc = {k: v[:4].cpu() for k, v in tg.items()}

            def cpu_step():
                ref.zero_grad()
                set_loss_ref.set_loss(ref(xc, mc), tc)[0]["total_loss"].backward()
            t_cpu = _time_cpu(cpu_step)
            line["cpu_baseline"] = {"value": round(4 / t_cpu, 2), "unit": "train traces/s", "cores": cores, "kind": "port",
                                    "sample": "batch 4 x 3000 points, torch CPU oracle + scipy matcher"}
        print(json.dumps(line), flush=True)

    # ---- row 3 alone and row 4: 4096 scenes ----
    B, Q, M = 4096, 30, 50
    gt = torch.cat([torch.randn(B, M, 3, generator=g) * 3, torch.rand(B, M, 3, generator=g) * 2 + 0.3], -1)
    valid = torch.rand(B, M, generator=g) < 0.4
    labels = torch.randint(0, 4, (B, M), generator=g)
    boxes = gt[:, :Q] + torch.randn(B, Q, 6, generator=g) * 0.12
    boxes[..., 3:] = boxes[..., 3:].clamp_min(0.05)
    logits = torch.randn(B, Q, 4, generator=g) * 2
    cb, cl = boxes.cuda().requires_grad_(True), logits.cuda().requires_grad_(True)
    tg = {"boxes": gt.cuda(), "labels": labels.cuda(), "valid_mask": valid.cuda()}
    crit = SetCriterion(W)

    def loss_step():
        cb.grad = None; cl.grad = None
        crit({"pred_boxes": cb, "pred_classes": cl}, tg)["total_loss"].backward()
    ms = _time_gpu(loss_step, args.steps * 4, 3)
    S = 256
    bs, ls = boxes[:S].clone().requires_grad_(True), logits[:S].clone().requires_grad_(True)
    ts = {"boxes": gt[:S], "labels": labels[:S], "valid_mask": valid[:S]}
    t_cpu = _time_cpu(lambda: set_loss_ref.set_loss({"pred_boxes": bs, "pred_classes": ls}, ts)[0]["total_loss"].backward())
    print(json.dumps({"row": "8(f)3 Hungarian matcher + set loss, fwd+bwd", "metric": "scenes/s", "value": round(B / ms * 1e3, 0),
                      "ms_per_step": round(ms, 3), "dtype": "f32 cost / f64 solver",
                      "config": {"workload": f"{B} scenes x {Q} queries x {M} collider slots (40% valid)"},
                      "cpu_baseline": {"value": round(S / t_cpu, 0), "unit": "scenes/s", "cores": cores, "kind": "port",
                                       "sample": f"{S} scenes, torch CPU + scipy.optimize.linear_sum_assignment"}}), flush=True)

    def eval_step():
        acc = MetricAccumulator("cuda")
        acc.update({"pred_boxes": cb, "pred_classes": cl}, tg)
        nms_batch(cb, cl)
        return acc.compute(), mean_average_precision(cb, cl, tg["boxes"], tg["labels"], tg["valid_mask"])[0]
    ms = _time_gpu(eval_step, args.steps, 3)
    S = 64
    o = {"pred_boxes": boxes[:S], "pred_classes": logits[:S]}
    ts = {"boxes": gt[:S], "labels": labels[:S], "valid_mask": valid[:S]}

    def cpu_eval():
        eval_ref.metrics_from_counts(eval_ref.batch_counts(o, ts))
        for b in range(S):
            eval_ref.nms_order(boxes[b], logits[b])
        eval_ref.mean_average_precision(boxes[:S], logits[:S], gt[:S], labels[:S], valid[:S])
    t_cpu = _time_cpu(cpu_eval)
    # ---- BASELINE config 5: batched inference + IoU / mAP evaluation of the GRU model, 262144 traces x 500 steps ----
    from roomslam_b200 import RoomSLAM, synth
    from roomslam_b200.evaluation import SlotEvaluator
    n5 = 262144
    model5 = RoomSLAM(precision="bf16").cuda().eval()
    x5, t5 = synth.make_sample(n5, SEQ_LEN, MAX_OBJECTS, seed=0, device="cuda")

    def c5_step():
        ev = SlotEvaluator(4, 0.5)
        with torch.no_grad():
            for s0 in range(0, n5, 16384):
                ev.update(model5(x5[s0:s0 + 16384]), {k: v[s0:s0 + 16384] for k, v in t5.items()})
        return ev.compute()
    ms5 = _time_gpu(c5_step, max(1, args.steps // 2), 1)
    print(json.dumps({"row": "BASELINE config 5: batched GRU inference + IoU / mAP evaluation (incl. the host read of the metrics)",
                      "metric": "traces/s", "value": round(n5 / ms5 * 1e3, 0), "ms_per_step": round(ms5, 2), "dtype": "bf16",
                      "config": {"workload": f"{n5} traces x {SEQ_LEN} steps, H 128, 2 layers, 10 slots; chunks of 16384"}}), flush=True)
    del x5, t5, model5

    print(json.dumps({"row": "8(f)4 evaluation: matched metrics + NMS + mAP (incl. the host read of the results)",
                      "metric": "scenes/s", "value": round(B / ms * 1e3, 0), "ms_per_step": round(ms, 3), "dtype": "f32",
                      "config": {"workload": f"{B} scenes x {Q} queries x {M} collider slots"},
                      "cpu_baseline": {"value": round(S / t_cpu, 1), "unit": "scenes/s", "cores": 1, "kind": "port",
                                       "sample": f"{S} scenes, python/numpy oracle"}}), flush=True)



def load_traffic():
    """DRAM bytes per launch from the round's committed `ncu --set full` captures (profiles/r2_traffic.json, stamped
    with the commit they were taken at): {"commit", "source", "batch_per_gpu", "kernels": {name: bytes}, "heatmap_bytes_per_point"}."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    try:
        return json.load(open(path))
    except Exception:
        return None


def train_roofline(kernel_ms, B, pk, precision, traffic):
    """Roofline object for the kernel with the largest share of the training step."""
    if not kernel_ms:
        return None
    name, (ms, calls, flops) = max(kernel_ms.items(), key=lambda kv: kv[1][0])
    if flops <= 0 or ms <= 0:
        return None
    ach = flops / (ms / 1e3) / 1e12
    out = {"bound": "tensor", "achieved": ach, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
           "frac": ach / pk["tflops_sustained"], "traffic": None, "kernel": name, "kernel_ms": ms, "launches": calls,
           "algorithmic_flops": flops,
           "note": "dominant kernel of the training step by CUDA-event time; the tensor figure is the algorithmic-FLOP view "
                   "SURVEY.md 8(d) asks for. Its achieved HBM bandwidth over the measured DRAM bytes is in hbm_view",
           "peak_source": pk["source"] + ", sustained (kernel timed inside a long step)"}
    per_launch = (traffic or {}).get("kernels", {}).get(name)
    if precision == "bf16" and traffic and B == traffic.get("batch_per_gpu") and per_launch:
        gbs = per_launch / (ms / calls / 1e3) / 1e9
        out["traffic"] = per_launch
        out["hbm_view"] = {"bytes_per_launch": per_launch, "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                           "frac": gbs / pk["hbm_gbs"], "source": traffic.get("source"), "commit": traffic.get("commit")}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="auto", choices=["auto", "bf16", "fp32"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default, BASELINE config 3): --batch / --heatmap-traces are GLOBAL and split over the GPUs; "
                         "weak: they are per GPU.  The other mode is measured too and reported under its name")
    ap.add_argument("--batch", type=int, default=TRAIN_BATCH, help="traces (global for strong scaling, per GPU for weak)")
    ap.add_argument("--heatmap-traces", type=int, default=HEATMAP_TRACES, help="traces (global / per GPU, as --batch)")
    ap.add_argument("--skip-c4", action="store_true", help="skip the BASELINE config 4 leg (H 256, T 4000; ~63 GB of HBM)")
    ap.add_argument("--suite", default="headline", choices=["headline", "next"],
                    help="'next': one JSON line per SURVEY.md 8(f) row instead of the headline line (single GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed training step and heatmap pass computed to DIR/<name>.npy (rank 0's "
                         "shard; float32, float64 for the heatmap counts; at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.suite != "headline"):
        ap.error("--dump-outputs applies to the GPU headline run (--impl ours --suite headline)")
    # Native libraries write banners to file descriptor 1 (NCCL prints its version at the first communicator init).
    # The contract is ONE JSON line on stdout: keep Python's stdout on the real descriptor and point fd 1 at stderr.
    sys.stdout.flush()
    sys.stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.suite == "next":
        return run_next_rows(args)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
