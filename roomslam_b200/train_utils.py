"""Training plumbing around the kernels: flat parameter / gradient buffers, bucketed gradient all-reduce
overlapped with backward (NCCL over NVLink), and the fused AdamW step.

Mirrors what the upstream loop does around the model (src/benchmark/train.py:218-221: zero_grad, backward,
clip_grad_norm_(1.0), optimizer.step with AdamW :440-444), for one process per GPU.
"""
from __future__ import annotations

import os
import re
from typing import List, Optional

import torch
import torch.distributed as dist
import torch.nn as nn

from . import _lib


def seed_everything(seed: int) -> None:
    """Seeds Python, numpy and torch (host and every GPU) and turns on torch.use_deterministic_algorithms, which the
    library follows with fixed-order split reductions: a rerun with the same seed, data and GPU model gives the same bits."""
    import random

    import numpy as np
    os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")     # torch's condition for deterministic cuBLAS calls
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.use_deterministic_algorithms(True)


class FlatParams:
    """Re-homes every parameter of `model` into ONE contiguous fp32 buffer (parameters become views) and gives
    each a persistent .grad view into ONE flat gradient buffer.  state_dict()/load_state_dict() keep working
    (they copy through the views).  Gradients are ordered so that the parameters whose gradients become final
    first in backward (decoder, then the top GRU layer ... then layer 0) form contiguous buckets."""

    def __init__(self, model: nn.Module, bucket_of=None):
        params = [p for p in model.parameters() if p.requires_grad]
        names = {id(p): n for n, p in model.named_parameters()}
        bucket_of = bucket_of or default_bucket
        order = sorted(range(len(params)), key=lambda i: (bucket_of(names[id(params[i])]), i))
        self.params = [params[i] for i in order]
        self.names = [names[id(p)] for p in self.params]
        self.buckets_idx = [bucket_of(n) for n in self.names]
        dev = self.params[0].device
        n = sum(p.numel() for p in self.params)
        self.flat = torch.empty(n, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(n, device=dev, dtype=torch.float32)
        self.offsets = []
        off = 0
        with torch.no_grad():
            for p in self.params:
                k = p.numel()
                self.flat[off:off + k].copy_(p.detach().reshape(-1))
                p.data = self.flat[off:off + k].view_as(p)
                p.grad = self.grad[off:off + k].view_as(p)
                self.offsets.append(off)
                off += k
        self.numel = n
        # bucket ranges in the flat buffer
        self.bucket_ranges = []
        start = 0
        for i in range(1, len(self.params) + 1):
            if i == len(self.params) or self.buckets_idx[i] != self.buckets_idx[start]:
                lo = self.offsets[start]
                hi = self.offsets[i - 1] + self.params[i - 1].numel()
                self.bucket_ranges.append((self.buckets_idx[start], lo, hi, list(range(start, i))))
                start = i

    def zero_grad(self):
        self.grad.zero_()
        for p, off in zip(self.params, self.offsets):       # re-attach in case something replaced .grad
            if p.grad is None or p.grad.data_ptr() != self.grad.data_ptr() + 4 * off:
                p.grad = self.grad[off:off + p.numel()].view_as(p)


def default_bucket(name: str) -> int:
    """Backward order of RoomSLAM: decoder first, then GRU layers from the top down."""
    if name.startswith("decoder."):
        return 0
    if name.startswith("encoder."):
        m = re.search(r"_l(\d+)", name)
        if m:
            return 1000 - int(m.group(1))          # higher layers earlier
        # the BiLSTM pipeline's encoder (lstm_model.py): out_proj is the last module of the forward pass, so its gradient
        # is final first; input_proj feeds layer 0 and finishes last
        return 500 if "out_proj" in name else 1500
    return 2000


class GradReducer:
    """Data-parallel gradient all-reduce (sum) of the flat gradient buffer, one NCCL call per bucket, launched on a
    side stream from a post-accumulate-grad hook as soon as the last gradient of the bucket has been written, so
    the reduce of (decoder + top layer) overlaps the backward-through-time of the layers below."""

    def __init__(self, flat: FlatParams, group=None, merge_small: bool = True):
        self.flat, self.group = flat, group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.stream = torch.cuda.Stream() if flat.flat.is_cuda else None
        ranges = flat.bucket_ranges
        if merge_small and len(ranges) > 2:      # decoder + all layers but the lowest in one bucket, layer 0 alone
            first = (ranges[0][0], ranges[0][1], ranges[-2][2], sum((r[3] for r in ranges[:-1]), []))
            ranges = [first, ranges[-1]]
        self.ranges = ranges
        self.pending = [0] * len(ranges)
        self.bucket_of_param = {}
        for b, (_, lo, hi, idxs) in enumerate(ranges):
            for i in idxs:
                self.bucket_of_param[i] = b
        self.launched: List[bool] = [False] * len(ranges)
        self.handles = []
        if self.world > 1:
            for i, p in enumerate(flat.params):
                p.register_post_accumulate_grad_hook(self._make_hook(i))

    def _make_hook(self, i):
        def hook(_p):
            b = self.bucket_of_param[i]
            self.pending[b] -= 1
            if self.pending[b] == 0:
                self._launch(b)
        return hook

    def _launch(self, b):
        _, lo, hi, _ = self.ranges[b]
        self.launched[b] = True
        if self.stream is not None:
            self.stream.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(self.stream):
                dist.all_reduce(self.flat.grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group)
        else:   # gloo / CPU tests
            dist.all_reduce(self.flat.grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group)

    def prepare(self):
        """Call before backward()."""
        for b, (_, _, _, idxs) in enumerate(self.ranges):
            self.pending[b] = len(idxs)
            self.launched[b] = False

    def finish(self):
        """Call after backward(): launches anything whose hooks did not all fire, then joins the side stream."""
        if self.world > 1:
            for b in range(len(self.ranges)):
                if not self.launched[b]:
                    self._launch(b)
            if self.stream is not None:
                torch.cuda.current_stream().wait_stream(self.stream)


class FusedAdamW:
    """AdamW + global-norm clipping in one pass over the flat buffers (csrc/optim.cu)."""

    def __init__(self, flat: FlatParams, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, max_grad_norm=1.0):
        self.flat, self.lr, self.betas, self.eps, self.wd, self.max_norm = flat, lr, betas, eps, weight_decay, max_grad_norm
        self.m = torch.zeros_like(flat.flat)
        self.v = torch.zeros_like(flat.flat)
        self.scratch = torch.zeros(1, dtype=torch.float64, device=flat.flat.device)
        self.t = 0

    def step(self, grad_scale: float = 1.0):
        if not self.flat.flat.is_cuda:
            raise _lib.RoomSlamError("FusedAdamW runs on CUDA only (no CPU fallback)")
        self.t += 1
        f = self.flat
        with torch.cuda.device(f.flat.device):
            _lib.call("rs_adamw_step_f32", f.flat.data_ptr(), f.grad.data_ptr(), self.m.data_ptr(), self.v.data_ptr(), f.numel,
                      self.lr, self.betas[0], self.betas[1], self.eps, self.wd, self.t, grad_scale, self.max_norm or 0.0,
                      self.scratch.data_ptr(), torch.cuda.current_stream(f.flat.device).cuda_stream)


class HostBatchPrefetcher:
    """Double-buffered host -> device staging: ``submit`` starts the copy of a (pinned) host batch on a side stream,
    ``get`` hands the device tensors to the current stream once the copy has landed.  Submitting batch k+1 right after
    getting batch k overlaps its PCIe transfer with step k's kernels (the upstream loop copies synchronously at the top
    of every iteration, src/benchmark/train.py:199-203)."""

    def __init__(self, device="cuda"):
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self._pending = None

    def submit(self, x_host: torch.Tensor, tgt_host: dict) -> None:
        if self._pending is not None:
            raise RuntimeError("HostBatchPrefetcher: get() the previous batch before submitting another one")
        self.stream.wait_stream(torch.cuda.current_stream(self.device))      # buffers freed by the compute stream are reusable
        with torch.cuda.stream(self.stream):
            x = x_host.to(self.device, non_blocking=True)
            tgt = {k: v.to(self.device, non_blocking=True) for k, v in tgt_host.items()}
            done = torch.cuda.Event()
            done.record(self.stream)
        self._pending = (x, tgt, done)

    def get(self):
        if self._pending is None:
            raise RuntimeError("HostBatchPrefetcher: nothing submitted")
        x, tgt, done = self._pending
        self._pending = None
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(done)
        x.record_stream(cur)
        for v in tgt.values():
            v.record_stream(cur)
        return x, tgt

    @property
    def has_pending(self) -> bool:
        return self._pending is not None
