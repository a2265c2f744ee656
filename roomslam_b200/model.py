"""RoomSLAM nn.Module on B200: bidirectional-GRU encoder + MLP decoder heads + multi-task loss.

Drop-in for the `src/models/room_slam.py` the upstream README describes (README.md:110-125, :147-157; no code
upstream, SURVEY.md section 0).  Constructor, forward(), compute_loss() and state_dict() keys are identical to the
CPU oracle (oracle/room_slam_ref.py), so `cuda_model.load_state_dict(oracle.state_dict())` is the parity harness
and checkpoints interchange.  The arithmetic runs in libroomslam_b200.so; nothing falls back to torch ops.

precision="fp32": CUDA-core kernels, parity 1e-4 relative to torch's CPU path.
precision="bf16": tcgen05 tensor-core kernels (bf16 operands, fp32 accumulate), parity 2e-2; hidden_size 128 or 256 and
                  input_size <= 16 (the layer-0 projection rides on the recurrence MMA; wider inputs: precision="fp32").
precision="auto": bf16 from 256 traces per step when hidden_size is 128 or 256 and input_size <= 2, fp32 otherwise.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _lib
from . import functional as F_

CLASS_NAMES = ("GROUND", "LOW", "MID", "BLOCK")    # README.md:20-23, decision D7
LOSS_KEYS = ("total", "class", "position", "size", "orientation", "validity")


class GRUParams(nn.Module):
    """Parameter container with torch.nn.GRU's names, shapes, order and U(-1/sqrt(H), 1/sqrt(H)) init
    (torch/nn/modules/rnn.py:1301), so that state_dicts interchange with the oracle's nn.GRU."""

    def __init__(self, input_size: int, hidden_size: int, num_layers: int):
        super().__init__()
        self.input_size, self.hidden_size, self.num_layers = input_size, hidden_size, num_layers
        H = hidden_size
        self._names = []
        for layer in range(num_layers):
            in_l = input_size if layer == 0 else 2 * H
            for sfx in ("", "_reverse"):
                for name, shape in ((f"weight_ih_l{layer}{sfx}", (3 * H, in_l)), (f"weight_hh_l{layer}{sfx}", (3 * H, H)),
                                    (f"bias_ih_l{layer}{sfx}", (3 * H,)), (f"bias_hh_l{layer}{sfx}", (3 * H,))):
                    self.register_parameter(name, nn.Parameter(torch.empty(*shape)))
                    self._names.append(name)
        stdv = 1.0 / math.sqrt(H)
        for p in self.parameters():
            nn.init.uniform_(p, -stdv, stdv)

    def flat_weights(self):
        return [getattr(self, n) for n in self._names]


class Decoder(nn.Module):
    """Parameter container for the MLP decoder (README.md:117-120; decision D6).  nn.Linear is used only to hold
    and initialise weights; the math runs in DecoderFn (fp32 CUDA-core GEMM) or DecoderBF16Fn (TMA-fed tcgen05 GEMM)."""

    def __init__(self, in_features: int, hidden: int, max_objects: int, num_classes: int, precision: str = "fp32"):
        super().__init__()
        self.max_objects, self.num_classes = max_objects, num_classes
        self.precision = precision
        self.trunk = nn.Sequential(nn.Linear(in_features, hidden), nn.ReLU(), nn.Linear(hidden, hidden), nn.ReLU())
        self.class_head = nn.Linear(hidden, max_objects * num_classes)
        self.pos_head = nn.Linear(hidden, max_objects * 2)
        self.size_head = nn.Linear(hidden, max_objects * 2)
        self.orient_head = nn.Linear(hidden, max_objects)
        self.valid_head = nn.Linear(hidden, max_objects)

    def forward(self, latent: torch.Tensor) -> Dict[str, torch.Tensor]:
        heads = []
        for h in (self.class_head, self.pos_head, self.size_head, self.orient_head, self.valid_head):
            heads += [h.weight, h.bias]
        fn = F_.DecoderFn
        # bf16 mode: tensor-core decoder for inference (any batch: predictions must not depend on the chunking) and for
        # training from 256 traces up.  Below that the training GEMMs are latency-bound anyway and a single bf16-induced
        # ReLU flip moves the gradient of a 3-trace batch by several per cent (tools/bf16_err_probe.py).
        if self.precision == "bf16" and (latent.shape[0] >= 256 or not torch.is_grad_enabled()) and latent.shape[1] % 64 == 0 \
                and self.trunk[0].out_features % 128 == 0 and self.trunk[2].out_features % 128 == 0:
            from .functional_bf16 import DecoderBF16Fn as fn
        cls, pos, size, orient, valid = fn.apply(
            latent, self.max_objects, self.num_classes, self.trunk[0].weight, self.trunk[0].bias,
            self.trunk[2].weight, self.trunk[2].bias, *heads)
        return {"class_logits": cls, "positions": pos, "sizes": size, "orientations": orient, "validity_logits": valid}


class RoomSLAM(nn.Module):
    def __init__(self, input_size: int = 2, hidden_size: int = 128, num_layers: int = 2, max_objects: int = 10,
                 num_classes: int = 4, dropout: float = 0.1, decoder_hidden: int = 256, precision: str = "fp32",
                 bf16_split_weights: Optional[bool] = None):
        super().__init__()
        if precision not in ("fp32", "bf16", "auto"):
            raise ValueError(f"precision must be 'fp32', 'bf16' or 'auto', got {precision!r}")
        if hidden_size % 32 or not (32 <= hidden_size <= 512):
            raise ValueError("hidden_size must be a multiple of 32 in [32, 512]")
        self.input_size, self.hidden_size, self.num_layers = input_size, hidden_size, num_layers
        self.max_objects, self.num_classes, self.dropout = max_objects, num_classes, dropout
        self.precision = precision
        # bf16 mode: feed every GRU weight to the tensor core as a bf16 PAIR hi + lo (~16 mantissa bits) instead of one bf16.
        # Rounding the weights is a coherent perturbation (it does not average out over the batch like activation rounding):
        # alone it moves the gradients by 2.3 % at batch 32.  None = automatic: split below SPLIT_WEIGHTS_BELOW traces per
        # step, where the recurrence is latency-bound and the doubled MMA work is free; plain bf16 weights above.
        self.bf16_split_weights = bf16_split_weights
        self.encoder = GRUParams(input_size, hidden_size, num_layers)
        self.decoder = Decoder(2 * hidden_size, decoder_hidden, max_objects, num_classes, precision)

    # -- dropout mask (decision D4: explicit Bernoulli mask so oracle and kernel see the same one) ----------
    def make_dropout_mask(self, batch: int, seq_len: int, generator: Optional[torch.Generator] = None,
                          device=None) -> Optional[torch.Tensor]:
        if self.num_layers < 2 or self.dropout <= 0.0:
            return None
        keep = 1.0 - self.dropout
        shape = (self.num_layers - 1, batch, seq_len, 2 * self.hidden_size)
        gen_dev = generator.device if generator is not None else (device or "cpu")
        m = (torch.rand(shape, generator=generator, device=gen_dev) < keep).to(torch.float32) / keep
        return m.to(device) if device is not None else m

    def _check_input(self, x: torch.Tensor):
        if x.dim() != 3 or x.shape[-1] != self.input_size:
            raise ValueError(f"expected input of shape (B, T, {self.input_size}), got {tuple(x.shape)}")
        if not x.is_cuda:
            raise _lib.RoomSlamError("RoomSLAM runs on CUDA (sm_100a) only: move the model and inputs to the GPU; "
                                     "there is no CPU fallback")

    def _check_lengths(self, x, lengths):
        if lengths is None:
            return None
        lengths = torch.as_tensor(lengths)
        if lengths.shape != (x.shape[0],) or (x.shape[0] and (int(lengths.min()) < 1 or int(lengths.max()) > x.shape[1])):
            raise ValueError("lengths must hold one value in [1, T] per trace (torch.nn.utils.rnn.pack_padded_sequence's rule)")
        return lengths

    def encode(self, x: torch.Tensor, dropout_mask: Optional[torch.Tensor] = None, lengths: Optional[torch.Tensor] = None):
        """(out (B,T,2H) of the top layer, h_n (2L,B,H)) with torch.nn.GRU semantics; with `lengths` (valid steps per
        trace) those of a packed sequence: zero outputs past a trace's end, h_n taken at its last valid step."""
        self._check_input(x)
        lengths = self._check_lengths(x, lengths)
        out, h_n = self._encode(x, dropout_mask, lengths)
        if isinstance(out, F_._LazyOut):
            out = out.materialize()
        return out, h_n

    AUTO_BF16_MIN_BATCH = 256
    SPLIT_WEIGHTS_BELOW = 1024

    def _use_bf16(self, batch: int) -> bool:
        """'auto': the tensor-core bf16 kernels from 256 traces per step (where their 2e-2 gradient bar holds, DESIGN.md 4.2)
        when the shape fits them (H = 128, at most 2 input columns); the fp32 kernels (1e-4) otherwise."""
        if self.precision == "auto":
            return batch >= self.AUTO_BF16_MIN_BATCH and self.hidden_size in (128, 256) and self.input_size <= 2
        return self.precision == "bf16"

    def _encode(self, x, dropout_mask, lengths=None):
        bf16 = self._use_bf16(x.shape[0])
        self.decoder.precision = "bf16" if bf16 else "fp32"
        layer_fn = _bf16_layer_fn(self.hidden_size) if bf16 else F_.GRULayerFn
        # inter-layer dropout (README.md:114): an explicit float mask (decision D4) is used as given; without one, training
        # mode draws it -- as packed bits on the device for the bf16 kernels, as a float mask for the fp32 kernels
        if dropout_mask is not None:
            if dropout_mask.dim() == 3:
                dropout_mask = dropout_mask.unsqueeze(0)
            dropout_mask = dropout_mask.to(device=x.device, dtype=torch.float32)
        elif self.training and self.dropout > 0 and self.num_layers > 1:
            if bf16:
                from .functional_bf16 import gen_drop_bits
                seeds = torch.randint(0, 2 ** 62, (self.num_layers - 1,))        # host RNG: reproducible under manual_seed
                dropout_mask = [gen_drop_bits(x.shape[0], x.shape[1], 2 * self.hidden_size, 1.0 - self.dropout, int(s), x.device)
                                for s in seeds]
            else:
                dropout_mask = self.make_dropout_mask(x.shape[0], x.shape[1], device=x.device)
        split = bf16 and self.hidden_size == 128 and (self.bf16_split_weights if self.bf16_split_weights is not None else x.shape[0] < self.SPLIT_WEIGHTS_BELOW)
        return F_.gru_encoder(x, dropout_mask, self.num_layers, self.encoder.flat_weights(), layer_fn, lengths, split_weights=split)

    def forward(self, x: torch.Tensor, dropout_mask: Optional[torch.Tensor] = None,
                lengths: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
        self._check_input(x)
        lengths = self._check_lengths(x, lengths)
        _, h_n = self._encode(x, dropout_mask, lengths)
        latent = torch.cat([h_n[-2], h_n[-1]], dim=-1)          # decision D5 (README.md:115)
        return self.decoder(latent)

    @torch.no_grad()
    def predict(self, x: torch.Tensor, batch_size: int = 16384) -> Dict[str, torch.Tensor]:
        """Batched inference (BASELINE config 5: hundreds of thousands of traces): forward in chunks of `batch_size`
        traces so that the per-timestep activations of one chunk fit in HBM; x may live on the host (each chunk is
        copied to the model's device) and the predictions come back on x's device."""
        was_training = self.training
        self.eval()
        dev = next(self.parameters()).device
        outs = []
        try:
            for s in range(0, x.shape[0], batch_size):
                xb = x[s:s + batch_size].to(dev, non_blocking=True)
                outs.append({k: v.to(x.device) for k, v in self.forward(xb).items()})
        finally:
            self.train(was_training)
        if not outs:
            return self.forward(x.to(dev))
        return {k: torch.cat([o[k] for o in outs], 0) for k in outs[0]}

    def compute_loss(self, pred: Dict[str, torch.Tensor], target: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
        losses = F_.MultiTaskLossFn.apply(pred["class_logits"], pred["positions"], pred["sizes"], pred["orientations"],
                                          pred["validity_logits"], target["classes"], target["positions"],
                                          target["sizes"], target["orientations"], target["valid"])
        return {k: losses[i] for i, k in enumerate(LOSS_KEYS)}


def _bf16_layer_fn(hidden_size: int):
    """The tensor-core recurrence exists for hidden_size 128 (W_hh resident in shared memory, csrc/rec_pair.cu) and 256
    (W_hh streamed from L2, csrc/rec_wide.cu); other sizes run the fp32 kernels."""
    from .functional_bf16 import GRULayerBF16Fn, GRULayerBF16WideFn
    if hidden_size == 128:
        return GRULayerBF16Fn
    if hidden_size == 256:
        return GRULayerBF16WideFn
    raise _lib.RoomSlamError(f"bf16 mode is built for hidden_size 128 or 256 (got {hidden_size}); use precision='fp32'")
