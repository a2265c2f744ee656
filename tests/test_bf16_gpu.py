"""GPU parity of the bf16 tensor-core mode (tcgen05 recurrence + block GEMMs) against the fp32 torch CPU oracle.
Tolerance: 2e-2 relative (BASELINE.json north_star).  Hidden states and losses: max|a-b| / max|b| per tensor.
Gradients: relative L2 error ||a-b|| / ||b|| per tensor (a 0.3 % perturbation of the latent flips a few ReLUs of
the decoder, which moves single gradient ENTRIES by more than their tensor-level error), plus a 1e-1 bound on the
max-norm error so that no entry is grossly off."""
import numpy as np
import pytest
import torch

from oracle.room_slam_ref import RoomSLAM as RefRoomSLAM
from roomslam_b200 import RoomSLAM, synth

pytestmark = pytest.mark.gpu
RTOL = 2e-2
LOSS_KEYS = ("total", "class", "position", "size", "orientation", "validity")


def rel_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-6))


def l2_err(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / b.norm().clamp_min(1e-12))


def to_cuda(d):
    return {k: v.cuda() for k, v in d.items()}


@pytest.mark.parametrize("B,T,L,use_mask", [(4, 12, 1, False), (130, 40, 2, False), (37, 25, 2, True), (256, 500, 2, False),
                                            (256, 500, 2, True), (1, 1, 2, False), (3, 2, 2, False), (129, 3, 1, False)])
def test_bf16_matches_oracle(B, T, L, use_mask):
    torch.manual_seed(B + T)
    ref = RefRoomSLAM(num_layers=L, dropout=0.1 if use_mask else 0.0)
    dev = RoomSLAM(num_layers=L, dropout=ref.dropout, precision="bf16").cuda()
    dev.load_state_dict(ref.state_dict())
    ref.train(use_mask); dev.train(use_mask)
    x, tgt = synth.make_sample(B, T, 10, seed=B)
    mask = ref.make_dropout_mask(B, T, torch.Generator().manual_seed(1)) if use_mask else None
    enc_ref, hn_ref = ref.encode(x, mask)
    loss_ref = ref.compute_loss(ref(x, mask), tgt)
    loss_ref["total"].backward()
    xm = mask.cuda() if mask is not None else None
    enc_dev, hn_dev = dev.encode(x.cuda(), xm)
    loss_dev = dev.compute_loss(dev(x.cuda(), xm), to_cuda(tgt))
    loss_dev["total"].backward()
    assert rel_err(enc_dev, enc_ref) < RTOL and rel_err(hn_dev, hn_ref) < RTOL
    for k in LOSS_KEYS:
        assert abs(loss_dev[k].item() - loss_ref[k].item()) <= RTOL * max(abs(loss_ref[k].item()), 1e-6), k
    ref_grads = dict(ref.named_parameters())
    errs = {pn: (l2_err(p.grad, ref_grads[pn].grad), rel_err(p.grad, ref_grads[pn].grad)) for pn, p in dev.named_parameters()}
    bad = {k: v for k, v in errs.items() if not (v[0] < RTOL and v[1] < 1e-1)}
    assert not bad, bad


def test_bf16_rejects_other_hidden_sizes():
    from roomslam_b200 import _lib
    dev = RoomSLAM(hidden_size=64, precision="bf16").cuda()
    with pytest.raises(_lib.RoomSlamError):
        dev(torch.zeros(2, 4, 2, device="cuda"))


@pytest.mark.parametrize("B,T,L,use_mask", [(130, 40, 2, False), (200, 64, 2, True), (3, 5, 1, False), (129, 7, 2, False)])
def test_hidden_256_matches_oracle(B, T, L, use_mask):
    """hidden_size = 256 (README.md:153: HIDDEN_SIZE is a hyper-parameter; BASELINE config 4) on the tensor-core path
    that streams W_hh from L2 (csrc/rec_wide.cu), against the fp32 CPU oracle: 2e-2."""
    torch.manual_seed(B + T)
    ref = RefRoomSLAM(hidden_size=256, num_layers=L, dropout=0.1 if use_mask else 0.0)
    dev = RoomSLAM(hidden_size=256, num_layers=L, dropout=ref.dropout, precision="bf16").cuda()
    dev.load_state_dict(ref.state_dict())
    ref.train(use_mask); dev.train(use_mask)
    x, tgt = synth.make_sample(B, T, 10, seed=B)
    mask = ref.make_dropout_mask(B, T, torch.Generator().manual_seed(1)) if use_mask else None
    enc_ref, hn_ref = ref.encode(x, mask)
    loss_ref = ref.compute_loss(ref(x, mask), tgt)
    loss_ref["total"].backward()
    xm = mask.cuda() if mask is not None else None
    enc_dev, hn_dev = dev.encode(x.cuda(), xm)
    loss_dev = dev.compute_loss(dev(x.cuda(), xm), to_cuda(tgt))
    loss_dev["total"].backward()
    assert rel_err(enc_dev, enc_ref) < RTOL and rel_err(hn_dev, hn_ref) < RTOL
    for k in LOSS_KEYS:
        assert abs(loss_dev[k].item() - loss_ref[k].item()) <= RTOL * max(abs(loss_ref[k].item()), 1e-6), k
    ref_grads = dict(ref.named_parameters())
    tol = RTOL if B >= 100 else 5e-2          # a handful of traces: bf16 rounding noise does not average out (see module doc)
    errs = {pn: l2_err(p.grad, ref_grads[pn].grad) for pn, p in dev.named_parameters() if pn.startswith("encoder.")}
    bad = {k: v for k, v in errs.items() if not v < tol}
    assert not bad, bad


def test_c4_shape_hidden_256_seq_4000():
    """BASELINE config 4's shape at a batch the CPU oracle can follow (64 traces x 4000 steps, H = 256): hidden states,
    losses and encoder gradients of the bf16 tensor-core path against the fp32 oracle within 2e-2; lengths vary so the
    packed-sequence path of the wide kernels is exercised at the full 4000 steps too (second half of the batch)."""
    torch.manual_seed(4)
    ref = RefRoomSLAM(hidden_size=256, dropout=0.0).train()
    dev = RoomSLAM(hidden_size=256, dropout=0.0, precision="bf16").cuda().train()
    dev.load_state_dict(ref.state_dict())
    x, tgt = synth.make_sample(64, 4000, 10, seed=2)
    _, hn_ref = ref.encode(x)
    loss_ref = ref.compute_loss(ref(x), tgt)
    loss_ref["total"].backward()
    _, hn_dev = dev.encode(x.cuda())
    loss_dev = dev.compute_loss(dev(x.cuda()), to_cuda(tgt))
    loss_dev["total"].backward()
    assert rel_err(hn_dev, hn_ref) < RTOL
    for k in LOSS_KEYS:
        assert abs(loss_dev[k].item() - loss_ref[k].item()) <= RTOL * max(abs(loss_ref[k].item()), 1e-6), k
    ref_grads = dict(ref.named_parameters())
    errs = {pn: l2_err(p.grad, ref_grads[pn].grad) for pn, p in dev.named_parameters() if pn.startswith("encoder.")}
    bad = {k: v for k, v in errs.items() if not v < RTOL}
    assert not bad, bad


def _grad_errs(dev, ref_grads):
    return {k: l2_err(p.grad, ref_grads[k]) for k, p in dev.named_parameters()}


def test_c1_shape_explicit_bf16_against_the_unmodified_fp32_oracle():
    """BASELINE config 1 (32 traces x 500 steps, README.md:151 BATCH_SIZE = 32) with EXPLICIT precision="bf16" against
    the fp32 oracle at its own fp32 weights: every loss and every gradient tensor within the 2e-2 bar of north_star.
    Below 1024 traces the bf16 mode feeds the GRU weights to the tensor core as bf16 pairs (hi + lo): rounding them to a
    single bf16 alone moves the oracle's gradients by 2.3 % here (a coherent perturbation, tools/bf16_attrib_probe.py)."""
    torch.manual_seed(0)
    ref = RefRoomSLAM(hidden_size=128, dropout=0.0).train()
    dev = RoomSLAM(hidden_size=128, dropout=0.0, precision="bf16")
    dev.load_state_dict(ref.state_dict())
    dev = dev.cuda().train()
    x, tgt = synth.make_sample(32, 500, 10, seed=3)
    lr = ref.compute_loss(ref(x), tgt)
    lr["total"].backward()
    ld = dev.compute_loss(dev(x.cuda()), to_cuda(tgt))
    ld["total"].backward()
    for k in LOSS_KEYS:
        assert abs(ld[k].item() - lr[k].item()) <= RTOL * max(abs(lr[k].item()), 1e-6), k
    errs = _grad_errs(dev, {k: p.grad for k, p in ref.named_parameters()})
    bad = {k: v for k, v in errs.items() if not v < RTOL}
    assert not bad, bad


def test_split_weights_flag_changes_only_the_weight_precision():
    """bf16_split_weights=True / False at the same shape: both within tolerance of each other at a batch where plain
    bf16 weights are fine, and the flag is honoured (the results differ)."""
    torch.manual_seed(1)
    ref = RefRoomSLAM(hidden_size=128, dropout=0.0).train()
    x, tgt = synth.make_sample(300, 60, 10, seed=5)
    outs = []
    for flag in (True, False):
        dev = RoomSLAM(hidden_size=128, dropout=0.0, precision="bf16", bf16_split_weights=flag)
        dev.load_state_dict(ref.state_dict())
        dev = dev.cuda().train()
        _, h_n = dev.encode(x.cuda())
        outs.append(h_n.detach().cpu())
    assert not torch.equal(outs[0], outs[1])
    assert rel_err(outs[0], outs[1]) < RTOL


def test_benchmark_shape_8192x500():
    """The shape every headline number is measured at (BASELINE config 3 on one GPU: 8192 traces x 500 steps, bf16):
    losses and h_n against the fp32 CPU oracle on a fixed 1024-trace slice (the oracle does ~33 traces/s), and every
    parameter gradient of the full batch against the fp32 CUDA mode (itself pinned to the oracle at 1e-4)."""
    torch.manual_seed(0)
    ref = RefRoomSLAM(hidden_size=128, dropout=0.0).train()
    x, tgt = synth.make_sample(8192, 500, 10, seed=11)
    grads, hn, losses = {}, {}, {}
    for precision in ("fp32", "bf16"):
        dev = RoomSLAM(hidden_size=128, dropout=0.0, precision=precision)
        dev.load_state_dict(ref.state_dict())
        dev = dev.cuda().train()
        xd = x.cuda()
        _, h_n = dev.encode(xd)
        hn[precision] = h_n[:, :1024].detach().cpu()
        loss = dev.compute_loss(dev(xd), to_cuda(tgt))
        loss["total"].backward()
        losses[precision] = {k: v.item() for k, v in loss.items()}
        grads[precision] = {k: p.grad.detach().cpu() for k, p in dev.named_parameters()}
        del dev, xd, loss, h_n
        torch.cuda.empty_cache()
    for k in LOSS_KEYS:
        assert abs(losses["bf16"][k] - losses["fp32"][k]) <= RTOL * max(abs(losses["fp32"][k]), 1e-6), k
    bad = {k: l2_err(grads["bf16"][k], grads["fp32"][k]) for k in grads["fp32"]}
    bad = {k: v for k, v in bad.items() if not v < RTOL}
    assert not bad, bad
    # the oracle itself on the first 1024 traces: hidden states of both modes, and the fp32 mode's slice loss at 1e-4
    with torch.no_grad():
        _, hn_ref = ref.encode(x[:1024])
    assert rel_err(hn["fp32"], hn_ref) < 1e-4
    assert rel_err(hn["bf16"], hn_ref) < RTOL


def test_device_drawn_dropout_bits_match_the_oracle_with_the_same_mask():
    """Training mode without an explicit mask: the bf16 path draws Bernoulli bits on the device (rs_gen_drop_bits) and the
    recurrence kernels apply them (out (.) mask written by the forward kernel, d_out masked inside the BPTT kernel).  The
    oracle run with the float mask those bits stand for must agree within the bf16 tolerance; the keep rate is 1 - p."""
    from roomslam_b200 import functional_bf16 as FB
    B, T, H = 300, 40, 128
    bits, scale = FB.gen_drop_bits(B, T, 2 * H, 0.9, 1234, torch.device("cuda"))
    mask = FB.unpack_drop_bits(bits, scale, B)
    keep = float((mask > 0).float().mean())
    assert abs(keep - 0.9) < 5e-3 and abs(float(scale) - 1 / 0.9) < 1e-3
    bits2, _ = FB.gen_drop_bits(B, T, 2 * H, 0.9, 1234, torch.device("cuda"))
    bits3, _ = FB.gen_drop_bits(B, T, 2 * H, 0.9, 1235, torch.device("cuda"))
    assert torch.equal(bits, bits2) and not torch.equal(bits, bits3)          # a pure function of the seed
    pb, ps = FB.drop_bits_from_mask(mask)                                      # packing the float mask gives the bits back
    assert torch.equal(FB.unpack_drop_bits(pb, ps, B), mask) and abs(float(ps) - float(scale)) < 1e-6

    torch.manual_seed(3)
    ref = RefRoomSLAM(dropout=0.1).train()
    dev = RoomSLAM(dropout=0.1, precision="bf16").cuda().train()
    dev.load_state_dict(ref.state_dict())
    x, tgt = synth.make_sample(B, T, 10, seed=9)
    loss_ref = ref.compute_loss(ref(x, mask.cpu().unsqueeze(0)), tgt)
    loss_ref["total"].backward()
    # the model's own training path: give it the same bits by patching the generator it calls
    orig = FB.gen_drop_bits
    FB.gen_drop_bits = lambda *a, **k: (bits, scale)
    try:
        loss_dev = dev.compute_loss(dev(x.cuda()), to_cuda(tgt))
    finally:
        FB.gen_drop_bits = orig
    loss_dev["total"].backward()
    for k in LOSS_KEYS:
        assert abs(loss_dev[k].item() - loss_ref[k].item()) <= RTOL * max(abs(loss_ref[k].item()), 1e-6), k
    # the dropout path sits in the encoder: its gradients (and the trunk's) are held to the bf16 bar.  The head gradients
    # of an untrained model are sums of +-1 L1 signs that nearly cancel (one flipped sign of ~1600 moves them by several
    # per cent); they are covered, without dropout, by test_bf16_matches_oracle
    ref_grads = {k: p.grad for k, p in ref.named_parameters()}
    bad = {k: l2_err(p.grad, ref_grads[k]) for k, p in dev.named_parameters() if k.startswith(("encoder.", "decoder.trunk."))}
    bad = {k: v for k, v in bad.items() if not v < RTOL}
    assert not bad, bad


@pytest.mark.parametrize("B,T,use_mask,varlen", [(130, 40, False, False), (300, 64, True, False), (260, 50, False, True), (1100, 30, False, False)])
def test_fused_projection_meets_the_oracle(B, T, use_mask, varlen):
    """Deeper layers with unsplit weights run the K = 256 input projection INSIDE the recurrence kernel (W_ih resident,
    no P tensor, no projection GEMM): h_n, the losses and the encoder gradients against the fp32 oracle within 2e-2."""
    torch.manual_seed(B)
    ref = RefRoomSLAM(dropout=0.1 if use_mask else 0.0)
    ref.train(use_mask)
    x, tgt = synth.make_sample(B, T, 10, seed=B)
    mask = ref.make_dropout_mask(B, T, torch.Generator().manual_seed(1)) if use_mask else None
    lengths = torch.randint(1, T + 1, (B,), generator=torch.Generator().manual_seed(2)) if varlen else None
    dev = RoomSLAM(dropout=ref.dropout, precision="bf16", bf16_split_weights=False).cuda()
    dev.load_state_dict(ref.state_dict())
    dev.train(use_mask)
    xm = mask.cuda() if mask is not None else None
    _, hn_dev = dev.encode(x.cuda(), xm, lengths)
    loss_dev = dev.compute_loss(dev(x.cuda(), xm, lengths), to_cuda(tgt))
    loss_dev["total"].backward()
    _, hn_ref = ref.encode(x, mask, lengths)
    loss_ref = ref.compute_loss(ref(x, mask, lengths), tgt)
    loss_ref["total"].backward()
    assert rel_err(hn_dev, hn_ref) < RTOL
    for k in LOSS_KEYS:
        assert abs(loss_dev[k].item() - loss_ref[k].item()) <= RTOL * max(abs(loss_ref[k].item()), 1e-6), k
    ref_grads = dict(ref.named_parameters())
    bad = {pn: l2_err(p.grad, ref_grads[pn].grad) for pn, p in dev.named_parameters() if pn.startswith("encoder.")}
    bad = {k: v for k, v in bad.items() if not v < RTOL}
    assert not bad, bad


@pytest.mark.parametrize("H,B,T", [(128, 300, 40), (128, 1100, 24), (256, 200, 24)])
def test_dropout_backward_in_dgrad_epilogue_equals_in_bptt_kernel(H, B, T):
    """The backward half of inter-layer dropout is applied by the CONSUMING layer (dX (.) mask in the epilogue of its dgrad
    GEMM, rs_blk_gemm_nt_drop); the BPTT kernel of the producing layer can do the same on the incoming gradient.  Same
    bits, same weights: the two placements must agree up to the bf16 rounding of dX (rounded after / before the scale)."""
    from roomslam_b200 import functional as F_, functional_bf16 as FB
    torch.manual_seed(H + B)
    dev = RoomSLAM(hidden_size=H, dropout=0.1, precision="bf16").cuda().train()
    x, tgt = synth.make_sample(B, T, 10, seed=4)
    bits = [FB.gen_drop_bits(B, T, 2 * H, 0.9, 77, torch.device("cuda"))]
    grads = []
    for in_bptt in (False, True):
        dev.zero_grad()
        w = dev.encoder.flat_weights()
        layer_fn = FB.GRULayerBF16Fn if H == 128 else FB.GRULayerBF16WideFn
        _, h_n = F_.gru_encoder(x.cuda(), bits, 2, w, layer_fn, None, split_weights=False, mask_in_bptt=in_bptt)
        (h_n ** 2).sum().backward()
        grads.append([p.grad.clone() for p in dev.encoder.parameters()])
    for a, b in zip(*grads):
        assert l2_err(a, b) < 1e-2 and float(b.abs().max()) > 0


@pytest.mark.parametrize("H,B,T", [(128, 1100, 60), (128, 300, 33), (256, 260, 20)])
def test_recurrence_is_reproducible(H, B, T):
    """The forward recurrence has no atomics: repeated runs must give BIT-identical outputs and hidden states.  The weight
    gradients end in fp32 atomic sums, so they may differ by summation order only (1e-5 relative L2).  A race between the
    epilogue warps, the issuing thread and the copy producers (arrivals before the last stores, loads issued after the
    arrival, single-thread tile copies) would show up here long before it moves a 2e-2 tolerance."""
    torch.manual_seed(H + T)
    dev = RoomSLAM(hidden_size=H, dropout=0.0, precision="bf16").cuda().train()
    x, _ = synth.make_sample(B, T, 10, seed=11)
    runs = []
    for _ in range(3):
        dev.zero_grad()
        out, h_n = dev.encode(x.cuda())
        (h_n.square().sum() + out.square().sum()).backward()
        runs.append((out.detach().clone(), h_n.detach().clone(), [p.grad.detach().clone() for p in dev.encoder.parameters()]))
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1])
        for a, b in zip(r[2], runs[0][2]):
            assert l2_err(a, b) < 1e-5
