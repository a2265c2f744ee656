"""CPU self-checks of oracle/decoder_ref.py, the float64 reference that tests/test_decoder_loss_gpu.py holds the decoder,
loss and AdamW kernels to: composed stage by stage, it must reproduce float64 autograd of oracle.room_slam_ref.Decoder +
RoomSLAM.compute_loss, and its AdamW step torch.optim.AdamW + clip_grad_norm_."""
import numpy as np
import pytest
import torch

from oracle import decoder_ref as D
from oracle import room_slam_ref as R

F64 = torch.float64


def _rel(a, b):
    a, b = a.to(F64), b.to(F64)
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


def _problem(seed, B, DL, DH, N, C, valid="fractional"):
    g = torch.Generator().manual_seed(seed)
    dec = R.Decoder(DL, DH, N, C).double()
    with torch.no_grad():
        for p in dec.parameters():
            p.copy_(torch.randn(p.shape, generator=g, dtype=F64) * 0.3)
    lat = torch.randn(B, DL, generator=g, dtype=F64)
    tgt = {"classes": torch.randint(0, C, (B, N), generator=g), "positions": torch.randn(B, N, 2, generator=g, dtype=F64),
           "sizes": torch.rand(B, N, 2, generator=g, dtype=F64) * 3, "orientations": torch.randn(B, N, generator=g, dtype=F64)}
    if valid == "fractional":
        tgt["valid"] = torch.rand(B, N, generator=g, dtype=F64)
    elif valid == "none":
        tgt["valid"] = torch.zeros(B, N, dtype=F64)
    else:
        tgt["valid"] = (torch.rand(B, N, generator=g) < 0.5).to(F64)
    return dec, lat, tgt


def _composed(dec, lat, tgt, d_losses):
    N, C = dec.max_objects, dec.num_classes
    heads = []
    for h in (dec.class_head, dec.pos_head, dec.size_head, dec.orient_head, dec.valid_head):
        heads += [h.weight.detach(), h.bias.detach()]
    Wh, bh = D.pad_heads(heads)
    W1, b1, W2, b2 = (t.detach() for t in (dec.trunk[0].weight, dec.trunk[0].bias, dec.trunk[2].weight, dec.trunk[2].bias))
    f = D.decoder_fwd(lat, W1, b1, W2, b2, Wh, bh)
    NH = N * (C + 6)
    assert (f["rawp"][:, NH:] == 0).all()
    raw = f["rawp"][:, :NH]
    pred = D.heads_split(raw, N, C)
    sums, g = D.loss_terms(*pred, tgt["classes"], tgt["positions"], tgt["sizes"], tgt["orientations"], tgt["valid"])
    losses = D.loss_finalize(sums, g[4].numel())
    d_pred = D.loss_bwd(sums, g, d_losses)
    d_raw = D.heads_merge(raw, N, C, *d_pred)
    d_rawp = torch.cat([d_raw, d_raw.new_zeros(d_raw.shape[0], Wh.shape[0] - NH)], 1)
    b = D.decoder_bwd(lat, W1, W2, Wh, f["f1"], f["f2"], d_rawp, d_raw)
    assert (b["dWh"][NH:] == 0).all()
    grads = [b["dW1"], b["db1"], b["dW2"], b["db2"], b["dWh"][:NH], b["dbh"]]
    return losses, grads, b["dlat"]


D_LOSSES = [torch.eye(6, dtype=F64)[k] for k in range(6)] + [torch.tensor([0.7, -1.3, 2.1, 0.4, -0.9, 1.6], dtype=F64)]


@pytest.mark.parametrize("shape", [(7, 64, 32, 5, 3), (3, 16, 24, 13, 1), (5, 32, 16, 2, 16)])
@pytest.mark.parametrize("valid", ["fractional", "binary", "none"])
def test_composed_reference_matches_autograd(shape, valid):
    """losses, every parameter gradient and d latent, for each loss component alone and for a random d(losses)."""
    B, DL, DH, N, C = shape
    dec, lat, tgt = _problem(11 + B, B, DL, DH, N, C, valid)
    with torch.no_grad():                              # some size pre-activations above the softplus threshold
        dec.size_head.bias[: N] += 25.0
    for d_losses in D_LOSSES:
        dec.zero_grad()
        latr = lat.clone().requires_grad_(True)
        pred = dec(latr)
        ref = R.RoomSLAM.compute_loss(None, pred, tgt)
        lv = torch.stack([ref[k] for k in ("total", "class", "position", "size", "orientation", "validity")])
        (lv * d_losses).sum().backward()
        losses, grads, dlat = _composed(dec, lat, tgt, d_losses)
        assert _rel(losses, lv.detach()) < 1e-12
        head_w = torch.cat([h.weight.grad for h in (dec.class_head, dec.pos_head, dec.size_head, dec.orient_head, dec.valid_head)])
        head_b = torch.cat([h.bias.grad for h in (dec.class_head, dec.pos_head, dec.size_head, dec.orient_head, dec.valid_head)])
        want = [dec.trunk[0].weight.grad, dec.trunk[0].bias.grad, dec.trunk[2].weight.grad, dec.trunk[2].bias.grad, head_w, head_b]
        for got, w in zip(grads, want):
            assert _rel(got, w) < 1e-12 or (w == 0).all() and (got == 0).all()
        assert _rel(dlat, latr.grad) < 1e-12 or (latr.grad == 0).all() and (dlat == 0).all()


def test_heads_split_threshold_and_blocks():
    N, C = 3, 2
    raw = torch.arange(2 * N * (C + 6), dtype=F64).reshape(2, -1)
    cls, pos, size, orient, valid = D.heads_split(raw, N, C)
    assert torch.equal(cls.reshape(2, -1), raw[:, :6]) and torch.equal(pos.reshape(2, -1), raw[:, 6:12])
    assert torch.equal(orient, raw[:, 18:21]) and torch.equal(valid, raw[:, 21:24])
    v = torch.tensor([[20.0, np.nextafter(np.float32(20), np.float32(30)), -100.0, 88.0]], dtype=F64)
    sp = D.softplus(v)
    assert float(sp[0, 0]) == pytest.approx(20 + np.log1p(np.exp(-20.0)), rel=1e-15)
    assert float(sp[0, 1]) == float(v[0, 1]) and float(sp[0, 3]) == 88.0
    assert torch.equal(D.softplus(v, 21.0)[0, 1], torch.log1p(torch.exp(v[0, 1])))


def _torch_adamw(p0, grads, lr, betas, eps, wd, grad_scale, max_norm):
    p = torch.nn.Parameter(p0.clone())
    opt = torch.optim.AdamW([p], lr=lr, betas=betas, eps=eps, weight_decay=wd)
    out, norms = [], []
    for g in grads:
        p.grad = g.clone() * grad_scale
        norms.append(float(p.grad.square().sum()))
        if max_norm > 0:
            torch.nn.utils.clip_grad_norm_([p], max_norm)
        opt.step()
        st = opt.state[p]
        out.append((p.detach().clone(), st["exp_avg"].clone(), st["exp_avg_sq"].clone()))
    return out, norms


@pytest.mark.parametrize("max_norm,grad_scale", [(0.5, 1.0), (0.5, 0.125), (0.0, 1.0), (1e3, 0.125)])
def test_adamw_reference_matches_torch(max_norm, grad_scale):
    """Five steps with float32-exact hyperparameters: the reference equals torch.optim.AdamW + clip_grad_norm_."""
    g = torch.Generator().manual_seed(3)
    n = 1000
    p0 = torch.randn(n, generator=g, dtype=F64)
    grads = [torch.randn(n, generator=g, dtype=F64) * 0.1 for _ in range(5)]
    hp = dict(lr=2.0 ** -7, eps=2.0 ** -20, wd=2.0 ** -4)
    betas = (0.875, 1 - 2.0 ** -10)
    want, norms = _torch_adamw(p0, grads, hp["lr"], betas, hp["eps"], hp["wd"], grad_scale, max_norm)
    p, m, v = p0, torch.zeros(n, dtype=F64), torch.zeros(n, dtype=F64)
    for t, (gr, (wp, wm, wv), nrm) in enumerate(zip(grads, want, norms), 1):
        p, m, v, sumsq = D.adamw_step(p, gr, m, v, hp["lr"], betas[0], betas[1], hp["eps"], hp["wd"], t, grad_scale, max_norm)
        assert _rel(p - p0, wp - p0) < 1e-12 and _rel(m, wm) < 1e-12 and _rel(v, wv) < 1e-12
        assert sumsq == (pytest.approx(nrm, rel=1e-13) if max_norm > 0 else 0.0)


def test_adamw_bias_corrections():
    """The float32 bias corrections of the C entry point, and the fault variants differ from the correct step."""
    assert D.bias_corrections(0.9, 0.999, 1, True) == (float(np.float32(1) - np.float32(0.9)), float(np.float32(1) - np.float32(0.999)))
    assert D.bias_corrections(0.875, 1 - 2.0 ** -10, 3, False) == (1 - 0.875 ** 3, 1 - (1 - 2.0 ** -10) ** 3)
    p, g, m, v = torch.ones(4, dtype=F64), torch.full((4,), 0.5, dtype=F64), torch.full((4,), 0.1, dtype=F64), torch.full((4,), 0.2, dtype=F64)
    base = D.adamw_step(p, g, m, v, 1e-2, 0.9, 0.999, 1e-8, 0.1, 2)[0]
    for kw in (dict(decay_after=True), dict(sqrt_bc2=False)):
        assert _rel(D.adamw_step(p, g, m, v, 1e-2, 0.9, 0.999, 1e-8, 0.1, 2, **kw)[0] - p, base - p) > 1e-6
