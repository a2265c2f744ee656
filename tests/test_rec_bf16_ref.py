"""Self-check of oracle/rec_bf16_ref.py (no GPU): with exact float64 weights its teacher-forced forward step and its
backward recursion must reproduce a bidirectional float64 torch.nn.GRU -- hidden states to 1e-12 and every weight and bias
gradient, assembled from its dG, to 1e-10.  That pins the gate order, the 1/2 convention of the r and z rows, the reverse
direction's indexing, the packed-sequence semantics of `lengths` and the meaning of the hn block before the GPU tests
(test_rec_kernels_gpu.py) rely on them."""
import pytest
import torch
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

from oracle import rec_bf16_ref as R

F64 = torch.float64


def gru_run(H, I, B, T, lengths, seed, x_mult=None):
    """x_mult (B, T, I) or None: a dropout multiplier on the input, GRU(x * x_mult); grads["x"] is d/dx."""
    g = torch.Generator().manual_seed(seed)
    gru = torch.nn.GRU(I, H, batch_first=True, bidirectional=True).double()
    with torch.no_grad():
        for p in gru.parameters():
            p.copy_((torch.rand(p.shape, generator=g, dtype=F64) - 0.5) * (2.0 / H ** 0.5))
    x = torch.randn(B, T, I, generator=g, dtype=F64).requires_grad_()
    d_out = torch.randn(B, T, 2 * H, generator=g, dtype=F64)
    d_h_n = torch.randn(2, B, H, generator=g, dtype=F64)
    xin = x * x_mult if x_mult is not None else x
    if lengths is not None:
        packed = pack_padded_sequence(xin, lengths, batch_first=True, enforce_sorted=False)
        out, h_n = gru(packed)
        out, _ = pad_packed_sequence(out, batch_first=True, total_length=T)
    else:
        out, h_n = gru(xin)
    ((out * d_out).sum() + (h_n * d_h_n).sum()).backward()
    names = ("weight_ih_l0", "weight_hh_l0", "bias_ih_l0", "bias_hh_l0")
    w = [getattr(gru, n + sfx).detach() for sfx in ("", "_reverse") for n in names]
    grads = {n: torch.stack([getattr(gru, n + "_l0" + sfx).grad for sfx in ("", "_reverse")], 0)
             for n in ("weight_ih", "weight_hh", "bias_ih", "bias_hh")}
    grads["x"] = x.grad
    return x.detach(), out.detach(), h_n.detach(), d_out, d_h_n, w, grads


CASES = [  # (H, I, B, T, lengths)
    (128, 2, 5, 7, None),
    (128, 11, 5, 7, [7, 1, 4, 7, 2]),
    (256, 2, 4, 6, [3, 6, 1, 5]),
    (256, 11, 3, 5, None),
]


@pytest.mark.parametrize("H,I,B,T,lengths", CASES)
def test_reference_matches_torch_gru(H, I, B, T, lengths):
    lt = torch.tensor(lengths, dtype=torch.int32) if lengths is not None else None
    x, out, h_n, d_out, d_h_n, w, grads = gru_run(H, I, B, T, lengths, seed=H + I + B)
    W = R.ref_weights(w, H, split=0, quant=False)
    act = R.active_mask(lt, B, T, x.device)
    # the decoded `out` layout (2, B, T + 2, H) with zero pad rows, as the kernels leave it
    outf = torch.zeros(2, B, T + 2, H, dtype=F64)
    outf[0, :, 1:-1], outf[1, :, 1:-1] = out[..., :H], out[..., H:]
    hp = R.h_prev_forward(outf, lt)
    inp = R.input_from_x(x, W, B)
    f = R.forward_step(hp, inp, W, act)

    # forward: the blend of the teacher-forced gates is torch's next hidden state at every valid step of both directions
    for d in (0, 1):
        err = (f["h"][d] - outf[d, :, 1:-1]).abs() * act[..., None]
        assert float(err.max()) < 1e-12, (d, float(err.max()))
    last = (lt.long() - 1) if lt is not None else torch.full((B,), T - 1)
    assert torch.allclose(f["h"][0, torch.arange(B), last], h_n[0], atol=1e-12, rtol=0)
    assert torch.allclose(f["h"][1, :, 0], h_n[1], atol=1e-12, rtol=0)
    # past a trace's length z = 1 holds the state (direction 0 keeps reading its last valid step)
    assert torch.equal(f["z"][:, ~act], torch.ones_like(f["z"][:, ~act]))

    # backward: dG assembles into autograd's weight and bias gradients; hn both from the forward and recomputed from `out`
    hpb = R.h_prev_backward(outf)
    hn_re = R.recompute_hn(hpb, W)
    assert float((hn_re - f["hn"])[:, act].abs().max()) < 1e-12
    d_out_r = torch.stack([d_out[..., :H], d_out[..., H:]], 0)
    dG = R.backward(f["r"], f["z"], f["n"], hn_re, hpb, W, act, d_out=d_out_r, d_h_n=d_h_n)
    assert torch.equal(dG[:, ~act], torch.zeros_like(dG[:, ~act]))
    gw = R.weight_grads(dG, torch.stack([x, x], 0), hpb)
    for mine, theirs in (("w_ih", "weight_ih"), ("w_hh", "weight_hh"), ("b_ih", "bias_ih"), ("b_hh", "bias_hh")):
        ref = grads[theirs]
        err = float((gw[mine] - ref).abs().max() / ref.abs().max())
        assert err < 1e-10, (mine, err)

    # the teacher-forced backward, fed its own r | z | hn gradients, is the same recursion
    dG_tf = R.backward(f["r"], f["z"], f["n"], hn_re, hpb, W, act, d_out=d_out_r, d_h_n=d_h_n, feedback=dG[:, :, :, [0, 1, 3]])
    assert torch.allclose(dG_tf, dG, atol=1e-14, rtol=0)


def test_reference_without_d_out_or_d_h_n():
    """d_out and d_h_n each absent: the recursion is the one with that input zero."""
    H, I, B, T = 128, 2, 3, 5
    x, out, h_n, d_out, d_h_n, w, _ = gru_run(H, I, B, T, None, seed=3)
    W = R.ref_weights(w, H, split=0, quant=False)
    act = R.active_mask(None, B, T, x.device)
    outf = torch.zeros(2, B, T + 2, H, dtype=F64)
    outf[0, :, 1:-1], outf[1, :, 1:-1] = out[..., :H], out[..., H:]
    f = R.forward_step(R.h_prev_forward(outf, None), R.input_from_x(x, W, B), W, act)
    hpb = R.h_prev_backward(outf)
    d_out_r = torch.stack([d_out[..., :H], d_out[..., H:]], 0)
    args = (f["r"], f["z"], f["n"], f["hn"], hpb, W, act)
    assert torch.equal(R.backward(*args, d_out=None, d_h_n=d_h_n), R.backward(*args, d_out=torch.zeros_like(d_out_r), d_h_n=d_h_n))
    assert torch.equal(R.backward(*args, d_out=d_out_r, d_h_n=None), R.backward(*args, d_out=d_out_r, d_h_n=torch.zeros_like(d_h_n)))
    assert torch.equal(R.backward(*args), torch.zeros(2, B, T, 4, H, dtype=F64))


def test_decoders_keep_pads_and_invert():
    """tm_full / to_tm are inverses over every row and trace, pads included; out_full / dG_full / gates_full / drop_full
    address the documented columns."""
    g = torch.Generator().manual_seed(0)
    H, T, nt = 128, 3, 2
    full = torch.randn(nt * 128, T + 2, 2 * H, generator=g).to(torch.bfloat16).double()
    tm = R.to_tm(full)
    assert tm.shape == (nt, T + 2, 2 * H // 8, 128, 8)
    assert torch.equal(R.tm_full(tm), full)
    # element (trace b, row t', column c) sits at [b // 128, t', c // 8, b % 128, c % 8]
    b, tp, c = 200, 4, 3 * 8 + 5 + H
    assert float(tm[b // 128, tp, c // 8, b % 128, c % 8]) == float(full[b, tp, c])
    of = R.out_full(tm, H)
    assert float(of[1, b, tp, c - H]) == float(full[b, tp, c])
    dg = torch.randn(nt * 128, T + 2, 8 * H, generator=g).double()
    dgf = R.dG_full(R.to_tm(dg, torch.float32), H)
    assert float(dgf[1, b, 2, 3, 7]) == float(dg[b, 2, 4 * H + 3 * H + 7])
    # gates: [tiles][T][2][NG H / 8][128][8] fp16 bits in a bf16 buffer
    gv = torch.randn(nt, T, 2, 4 * H // 8, 128, 8, generator=g).to(torch.float16)
    gf = R.gates_full(gv.view(torch.bfloat16), H)
    assert float(gf[1, 130, 2, 3, 17]) == float(gv[1, 2, 1, (3 * H + 17) // 8, 2, 17 % 8])
    # dropout bits: byte c / 8, bit c % 8 of column c = d H + u
    bits = torch.zeros(nt, T, 128, 2 * H // 8, dtype=torch.uint8)
    bits[1, 2, 5, (H + 9) // 8] = 1 << ((H + 9) % 8)
    m = R.drop_full(bits, torch.tensor([2.0]), H)
    assert float(m.sum()) == 2.0 and float(m[1, 133, 2, 9]) == 2.0


def test_quantised_weights_follow_pack_w():
    """The operand values of the quantised weights: bf16(w / 2) on r, z rows, hi + lo with split, the bias as b_hi + b_lo."""
    g = torch.Generator().manual_seed(1)
    H, I = 128, 3
    w = [torch.randn(3 * H, I, generator=g), torch.randn(3 * H, H, generator=g), torch.randn(3 * H, generator=g),
         torch.randn(3 * H, generator=g)] * 2
    for split in (0, 1):
        W = R.ref_weights(w, H, split)
        w_hh = w[1]
        hi = (w_hh[:H] * 0.5).to(torch.bfloat16).float()
        exp = hi.double() + ((w_hh[:H] * 0.5 - hi).to(torch.bfloat16).double() if split else 0.0)
        assert torch.equal(W.whh[0, :H], exp)
        assert torch.equal(W.whh[1, 2 * H:], R.hi_lo(w_hh[2 * H:], split))
        assert torch.equal(W.whh_bwd[0], R.hi_lo(w_hh, split))
        # split weights carry ~16 mantissa bits
        err = float((W.whh[0] - torch.cat([w_hh[:2 * H] * 0.5, w_hh[2 * H:]]).double()).abs().max())
        assert err < (2.0 ** -14 if split else 2.0 ** -6) * float(w_hh.abs().max())
    bx = (w[2] + torch.cat([w[3][:2 * H], torch.zeros(H)])) * torch.cat([torch.full((2 * H,), 0.5), torch.ones(H)])
    assert torch.equal(R.bias_x(w[2], w[3], H), bx)
    assert float((W.bias[0] - bx.double()).abs().max()) <= 2.0 ** -16 * float(bx.abs().max())


@pytest.mark.parametrize("H,I,lengths,dropout", [(128, 256, None, False), (128, 256, [5, 1, 3, 5], True),
                                                 (256, 512, [2, 5, 5, 4], True)])
def test_data_grad_matches_torch_gru_input_grad(H, I, lengths, dropout):
    """data_grad over the reference's dG, with exact weights, is autograd's gradient of the layer input -- through a
    dropout multiplier on the input too, which data_grad applies at rows 1 .. T only (the pad rows stay unscaled)."""
    B, T = 4, 5
    g = torch.Generator().manual_seed(H + I)
    mult = (torch.rand(B, T, I, generator=g) < 0.75).to(F64) / 0.75 if dropout else None
    lt = torch.tensor(lengths, dtype=torch.int32) if lengths is not None else None
    x, out, _, d_out, d_h_n, w, grads = gru_run(H, I, B, T, lengths, seed=7, x_mult=mult)
    W = R.ref_weights(w, H, split=0, quant=False)
    act = R.active_mask(lt, B, T, x.device)
    outf = torch.zeros(2, B, T + 2, H, dtype=F64)
    outf[0, :, 1:-1], outf[1, :, 1:-1] = out[..., :H], out[..., H:]
    xin = x * mult if dropout else x
    inp = torch.stack([xin @ W.wih[d].T + W.bias[d] for d in (0, 1)], 0)
    f = R.forward_step(R.h_prev_forward(outf, lt), inp, W, act)
    hpb = R.h_prev_backward(outf)
    d_out_r = torch.stack([d_out[..., :H], d_out[..., H:]], 0)
    dG = R.backward(f["r"], f["z"], f["n"], R.recompute_hn(hpb, W), hpb, W, act, d_out=d_out_r, d_h_n=d_h_n)
    dGf = torch.zeros(2, B, T + 2, 4, H, dtype=F64)
    dGf[:, :, 1:-1] = dG
    dGf[:, :, 0], dGf[:, :, -1] = 1.0, -1.0                    # pad rows: they reach dX's pad rows and nothing else
    w_ih = torch.stack([w[0], w[4]], 0).to(F64)
    dx = R.data_grad(dGf, w_ih, mult)
    err = float((dx[:, 1:-1] - grads["x"]).abs().max() / grads["x"].abs().max())
    assert err < 1e-10, err
    pads = sum(dGf[d, :, [0, -1], :3].flatten(2) @ w_ih[d] for d in (0, 1))
    assert torch.allclose(dx[:, [0, -1]], pads, rtol=1e-12, atol=1e-12)


def test_projection_is_the_input_pre_activation():
    """projection with the reference's scaled weights and bias is X W_ih^T + b_ih (+ b_hh on r, z), r and z halved, at
    every row (pad rows included), per direction r | z | n."""
    H, I, Bp, T = 128, 256, 3, 4
    g = torch.Generator().manual_seed(5)
    w = [torch.randn(3 * H, I, generator=g), torch.randn(3 * H, H, generator=g), torch.randn(3 * H, generator=g),
         torch.randn(3 * H, generator=g)] * 2
    w[4:] = [t * 2 for t in w[4:]]
    W = R.ref_weights(w, H, split=0, quant=False)
    X = torch.randn(Bp, T + 2, I, generator=g, dtype=F64)
    P = R.projection(X, W.wih, W.bias)
    s = R.gate_scale(H, "cpu", F64)
    for d in (0, 1):
        w_ih, _, b_ih, b_hh = [t.to(F64) for t in w[4 * d: 4 * d + 4]]
        want = (X @ w_ih.T + b_ih + torch.cat([b_hh[:2 * H], torch.zeros(H, dtype=F64)])) * s
        assert float((P[..., 3 * H * d: 3 * H * (d + 1)] - want).abs().max()) < 1e-12


def test_x_operand_layout():
    """x_operand: bf16(x) in columns < I of rows 1 .. T of the real traces; zero columns >= I, pad rows and pad traces."""
    B, T, I, Bp = 3, 4, 5, 128
    x = torch.randn(B, T, I, generator=torch.Generator().manual_seed(2))
    xo = R.x_operand(x, Bp, T)
    assert xo.shape == (Bp, T + 2, 16) and xo.dtype == F64
    assert torch.equal(xo[:B, 1:-1, :I], x.to(torch.bfloat16).to(F64))
    rest = xo.clone()
    rest[:B, 1:-1, :I] = 0
    assert torch.equal(rest, torch.zeros_like(rest))
