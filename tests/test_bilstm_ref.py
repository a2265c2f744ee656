"""CPU self-checks of oracle/bilstm_ref.py, the float64 reference the BiLSTM kernel tests (test_bilstm_kernels_gpu.py)
compare against: the LSTM forward and backward recursions against float64 torch.nn.LSTM and autograd, the query
attention against float64 autograd of the oracle decoder's attention (k / v folded as SimpleQueryDecoder folds them),
and trace_stats against TraceEncoderRef.stats."""
import pytest
import torch

from oracle import bilstm_ref as R
from oracle.lstm_ref import QueryDecoderRef, TraceEncoderRef

F64 = torch.float64


def lstm_case(H, B, T, I, drop, seed):
    g = torch.Generator().manual_seed(seed)
    lstm = torch.nn.LSTM(I, H, batch_first=True, bidirectional=True).double()
    with torch.no_grad():
        for p in lstm.parameters():
            p.copy_((torch.rand(p.shape, generator=g, dtype=F64) * 2 - 1) * 1.5 / H ** 0.5)
    xin = torch.zeros(B, T + 2, I, dtype=F64)
    xin[:, 1:-1] = torch.randn(B, T, I, generator=g, dtype=F64)
    mask = (torch.rand(B, T, I, generator=g) < 0.8).to(F64) / 0.8 if drop else None
    return lstm, xin, mask, torch.randn(B, T, 2 * H, generator=g, dtype=F64)


def layer_operands(lstm, H):
    w_ih = torch.cat([lstm.weight_ih_l0, lstm.weight_ih_l0_reverse], 0).detach()
    w_hh = torch.stack([lstm.weight_hh_l0, lstm.weight_hh_l0_reverse]).detach()
    b = torch.cat([lstm.bias_ih_l0 + lstm.bias_hh_l0, lstm.bias_ih_l0_reverse + lstm.bias_hh_l0_reverse]).detach()
    return w_ih, w_hh, b


@pytest.mark.parametrize("H", [32, 64, 96, 128])
@pytest.mark.parametrize("B,T", [(1, 7), (5, 13)])
@pytest.mark.parametrize("drop", [False, True])
def test_lstm_reference_against_torch(H, B, T, drop):
    I = 2 * H
    lstm, xin, mask, d_out = lstm_case(H, B, T, I, drop, seed=H + B + T)
    w_ih, w_hh, b = layer_operands(lstm, H)
    x = xin.clone().requires_grad_(True)
    xm = R.masked_input(x, mask)
    want, _ = lstm(xm[:, 1:-1])
    (want * d_out).sum().backward()

    # forward: P with the bias folded in, the free recursion, and the teacher-forced step on its own h and c
    P = R.masked_input(xin, mask) @ w_ih.t() + b
    Pd = R.dirs(P[:, 1:-1], 4)
    fr = R.forward_free(Pd, w_hh)
    h = R.undirs(fr["h"].unsqueeze(3))
    assert (h - want.detach()).abs().max() < 1e-12
    tf = R.forward_step(Pd, w_hh, R.prev_step(fr["h"]))
    assert (tf["gates"] - fr["gates"]).abs().max() < 1e-12
    c, _ = R.cell(fr["gates"], R.prev_step(fr["c"]))
    assert (c - fr["c"]).abs().max() < 1e-12
    assert (R.h_of(fr["gates"][:, :, :, 3], fr["c"])[0] - fr["h"]).abs().max() < 1e-12

    # backward: free and teacher-forced on its own dG agree; assembled, they are torch's gradients
    dod = R.dirs(d_out, 1)[:, :, :, 0]
    bw = R.backward(fr["gates"], fr["c"], w_hh, dod)
    bt = R.backward(fr["gates"], fr["c"], w_hh, dod, feedback=bw["dG"])
    assert (bw["dG"] - bt["dG"]).abs().max() < 1e-12
    dG = torch.zeros(B, T + 2, 8 * H, dtype=F64)
    dG[:, 1:-1] = R.undirs(bw["dG"])
    out = torch.zeros(B, T + 2, 2 * H, dtype=F64)
    out[:, 1:-1] = h
    dW_ih, dW_hh, db = R.lstm_weight_grads(dG, out, xin, mask)
    tol = 1e-10
    assert (dW_ih[:4 * H] - lstm.weight_ih_l0.grad).abs().max() < tol
    assert (dW_ih[4 * H:] - lstm.weight_ih_l0_reverse.grad).abs().max() < tol
    assert (dW_hh[0] - lstm.weight_hh_l0.grad).abs().max() < tol
    assert (dW_hh[1] - lstm.weight_hh_l0_reverse.grad).abs().max() < tol
    for n in ("bias_ih_l0", "bias_hh_l0"):
        assert (db[:4 * H] - getattr(lstm, n).grad).abs().max() < tol
        assert (db[4 * H:] - getattr(lstm, n + "_reverse").grad).abs().max() < tol
    assert (R.data_grad(dG, w_ih, mask) - x.grad).abs().max() < tol


def test_lstm_backward_fault_reference_differs():
    """dc_no_f (a deliberately wrong reference) must change dG: the sensitivity test relies on it."""
    lstm, xin, _, d_out = lstm_case(32, 2, 9, 64, False, 0)
    w_ih, w_hh, b = layer_operands(lstm, 32)
    fr = R.forward_free(R.dirs((xin @ w_ih.t() + b)[:, 1:-1], 4), w_hh)
    dod = R.dirs(d_out, 1)[:, :, :, 0]
    a = R.backward(fr["gates"], fr["c"], w_hh, dod)["dG"]
    z = R.backward(fr["gates"], fr["c"], w_hh, dod, dc_no_f=True)["dG"]
    assert (a - z).abs().max() > 1e-3


# ------------------------------------------------------------------------------------------------------- attention
def attn_case(B, N, D, Q, mask_kind, seed):
    g = torch.Generator().manual_seed(seed)
    dec = QueryDecoderRef(D, Q).double()
    memory = torch.randn(B, N, D, generator=g, dtype=F64)
    traces = torch.randn(B, N, 11, generator=g, dtype=F64) * 2 + 1
    if mask_kind is None:
        mask = None
    else:
        mask = torch.rand(B, N, generator=g) < 0.7
        mask[:, 0] = True
        if mask_kind == "dead":
            mask[1] = False
    return dec, memory, traces, mask


@pytest.mark.parametrize("mask_kind", [None, "rand", "dead"])
@pytest.mark.parametrize("D,Q,N", [(32, 5, 17), (64, 33, 40)])
def test_attention_reference_against_autograd(mask_kind, D, Q, N):
    B = 3
    dec, memory, traces, mask = attn_case(B, N, D, Q, mask_kind, D + Q + N)
    valid = mask if mask is not None else torch.ones(B, N, dtype=torch.bool)
    mean, rms, count = R.trace_stats(traces, mask, fp32=False)
    g = torch.Generator().manual_seed(7)
    d_feat = torch.randn(B, Q, D, generator=g, dtype=F64)
    d_anchor = torch.randn(B, Q, 3, generator=g, dtype=F64)
    d_summary = torch.randn(B, D, generator=g, dtype=F64)

    # the oracle decoder's attention over the traces with a valid token, differentiated by autograd
    live = valid.any(1)
    mem = memory[live].clone().requires_grad_(True)
    q = dec.q_proj(dec.query_embed.weight).detach()
    k, v = dec.k_proj(mem), dec.v_proj(mem)
    logits = torch.einsum("qd,bnd->bqn", q, k) * dec.inv_temp / dec.scale
    logits = logits.masked_fill(~valid[live][:, None, :], float("-inf"))
    attn = torch.softmax(logits, -1)
    feat = attn @ v
    anchor = attn @ ((traces[live][..., :3] - mean[live][:, None]) / rms[live][:, None, None])
    summary = (mem * valid[live][..., None]).sum(1) / count[live][:, None]
    loss = (feat * d_feat[live]).sum() + (anchor * d_anchor[live]).sum() + (summary * d_summary[live]).sum()
    loss.backward()

    # the folded form the kernels compute
    tau = (dec.inv_temp / dec.scale).detach()
    qk = (q @ dec.k_proj.weight).detach() * tau
    qb = (q * dec.k_proj.bias).sum(-1).detach() * tau
    fw = R.attn_fwd(memory, qk, qb, traces, mask, mean, rms)
    Wv, bv = dec.v_proj.weight.detach(), dec.v_proj.bias.detach()
    tol = 1e-12
    assert ((fw["ctx"] @ Wv.t() + bv)[live] - feat.detach()).abs().max() < tol
    assert (fw["anchor"][live] - anchor.detach()).abs().max() < tol
    assert (fw["summary"][live] - summary.detach()).abs().max() < tol
    lse = torch.logsumexp(logits.detach(), -1)
    st = fw["stats"]
    assert ((st[..., 0] + torch.log(st[..., 1]))[live] - lse).abs().max() < tol
    d_ctx = d_feat @ Wv
    d_ctx[~live] = 0
    d_anc = d_anchor.clone()
    d_anc[~live] = 0
    bw = R.attn_bwd(memory, qk, fw, count, d_ctx, d_anc, d_summary)
    assert (bw["d_memory"][live] - mem.grad).abs().max() < 1e-11
    assert (tau * q.t() @ bw["dqk"] - dec.k_proj.weight.grad).abs().max() < 1e-11
    assert (tau * q.t() @ bw["dqb"] - dec.k_proj.bias.grad).abs().max() < 1e-11
    if mask_kind == "dead":         # the documented outputs of a trace without a valid token
        assert bool(torch.isnan(fw["ctx"][1]).all() and torch.isnan(fw["anchor"][1]).all())
        assert bool((fw["summary"][1] == 0).all())
        assert bool((st[1, :, 0] == float("-inf")).all() and (st[1, :, 1] == 0).all())
        bw2 = R.attn_bwd(memory, qk, fw, count, torch.randn(B, Q, D, dtype=F64), torch.randn(B, Q, 3, dtype=F64))
        assert bool((bw2["d_memory"][1] == 0).all()) and bool(torch.isfinite(bw2["dqk"]).all())


@pytest.mark.parametrize("mask_kind", [None, "rand", "dead"])
def test_trace_stats_reference(mask_kind):
    _, _, traces, mask = attn_case(4, 300, 32, 1, mask_kind, 3)
    valid = mask if mask is not None else torch.ones(4, 300, dtype=torch.bool)
    mean_w, rms_w = TraceEncoderRef.stats(traces, valid)
    mean, rms, count = R.trace_stats(traces, mask, fp32=False)
    assert (mean - mean_w[:, 0]).abs().max() < 1e-12
    assert (rms - rms_w[:, 0, 0]).abs().max() < 1e-12
    assert torch.equal(count, valid.sum(1).clamp_min(1).to(F64))
    m32, r32, _ = R.trace_stats(traces.float(), mask, fp32=True)
    assert torch.equal(m32, m32.float().double()) and torch.equal(r32, r32.float().double())
    assert torch.allclose(m32, mean, rtol=1e-6, atol=1e-6) and torch.allclose(r32, rms, rtol=1e-6, atol=1e-6)
