"""GPU: the tcgen05 GEMM entry points against torch.matmul (bf16 operands, fp32 accumulate)."""
import ctypes

import pytest
import torch

from roomslam_b200 import _lib, layout as L

pytestmark = pytest.mark.gpu


def st():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("M,N,K,bias", [(128, 128, 64, False), (1000, 256, 128, True), (20497, 768, 256, True)])
def test_gemm_bf16_nt_row_major(M, N, K, bias):
    torch.manual_seed(0)
    A = torch.randn(M, K, device="cuda").bfloat16(); B = torch.randn(N, K, device="cuda").bfloat16()
    b = torch.randn(N, device="cuda") if bias else None
    C = torch.full((M, N), 7.0, device="cuda").bfloat16()
    _lib.call("rs_gemm_bf16_nt", A.data_ptr(), K, B.data_ptr(), K, C.data_ptr(), N, b.data_ptr() if bias else 0, M, N, K, 0, st())
    ref = A.float() @ B.float().t() + (b if bias else 0)
    assert float((C.float() - ref).abs().max() / ref.abs().max()) < 6e-3       # bf16 output rounding


@pytest.mark.parametrize("rows,M,N,sa,sb,ca,cb", [(64, 128, 128, 0, 0, 0, 0), (5000, 256, 128, 1, 0, 0, 0),
                                                   (70000, 768, 256, 0, 1, 0, 0), (3000, 128, 128, 0, 0, 128, 256)])
def test_gemm_bf16_tn_row_major(rows, M, N, sa, sb, ca, cb):
    torch.manual_seed(1)
    lda, ldb = max(ca + M, 512 if ca else M), max(cb + N, 512 if cb else N)
    A = torch.randn(rows + 3, lda, device="cuda").bfloat16(); B = torch.randn(rows + 3, ldb, device="cuda").bfloat16()
    C = torch.ones(M, N, device="cuda")
    _lib.call("rs_gemm_bf16_tn_acc", A.data_ptr(), lda, A.shape[0], ca, sa, B.data_ptr(), ldb, B.shape[0], cb, sb,
              C.data_ptr(), N, M, N, rows, st())
    ref = 1.0 + A[sa:sa + rows, ca:ca + M].float().t() @ B[sb:sb + rows, cb:cb + N].float()
    assert float((C - ref).abs().max() / ref.abs().max()) < 1e-4


@pytest.mark.parametrize("B,T,Ca,kcols,N,Cc,c0", [(128, 1, 64, [0], 128, 128, 0), (200, 5, 256, [0, 64, 128, 192], 768, 768, 0),
                                                    (300, 7, 1024, [0, 64, 128, 192, 256, 320, 512, 576, 640, 704, 768, 832], 256, 256, 0),
                                                    (128, 3, 128, [64], 128, 512, 256),
                                                    (700, 60, 256, [0, 64, 128, 192], 768, 768, 0), (256, 149, 128, [0, 64], 256, 512, 128),
                                                    (1300, 40, 256, [64, 128, 192], 512, 1024, 256)])
def test_blk_gemm_nt_tile_major(B, T, Ca, kcols, N, Cc, c0):
    torch.manual_seed(2)
    x = torch.randn(B, T, Ca, device="cuda")
    xt = L.to_tile_major(x)
    K = len(kcols) * 64
    w = torch.randn(N, K, device="cuda") * 0.1
    b = torch.randn(N, device="cuda")
    ct = torch.zeros(L.n_tiles(B), T + 2, Cc // 8, 128, 8, device="cuda", dtype=torch.bfloat16)
    kch = L.int_array([c // 8 for c in kcols])
    _lib.call("rs_blk_gemm_nt", xt.data_ptr(), Ca, ctypes.addressof(kch), len(kcols), L.tile_weight_nt(w).data_ptr(), N // 128,
              ct.data_ptr(), Cc, c0 // 8, b.data_ptr(), xt.shape[0] * xt.shape[1], st())
    xa = torch.cat([x[..., c:c + 64] for c in kcols], -1).bfloat16().float()
    ref = xa @ w.bfloat16().float().t() + b
    got = L.from_tile_major(ct, B, T).float()
    assert float((got[..., c0:c0 + N] - ref).abs().max() / ref.abs().max()) < 6e-3
    got[..., c0:c0 + N] = 0
    assert float(got.abs().max()) == 0.0            # nothing written outside the requested columns


@pytest.mark.parametrize("shift", [0, -1, 1])
def test_blk_wgrad_tile_major_with_time_shift(shift):
    """rs_blk_wgrad with three roles on dG columns 0, 128 and 384 against the time-shifted B columns 128..255, no bias, no
    B2: C += sum over blocks dG_blk^T . B_blk'."""
    from roomslam_b200.functional_bf16 import _ones_block, _wgrad
    torch.manual_seed(3)
    B, T, Ca, Cb, n_cols = 300, 9, 1024, 256, 128
    mcols = [0, 128, 384]
    a = torch.randn(B, T, Ca, device="cuda"); b = torch.randn(B, T, Cb, device="cuda")
    at, bt = L.to_tile_major(a), L.to_tile_major(b)
    C = torch.ones(len(mcols) * 128, n_cols, device="cuda")
    roles = [(c // 8, bt, Cb, 128 // 8, n_cols, shift, C[i * 128:(i + 1) * 128], n_cols, None, None, None) for i, c in enumerate(mcols)]
    _wgrad(at, Ca, _ones_block(torch.device("cuda")), roles, at.shape[0], T, st())
    aa = torch.cat([a[..., c:c + 128] for c in mcols], -1).bfloat16().float()
    src = b[..., 128:128 + n_cols].bfloat16().float()
    bb = torch.zeros_like(src)
    if shift == 0:
        bb = src
    elif shift == -1:
        bb[:, 1:] = src[:, :-1]
    else:
        bb[:, :-1] = src[:, 1:]
    ref = 1.0 + torch.einsum("btm,btn->mn", aa, bb)
    assert float((C - ref).abs().max() / ref.abs().max()) < 1e-4


@pytest.mark.parametrize("M,N,K", [(5000, 512, 128), (4100, 128, 11), (9000, 128, 512)])
def test_bf16x6_split_gemm_is_fp32_grade(M, N, K):
    """rs_split_bf16x6 + rs_gemm_bf16_nt / rs_gemm_bf16_tn_acc against an fp64 matmul: error at the fp32 level."""
    from roomslam_b200.lstm_model import nt_tc, split3, tn_tc
    torch.manual_seed(M)
    a = torch.randn(M, K, device="cuda") * torch.rand(M, 1, device="cuda") * 10
    w = torch.randn(N, K, device="cuda")
    bias = torch.randn(N, device="cuda")
    a3, kp = split3(a)
    out = torch.empty(M, N, device="cuda")
    nt_tc(a3, split3(w, role_b=True)[0], bias, out)
    ref = a.double() @ w.double().t() + bias.double()
    # the tensor core truncates its fp32 accumulator at every K=16 step of the final (hi.hi) sixth: ~6e-8 x K/16
    assert float((out.double() - ref).abs().max() / ref.abs().max()) < 2e-6
    # hi + mid + lo reproduces x to 24 bits
    thirds = a3.view(M, 6, kp)[:, [0, 2, 5], :K].double().sum(1)            # lo, mid, hi sixths of the A role
    assert float((thirds - a.double()).abs().max() / a.abs().max()) < 2e-7
    # weight gradient: dW[N, K] = dY^T A with a one-row shift between the operands
    dy = torch.randn(M, N, device="cuda")
    dy3, kpy = split3(dy)
    dw = torch.zeros(N, kp, device="cuda")
    tn_tc(dy3, kpy, 0, N, a3, kp, kp, dw, a_shift=1, b_shift=0)
    ref_w = dy[1:].double().t() @ a[:-1].double()
    assert float((dw[:, :K].double() - ref_w).abs().max() / ref_w.abs().max()) < 5e-6
