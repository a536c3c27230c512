"""The fp64 GEMM reference of tests/gemm_ref.py against torch on the CPU: F.linear, LayerNorm + Linear for the fold, F.gelu and
its autograd gradient, and a loop over groups for the grouped addressing."""
import math

import pytest
import torch
import torch.nn.functional as F

from tests import gemm_ref as R

F64 = torch.float64


def _ab(M, N, K, seed, dtype=torch.bfloat16):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(M, K, generator=g).to(dtype), torch.randn(N, K, generator=g).to(dtype), g


@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, True)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_operand_majors_match_linear(a_mn, b_mn, dtype):
    M, N, K = 37, 24, 19
    A, B, g = _ab(M, N, K, 1, dtype)
    bias = torch.randn(N, generator=g)
    a_st = A.t().contiguous() if a_mn else A
    b_st = B.t().contiguous() if b_mn else B
    r = R.gemm(a_st, b_st, M, N, K, a_mn, b_mn, bias=bias, out_dtype=torch.float32)
    ref = F.linear(A.double(), B.double(), bias.double())
    assert torch.allclose(r["c"], ref, rtol=0, atol=1e-12)
    assert bool((r["c_bound"] > 0).all())


def test_strided_operands():
    M, N, K = 20, 16, 12
    A, B, _ = _ab(M, N, K + 5, 2)
    r = R.gemm(A[:, :K], B[:, 3:3 + K], M, N, K)
    assert torch.allclose(r["c"], A[:, :K].double() @ B[:, 3:3 + K].double().t(), rtol=0, atol=1e-12)


def test_layernorm_fold_matches_layer_norm_then_linear():
    M, N, K, eps = 33, 40, 64, 1e-5
    g = torch.Generator().manual_seed(3)
    x = (torch.randn(M, K, generator=g) * 2 + 0.7).half()
    gamma, beta = torch.rand(K, generator=g) + 0.5, torch.randn(K, generator=g) * 0.1
    W, b = torch.randn(N, K, generator=g) * 0.05, torch.randn(N, generator=g) * 0.1
    wg = (W * gamma).half()                                 # the folded weight the library is given, and its column sums
    stats = torch.stack([x.double().sum(1), (x.double() ** 2).sum(1)], 1).float()
    r = R.gemm(x, wg, M, N, K, bias=(W.double() @ beta.double() + b.double()), ln=(stats, wg.double().sum(1), 1.0 / K, eps),
               out_dtype=torch.float32)
    ref = F.linear(F.layer_norm(x.double(), (K,), None, None, eps), wg.double(), W.double() @ beta.double() + b.double())
    # the only difference: statistics rounded to fp32 by the producer of x
    assert (r["c"] - ref).abs().max().item() < 1e-5
    assert bool(((r["c"] - ref).abs() <= r["c_bound"]).all())


def test_gelu_and_its_autograd_gradient():
    x = torch.linspace(-8, 8, 4001, dtype=F64, requires_grad=True)
    y = F.gelu(x)
    y.sum().backward()
    assert torch.allclose(R.gelu(x.detach()), y.detach(), rtol=0, atol=1e-15)
    assert torch.allclose(R.gelu_grad(x.detach()), x.grad, rtol=0, atol=1e-14)
    xq = x.detach()
    assert torch.allclose(R.quick_gelu(xq), xq * torch.sigmoid(1.702 * xq), rtol=0, atol=0)
    # the documented accuracy of the default build's tanh form (DESIGN §2)
    assert (R.gelu_tanh_form(xq) - R.gelu(xq)).abs().max().item() <= R.GELU_TANH_FORM
    # GELU and QuickGELU slopes stay under the factor the bounds propagate input errors with
    xs = torch.linspace(-20, 20, 100001, dtype=F64)
    assert R.gelu_grad(xs).abs().max().item() <= R.GELU_SLOPE
    xq2 = xs.clone().requires_grad_()
    R.quick_gelu(xq2).sum().backward()
    assert xq2.grad.abs().max().item() <= R.GELU_SLOPE


@pytest.mark.parametrize("act", [R.ACT_GELU, R.ACT_QUICKGELU, R.ACT_DGELU])
def test_activation_epilogues_order(act):
    M, N, K = 16, 24, 8
    A, B, g = _ab(M, N, K, 4)
    bias = torch.randn(N, generator=g)
    rs = torch.tensor([0.0, 1.25, 0.5, 2.0])
    aux = torch.randn(M, N, generator=g).bfloat16()
    colsum0 = torch.randn(N, generator=g)
    pre = A.double() @ B.double().t() + (0 if act == R.ACT_DGELU else bias.double())
    if act == R.ACT_DGELU:
        y = pre * R.gelu_grad(aux.double())
    else:
        y = F.gelu(pre) if act == R.ACT_GELU else pre * torch.sigmoid(1.702 * pre)
    y = y * rs.double().repeat_interleave(4)[:, None]
    r = R.gemm(A, B, M, N, K, bias=None if act == R.ACT_DGELU else bias, act=act, aux_in=aux, row_scale=rs, rows_per_scale=4,
               colsum_in=colsum0 if act == R.ACT_DGELU else None)
    assert torch.allclose(r["c"], y, rtol=0, atol=1e-12)
    if act == R.ACT_GELU:
        assert torch.allclose(r["aux"], pre, rtol=0, atol=1e-12)
    if act == R.ACT_DGELU:
        assert torch.allclose(r["colsum"], colsum0.double() + y.sum(0), rtol=0, atol=1e-12)
    # zero-scaled rows are exact zeros, with a zero bound
    assert bool((r["c"][:4] == 0).all()) and bool((r["c_bound"][:4] == 0).all())


def test_residual_and_accumulate():
    M, N, K = 12, 16, 8
    A, B, g = _ab(M, N, K, 5)
    res = torch.randn(M, N, generator=g)
    c0 = torch.randn(M, N, generator=g)
    base = A.double() @ B.double().t()
    assert torch.allclose(R.gemm(A, B, M, N, K, residual=res, out_dtype=torch.float32)["c"], base + res.double(), rtol=0, atol=1e-12)
    r16 = R.gemm(A, B, M, N, K, residual=res.half(), out_dtype=torch.float16)
    assert torch.allclose(r16["c"], base + res.half().double(), rtol=0, atol=1e-12)
    acc = R.gemm(A.t().contiguous(), B.t().contiguous(), M, N, K, True, True, c_in=c0, out_dtype=torch.float32, split_k=3)
    assert torch.allclose(acc["c"], c0.double() + base, rtol=0, atol=1e-12)


def test_row_stats_and_head_dot():
    g = torch.Generator().manual_seed(6)
    c = torch.randn(6, 128, generator=g).half()
    s0 = torch.randn(6, 2, generator=g)
    ref, bound = R.row_stats(c, s0)
    x = c.double()
    assert torch.allclose(ref[:, 0], s0[:, 0].double() + x.sum(1)) and torch.allclose(ref[:, 1], s0[:, 1].double() + (x * x).sum(1))
    assert bool((bound > 0).all())
    cb, aux = torch.randn(6, 128, generator=g).bfloat16(), torch.randn(6, 128, generator=g).bfloat16()
    d, _ = R.head_dot(cb, aux, 3)                       # [2 sequences, 2 heads, 3 rows]
    p = cb.double() * aux.double()
    assert d.shape == (2, 2, 3)
    assert math.isclose(d[1, 0, 2].item(), p[5, :64].sum().item(), rel_tol=1e-14)
    assert math.isclose(d[0, 1, 1].item(), p[1, 64:].sum().item(), rel_tol=1e-14)


@pytest.mark.parametrize("form", ["fwd", "dgrad", "wgrad"])
def test_grouped_addressing_matches_a_loop_over_groups(form):
    """The three grouped calls of the decoders (modeling_adaptation.py): y_k = z_k W_k^T + b_k, dz_k = dy_k W_k and
    dW_k = dy_k^T z_k, each group stacked along M."""
    Kd, rows, D, Cc = 3, 8, 16, 24
    g = torch.Generator().manual_seed(7)
    z = torch.randn(Kd * rows, D, generator=g).bfloat16()          # decoder inputs, stacked
    dy = torch.randn(Kd * rows, Cc, generator=g).bfloat16()        # decoder output gradients, stacked
    W = torch.randn(Kd * Cc, D, generator=g).bfloat16()            # the K weights [C, D], stacked
    bias_stride = 32
    bias = torch.randn((Kd - 1) * bias_stride + Cc, generator=g)
    if form == "fwd":
        r = R.gemm(z, W, Kd * rows, Cc, D, bias=bias, group=dict(rows=rows, b_n=Cc, bias=bias_stride), out_dtype=torch.float32)
        ref = torch.cat([F.linear(z[k * rows:(k + 1) * rows].double(), W[k * Cc:(k + 1) * Cc].double(),
                                  bias[k * bias_stride:k * bias_stride + Cc].double()) for k in range(Kd)])
    elif form == "dgrad":
        r = R.gemm(dy, W, Kd * rows, D, Cc, False, True, group=dict(rows=rows, b_k=Cc))
        ref = torch.cat([dy[k * rows:(k + 1) * rows].double() @ W[k * Cc:(k + 1) * Cc].double() for k in range(Kd)])
    else:
        r = R.gemm(dy, z, Kd * Cc, D, rows, True, True, group=dict(rows=Cc, a_k=rows, a_m=Cc, b_k=rows), out_dtype=torch.float32)
        ref = torch.cat([dy[k * rows:(k + 1) * rows].double().t() @ z[k * rows:(k + 1) * rows].double() for k in range(Kd)])
    assert torch.allclose(r["c"], ref, rtol=0, atol=1e-12)
