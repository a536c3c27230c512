"""fp64 reference of ub_gemm_bf16 (include/unite_b200.h) and the per-element error bounds its outputs are judged by.

The reference restates the header: C[m, n] = epilogue(sum_k A[m, k] B[n, k]) with the operands read through their storage
(K-major: A[m, k] = A_st[m, k]; MN-major: A[m, k] = A_st[k, m]; the same for B) and, for a grouped GEMM, row m of group
g = m // group_rows reading A at (m - g a_m, k + g a_k), B at (n + g b_n, k + g b_k) and the bias at n + g bias.  The epilogue
runs in the kernel's order: LayerNorm fold -> bias -> activation (QuickGELU, GELU, DGELU) -> row_scale -> residual or
accumulate -> one rounding to C's type.  Inputs are the library's (bf16 / fp16 operands, fp32 bias, ...); everything here is fp64
and runs on whatever device the inputs are on.

Every output element gets its own bound, the sum of
    fp32 accumulation   K 2^-23 (|A| |B|^T)_mn      (recursive fp32 summation of exact products, twice the unit roundoff)
    epilogue arithmetic 2^-23 of each fp32 intermediate, and the LayerNorm statistics' cancellation
    approximations      |form - exact| + 2^-10 sensitivity: the tanh form of GELU / GELU' the default build evaluates with
                        tanh.approx (within 4.7e-4 of GELU, DESIGN §2; QuickGELU's tanh form is exact), 2^-10 on tanh.approx
    output rounding     2^-8 |C| for bf16 (8 significant bits), 2^-11 for fp16, 2^-24 for fp32
propagated through the later steps (GELU's slope is at most 1.13).  Column sums, row statistics and head dot products have
their own bounds (summation order and count).  No norms: one element outside its bound fails.
"""
import math

import torch

ACT_NONE, ACT_QUICKGELU, ACT_GELU, ACT_DGELU, ACT_DOT_AUX = 0, 1, 2, 3, 4
UNIT = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float32: 2.0 ** -24}
F32_OP = 2.0 ** -23                 # one fp32 rounding, with a factor 2 of margin
TANH_APPROX = 2.0 ** -10            # tanh.approx.f32 (2^-11 in the PTX ISA), with a factor 2 of margin
GELU_TANH_FORM = 4.74e-4            # max |tanh form - erf form| of GELU, at x = 2.70 (DESIGN §2: 4.7e-4)
GELU_SLOPE = 1.13                   # max |GELU'| and max |QuickGELU'|
F64 = torch.float64
SQRT2 = math.sqrt(2.0)


# ---------------------------------------------------------------------------------------------------------------- activations
def gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / SQRT2))


def gelu_grad(x):
    return 0.5 * (1.0 + torch.erf(x / SQRT2)) + x * torch.exp(-0.5 * x * x) / math.sqrt(2.0 * math.pi)


def quick_gelu(x):
    return x * torch.sigmoid(1.702 * x)


def _tanh_form(x):
    return torch.tanh(x * (0.7978845608 + 0.0356774081 * x * x)), 0.7978845608 + 0.1070322243 * x * x


def gelu_tanh_form(x):
    """GELU as the default build evaluates it (csrc/common.cuh), in fp64."""
    t, _ = _tanh_form(x)
    return 0.5 * x * (1.0 + t)


def gelu_grad_tanh_form(x):
    t, dudx = _tanh_form(x)
    return 0.5 * (1.0 + t) + 0.5 * x * (1.0 - t * t) * dudx


def act_bound(act, x):
    """Bound of |kernel activation - exact activation| at the fp32 input x (fp64 tensor), beyond fp32 rounding."""
    if act == ACT_GELU:
        return (gelu_tanh_form(x) - gelu(x)).abs() + 0.5 * TANH_APPROX * x.abs()
    if act == ACT_QUICKGELU:                  # 0.5 x (1 + tanh(0.851 x)) is x sigmoid(1.702 x) exactly
        return 0.5 * TANH_APPROX * x.abs()
    raise ValueError(act)


def dgelu_bound(x):
    """Bound of |kernel gelu'(x) - gelu'(x)|: the tanh form's own error and tanh.approx's, through d gelu'/d tanh."""
    _, dudx = _tanh_form(x)
    return (gelu_grad_tanh_form(x) - gelu_grad(x)).abs() + TANH_APPROX * (0.5 + x.abs() * dudx)


# ---------------------------------------------------------------------------------------------------------------- operands
def operand_views(A, a_mn, B, b_mn, M, N, K, group=None):
    """[(rows, A_g [rows, K], B_g [N, K], bias offset)] per group, fp64; one entry for an ungrouped GEMM."""
    gr = group["rows"] if group else M
    out = []
    for g in range(M // gr):
        ak, am, bk, bn, bo = ((g * group.get(x, 0)) for x in ("a_k", "a_m", "b_k", "b_n", "bias")) if group else (0,) * 5
        m0 = g * gr - am
        a = A[ak:ak + K, m0:m0 + gr].t() if a_mn else A[m0:m0 + gr, ak:ak + K]
        b = B[bk:bk + K, bn:bn + N].t() if b_mn else B[bn:bn + N, bk:bk + K]
        assert a.shape == (gr, K) and b.shape == (N, K), "operand storage too small for the group layout"
        out.append((slice(g * gr, (g + 1) * gr), a.to(F64), b.to(F64), bo))
    return out


# ---------------------------------------------------------------------------------------------------------------- the GEMM
def gemm(A, B, M, N, K, a_mn=False, b_mn=False, *, bias=None, act=ACT_NONE, aux_in=None, row_scale=None, rows_per_scale=1,
         residual=None, c_in=None, out_dtype=torch.bfloat16, split_k=1, ln=None, colsum_in=None, group=None):
    """Exact result of ub_gemm_bf16 and its bounds.  ln = (stats fp32 [M,2], c fp32 [N], inv_d, eps); c_in: C before an
    accumulating call; colsum_in: colsum_out before the call.  Returns a dict of fp64 tensors: c / c_bound, and aux / aux_bound
    (GELU's pre-activation copy) and colsum / colsum_bound where they apply."""
    dev = A.device
    acc = torch.empty(M, N, dtype=F64, device=dev)
    mag = torch.empty_like(acc)                    # (|A| |B|^T)_mn
    bias_m = torch.zeros_like(acc) if bias is not None else None
    for rows, a, b, bo in operand_views(A, a_mn, B, b_mn, M, N, K, group):
        acc[rows] = a @ b.t()
        mag[rows] = a.abs() @ b.abs().t()
        if bias is not None:
            bias_m[rows] = bias[bo:bo + N].to(F64)[None, :]
    v, e = acc, K * F32_OP * mag
    if ln is not None:
        stats, c, inv_d, eps = ln
        st = stats.to(F64)
        mu, ex2 = st[:, 0:1] * inv_d, st[:, 1:2] * inv_d
        var = (ex2 - mu * mu).clamp_min(0.0)
        rstd = 1.0 / torch.sqrt(var + eps)
        rel = F32_OP * (ex2 + mu * mu) / (var + eps) + 4 * F32_OP       # fp32 variance cancellation, rsqrtf
        mc = mu * c.to(F64)[None, :]
        v = rstd * (acc - mc)
        e = rstd * e + rel * v.abs() + 2 * F32_OP * rstd * (acc.abs() + mc.abs())
    if bias_m is not None:
        v = v + bias_m
        e = e + F32_OP * v.abs()
    out = {}
    if act in (ACT_GELU, ACT_QUICKGELU):
        if act == ACT_GELU:
            out["aux"], out["aux_bound"] = v, e * (1 + UNIT[torch.bfloat16]) + UNIT[torch.bfloat16] * v.abs()
        y = gelu(v) if act == ACT_GELU else quick_gelu(v)
        e = GELU_SLOPE * e + act_bound(act, v) + F32_OP * y.abs()
        v = y
    elif act == ACT_DGELU:
        x = aux_in.to(F64)
        g = gelu_grad(x)
        y = v * g
        e = e * g.abs() + v.abs() * dgelu_bound(x) + F32_OP * y.abs()
        v = y
    if row_scale is not None:
        s = row_scale.to(F64)[torch.arange(M, device=dev) // rows_per_scale][:, None]
        v = v * s
        e = e * s.abs() + F32_OP * v.abs()
    if colsum_in is not None:
        # per column: 31 adds inside a warp's 32-row slab, then one fp32 red.add per slab of every (padded) tile row
        n_add = 32 + 16 * -(-M // 512) + 1
        c0 = colsum_in.to(F64)
        out["colsum"] = c0 + v.sum(0)
        out["colsum_bound"] = e.sum(0) + n_add * F32_OP * (c0.abs() + v.abs().sum(0))
    if residual is not None:
        v = v + residual.to(F64)
        e = e + F32_OP * v.abs()
    if c_in is not None:
        c0 = c_in.to(F64)
        v = c0 + v
        e = e + (split_k + 1) * F32_OP * (c0.abs() + mag)
    u = UNIT[out_dtype]
    out["c"], out["c_bound"] = v, e * (1 + u) + u * v.abs()
    return out


def row_stats(c, stats_in):
    """stats_out of the fp16-residual epilogue: stats_in + row (sum, sumsq) of the written fp16 C, with its summation bound."""
    x = c.to(F64)
    s0 = stats_in.to(F64)
    n_add = x.shape[1] + 16
    ref = s0 + torch.stack([x.sum(1), (x * x).sum(1)], 1)
    bound = n_add * F32_OP * (s0.abs() + torch.stack([x.abs().sum(1), (x * x).sum(1)], 1))
    return ref, bound


def head_dot(c, aux, seq_len):
    """dot_out of UB_ACT_DOT_AUX: [M / seq_len, N / 64, seq_len] sums over each 64-column head of the written bf16 C times aux_in,
    with the bound of a 64-term fp32 fma chain."""
    M, N = c.shape
    p = (c.to(F64) * aux.to(F64)).view(M, N // 64, 64)
    ref = p.sum(-1).view(M // seq_len, seq_len, N // 64).permute(0, 2, 1)
    bound = 64 * F32_OP * p.abs().sum(-1).view(M // seq_len, seq_len, N // 64).permute(0, 2, 1)
    return ref, bound


def ratio(err, bound):
    """err / bound, with 0 / 0 = 0."""
    return torch.where(err == 0, torch.zeros_like(err), err / bound)
