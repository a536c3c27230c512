"""Typed torch-tensor front end of the C ABI (include/unite_b200.h).

Every function here checks dtype / device / contiguity, takes the raw pointers and the CURRENT torch CUDA stream
and calls straight into libunite_b200.so.  torch is used for memory and streams only — there is no torch
implementation of any op behind these functions, and no fallback.
"""
import ctypes as C
from typing import Optional

import torch

from . import _cabi
from ._cabi import lib, check, GemmEpilogue, UB_ACT_NONE, UB_ACT_QUICKGELU, UB_ACT_GELU, UB_ACT_DGELU, UB_ACT_DOT_AUX  # noqa: F401

BF16, F32, I32, U8 = torch.bfloat16, torch.float32, torch.int32, torch.uint8
F16 = torch.float16


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# ---- instrumentation: launch counter (bench.py's gpu_launches) and optional per-op CUDA-event timing ------------
LAUNCHES = 0          # kernels launched through this module since import
PROFILE = None        # set to a list to collect (name, info, start_event, end_event) per op on the launching stream


def _instrument(name, n_kernels):
    def deco(fn):
        def wrapped(*a, **k):
            global LAUNCHES
            LAUNCHES += n_kernels
            if PROFILE is None:
                return fn(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            info = None
            if name == "gemm" and fn.__name__ == "gemm_wgrad_multi":
                probs = a[0]                          # counted as one GEMM of sum(M_i * N_i) x 1 x K (same 2 M N K flops)
                info = (sum(gw.shape[0] * gw.shape[1] for _, _, gw in probs), 1, probs[0][0].shape[0], True, True, True)
            elif name == "gemm":
                out = a[2]
                K = k["group"]["K"] if k.get("group") else (a[0].shape[0] if k.get("a_t") else a[0].shape[1])
                info = (out.shape[0], out.shape[1], K, bool(k.get("a_t")), bool(k.get("b_t")), out.dtype == F32)
            PROFILE.append((name, info, e0, e1))
            return r
        wrapped.__name__, wrapped.__doc__ = fn.__name__, fn.__doc__
        return wrapped
    return deco


def _p(t: Optional[torch.Tensor], dtype=None, what="tensor") -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise _cabi.UBError(f"{what}: expected a CUDA tensor (unite_b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise _cabi.UBError(f"{what}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise _cabi.UBError(f"{what}: expected a contiguous tensor, got strides {t.stride()}")
    return t.data_ptr()


def _p2d(t: torch.Tensor, dtype, what):
    """2-D row-major view with arbitrary leading dimension."""
    if not t.is_cuda or t.dtype != dtype or t.dim() != 2 or t.stride(1) != 1:
        raise _cabi.UBError(f"{what}: expected a 2-D row-major CUDA {dtype} tensor, got {t.dtype} {tuple(t.shape)} {t.stride()}")
    return t.data_ptr(), t.stride(0)


@_instrument("gemm", 1)
def gemm(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor, *, a_t=False, b_t=False, bias=None, residual=None,
         row_scale=None, rows_per_scale=0, act=UB_ACT_NONE, aux_in=None, aux_out=None, accumulate=False, split_k=1, tile_ctas=0,
         max_ctas=0, ln_stats=None, ln_c=None, ln_eps=0.0, stats_out=None, colsum_out=None, group=None, dot_out=None, dot_seq_len=0):
    """out[M,N] = epilogue(A[M,K] @ B[N,K]^T).  a_t / b_t: the operand is stored transposed ([K,M] / [K,N]).
    A and B are both bf16 or both fp16.  ln_stats / ln_c: LayerNorm of A's rows folded into the epilogue (see the header);
    stats_out: row (sum, sumsq) of an fp16-residual output, accumulated.  colsum_out (DGELU epilogue): fp32 [N], += column sums
    of the output over its M rows (the bias gradient of the Linear whose pre-activation is aux_in).
    group: dict(rows=, K=, a_k=0, a_m=0, b_k=0, b_n=0, bias=0) — a grouped GEMM (see ub_gemm_epilogue.group_*): `out` stacks the
    groups' outputs along M, K is the per-group contraction length and the operands are addressed with the group offsets.
    act=UB_ACT_DOT_AUX with aux_in, dot_out (fp32 [M // dot_seq_len, N // 64, dot_seq_len]) and dot_seq_len: besides C, the per-(row,
    64-column head) dot product of the bf16 output with aux_in (D = rowsum(dO o O) for the attention backward, from the GEMM that
    produces dO)."""
    ab = F16 if a.dtype == F16 else BF16
    pa, lda = _p2d(a, ab, "gemm A")
    pb, ldb = _p2d(b, ab, "gemm B")
    if out.dtype not in (BF16, F32, F16):
        raise _cabi.UBError("gemm out: bf16, fp32 or (with an fp16 residual) fp16 expected")
    if out.dtype == F16 and (residual is None or residual.dtype != F16):
        raise _cabi.UBError("gemm out: fp16 output is only produced by the fp16-residual epilogue")
    pc, ldc = _p2d(out, out.dtype, "gemm C")
    M, N = out.shape
    ep = GemmEpilogue()
    if group is None:
        K = a.shape[0] if a_t else a.shape[1]
        am, bn = (a.shape[1] if a_t else a.shape[0]), (b.shape[1] if b_t else b.shape[0])
        bk = b.shape[0] if b_t else b.shape[1]
        if am != M or bn != N or bk != K:
            raise _cabi.UBError(f"gemm: shape mismatch A{tuple(a.shape)} a_t={a_t} B{tuple(b.shape)} b_t={b_t} C{tuple(out.shape)}")
    else:
        K, G = int(group["K"]), M // int(group["rows"])
        ep.group_rows, ep.group_a_k, ep.group_a_m = int(group["rows"]), int(group.get("a_k", 0)), int(group.get("a_m", 0))
        ep.group_b_k, ep.group_b_n, ep.group_bias = int(group.get("b_k", 0)), int(group.get("b_n", 0)), int(group.get("bias", 0))
        a_k_ext, a_m_ext = K + (G - 1) * ep.group_a_k, (ep.group_a_m or M)
        b_k_ext, b_n_ext = K + (G - 1) * ep.group_b_k, N + (G - 1) * ep.group_b_n
        if tuple(a.shape) != ((a_k_ext, a_m_ext) if a_t else (a_m_ext, a_k_ext)) or tuple(b.shape) != ((b_k_ext, b_n_ext) if b_t else (b_n_ext, b_k_ext)):
            raise _cabi.UBError(f"grouped gemm: operand shapes A{tuple(a.shape)} B{tuple(b.shape)} do not match the group layout {group} for C{tuple(out.shape)}")
    if bias is not None:
        if group is None and bias.numel() != N:
            raise _cabi.UBError("gemm bias: wrong length")
        ep.bias = _p(bias, F32, "gemm bias")
    if residual is not None:
        if residual.dtype == F16:
            if out.dtype != F16:
                raise _cabi.UBError("gemm: an fp16 residual needs an fp16 output (the teacher's residual stream)")
            ep.residual_f16 = 1
        pr, ldr = _p2d(residual, residual.dtype if residual.dtype == F16 else F32, "gemm residual")
        if tuple(residual.shape) != (M, N):
            raise _cabi.UBError("gemm residual: wrong shape")
        ep.residual, ep.ldr = pr, ldr
    if row_scale is not None:
        ep.row_scale = _p(row_scale, F32, "gemm row_scale")
        ep.rows_per_scale = rows_per_scale
    if aux_in is not None:
        px, ldx = _p2d(aux_in, BF16, "gemm aux_in")
        ep.aux_in, ep.ld_aux = px, ldx
    if aux_out is not None:
        px, ldx = _p2d(aux_out, BF16, "gemm aux_out")
        ep.aux_out, ep.ld_aux = px, ldx
    ep.act = act
    ep.out_fp32 = 1 if out.dtype == F32 else 0
    ep.accumulate = 1 if accumulate else 0
    ep.tile_ctas, ep.max_ctas = tile_ctas, max_ctas
    ep.ab_f16 = 1 if ab == F16 else 0
    if ln_stats is not None:
        if ln_c is None or ln_c.numel() != N or tuple(ln_stats.shape) != (M, 2):
            raise _cabi.UBError("gemm: ln_stats must be fp32 [M,2] and ln_c fp32 [N]")
        ep.ln_stats, ep.ln_c = _p(ln_stats, F32, "ln_stats"), _p(ln_c, F32, "ln_c")
        ep.ln_inv_d, ep.ln_eps = 1.0 / K, ln_eps
    if stats_out is not None:
        if tuple(stats_out.shape) != (M, 2):
            raise _cabi.UBError("gemm: stats_out must be fp32 [M,2]")
        ep.stats_out = _p(stats_out, F32, "stats_out")
    if colsum_out is not None:
        if colsum_out.numel() != N:
            raise _cabi.UBError("gemm: colsum_out must be fp32 [N]")
        ep.colsum_out = _p(colsum_out, F32, "colsum_out")
    if dot_out is not None:
        if act != UB_ACT_DOT_AUX or aux_in is None or dot_seq_len <= 0 or M % dot_seq_len or N % 64 or dot_out.numel() != M * (N // 64):
            raise _cabi.UBError("gemm: dot_out needs act=UB_ACT_DOT_AUX, aux_in, dot_seq_len dividing M and fp32 [M / S, N / 64, S]")
        ep.dot_out, ep.dot_seq_len = _p(dot_out, F32, "dot_out"), int(dot_seq_len)
    check(lib.ub_gemm_bf16(pa, lda, int(a_t), pb, ldb, int(b_t), pc, ldc, M, N, K, C.byref(ep), split_k, _stream()), "ub_gemm_bf16")
    return out


@_instrument("gemm", 1)
def gemm_wgrad_multi(problems, split_k=1):
    """problems: up to four (dy [K, M_i] bf16, x [K, N_i] bf16, gw [M_i, N_i] fp32): gw_i += dy_i^T x_i, one launch."""
    if not 1 <= len(problems) <= 4:
        raise _cabi.UBError("gemm_wgrad_multi: 1..4 problems")
    arr = (_cabi.GemmProblem * len(problems))()
    K = problems[0][0].shape[0]
    for i, (dy, x, gw) in enumerate(problems):
        pa, lda = _p2d(dy, BF16, "wgrad dy")
        pb, ldb = _p2d(x, BF16, "wgrad x")
        pc, ldc = _p2d(gw, F32, "wgrad out")
        if dy.shape[0] != K or x.shape[0] != K or tuple(gw.shape) != (dy.shape[1], x.shape[1]):
            raise _cabi.UBError(f"gemm_wgrad_multi: problem {i}: dy{tuple(dy.shape)} x{tuple(x.shape)} gw{tuple(gw.shape)}")
        arr[i].A, arr[i].lda, arr[i].B, arr[i].ldb, arr[i].C, arr[i].ldc = pa, lda, pb, ldb, pc, ldc
        arr[i].M, arr[i].N = gw.shape
    check(lib.ub_gemm_wgrad_multi(arr, len(problems), K, split_k, _stream()), "ub_gemm_wgrad_multi")


@_instrument("attn_fwd", 1)
def attn_fwd(qkv, o, lse, n_seq, S, H, scale):
    check(lib.ub_attn_fwd(_p(qkv, BF16, "qkv"), _p(o, BF16, "o"), _p(lse, F32, "lse"), n_seq, S, H, scale, _stream()), "ub_attn_fwd")


@_instrument("attn_bwd", 3)
def attn_bwd(qkv, o, d_o, lse, d_ws, dqkv, n_seq, S, H, scale, dbias=None):
    """dbias: optional fp32 [3*H*64], += column sums of the dq / dv thirds of dqkv (q_bias / v_bias gradients; the key third is untouched)."""
    if dbias is not None and dbias.numel() != 3 * H * 64:
        raise _cabi.UBError("attn_bwd dbias: fp32 [3*H*64] expected")
    if S <= 320:
        global LAUNCHES
        LAUNCHES -= 1          # D pre-pass + ONE backward kernel for resident items; longer sequences run the dK/dV and dQ passes
    if o is None:
        LAUNCHES -= 1          # D was written by the GEMM that produced d_o (gemm(..., act=UB_ACT_DOT_AUX, dot_out=d_ws)): no prep kernel
    check(lib.ub_attn_bwd(_p(qkv, BF16, "qkv"), _p(o, BF16, "o"), _p(d_o, BF16, "d_o"), _p(lse, F32, "lse"),
                          _p(d_ws, F32, "D_ws"), _p(dqkv, BF16, "dqkv"), _p(dbias, F32, "dbias"), n_seq, S, H, scale, _stream()), "ub_attn_bwd")


@_instrument("cls_attn", 1)
def cls_attn(qkv, out, n_seq, S, H, scale):
    check(lib.ub_cls_attn(_p(qkv, BF16, "qkv"), _p(out, F32, "attn"), n_seq, S, H, scale, _stream()), "ub_cls_attn")


@_instrument("layernorm_fwd", 1)
def layernorm_fwd(x, gamma, beta, eps, out, *, src_rows=None, post_add=None, post_idx=None):
    rows, D = out.shape
    if x.dtype not in (F32, F16):
        raise _cabi.UBError(f"ln x: fp32 or fp16 rows expected, got {x.dtype}")
    check(lib.ub_layernorm_fwd(_p(x, None, "ln x"), 1 if x.dtype == F16 else 0, _p(src_rows, I32, "src_rows"), _p(gamma, F32, "gamma"), _p(beta, F32, "beta"),
                               eps, _p(post_add, F32, "post_add"), _p(post_idx, I32, "post_idx"), _p(out, None, "ln out"),
                               1 if out.dtype == F32 else 0, rows, D, _stream()), "ub_layernorm_fwd")
    return out


@_instrument("teacher_embed_ln", 1)
def teacher_embed_ln(E, cls, pos, gamma, beta, eps, out, frames, P, D, stats=None):
    check(lib.ub_teacher_embed_ln(_p(E, F32, "E"), _p(cls, F32, "cls"), _p(pos, F32, "pos"), _p(gamma, F32, "gamma"),
                                  _p(beta, F32, "beta"), eps, _p(out, None, "out"), 1 if out.dtype == F16 else 0,
                                  _p(stats, F32, "stats"), frames, P, D, _stream()),
          "ub_teacher_embed_ln")


@_instrument("layernorm_bwd", 1)
def layernorm_bwd(dy, x, gamma, eps, dx_in, dx_out, dxs_out, row_scale, rows_per_scale, dgamma, dbeta, dsum=None):
    rows, D = x.shape
    check(lib.ub_layernorm_bwd(_p(dy, BF16, "dy"), _p(x, F32, "x"), _p(gamma, F32, "gamma"), eps, _p(dx_in, F32, "dx_in"),
                               _p(dx_out, F32, "dx_out"), _p(dxs_out, BF16, "dxs_out"), _p(row_scale, F32, "row_scale"),
                               rows_per_scale, _p(dgamma, F32, "dgamma"), _p(dbeta, F32, "dbeta"), _p(dsum, F32, "dsum"), rows, D,
                               _stream()),
          "ub_layernorm_bwd")


@_instrument("dec_tail_fwd", 1)
def dec_tail_fwd(y, gamma, beta, eps, out, tgt=None, loss_acc=None, loss_scale=0.0, loss_rows=None):
    """loss_rows = (lo, hi): only these rows enter the loss (clip_loss_data 'source' / 'target'); None = all."""
    rows, D = y.shape
    lo, hi = loss_rows if loss_rows is not None else (0, rows)
    check(lib.ub_dec_tail_fwd(_p(y, F32, "y"), _p(gamma, F32, "gamma"), _p(beta, F32, "beta"), eps, _p(out, F32, "out"),
                              _p(tgt, F32, "tgt"), _p(loss_acc, F32, "loss_acc"), loss_scale, lo, hi, rows, D, _stream()), "ub_dec_tail_fwd")


@_instrument("dec_tail_bwd", 1)
def dec_tail_bwd(y, gamma, beta, eps, go, go_scale, dy_out, dgamma, dbeta, go_rows=None):
    rows, D = y.shape
    lo, hi = go_rows if go_rows is not None else (0, rows)
    check(lib.ub_dec_tail_bwd(_p(y, F32, "y"), _p(gamma, F32, "gamma"), _p(beta, F32, "beta"), eps, _p(go, F32, "go"), go_scale, lo, hi,
                              _p(dy_out, BF16, "dy_out"), _p(dgamma, F32, "dgamma"), _p(dbeta, F32, "dbeta"), rows, D, _stream()),
          "ub_dec_tail_bwd")


@_instrument("l2norm_rows", 1)
def l2norm_rows(x):
    rows, D = x.shape
    check(lib.ub_l2norm_rows(_p(x, F32, "x"), rows, D, _stream()), "ub_l2norm_rows")


@_instrument("patchify", 1)
def patchify(x, out, tubelet):
    B, Cc, T, H, W = x.shape
    if Cc != 3:
        raise _cabi.UBError("patchify: 3 input channels expected")
    check(lib.ub_patchify(_p(x, F32, "videos"), _p(out, BF16, "patches"), B, T, H, W, tubelet, _stream()), "ub_patchify")
    return out


@_instrument("patchify_mix", 1)
def patchify_mix(x, out, mix, tubelet):
    """patchify of the batch-mode mixup / cutmix of x, x untouched.  mix: device fp32 [10] (see ub_patchify_mix; built by
    unite_b200.mixup)."""
    B, Cc, T, H, W = x.shape
    if Cc != 3:
        raise _cabi.UBError("patchify_mix: 3 input channels expected")
    if mix.numel() < 10:
        raise _cabi.UBError("patchify_mix: mix must hold 10 floats")
    check(lib.ub_patchify_mix(_p(x, F32, "videos"), _p(out, BF16, "patches"), _p(mix, F32, "mix"), B, T, H, W, tubelet, _stream()),
          "ub_patchify_mix")
    return out


IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)      # kinetics_sparse.py:241-243


@_instrument("patchify", 1)
def patchify_u8(x, out, tubelet, mean=IMAGENET_MEAN, std=IMAGENET_STD):
    """x uint8 [B,T,H,W,3] (decoder layout) -> normalised bf16 im2col rows (ToTensor + tensor_normalize + permute + patchify)."""
    if x.dim() != 5 or x.shape[-1] != 3 or not x.is_contiguous():
        raise _cabi.UBError(f"patchify_u8: contiguous uint8 [B,T,H,W,3] expected, got {tuple(x.shape)}")
    B, T, H, W, _ = x.shape
    m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
    check(lib.ub_patchify_u8(_p(x, U8, "frames"), _p(out, BF16, "patches"), m3, s3, B, T, H, W, tubelet, _stream()), "ub_patchify_u8")
    return out


@_instrument("patchify_mix", 1)
def patchify_mix_u8(x, out, mix, tubelet, mean=IMAGENET_MEAN, std=IMAGENET_STD):
    """patchify_mix of the clip patchify_u8 normalises from x uint8 [B,T,H,W,3]: normalised, then mixed by the device draw mix
    (fp32 [10], see patchify_mix); x untouched."""
    if x.dim() != 5 or x.shape[-1] != 3 or not x.is_contiguous():
        raise _cabi.UBError(f"patchify_mix_u8: contiguous uint8 [B,T,H,W,3] expected, got {tuple(x.shape)}")
    if mix.numel() < 10:
        raise _cabi.UBError("patchify_mix_u8: mix must hold 10 floats")
    B, T, H, W, _ = x.shape
    m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
    check(lib.ub_patchify_mix_u8(_p(x, U8, "frames"), _p(out, BF16, "patches"), _p(mix, F32, "mix"), m3, s3, B, T, H, W, tubelet,
                                 _stream()), "ub_patchify_mix_u8")
    return out


@_instrument("patchify_aug", 1)
def patchify_aug_u8(x, out, draw, crop_size, tubelet, erase_mode=0, mix=None, noise=None, rng=None, seed=0, mean=IMAGENET_MEAN,
                    std=IMAGENET_STD):
    """Rows of the stage-2 training crop, flip and random erasing of decoded uint8 frames x [B,T,H,W,3] (any H, W), normalised on the
    way: out bf16 [B*(T/tubelet)*(crop_size/16)^2, 3*tubelet*256].  draw: device int32 [B,10] per-clip draws (augment.AugBuffer.draw);
    erase_mode 0 const, 1 rand, 2 pixel; noise: fp32 [B,T,3] (rand) or [B,T,3,S,S] (pixel) normals in place of the generator, whose
    counter rng (device int64 [2]) the launch advances; mix: ub_patchify_mix's device draw (fp32 [10]) or None.  x is not written."""
    if x.dim() != 5 or x.shape[-1] != 3 or not x.is_contiguous():
        raise _cabi.UBError(f"patchify_aug_u8: contiguous uint8 [B,T,H,W,3] expected, got {tuple(x.shape)}")
    B, T, H, W, _ = x.shape
    S = int(crop_size)
    if tuple(draw.shape) != (B, 10):
        raise _cabi.UBError(f"patchify_aug_u8: draw must be int32 [{B}, 10], got {tuple(draw.shape)}")
    if mix is not None and mix.numel() < 10:
        raise _cabi.UBError("patchify_aug_u8: mix must hold 10 floats")
    if noise is not None and tuple(noise.shape) != ((B, T, 3) if erase_mode == 1 else (B, T, 3, S, S)):
        raise _cabi.UBError(f"patchify_aug_u8: noise of shape {tuple(noise.shape)} does not fit erase mode {erase_mode}")
    if rng is not None and (rng.dtype != torch.int64 or rng.numel() != 2):
        raise _cabi.UBError("patchify_aug_u8: rng must be a device int64 [2] counter")
    n_tok = B * (T // tubelet) * (S // 16) ** 2
    if tuple(out.shape) != (n_tok, 3 * tubelet * 256):
        raise _cabi.UBError(f"patchify_aug_u8: out must be [{n_tok}, {3 * tubelet * 256}], got {tuple(out.shape)}")
    m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
    check(lib.ub_patchify_aug_u8(_p(x, U8, "frames"), _p(out, BF16, "patches"), _p(draw, I32, "draw"), _p(mix, F32, "mix"), int(erase_mode),
                                 _p(noise, F32, "noise"), int(seed) & 0xFFFFFFFFFFFFFFFF, _p(rng, torch.int64, "rng"), m3, s3, B, T, H, W, S,
                                 tubelet, _stream()), "ub_patchify_aug_u8")
    return out


def clip_shape(x, paired=False, crop_size=None):
    """The [B,3,T,H,W] shape of the clip a batch stands for: an fp32 clip's own shape, or that of the clip decoded uint8 frames
    [B,T,H,W,3] normalise to.  A uint8 batch that patchify_u8 / patchify_mix_u8 cannot read raises ValueError here, before any
    launch: not contiguous [B,T,H,W,3], H or W not a multiple of 16, or (paired: clip b is mixed with clip B-1-b) an odd batch.
    crop_size S (a spatial augmentation, patchify_aug_u8): the batch must be uint8 frames, of any H, W, and stands for the augmented
    clip [B,3,T,S,S]."""
    if crop_size is not None and x.dtype != U8:
        raise ValueError(f"the spatial augmentation runs on decoded uint8 frames [B,T,H,W,3]; got a {x.dtype} batch (a loader that "
                         "augments on the host feeds the augmented fp32 clip without spatial_aug)")
    if x.dtype != U8:
        return tuple(x.shape)
    if x.dim() != 5 or x.shape[-1] != 3:
        raise ValueError(f"uint8 batches are decoded frames [B,T,H,W,3] (channels last); got shape {tuple(x.shape)}")
    if not x.is_contiguous():
        raise ValueError(f"uint8 frames must be contiguous; got shape {tuple(x.shape)} with strides {x.stride()}")
    B, T, H, W, _ = x.shape
    if crop_size is None and (H % 16 or W % 16):
        raise ValueError(f"uint8 frames of {H}x{W} pixels: H and W must be multiples of the 16-pixel patch")
    if paired and B % 2:
        raise ValueError(f"mixup: the batch size must be even (clip b is mixed with clip B-1-b), got {B}")
    return (B, 3, T, H, W) if crop_size is None else (B, 3, T, crop_size, crop_size)


def padded_k(features: int) -> int:
    """Row pitch of resize_patchify's output: the im2col width rounded up to 64 elements (one GEMM K block; also keeps the
    rows 16-byte aligned for TMA, which 3*14*14 = 588 bf16 would not be)."""
    return (features + 63) // 64 * 64


@_instrument("resize_patchify", 1)
def resize_patchify(x, out, resolution, patch, tubelet, mean=IMAGENET_MEAN, std=IMAGENET_STD):
    """Teacher im2col rows of a clip seen at `resolution` x `resolution` with `patch`-pixel patches.
    x: fp32 clip [B,3,T,H,W], or decoded uint8 frames [B,T,H,W,3] (normalised with mean / std before the resize).
    out: bf16 [B*(T/tubelet)*(resolution/patch)^2, ld], ld >= 3*tubelet*patch^2 (columns past that are written as zeros).
    When resolution != H or W the clip is resized as F.interpolate(mode="bicubic", align_corners=False) does."""
    if x.dtype == U8:
        if x.dim() != 5 or x.shape[-1] != 3:
            raise _cabi.UBError(f"resize_patchify: uint8 frames [B,T,H,W,3] expected, got {tuple(x.shape)}")
        B, T, H, W, _ = x.shape
    else:
        if x.dim() != 5 or x.shape[1] != 3:
            raise _cabi.UBError(f"resize_patchify: fp32 clip [B,3,T,H,W] expected, got {tuple(x.shape)}")
        B, _, T, H, W = x.shape
    n_tok = B * (T // tubelet) * (resolution // patch) ** 2
    if out.dim() != 2 or out.shape[0] != n_tok:
        raise _cabi.UBError(f"resize_patchify: out must be [{n_tok}, ld], got {tuple(out.shape)}")
    m3, s3 = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
    check(lib.ub_resize_patchify(_p(x, U8 if x.dtype == U8 else F32, "videos"), int(x.dtype == U8), m3, s3, _p(out, BF16, "patches"),
                                 out.shape[1], B, T, H, W, resolution, patch, tubelet, _stream()), "ub_resize_patchify")
    return out


@_instrument("mask_select", 1)
def mask_select(attn, q, mask, vis_idx, tea_rows, T, k, n_vis):
    frames, P = attn.shape
    check(lib.ub_mask_select(_p(attn, F32, "attn"), _p(q, F32, "q"), _p(mask, U8, "mask"), _p(vis_idx, I32, "vis_idx"),
                             _p(tea_rows, I32, "tea_rows"), frames, P, T, k, n_vis, _stream()), "ub_mask_select")


@_instrument("gather_rows", 1)
def gather_rows(src, idx, out, rows_per_group=0, group_stride_rows=0):
    n_rows = idx.numel()
    row_bytes = out.shape[-1] * out.element_size()
    check(lib.ub_gather_rows(_p(src, out.dtype, "gather src"), _p(idx, I32, "gather idx"), _p(out, None, "gather out"), n_rows,
                             row_bytes, rows_per_group, group_stride_rows, _stream()), "ub_gather_rows")
    return out


@_instrument("colsum_bf16", 1)
def colsum_bf16(x, out, skip=(0, 0)):
    """out[n] += sum_m x[m, n]; columns skip[0] <= n < skip[1] are left untouched."""
    px, ld = _p2d(x, BF16, "colsum x")
    M, N = x.shape
    check(lib.ub_colsum_bf16(px, ld, _p(out, F32, "colsum out"), M, N, skip[0], skip[1], _stream()), "ub_colsum_bf16")


@_instrument("cast_scale_bf16", 1)
def cast_scale_bf16(x, out, row_scale=None, rows_per_scale=0):
    rows, D = x.shape
    check(lib.ub_cast_scale_bf16(_p(x, F32, "x"), _p(out, BF16, "out"), _p(row_scale, F32, "row_scale"), rows_per_scale, rows, D,
                                 _stream()), "ub_cast_scale_bf16")


@_instrument("sumsq", 1)
def sumsq(g, out):
    check(lib.ub_sumsq(_p(g, F32, "g"), g.numel(), _p(out, F32, "out"), _stream()), "ub_sumsq")


@_instrument("adamw", 1)
def adamw(p, g, m, v, w16, n_decay, lr, wd, beta1, beta2, eps, step, grad_scale=1.0):
    check(lib.ub_adamw(_p(p, F32, "p"), _p(g, F32, "g"), _p(m, F32, "m"), _p(v, F32, "v"), _p(w16, BF16, "w16"), p.numel(), n_decay,
                       lr, wd, beta1, beta2, eps, step, grad_scale, _stream()), "ub_adamw")


@_instrument("adamw", 1)
def adamw_dev(p, g, m, v, w16, n_decay, hyper, gnorm_sq=None):
    check(lib.ub_adamw_dev(_p(p, F32, "p"), _p(g, F32, "g"), _p(m, F32, "m"), _p(v, F32, "v"), _p(w16, BF16, "w16"), p.numel(), n_decay,
                           _p(hyper, F32, "hyper"), _p(gnorm_sq, F32, "gnorm_sq"), _stream()), "ub_adamw_dev")


@_instrument("adamw", 1)
def adamw_seg(p, g, m, v, w16, seg_end4, hyper, gnorm_sq=None):
    """Segmented AdamW: seg_end4 int32 [S] (device), hyper fp32 [8 + 2S] (device) — see include/unite_b200.h."""
    S = seg_end4.numel()
    if hyper.numel() != 8 + 2 * S:
        raise _cabi.UBError(f"adamw_seg: hyper has {hyper.numel()} floats, expected {8 + 2 * S}")
    check(lib.ub_adamw_seg(_p(p, F32, "p"), _p(g, F32, "g"), _p(m, F32, "m"), _p(v, F32, "v"), _p(w16, BF16, "w16"), p.numel(),
                           _p(seg_end4, I32, "seg_end4"), S, _p(hyper, F32, "hyper"), _p(gnorm_sq, F32, "gnorm_sq"), _stream()), "ub_adamw_seg")


@_instrument("sumsq", 1)
def sumsq_seg(g, seg_end4, hyper, out):
    check(lib.ub_sumsq_seg(_p(g, F32, "g"), g.numel(), _p(seg_end4, I32, "seg_end4"), seg_end4.numel(), _p(hyper, F32, "hyper"),
                           _p(out, F32, "out"), _stream()), "ub_sumsq_seg")


@_instrument("drop_path_draw", 1)
def drop_path_draw(rates, out, seed, step):
    """out fp32 [depth, 2, B] <- DropPath factors of one step; `step` int64 [1] device counter, advanced by the kernel."""
    depth, two, B = out.shape
    if two != 2 or rates.numel() != depth or step.dtype != torch.int64 or step.numel() != 1:
        raise _cabi.UBError("drop_path_draw: out [depth,2,B], rates [depth], step int64 [1] expected")
    check(lib.ub_drop_path_draw(_p(rates, F32, "rates"), _p(out, F32, "out"), depth, B, int(seed) & 0xFFFFFFFFFFFFFFFF, _p(step, torch.int64, "step"),
                                _stream()), "ub_drop_path_draw")
    return out


@_instrument("adamw_nvls", 1)
def adamw_nvls(p, g_mc, m, v, w16, w16_mc, n_decay, rank, world, hyper, gnorm_mc, flags, flags_mc, epoch, err, g_peers=None,
               w16_peers=None, stage_peers=None, prepushed=False):
    """g_mc / w16_mc / gnorm_mc / flags / flags_mc are raw addresses (ints): multicast mappings of symmetric allocations;
    g_peers / w16_peers: ctypes arrays of every rank's mapping of the gradient arena / shadow (or None)."""
    check(lib.ub_adamw_nvls(_p(p, F32, "p"), g_mc, _p(m, F32, "m"), _p(v, F32, "v"), _p(w16, BF16, "w16"), w16_mc, p.numel(), n_decay,
                            rank, world, _p(hyper, F32, "hyper"), gnorm_mc, flags, flags_mc, epoch.data_ptr(), err.data_ptr(),
                            None if g_peers is None else _cabi.C.addressof(g_peers),
                            None if w16_peers is None else _cabi.C.addressof(w16_peers),
                            None if stage_peers is None else _cabi.C.addressof(stage_peers), int(bool(prepushed)), _stream()),
          "ub_adamw_nvls")


@_instrument("cast_bf16", 1)
def cast_bf16(x, out):
    check(lib.ub_cast_bf16(_p(x, F32, "x"), _p(out, BF16, "out"), x.numel(), _stream()), "ub_cast_bf16")


@_instrument("ema_update", 1)
def ema_update(ema_params, ema_w16, params, decay):
    """ema_params = ema_params * decay + (1 - decay) * params in fp32 (timm ModelEma.update, bit for bit), and ema_w16 = its bf16
    shadow, in one pass.  decay is rounded to fp32 and 1 - decay is computed in double first, as torch does with the scalars."""
    n = ema_params.numel()
    if params.numel() != n or ema_w16.numel() != n:
        raise _cabi.UBError(f"ema_update: ema {n}, shadow {ema_w16.numel()} and params {params.numel()} elements differ")
    check(lib.ub_ema_update(_p(ema_params, F32, "ema_params"), _p(ema_w16, BF16, "ema_w16"), _p(params, F32, "params"), n, float(decay),
                            float(1.0 - decay), _stream()), "ub_ema_update")


@_instrument("meanpool_fwd", 1)
def meanpool_fwd(x, out):
    B, N, D = x.shape
    check(lib.ub_meanpool_fwd(_p(x, F32, "x"), _p(out, F32, "out"), B, N, D, _stream()), "ub_meanpool_fwd")
    return out


@_instrument("meanpool_bwd", 1)
def meanpool_bwd(g, dx):
    B, N, D = dx.shape
    check(lib.ub_meanpool_bwd(_p(g, F32, "g"), _p(dx, F32, "dx"), B, N, D, _stream()), "ub_meanpool_bwd")
    return dx


@_instrument("linear_small_fwd", 1)
def linear_small_fwd(x, W, bias, out):
    B, D = x.shape
    Cc = W.shape[0]
    check(lib.ub_linear_small_fwd(_p(x, F32, "x"), _p(W, F32, "W"), _p(bias, F32, "bias"), _p(out, F32, "out"), B, Cc, D, _stream()),
          "ub_linear_small_fwd")
    return out


@_instrument("linear_small_bwd", 1)
def linear_small_bwd(x, W, dout, dx, dW, db):
    B, D = x.shape
    Cc = W.shape[0]
    check(lib.ub_linear_small_bwd(_p(x, F32, "x"), _p(W, F32, "W"), _p(dout, F32, "dout"), _p(dx, F32, "dx"), _p(dW, F32, "dW"),
                                  _p(db, F32, "db"), B, Cc, D, _stream()), "ub_linear_small_bwd")


@_instrument("softmax_ce", 1)
def softmax_ce(logits, labels, weights, scale, loss_acc, dlogits):
    B, Cc = logits.shape
    check(lib.ub_softmax_ce(_p(logits, F32, "logits"), _p(labels, I32, "labels"), _p(weights, F32, "weights"), scale,
                            _p(loss_acc, F32, "loss_acc"), _p(dlogits, F32, "dlogits"), B, Cc, _stream()), "ub_softmax_ce")


@_instrument("soft_target_ce", 1)
def soft_target_ce(logits, labels, mix, scale, loss_acc, dlogits):
    """Soft-target CE of the mixup target built on the device from labels and mix = device fp32 [lam, on, off]."""
    B, Cc = logits.shape
    if mix.numel() < 3:
        raise _cabi.UBError("soft_target_ce: mix must hold lam, on, off")
    check(lib.ub_soft_target_ce(_p(logits, F32, "logits"), _p(labels, I32, "labels"), _p(mix, F32, "mix"), scale,
                                _p(loss_acc, F32, "loss_acc"), _p(dlogits, F32, "dlogits"), B, Cc, _stream()), "ub_soft_target_ce")


@_instrument("clip_zero_shot", 1)
def clip_zero_shot(img_feat, text_feat, probs, T):
    BT, D = img_feat.shape
    Cc = text_feat.shape[0]
    check(lib.ub_clip_zero_shot(_p(img_feat, F32, "img_feat"), _p(text_feat, F32, "text_feat"), _p(probs, F32, "probs"), BT // T, T, Cc, D,
                                _stream()), "ub_clip_zero_shot")
    return probs


@_instrument("pseudo_label_fusion", 1)
def pseudo_label_fusion(logits_full, clip_probs, threshold, conf_weighted, msp, pseudo, sel, weight):
    B, Cc = logits_full.shape
    check(lib.ub_pseudo_label_fusion(_p(logits_full, F32, "logits_full"), _p(clip_probs, F32, "clip_probs"), threshold, int(conf_weighted),
                                     _p(msp, F32, "msp"), _p(pseudo, I32, "pseudo"), _p(sel, U8, "sel"), _p(weight, F32, "weight"), B, Cc,
                                     _stream()), "ub_pseudo_label_fusion")
