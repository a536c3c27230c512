"""ctypes binding of the C ABI in include/unite_b200.h.

This is the only place the shared library is loaded.  It fails loudly (ImportError) when the library has
not been built — there is no Python/torch fallback for any op on the product path.
"""
import ctypes as C
import os

# UB_LIB_VARIANT=<suffix> loads lib/libunite_b200_<suffix>.so instead (A/B runs of two builds on one GPU box)
_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib",
                         "libunite_b200%s.so" % ("_" + os.environ["UB_LIB_VARIANT"] if os.environ.get("UB_LIB_VARIANT") else ""))

UB_ACT_NONE, UB_ACT_QUICKGELU, UB_ACT_GELU, UB_ACT_DGELU, UB_ACT_DOT_AUX = 0, 1, 2, 3, 4


class GemmEpilogue(C.Structure):
    _fields_ = [
        ("bias", C.c_void_p),
        ("residual", C.c_void_p),
        ("row_scale", C.c_void_p),
        ("aux_in", C.c_void_p),
        ("aux_out", C.c_void_p),
        ("ldr", C.c_int64),
        ("ld_aux", C.c_int64),
        ("rows_per_scale", C.c_int32),
        ("act", C.c_int32),
        ("out_fp32", C.c_int32),
        ("accumulate", C.c_int32),
        ("tile_ctas", C.c_int32),
        ("max_ctas", C.c_int32),
        ("residual_f16", C.c_int32),
        ("ab_f16", C.c_int32),
        ("ln_stats", C.c_void_p),
        ("ln_c", C.c_void_p),
        ("stats_out", C.c_void_p),
        ("ln_inv_d", C.c_float),
        ("ln_eps", C.c_float),
        ("colsum_out", C.c_void_p),
        ("group_rows", C.c_int32),
        ("group_a_k", C.c_int32),
        ("group_a_m", C.c_int32),
        ("group_b_k", C.c_int32),
        ("group_b_n", C.c_int32),
        ("group_bias", C.c_int32),
        ("dot_out", C.c_void_p),
        ("dot_seq_len", C.c_int32),
        ("reserved0", C.c_int32),
    ]


class GemmProblem(C.Structure):
    _fields_ = [("A", C.c_void_p), ("lda", C.c_int64), ("B", C.c_void_p), ("ldb", C.c_int64), ("C", C.c_void_p), ("ldc", C.c_int64),
                ("M", C.c_int32), ("N", C.c_int32)]


def _load():
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"unite_b200: {_LIB_PATH} is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C unite_b200/csrc`). There is no fallback path."
        )
    return C.CDLL(_LIB_PATH)


lib = _load()

# name -> (restype, argtypes); kept in one table so tests can check it against the header.
_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float
SIGNATURES = {
    "ub_version": (C.c_int, []),
    "ub_last_error": (C.c_char_p, []),
    "ub_sm_count": (C.c_int, []),
    "ub_set_sm_limit": (C.c_int, [_I]),
    "ub_gemm_cluster4_capacity": (C.c_int, []),
    "ub_gemm_bf16": (C.c_int, [_P, _L, _I, _P, _L, _I, _P, _L, _I, _I, _I, C.POINTER(GemmEpilogue), _I, _P]),
    "ub_gemm_wgrad_multi": (C.c_int, [C.POINTER(GemmProblem), _I, _I, _I, _P]),
    "ub_attn_fwd": (C.c_int, [_P, _P, _P, _I, _I, _I, _F, _P]),
    "ub_attn_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _F, _P]),
    "ub_cls_attn": (C.c_int, [_P, _P, _I, _I, _I, _F, _P]),
    "ub_layernorm_fwd": (C.c_int, [_P, _I, _P, _P, _P, _F, _P, _P, _P, _I, _I, _I, _P]),
    "ub_teacher_embed_ln": (C.c_int, [_P, _P, _P, _P, _P, _F, _P, _I, _P, _I, _I, _I, _P]),
    "ub_layernorm_bwd": (C.c_int, [_P, _P, _P, _F, _P, _P, _P, _P, _I, _P, _P, _P, _I, _I, _P]),
    "ub_dec_tail_fwd": (C.c_int, [_P, _P, _P, _F, _P, _P, _P, _F, _I, _I, _I, _I, _P]),
    "ub_dec_tail_bwd": (C.c_int, [_P, _P, _P, _F, _P, _F, _I, _I, _P, _P, _P, _I, _I, _P]),
    "ub_l2norm_rows": (C.c_int, [_P, _I, _I, _P]),
    "ub_patchify": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "ub_patchify_mix": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ub_patchify_u8": (C.c_int, [_P, _P, C.POINTER(C.c_float), C.POINTER(C.c_float), _I, _I, _I, _I, _I, _P]),
    "ub_patchify_mix_u8": (C.c_int, [_P, _P, _P, C.POINTER(C.c_float), C.POINTER(C.c_float), _I, _I, _I, _I, _I, _P]),
    "ub_patchify_aug_u8": (C.c_int, [_P, _P, _P, _P, _I, _P, C.c_uint64, _P, C.POINTER(C.c_float), C.POINTER(C.c_float), _I, _I, _I, _I,
                                     _I, _I, _P]),
    "ub_resize_patchify":(C.c_int, [_P, _I, C.POINTER(C.c_float), C.POINTER(C.c_float), _P, _L, _I, _I, _I, _I, _I, _I, _I, _P]),
    "ub_mask_select": (C.c_int, [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P]),
    "ub_gather_rows": (C.c_int, [_P, _P, _P, _L, _L, _I, _L, _P]),
    "ub_colsum_bf16": (C.c_int, [_P, _L, _P, _I, _I, _I, _I, _P]),
    "ub_cast_scale_bf16": (C.c_int, [_P, _P, _P, _I, _L, _I, _P]),
    "ub_sumsq": (C.c_int, [_P, _L, _P, _P]),
    "ub_adamw": (C.c_int, [_P, _P, _P, _P, _P, _L, _L, _F, _F, _F, _F, _F, _I, _F, _P]),
    "ub_adamw_dev": (C.c_int, [_P, _P, _P, _P, _P, _L, _L, _P, _P, _P]),
    "ub_adamw_seg": (C.c_int, [_P, _P, _P, _P, _P, _L, _P, _I, _P, _P, _P]),
    "ub_sumsq_seg": (C.c_int, [_P, _L, _P, _I, _P, _P, _P]),
    "ub_cast_bf16": (C.c_int, [_P, _P, _L, _P]),
    "ub_ema_update": (C.c_int, [_P, _P, _P, _L, _F, _F, _P]),
    "ub_drop_path_draw": (C.c_int, [_P, _P, _I, _I, C.c_uint64, _P, _P]),
    "ub_nvls_slots": (C.c_int, []),
    "ub_adamw_nvls": (C.c_int, [_P, _P, _P, _P, _P, _P, _L, _L, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _P]),
    "ub_meanpool_fwd": (C.c_int, [_P, _P, _I, _I, _I, _P]),
    "ub_meanpool_bwd": (C.c_int, [_P, _P, _I, _I, _I, _P]),
    "ub_linear_small_fwd": (C.c_int, [_P, _P, _P, _P, _I, _I, _I, _P]),
    "ub_linear_small_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _I, _I, _P]),
    "ub_softmax_ce": (C.c_int, [_P, _P, _P, _F, _P, _P, _I, _I, _P]),
    "ub_soft_target_ce": (C.c_int, [_P, _P, _P, _F, _P, _P, _I, _I, _P]),
    "ub_clip_zero_shot": (C.c_int, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "ub_pseudo_label_fusion": (C.c_int, [_P, _P, _F, _I, _P, _P, _P, _P, _I, _I, _P]),
}


def _bind():
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args


_bind()


class UBError(RuntimeError):
    pass


def check(rc, what=""):
    if rc != 0:
        raise UBError(f"{what}: {lib.ub_last_error().decode()}")
