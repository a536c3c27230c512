"""Kernel-level parity on the GPU (through the C ABI) against plain torch references: every entry point of
include/unite_b200.h is exercised here or in test_stage1_gpu.py.  Bit-exact for integer / byte / index work
(patchify rounding, mask select, gathers); fp tolerances are written next to each comparison in tools/*_check.py."""
import importlib
import os
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))


def _kc():
    m = importlib.import_module("kernels_check")
    m.OK = True
    return m


def test_tokens_patchify_mask_gather_bit_exact():
    m = _kc(); m.check_tokens(); assert m.OK


# (10240, 768), (5003, 1024), (6000, 256): large enough for the bulk-copy-staged backward (ragged last row block included)
@pytest.mark.parametrize("rows,D", [(4096, 768), (1024, 128), (512, 1024), (10240, 768), (5008, 1024), (6000, 256)])
def test_layernorm_family(rows, D):
    m = _kc(); m.check_ln(rows, D); assert m.OK


@pytest.mark.parametrize("rows,D", [(4096, 512), (300, 128)])
def test_decoder_tail_and_loss(rows, D):
    m = _kc(); m.check_dec_tail(rows, D); assert m.OK


def test_fused_adamw_matches_torch():
    m = _kc(); m.check_optim(); assert m.OK


@pytest.mark.parametrize("n_seq,S,H", [(2, 17, 2), (4, 197, 12), (3, 128, 4), (5, 240, 3), (2, 256, 3), (3, 320, 12), (1, 1568, 4)])
def test_attention_forward_backward_cls(n_seq, S, H):
    m = _kc(); m.check_attention(n_seq, S, H); assert m.OK


def test_teacher_attention_first_half_reference_and_its_redo_path():
    m = _kc(); m.check_attention_tc_late_maximum(); assert m.OK


@pytest.mark.parametrize("B,N,H", [(5, 320, 12), (3, 197, 4), (2, 1568, 12), (1, 40, 2)])
def test_gemm_epilogue_leaves_rowsum_dO_O_for_the_attention_backward(B, N, H):
    m = _kc(); m.check_gemm_dot_aux(B, N, H); assert m.OK


def test_gemm_all_operand_majors_and_epilogues():
    g = importlib.import_module("gemm_check")
    ok = True
    ok &= g.run(128, 128, 64)
    ok &= g.run(128, 256, 256)
    ok &= g.run(256, 512, 768, out_fp32=1)
    ok &= g.run(200, 264, 200, out_fp32=1)                      # ragged M, N, K: TMA zero-fill / clipping
    ok &= g.run(1000, 768, 768, bias=True, resid=True, out_fp32=1)
    ok &= g.run(2048, 2304, 768, bias=True)
    ok &= g.run(2048, 3072, 768, bias=True, act=1)
    ok &= g.run(2048, 3072, 768, bias=True, act=2)
    ok &= g.run(256, 256, 128, b_mn=1)                          # dgrad form
    ok &= g.run(2048, 768, 3072, b_mn=1)
    ok &= g.run(256, 256, 256, a_mn=1, b_mn=1, out_fp32=1)      # wgrad form
    ok &= g.run(768, 768, 4096, a_mn=1, b_mn=1, out_fp32=1, split_k=4, accumulate=1)
    assert ok


@pytest.mark.parametrize("M,N,K", [(2048, 3072, 768), (1000, 520, 256), (10240, 3072, 768)])
def test_gemm_dgelu_epilogue_with_fused_bias_gradient(M, N, K):
    """dX = (dY @ W) * gelu'(pre) in bf16 and, from the same epilogue, colsum_out += sum over rows of dX (the fc1 bias gradient,
    modeling_finetune.py:66-73 backward).  Reference: fp32 torch on the same bf16 operands; ragged M / N / K included."""
    import torch
    from unite_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(M + N + K)
    dy = (torch.randn(M, K, device="cuda", generator=g) * 0.5).bfloat16()
    w = (torch.randn(K, N, device="cuda", generator=g) * 0.05).bfloat16()            # stored [K, N]: b_t form, as in backward
    pre = torch.randn(M, N, device="cuda", generator=g).bfloat16()
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    bias_grad = torch.full((N,), 3.0, device="cuda")                                 # accumulates on top of what is there
    ops.gemm(dy, w, out, b_t=True, act=ops.UB_ACT_DGELU, aux_in=pre, colsum_out=bias_grad)
    torch.cuda.synchronize()
    x = pre.float()
    dgelu = 0.5 * (1 + torch.erf(x / 2 ** 0.5)) + x * torch.exp(-0.5 * x * x) / (2 * torch.pi) ** 0.5
    ref = (dy.float() @ w.float()) * dgelu
    assert ((out.float() - ref).norm() / ref.norm()).item() < 6e-3
    ref_sum = ref.sum(0) + 3.0
    err = (bias_grad - ref_sum).abs().max().item()
    assert err < 2e-3 * ref.abs().sum(0).max().item() + 1e-3, err
    # and against the separate pass over the bf16 output it replaces
    sep = torch.full((N,), 3.0, device="cuda")
    ops.colsum_bf16(out, sep)
    assert (bias_grad - sep).abs().max().item() < 5e-3 * out.float().abs().sum(0).max().item() + 1e-3


def test_gemm_layernorm_fold_and_fp16_residual_statistics():
    """Teacher path: x = residual + A W^T written in fp16 with its row (sum, sumsq); the next GEMM consumes x directly and applies
    LayerNorm in its epilogue (fp16 operands).  Against torch layer_norm + linear in fp32."""
    g = importlib.import_module("gemm_check")
    assert g.run_lnfold(1000, 2304, 768)
    assert g.run_lnfold(2048, 3072, 768, act=1)
    assert g.run_lnfold(300, 512, 256)


@pytest.mark.parametrize("tub", [1, 2])
def test_uint8_frames_to_normalised_patches_bit_exact(tub):
    """SURVEY.md §8 row f2: decoded uint8 frames [B,T,H,W,3] -> ToTensor + tensor_normalize + THWC->CTHW + patchify in one
    kernel, bit-exact against the CPU restatement of src/datasets/kinetics_sparse.py:236-247,434-451."""
    import torch
    from oracle import unite_oracle as orc
    from unite_b200 import ops
    B, T, H, W = 2, 4, 64, 96
    fr = torch.randint(0, 256, (B, T, H, W, 3), generator=torch.Generator().manual_seed(3 + tub), dtype=torch.uint8)
    fr[0, 0, 0, :4] = torch.tensor([[0, 0, 0], [255, 255, 255], [1, 128, 254], [127, 0, 255]], dtype=torch.uint8)   # extremes
    n_tok = B * (T // tub) * (H // 16) * (W // 16)
    out = torch.empty(n_tok, 3 * tub * 256, device="cuda", dtype=torch.bfloat16)
    ops.patchify_u8(fr.cuda(), out, tub)
    ref = orc.patchify(orc.normalize_frames_u8(fr), tub, 16).reshape(n_tok, -1).bfloat16()
    assert torch.equal(out.cpu(), ref)
    with pytest.raises(Exception):
        ops.patchify_u8(fr.cuda()[..., :2], out, tub)          # not [.., 3]


@pytest.mark.parametrize("variant", ["", "erf"])
def test_gelu_epilogue_default_and_exact_erf_builds(variant):
    """DESIGN §2: the student's GELU is evaluated with the hardware tanh.approx form (|err| <= 4.7e-4, a deliberate deviation);
    -DUB_GELU_ERF (libunite_b200_erf.so, built by build()) restores an erf accurate to 1.5e-7.  Both builds are kept under test."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if variant:
        assert os.path.exists(os.path.join(root, "unite_b200", "lib", f"libunite_b200_{variant}.so")), "build() did not produce the erf variant"
    env = dict(os.environ)
    env.pop("UB_LIB_VARIANT", None)
    if variant:
        env["UB_LIB_VARIANT"] = variant
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "gelu_variant_check.py")], capture_output=True, text=True, env=env, timeout=300)
    print(r.stdout[-400:])
    assert r.returncode == 0 and "GELU VARIANT OK" in r.stdout, (r.stdout[-1500:], r.stderr[-1500:])


def test_multi_problem_weight_gradient_gemm():
    """ub_gemm_wgrad_multi: several dW_i += dY_i^T X_i over the same tokens in one launch — ragged widths (TMA clipping), a token
    count that is not a multiple of the k-block, accumulation into non-zero dW, 1 to 4 problems, several split-K factors."""
    import torch
    from unite_b200 import ops
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(11)
    for K, widths, split in ((10240, [(768, 3072), (3072, 768), (768, 768), (2304, 768)], 2), (1000, [(200, 328), (512, 64), (8, 1032)], 3),
                             (4096, [(520, 264)], 1), (320, [(128, 128), (384, 512)], 7)):
        probs, refs = [], []
        for (M, N) in widths:
            dy = (torch.randn(K, M, device=dev, generator=g) * 0.5).bfloat16()
            x = (torch.randn(K, N, device=dev, generator=g) * 0.5).bfloat16()
            gw = torch.randn(M, N, device=dev, generator=g)
            refs.append(gw.double() + dy.double().t() @ x.double())
            probs.append((dy, x, gw))
        ops.gemm_wgrad_multi(probs, split_k=split)
        torch.cuda.synchronize()
        for (dy, x, gw), ref in zip(probs, refs):
            err = ((gw.double() - ref).norm() / ref.norm()).item()
            assert err < 2e-5 and torch.isfinite(gw).all(), (K, tuple(gw.shape), split, err)
