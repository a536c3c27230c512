"""CLIP ViT-L/14 teacher without a GPU: the factories construct, the checkpoint adapter maps OpenAI L/14 shapes onto a 196-px
teacher, the test-side reference for a resized teacher view agrees with the oracle, and the configurations the CUDA path refuses are refused."""
import types

import pytest
import torch
import torch.nn.functional as F

from oracle import unite_oracle as O
from tests.util import load_golden, oracle_cfgs, seeded_states


@pytest.mark.parametrize("factory", ["clip_l14", "clip_l14_336"])
def test_l14_factories_construct_at_196(factory):
    from unite_b200 import clip
    m = getattr(clip, factory)(pretrained=False, input_resolution=196, return_attn=True)
    assert m.patch_size == 14 and m.width == 1024 and m.heads == 16 and m.output_dim == 768
    assert tuple(m.positional_embedding.shape) == (197, 1024)
    assert m.k_pad == 640                                        # 3*14*14 = 588 features, padded to a multiple of 64
    assert tuple(m.conv1.weight.shape) == (1024, 3, 1, 14, 14)


@pytest.mark.parametrize("orig_tokens", [257, 577])           # OpenAI ViT-L/14 at 224 px (16x16 grid) and at 336 px (24x24)
def test_checkpoint_adapter_maps_l14_weights_onto_a_196px_teacher_with_kernel_size_2(orig_tokens):
    from unite_b200 import clip
    m = clip.clip_l14(pretrained=False, input_resolution=196, kernel_size=2)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(orig_tokens)
    pos = torch.randn(orig_tokens, 1024, generator=g)
    w2d = torch.randn(1024, 3, 14, 14, generator=g)
    sd["positional_embedding"], sd["conv1.weight"] = pos, w2d
    clip.load_state_dict(m, sd, input_resolution=196, patch_size=14)
    n = int((orig_tokens - 1) ** 0.5)
    grid = pos[1:].reshape(1, n, n, 1024).permute(0, 3, 1, 2)
    want = F.interpolate(grid, size=(14, 14), mode="bicubic", align_corners=False).permute(0, 2, 3, 1).reshape(196, 1024)
    got = m.positional_embedding.detach()
    assert got.shape == (197, 1024)
    assert torch.equal(got[0], pos[0]) and torch.equal(got[1:], want)
    w3 = m.conv1.weight.detach()
    assert w3.shape == (1024, 3, 2, 14, 14)
    assert torch.equal(w3[:, :, 1], w2d) and not w3[:, :, 0].any()      # centre inflation: time_dim // 2 = 1 holds the 2-D kernel


def test_resized_reference_without_a_resize_is_the_oracle_step():
    """tests/teacher_resize_ref.stage1_step_at at the clip's own size reproduces oracle.stage1_step bit for bit."""
    from tests.teacher_resize_ref import stage1_step_at
    fix = load_golden("tiny_stage12.pt")
    scfg, tcfg = oracle_cfgs(fix)
    ssd, tsd, _ = seeded_states(fix)
    args = (ssd, tsd, fix["videos"], fix["q"], scfg, tcfg)
    base = O.stage1_step(*args, mask_ratio=fix["cfg"]["mask_ratio"])
    r = stage1_step_at(*args, fix["videos"].shape[3], mask_ratio=fix["cfg"]["mask_ratio"])
    for key in ("attn", "mask", "vis_idx", "targets", "outputs", "loss", "grad_norm"):
        assert torch.equal(r[key], base[key]), key
    for k, gr in base["grads"].items():
        assert torch.equal(r["grads"][k], gr), k


def test_resized_reference_resizes_the_teacher_copy_only():
    """A 14-pixel teacher at 56 px behind a 16-pixel student at 64 px: both see 16 patches per frame."""
    from oracle.weights import seeded_state
    from tests.teacher_resize_ref import stage1_step_at
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    ssd, _, _ = seeded_states(fix)
    tcfg = O.TeacherCfg(width=128, layers=3, heads=2, output_dim=128, input_resolution=56, patch_size=14, return_layers=(1, 2))
    shapes = {"conv1.weight": (128, 3, 1, 14, 14), "class_embedding": (128,), "positional_embedding": (17, 128), "proj": (128, 128),
              "ln_pre.weight": (128,), "ln_pre.bias": (128,), "ln_post.weight": (128,), "ln_post.bias": (128,)}
    for i in range(3):
        p = f"transformer.resblocks.{i}."
        shapes.update({p + "attn.in_proj_weight": (384, 128), p + "attn.in_proj_bias": (384,), p + "attn.out_proj.weight": (128, 128),
                       p + "attn.out_proj.bias": (128,), p + "ln_1.weight": (128,), p + "ln_1.bias": (128,), p + "mlp.c_fc.weight": (512, 128),
                       p + "mlp.c_fc.bias": (512,), p + "mlp.c_proj.weight": (128, 512), p + "mlp.c_proj.bias": (128,),
                       p + "ln_2.weight": (128,), p + "ln_2.bias": (128,)})
    tsd = seeded_state(shapes, 3)
    videos, q = fix["videos"], fix["q"]
    r = stage1_step_at(ssd, tsd, videos, q, scfg, tcfg, 56, mask_ratio=0.75, with_grads=False)
    B, C, T, H, W = videos.shape
    tv = F.interpolate(videos.view(B, C * T, H, W), size=(56, 56), mode="bicubic", align_corners=False).view(B, C, T, 56, 56)
    _, attn = O.teacher_forward(tsd, tv, tcfg)
    assert torch.equal(r["attn"], attn) and r["attn"].shape == (B * T, 16)
    # the student still saw the 64-px clip: its outputs are those of student_forward on it
    out = O.student_forward(ssd, videos, r["mask"], scfg, clip_only=True)
    assert torch.equal(out, r["outputs"])


def test_oracle_patchify_at_14_pixels_is_conv3d():
    g = torch.Generator().manual_seed(4)
    x = torch.randn(2, 3, 4, 28, 42, generator=g)
    w = torch.randn(8, 3, 2, 14, 14, generator=g)
    ref = F.conv3d(x, w, stride=(2, 14, 14)).flatten(2).transpose(1, 2)        # [B, T'*h*w, D], token order (t, h, w)
    got = O.patchify(x, 2, 14) @ w.reshape(8, -1).t()
    assert torch.allclose(got, ref, rtol=1e-4, atol=1e-4)


def test_teacher_forward_refuses_a_clip_off_its_patch_grid():
    from unite_b200 import clip
    m = clip.VisionTransformer(input_resolution=56, patch_size=14, width=128, layers=1, heads=2, output_dim=64, return_attn=True,
                               clip_return_layers=[0])
    with pytest.raises(ValueError, match="does not resize"):
        m(torch.zeros(1, 3, 1, 64, 64))                          # 64 px: not a multiple of 14, and 4x4 would be another grid
    with pytest.raises(NotImplementedError):
        clip.VisionTransformer(input_resolution=64, patch_size=8, width=128, layers=1, heads=2, output_dim=64)


def test_stage3_refuses_a_14_pixel_teacher():
    from unite_b200.engine_stage3 import Stage3Engine
    teacher = types.SimpleNamespace(patch_size=14)
    with pytest.raises(NotImplementedError, match="patch size 14"):
        Stage3Engine(None, teacher, None, None, None)
