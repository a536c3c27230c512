"""CLIP ViT-L/14 teacher on the GPU: the resize + patchify kernel against F.interpolate + the oracle's im2col, the full-depth
teacher and the stage-1 step against the CPU oracle (tests/teacher_resize_ref.py) (tolerances of tests/test_stage1_gpu.py), and the training loop with
clip_input_resolution."""
import pytest
import torch

from tests.util import build_student, build_teacher, per_token_rel, rel_l2

pytestmark = pytest.mark.gpu
FEAT_TOL = 1e-2


def _seeded(model, seed):
    from oracle.weights import seeded_state
    sd = seeded_state({k: tuple(v.shape) for k, v in model.state_dict().items()}, seed)
    model.load_state_dict(sd, strict=True)
    return sd


def _l14_cfg(kernel_size=1, return_layers=(18, 19, 20, 21, 22, 23)):
    from oracle import unite_oracle as O
    return O.TeacherCfg(width=1024, layers=24, heads=16, output_dim=768, input_resolution=196, patch_size=14, kernel_size=kernel_size,
                        return_layers=return_layers)


def _within_one_bf16_ulp(got, ref):
    """|got - bf16(ref)| <= 1 bf16 ulp at max(|got|, |bf16(ref)|, 1/64).  The floor: on O(1) inputs the kernel's fp32 sums and
    ATen's CPU kernel differ by up to ~2.4e-6 absolute (rounding order), more than one ulp of a value that cancels to near zero."""
    a, b = got.float().cpu(), ref.bfloat16().float()
    _, e = torch.frexp(torch.maximum(torch.maximum(a.abs(), b.abs()), torch.full_like(a, 1 / 64)))
    ulp = torch.ldexp(torch.ones_like(a), e - 8)                  # bf16 keeps 8 significant bits
    return (a - b).abs() <= ulp


# ---- kernel -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["fp32", "uint8"])
@pytest.mark.parametrize("B,T,H,R,p,ks", [(2, 8, 224, 196, 14, 1), (2, 8, 224, 196, 14, 2), (2, 8, 224, 224, 14, 1), (3, 4, 224, 196, 14, 1)])
def test_resize_patchify_matches_interpolate_then_im2col(kind, B, T, H, R, p, ks):
    from oracle import unite_oracle as O
    from tests.teacher_resize_ref import resize_for_teacher
    from unite_b200 import ops
    g = torch.Generator().manual_seed(B * 1000 + R + ks)
    if kind == "uint8":
        frames = torch.randint(0, 256, (B, T, H, H, 3), generator=g, dtype=torch.uint8)
        x, dev_in = O.normalize_frames_u8(frames), frames.cuda()
    else:
        x = torch.randn(B, 3, T, H, H, generator=g)
        dev_in = x.cuda()
    feat = 3 * ks * p * p
    ld = ops.padded_k(feat)
    n_tok = B * (T // ks) * (R // p) ** 2
    out = torch.full((n_tok, ld), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.resize_patchify(dev_in, out, R, p, ks)
    torch.cuda.synchronize()
    ref = O.patchify(resize_for_teacher(x, R), ks, p).reshape(n_tok, feat)
    ok = _within_one_bf16_ulp(out[:, :feat], ref)
    assert ok.all(), f"{int((~ok).sum())} of {ok.numel()} elements more than 1 bf16 ulp away"
    assert torch.equal(out[:, feat:].cpu(), torch.zeros(n_tok, ld - feat, dtype=torch.bfloat16)), "padding columns not zero"
    if R == H:
        assert torch.equal(out[:, :feat].cpu(), ref.bfloat16())   # no resize: a plain im2col, bit-exact


# ---- teacher ------------------------------------------------------------------------------------------------------------
def test_full_depth_l14_teacher_at_196_against_oracle():
    from oracle import unite_oracle as O
    tcfg = _l14_cfg()
    teacher = build_teacher(tcfg)
    tsd = _seeded(teacher, 31)
    g = torch.Generator().manual_seed(32)
    videos = torch.randn(2, 3, 8, 196, 196, generator=g)
    feat_ref, attn_ref = O.teacher_forward(tsd, videos, tcfg)
    feat, attn = teacher.cuda()(videos.cuda())
    torch.cuda.synchronize()
    err = per_token_rel(feat, feat_ref)
    a_err = rel_l2(attn, attn_ref)
    print(f"L/14 teacher, 24 layers at 196 px: per-token feature error mean {err.mean():.2e} max {err.max():.2e}; attention rel L2 {a_err:.2e}")
    assert err.max() < FEAT_TOL
    assert a_err < FEAT_TOL


# ---- stage-1 step -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("large", [False, True], ids=["vitb16_student", "vitl16_student_tubelet2"])
def test_stage1_step_with_l14_teacher_against_oracle(large):
    """Clips at 224 px, the teacher's copy resized to 196 on the device (14x14 patches of 14 px = the student's 14x14 of 16 px).
    large: ViT-L/16 student at 16 frames / tubelet 2 and the teacher at kernel_size 2 (K = 1176 before padding), B = 1."""
    from oracle import unite_oracle as O
    from unite_b200.engine import Stage1Engine
    from tests.test_stage1_gpu import _check_step
    from tests.teacher_resize_ref import stage1_step_at
    if large:
        scfg = O.StudentCfg(embed_dim=1024, depth=24, num_heads=16, num_frames=16, tubelet_size=2, clip_output_dim=768)
        tcfg, B = _l14_cfg(kernel_size=2), 1
    else:
        scfg, tcfg, B = O.StudentCfg(clip_output_dim=768), _l14_cfg(), 2
    student, teacher = build_student(scfg), build_teacher(tcfg)
    ssd, tsd = _seeded(student, 41), _seeded(teacher, 42)
    g = torch.Generator().manual_seed(43)
    videos = torch.randn(B, 3, scfg.num_frames, 224, 224, generator=g)
    q = torch.empty(B * scfg.num_frames // scfg.tubelet_size, 196).exponential_(1, generator=g)
    ref = stage1_step_at(ssd, tsd, videos, q, scfg, tcfg, 196, mask_ratio=0.8)
    assert ref["vis_idx"].shape == (B, 320)
    eng = Stage1Engine(student.cuda().train(), teacher.cuda().eval(), mask_ratio=0.8)
    assert eng.teacher_resolution == 196 and not eng.share_patches
    _check_step(eng, ref, videos, q, big_grad_only=True)


# ---- loop ---------------------------------------------------------------------------------------------------------------
def _tiny(teacher_res=196, output_dim=128, seed=0):
    """Three-block student at 224 px / 4 frames and a three-block 14-pixel teacher (width 128, head_dim 64)."""
    from oracle import unite_oracle as O
    scfg = O.StudentCfg(embed_dim=128, depth=3, num_heads=2, num_frames=4, return_layers=(1, 2), clip_output_dim=128)
    tcfg = O.TeacherCfg(width=128, layers=3, heads=2, output_dim=output_dim, input_resolution=teacher_res, patch_size=14,
                        return_layers=(1, 2))
    student, teacher = build_student(scfg), build_teacher(tcfg)
    _seeded(student, seed + 1)
    _seeded(teacher, seed + 2)
    g = torch.Generator().manual_seed(seed + 3)
    videos = torch.randn(2, 3, 4, 224, 224, generator=g)
    q = torch.empty(2 * 4, 196).exponential_(1, generator=g)
    return student.cuda().train(), teacher.cuda().eval(), videos, q


class _Args:
    log_freq = 1


def test_train_one_epoch_at_clip_input_resolution_196_lowers_the_loss():
    from unite_b200.engine_for_pretraining import train_one_epoch
    student, teacher, videos, q = _tiny()
    kw = dict(teacher_model=teacher, clip_input_resolution=196, mask_type="attention", mask_ratio=0.8, args=_Args,
              lr_schedule_values=[1e-3] * 100)
    first = train_one_epoch(student, [(videos, -1, torch.zeros(2), q)], None, None, "cuda", 0, None, **kw)["loss"]
    train_one_epoch(student, [(videos, -1, torch.zeros(2), q)] * 10, None, None, "cuda", 1, None, **kw)
    train_one_epoch(student, [(videos, -1, torch.zeros(2))] * 2, None, None, "cuda", 2, None, **kw)     # noise drawn on the device
    last = train_one_epoch(student, [(videos, -1, torch.zeros(2), q)], None, None, "cuda", 3, None, **kw)["loss"]
    eng = student.__dict__["_ub_stage1_engine"][1]
    assert eng.teacher_resolution == 196 and eng.last["attn"].shape == (8, 196)
    print(f"loss {first:.5f} -> {last:.5f}")
    assert last < first


def test_uint8_frames_give_the_same_step_as_the_normalised_clip():
    from oracle.unite_oracle import normalize_frames_u8
    from unite_b200.engine import Stage1Engine
    student, teacher, _, q = _tiny(seed=10)
    eng = Stage1Engine(student, teacher, mask_ratio=0.8)
    frames = torch.randint(0, 256, (2, 4, 224, 224, 3), generator=torch.Generator().manual_seed(11), dtype=torch.uint8)
    q = q.cuda()
    eng.optimizer.zero_grad()
    l_u8 = eng.forward_backward(frames.cuda(), q).clone()
    mask_u8 = eng.last["mask"].clone()
    g_u8 = eng.core.arena.grads.clone()
    eng.optimizer.zero_grad()
    l_f32 = eng.forward_backward(normalize_frames_u8(frames).cuda(), q).clone()
    torch.cuda.synchronize()
    assert torch.equal(mask_u8, eng.last["mask"])
    assert abs(l_u8.item() - l_f32.item()) <= 2e-6 * abs(l_f32.item()), (l_u8.item(), l_f32.item())
    assert rel_l2(g_u8, eng.core.arena.grads) < 1e-5


def test_graph_replayed_step_matches_an_eager_step():
    """The resize runs inside the captured step: a replay and an eager forward/backward from the same parameters agree."""
    from unite_b200.engine import Stage1Engine
    student, teacher, videos, q = _tiny(seed=20)
    eng = Stage1Engine(student, teacher, mask_ratio=0.8, lr=1e-3, use_graph=True)
    videos, q = videos.cuda(), q.cuda()
    for _ in range(2):
        eng.step(videos, q)                                       # eager warm-up steps of this shape
    torch.cuda.synchronize()
    p0 = eng.core.arena.params.clone()
    eng.step(videos, q)                                           # captured, then replayed
    torch.cuda.synchronize()
    assert len(eng._graphs) == 1
    loss_g, mask_g = eng.loss.clone(), eng.last["mask"].clone()
    out_g, grads_g = eng.last["outputs"].clone(), eng.core.arena.grads.clone()
    eng.core.arena.params.copy_(p0)
    eng.core.sync_shadow(force=True)
    eng.optimizer.zero_grad()
    loss_e = eng.forward_backward(videos, q).clone()
    torch.cuda.synchronize()
    assert torch.equal(mask_g, eng.last["mask"])
    assert abs(loss_g.item() - loss_e.item()) <= 2e-6 * abs(loss_e.item()), (loss_g.item(), loss_e.item())
    assert rel_l2(out_g, eng.last["outputs"]) < 1e-5
    assert rel_l2(grads_g, eng.core.arena.grads) < 1e-5


def test_misconfigurations_are_refused_with_both_numbers():
    from unite_b200.engine import Stage1Engine
    from unite_b200.engine_for_pretraining import train_one_epoch
    # a 14-pixel teacher at 224 px sees 16x16 = 256 patches per frame, the 16-pixel student 196
    student, teacher, videos, q = _tiny(teacher_res=224)
    with pytest.raises(ValueError, match=r"256.*196"):
        train_one_epoch(student, [(videos, -1, torch.zeros(2), q)], None, None, "cuda", 0, None, teacher_model=teacher,
                        clip_input_resolution=224, mask_type="attention", mask_ratio=0.8, args=_Args)
    # a resolution that is not a multiple of the patch size
    student, teacher, videos, q = _tiny(seed=30)
    with pytest.raises(ValueError, match=r"200.*14"):
        train_one_epoch(student, [(videos, -1, torch.zeros(2), q)], None, None, "cuda", 0, None, teacher_model=teacher,
                        clip_input_resolution=200, mask_type="attention", mask_ratio=0.8, args=_Args)
    # the student's clip_output_dim must be the teacher's output_dim
    student, teacher, _, _ = _tiny(output_dim=96, seed=40)
    with pytest.raises(ValueError, match=r"128.*96"):
        Stage1Engine(student, teacher)
