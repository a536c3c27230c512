"""uint8 frames for stages 2 and 3 without a GPU: the batches refused before anything is launched, the clip shape the mixup draw
sees, the synthetic loaders' uint8 option and the fp32 path's unchanged launches."""
import types

import numpy as np
import pytest
import torch


def _frames(*shape):
    return torch.randint(0, 256, shape, generator=torch.Generator().manual_seed(0), dtype=torch.uint8)


BAD = [
    (lambda: _frames(2, 3, 4, 32, 32), "channels last"),                              # uint8 in [B,3,T,H,W] layout
    (lambda: _frames(2, 4, 32, 64, 3)[:, :, :, ::2], "contiguous"),                   # a non-contiguous batch
    (lambda: _frames(2, 4, 32, 64, 3).transpose(2, 3), "contiguous"),
    (lambda: _frames(2, 4, 40, 32, 3), "multiples of the 16-pixel patch"),            # H not a multiple of 16
    (lambda: _frames(2, 4, 32, 24, 3), "multiples of the 16-pixel patch"),            # W not a multiple of 16
]


@pytest.mark.parametrize("make,msg", BAD)
def test_clip_shape_refuses_frames_the_kernels_cannot_read(make, msg):
    from unite_b200 import ops
    with pytest.raises(ValueError, match=msg):
        ops.clip_shape(make())


def test_clip_shape_maps_frames_to_the_clip_they_stand_for():
    from unite_b200 import ops
    assert ops.clip_shape(_frames(4, 8, 224, 160, 3)) == (4, 3, 8, 224, 160)
    assert ops.clip_shape(_frames(3, 8, 32, 32, 3)) == (3, 3, 8, 32, 32)
    with pytest.raises(ValueError, match="even"):
        ops.clip_shape(_frames(3, 8, 32, 32, 3), paired=True)
    x = torch.zeros(3, 3, 4, 24, 40)                                                  # fp32: today's checks only, in the kernels
    assert ops.clip_shape(x, paired=True) == tuple(x.shape)


def test_the_mixup_draw_of_frames_is_the_draw_of_their_clip():
    """timm draws the cutmix box from the last two axes of the shape it is given: frames must be drawn as their [B,3,T,H,W] clip."""
    from unite_b200 import mixup as M
    from unite_b200 import ops
    frames = _frames(4, 8, 48, 32, 3)
    cfg = dict(mixup_alpha=0., cutmix_alpha=1.0, label_smoothing=0.1, num_classes=12)
    np.random.seed(10)
    want = M.draw(M.Mixup(**cfg), (4, 3, 8, 48, 32))
    np.random.seed(10)
    got = M.draw(M.Mixup(**cfg), ops.clip_shape(frames))
    assert got == want and got.use_cutmix and got.box[0][1] > got.box[0][0]


@pytest.mark.parametrize("bad,msg", [(lambda f: f[:3], "even"), (lambda f: _frames(4, 4, 40, 32, 3), "16-pixel")] +
                         [(lambda f, m=m: m(), msg) for m, msg in BAD[:2]])
def test_stage2_refuses_before_any_launch(bad, msg):
    """Stage2Engine.step (before the optimizer's upload), finetune_step (before the DropPath draw) and the model's forward refuse a
    bad uint8 batch with ValueError on a machine without a GPU: nothing is launched first."""
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import Stage2Engine, finetune_step
    from unite_b200.modeling_finetune import VisionTransformer
    frames = bad(_frames(4, 4, 48, 32, 3))
    d = M.MixDraw(True, 0.3, False, ((0, 0), (0, 0), (0, 0)), 0.3)
    eng = Stage2Engine.__new__(Stage2Engine)                       # no arena, no optimizer: any use of them would fail otherwise
    with pytest.raises(ValueError, match=msg):
        eng.step(frames, torch.zeros(frames.shape[0], dtype=torch.long), mix=d, smoothing=0.1)
    mix = types.SimpleNamespace(clip=object(), target=object())
    with pytest.raises(ValueError, match=msg):
        finetune_step(None, frames, None, None, mix=mix)
    if msg != "even":
        with pytest.raises(ValueError, match=msg):
            VisionTransformer.forward(None, frames)


def test_stage2_loop_refuses_an_odd_uint8_batch_under_mixup():
    from unite_b200 import mixup as M
    from unite_b200 import ops
    mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, num_classes=12)
    with pytest.raises(ValueError, match="even"):
        M.draw(mixer, ops.clip_shape(_frames(3, 4, 32, 32, 3)))


@pytest.mark.parametrize("views,msg", [
    ((_frames(2, 4, 32, 32, 3), torch.zeros(2, 3, 4, 32, 32), None), "share a dtype"),
    ((_frames(2, 4, 32, 32, 3), _frames(2, 4, 32, 32, 3), torch.zeros(2, 3, 4, 32, 32)), "share a dtype"),
    ((torch.zeros(2, 3, 4, 32, 32), torch.zeros(2, 3, 4, 32, 32), _frames(2, 4, 32, 32, 3)), "share a dtype"),
    ((_frames(2, 4, 32, 32, 3), _frames(2, 3, 4, 32, 32), None), "channels last"),
    ((_frames(2, 4, 32, 32, 3), _frames(2, 4, 32, 64, 3)[:, :, :, ::2], None), "contiguous"),
    ((_frames(2, 4, 32, 32, 3), _frames(2, 4, 32, 32, 3), _frames(2, 4, 32, 40, 3)), "16-pixel"),
])
def test_stage3_refuses_mixed_or_unreadable_views_before_any_launch(views, msg):
    from unite_b200.engine_stage3 import Stage3Engine
    eng = Stage3Engine.__new__(Stage3Engine)                       # no model, no optimizer: any use of them would fail otherwise
    vs, vt, va = views
    ys = torch.zeros(2, dtype=torch.long)
    with pytest.raises(ValueError, match=msg):
        eng.forward_backward(vs, ys, vt, va)
    with pytest.raises(ValueError, match=msg):
        eng.step(vs, ys, vt, va)


def test_stage3_view_dtype():
    from unite_b200.engine_stage3 import view_dtype
    f = _frames(2, 4, 32, 32, 3)
    assert view_dtype(f, f, None) == torch.uint8
    assert view_dtype(torch.zeros(2, 3, 4, 24, 24), torch.zeros(2, 3, 4, 24, 24), None) == torch.float32


def test_synthetic_stage2_and_stage3_loaders_carry_uint8_frames():
    from unite_b200.synthetic import SyntheticStage2Loader, SyntheticStage3Loader
    v, y, idx, extra = next(iter(SyntheticStage2Loader(4, num_frames=4, img_size=32, steps=1, uint8=True)))
    assert v.dtype == torch.uint8 and v.shape == (4, 4, 32, 32, 3) and y.shape == (4,) and extra == {}
    ld = SyntheticStage3Loader(4, 6, num_frames=4, img_size=32, steps=2, uint8=True)
    vs, ys, _, _ = next(iter(ld.source))
    vt, va, yt, names = next(iter(ld.target))
    assert vs.dtype == vt.dtype == va.dtype == torch.uint8
    assert vs.shape == (4, 4, 32, 32, 3) and vt.shape == va.shape == (6, 4, 32, 32, 3) and len(names) == 6
    d = va.short() - vt.short()
    assert d.abs().max() <= 8 and (d != 0).any()
    # the fp32 loaders are unchanged: same draws from the same seed
    g = torch.Generator().manual_seed(0)
    want = torch.randn(4, 3, 4, 32, 32, generator=g)
    assert torch.equal(next(iter(SyntheticStage2Loader(4, num_frames=4, img_size=32, steps=1)))[0], want)


def test_fp32_stage2_launch_list_is_unchanged(monkeypatch):
    """The fp32 path of FinetuneCore.run_forward, run against recording stand-ins for every op: the same kernels in the same order
    as before uint8 frames were accepted."""
    from unite_b200 import finetune_core, ops
    calls = []

    def rec(name):
        def f(*a, **k):
            calls.append(name)
            return a[1] if name.startswith("patchify") else None
        return f
    for name in ("patchify", "patchify_mix", "patchify_u8", "patchify_mix_u8", "meanpool_fwd", "layernorm_fwd", "linear_small_fwd"):
        monkeypatch.setattr(ops, name, rec(name))
    core = finetune_core.FinetuneCore.__new__(finetune_core.FinetuneCore)
    core.sync_shadow = lambda: calls.append("sync_shadow")
    core.N, core.tubelet, core.D, core.depth, core.C, core.eps = 16, 1, 8, 1, 3, 1e-6
    core._pos_full = {2: None}
    core.arena = types.SimpleNamespace(p32=lambda n: None)
    ws = types.SimpleNamespace(x_at=lambda l: torch.zeros(2 * 16 * 8))
    core.trunk = types.SimpleNamespace(forward=lambda *a: calls.append("trunk") or ws)
    x = torch.zeros(2, 3, 4, 16, 16)
    core.run_forward(x, None, False)
    core.run_forward(x, None, False, mix=torch.zeros(10))
    assert calls == ["sync_shadow", "patchify", "trunk", "meanpool_fwd", "layernorm_fwd", "linear_small_fwd",
                     "sync_shadow", "patchify_mix", "trunk", "meanpool_fwd", "layernorm_fwd", "linear_small_fwd"]


@pytest.mark.parametrize("kernel_size", [1, 2])
@pytest.mark.parametrize("dual", [False, True])
def test_fp32_stage3_launch_list_is_unchanged(monkeypatch, dual, kernel_size):
    """Stage3Engine.forward_backward on fp32 clips with recording stand-ins for the towers and every op: the teacher patchifies
    each view itself, the student reads the teacher's im2col when the kernels agree and patchifies the clip itself otherwise,
    in the same order as before uint8 frames were accepted."""
    from unite_b200 import ops
    from unite_b200.engine_stage3 import Stage3Engine
    calls = []
    Bs, Bt, T, P, D, C, k = 2, 2, 4 // kernel_size, 16, 8, 3, 2
    for name in ("meanpool_fwd", "linear_small_fwd", "linear_small_bwd", "meanpool_bwd", "softmax_ce", "mask_select",
                 "clip_zero_shot", "pseudo_label_fusion"):
        monkeypatch.setattr(ops, name, lambda *a, name=name, **kw: calls.append(name))

    def teacher_fwd(x, patches=None):
        calls.append(("teacher", patches))
        return None, torch.zeros(x.shape[0] * T, P), f"rows{len(calls)}"

    def student_fwd(x, vis, patches, dp, clip_only, save, want_clip=True, abs_rows=None):
        calls.append(("student", patches, abs_rows is None))
        return torch.zeros(x.shape[0], vis.shape[1], D), None, None
    eng = Stage3Engine.__new__(Stage3Engine)
    eng.teacher = types.SimpleNamespace(forward_features=teacher_fwd, kernel_size=kernel_size,
                                        cls_features=lambda *a: calls.append("cls_features"))
    eng.core = types.SimpleNamespace(N=64, tubelet=1, run_forward=student_fwd, run_backward=lambda *a, **kw: calls.append("backward"))
    eng.student = types.SimpleNamespace(training=False)
    eng.W, eng.b, eng.text = torch.zeros(C, D), torch.zeros(C), torch.zeros(C, 4)
    eng.k, eng.mask_ratio, eng.thr, eng.src_ratio, eng.tgt_ratio, eng.conf_weighted = k, 0.75, 0.5, 1.0, 1.0, True
    eng.nvls = eng.grad_sync = None
    eng.loss, eng.loss_s, eng.loss_t = torch.zeros(1), torch.zeros(1), torch.zeros(1)
    eng._full_idx = {}
    clip = lambda B: torch.zeros(B, 3, 4, 32, 32)
    eng.forward_backward(clip(Bs), torch.zeros(Bs, dtype=torch.long), clip(Bt), clip(Bt) if dual else None)
    share = kernel_size == 1
    teacher = [("teacher", None), "cls_features"] if not dual else [("teacher", None), ("teacher", None), "cls_features"]
    rows_t = "rows2" if dual else "rows1"
    want = teacher + [("student", None, True), "meanpool_fwd", "linear_small_fwd", "softmax_ce", "linear_small_bwd", "meanpool_bwd",
                      "backward", ("student", rows_t if share else None, True), "meanpool_fwd", "linear_small_fwd", "mask_select"]
    for m in range(k):
        want += [("student", "rows1" if share else None, not share), "meanpool_fwd", "linear_small_fwd"]
    want += ["clip_zero_shot", "pseudo_label_fusion", "softmax_ce", "linear_small_bwd", "meanpool_bwd", "backward"]
    assert calls == want
