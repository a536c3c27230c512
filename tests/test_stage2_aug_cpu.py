"""The stage-2 spatial augmentation's host side without a GPU: unite_b200.augment draws call for call what the reference's
loader draws (tests/augment_ref.py, from the same Python and numpy seeds), the packed per-clip layout, and the refusals, raised
before any device work."""
import random
import types

import numpy as np
import pytest
import torch

from tests import augment_ref as R


def _seed(s):
    random.seed(s)
    np.random.seed(s)


def _ref_draws(B, H, W, S=224, scale=(0.08, 1.0), ratio=(0.75, 1.3333), hflip=True, reprob=0.25):
    """Per clip, the reference's calls in the loader's order; the erasing box is read back from a const erase of a ones plane."""
    rows = []
    for _ in range(B):
        i, j, h, w = R._get_param_spatial_crop(scale, ratio, H, W)
        flip = int(np.random.uniform() < 0.5) if hflip else 0
        box = (0, 0, 0, 0, 0)
        if reprob > 0:
            plane = torch.ones(1, 1, S, S)
            R.RandomErasing(reprob, mode="const", max_count=1, num_splits=1, device="cpu")(plane)
            ys, xs = torch.nonzero(plane[0, 0] == 0, as_tuple=True)
            if ys.numel():
                box = (1, int(ys.min()), int(xs.min()), int(ys.max()) - int(ys.min()) + 1, int(xs.max()) - int(xs.min()) + 1)
        rows.append([i, j, h, w, flip, *box])
    return np.array(rows, dtype=np.int32)


CASES = [
    # H, W, SpatialAugment kwargs
    (256, 320, {}),
    (240, 427, dict(reprob=1.0, remode="const")),
    (224, 224, dict(reprob=0.0)),                              # no RandomErasing: no erase draw at all
    (256, 32, dict(scale=(0.9, 1.0))),                         # narrower than the ratio range: every attempt misses, fallback
    (256, 320, dict(scale=(1.0, 1.0), reprob=1.0)),            # the whole frame's area: mostly the whole-image fallback
    (300, 200, dict(hflip=False, crop_size=112, remode="rand")),
]


@pytest.mark.parametrize("H,W,kw", CASES)
def test_host_draws_equal_the_reference_call_for_call(H, W, kw):
    from unite_b200.augment import SpatialAugment
    aug = SpatialAugment(**kw)
    B = 24
    for seed in (0, 1, 7):
        _seed(seed)
        got = aug.draw((B, 8, H, W, 3))
        after = (random.random(), np.random.uniform())
        _seed(seed)
        want = _ref_draws(B, H, W, S=aug.crop_size, scale=aug.scale, ratio=aug.ratio, hflip=aug.hflip, reprob=aug.reprob)
        assert (random.random(), np.random.uniform()) == after, "the two paths consumed different numbers of draws"
        assert got.params.dtype == np.int32 and got.params.shape == (B, 10) and got.frames_hw == (H, W)
        assert np.array_equal(got.params, want), (got.params, want)
    p = got.params
    assert ((p[:, 0] >= 0) & (p[:, 0] + p[:, 2] <= H) & (p[:, 1] >= 0) & (p[:, 1] + p[:, 3] <= W)).all()
    if kw.get("scale") == (0.9, 1.0):
        assert (p[:, :4] == [(256 - 43) // 2, 0, 43, 32]).all()            # the central crop at the narrowest admissible ratio
    if kw.get("reprob") == 1.0:
        assert (p[:, 5] == 1).all()
    if kw.get("reprob") == 0.0:
        assert (p[:, 5:] == 0).all()
    if kw.get("hflip") is False:
        assert (p[:, 4] == 0).all()
    elif B >= 24:
        assert 0 < p[:, 4].sum() < B


def test_crop_fallback_and_flip_functions():
    from unite_b200.augment import crop_params, erase_box, flip_draw
    _seed(3)
    a = [crop_params((0.9, 1.0), (0.75, 1.3333), 256, 32) for _ in range(5)]
    _seed(3)
    b = [R._get_param_spatial_crop((0.9, 1.0), (0.75, 1.3333), 256, 32) for _ in range(5)]
    assert a == b and all(x == (106, 0, 43, 32) for x in a)
    _seed(5)
    f = [flip_draw() for _ in range(64)]
    _seed(5)
    assert f == [np.random.uniform() < 0.5 for _ in range(64)]
    _seed(9)
    assert erase_box(0.0, 224, 224) is None                               # random.random() > 0
    assert all(erase_box(1.0, 224, 224) is not None for _ in range(32))


def test_packed_layout():
    """{i, j, h, w, flip, erase, top, left, eh, ew} per clip, int32, in batch order."""
    from unite_b200.augment import SpatialAugment
    aug = SpatialAugment(reprob=1.0)
    _seed(11)
    d = aug.draw((3, 4, 256, 320, 3))
    _seed(11)
    for b in range(3):
        i, j, h, w = R._get_param_spatial_crop(aug.scale, aug.ratio, 256, 320)
        flip = int(np.random.uniform() < 0.5)
        assert random.random() <= 1.0
        assert tuple(d.params[b, :5]) == (i, j, h, w, flip)
        # the erase draw: replay it on the host from the state RandomErasing leaves after its probability draw
        S = aug.crop_size
        while True:
            ta = random.uniform(0.02, 1 / 3) * S * S
            ar = np.exp(random.uniform(np.log(0.3), np.log(1 / 0.3)))
            eh, ew = int(round(np.sqrt(ta * ar))), int(round(np.sqrt(ta / ar)))
            if ew < S and eh < S:
                top, left = random.randint(0, S - eh), random.randint(0, S - ew)
                break
        assert tuple(d.params[b, 5:]) == (1, top, left, eh, ew)


def test_refusals_are_raised_at_construction():
    from unite_b200.augment import SpatialAugment
    with pytest.raises(ValueError, match="recount"):
        SpatialAugment(recount=2)
    with pytest.raises(ValueError, match="remode"):
        SpatialAugment(remode="gauss")
    with pytest.raises(ValueError, match="multiple of the 16-pixel"):
        SpatialAugment(crop_size=200)
    assert SpatialAugment().remode == "pixel" and SpatialAugment().erase_mode == 2 and SpatialAugment(remode="const").erase_mode == 0


def _frames(*shape):
    return torch.randint(0, 256, shape, generator=torch.Generator().manual_seed(0), dtype=torch.uint8)


def test_clip_shape_under_augmentation():
    """Frames of any size stand for the augmented [B,3,T,S,S] clip (the cutmix box is drawn on it); fp32 clips are refused."""
    from unite_b200 import ops
    assert ops.clip_shape(_frames(4, 8, 240, 427, 3), paired=True, crop_size=224) == (4, 3, 8, 224, 224)
    assert ops.clip_shape(_frames(3, 8, 17, 5, 3), crop_size=16) == (3, 3, 8, 16, 16)
    with pytest.raises(ValueError, match="uint8 frames"):
        ops.clip_shape(torch.zeros(2, 3, 8, 224, 224), crop_size=224)
    with pytest.raises(ValueError, match="even"):
        ops.clip_shape(_frames(3, 8, 240, 427, 3), paired=True, crop_size=224)
    with pytest.raises(ValueError, match="contiguous"):
        ops.clip_shape(_frames(2, 4, 32, 64, 3)[:, :, :, ::2], crop_size=16)


def test_the_mixup_draw_sees_the_augmented_clip():
    from unite_b200 import mixup as M
    from unite_b200 import ops
    cfg = dict(mixup_alpha=0., cutmix_alpha=1.0, label_smoothing=0.1, num_classes=12)
    np.random.seed(10)
    want = M.draw(M.Mixup(**cfg), (4, 3, 8, 224, 224))
    np.random.seed(10)
    got = M.draw(M.Mixup(**cfg), ops.clip_shape(_frames(4, 8, 240, 427, 3), crop_size=224))
    assert got == want and got.use_cutmix


@pytest.mark.parametrize("bad,msg", [(lambda: torch.zeros(4, 3, 8, 32, 32), "uint8 frames"),
                                     (lambda: _frames(3, 8, 40, 40, 3), "even")])
def test_stage2_refuses_before_any_device_work(bad, msg):
    """Stage2Engine.step (before the draw's upload and the optimizer's), finetune_step (before the DropPath draw) refuse an fp32
    batch under spatial_aug, and an odd uint8 batch under mixup, with ValueError on a machine without a GPU."""
    from unite_b200 import mixup as M
    from unite_b200.augment import SpatialAugment
    from unite_b200.engine_for_finetuning import Stage2Engine, finetune_step
    x = bad()
    aug = SpatialAugment(crop_size=32)
    _seed(0)
    d = aug.draw((x.shape[0], 8, 40, 40, 3))
    eng = Stage2Engine.__new__(Stage2Engine)                       # no arena, no optimizer, no buffers: any use would fail otherwise
    mix = M.MixDraw(True, 0.3, False, ((0, 0), (0, 0), (0, 0)), 0.3)
    with pytest.raises(ValueError, match=msg):
        eng.step(x, torch.zeros(x.shape[0], dtype=torch.long), mix=mix, smoothing=0.1, aug=d)
    buf = types.SimpleNamespace(aug=aug, batch=x.shape[0])
    with pytest.raises(ValueError, match=msg):
        finetune_step(None, x, None, None, mix=types.SimpleNamespace(clip=object(), target=object()), aug=buf)


def test_run_forward_refuses_a_crop_the_model_cannot_take():
    """num_patches follows crop_size: a crop giving another token count is refused before the shadow cast or any launch."""
    from unite_b200 import finetune_core
    from unite_b200.augment import SpatialAugment
    core = finetune_core.FinetuneCore.__new__(finetune_core.FinetuneCore)
    core.N, core.tubelet = 8 * 14 * 14, 1
    core.sync_shadow = lambda: pytest.fail("launched before the refusal")
    buf = types.SimpleNamespace(aug=SpatialAugment(crop_size=112), batch=2)
    with pytest.raises(ValueError, match="tokens"):
        core.run_forward(_frames(2, 8, 240, 320, 3), None, False, aug=buf)
    with pytest.raises(ValueError, match="uint8"):
        core.run_forward(torch.zeros(2, 3, 8, 224, 224), None, False, aug=buf)


def test_fp32_and_uint8_launch_lists_are_unchanged_without_augmentation(monkeypatch):
    """FinetuneCore.run_forward with no augmentation launches what it launched before (the augmented im2col is never reached);
    with one, the augmented im2col replaces the other im2cols."""
    from unite_b200 import finetune_core, ops
    from unite_b200.augment import SpatialAugment
    calls = []

    def rec(name):
        def f(*a, **k):
            calls.append(name)
            return a[1] if name.startswith("patchify") else None
        return f
    for name in ("patchify", "patchify_mix", "patchify_u8", "patchify_mix_u8", "patchify_aug_u8", "meanpool_fwd", "layernorm_fwd",
                 "linear_small_fwd"):
        monkeypatch.setattr(ops, name, rec(name))
    core = finetune_core.FinetuneCore.__new__(finetune_core.FinetuneCore)
    core.sync_shadow = lambda: None
    core.N, core.tubelet, core.D, core.depth, core.C, core.eps = 16, 1, 8, 1, 3, 1e-6
    core._pos_full = {2: None}
    core.arena = types.SimpleNamespace(p32=lambda n: None)
    ws = types.SimpleNamespace(x_at=lambda l: torch.zeros(2 * 16 * 8))
    core.trunk = types.SimpleNamespace(forward=lambda *a: ws)
    f32, u8 = torch.zeros(2, 3, 4, 16, 16), _frames(2, 4, 16, 16, 3)
    for x in (f32, u8):
        for mix in (None, torch.zeros(10)):
            core.run_forward(x, None, False, mix=mix)
    buf = types.SimpleNamespace(aug=SpatialAugment(crop_size=32), batch=2, draw=None, rng=None)
    core.run_forward(_frames(2, 4, 23, 37, 3), None, False, aug=buf)
    core.run_forward(_frames(2, 4, 23, 37, 3), None, False, mix=torch.zeros(10), aug=buf)
    im2col = [c for c in calls if c.startswith("patchify")]
    assert im2col == ["patchify", "patchify_mix", "patchify_u8", "patchify_mix_u8", "patchify_aug_u8", "patchify_aug_u8"]
