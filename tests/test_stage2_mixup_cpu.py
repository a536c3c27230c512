"""Stage-2 mixup without a GPU: the package's host draws against timm 0.4.12's (tests/mixup_ref.py), the box mapping against the
literal 5-D slice, the packed device values, and the configurations the fused loop refuses."""
import numpy as np
import pytest
import torch

from tests import mixup_ref as R

SHAPE = (4, 3, 8, 32, 48)          # [B,C,T,H,W]: H > T, so timm's H range (applied to T) is often clamped; W != H

CONFIGS = {
    "mixup": dict(mixup_alpha=0.8, cutmix_alpha=0.),
    "cutmix": dict(mixup_alpha=0., cutmix_alpha=1.0),
    "both": dict(mixup_alpha=0.8, cutmix_alpha=1.0),
    "minmax": dict(mixup_alpha=0., cutmix_minmax=(0.2, 0.8)),
    "prob": dict(mixup_alpha=0.8, cutmix_alpha=1.0, prob=0.5, switch_prob=0.3),
    "no_correct_lam": dict(mixup_alpha=0.8, cutmix_alpha=1.0, correct_lam=False),
}


def _ref_sequence(cfg, seed, n):
    np.random.seed(seed)
    ref = R.Mixup(label_smoothing=0.1, num_classes=10, **cfg)
    out = []
    for _ in range(n):
        x = torch.zeros(SHAPE)
        ref(x, torch.arange(SHAPE[0]) % 10)
        out.append(dict(ref.last))
    return out


@pytest.mark.parametrize("seed", [0, 1, 12345])
@pytest.mark.parametrize("name", list(CONFIGS))
def test_host_draws_match_timm_batch_mixup(name, seed):
    from unite_b200 import mixup as M
    n = 40
    ref = _ref_sequence(CONFIGS[name], seed, n)
    np.random.seed(seed)
    mine = M.Mixup(label_smoothing=0.1, num_classes=10, **CONFIGS[name])
    kinds = set()
    for r in ref:
        d = M.draw(mine, SHAPE)
        assert d.apply == (r["lam"] != 1.)
        assert d.lam == r["lam"] and d.use_cutmix == (r["use_cutmix"] and d.apply)
        assert d.target_lam == r["target_lam"]
        if d.use_cutmix:
            assert d.box == M.clip_box(SHAPE, *r["bbox"])
        kinds.add("cut" if d.use_cutmix else ("mix" if d.apply else "none"))
    want = {"mixup": {"mix"}, "cutmix": {"cut"}, "both": {"mix", "cut"}, "minmax": {"cut"}, "prob": {"mix", "cut", "none"},
            "no_correct_lam": {"mix", "cut"}}[name]
    assert kinds == want
    assert np.random.rand() == _after(CONFIGS[name], seed, n), "the draws must consume the global RNG exactly as timm does"


def _after(cfg, seed, n):
    _ref_sequence(cfg, seed, n)
    return np.random.rand()


def test_reference_mixup_object_draws_the_same_through_the_package():
    """The loop accepts the reference's own Mixup: it calls that object's _params_per_batch and maps the box itself."""
    from unite_b200 import mixup as M
    cfg = CONFIGS["both"]
    np.random.seed(7)
    theirs = R.Mixup(**cfg)
    a = [M.draw(theirs, SHAPE) for _ in range(21)]
    np.random.seed(7)
    b = [M.draw(M.Mixup(**cfg), SHAPE) for _ in range(21)]
    assert a == b


def test_uncorrected_lam_is_the_beta_draw_and_corrected_lam_uses_the_hw_area():
    from unite_b200 import mixup as M
    for correct in (True, False):
        np.random.seed(3)
        d = next(d for d in (M.draw(M.Mixup(mixup_alpha=0., cutmix_alpha=1.0, correct_lam=correct), SHAPE) for _ in range(50))
                 if d.apply)
        if not correct:
            assert d.target_lam == d.lam
        else:
            np.random.seed(3)
            ref = R.Mixup(mixup_alpha=0., cutmix_alpha=1.0)
            ref(torch.zeros(SHAPE), torch.zeros(SHAPE[0], dtype=torch.long))
            yl, yh, xl, xh = ref.last["bbox"]
            assert d.target_lam == 1. - (yh - yl) * (xh - xl) / float(SHAPE[3] * SHAPE[4])


@pytest.mark.parametrize("bbox", [(0, 8, 0, 32), (2, 5, 10, 30), (6, 20, 4, 40), (9, 30, 0, 48), (0, 0, 3, 3), (31, 32, 47, 48),
                                  (0, 32, 0, 48)])
def test_box_mapping_matches_the_literal_slice_of_a_5d_clip(bbox):
    from unite_b200.mixup import clip_box
    x = torch.arange(np.prod(SHAPE), dtype=torch.float32).view(SHAPE)
    yl, yh, xl, xh = bbox
    lit = x.clone()
    lit[:, :, yl:yh, xl:xh] = lit.flip(0)[:, :, yl:yh, xl:xh]
    (t0, t1), (h0, h1), (w0, w1) = clip_box(SHAPE, yl, yh, xl, xh)
    assert 0 <= t0 <= t1 <= SHAPE[2] and 0 <= h0 <= h1 <= SHAPE[3] and (w0, w1) == (0, SHAPE[4])
    mine = x.clone()
    mine[:, :, t0:t1, h0:h1, w0:w1] = x.flip(0)[:, :, t0:t1, h0:h1, w0:w1]
    assert torch.equal(mine, lit)


def test_packed_values_follow_timm_rounding():
    from unite_b200.mixup import NO_MIX, MixDraw
    d = MixDraw(True, 0.3, False, ((0, 0), (0, 0), (0, 0)), 0.3)
    v = torch.tensor(d.packed(0.1, 400), dtype=torch.float32)
    assert v[0] == 1 and v[1] == np.float32(0.3) and v[2] == np.float32(1. - 0.3) and v[3] == 0
    assert v[10] == np.float32(0.3) and v[11] == np.float32(1. - 0.1 + 0.1 / 400) and v[12] == np.float32(0.1 / 400)
    t = R.mixup_target(torch.tensor([3, 5]), 400, 0.3, 0.1, "cpu")
    assert t[0, 3] == np.float32(np.float32(0.3) * v[11] + np.float32(0.7) * v[12])
    n = torch.tensor(NO_MIX.packed(0.0, 12))
    assert n[0] == 0 and n[1] == 1 and n[2] == 0 and n[10] == 1 and n[11] == 1 and n[12] == 0


def test_loss_table():
    from unite_b200 import mixup as M
    mix = M.Mixup(label_smoothing=0.1, num_classes=10)
    ce = torch.nn.CrossEntropyLoss
    assert M.resolve_loss(M.SoftTargetCrossEntropy(), mix) == 0.1
    assert M.resolve_loss(R.SoftTargetCrossEntropy(), mix) == 0.1                     # recognised by class name
    assert M.resolve_loss(ce(), mix) == 0.1
    assert M.resolve_loss(None, None) is None and M.resolve_loss(ce(), None) is None
    assert M.resolve_loss(M.LabelSmoothingCrossEntropy(0.2), None) == 0.2
    assert M.resolve_loss(R.LabelSmoothingCrossEntropy(0.3), None) == 0.3
    assert M.resolve_loss(ce(label_smoothing=0.1), None) == pytest.approx(0.1)
    for crit, fn in ((M.SoftTargetCrossEntropy(), None), (M.LabelSmoothingCrossEntropy(0.1), mix), (ce(label_smoothing=0.1), mix),
                     (ce(weight=torch.ones(10)), None), (ce(reduction="sum"), mix), (torch.nn.MSELoss(), None)):
        with pytest.raises(NotImplementedError):
            M.resolve_loss(crit, fn)


def test_refusals():
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import train_one_epoch
    for mode in ("elem", "pair"):
        with pytest.raises(NotImplementedError):
            M.Mixup(mode=mode)
        with pytest.raises(NotImplementedError):
            M.resolve_loss(M.SoftTargetCrossEntropy(), R.Mixup(mode=mode))
        with pytest.raises(NotImplementedError):
            train_one_epoch(torch.nn.Linear(2, 2), M.SoftTargetCrossEntropy(), [], None, "cpu", 0, mixup_fn=R.Mixup(mode=mode))
    np.random.seed(0)
    state = np.random.get_state()[1].copy()
    with pytest.raises(ValueError):
        M.draw(M.Mixup(), (7, 3, 8, 32, 32))                                             # stage2.sh's 7 clips per GPU
    assert np.array_equal(np.random.get_state()[1], state), "an odd batch is refused before any draw"
    with pytest.raises(NotImplementedError):
        M.Mixup()(torch.zeros(SHAPE), torch.zeros(4, dtype=torch.long))
    for crit, fn in ((M.SoftTargetCrossEntropy(), None), (torch.nn.MSELoss(), M.Mixup())):
        with pytest.raises(NotImplementedError):
            train_one_epoch(torch.nn.Linear(2, 2), crit, [], None, "cpu", 0, mixup_fn=fn)
    with pytest.raises(NotImplementedError, match="EMA"):
        train_one_epoch(torch.nn.Linear(2, 2), None, [], None, "cpu", 0, model_ema=object())


def test_timm_losses_agree_with_the_soft_target_form():
    """LabelSmoothingCrossEntropy(s) == SoftTargetCrossEntropy(mixup_target(lam=1, s)) == CrossEntropyLoss(label_smoothing=s):
    the three criteria the fused loss stands for with lam = 1."""
    g = torch.Generator().manual_seed(0)
    x = torch.randn(6, 12, generator=g, dtype=torch.float64)
    y = torch.randint(0, 12, (6,), generator=g)
    a = R.LabelSmoothingCrossEntropy(0.1)(x, y)
    b = R.SoftTargetCrossEntropy()(x, R.mixup_target(y, 12, 1.0, 0.1, "cpu").double())
    c = torch.nn.CrossEntropyLoss(label_smoothing=0.1)(x, y)
    assert torch.allclose(a, c, rtol=1e-12) and torch.allclose(a, b, rtol=1e-6)        # mixup_target is fp32
