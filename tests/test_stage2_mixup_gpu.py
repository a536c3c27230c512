"""Stage-2 mixup / cutmix / label smoothing on the GPU against tests/mixup_ref.py (timm 0.4.12 restated) and the oracle: the fused
im2col bit for bit, the soft-target loss against fp64 torch, the whole step, CUDA-graph replay and train_one_epoch."""
from functools import partial

import numpy as np
import pytest
import torch

from tests import mixup_ref as R
from tests.util import cosine, load_golden, oracle_cfgs, rel_l2, seeded_states

pytestmark = pytest.mark.gpu
LOSS_TOL = 1e-3


def _build_vit(scfg, drop_path_rate=0.0):
    import torch.nn as nn
    from unite_b200.modeling_finetune import VisionTransformer
    return VisionTransformer(img_size=scfg.img_size, patch_size=scfg.patch_size, embed_dim=scfg.embed_dim, depth=scfg.depth,
                             num_heads=scfg.num_heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                             num_classes=scfg.num_classes, all_frames=scfg.num_frames, tubelet_size=scfg.tubelet_size,
                             init_scale=0.001, use_mean_pooling=True, drop_path_rate=drop_path_rate)


def _tiny_vit(head_std=None, drop_path_rate=0.0, seed=17):
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    _, _, vsd = seeded_states(fix)
    vsd = dict(vsd)
    if head_std is not None:
        g = torch.Generator().manual_seed(seed)
        vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=g) * head_std
    vit = _build_vit(scfg, drop_path_rate)
    vit.load_state_dict(vsd, strict=True)
    return scfg, vsd, vit.cuda()


def _buffer(d, smoothing, C, mix_clips=True):
    from unite_b200.mixup import MixBuffer
    buf = MixBuffer(torch.device("cuda"), mix_clips=mix_clips)
    buf.upload(d.packed(smoothing, C))
    return buf


# ---- 1. ub_patchify_mix: bit-exact against patchify of the clip mixed by timm's code on the device ----------------------------------
CASES = [
    # B, T, H, W, tubelet, kind, parameter (lam for mixup, timm's (yl, yh, xl, xh) for cutmix, "minmax" for a rand_bbox_minmax box)
    (2, 4, 32, 32, 2, "mix", 0.37),
    (2, 4, 32, 32, 1, "mix", 1.0),
    (2, 4, 32, 32, 1, "copy", None),
    (4, 8, 48, 32, 2, "cut", (8, 20, 5, 30)),          # T slice [8, 8): empty
    (4, 8, 48, 32, 1, "cut", (3, 6, 10, 40)),          # partial T slice
    (2, 4, 32, 32, 2, "cut", (0, 32, 0, 32)),          # whole T and H
    (6, 8, 64, 96, 2, "cut", "minmax"),
    (6, 8, 64, 96, 1, "mix", 0.81),                    # non-square
    (32, 8, 224, 224, 2, "mix", 0.4217),               # the bench shape
    (32, 8, 224, 224, 2, "cut", (2, 7, 30, 190)),
]


@pytest.mark.parametrize("B,T,H,W,tub,kind,par", CASES)
def test_patchify_mix_is_bit_exact_against_timm_mix_then_patchify(B, T, H, W, tub, kind, par):
    from unite_b200 import ops
    from unite_b200.mixup import NO_MIX, MixDraw, clip_box
    g = torch.Generator().manual_seed(B * 1000 + T + H)
    x = torch.randn(B, 3, T, H, W, generator=g).cuda()
    keep = x.clone()
    ref = x.clone()
    if kind == "copy":
        d = NO_MIX
    elif kind == "mix":
        lam = par
        x_flipped = ref.flip(0).mul_(1. - lam)                                        # timm Mixup._mix_batch, literally
        ref.mul_(lam).add_(x_flipped)
        d = MixDraw(True, lam, False, ((0, 0), (0, 0), (0, 0)), lam)
    else:
        if par == "minmax":
            np.random.seed(5)
            (yl, yh, xl, xh), lam = R.cutmix_bbox_and_lam(ref.shape, 0.5, ratio_minmax=(0.2, 0.8))
        else:
            (yl, yh, xl, xh), lam = par, 0.5
        ref[:, :, yl:yh, xl:xh] = ref.flip(0)[:, :, yl:yh, xl:xh]
        d = MixDraw(True, 0.5, True, clip_box(ref.shape, yl, yh, xl, xh), float(lam))
    n_tok = B * (T // tub) * (H // 16) * (W // 16)
    want = torch.empty(n_tok, 3 * tub * 256, device="cuda", dtype=torch.bfloat16)
    got = torch.full_like(want, float("nan"))
    ops.patchify(ref, want, tub)
    ops.patchify_mix(x, got, _buffer(d, 0.1, 10).clip, tub)
    torch.cuda.synchronize()
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
    assert torch.equal(x, keep), "the input clip must not be written"


def test_patchify_mix_refuses_an_odd_batch():
    from unite_b200 import ops
    from unite_b200._cabi import UBError
    from unite_b200.mixup import NO_MIX
    x = torch.zeros(3, 3, 2, 16, 16, device="cuda")
    with pytest.raises(UBError, match="even"):
        ops.patchify_mix(x, torch.empty(6, 3 * 256, device="cuda", dtype=torch.bfloat16), _buffer(NO_MIX, 0., 10).clip, 1)


# ---- 2. ub_soft_target_ce against fp64 torch --------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [12, 400])
@pytest.mark.parametrize("lam,smoothing", [(0.3, 0.1), (0.77, 0.0), (1.0, 0.1)])
def test_soft_target_ce_against_fp64_timm_losses(C, lam, smoothing):
    from unite_b200 import ops
    from unite_b200.mixup import MixDraw
    B = 16
    g = torch.Generator().manual_seed(C + int(lam * 100))
    logits = torch.randn(B, C, generator=g) * 3
    labels = torch.randint(0, C, (B,), generator=g)
    x = logits.double().requires_grad_(True)
    target = R.mixup_target(labels, C, lam, smoothing, "cpu").double()
    loss = R.SoftTargetCrossEntropy()(x, target)
    loss.backward()
    if lam == 1.0:
        ls = R.LabelSmoothingCrossEntropy(smoothing)(logits.double(), labels)
        assert abs(ls.item() - loss.item()) < 1e-6 * loss.item()
    buf = _buffer(MixDraw(lam != 1.0, lam, False, ((0, 0), (0, 0), (0, 0)), lam), smoothing, C)
    acc = torch.zeros(1, device="cuda")
    dl = torch.empty(B, C, device="cuda")
    ops.soft_target_ce(logits.cuda(), labels.cuda().int(), buf.target, 1.0 / B, acc, dl)
    torch.cuda.synchronize()
    l_rel = abs(acc.item() - loss.item()) / loss.item()
    d_err = (dl.cpu().double() - x.grad).abs().max().item() / x.grad.abs().max().item()
    print(f"C={C} lam={lam} s={smoothing}: loss rel {l_rel:.1e}, dlogits {d_err:.1e}")
    assert l_rel < 1e-6 and d_err < 1e-6


# ---- 3. the whole step against the oracle ---------------------------------------------------------------------------------------
def _oracle_soft_step(vsd, videos, target, scfg, with_grads):
    from oracle import unite_oracle as O
    params = {k: v.detach().clone().requires_grad_(with_grads) for k, v in vsd.items()}
    logits = O.vit_forward(params, videos, scfg)
    loss = R.SoftTargetCrossEntropy()(logits, target)
    res = dict(logits=logits.detach(), loss=loss.detach())
    if with_grads:
        loss.backward()
        res["grads"] = {k: v.grad for k, v in params.items() if v.grad is not None}
    return res


@pytest.mark.parametrize("kind", ["mixup", "cutmix", "smoothing"])
def test_stage2_soft_loss_at_256_clips_meets_the_loss_gate(kind):
    """As test_stage2_loss_at_256_clips_meets_the_loss_gate, with the clip mixed by timm's Mixup and timm's loss on top."""
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import finetune_step
    scfg, vsd, vit = _tiny_vit(head_std=0.05)
    vit.eval()
    n, C = 256, scfg.num_classes
    g = torch.Generator().manual_seed(23)
    videos = torch.randn(n, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g)
    labels = torch.randint(0, C, (n,), generator=g)
    if kind == "smoothing":
        mixed, target = videos, R.mixup_target(labels, C, 1.0, 0.1, "cpu")
        buf = _buffer(M.NO_MIX, 0.1, C, mix_clips=False)
    else:
        cfg = dict(mixup_alpha=0.8, cutmix_alpha=0.) if kind == "mixup" else dict(mixup_alpha=0., cutmix_alpha=1.0)
        np.random.seed(4)
        mixed, target = R.Mixup(label_smoothing=0.1, num_classes=C, **cfg)(videos.clone(), labels)
        np.random.seed(4)
        d = M.draw(M.Mixup(label_smoothing=0.1, num_classes=C, **cfg), videos.shape)
        assert d.apply and d.use_cutmix == (kind == "cutmix")
        buf = _buffer(d, 0.1, C)
    ref = _oracle_soft_step(vsd, mixed, target, scfg, with_grads=False)
    loss = torch.zeros(1, device="cuda")
    dev_videos = videos.cuda()
    logits = finetune_step(vit, dev_videos, labels.cuda(), loss, mix=buf)
    torch.cuda.synchronize()
    assert rel_l2(logits, ref["logits"]) < 1e-2
    l_rel = abs(loss.item() - ref["loss"].item()) / ref["loss"].item()
    print(f"stage-2 {kind} @{n} clips: {loss.item():.6f} vs {ref['loss'].item():.6f} ({l_rel:.1e})")
    assert l_rel < LOSS_TOL
    assert torch.equal(dev_videos.cpu(), videos)


def test_full_vitb16_stage2_mixup_gradients_against_oracle():
    from oracle import unite_oracle as O
    from oracle.weights import seeded_state
    from unite_b200.engine_for_finetuning import finetune_step
    from unite_b200.mixup import MixDraw
    scfg = O.StudentCfg(num_classes=12)
    vit = _build_vit(scfg)
    vsd = seeded_state({k: tuple(v.shape) for k, v in vit.state_dict().items()}, 3)
    g = torch.Generator().manual_seed(41)
    vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=g) * 0.02
    vit.load_state_dict(vsd, strict=True)
    vit = vit.cuda().eval()
    videos = torch.randn(2, 3, 8, 224, 224, generator=g)
    labels = torch.tensor([3, 7])
    lam = 0.62
    mixed = videos.clone()
    x_flipped = mixed.flip(0).mul_(1. - lam)
    mixed.mul_(lam).add_(x_flipped)
    ref = _oracle_soft_step(vsd, mixed, R.mixup_target(labels, 12, lam, 0.1, "cpu"), scfg, with_grads=True)
    loss = torch.zeros(1, device="cuda")
    buf = _buffer(MixDraw(True, lam, False, ((0, 0), (0, 0), (0, 0)), lam), 0.1, 12)
    finetune_step(vit, videos.cuda(), labels.cuda(), loss, mix=buf)
    torch.cuda.synchronize()
    assert abs(loss.item() - ref["loss"].item()) < 5e-3 * ref["loss"].item()
    arena = vit.core().arena
    worst_c, worst_r = 1.0, 0.0
    for k, g_ref in ref["grads"].items():
        if g_ref.numel() < 4096:
            continue
        c, r = cosine(arena.g32(k), g_ref), rel_l2(arena.g32(k), g_ref)
        worst_c, worst_r = min(worst_c, c), max(worst_r, r)
        assert c >= 0.999 and r <= 2e-2, (k, c, r)
    print(f"stage-2 full size mixup grads: worst cosine {worst_c:.6f}, worst rel-L2 {worst_r:.2e}")


# ---- 4. CUDA-graph replay ----------------------------------------------------------------------------------------------------------
def test_stage2_mixup_graph_replay_matches_eager_steps():
    """Six Stage2Engine steps under a graph and six eager ones from the same numpy seed, prob < 1 so that unmixed, mixup and
    cutmix steps all occur (seed 1 draws mixup, cutmix, cutmix, mixup, cutmix, none): one graph serves them all, each replay
    reading its own draw."""
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    g = torch.Generator().manual_seed(78)
    shape = (3, scfg.num_frames, scfg.img_size, scfg.img_size)
    x = torch.randn(6, *shape, generator=g).cuda()
    y = torch.randint(0, scfg.num_classes, (6,), generator=g).cuda()

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 2e-4, 0.05, (0.9, 0.999), 1e-8
    runs = []
    for use_graph in (True, False, False):
        _, _, vit = _tiny_vit(drop_path_rate=0.2)
        vit.train()
        L = vit.get_num_layers()
        asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])
        opt = create_optimizer(Args, vit, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
        eng = Stage2Engine(vit, opt, use_graph=use_graph)
        np.random.seed(1)
        mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, prob=0.6, switch_prob=0.5, label_smoothing=0.1, num_classes=scfg.num_classes)
        losses, kinds = [], []
        for s in range(6):
            d = M.draw(mixer, x.shape)
            kinds.append("cut" if d.use_cutmix else ("mix" if d.apply else "none"))
            losses.append(eng.step(x, y, mix=d, smoothing=0.1).clone())
        torch.cuda.synchronize()
        runs.append((torch.cat(losses).cpu(), eng.stats.cpu(), vit.core().arena.params.clone().cpu(), eng, kinds))
    (l_g, st_g, p_g, eng_g, kinds), (l_e, st_e, p_e, _, _), (l_e2, _, p_e2, _, _) = runs
    assert set(kinds[2:]) == {"none", "mix", "cut"}, kinds
    assert len(eng_g.graphs._graphs) == 1
    noise_l, noise_p = ((l_e - l_e2).abs() / l_e.abs()).max().item(), rel_l2(p_e, p_e2)
    d_l, d_p = ((l_g - l_e).abs() / l_e.abs()).max().item(), rel_l2(p_g, p_e)
    print(f"stage-2 mixup graph vs eager: loss {d_l:.2e} (eager vs eager {noise_l:.2e}), weights {d_p:.2e} (eager vs eager {noise_p:.2e})")
    assert d_l <= max(2e-5, 4 * noise_l), (l_g, l_e)
    assert torch.allclose(st_g, st_e, rtol=1e-4), (st_g, st_e)
    assert d_p <= max(1e-5, 4 * noise_p)


# ---- 5. train_one_epoch ------------------------------------------------------------------------------------------------------------
def _fresh_opt(vit):
    from unite_b200.optim_factory import create_optimizer

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    return create_optimizer(Args, vit)


def test_train_one_epoch_with_mixup_learns_and_reports_no_class_acc():
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import train_one_epoch
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    g = torch.Generator().manual_seed(5)
    batch = (torch.randn(4, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g),
             torch.randint(0, scfg.num_classes, (4,), generator=g), torch.zeros(4), {})
    crit = M.SoftTargetCrossEntropy()
    cfg = dict(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1, num_classes=scfg.num_classes)
    _, _, vit = _tiny_vit(drop_path_rate=0.1)
    opt = _fresh_opt(vit)
    np.random.seed(0)
    mixer = M.Mixup(**cfg)
    s0 = train_one_epoch(vit, crit, [batch] * 2, opt, "cuda", 0, None, mixup_fn=mixer, lr_schedule_values=[2e-3] * 60)
    s1 = train_one_epoch(vit, crit, [batch] * 40, opt, "cuda", 1, None, mixup_fn=mixer, lr_schedule_values=[2e-3] * 60, start_steps=2)
    assert "class_acc" not in s0 and "class_acc" not in s1
    print(f"mixup train_one_epoch: {s0['loss']:.4f} -> {s1['loss']:.4f}")
    assert opt.step_count == 42 and s1["loss"] < s0["loss"]
    s2 = train_one_epoch(vit, crit, [batch] * 4, opt, "cuda", 2, None, mixup_fn=mixer, update_freq=2)
    assert "class_acc" not in s2 and np.isfinite(s2["loss"]) and opt.step_count == 44
    s3 = train_one_epoch(vit, M.LabelSmoothingCrossEntropy(0.1), [batch] * 2, opt, "cuda", 3, None)
    assert "class_acc" in s3 and np.isfinite(s3["loss"])
    with pytest.raises(ValueError):
        train_one_epoch(vit, crit, [(batch[0][:3], batch[1][:3])], opt, "cuda", 4, None, mixup_fn=mixer)


def test_package_and_reference_mixup_objects_train_alike():
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import train_one_epoch
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    g = torch.Generator().manual_seed(6)
    batches = [(torch.randn(4, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g),
                torch.randint(0, scfg.num_classes, (4,), generator=g)) for _ in range(5)]
    cfg = dict(mixup_alpha=0.8, cutmix_alpha=1.0, prob=0.7, label_smoothing=0.1, num_classes=scfg.num_classes)
    out = []
    for cls in (M.Mixup, R.Mixup):
        _, _, vit = _tiny_vit()
        opt = _fresh_opt(vit)
        np.random.seed(11)
        st = train_one_epoch(vit, M.SoftTargetCrossEntropy(), batches, opt, "cuda", 0, None, mixup_fn=cls(**cfg))
        out.append((st["loss"], vit.core().arena.params.clone().cpu(), np.random.rand()))
    assert out[0][2] == out[1][2], "both objects must consume the global RNG alike"
    # same draws; what remains is the run-to-run noise of fp32 reduce-adds
    assert abs(out[0][0] - out[1][0]) < 1e-4 * abs(out[1][0])
    assert rel_l2(out[0][1], out[1][1]) < 1e-3


def test_train_class_batch_with_soft_target_ce_gives_the_fused_gradients():
    from unite_b200 import mixup as M
    from unite_b200.engine_for_finetuning import finetune_step, train_class_batch
    scfg, _, vit = _tiny_vit(head_std=0.05)
    vit.eval()                                                                     # no DropPath draw in either pass
    C = scfg.num_classes
    g = torch.Generator().manual_seed(8)
    videos = torch.randn(8, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g).cuda()
    labels = torch.randint(0, C, (8,), generator=g).cuda()
    np.random.seed(2)
    mixed, target = R.Mixup(mixup_alpha=0.8, cutmix_alpha=0., label_smoothing=0.1, num_classes=C)(videos.clone(), labels)
    arena = vit.core().arena
    arena.grads.zero_()
    loss, _ = train_class_batch(vit, mixed, target, M.SoftTargetCrossEntropy())
    loss.backward()
    g_autograd = arena.grads.clone()
    arena.grads.zero_()
    np.random.seed(2)
    buf = _buffer(M.draw(M.Mixup(mixup_alpha=0.8, cutmix_alpha=0., label_smoothing=0.1, num_classes=C), videos.shape), 0.1, C)
    acc = torch.zeros(1, device="cuda")
    finetune_step(vit, videos, labels, acc, mix=buf)
    torch.cuda.synchronize()
    assert abs(acc.item() - loss.item()) < 1e-5 * loss.item()
    r = rel_l2(arena.grads, g_autograd)
    print(f"train_class_batch vs fused: loss {loss.item():.6f} / {acc.item():.6f}, grads rel-L2 {r:.2e}")
    assert r < 1e-4
