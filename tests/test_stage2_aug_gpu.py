"""ub_patchify_aug_u8 and the stage-2 step under SpatialAugment, on the device.  The reference is the loader's order in torch:
normalise (oracle.unite_oracle.normalize_frames_u8), slice the crop, F.interpolate(bilinear, align_corners=False), flip, erase
(zeros, or the noise the test supplies), mix as timm does, then the im2col — the kernel resamples normalised taps, so its rows may
differ from it by fp32 rounding, turned into at most one bf16 ulp where the rounding of a value changes."""
import random
from functools import partial

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.util import load_golden, oracle_cfgs, rel_l2, seeded_states

pytestmark = pytest.mark.gpu
GUARD = 64                                                      # NaN rows before and after the output


def _frames(shape, seed):
    return torch.randint(0, 256, shape, generator=torch.Generator().manual_seed(seed), dtype=torch.uint8)


def _norm(frames):
    from oracle.unite_oracle import normalize_frames_u8
    return normalize_frames_u8(frames)


def _augment_ref(frames, params, S, mode=0, noise=None):
    """The loader's order on the normalised clip [B,3,T,S,S] (fp32, on the device), with the draws `params` [B,10]."""
    x = _norm(frames).cuda()
    out = []
    for b in range(x.shape[0]):
        i, j, h, w, flip, erase, top, left, eh, ew = (int(v) for v in params[b])
        c = F.interpolate(x[b][..., i:i + h, j:j + w], size=(S, S), mode="bilinear", align_corners=False)     # [3,T,S,S]
        if flip:
            c = c.flip(-1)
        if erase:
            if mode == 0:
                c[:, :, top:top + eh, left:left + ew] = 0.
            elif mode == 1:
                c[:, :, top:top + eh, left:left + ew] = noise[b].permute(1, 0)[:, :, None, None]
            else:
                c[:, :, top:top + eh, left:left + ew] = noise[b].permute(1, 0, 2, 3)[:, :, top:top + eh, left:left + ew]
        out.append(c)
    return torch.stack(out)


def _mix_ref(ref, d):
    if not d.apply:
        return ref
    if d.use_cutmix:
        (t0, t1), (h0, h1), (w0, w1) = d.box
        ref[:, :, t0:t1, h0:h1, w0:w1] = ref.flip(0)[:, :, t0:t1, h0:h1, w0:w1].clone()
        return ref
    x_flipped = ref.flip(0).mul_(1. - d.lam)                                       # timm Mixup._mix_batch, literally
    return ref.mul_(d.lam).add_(x_flipped)


def _rows32(clip, tub):
    B, _, T, S, _ = clip.shape
    g = S // 16
    return clip.reshape(B, 3, T // tub, tub, g, 16, g, 16).permute(0, 2, 4, 6, 1, 3, 5, 7).reshape(-1, 3 * tub * 256)


def _run_kernel(x, draw_dev, S, tub, mode=0, mix=None, noise=None, rng=None):
    from unite_b200 import ops
    B, T = x.shape[:2]
    n = B * (T // tub) * (S // 16) ** 2
    buf = torch.full((n + 2 * GUARD, 3 * tub * 256), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.patchify_aug_u8(x, buf[GUARD:GUARD + n], draw_dev, S, tub, mode, mix=mix, noise=noise, rng=rng)
    torch.cuda.synchronize()
    assert torch.isnan(buf[:GUARD].float()).all() and torch.isnan(buf[GUARD + n:].float()).all(), "wrote outside its rows"
    return buf[GUARD:GUARD + n]


def _assert_close(got, ref32):
    """At most one bf16 ulp, and only where the fp32 reference lies within 1e-5 of the rounding boundary between the two."""
    want = ref32.to(torch.bfloat16)
    assert not torch.isnan(got.float()).any()
    diff = got.view(torch.int16) != want.view(torch.int16)
    if not diff.any():
        return
    g, w, r = got.float()[diff], want.float()[diff], ref32[diff]
    ulps = (got.view(torch.int16)[diff].int() - want.view(torch.int16)[diff].int()).abs()
    boundary = (g + w) / 2
    print(f"{int(diff.sum())} of {got.numel()} elements one ulp apart; max distance to the boundary {(r - boundary).abs().max().item():.2e}")
    assert (ulps <= 1).all(), ulps.max()
    assert ((r - boundary).abs() <= 1e-5 * torch.clamp(r.abs(), min=1.0)).all()


def _draws(B, H, W, S, seed, **kw):
    from unite_b200.augment import SpatialAugment
    random.seed(seed)
    np.random.seed(seed)
    return SpatialAugment(crop_size=S, **kw).draw((B, 1, H, W, 3)).params


EDGE = np.array([[0, 0, 20, 30, 1, 1, 0, 0, 10, 12],             # crop and erasing box at the top-left corner, flipped
                 [0, 0, 0, 0, 0, 1, 0, 0, 0, 0],                # (filled per shape below)
                 [0, 0, 1, 1, 0, 1, 20, 30, 12, 2],             # a 1x1 crop; box at the bottom-right of the S=32 crop
                 [0, 0, 0, 0, 1, 0, 0, 0, 0, 0]], dtype=np.int32)


def _edge_draws(B, H, W, S):
    p = np.tile(EDGE, (B // 4 + 1, 1))[:B].copy()
    for k in range(B):
        if k % 4 == 0:
            p[k, 2:4] = (min(20, H), min(30, W))
        if k % 4 == 1:
            p[k, 0:4] = (H - min(H, 17), W - min(W, 23), min(H, 17), min(W, 23))   # bottom-right crop
            p[k, 6:10] = (S - 5, 0, 5, S)                                           # full-width box on the last rows
        if k % 4 == 2:
            p[k, 0:2] = (H - 1, W - 1)
            p[k, 6:10] = (S - 12, S - 2, 12, 2)
        if k % 4 == 3:
            p[k, 0:4] = (0, 0, H, W)                                                # the whole frame
    return p


CASES = [
    # B, T, H, W, S, tub, draws, mix kind, erase mode
    (3, 4, 256, 320, 224, 2, "drawn", None, 0),
    (5, 4, 240, 427, 224, 1, "drawn", None, 2),
    (4, 4, 240, 427, 224, 2, "drawn", "mixup", 1),
    (4, 2, 256, 320, 224, 1, "drawn", "cutmix", 0),
    (8, 4, 40, 56, 32, 2, "edge", None, 0),
    (8, 4, 40, 56, 32, 1, "edge", "mixup", 2),
    (8, 2, 33, 17, 32, 2, "edge", "cutmix", 1),
    (7, 2, 12, 9, 32, 1, "drawn", None, 2),                       # upsampling from frames smaller than the crop
]


@pytest.mark.parametrize("B,T,H,W,S,tub,kind,mixk,mode", CASES)
def test_patchify_aug_u8_matches_the_loader_order_in_torch(B, T, H, W, S, tub, kind, mixk, mode):
    from unite_b200 import mixup as M
    from unite_b200 import ops
    frames = _frames((B, T, H, W, 3), B * 100 + H + W)
    params = _edge_draws(B, H, W, S) if kind == "edge" else _draws(B, H, W, S, B + T, reprob=0.7)
    g = torch.Generator().manual_seed(5)
    noise = None
    if mode == 1:
        noise = torch.randn(B, T, 3, generator=g).cuda()
    elif mode == 2:
        noise = torch.randn(B, T, 3, S, S, generator=g).cuda()
    d = M.NO_MIX
    if mixk == "mixup":
        d = M.MixDraw(True, 0.37, False, ((0, 0), (0, 0), (0, 0)), 0.37)
    elif mixk == "cutmix":
        d = M.MixDraw(True, 0.5, True, M.clip_box((B, 3, T, S, S), 1, T, 3, S - 4), 0.5)
    mix = None
    if mixk is not None:
        mix = M.MixBuffer(torch.device("cuda"))
        mix.upload(d.packed(0.1, 12))
    x = frames.cuda()
    got = _run_kernel(x, torch.from_numpy(params).cuda(), S, tub, mode, mix=None if mix is None else mix.clip, noise=noise)
    ref = _mix_ref(_augment_ref(frames, params, S, mode, noise), d)
    _assert_close(got, _rows32(ref, tub))
    want16 = torch.empty_like(got)
    ops.patchify(ref.contiguous(), want16, tub)                   # the existing im2col of the torch-augmented clip
    torch.cuda.synchronize()
    assert ((got.view(torch.int16).int() - want16.view(torch.int16).int()).abs() <= 1).all()
    assert torch.equal(x.cpu(), frames), "the input frames must not be written"


@pytest.mark.parametrize("tub", [1, 2])
def test_identity_crop_equals_patchify_u8_bit_for_bit(tub):
    from unite_b200 import ops
    B, T, S = 3, 4, 224
    frames = _frames((B, T, S, S, 3), 77)
    x = frames.cuda()
    params = np.zeros((B, 10), dtype=np.int32)
    params[:, 2:4] = S
    got = _run_kernel(x, torch.from_numpy(params).cuda(), S, tub)
    want = ops.patchify_u8(x, torch.empty_like(got), tub)
    torch.cuda.synchronize()
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))


def _noise_setup(B=4, T=4, H=240, W=320, S=224, seed=3):
    frames = _frames((B, T, H, W, 3), seed)
    params = _draws(B, H, W, S, seed, reprob=1.0)
    params[:, 6:10] = (10, 20, 150, 140)                        # a large box: ~21000 pixels per frame
    return frames.cuda(), torch.from_numpy(params).cuda(), params


def test_pixel_noise_from_the_generator():
    """Outside the box the rows are those of the const erase; inside, standard normals: mean and variance within sampling bounds,
    different from one launch to the next (the device counter advances)."""
    x, dev_p, params = _noise_setup()
    B, T, S = 4, 4, 224
    rng = torch.zeros(2, dtype=torch.int64, device="cuda")
    const = _run_kernel(x, dev_p, S, 1, 0)
    a = _run_kernel(x, dev_p, S, 1, 2, rng=rng)
    assert rng.tolist() == [1, 0]
    b = _run_kernel(x, dev_p, S, 1, 2, rng=rng)
    assert rng.tolist() == [2, 0]
    mask = torch.zeros(B, 3, T, S, S, dtype=torch.bool, device="cuda")
    mask[:, :, :, 10:160, 20:160] = True
    inside = _rows32(mask, 1)
    assert torch.equal(a[~inside].view(torch.int16), const[~inside].view(torch.int16))
    assert torch.equal(b[~inside].view(torch.int16), const[~inside].view(torch.int16))
    v = a[inside].double()
    n = v.numel()
    print(f"pixel noise: n={n} mean {v.mean().item():.4f} var {v.var().item():.4f}")
    assert abs(v.mean().item()) < 5 / n ** 0.5 and abs(v.var().item() - 1) < 10 * (2 / n) ** 0.5
    assert (a[inside] != b[inside]).float().mean().item() > 0.99


def test_rand_noise_is_one_normal_per_frame_and_channel():
    x, dev_p, _ = _noise_setup()
    rng = torch.zeros(2, dtype=torch.int64, device="cuda")
    a = _run_kernel(x, dev_p, 224, 1, 1, rng=rng)
    # the clip back from its tubelet-1 im2col rows
    clip = a.float().reshape(4, 4, 14, 14, 3, 16, 16).permute(0, 4, 1, 2, 5, 3, 6).reshape(4, 3, 4, 224, 224)
    box = clip[:, :, :, 10:160, 20:160]
    per = box.amax(dim=(-1, -2))
    assert torch.equal(per, box.amin(dim=(-1, -2))), "one value per (clip, channel, frame)"
    n = per.numel()                                            # 48 normals, rounded to bf16 (a repeated value is possible)
    assert per.unique().numel() >= n - 4 and abs(per.double().var().item() - 1) < 0.6


def test_graph_replays_draw_fresh_noise_and_identical_rows_elsewhere():
    from unite_b200 import ops
    x, dev_p, _ = _noise_setup()
    rng = torch.zeros(2, dtype=torch.int64, device="cuda")
    n = 4 * 4 * 14 * 14
    out = torch.empty(n, 3 * 256, device="cuda", dtype=torch.bfloat16)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.patchify_aug_u8(x, out, dev_p, 224, 1, 2, rng=rng)                     # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        ops.patchify_aug_u8(x, out, dev_p, 224, 1, 2, rng=rng)
    g.replay()
    first = out.clone()
    g.replay()
    torch.cuda.synchronize()
    second = out.clone()
    mask = torch.zeros(4, 3, 4, 224, 224, dtype=torch.bool, device="cuda")
    mask[:, :, :, 10:160, 20:160] = True
    inside = _rows32(mask, 1)
    assert rng[0].item() == 3
    assert torch.equal(first[~inside].view(torch.int16), second[~inside].view(torch.int16))
    assert (first[inside] != second[inside]).float().mean().item() > 0.99


# ---- the stage-2 step ----------------------------------------------------------------------------------------------------------
def _tiny_vit(drop_path_rate=0.0):
    import torch.nn as nn
    from unite_b200.modeling_finetune import VisionTransformer
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    _, _, vsd = seeded_states(fix)
    vsd = dict(vsd)
    vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=torch.Generator().manual_seed(17)) * 0.05
    vit = VisionTransformer(img_size=scfg.img_size, patch_size=scfg.patch_size, embed_dim=scfg.embed_dim, depth=scfg.depth,
                            num_heads=scfg.num_heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                            num_classes=scfg.num_classes, all_frames=scfg.num_frames, tubelet_size=scfg.tubelet_size,
                            init_scale=0.001, use_mean_pooling=True, drop_path_rate=drop_path_rate)
    vit.load_state_dict(vsd, strict=True)
    return scfg, vit.cuda()


def _opt(vit):
    from unite_b200.optim_factory import create_optimizer

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    return create_optimizer(Args, vit)


def test_stage2_engine_with_spatial_aug_equals_the_fp32_step_on_the_torch_augmented_clip():
    """Stage2Engine (graph-replayed) fed uint8 frames of 80x104 pixels + SpatialAugment(remode='const'), with mixup / cutmix draws,
    against the same engine path fed the fp32 clip augmented in torch with the same draws."""
    from unite_b200 import mixup as M
    from unite_b200.augment import SpatialAugment
    from unite_b200.engine_for_finetuning import Stage2Engine
    scfg, _ = _tiny_vit()
    S, T, B, C = scfg.img_size, scfg.num_frames, 4, scfg.num_classes
    aug = SpatialAugment(crop_size=S, reprob=0.8, remode="const")
    frames = [_frames((B, T, 80, 104, 3), 400 + i) for i in range(3)]
    y = torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(4)).cuda()
    random.seed(0)
    np.random.seed(0)
    mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1, num_classes=C)
    steps = []
    for s in range(6):
        d = aug.draw(frames[s % 3].shape)
        steps.append((frames[s % 3], d, M.draw(mixer, (B, 3, T, S, S))))
    assert {m.use_cutmix for _, _, m in steps if m.apply} == {False, True}
    out = {}
    for name in ("u8", "f32"):
        _, vit = _tiny_vit()
        vit.train()
        eng = Stage2Engine(vit, _opt(vit), use_graph=True)
        losses = []
        for f, d, m in steps:
            if name == "u8":
                losses.append(eng.step(f.cuda(), y, private_inputs=True, mix=m, smoothing=0.1, aug=d).clone())
            else:
                losses.append(eng.step(_augment_ref(f, d.params, S).contiguous(), y, private_inputs=True, mix=m, smoothing=0.1).clone())
        torch.cuda.synchronize()
        out[name] = (torch.cat(losses).cpu(), eng.logits.clone().cpu(), vit.core().arena.params.clone().cpu(), len(eng.graphs._graphs))
    (l_u, lg_u, p_u, ng), (l_f, lg_f, p_f, _) = out["u8"], out["f32"]
    print(f"spatial_aug step vs torch-augmented fp32: loss {((l_u - l_f).abs() / l_f.abs()).max().item():.2e}, "
          f"logits {rel_l2(lg_u, lg_f):.2e}, weights {rel_l2(p_u, p_f):.2e}")
    assert ng == 1
    assert ((l_u - l_f).abs() <= 1e-3 * l_f.abs()).all(), (l_u, l_f)
    assert rel_l2(lg_u, lg_f) < 1e-3 and rel_l2(p_u, p_f) < 1e-3


@pytest.mark.parametrize("update_freq", [1, 2])
def test_train_one_epoch_with_spatial_aug_equals_the_loop_on_torch_augmented_clips(update_freq):
    from unite_b200.augment import SpatialAugment
    from unite_b200.engine_for_finetuning import train_one_epoch
    scfg, _ = _tiny_vit()
    S, T, B, C = scfg.img_size, scfg.num_frames, 4, scfg.num_classes
    aug = SpatialAugment(crop_size=S, reprob=0.5, remode="const")
    frames = [_frames((B, T, 72, 90, 3), 500 + i) for i in range(4)]
    labels = [torch.randint(0, C, (B,), generator=torch.Generator().manual_seed(60 + i)) for i in range(4)]
    random.seed(1)
    np.random.seed(1)
    clips = [_augment_ref(f, aug.draw(f.shape).params, S).cpu() for f in frames]
    out = {}
    for name in ("u8", "f32"):
        _, vit = _tiny_vit(drop_path_rate=0.1)
        batches = [((f if name == "u8" else c), yy, torch.zeros(B), {}) for f, c, yy in zip(frames, clips, labels)]
        random.seed(1)
        np.random.seed(1)
        st = train_one_epoch(vit, None, batches, _opt(vit), "cuda", 0, None, update_freq=update_freq, lr_schedule_values=[1e-3] * 8,
                             spatial_aug=aug if name == "u8" else None)
        torch.cuda.synchronize()
        out[name] = (st, vit.core().arena.params.clone().cpu())
    (a, p_u), (b, p_f) = out["u8"], out["f32"]
    print(f"train_one_epoch spatial_aug (update_freq {update_freq}): loss {a['loss']:.6f} / {b['loss']:.6f}, weights {rel_l2(p_u, p_f):.1e}")
    assert abs(a["loss"] - b["loss"]) < 1e-3 * abs(b["loss"]) and a["class_acc"] == b["class_acc"]
    assert rel_l2(p_u, p_f) < 1e-3
    with pytest.raises(ValueError, match="uint8 frames"):
        train_one_epoch(vit, None, [(clips[0], labels[0])], _opt(vit), "cuda", 0, None, spatial_aug=aug, update_freq=update_freq)
