"""Decoded uint8 frames [B,T,H,W,3] fed to stages 2 and 3, normalised on the device inside the im2col.  The reference is always
oracle.unite_oracle.normalize_frames_u8 of the same frames (the reference loader's ToTensor + tensor_normalize): ub_patchify_mix_u8
bit for bit against ub_patchify of the torch-mixed normalised clip, and every step, loop and evaluation fed uint8 frames against the
same call fed that normalised fp32 clip."""
from functools import partial

import numpy as np
import pytest
import torch

from tests import mixup_ref as R
from tests.util import build_student, build_teacher, load_golden, oracle_cfgs, rel_l2, seeded_states

pytestmark = pytest.mark.gpu
LOSS_REL, GRAD_REL = 2e-6, 1e-5          # test_stage1_step_from_uint8_frames_equals_step_from_normalised_clip: fp32 atomic order only


def _norm(frames):
    from oracle.unite_oracle import normalize_frames_u8
    return normalize_frames_u8(frames)


def _frames(shape, seed):
    return torch.randint(0, 256, shape, generator=torch.Generator().manual_seed(seed), dtype=torch.uint8)


def _buffer(d, smoothing=0.1, C=12, mix_clips=True):
    from unite_b200.mixup import MixBuffer
    buf = MixBuffer(torch.device("cuda"), mix_clips=mix_clips)
    buf.upload(d.packed(smoothing, C))
    return buf


# ---- 1. ub_patchify_mix_u8 bit for bit --------------------------------------------------------------------------------------------
CASES = [
    # B, T, H, W, tubelet, kind, parameter (lam for mixup, timm's (yl, yh, xl, xh) for cutmix)
    (2, 4, 32, 32, 2, "mix", 0.37),
    (2, 4, 32, 32, 1, "mix", 0.81),
    (4, 8, 48, 32, 2, "mix", 0.05),
    (2, 4, 32, 32, 1, "mix", 1.0),                      # lam = 1 mixed: the clip itself
    (2, 4, 32, 32, 2, "copy", None),                    # the draw left the batch unmixed
    (4, 8, 48, 32, 2, "cut", (8, 20, 5, 30)),          # T slice [8, 8): empty
    (4, 8, 48, 32, 1, "cut", (0, 3, 40, 48)),          # on the borders: first frames, last rows
    (4, 8, 48, 32, 2, "cut", (5, 8, 0, 7)),            # last frames, first rows
    (2, 4, 32, 32, 2, "cut", (0, 32, 0, 32)),          # the whole clip
    (32, 8, 224, 224, 2, "mix", 0.4217),               # the bench shape
    (32, 8, 224, 224, 2, "cut", (2, 7, 30, 190)),
    (4, 8, 224, 160, 2, "mix", 0.63),                  # non-square
    (4, 8, 224, 160, 1, "cut", (1, 6, 20, 150)),
    (4, 8, 48, 32, 2, "timm", 0),                      # tests/mixup_ref.Mixup against unite_b200.mixup.draw at a numpy seed:
    (4, 8, 48, 32, 1, "timm", 10),                     # mixup, and cutmix boxes T [0,8) x H [1,17), T [2,8) x H [6,32)
    (4, 8, 48, 32, 2, "timm", 29),
]


@pytest.mark.parametrize("B,T,H,W,tub,kind,par", CASES)
def test_patchify_mix_u8_is_bit_exact_against_normalise_then_timm_mix_then_patchify(B, T, H, W, tub, kind, par):
    from unite_b200 import ops
    from unite_b200 import mixup as M
    from unite_b200.mixup import NO_MIX, MixDraw, clip_box
    frames = _frames((B, T, H, W, 3), B * 1000 + T + H + W)
    frames[0, 0, 0, :4] = torch.tensor([[0, 0, 0], [255, 255, 255], [1, 128, 254], [127, 0, 255]], dtype=torch.uint8)
    x = frames.cuda()
    ref = _norm(frames).cuda()
    if kind == "copy":
        d = NO_MIX
    elif kind == "mix":
        lam = par
        x_flipped = ref.flip(0).mul_(1. - lam)                                        # timm Mixup._mix_batch, literally
        ref.mul_(lam).add_(x_flipped)
        d = MixDraw(True, lam, False, ((0, 0), (0, 0), (0, 0)), lam)
    elif kind == "timm":
        cfg = dict(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1, num_classes=12)
        np.random.seed(par)
        R.Mixup(**cfg)(ref, torch.zeros(B, dtype=torch.long, device="cuda"))
        np.random.seed(par)
        d = M.draw(M.Mixup(**cfg), ops.clip_shape(x))                            # the box from the clip's shape, not the frames'
        assert d.apply
    else:
        yl, yh, xl, xh = par
        ref[:, :, yl:yh, xl:xh] = ref.flip(0)[:, :, yl:yh, xl:xh]
        d = MixDraw(True, 0.5, True, clip_box(ref.shape, yl, yh, xl, xh), 0.5)
    n_tok = B * (T // tub) * (H // 16) * (W // 16)
    want = torch.empty(n_tok, 3 * tub * 256, device="cuda", dtype=torch.bfloat16)
    got = torch.full_like(want, float("nan"))
    ops.patchify(ref, want, tub)
    ops.patchify_mix_u8(x, got, _buffer(d).clip, tub)
    torch.cuda.synchronize()
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))
    assert torch.equal(x.cpu(), frames), "the input frames must not be written"
    if kind == "copy" or (kind == "mix" and par == 1.0):
        plain = ops.patchify_u8(x, torch.empty_like(want), tub)
        assert torch.equal(got.view(torch.int16), plain.view(torch.int16))


def test_patchify_mix_u8_refuses_an_odd_batch_and_a_short_draw():
    from unite_b200 import ops
    from unite_b200._cabi import UBError
    from unite_b200.mixup import NO_MIX
    x = torch.zeros(3, 2, 16, 16, 3, device="cuda", dtype=torch.uint8)
    out = torch.empty(6, 3 * 256, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(UBError, match="even"):
        ops.patchify_mix_u8(x, out, _buffer(NO_MIX).clip, 1)
    with pytest.raises(UBError, match="10 floats"):
        ops.patchify_mix_u8(x[:2], out[:4], torch.zeros(4, device="cuda"), 1)


# ---- 2. stage 2 ---------------------------------------------------------------------------------------------------------------------
def _build_vit(scfg, drop_path_rate=0.0):
    import torch.nn as nn
    from unite_b200.modeling_finetune import VisionTransformer
    return VisionTransformer(img_size=scfg.img_size, patch_size=scfg.patch_size, embed_dim=scfg.embed_dim, depth=scfg.depth,
                             num_heads=scfg.num_heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                             num_classes=scfg.num_classes, all_frames=scfg.num_frames, tubelet_size=scfg.tubelet_size,
                             init_scale=0.001, use_mean_pooling=True, drop_path_rate=drop_path_rate)


def _tiny_vit(drop_path_rate=0.0, tubelet=None):
    from dataclasses import replace
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    _, _, vsd = seeded_states(fix)
    vsd = dict(vsd)
    g = torch.Generator().manual_seed(17)
    vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=g) * 0.05          # O(1) logits
    if tubelet is not None and tubelet != scfg.tubelet_size:
        from oracle.weights import seeded_state
        scfg = replace(scfg, tubelet_size=tubelet)
        vit = _build_vit(scfg, drop_path_rate)
        vsd = seeded_state({k: tuple(v.shape) for k, v in vit.state_dict().items()}, 9)
        vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=g) * 0.05
    else:
        vit = _build_vit(scfg, drop_path_rate)
    vit.load_state_dict(vsd, strict=True)
    return scfg, vit.cuda()


def _frames_like(scfg, B, seed):
    return _frames((B, scfg.num_frames, scfg.img_size, scfg.img_size, 3), seed)


def _draw_for(kind, shape, C):
    from unite_b200 import mixup as M
    if kind == "ce":
        return None
    if kind == "smoothing":
        return _buffer(M.NO_MIX, 0.1, C, mix_clips=False)
    cfg = dict(mixup_alpha=0.8, cutmix_alpha=0.) if kind == "mixup" else dict(mixup_alpha=0., cutmix_alpha=1.0)
    np.random.seed(4)
    d = M.draw(M.Mixup(label_smoothing=0.1, num_classes=C, **cfg), shape)
    assert d.apply and d.use_cutmix == (kind == "cutmix")
    return _buffer(d, 0.1, C)


@pytest.mark.parametrize("tubelet", [1, 2])
@pytest.mark.parametrize("kind", ["ce", "smoothing", "mixup", "cutmix"])
def test_stage2_step_from_uint8_frames_equals_step_from_normalised_clip(kind, tubelet):
    from unite_b200 import ops
    from unite_b200.engine_for_finetuning import finetune_step
    scfg, vit = _tiny_vit(tubelet=tubelet)
    vit.eval()                                                                     # no DropPath draw in either pass
    C = scfg.num_classes
    frames = _frames_like(scfg, 8, 31 + tubelet)
    labels = torch.randint(0, C, (8,), generator=torch.Generator().manual_seed(5)).cuda()
    buf = _draw_for(kind, ops.clip_shape(frames), C)
    arena = vit.core().arena
    out = {}
    for name, x in (("u8", frames.cuda()), ("f32", _norm(frames).cuda())):
        arena.grads.zero_()
        loss = torch.zeros(1, device="cuda")
        logits = finetune_step(vit, x, labels, loss, mix=buf)
        torch.cuda.synchronize()
        out[name] = (loss.item(), logits.clone(), arena.grads.clone())
    (l_u, lg_u, g_u), (l_f, lg_f, g_f) = out["u8"], out["f32"]
    print(f"stage-2 {kind} tub {tubelet}: loss {l_u:.7f} / {l_f:.7f}, grads rel-L2 {rel_l2(g_u, g_f):.1e}")
    assert abs(l_u - l_f) <= LOSS_REL * abs(l_f)
    assert rel_l2(g_u, g_f) < GRAD_REL
    assert torch.equal(lg_u.argmax(-1), lg_f.argmax(-1))


def test_stage2_uint8_graph_replay_matches_eager_uint8_steps():
    """As test_stage2_mixup_graph_replay_matches_eager_steps, with uint8 frames: six Stage2Engine steps replayed from one graph
    (unmixed, mixup and cutmix draws) against six eager uint8 steps from the same numpy seed."""
    from unite_b200 import mixup as M
    from unite_b200 import ops
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    scfg, _ = _tiny_vit()
    x = _frames_like(scfg, 6, 78).cuda()
    y = torch.randint(0, scfg.num_classes, (6,), generator=torch.Generator().manual_seed(78)).cuda()

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 2e-4, 0.05, (0.9, 0.999), 1e-8
    runs = []
    for use_graph in (True, False, False):
        _, vit = _tiny_vit(drop_path_rate=0.2)
        vit.train()
        L = vit.get_num_layers()
        asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])
        opt = create_optimizer(Args, vit, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
        eng = Stage2Engine(vit, opt, use_graph=use_graph)
        np.random.seed(1)
        mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, prob=0.6, switch_prob=0.5, label_smoothing=0.1, num_classes=scfg.num_classes)
        losses, kinds = [], []
        for s in range(6):
            d = M.draw(mixer, ops.clip_shape(x))
            kinds.append("cut" if d.use_cutmix else ("mix" if d.apply else "none"))
            losses.append(eng.step(x, y, mix=d, smoothing=0.1).clone())
        for s in range(3):
            losses.append(eng.step(x, y).clone())                                 # plain CE: a second graph
        torch.cuda.synchronize()
        runs.append((torch.cat(losses).cpu(), eng.stats.cpu(), vit.core().arena.params.clone().cpu(), eng, kinds))
    (l_g, st_g, p_g, eng_g, kinds), (l_e, st_e, p_e, _, _), (l_e2, _, p_e2, _, _) = runs
    assert set(kinds[2:]) == {"none", "mix", "cut"}, kinds
    assert len(eng_g.graphs._graphs) == 2
    noise_l, noise_p = ((l_e - l_e2).abs() / l_e.abs()).max().item(), rel_l2(p_e, p_e2)
    d_l, d_p = ((l_g - l_e).abs() / l_e.abs()).max().item(), rel_l2(p_g, p_e)
    print(f"stage-2 uint8 graph vs eager: loss {d_l:.2e} (eager vs eager {noise_l:.2e}), weights {d_p:.2e} (eager vs eager {noise_p:.2e})")
    assert d_l <= max(2e-5, 4 * noise_l), (l_g, l_e)
    assert torch.allclose(st_g, st_e, rtol=1e-4), (st_g, st_e)
    assert d_p <= max(1e-5, 4 * noise_p)


def _fresh_opt(vit):
    from unite_b200.optim_factory import create_optimizer

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    return create_optimizer(Args, vit)


@pytest.mark.parametrize("update_freq", [1, 2])
@pytest.mark.parametrize("with_ema", [False, True])
def test_stage2_train_one_epoch_on_uint8_batches_equals_the_normalised_clip(update_freq, with_ema):
    """Both loops (graph-replayed update_freq 1, eager update_freq 2), with mixup / cutmix / label smoothing drawn from one numpy
    seed, and the model EMA: uint8 batches train as their normalised fp32 clips do.  The cutmix box comes from the clip's shape,
    not the frames' ([B,T,H,W,3]), or the two runs would cut different boxes."""
    from unite_b200 import mixup as M
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import train_one_epoch
    scfg, _ = _tiny_vit()
    C = scfg.num_classes
    frames = [_frames_like(scfg, 4, 50 + i) for i in range(4)]
    labels = [torch.randint(0, C, (4,), generator=torch.Generator().manual_seed(60 + i)) for i in range(4)]
    out = {}
    for name in ("u8", "f32"):
        _, vit = _tiny_vit(drop_path_rate=0.1)
        opt = _fresh_opt(vit)
        ema = ModelEma(vit, decay=0.9) if with_ema else None
        batches = [((f if name == "u8" else _norm(f)), y, torch.zeros(4), {}) for f, y in zip(frames, labels)]
        np.random.seed(3)
        mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, switch_prob=0.5, label_smoothing=0.1, num_classes=C)
        s0 = train_one_epoch(vit, M.SoftTargetCrossEntropy(), batches * 2, opt, "cuda", 0, None, model_ema=ema, mixup_fn=mixer,
                             update_freq=update_freq, lr_schedule_values=[1e-3] * 40)
        s1 = train_one_epoch(vit, M.LabelSmoothingCrossEntropy(0.1), batches, opt, "cuda", 1, None, model_ema=ema,
                             update_freq=update_freq, start_steps=8, lr_schedule_values=[1e-3] * 40)
        torch.cuda.synchronize()
        out[name] = (s0, s1, vit.core().arena.params.clone().cpu(), ema.ema.core().arena.params.clone().cpu() if with_ema else None)
    (a0, a1, p_u, e_u), (b0, b1, p_f, e_f) = out["u8"], out["f32"]
    print(f"uint8 vs fp32 train_one_epoch (update_freq {update_freq}, ema {with_ema}): loss {a0['loss']:.6f} / {b0['loss']:.6f}, "
          f"{a1['loss']:.6f} / {b1['loss']:.6f}; weights rel-L2 {rel_l2(p_u, p_f):.1e}")
    for a, b in ((a0, b0), (a1, b1)):
        assert abs(a["loss"] - b["loss"]) < 1e-4 * abs(b["loss"])
        assert abs(a["grad_norm"] - b["grad_norm"]) < 1e-3 * abs(b["grad_norm"])
    assert "class_acc" not in a0 and a1["class_acc"] == b1["class_acc"]
    assert rel_l2(p_u, p_f) < 1e-3                  # AdamW turns noise on a near-zero gradient into a +-lr step
    if with_ema:
        assert rel_l2(e_u, e_f) < 1e-3


def test_validation_and_final_test_on_uint8_batches(tmp_path):
    from unite_b200.engine_for_finetuning import final_test, validation_one_epoch
    scfg, vit = _tiny_vit()
    vit.eval()
    C = scfg.num_classes
    frames = [_frames_like(scfg, 4, 70 + i) for i in range(3)]
    labels = [torch.randint(0, C, (4,), generator=torch.Generator().manual_seed(80 + i)) for i in range(3)]
    with torch.no_grad():
        lg_u = torch.cat([vit(f.cuda()) for f in frames])
        lg_f = torch.cat([vit(_norm(f).cuda()) for f in frames])
    assert rel_l2(lg_u, lg_f) < GRAD_REL and torch.equal(lg_u.argmax(-1), lg_f.argmax(-1))
    (s_u, ece_u) = validation_one_epoch(list(zip(frames, labels)), vit, "cuda")
    (s_f, ece_f) = validation_one_epoch(list(zip([_norm(f) for f in frames], labels)), vit, "cuda")
    assert s_u["acc1"] == s_f["acc1"] and s_u["acc5"] == s_f["acc5"]
    assert abs(s_u["loss"] - s_f["loss"]) <= 1e-5 * abs(s_f["loss"]) and abs(ece_u - ece_f) < 1e-5
    files = {}
    for name, fr in (("u8", frames), ("f32", [_norm(f) for f in frames])):
        batches = [(f, y, [f"vid{4 * i + j}" for j in range(4)], torch.zeros(4), torch.zeros(4)) for i, (f, y) in enumerate(zip(fr, labels))]
        files[name] = str(tmp_path / f"{name}.txt")
        st, _ = final_test(batches, vit, "cuda", files[name])
        assert st["acc1"] == s_f["acc1"] and st["acc5"] == s_f["acc5"]
    rows = {}
    for name, path in files.items():
        with open(path) as f:
            lines = f.readlines()
        rows[name] = lines
    assert rows["u8"][0] == rows["f32"][0] and len(rows["u8"]) == len(rows["f32"]) == 13

    def scores(line):
        return torch.tensor([float(t) for t in line.rsplit("[", 1)[1].rsplit("]", 1)[0].split(",")])
    for a, b in zip(rows["u8"][1:], rows["f32"][1:]):
        assert a.split(" ")[0] == b.split(" ")[0] and a.rsplit("]", 1)[1] == b.rsplit("]", 1)[1]
        assert rel_l2(scores(a), scores(b)) < GRAD_REL


# ---- 3. stage 3 ---------------------------------------------------------------------------------------------------------------------
def _stage3_models(kernel_size=None, drop_path_rate=0.0):
    """The tiny student (tubelet 1) and teacher.  kernel_size=2: a teacher whose temporal kernel is not the student's tubelet, so
    the student needs its own im2col."""
    from oracle import unite_oracle as O
    from oracle.weights import seeded_state
    fix = load_golden("tiny_stage12.pt")
    scfg, tcfg = oracle_cfgs(fix)
    ssd, tsd, _ = seeded_states(fix)
    if kernel_size is not None and kernel_size != tcfg.kernel_size:
        tcfg = O.TeacherCfg(**{**fix["cfg"]["teacher"], "kernel_size": kernel_size})
        tsd = seeded_state({k: tuple(v.shape) for k, v in build_teacher(tcfg).state_dict().items()}, 6)
    student, teacher = build_student(scfg, drop_path_rate=drop_path_rate), build_teacher(tcfg)
    student.load_state_dict(ssd, strict=True)
    teacher.load_state_dict(tsd, strict=True)
    return scfg, tcfg, student.cuda(), teacher.cuda().eval()


def _stage3_head(scfg, tcfg, seed=31):
    g = torch.Generator().manual_seed(seed)
    C = 12
    return torch.randn(C, scfg.embed_dim, generator=g) * 0.5, torch.randn(C, generator=g) * 0.1, torch.randn(C, tcfg.output_dim, generator=g)


def _stage3_views(scfg, Bs, Bt, seed):
    shape = lambda B: (B, scfg.num_frames, scfg.img_size, scfg.img_size, 3)
    vs, vt = _frames(shape(Bs), seed), _frames(shape(Bt), seed + 1)
    va = (vt.short() + _frames(shape(Bt), seed + 2).short() // 16 - 8).clamp(0, 255).to(torch.uint8)
    ys = torch.randint(0, 12, (Bs,), generator=torch.Generator().manual_seed(seed))
    return vs, ys, vt, va


@pytest.mark.parametrize("kernel_size", [1, 2], ids=["shared_im2col", "own_im2col"])
@pytest.mark.parametrize("dual", [False, True], ids=["single_view", "dual_view"])
def test_stage3_step_from_uint8_frames_equals_step_from_normalised_clips(dual, kernel_size):
    from unite_b200.engine_stage3 import Stage3Engine
    scfg, tcfg, student, teacher = _stage3_models(kernel_size)
    cls_w, cls_b, text = _stage3_head(scfg, tcfg)
    eng = Stage3Engine(student.eval(), teacher, cls_w, cls_b, text, mask_ratio=0.75, k=2)
    assert (eng.core.tubelet == teacher.kernel_size) == (kernel_size == 1)
    vs, ys, vt, va = _stage3_views(scfg, 4, 8, 90)
    views = {"u8": (vs, vt, va if dual else None)}
    views["f32"] = tuple(None if v is None else _norm(v) for v in views["u8"])
    out = {}
    for name, (s, t, a) in views.items():
        eng.optimizer.zero_grad()
        loss = eng.forward_backward(s.cuda(), ys.cuda(), t.cuda(), None if a is None else a.cuda())
        torch.cuda.synchronize()
        out[name] = (torch.cat([loss, eng.loss_s, eng.loss_t]).cpu(), {k: v.clone() for k, v in eng.last.items()},
                     eng.core.arena.grads.clone())
    (l_u, L_u, g_u), (l_f, L_f, g_f) = out["u8"], out["f32"]
    print(f"stage-3 dual={dual} kernel={kernel_size}: losses {l_u.tolist()} / {l_f.tolist()}, grads rel-L2 {rel_l2(g_u, g_f):.1e}, "
          f"selected {int(L_f['sel_mask'].sum())}/8")
    for key in ("attn", "masks", "sel_mask", "pseudo"):
        assert torch.equal(L_u[key], L_f[key]), key
    for key in ("logits_s", "logits_full_t", "logits_masked", "clip_probs", "msp"):
        assert rel_l2(L_u[key], L_f[key]) < GRAD_REL, key
    assert ((l_u - l_f).abs() <= LOSS_REL * l_f.abs()).all(), (l_u, l_f)
    assert rel_l2(g_u, g_f) < GRAD_REL


def test_stage3_uint8_graph_replay_matches_eager_steps():
    """As test_stage3_graph_replay_matches_eager_steps, with dual-view uint8 frames."""
    from unite_b200.engine_stage3 import Stage3Engine
    batches = []
    runs = []
    for use_graph in (True, False):
        scfg, tcfg, student, teacher = _stage3_models(drop_path_rate=0.2)
        cls_w, cls_b, text = _stage3_head(scfg, tcfg)
        if not batches:
            for i in range(2):
                vs, ys, vt, va = _stage3_views(scfg, 4, 4, 200 + 10 * i)
                batches.append((vs.cuda(), ys.cuda(), vt.cuda(), va.cuda()))
        eng = Stage3Engine(student.train(), teacher, cls_w, cls_b, text, mask_ratio=0.75, k=2, lr=2e-5, use_graph=use_graph)
        p0 = eng.core.arena.params.clone().cpu()
        losses = []
        for s in range(6):
            eng.step(*batches[s % 2])
            losses.append(torch.cat([eng.loss, eng.loss_s, eng.loss_t]).clone())
        torch.cuda.synchronize()
        runs.append((torch.stack(losses).cpu(), eng.core.arena.params.clone().cpu(), eng))
    (l_g, p_g, eng_g), (l_e, p_e, _) = runs
    assert len(eng_g.graphs._graphs) == 2
    travelled, d_p = rel_l2(p_g, p0), rel_l2(p_g, p_e)
    print(f"stage-3 uint8 graph vs eager: losses {(l_g - l_e).abs().max().item():.2e}, weights {d_p:.2e} of {travelled:.2e} travelled")
    assert torch.allclose(l_g, l_e, rtol=3e-5, atol=1e-6), (l_g, l_e)
    assert travelled > 3e-4 and d_p < 0.02 * travelled
    assert len(set(round(v, 4) for v in l_g[:, 0].tolist())) >= 5


def test_stage3_train_one_epoch_on_uint8_target_batches():
    """The drop-in loop over (vid, vid_aug, label, name) uint8 target batches and uint8 source batches, against the same loop over
    the normalised clips."""
    from unite_b200.engine_stage3 import train_one_epoch
    out = {}
    for name in ("u8", "f32"):
        scfg, tcfg, student, teacher = _stage3_models()
        cls_w, cls_b, text = _stage3_head(scfg, tcfg)

        class Args:
            masking_type, selection_strategy, train_masked, conf_weighted_loss = "clip_attention", "clip_matchORconf", True, True
            class_loss_src_ratio, class_loss_src_ratio_pl, class_loss_tgt_ratio, clip_threshold = 1.0, 1.0, 1.0, 0.5
            return_aug_for_val, full_oracle, log_freq = True, False, 10
            text_features = text
        src_classifier = torch.nn.Linear(scfg.embed_dim, 12)
        with torch.no_grad():
            src_classifier.weight.copy_(cls_w); src_classifier.bias.copy_(cls_b)
        f = (lambda v: v) if name == "u8" else _norm
        src, tgt = [], []
        for i in range(2):
            vs, ys, vt, va = _stage3_views(scfg, 4, 4, 300 + 10 * i)
            src.append((f(vs), ys, torch.arange(4), {}))
            tgt.append((f(vt), f(va), torch.zeros(4, dtype=torch.long), ["a", "b", "c", "d"]))
        stats = train_one_epoch(student, src * 2, tgt, None, "cuda", 0, None, src_classifier=src_classifier.cuda(), teacher_model=teacher,
                                mask_type="attention", mask_ratio=0.75, args=Args, lr_schedule_values=[1e-5] * 10)
        out[name] = (stats, student.core().arena.params.clone().cpu())
    (s_u, p_u), (s_f, p_f) = out["u8"], out["f32"]
    print(f"stage-3 train_one_epoch uint8 vs fp32: {s_u['loss']:.6f} / {s_f['loss']:.6f}, weights rel-L2 {rel_l2(p_u, p_f):.1e}")
    for k in ("loss", "loss_class", "loss_class_t", "grad_norm"):
        assert np.isfinite(s_u[k]) and abs(s_u[k] - s_f[k]) <= 1e-4 * abs(s_f[k]) + 1e-7, k
    assert rel_l2(p_u, p_f) < 1e-4
