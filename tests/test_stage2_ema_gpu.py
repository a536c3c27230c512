"""Stage-2 model EMA on the GPU against tests/ema_ref.py (timm 0.4.12's ModelEma restated, i.e. torch's own fp32 update): the fused
kernel bit for bit, the EMA of the eager and the graph-replayed step over recorded weights, train_one_epoch with the package's and
the reference's ModelEma, evaluation of the EMA model, the checkpoint round trip, full-size ViT-B/16, and several GPUs."""
import os
import subprocess
import sys
from functools import partial

import numpy as np
import pytest
import torch

from tests import ema_ref as R
from tests.util import load_golden, oracle_cfgs, rel_l2, seeded_states

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DECAY = 0.99                   # far enough from 1 that every update moves the EMA visibly


def _build_vit(scfg, drop_path_rate=0.0):
    import torch.nn as nn
    from unite_b200.modeling_finetune import VisionTransformer
    return VisionTransformer(img_size=scfg.img_size, patch_size=scfg.patch_size, embed_dim=scfg.embed_dim, depth=scfg.depth,
                             num_heads=scfg.num_heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                             num_classes=scfg.num_classes, all_frames=scfg.num_frames, tubelet_size=scfg.tubelet_size,
                             init_scale=0.001, use_mean_pooling=True, drop_path_rate=drop_path_rate)


def _tiny_vit(drop_path_rate=0.0):
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    _, _, vsd = seeded_states(fix)
    vit = _build_vit(scfg, drop_path_rate)
    vit.load_state_dict(vsd, strict=True)
    return scfg, vit.cuda()


def _bits(t):
    return t.detach().contiguous().view(torch.int32) if t.dtype == torch.float32 else t.detach().contiguous().view(torch.int16)


def _same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def _bf16(t):
    """ub_cast_bf16 of an fp32 tensor (the shadow a model's arena gets from its fp32 weights)."""
    from unite_b200 import ops
    out = torch.empty(t.numel(), device=t.device, dtype=torch.bfloat16)
    ops.cast_bf16(t.contiguous().view(-1), out)
    return out


def _replay_reference(e0, recorded, decay):
    """The EMA timm's update produces over a sequence of recorded weight arenas, after each update."""
    e, out = e0.clone(), []
    for p in recorded:
        R.update_tensor(e, p, decay)
        out.append(e.clone())
    return out


def _vitb16_stage2(C=12):
    from unite_b200 import modeling_finetune  # noqa: F401  (registers the factories)
    from unite_b200.registry import create_model
    torch.manual_seed(0)
    return create_model("vit_base_patch16_224", pretrained=False, num_classes=C, all_frames=8, tubelet_size=1, drop_rate=0.0,
                        drop_path_rate=0.1, attn_drop_rate=0.0, drop_block_rate=None, use_mean_pooling=True, init_scale=0.001,
                        fc_drop_rate=0.0, use_checkpoint=False, checkpoint_num=0)


@pytest.fixture(scope="module")
def vitb_numel():
    return _vitb16_stage2().cuda().core().arena.numel


# ---- 1. ub_ema_update bit for bit against torch's fp32 update ---------------------------------------------------------------------
GRID = 148 * 8 * 256 * 4       # elements one pass of the grid-stride loop covers on a 148-SM B200
LENGTHS = [4, 1028, 2 * GRID + 12, "vitb"]
GUARD = 64


@pytest.mark.parametrize("decay", [0.9999, 0.99996, 0.5, 0.0, 1.0])
@pytest.mark.parametrize("n", LENGTHS)
def test_ema_update_kernel_is_bit_exact(n, decay, vitb_numel):
    from unite_b200 import ops
    n = vitb_numel if n == "vitb" else n
    g = torch.Generator(device="cuda").manual_seed(n % 1000 + int(decay * 1e5))
    scale = lambda: torch.exp(torch.randn(n + GUARD, device="cuda", generator=g) * 3)      # magnitudes over ~ e^+-9
    ema = torch.randn(n + GUARD, device="cuda", generator=g) * scale()
    p = torch.randn(n + GUARD, device="cuda", generator=g) * scale()
    ema[n:] = float("nan")
    w16 = torch.full((n + GUARD,), float("nan"), device="cuda", dtype=torch.bfloat16)
    p_keep = p.clone()
    want = R.update_tensor(ema[:n].clone(), p[:n], decay)
    ops.ema_update(ema[:n], w16[:n], p[:n], decay)
    torch.cuda.synchronize()
    assert _same_bits(ema[:n], want)
    assert _same_bits(w16[:n], _bf16(want))
    assert _same_bits(p, p_keep), "p must not be written"
    assert ema[n:].isnan().all() and w16[n:].isnan().all(), "nothing past n may be written"


def test_ema_update_refuses_bad_arguments():
    from unite_b200 import ops
    from unite_b200._cabi import UBError, lib
    a = torch.zeros(8, device="cuda")
    w = torch.zeros(8, device="cuda", dtype=torch.bfloat16)
    s = torch.cuda.current_stream().cuda_stream
    for n in (6, 0, -4):
        assert lib.ub_ema_update(a.data_ptr(), w.data_ptr(), a.data_ptr(), n, 0.9, 0.1, s) != 0
        assert b"multiple of 4" in lib.ub_last_error()
    for ptrs in ((None, w.data_ptr(), a.data_ptr()), (a.data_ptr(), None, a.data_ptr()), (a.data_ptr(), w.data_ptr(), None)):
        assert lib.ub_ema_update(*ptrs, 8, 0.9, 0.1, s) != 0
        assert b"null pointer" in lib.ub_last_error()
    with pytest.raises(UBError, match="multiple of 4"):
        ops.ema_update(a[:6], w[:6], a[2:], 0.9)
    with pytest.raises(UBError, match="differ"):
        ops.ema_update(a, w[:4], a, 0.9)


# ---- 2./3. Stage2Engine: the EMA over recorded weights, eager and graph-replayed; training unchanged ------------------------------------
def _engine_runs():
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    g = torch.Generator().manual_seed(77)
    shape = (3, scfg.num_frames, scfg.img_size, scfg.img_size)
    batches = [(torch.randn(6, *shape, generator=g).cuda(), torch.randint(0, scfg.num_classes, (6,), generator=g).cuda()) for _ in range(2)]

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 2e-4, 0.05, (0.9, 0.999), 1e-8
    runs = {}
    for name, use_graph, with_ema in (("eager", False, False), ("eager2", False, False), ("eager_ema", False, True),
                                      ("graph_ema", True, True)):
        _, vit = _tiny_vit(drop_path_rate=0.2)
        vit.train()
        L = vit.get_num_layers()
        asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])
        opt = create_optimizer(Args, vit, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
        ema = ModelEma(vit, decay=DECAY) if with_ema else None                   # taken after the model's arena exists
        w0 = vit.core().arena.params.clone()
        eng = Stage2Engine(vit, opt, use_graph=use_graph, model_ema=ema)
        eng.max_norm = 1.0
        e0 = ema.ema.core().arena.params.clone() if with_ema else None
        losses, weights, emas, shadows = [], [], [], []
        for s in range(7):
            for grp in opt.param_groups:
                grp["lr"] = 2e-4 * (1 + s) / 7 * grp["lr_scale"]
            losses.append(eng.step(*batches[s % 2]).clone())
            weights.append(vit.core().arena.params.clone())
            if with_ema:
                emas.append(ema.ema.core().arena.params.clone())
                shadows.append(ema.ema.core().arena.w16.clone())
        torch.cuda.synchronize()
        runs[name] = dict(loss=torch.cat(losses).cpu(), stats=eng.stats.cpu(), weights=weights, emas=emas, shadows=shadows, e0=e0,
                          w0=w0, eng=eng, vit=vit, ema=ema)
    return runs


@pytest.fixture(scope="module")
def engine_runs():
    return _engine_runs()


@pytest.mark.parametrize("mode", ["eager_ema", "graph_ema"])
def test_stage2_engine_ema_equals_the_reference_update_over_recorded_weights(engine_runs, mode):
    r = engine_runs[mode]
    assert _same_bits(r["e0"], r["w0"]), "the EMA starts from the model's weights"
    want = _replay_reference(r["e0"], r["weights"], DECAY)
    for s, (got, exp, w16) in enumerate(zip(r["emas"], want, r["shadows"])):
        assert _same_bits(got, exp), f"update {s}: EMA differs from timm's update"
        assert _same_bits(w16, _bf16(exp)), f"update {s}: the EMA's bf16 shadow is stale"
    assert rel_l2(r["emas"][-1], r["weights"][-1]) > 0 and not torch.equal(r["emas"][-1], r["weights"][-1])
    if mode == "graph_ema":
        eng = r["eng"]
        assert len(eng.graphs._graphs) == 2, "one graph per resident batch expected"
        assert int(eng.core.drop_path.step.item()) == 7, "capture must not consume a DropPath draw"
        assert all(("ema", DECAY) in k for k in eng.graphs._graphs)


def test_stage2_ema_does_not_perturb_training(engine_runs):
    base, noise = engine_runs["eager"], engine_runs["eager2"]
    noise_l = ((base["loss"] - noise["loss"]).abs() / base["loss"].abs()).max().item()
    noise_p = rel_l2(base["weights"][-1], noise["weights"][-1])
    for mode in ("eager_ema", "graph_ema"):
        r = engine_runs[mode]
        d_l = ((r["loss"] - base["loss"]).abs() / base["loss"].abs()).max().item()
        d_p = rel_l2(r["weights"][-1], base["weights"][-1])
        print(f"stage-2 {mode} vs eager without EMA: loss {d_l:.2e} (noise {noise_l:.2e}), weights {d_p:.2e} (noise {noise_p:.2e})")
        assert d_l <= max(2e-5, 4 * noise_l)
        assert torch.allclose(r["stats"], base["stats"], rtol=1e-4)
        assert d_p <= max(1e-5, 4 * noise_p)


# ---- 4. train_one_epoch with the package's and the reference's ModelEma -----------------------------------------------------------------
def _fresh_opt(vit):
    from unite_b200.optim_factory import create_optimizer

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    return create_optimizer(Args, vit)


@pytest.mark.parametrize("update_freq", [1, 2])
@pytest.mark.parametrize("kind", ["package", "timm"])
def test_train_one_epoch_updates_the_ema_once_per_optimizer_step(kind, update_freq):
    """One train_one_epoch call per optimizer update (update_freq loader batches), the weights recorded after each: the EMA must be
    timm's update over exactly that sequence (an update per micro-step, or none, would differ).  With update_freq 1 the later calls
    replay the held engine's CUDA graph."""
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import train_one_epoch
    scfg, vit = _tiny_vit(drop_path_rate=0.1)
    opt = _fresh_opt(vit)
    cls = ModelEma if kind == "package" else R.ModelEma
    ema = cls(vit, decay=DECAY)                                                     # deepcopy after the core exists
    e0 = vit.core().arena.params.clone()
    g = torch.Generator().manual_seed(9)
    batches = [(torch.randn(4, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g),
                torch.randint(0, scfg.num_classes, (4,), generator=g)) for _ in range(2 * update_freq)]
    recorded = []
    n_calls = 5
    for it in range(n_calls):
        st = train_one_epoch(vit, None, batches[(it % 2) * update_freq:(it % 2 + 1) * update_freq], opt, "cuda", it, None,
                             model_ema=ema, update_freq=update_freq, lr_schedule_values=[1e-3] * 10, start_steps=it)
        assert np.isfinite(st["loss"])
        recorded.append(vit.core().arena.params.clone())
    torch.cuda.synchronize()
    assert opt.step_count == n_calls
    if update_freq == 1:
        eng = vit.__dict__["_ub_stage2_engine"]
        assert eng.ema.source is ema and len(eng.graphs._graphs) == 1
    ema_arena = ema.ema.core().arena
    want = _replay_reference(e0, recorded, DECAY)[-1]
    assert _same_bits(ema_arena.params, want)
    assert _same_bits(ema_arena.w16, _bf16(want))
    # a model wrapped the reference's way: the EMA state_dict keys line up with the model's (timm's update would work too)
    assert list(ema.ema.state_dict()) == list(vit.state_dict())
    # the copy and the source share no storage
    src, cpy = vit.core().arena, ema_arena
    before = src.params.clone()
    with torch.no_grad():
        for p in ema.ema.parameters():
            p.add_(1.0)
    assert torch.equal(src.params, before), "writing the EMA's parameters changed the model"
    before = cpy.params.clone()
    with torch.no_grad():
        for p in vit.parameters():
            p.add_(1.0)
    assert torch.equal(cpy.params, before), "writing the model's parameters changed the EMA"


def test_a_new_ema_object_gets_a_new_engine():
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import train_one_epoch
    scfg, vit = _tiny_vit()
    opt = _fresh_opt(vit)
    g = torch.Generator().manual_seed(3)
    batch = [(torch.randn(2, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g), torch.randint(0, scfg.num_classes, (2,), generator=g))]
    engines = []
    for ema in (None, ModelEma(vit, DECAY), None):
        train_one_epoch(vit, None, batch, opt, "cuda", 0, None, model_ema=ema)
        engines.append(vit.__dict__["_ub_stage2_engine"])
    e_ema = engines[1].ema
    assert engines[0].ema is None and e_ema is not None and engines[2].ema is None
    assert len({id(e) for e in engines}) == 3
    ema2 = ModelEma(vit, 0.999)
    train_one_epoch(vit, None, batch, opt, "cuda", 1, None, model_ema=ema2)
    assert vit.__dict__["_ub_stage2_engine"].ema.source is ema2


# ---- 5. evaluation of the EMA model --------------------------------------------------------------------------------------------------
def test_ema_model_evaluates_like_a_fresh_model_with_its_weights(tmp_path):
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import final_test, train_one_epoch, validation_one_epoch
    scfg, vit = _tiny_vit(drop_path_rate=0.1)
    opt = _fresh_opt(vit)
    ema = ModelEma(vit, decay=0.9)
    g = torch.Generator().manual_seed(12)
    mk = lambda n: (torch.randn(n, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g),
                    torch.randint(0, scfg.num_classes, (n,), generator=g))
    train_one_epoch(vit, None, [mk(4) for _ in range(4)], opt, "cuda", 0, None, model_ema=ema, lr_schedule_values=[5e-3] * 4)
    assert all(not p.requires_grad for p in ema.ema.parameters())
    fresh = _build_vit(scfg)
    fresh.load_state_dict(ema.ema.state_dict())
    fresh = fresh.cuda()
    assert not torch.equal(fresh.head.weight, vit.head.weight)
    val = [mk(3) for _ in range(2)]
    test = [(v, y, [f"vid{i}_{j}" for j in range(3)], torch.zeros(3, dtype=torch.long), torch.arange(3)) for i, (v, y) in enumerate(val)]
    out = {}
    for name, m in (("ema", ema.ema), ("fresh", fresh)):
        stats, ece = validation_one_epoch(val, m, "cuda")
        path = os.path.join(tmp_path, f"{name}.txt")
        tstats, _ = final_test(test, m, "cuda", path)
        with torch.no_grad():
            logits = m(val[0][0].cuda())
        with open(path) as f:
            out[name] = (stats, ece, tstats, f.read(), logits)
    a, b = out["ema"], out["fresh"]
    assert a[0] == b[0] and a[1] == b[1] and a[2] == b[2]
    assert a[3] == b[3], "final_test logits differ"
    assert _same_bits(a[4], b[4])
    assert _same_bits(ema.ema.core().arena.w16, fresh.core().arena.w16)


# ---- 6. checkpoint round trip ----------------------------------------------------------------------------------------------------------
def test_checkpoint_round_trip_restores_the_ema_arena_and_shadow(tmp_path):
    from unite_b200.checkpoint import auto_load_model, save_model
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import train_one_epoch
    scfg, vit = _tiny_vit()
    opt = _fresh_opt(vit)
    ema = ModelEma(vit, decay=0.9)
    g = torch.Generator().manual_seed(13)
    data = [(torch.randn(2, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g), torch.randint(0, scfg.num_classes, (2,), generator=g))
            for _ in range(3)]
    train_one_epoch(vit, None, data, opt, "cuda", 0, None, model_ema=ema, lr_schedule_values=[5e-3] * 3)
    save_model(str(tmp_path), 0, vit, opt, model_ema=ema)
    _, vit2 = _tiny_vit()
    opt2 = _fresh_opt(vit2)
    ema2 = ModelEma(vit2, decay=0.9)
    with torch.no_grad():
        ema2.ema(data[0][0].cuda())                                              # the core and its shadow exist before the load
    assert auto_load_model(str(tmp_path), vit2, opt2, model_ema=ema2) == 1
    a, b = ema.ema.core().arena, ema2.ema.core().arena
    assert _same_bits(a.params, b.params) and _same_bits(a.w16, b.w16)
    assert _same_bits(vit.core().arena.params, vit2.core().arena.params)


# ---- 7. full-size ViT-B/16, graph step -------------------------------------------------------------------------------------------------
def test_full_vitb16_stage2_graph_step_ema_is_bit_exact():
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    vit = _vitb16_stage2().cuda().train()
    L = vit.get_num_layers()
    asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(Args, vit, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
    ema = ModelEma(vit, decay=0.9999)
    eng = Stage2Engine(vit, opt, use_graph=True, model_ema=ema)
    e0 = ema.ema.core().arena.params.clone()
    g = torch.Generator().manual_seed(21)
    x = torch.randn(4, 3, 8, 224, 224, generator=g).cuda()
    y = torch.randint(0, 12, (4,), generator=g).cuda()
    recorded, emas = [], []
    for _ in range(4):                                                                # 2 eager warm-up steps, then 2 graph replays
        eng.step(x, y)
        recorded.append(vit.core().arena.params.clone())
        emas.append(ema.ema.core().arena.params.clone())
    torch.cuda.synchronize()
    assert len(eng.graphs._graphs) == 1
    for s, (got, exp) in enumerate(zip(emas, _replay_reference(e0, recorded, 0.9999))):
        assert _same_bits(got, exp), f"update {s}"
    assert _same_bits(ema.ema.core().arena.w16, _bf16(emas[-1]))


# ---- 8. several GPUs: every rank's EMA is the same -----------------------------------------------------------------------------------
def test_ema_is_identical_across_ranks():
    n_gpu = torch.cuda.device_count()
    if n_gpu < 2:
        pytest.skip("needs 2 GPUs")
    world = min(n_gpu, 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                        "--master-port", "29571", os.path.join(ROOT, "tools", "ema_ddp_check.py"), "--steps", "4"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0 and "EMA PARITY OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])
