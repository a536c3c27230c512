"""Round-2 parity cases on the GPU (through the C ABI), each against the CPU oracle on the same seeded inputs:
DropPath (injected factors, device generator, CUDA-graph replay), the benchmarked B=32 shapes, clip_loss_data source/target,
layer-decay AdamW groups and frozen parameters, many-sample stage-2 / stage-3 / alternative losses at the 1e-3 loss gate,
and the stage-3 drop-in loop with the dual-view target batch."""
from functools import partial

import numpy as np
import pytest
import torch

from tests.util import (build_student, build_teacher, cosine, load_golden, oracle_cfgs, per_token_rel, rel_l2, seeded_states)

pytestmark = pytest.mark.gpu
FEAT_TOL, LOSS_TOL = 1e-2, 1e-3


def _tiny(drop_path_rate=0.0):
    fix = load_golden("tiny_stage12.pt")
    scfg, tcfg = oracle_cfgs(fix)
    ssd, tsd, vsd = seeded_states(fix)
    student, teacher = build_student(scfg, drop_path_rate=drop_path_rate), build_teacher(tcfg)
    student.load_state_dict(ssd, strict=True)
    teacher.load_state_dict(tsd, strict=True)
    return fix, scfg, tcfg, ssd, tsd, vsd, student.cuda().train(), teacher.cuda().eval()


def _tiny_batch(scfg, B, seed):
    g = torch.Generator().manual_seed(seed)
    videos = torch.randn(B, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g)
    q = torch.empty(B * scfg.num_frames // scfg.tubelet_size, (scfg.img_size // 16) ** 2).exponential_(1, generator=g)
    return videos, q


# ---- DropPath -----------------------------------------------------------------------------------------------------------
def test_drop_path_draw_is_bit_exact_against_host_philox_and_advances_its_counter():
    from oracle.philox import drop_path_factors
    from unite_b200 import ops
    for depth, B, rate, seed in ((12, 32, 0.1, 0), (24, 5, 0.3, 0x1234567887654321), (3, 1, 0.0, 7)):
        rates = torch.linspace(0, rate, depth)
        step = torch.zeros(1, dtype=torch.int64, device="cuda")
        out = torch.empty(depth, 2, B, device="cuda")
        for s in range(3):
            ops.drop_path_draw(rates.cuda(), out, seed, step)
            torch.cuda.synchronize()
            ref = drop_path_factors(rates.numpy(), B, seed, s)
            assert np.array_equal(out.cpu().numpy(), ref), (depth, B, rate, s)
            assert int(step.item()) == s + 1
        if rate > 0:
            assert float((out == 0).float().mean()) < rate                       # dropped fraction below the largest rate
            assert torch.all((out == 0) | (out >= 1.0))


def test_stage1_with_injected_drop_path_factors_against_oracle():
    """SURVEY.md §7: one run with an injected keep mask.  modeling_finetune.py:42-50 (DropPath on both residual branches)."""
    from oracle import unite_oracle as O
    from unite_b200.engine import Stage1Engine
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny(drop_path_rate=0.4)
    B = 8
    videos, q = _tiny_batch(scfg, B, 5)
    g = torch.Generator().manual_seed(9)
    keep = 1.0 - torch.linspace(0, 0.4, scfg.depth).view(-1, 1, 1)
    dp = (torch.floor(keep + torch.rand(scfg.depth, 2, B, generator=g)) / keep).contiguous()
    assert 0 < int((dp == 0).sum()) < dp.numel() // 2
    ref = O.stage1_step(ssd, tsd, videos, q, scfg, tcfg, mask_ratio=fix["cfg"]["mask_ratio"], keep_scales=dp)
    eng = Stage1Engine(student, teacher, mask_ratio=fix["cfg"]["mask_ratio"])
    eng.optimizer.zero_grad()
    loss = eng.forward_backward(videos.cuda(), q.cuda(), dp=dp.cuda(), attn_override=ref["attn"].cuda().contiguous())
    torch.cuda.synchronize()
    assert torch.equal(eng.last["mask"].cpu(), ref["mask"])
    assert per_token_rel(eng.last["outputs"], ref["outputs"]).max() < FEAT_TOL
    assert abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item()) < LOSS_TOL
    for k, g_ref in ref["grads"].items():
        if g_ref.numel() < 4096:
            continue
        assert cosine(eng.core.arena.g32(k), g_ref) >= 0.999, k
        assert rel_l2(eng.core.arena.g32(k), g_ref) <= 2e-2, k


def test_cuda_graph_step_draws_fresh_drop_path_factors_on_every_replay():
    """The shipped drop_path: 0.1 runs INSIDE the captured step: the generator's step counter lives on the device, so replay s
    uses the factors of draw s — checked against an eager engine fed with the host-reproduced factors (lr = 0 keeps weights fixed)."""
    from oracle.philox import drop_path_factors
    from unite_b200.engine import Stage1Engine
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny(drop_path_rate=0.5)
    videos, q = _tiny_batch(scfg, 8, 6)
    videos, q = videos.cuda(), q.cuda()
    eng = Stage1Engine(student, teacher, mask_ratio=fix["cfg"]["mask_ratio"], lr=0.0, weight_decay=0.0, use_graph=True)
    rates = student.encoder.drop_path_rates
    losses = []
    for s in range(6):                                                            # 2 eager warm-up steps, then capture + replays
        losses.append(eng.step(videos, q).clone())
        torch.cuda.synchronize()
    assert len(eng.graphs._graphs) == 1, "the DropPath step was not captured in a CUDA graph"
    n_draws = int(eng.drop_path.step.item())
    assert n_draws == 6, f"{n_draws} draws for 6 steps (capture itself must not consume a draw)"
    student2 = build_student(scfg, drop_path_rate=0.5)
    student2.load_state_dict(ssd, strict=True)
    eng2 = Stage1Engine(student2.cuda().train(), teacher, mask_ratio=fix["cfg"]["mask_ratio"], lr=0.0, weight_decay=0.0)
    distinct = set()
    for s in range(6):
        dp = torch.from_numpy(drop_path_factors(np.asarray(rates, dtype=np.float32), 8, 0, s)).cuda()
        eng2.optimizer.zero_grad()
        ref = eng2.forward_backward(videos, q, dp=dp)
        torch.cuda.synchronize()
        assert abs(ref.item() - losses[s].item()) <= 2e-5 * abs(ref.item()), (s, ref.item(), losses[s].item())
        distinct.add(round(ref.item(), 6))
    assert len(distinct) >= 5, "replays reused the same DropPath factors"


# ---- the benchmarked shapes ----------------------------------------------------------------------------------------------
def test_full_vitb16_stage1_at_bench_batch_32_against_oracle():
    """B = 32 (BASELINE configs[1]: M = 10 240 student rows, 50 432 teacher rows — the tile / pair / split-K choices bench.py
    actually runs).  Forward quantities against the oracle on the CPU: mask bit-exact, features 1e-2, loss 1e-3."""
    from oracle import unite_oracle as O
    from oracle.weights import seeded_state
    from unite_b200.engine import Stage1Engine
    scfg, tcfg = O.StudentCfg(), O.TeacherCfg()
    student, teacher = build_student(scfg), build_teacher(tcfg)
    ssd = seeded_state({k: tuple(v.shape) for k, v in student.state_dict().items()}, 0)
    tsd = seeded_state({k: tuple(v.shape) for k, v in teacher.state_dict().items()}, 1)
    student.load_state_dict(ssd); teacher.load_state_dict(tsd)
    g = torch.Generator().manual_seed(32)
    B = 32
    videos = torch.randn(B, 3, 8, 224, 224, generator=g)
    q = torch.empty(B * 8, 196).exponential_(1, generator=g)
    ref = O.stage1_step(ssd, tsd, videos, q, scfg, tcfg, mask_ratio=0.8, with_grads=False)
    eng = Stage1Engine(student.cuda().train(), teacher.cuda().eval(), mask_ratio=0.8)
    eng.optimizer.zero_grad()
    loss = eng.forward_backward(videos.cuda(), q.cuda(), attn_override=ref["attn"].cuda().contiguous())
    torch.cuda.synchronize()
    assert rel_l2(eng.last["attn"], ref["attn"]) < FEAT_TOL
    assert torch.equal(eng.last["mask"].cpu(), ref["mask"])
    assert torch.equal(eng.last["vis_idx"].cpu().long(), O.visible_indices(ref["mask"]))
    K, _, Nv, C = ref["targets"].shape
    t_err = per_token_rel(eng.last["targets"].view(K, B, Nv, C), ref["targets"])
    o_err = per_token_rel(eng.last["outputs"], ref["outputs"])
    l_rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
    print(f"B=32: targets max {t_err.max():.2e}, outputs max {o_err.max():.2e}, loss {loss.item():.6f} vs {ref['loss'].item():.6f} ({l_rel:.1e})")
    assert t_err.max() < FEAT_TOL and o_err.max() < FEAT_TOL and l_rel < LOSS_TOL
    # grouped decoder GEMMs (one launch for the K heads: forward, dgrad, wgrad — active at these shapes) against the K separate
    # launches on the same inputs: identical math, different fp32 accumulation order
    assert eng.core._grouped(B * 320), "the grouped decoder path is not active at the benchmarked shapes"
    arena = eng.core.arena
    names = [f"clip_decoder.{k}.head.weight" for k in range(6)] + ["clip_decoder.3.head.bias", "encoder.blocks.11.mlp.fc2.weight",
                                                                    "encoder.blocks.6.attn.qkv.weight", "encoder.blocks.0.mlp.fc1.weight"]
    g_grouped = {n: arena.g32(n).clone() for n in names}
    out_grouped = eng.last["outputs"].clone()
    eng.core._group_dec = False
    eng.core._dec_ws.clear()
    eng.optimizer.zero_grad()
    eng.forward_backward(videos.cuda(), q.cuda(), attn_override=ref["attn"].cuda().contiguous())
    torch.cuda.synchronize()
    assert rel_l2(out_grouped, eng.last["outputs"]) < 1e-6
    for n in names:
        # the decoders' own gradients see a different split-K factor (fp32 partial sums over 10 240 tokens with cancellation:
        # ~1e-4 relative); the trunk's also carry the run-to-run order of the fp32 red.adds of 12 layers of weight gradients
        tol = 3e-4 if n.startswith("clip_decoder") else 1e-3
        assert rel_l2(g_grouped[n], arena.g32(n)) < tol, (n, rel_l2(g_grouped[n], arena.g32(n)))
    eng.core._group_dec = True
    eng.core._dec_ws.clear()
    # the mask the engine derives from ITS OWN attention differs from the oracle's only where attn/q ties are within fp noise
    eng.forward_backward(videos.cuda(), q.cuda())
    torch.cuda.synchronize()
    own = eng.last["mask"].cpu()
    assert int(own.sum()) == int(ref["mask"].sum())
    assert float((own != ref["mask"]).float().mean()) < 2e-3


# ---- clip_loss_data ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("data,kind", [("source", "l2"), ("target", "l2"), ("source", "mse"), ("target", "smooth_l1")])
def test_clip_loss_data_source_and_target_against_oracle(data, kind):
    """run_stage1.py:418-423: outputs / targets sliced to the first B_s clips or the rest before the loss."""
    from oracle import unite_oracle as O
    from unite_b200.engine import Stage1Engine
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny()
    B, Bs = 8, 3
    videos, q = _tiny_batch(scfg, B, 11)
    ref = O.stage1_step(ssd, tsd, videos, q, scfg, tcfg, mask_ratio=fix["cfg"]["mask_ratio"], clip_loss_type=kind, clip_loss_data=data,
                        n_source=Bs)
    eng = Stage1Engine(student, teacher, mask_ratio=fix["cfg"]["mask_ratio"], clip_loss_type=kind)
    eng.clip_loss_data, eng.n_source = data, Bs
    eng.optimizer.zero_grad()
    loss = eng.forward_backward(videos.cuda(), q.cuda(), attn_override=ref["attn"].cuda().contiguous())
    torch.cuda.synchronize()
    l_rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
    assert l_rel < (LOSS_TOL if kind == "l2" else 2e-3), (loss.item(), ref["loss"].item())
    assert per_token_rel(eng.last["outputs"], ref["outputs"]).max() < FEAT_TOL          # every clip is still computed
    for k, g_ref in ref["grads"].items():
        if g_ref.numel() < 4096:
            continue
        assert cosine(eng.core.arena.g32(k), g_ref) >= 0.999, (data, kind, k)
        assert rel_l2(eng.core.arena.g32(k), g_ref) <= 2e-2, (data, kind, k)


def test_train_one_epoch_passes_clip_loss_data_and_source_count():
    from unite_b200.engine_for_pretraining import train_one_epoch
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny()
    vs, qs = _tiny_batch(scfg, 2, 1)
    vt, qt = _tiny_batch(scfg, 3, 2)

    class A:
        log_freq = 1
        clip_loss_data = "target"
    stats = train_one_epoch(student, [(vs, -1, torch.zeros(2), qs)] * 2, [(vt, -1, torch.zeros(3), qt)], None, "cuda", 0, None,
                            teacher_model=teacher, mask_type="attention", mask_ratio=fix["cfg"]["mask_ratio"], args=A)
    eng = student.__dict__["_ub_stage1_engine"][1]
    assert eng.clip_loss_data == "target" and eng.n_source == 2 and eng.last["outputs"].shape[1] == 5
    assert np.isfinite(stats["loss"])
    with pytest.raises(TypeError):
        train_one_epoch(student, [(vs, -1, torch.zeros(2), qs)], None, torch.optim.AdamW(student.parameters(), lr=1e-3), "cuda", 0, None,
                        teacher_model=teacher, mask_type="attention", mask_ratio=fix["cfg"]["mask_ratio"], args=A)


# ---- optimizer groups ----------------------------------------------------------------------------------------------------
def _build_vit(scfg, drop_path_rate=0.0):
    import torch.nn as nn
    from unite_b200.modeling_finetune import VisionTransformer
    return VisionTransformer(img_size=scfg.img_size, patch_size=scfg.patch_size, embed_dim=scfg.embed_dim, depth=scfg.depth,
                             num_heads=scfg.num_heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                             num_classes=scfg.num_classes, all_frames=scfg.num_frames, tubelet_size=scfg.tubelet_size,
                             init_scale=0.001, use_mean_pooling=True, drop_path_rate=drop_path_rate)


def test_layer_decay_groups_and_frozen_parameters_match_torch_adamw():
    """src/optim_factory.py:45-118 with LayerDecayValueAssigner(0.65 ** (L + 1 - i)) (run_stage2.py:616-617,
    configs/stage2_config.yaml:35) and two frozen tensors, 3 steps with a per-step lr schedule, against torch.optim.AdamW over
    the same groups."""
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    fix, scfg, *_ = _tiny()
    _, _, vsd = seeded_states(fix)
    vit = _build_vit(scfg)
    vit.load_state_dict(vsd, strict=True)
    vit = vit.cuda()
    vit.blocks[0].mlp.fc1.weight.requires_grad_(False)                            # run_stage2.py frozen_layers-style freezing
    vit.patch_embed.proj.bias.requires_grad_(False)
    L = vit.get_num_layers()
    assigner = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(Args, vit, skip_list=vit.no_weight_decay(), get_num_layer=assigner.get_layer_id,
                           get_layer_scale=assigner.get_scale)
    scales = {g["name"]: g["lr_scale"] for g in opt.param_groups}
    assert abs(scales["layer_1_decay"] - 0.65 ** L) < 1e-12 and abs(scales[f"layer_{L + 1}_decay"] - 1.0) < 1e-12
    arena = vit.core().arena
    # torch reference over the same groups (optim_factory.py:76-118 restated)
    ps = {k: p.detach().clone().requires_grad_(p.requires_grad) for k, p in vit.named_parameters()}
    groups = {}
    skip = vit.no_weight_decay()
    for k, p in ps.items():
        if not p.requires_grad:
            continue
        nd = p.ndim == 1 or k.endswith(".bias") or k in skip
        lid = assigner.get_layer_id(k)
        gname = "layer_%d_%s" % (lid, "no_decay" if nd else "decay")
        groups.setdefault(gname, dict(params=[], weight_decay=0.0 if nd else 0.05, lr_scale=assigner.get_scale(lid)))["params"].append(p)
    assert {g_["name"] for g_ in opt.param_groups} == set(groups), "group names differ from get_parameter_groups'"
    ref = torch.optim.AdamW(list(groups.values()), lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    g = torch.Generator(device="cuda").manual_seed(3)
    sched = [1e-3, 7e-4, 4e-4]
    frozen_before = {k: ps[k].clone() for k in ("blocks.0.mlp.fc1.weight", "patch_embed.proj.bias")}
    for it in range(3):
        for grp in opt.param_groups:
            grp["lr"] = sched[it] * grp["lr_scale"]
        for grp in ref.param_groups:
            grp["lr"] = sched[it] * grp["lr_scale"]
        arena.grads.zero_()                                                      # alignment gaps and the zero key-bias gap stay 0
        for k in ps:
            arena.g32(k).copy_(torch.randn(arena.g32(k).shape, device="cuda", generator=g) * 1e-2)
        for k, p in ps.items():
            p.grad = arena.g32(k).clone() if p.requires_grad else None
        opt.step()
        ref.step()
    torch.cuda.synchronize()
    sd = vit.state_dict()
    for k, p in ps.items():
        assert rel_l2(sd[k], p) < 1e-6, k
    for k, v in frozen_before.items():
        assert torch.equal(sd[k], v), f"frozen parameter {k} was updated"
    assert torch.equal(arena.b16("blocks.1.attn.qkv.weight").float(), sd["blocks.1.attn.qkv.weight"].bfloat16().float())
    # the gradient norm covers trainable parameters only (utils.py:631-643 over p.grad is not None)
    want = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in ps.values() if p.grad is not None)).item()
    assert abs(opt.grad_norm().item() - want) < 1e-4 * want


def test_stage2_train_one_epoch_uses_the_callers_layer_decay_optimizer():
    from unite_b200.engine_for_finetuning import train_one_epoch
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    fix, scfg, *_ = _tiny()
    _, _, vsd = seeded_states(fix)
    vit = _build_vit(scfg, drop_path_rate=0.1)
    vit.load_state_dict(vsd, strict=True)
    vit = vit.cuda()
    L = vit.get_num_layers()
    assigner = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(Args, vit, get_num_layer=assigner.get_layer_id, get_layer_scale=assigner.get_scale)
    batch = (fix["videos"], fix["labels"], torch.zeros(2), {})
    s0 = train_one_epoch(vit, torch.nn.CrossEntropyLoss(), [batch] * 2, opt, "cuda", 0, None, update_freq=1, lr_schedule_values=[2e-3] * 50)
    s1 = train_one_epoch(vit, torch.nn.CrossEntropyLoss(), [batch] * 20, opt, "cuda", 1, None, update_freq=1, lr_schedule_values=[2e-3] * 50,
                         start_steps=2)
    assert opt.step_count == 22 and s1["loss"] < s0["loss"]
    assert abs(s1["min_lr"] - 2e-3 * 0.65 ** (L + 1)) < 1e-12 and abs(s1["lr"] - 2e-3) < 1e-12      # layer 0 = patch_embed
    with pytest.raises(TypeError):
        train_one_epoch(vit, None, [batch], torch.optim.AdamW(vit.parameters(), lr=1e-3), "cuda", 0, None)


# ---- many-sample losses at the 1e-3 gate -----------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["mse", "smooth_l1", "l1"])
def test_alternative_alignment_losses_at_32_clips_meet_the_loss_gate(kind):
    from oracle import unite_oracle as O
    from unite_b200.engine import Stage1Engine
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny()
    videos, q = _tiny_batch(scfg, 32, 13)
    ref = O.stage1_step(ssd, tsd, videos, q, scfg, tcfg, mask_ratio=fix["cfg"]["mask_ratio"], clip_loss_type=kind, with_grads=False)
    eng = Stage1Engine(student, teacher, mask_ratio=fix["cfg"]["mask_ratio"], clip_loss_type=kind)
    eng.optimizer.zero_grad()
    loss = eng.forward_backward(videos.cuda(), q.cuda(), attn_override=ref["attn"].cuda().contiguous())
    torch.cuda.synchronize()
    l_rel = abs(loss.item() - ref["loss"].item()) / abs(ref["loss"].item())
    print(f"{kind} @32 clips: {loss.item():.6e} vs {ref['loss'].item():.6e} ({l_rel:.1e})")
    assert l_rel < LOSS_TOL


def test_stage2_loss_at_256_clips_meets_the_loss_gate():
    from oracle import unite_oracle as O
    from unite_b200.engine_for_finetuning import finetune_step
    fix, scfg, *_ = _tiny()
    _, _, vsd = seeded_states(fix)
    # a head with O(1) logits (init_scale 0.001 gives CE == ln C whatever the trunk does; logits of std >> 1 make CE linear in
    # the logits, so that its relative error is the logit error, 3e-3, whatever the sample size)
    g = torch.Generator().manual_seed(17)
    vsd = dict(vsd)
    vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=g) * 0.05
    vit = _build_vit(scfg)
    vit.load_state_dict(vsd, strict=True)
    vit = vit.cuda().eval()                                                        # eval: no DropPath draw
    n = 256           # the CE error is the mean of per-sample logit noise (bf16 operands): it averages down like 1 / sqrt(n)
    videos = torch.randn(n, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g)
    labels = torch.randint(0, scfg.num_classes, (n,), generator=g)
    ref = O.stage2_step(vsd, videos, labels, scfg, with_grads=False)
    loss = torch.zeros(1, device="cuda")
    logits = finetune_step(vit, videos.cuda(), labels.cuda(), loss)
    torch.cuda.synchronize()
    assert rel_l2(logits, ref["logits"]) < FEAT_TOL
    l_rel = abs(loss.item() - ref["loss"].item()) / ref["loss"].item()
    print(f"stage-2 CE @{n} clips: {loss.item():.6f} vs {ref['loss'].item():.6f} ({l_rel:.1e})")
    assert l_rel < LOSS_TOL


def _stable_rows(ref, m_logit=2e-2, m_clip=3e-2):
    p = torch.softmax(ref["logits_full_t"], -1)
    top2 = p.topk(2, -1).values
    stable = (top2[:, 0] - top2[:, 1] > m_logit) & ((ref["msp"] - 0.5).abs() > m_logit)
    cp = ref["clip_probs"].topk(2, -1).values
    return stable & (cp[:, 0] - cp[:, 1] > m_clip) & ((cp[:, 0] - 0.5).abs() > m_clip)


def test_stage3_dual_view_at_256_clips_meets_the_loss_gate_and_trains_through_train_one_epoch():
    """run_stage3.py:405-413: the teacher attention and the masked committee see vid_aug, the full-token pass and the zero-shot
    head see vid.  256 target clips picked (by the ORACLE, clips are independent) so that every discrete decision has a margin
    above fp noise; then masks / pseudo labels / selection bit-exact and all three losses within 1e-3."""
    from oracle import unite_oracle as O
    from unite_b200.engine_stage3 import Stage3Engine, train_one_epoch
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny()
    C, D, Bs, Bt, pool = 12, scfg.embed_dim, 128, 256, 640
    g = torch.Generator().manual_seed(2024)
    cls_w = torch.randn(C, D, generator=g) * 0.1                                  # logits of std ~1: a mix of confident / unsure clips
    cls_b = torch.randn(C, generator=g) * 0.1
    text = torch.randn(C, tcfg.output_dim, generator=g)
    shape = (3, scfg.num_frames, scfg.img_size, scfg.img_size)
    videos_s = torch.randn(Bs, *shape, generator=g)
    labels_s = torch.randint(0, C, (Bs,), generator=g)
    cand = torch.randn(pool, *shape, generator=g)
    cand_aug = cand + 0.1 * torch.randn(pool, *shape, generator=g)
    r = O.stage3_step(ssd, tsd, cls_w, cls_b, text, videos_s[:2], labels_s[:2], cand, scfg, tcfg, mask_ratio=0.75, k=2, with_grads=False,
                      videos_t_aug=cand_aug)
    ok = _stable_rows(r).nonzero().flatten()
    assert ok.numel() >= Bt, f"only {ok.numel()} of {pool} candidate clips have stable decisions"
    videos_t, videos_t_aug = cand[ok[:Bt]].contiguous(), cand_aug[ok[:Bt]].contiguous()
    ref = O.stage3_step(ssd, tsd, cls_w, cls_b, text, videos_s, labels_s, videos_t, scfg, tcfg, mask_ratio=0.75, k=2,
                        videos_t_aug=videos_t_aug)
    assert int(ref["sel_mask"].sum()) >= 32
    student.eval()                                                                 # parity run without DropPath draws
    eng = Stage3Engine(student, teacher, cls_w, cls_b, text, mask_ratio=0.75, k=2)
    eng.optimizer.zero_grad()
    loss = eng.forward_backward(videos_s.cuda(), labels_s.cuda(), videos_t.cuda(), videos_t_aug.cuda(),
                                attn_override=ref["attn"].cuda().contiguous())
    torch.cuda.synchronize()
    Lr = eng.last
    assert rel_l2(Lr["attn"], ref["attn"]) < FEAT_TOL
    assert torch.equal(Lr["masks"].cpu(), ref["masks"])
    for key in ("logits_s", "logits_full_t", "logits_masked", "msp"):
        assert rel_l2(Lr[key], ref[key]) < FEAT_TOL, key
    assert torch.equal(Lr["pseudo"].cpu().long(), ref["pseudo"]) and torch.equal(Lr["sel_mask"].cpu(), ref["sel_mask"])
    for name, got, want in (("loss_s", eng.loss_s, ref["loss_s"]), ("loss_t", eng.loss_t, ref["loss_t"]), ("loss", loss, ref["loss"])):
        rel = abs(got.item() - want.item()) / abs(want.item())
        print(f"stage-3 {name} @{Bs}+{Bt} clips: {got.item():.6f} vs {want.item():.6f} ({rel:.1e})")
        assert rel < LOSS_TOL, name
    for k in ("encoder.blocks.0.attn.qkv.weight", "encoder.blocks.2.mlp.fc2.weight", "encoder.patch_embed.proj.weight"):
        assert cosine(eng.core.arena.g32(k), ref["grads"][k]) >= 0.999, k
    # ---- the drop-in loop (run_stage3.py:340-350 signature) over the dual-view loader contract
    student.train()

    class Args:
        masking_type, selection_strategy, train_masked, conf_weighted_loss = "clip_attention", "clip_matchORconf", True, True
        class_loss_src_ratio, class_loss_src_ratio_pl, class_loss_tgt_ratio, clip_threshold = 1.0, 1.0, 1.0, 0.5
        return_aug_for_val, full_oracle, log_freq = True, False, 10
        text_features = text
    src_classifier = torch.nn.Linear(D, C)
    with torch.no_grad():
        src_classifier.weight.copy_(cls_w); src_classifier.bias.copy_(cls_b)
    src = [(videos_s[:4], labels_s[:4], torch.arange(4), {})] * 3
    tgt = [(videos_t[:4], videos_t_aug[:4], torch.zeros(4, dtype=torch.long), ["a", "b", "c", "d"])] * 2      # shorter: must cycle (:369-375)
    stats = train_one_epoch(student, src, tgt, None, "cuda", 0, None, src_classifier=src_classifier.cuda(), teacher_model=teacher,
                            mask_type="attention", mask_ratio=0.75, args=Args, lr_schedule_values=[1e-4] * 10)
    assert set(stats) >= {"loss", "loss_class", "loss_class_t", "lr", "min_lr", "weight_decay", "grad_norm"}
    assert all(np.isfinite(stats[k]) for k in ("loss", "loss_class", "loss_class_t", "grad_norm"))
    assert abs(stats["loss"] - (stats["loss_class"] + stats["loss_class_t"])) < 1e-5


# ---- stage 2 at full size: all 1568 tokens through the long-sequence tcgen05 attention ---------------------------------------
def test_full_vitb16_stage2_all_tokens_against_oracle():
    """BASELINE configs[0] shape on the GPU: ViT-B/16, 8x224^2, every one of the 1568 tokens (S = 1568 attention runs on
    csrc/attention_long_tc.cu: forward with LSE + two-pass backward), B = 2, against the oracle on the CPU."""
    from oracle import unite_oracle as O
    from oracle.weights import seeded_state
    from unite_b200.engine_for_finetuning import finetune_step
    scfg = O.StudentCfg(num_classes=12)
    vit = _build_vit(scfg)
    vsd = seeded_state({k: tuple(v.shape) for k, v in vit.state_dict().items()}, 3)
    g = torch.Generator().manual_seed(41)
    vsd["head.weight"] = torch.randn(vsd["head.weight"].shape, generator=g) * 0.02         # O(1) logits
    vit.load_state_dict(vsd, strict=True)
    vit = vit.cuda().eval()
    videos = torch.randn(2, 3, 8, 224, 224, generator=g)
    labels = torch.randint(0, 12, (2,), generator=g)
    ref = O.stage2_step(vsd, videos, labels, scfg)
    loss = torch.zeros(1, device="cuda")
    logits = finetune_step(vit, videos.cuda(), labels.cuda(), loss)
    torch.cuda.synchronize()
    l_rel = abs(loss.item() - ref["loss"].item()) / ref["loss"].item()
    print(f"stage-2 full size: logits rel {rel_l2(logits, ref['logits']):.2e}, loss {loss.item():.5f} vs {ref['loss'].item():.5f} ({l_rel:.1e})")
    assert rel_l2(logits, ref["logits"]) < FEAT_TOL
    assert l_rel < 5e-3            # a 2-sample CE: its budget is the logit tolerance; the 1e-3 gate is checked at 256 clips above
    arena = vit.core().arena
    worst_c, worst_r = 1.0, 0.0
    for k, g_ref in ref["grads"].items():
        if g_ref.numel() < 4096:
            continue
        c, r = cosine(arena.g32(k), g_ref), rel_l2(arena.g32(k), g_ref)
        worst_c, worst_r = min(worst_c, c), max(worst_r, r)
        assert c >= 0.999 and r <= 2e-2, (k, c, r)
    print(f"stage-2 full size grads: worst cosine {worst_c:.6f}, worst rel-L2 {worst_r:.2e}")


# ---- several optimizer steps in a row: the whole loop (forward, backward, AdamW, bf16 shadow refresh) tracks the reference ---------
def test_four_training_steps_track_the_oracle_with_torch_adamw():
    """run_stage1.py:360-456 repeated: oracle step -> torch.optim.AdamW (decay / no-decay groups, optim_factory.py:76-118) on the CPU
    against Stage1Engine.step (with the CUDA graph: steps 3 and 4 are replays).  Losses within 1e-3 at every step; the accumulated
    UPDATE of every large tensor points where the reference's does (cosine >= 0.97) and the weights stay within 2e-2 relative (Adam's
    m / sqrt(v) turns the bf16 noise of near-zero gradient elements into sign flips of lr-sized steps, so the weights themselves
    cannot be held to the per-step gradient tolerance)."""
    from oracle import unite_oracle as O
    from unite_b200.engine import Stage1Engine
    fix, scfg, tcfg, ssd, tsd, _, student, teacher = _tiny()
    student.eval()                                                                  # no DropPath in this trajectory
    B, lr, wd = 8, 2e-3, 0.05
    batches = [_tiny_batch(scfg, B, 100 + i) for i in range(2)]
    ps = {k: v.clone().requires_grad_() for k, v in ssd.items()}
    dec = [p for k, p in ps.items() if not (p.ndim == 1 or k.endswith(".bias"))]
    nod = [p for k, p in ps.items() if (p.ndim == 1 or k.endswith(".bias"))]
    opt = torch.optim.AdamW([dict(params=dec, weight_decay=wd), dict(params=nod, weight_decay=0.0)], lr=lr, betas=(0.9, 0.95), eps=1e-8)
    eng = Stage1Engine(student, teacher, mask_ratio=fix["cfg"]["mask_ratio"], lr=lr, weight_decay=wd, use_graph=True)
    dev_batches = [(v.cuda(), q.cuda()) for v, q in batches]
    for it in range(4):
        v, q = batches[it % 2]
        cur = {k: p.detach() for k, p in ps.items()}
        ref = O.stage1_step(cur, tsd, v, q, scfg, tcfg, mask_ratio=fix["cfg"]["mask_ratio"])
        for k, p in ps.items():
            p.grad = ref["grads"][k]
        opt.step()
        loss = eng.step(*dev_batches[it % 2]).item()
        rel = abs(loss - ref["loss"].item()) / abs(ref["loss"].item())
        print(f"step {it}: loss {loss:.6f} vs {ref['loss'].item():.6f} ({rel:.1e})")
        assert rel < LOSS_TOL, (it, loss, ref["loss"].item())
    assert len(eng.graphs._graphs) >= 1
    sd = student.state_dict()
    worst, worst_cos = 0.0, 1.0
    for k, p in ps.items():
        if p.numel() < 4096:
            continue
        worst = max(worst, rel_l2(sd[k], p))
        worst_cos = min(worst_cos, cosine(sd[k].detach().cpu() - ssd[k], p.detach() - ssd[k]))
    print(f"after 4 steps: worst weight rel-L2 {worst:.2e}, worst update cosine {worst_cos:.4f}")
    assert worst < 2e-2 and worst_cos >= 0.97


# ---- CUDA-graph replay of the stage-2 / stage-3 steps ---------------------------------------------------------------------------
def test_stage2_graph_replay_matches_eager_steps():
    """Stage2Engine(use_graph=True): two eager steps, then one captured graph per resident batch, replayed — against an identical
    engine that runs every step eagerly (same weights, same DropPath seed, layer-decay groups, clip_grad on): per-step losses,
    running statistics and the weights after 7 updates agree to accumulation-order noise."""
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    fix, scfg, *_ = _tiny()
    _, _, vsd = seeded_states(fix)
    g = torch.Generator().manual_seed(77)
    shape = (3, scfg.num_frames, scfg.img_size, scfg.img_size)
    batches = [(torch.randn(6, *shape, generator=g).cuda(), torch.randint(0, scfg.num_classes, (6,), generator=g).cuda()) for _ in range(2)]

    class Args:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 2e-4, 0.05, (0.9, 0.999), 1e-8
    runs = []
    # a third, eager, run measures the run-to-run noise of the step itself (fp32 reduce-adds in the weight / LayerNorm gradients
    # arrive in any order): the graph must agree with eager as well as eager agrees with itself
    for use_graph in (True, False, False):
        vit = _build_vit(scfg, drop_path_rate=0.2)
        vit.load_state_dict(vsd, strict=True)
        vit = vit.cuda().train()
        L = vit.get_num_layers()
        asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])
        opt = create_optimizer(Args, vit, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
        eng = Stage2Engine(vit, opt, use_graph=use_graph)
        eng.max_norm = 1.0
        losses = []
        for s in range(7):
            for grp in opt.param_groups:                                          # a schedule: the graph must read lr from device memory
                grp["lr"] = 2e-4 * (1 + s) / 7 * grp["lr_scale"]
            losses.append(eng.step(*batches[s % 2]).clone())
        torch.cuda.synchronize()
        runs.append((torch.cat(losses).cpu(), eng.stats.cpu(), vit.core().arena.params.clone().cpu(), eng))
    (l_g, st_g, p_g, eng_g), (l_e, st_e, p_e, _), (l_e2, _, p_e2, _) = runs
    assert len(eng_g.graphs._graphs) == 2, "one graph per resident batch expected"
    assert int(eng_g.core.drop_path.step.item()) == 7, "capture must not consume a DropPath draw"
    noise_l, noise_p = ((l_e - l_e2).abs() / l_e.abs()).max().item(), rel_l2(p_e, p_e2)
    d_l, d_p = ((l_g - l_e).abs() / l_e.abs()).max().item(), rel_l2(p_g, p_e)
    print(f"stage-2 graph vs eager: loss {d_l:.2e} (eager vs eager {noise_l:.2e}), weights {d_p:.2e} (eager vs eager {noise_p:.2e})")
    assert d_l <= max(2e-5, 4 * noise_l), (l_g, l_e)
    assert len(set(round(v, 5) for v in l_g.tolist())) >= 6, "replays did not see fresh DropPath factors / weights"
    assert torch.allclose(st_g, st_e, rtol=1e-4), (st_g, st_e)
    assert d_p <= max(1e-5, 4 * noise_p)


def test_stage3_graph_replay_matches_eager_steps():
    """Stage3Engine(use_graph=True) against the eager engine: the five forwards, both backwards and AdamW of 6 updates (dual-view
    target batch, DropPath 0.2 in every pass) replayed from the graph give the same losses and weights.  One step from identical
    state is reproducible to fp32 reduction order (tools/stage3_determinism.py: gradients 3.5e-7 of their maximum, every discrete
    decision identical); AdamW turns noise on a near-zero gradient into a full +-lr update of a weight the loss does not depend
    on, so the learning rate is kept small, losses are compared tightly and weights against the distance they travelled."""
    from unite_b200.engine_stage3 import Stage3Engine
    fix, scfg, tcfg, ssd, tsd, *_ = _tiny()
    C, D = 12, scfg.embed_dim
    g = torch.Generator().manual_seed(31)
    cls_w, cls_b, text = torch.randn(C, D, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1, torch.randn(C, tcfg.output_dim, generator=g)
    shape = (3, scfg.num_frames, scfg.img_size, scfg.img_size)
    batches = []
    for _ in range(2):
        vt = torch.randn(4, *shape, generator=g)
        batches.append((torch.randn(4, *shape, generator=g).cuda(), torch.randint(0, C, (4,), generator=g).cuda(), vt.cuda(),
                        (vt + 0.1 * torch.randn(4, *shape, generator=g)).cuda()))
    runs = []
    for use_graph in (True, False):
        student, teacher = build_student(scfg, drop_path_rate=0.2), build_teacher(tcfg)
        student.load_state_dict(ssd, strict=True)
        teacher.load_state_dict(tsd, strict=True)
        eng = Stage3Engine(student.cuda().train(), teacher.cuda().eval(), cls_w, cls_b, text, mask_ratio=0.75, k=2, lr=2e-5, use_graph=use_graph)
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
    print(f"stage-3 graph vs eager: losses {(l_g - l_e).abs().max().item():.2e}, weights {d_p:.2e} of {travelled:.2e} travelled")
    assert torch.allclose(l_g, l_e, rtol=3e-5, atol=1e-6), (l_g, l_e)
    assert travelled > 3e-4 and d_p < 0.02 * travelled
    assert len(set(round(v, 4) for v in l_g[:, 0].tolist())) >= 5, "replays did not see fresh inputs / DropPath factors"
    assert eng_g.last["sel_mask"].shape[0] == 4 and torch.isfinite(eng_g.last["logits_masked"]).all()
