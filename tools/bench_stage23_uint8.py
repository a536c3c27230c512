#!/usr/bin/env python
"""Stages 2 and 3 fed decoded uint8 frames against the fp32 clip: the fused im2col kernels and train_one_epoch end to end, one JSON
line (written to --out as well).

    python tools/bench_stage23_uint8.py [--batch 32] [--steps 10] [--rounds 2] [--launches 200] [--out profiles/x.json]
    torchrun --nproc_per_node N tools/bench_stage23_uint8.py ...        (data parallel: every rank feeds its own pinned batches)

  patchify   ub_patchify_mix (fp32 clip [B,3,8,224,224], 154 MB at B = 32) against ub_patchify_mix_u8 (uint8 frames [B,8,224,224,3],
             38.5 MB), tubelet 1, on a mixup draw and on a cutmix draw.  CUDA events over `launches` back-to-back launches, the four
             alternated `rounds` times; rank 0 only.  Bytes are what the algorithm must move: the input read once and the bf16 rows
             written once; TB/s and the share of the B200's 7.7 TB/s data-sheet HBM bandwidth.
  e2e        train_one_epoch of stage 2 (ViT-B/16, all 1568 tokens, drop_path 0.1, layer-decay AdamW, update_freq 1: CUDA-graph replay)
             plain (CrossEntropyLoss) and with Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1) +
             SoftTargetCrossEntropy, and of stage 3 (ViT-B/16 student, CLIP ViT-B/16 teacher, dual-view target batches, B source +
             B target clips) — each fed from pinned host memory by the synthetic loaders, fp32 clips and uint8 frames alternated
             per round on one model.  Every epoch is warmed first (eager steps and graph capture outside the timed region); the
             timed region includes the host-to-device copies and the loop's final read-back.  ms per step is the slowest rank's.  The two
             feeds are different synthetic draws (Gaussian clips, uniform bytes), so their losses are not comparable.
  gpu        card name, power limit and SM clocks of every local GPU, read in the same run
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_clip_l14 import gpu_info  # noqa: E402

HBM_TBS = 7.7


def kernel_times(args, dev):
    import torch
    from unite_b200 import mixup as M
    from unite_b200 import ops
    B, T, S, C = args.batch, 8, 224, 12
    g = torch.Generator().manual_seed(1000)
    shape = (B, 3, T, S, S)
    x = torch.randn(*shape, generator=g).to(dev)
    fr = torch.randint(0, 256, (B, T, S, S, 3), generator=g, dtype=torch.uint8).to(dev)
    rows = torch.empty(B * T * (S // 16) ** 2, 3 * 256, device=dev, dtype=torch.bfloat16)
    buf_mix, buf_cut = M.MixBuffer(dev), M.MixBuffer(dev)
    buf_mix.upload(M.MixDraw(True, 0.4217, False, ((0, 0), (0, 0), (0, 0)), 0.4217).packed(0.1, C))
    buf_cut.upload(M.MixDraw(True, 0.5, True, M.clip_box(shape, 2, 7, 30, 190), 0.5).packed(0.1, C))
    kernels = dict(patchify_mix_mixup=(lambda: ops.patchify_mix(x, rows, buf_mix.clip, 1), x.numel() * 4),
                   patchify_mix_u8_mixup=(lambda: ops.patchify_mix_u8(fr, rows, buf_mix.clip, 1), fr.numel()),
                   patchify_mix_cutmix=(lambda: ops.patchify_mix(x, rows, buf_cut.clip, 1), x.numel() * 4),
                   patchify_mix_u8_cutmix=(lambda: ops.patchify_mix_u8(fr, rows, buf_cut.clip, 1), fr.numel()))
    us = {k: [] for k in kernels}
    for fn, _ in kernels.values():
        for _ in range(10):
            fn()
    for _ in range(args.rounds):
        for name, (fn, _) in kernels.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.launches):
                fn()
            e1.record()
            torch.cuda.synchronize()
            us[name].append(e0.elapsed_time(e1) * 1e3 / args.launches)
    out = {}
    for name, (_, in_bytes) in kernels.items():
        moved = in_bytes + rows.numel() * 2
        best = min(us[name])
        out[name] = dict(bytes_per_launch=moved, us_per_launch=[round(t, 2) for t in us[name]],
                         tb_s_best=round(moved / (best * 1e-6) / 1e12, 3), hbm_fraction_best=round(moved / (best * 1e-6) / 1e12 / HBM_TBS, 3))
    return dict(shape=list(shape), tubelet=1, launches=args.launches, rounds=args.rounds, l2="inputs exceed the 126 MB L2 only for fp32",
                **out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench_stage23_uint8: no CUDA device")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    gs = None
    if world > 1:
        from unite_b200.ddp import GradSync
        dist.init_process_group("nccl", device_id=dev)
        gs = GradSync()
    import bench
    from unite_b200 import mixup as M
    from unite_b200 import modeling_finetune  # noqa: F401  (registers the factories)
    from unite_b200.engine_for_finetuning import train_one_epoch as train_stage2
    from unite_b200.engine_stage3 import train_one_epoch as train_stage3
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    from unite_b200.registry import create_model
    from unite_b200.synthetic import SyntheticStage2Loader, SyntheticStage3Loader
    B, C = args.batch, 12
    kern = kernel_times(args, dev) if rank == 0 else None

    def timed(run):
        """ms per step of one epoch of `steps` steps (slowest rank), after a warm-up epoch through the same pinned batches."""
        run(args.warmup)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st = run(args.steps)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / args.steps, st

    # ---- stage 2 ----------------------------------------------------------------------------------------------------------------
    torch.manual_seed(0)
    model = create_model("vit_base_patch16_224", pretrained=False, num_classes=C, all_frames=8, tubelet_size=1, drop_rate=0.0,
                         drop_path_rate=bench.DROP_PATH, attn_drop_rate=0.0, drop_block_rate=None, use_mean_pooling=True,
                         init_scale=0.001, fc_drop_rate=0.0, use_checkpoint=False, checkpoint_num=0).to(dev).train()
    L = model.get_num_layers()
    asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class A:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(A, model, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
    if gs is not None:
        gs.arena = model.core().arena
        model.grad_sync = gs
    loaders2 = {u8: SyntheticStage2Loader(B, steps=args.steps, seed=0, rank=rank, n_distinct=2, num_classes=C, uint8=u8)
                for u8 in (False, True)}
    np.random.seed(rank)
    mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1, num_classes=C)

    def stage2(u8, mixed):
        def run(n):
            ld = loaders2[u8]
            ld.steps = n
            if mixed:
                return train_stage2(model, M.SoftTargetCrossEntropy(), ld, opt, dev, 0, None, mixup_fn=mixer)
            return train_stage2(model, None, ld, opt, dev, 0, None)
        return run

    # ---- stage 3 ----------------------------------------------------------------------------------------------------------------
    student, teacher = bench.build_models(seed=0)
    student, teacher = student.to(dev).train(), teacher.to(dev).eval()
    gw = torch.Generator().manual_seed(5)
    cls = torch.nn.Linear(768, C).to(dev)
    with torch.no_grad():
        cls.weight.copy_(torch.randn(C, 768, generator=gw) * 0.5)
        cls.bias.zero_()

    class Args3:
        masking_type, selection_strategy, train_masked, conf_weighted_loss = "clip_attention", "clip_matchORconf", True, True
        class_loss_src_ratio, class_loss_src_ratio_pl, class_loss_tgt_ratio, clip_threshold = 1.0, 1.0, 1.0, 0.5
        return_aug_for_val, full_oracle = True, False
        text_features = torch.randn(C, 512, generator=gw)
    if gs is not None:
        student.grad_sync = gs                            # engine_stage3._engine_for points it at the student's arena
    loaders3 = {u8: SyntheticStage3Loader(B, steps=args.steps, seed=0, rank=rank, n_distinct=2, num_classes=C, uint8=u8)
                for u8 in (False, True)}

    def stage3(u8):
        def run(n):
            ld = loaders3[u8]
            ld.source.steps = ld.target.steps = n
            return train_stage3(student, ld.source, ld.target, None, dev, 0, None, src_classifier=cls, teacher_model=teacher,
                                mask_type="attention", mask_ratio=0.8, args=Args3)
        return run

    legs = {"stage2_plain": lambda u8: stage2(u8, False), "stage2_mixup_cutmix": lambda u8: stage2(u8, True), "stage3_dual_view": stage3}
    ms = {leg: {"fp32": [], "uint8": []} for leg in legs}
    losses = {leg: {} for leg in legs}
    for _ in range(args.rounds):
        for leg, make in legs.items():
            for name, u8 in (("fp32", False), ("uint8", True)):
                t, st = timed(make(u8))
                ms[leg][name].append(round(t, 3))
                losses[leg][name] = round(st["loss"], 5)
    h2d = dict(stage2=dict(fp32=B * 3 * 8 * 224 * 224 * 4, uint8=B * 8 * 224 * 224 * 3))
    h2d["stage3"] = {k: 3 * v for k, v in h2d["stage2"].items()}              # source, target and augmented-target views
    e2e = {}
    for leg in legs:
        per = {}
        for name in ("fp32", "uint8"):
            best = min(ms[leg][name])
            per[name] = dict(ms_per_step=ms[leg][name], clips_per_s_best=round(world * B / (best * 1e-3), 1),
                             h2d_bytes_per_step_per_gpu=h2d["stage3" if leg.startswith("stage3") else "stage2"][name],
                             last_epoch_loss=losses[leg][name])
        per["uint8_over_fp32_best"] = round(min(ms[leg]["uint8"]) / min(ms[leg]["fp32"]), 4)
        e2e[leg] = per
    if rank == 0:
        out = dict(tool="bench_stage23_uint8", n_gpus=world, batch_per_gpu=B, clip=[3, 8, 224, 224],
                   gpu=[gpu_info(i) for i in range(max(world, 1))], patchify=kern,
                   e2e=dict(steps=args.steps, warmup_steps=args.warmup, rounds=args.rounds,
                            order="per round: stage2_plain, stage2_mixup_cutmix, stage3_dual_view, each fp32 then uint8",
                            api="train_one_epoch of engine_for_finetuning / engine_stage3, SyntheticStage2Loader / SyntheticStage3Loader "
                                "(pinned, 2 distinct batches)", clips_note="stage 3 counts source + target pairs", **e2e))
        line = json.dumps(out)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
