#!/usr/bin/env python
"""Stage 2 with mixup / cutmix / label smoothing: the fused im2col kernel and the whole graph-replayed step, one JSON line.

    python tools/bench_stage2_mixup.py [--batch 32] [--steps 20] [--warmup 5] [--rounds 3] [--launches 200]

  patchify              ub_patchify, ub_patchify_mix on a mixup draw and on a cutmix draw, at B x 3 x 8 x 224^2 fp32 (154 MB at
                        B = 32: more than the 126 MB L2, so every pass reads HBM).  CUDA events over `launches` back-to-back
                        launches, the three kernels alternated `rounds` times.  Bytes are what the algorithm must move: the fp32
                        clip read once and the bf16 rows written once (the same for all three); TB/s and the share of the
                        B200's 7.7 TB/s data-sheet HBM bandwidth.
  step                  the bench.py --workload stage2 step (ViT-B/16, all 1568 tokens, drop_path 0.1, layer-decay AdamW, CUDA
                        graph) run plain (CrossEntropyLoss) and with VideoMAE-style regularisation (Mixup(mixup_alpha=0.8,
                        cutmix_alpha=1.0, label_smoothing=0.1), SoftTargetCrossEntropy), alternated A/B/A/B/... on one engine
                        and one box; ms per step of each segment.
  gpu                   card name, power limit and SM clocks read in the same run
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=200)
    args = ap.parse_args()
    import numpy as np
    import torch
    from unite_b200 import modeling_finetune  # noqa: F401  (registers the factories)
    from unite_b200 import mixup as M
    from unite_b200 import ops
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    from unite_b200.registry import create_model
    if not torch.cuda.is_available():
        raise SystemExit("bench_stage2_mixup: no CUDA device")
    import bench
    dev = torch.device("cuda", 0)
    B, T, S, C = args.batch, 8, 224, 12
    g = torch.Generator().manual_seed(1000)
    shape = (B, 3, T, S, S)

    # ---- the kernel alone ----------------------------------------------------------------------------------------------------
    x = torch.randn(*shape, generator=g).to(dev)
    rows = torch.empty(B * T * (S // 16) ** 2, 3 * 256, device=dev, dtype=torch.bfloat16)
    buf_mix, buf_cut = M.MixBuffer(dev), M.MixBuffer(dev)
    buf_mix.upload(M.MixDraw(True, 0.4217, False, ((0, 0), (0, 0), (0, 0)), 0.4217).packed(0.1, C))
    buf_cut.upload(M.MixDraw(True, 0.5, True, M.clip_box(shape, 2, 7, 30, 190), 0.5).packed(0.1, C))
    kernels = dict(patchify=lambda: ops.patchify(x, rows, 1), patchify_mix_mixup=lambda: ops.patchify_mix(x, rows, buf_mix.clip, 1),
                   patchify_mix_cutmix=lambda: ops.patchify_mix(x, rows, buf_cut.clip, 1))
    bytes_moved = x.numel() * 4 + rows.numel() * 2
    us = {k: [] for k in kernels}
    for fn in kernels.values():
        for _ in range(10):
            fn()
    for _ in range(args.rounds):
        for name, fn in kernels.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.launches):
                fn()
            e1.record()
            torch.cuda.synchronize()
            us[name].append(e0.elapsed_time(e1) * 1e3 / args.launches)
    kern = {}
    for name, v in us.items():
        best = min(v)
        kern[name] = dict(us_per_launch=[round(t, 2) for t in v], tb_s_best=round(bytes_moved / (best * 1e-6) / 1e12, 3),
                          hbm_fraction_best=round(bytes_moved / (best * 1e-6) / 1e12 / HBM_TBS, 3))
    del x, rows

    # ---- the whole step, plain vs mixup / cutmix / smoothing, alternated ------------------------------------------------------------
    torch.manual_seed(0)
    model = create_model("vit_base_patch16_224", pretrained=False, num_classes=C, all_frames=T, tubelet_size=1, drop_rate=0.0,
                         drop_path_rate=bench.DROP_PATH, attn_drop_rate=0.0, drop_block_rate=None, use_mean_pooling=True,
                         init_scale=0.001, fc_drop_rate=0.0, use_checkpoint=False, checkpoint_num=0).to(dev).train()
    L = model.get_num_layers()
    asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class A:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(A, model, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
    batches = [(torch.randn(*shape, generator=g).to(dev), torch.randint(0, C, (B,), generator=g).to(dev)) for _ in range(2)]
    eng = Stage2Engine(model, opt, use_graph=os.environ.get("UB_NO_GRAPH", "0") != "1")
    np.random.seed(0)
    mixer = M.Mixup(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1, num_classes=C)
    i = [0]
    kinds = {"none": 0, "mixup": 0, "cutmix": 0}

    def plain():
        v, y = batches[i[0] % 2]
        i[0] += 1
        return eng.step(v, y)

    def mixed():
        v, y = batches[i[0] % 2]
        i[0] += 1
        d = M.draw(mixer, v.shape)
        kinds["cutmix" if d.use_cutmix else ("mixup" if d.apply else "none")] += 1
        return eng.step(v, y, mix=d, smoothing=0.1)

    ms = {"plain": [], "mixup": []}
    for _ in range(args.rounds):
        for name, fn in (("plain", plain), ("mixup", mixed)):
            for _ in range(args.warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                loss = fn()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(round(e0.elapsed_time(e1) / args.steps, 3))
            assert np.isfinite(loss.item())
    out = dict(
        tool="bench_stage2_mixup", batch=B, clip=[3, T, S, S], gpu=gpu_info(0),
        patchify=dict(bytes_per_launch=bytes_moved, launches=args.launches, rounds=args.rounds, **kern),
        step=dict(ms_per_step=ms, clips_per_s_best={k: round(B * 1e3 / min(v), 1) for k, v in ms.items()},
                  mixup_over_plain_best=round(min(ms["mixup"]) / min(ms["plain"]), 4), steps=args.steps, warmup=args.warmup,
                  order="A/B alternated per round: plain, mixup", draws=kinds, cuda_graph=eng.use_graph,
                  mixup_settings=dict(mixup_alpha=0.8, cutmix_alpha=1.0, label_smoothing=0.1, prob=1.0, switch_prob=0.5)))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
