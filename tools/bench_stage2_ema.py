#!/usr/bin/env python
"""Stage-2 model EMA: the fused update kernel alone and the whole graph-replayed step with and without it, one JSON line.

    python tools/bench_stage2_ema.py [--batch 32] [--steps 20] [--warmup 5] [--rounds 3] [--launches 100]

  kernel                ub_ema_update over the fp32 parameter arena of the ViT-B/16 and the ViT-L/16 stage-2 classifier (88 M and
                        304 M parameters: 1.2 and 4.3 GB of traffic per launch, far above the 126 MB L2, so every launch reads and
                        writes HBM).  CUDA events over `launches` back-to-back launches, `rounds` times.  Bytes are what the update
                        must move: p and ema read, ema and its bf16 shadow written, 14 B per parameter; TB/s and the share of the
                        B200's 7.7 TB/s data-sheet HBM bandwidth.
  step                  the bench.py --workload stage2 step (ViT-B/16, all 1568 tokens, drop_path 0.1, layer-decay AdamW, CUDA
                        graph) without and with ModelEma(decay=0.9999), alternated A/B/A/B/... on one engine (one graph each) and
                        one box; ms per step of each segment.
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
BYTES_PER_PARAM = 14


def _stage2_model(name, C, T, dev):
    import bench
    from unite_b200.registry import create_model
    return create_model(name, pretrained=False, num_classes=C, all_frames=T, tubelet_size=1, drop_rate=0.0, drop_path_rate=bench.DROP_PATH,
                        attn_drop_rate=0.0, drop_block_rate=None, use_mean_pooling=True, init_scale=0.001, fc_drop_rate=0.0,
                        use_checkpoint=False, checkpoint_num=0).to(dev).train()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--launches", type=int, default=100)
    args = ap.parse_args()
    import torch
    from unite_b200 import modeling_finetune  # noqa: F401  (registers the factories)
    from unite_b200 import ops
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    if not torch.cuda.is_available():
        raise SystemExit("bench_stage2_ema: no CUDA device")
    dev = torch.device("cuda", 0)
    B, T, S, C = args.batch, 8, 224, 12
    torch.manual_seed(0)

    # ---- the kernel alone ----------------------------------------------------------------------------------------------------
    kern = {}
    for label, name in (("vit_b16", "vit_base_patch16_224"), ("vit_l16", "vit_large_patch16_224")):
        m = _stage2_model(name, C, T, dev)
        n = m.core().arena.numel
        del m
        torch.cuda.empty_cache()
        ema = torch.randn(n, device=dev)
        p = torch.randn(n, device=dev)
        w16 = torch.empty(n, device=dev, dtype=torch.bfloat16)
        for _ in range(5):
            ops.ema_update(ema, w16, p, 0.9999)
        us = []
        for _ in range(args.rounds):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.launches):
                ops.ema_update(ema, w16, p, 0.9999)
            e1.record()
            torch.cuda.synchronize()
            us.append(e0.elapsed_time(e1) * 1e3 / args.launches)
        best = min(us)
        bytes_moved = n * BYTES_PER_PARAM
        kern[label] = dict(arena_elements=n, bytes_per_launch=bytes_moved, us_per_launch=[round(t, 2) for t in us],
                           tb_s_best=round(bytes_moved / (best * 1e-6) / 1e12, 3),
                           hbm_fraction_best=round(bytes_moved / (best * 1e-6) / 1e12 / HBM_TBS, 3))
        del ema, p, w16
        torch.cuda.empty_cache()

    # ---- the whole step, without and with the EMA, alternated on one engine -----------------------------------------------------------
    torch.manual_seed(0)
    model = _stage2_model("vit_base_patch16_224", C, T, dev)
    L = model.get_num_layers()
    asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class A:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(A, model, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale)
    g = torch.Generator().manual_seed(1000)
    batches = [(torch.randn(B, 3, T, S, S, generator=g).to(dev), torch.randint(0, C, (B,), generator=g).to(dev)) for _ in range(2)]
    model_ema = ModelEma(model, decay=0.9999)
    eng = Stage2Engine(model, opt, use_graph=os.environ.get("UB_NO_GRAPH", "0") != "1", model_ema=model_ema)
    with_ema = eng.ema
    i = [0]

    def run(ema):
        eng.ema = ema
        v, y = batches[i[0] % 2]
        i[0] += 1
        return eng.step(v, y)

    ms = {"plain": [], "ema": []}
    for _ in range(args.rounds):
        for name, ema in (("plain", None), ("ema", with_ema)):
            for _ in range(args.warmup):
                run(ema)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                loss = run(ema)
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(round(e0.elapsed_time(e1) / args.steps, 3))
            assert torch.isfinite(loss).all()
    out = dict(
        tool="bench_stage2_ema", batch=B, clip=[3, T, S, S], gpu=gpu_info(0), kernel=dict(launches=args.launches, rounds=args.rounds, **kern),
        step=dict(ms_per_step=ms, clips_per_s_best={k: round(B * 1e3 / min(v), 1) for k, v in ms.items()},
                  ema_over_plain_best=round(min(ms["ema"]) / min(ms["plain"]), 4),
                  ema_minus_plain_best_ms=round(min(ms["ema"]) - min(ms["plain"]), 3), steps=args.steps, warmup=args.warmup,
                  order="A/B alternated per round: plain, ema", graphs=len(eng.graphs._graphs), cuda_graph=eng.use_graph, decay=0.9999))
    print(json.dumps(out))


if __name__ == "__main__":
    main()
