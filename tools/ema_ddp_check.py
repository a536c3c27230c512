#!/usr/bin/env python
"""Stage-2 model EMA on several GPUs: every rank trains the replicated model on its own batches through train_one_epoch (NCCL
gradient all-reduce, CUDA-graph step) and updates its own EMA; afterwards the EMA arenas (and the weights) must be bitwise
identical across ranks, with no communication for the EMA.

    python -m torch.distributed.run --nproc-per-node=N tools/ema_ddp_check.py [--steps 4]
Prints "EMA PARITY OK" on rank 0 and exits 0 when they are.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=4)
    args = ap.parse_args()
    from functools import partial

    import torch
    import torch.distributed as dist
    import torch.nn as nn
    from tests.util import load_golden, oracle_cfgs, seeded_states
    from unite_b200.ddp import DataParallel, init_distributed_from_env
    from unite_b200.ema import ModelEma
    from unite_b200.engine_for_finetuning import train_one_epoch
    from unite_b200.modeling_finetune import VisionTransformer
    from unite_b200.optim_factory import create_optimizer
    rank, _, world = init_distributed_from_env()
    fix = load_golden("tiny_stage12.pt")
    scfg, _ = oracle_cfgs(fix)
    _, _, vsd = seeded_states(fix)
    vit = VisionTransformer(img_size=scfg.img_size, patch_size=scfg.patch_size, embed_dim=scfg.embed_dim, depth=scfg.depth,
                            num_heads=scfg.num_heads, mlp_ratio=4, qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6),
                            num_classes=scfg.num_classes, all_frames=scfg.num_frames, tubelet_size=scfg.tubelet_size, init_scale=0.001,
                            drop_path_rate=0.1)
    vit.load_state_dict(vsd, strict=True)
    vit = vit.cuda()
    ema = ModelEma(vit, decay=0.99)                               # built before the data-parallel wrapper, as VideoMAE does
    model = DataParallel(vit)

    class A:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-3, 0.05, (0.9, 0.999), 1e-8
    opt = create_optimizer(A, model)
    g = torch.Generator().manual_seed(100 + rank)                 # every rank its own batches
    batches = [(torch.randn(4, 3, scfg.num_frames, scfg.img_size, scfg.img_size, generator=g),
                torch.randint(0, scfg.num_classes, (4,), generator=g)) for _ in range(args.steps)]
    train_one_epoch(model, None, batches, opt, "cuda", 0, None, model_ema=ema)
    torch.cuda.synchronize()
    ok = True
    for name, t in (("weights", vit.core().arena.params), ("ema", ema.ema.core().arena.params), ("ema shadow", ema.ema.core().arena.w16)):
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        same = all(torch.equal(parts[0].view(torch.int16), q.view(torch.int16)) for q in parts)
        ok &= same
        if rank == 0:
            print(f"{name}: {'identical' if same else 'DIFFERENT'} on {world} ranks")
    moved = not torch.equal(ema.ema.core().arena.params, vit.core().arena.params)
    ok &= moved
    if rank == 0:
        print("EMA PARITY OK" if ok else f"EMA PARITY FAILED (EMA differs from the weights: {moved})")
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
