#!/usr/bin/env python
"""The stage-2 training crop, flip and random erasing on the device (ub_patchify_aug_u8, augment.SpatialAugment): one JSON line
(written to --out as well).

    python tools/bench_stage2_aug.py [--batch 32] [--launches 200] [--rounds 3] [--steps 10] [--host-clips 16] [--out profiles/x.json]

  kernel  B = 32, T = 8 decoded 256x320 uint8 frames -> 224^2, SpatialAugment() draws (remode 'pixel', device noise), tubelet 1, with
          and without a mixup draw, against ub_patchify_u8 / ub_patchify_mix_u8 of 224^2 frames.  CUDA events over `launches`
          back-to-back launches, the kernels alternated `rounds` times.  Bytes: the bf16 rows written once plus the input bytes the
          clips' crop boxes cover (read once; `bytes_frames` counts the whole frames instead), TB/s and the share of the B200's 7.7 TB/s
          data-sheet HBM bandwidth.  The inputs (63 MB of frames) fit the 126 MB L2, so repeated launches read them from there.
  step    Stage2Engine.step (ViT-B/16, 1568 tokens, drop_path 0.1, layer-decay AdamW, CUDA-graph replay) on device-resident batches:
          224^2 uint8 frames without augmentation against 256x320 frames with SpatialAugment, fresh draws every step, alternated per
          round on one engine.
  host    (a CPU measurement, on this machine's host cores) the reference loader's float work per clip after RandAugment: ToTensor +
          tensor_normalize, random_resized_crop, horizontal_flip, RandomErasing('pixel') on [T,C,H,W] (tests/augment_ref.py, torch
          with one intra-op thread, as a loader worker runs), against the uint8 hand-off's host work per clip (SpatialAugment.draw).
  gpu     card name, power limit and SM clocks, read in the same run
"""
import argparse
import json
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from bench_clip_l14 import gpu_info  # noqa: E402

HBM_TBS = 7.7


def kernel_times(args, dev):
    import numpy as np
    import torch
    from unite_b200 import mixup as M
    from unite_b200 import ops
    from unite_b200.augment import AugBuffer, SpatialAugment
    B, T, H, W, S = args.batch, 8, 256, 320, 224
    g = torch.Generator().manual_seed(1000)
    fr = torch.randint(0, 256, (B, T, H, W, 3), generator=g, dtype=torch.uint8).to(dev)
    fr224 = torch.randint(0, 256, (B, T, S, S, 3), generator=g, dtype=torch.uint8).to(dev)
    rows = torch.empty(B * T * (S // 16) ** 2, 3 * 256, device=dev, dtype=torch.bfloat16)
    aug = SpatialAugment()
    random.seed(0)
    np.random.seed(0)
    d = aug.draw(fr.shape)
    buf = AugBuffer(aug, B, dev)
    buf.upload(d)
    mix = M.MixBuffer(dev)
    mix.upload(M.MixDraw(True, 0.4217, False, ((0, 0), (0, 0), (0, 0)), 0.4217).packed(0.1, 12))
    p = d.params
    crop_bytes = int((p[:, 2].astype(np.int64) * p[:, 3]).sum()) * T * 3
    out_bytes = rows.numel() * 2
    aug_call = lambda m: ops.patchify_aug_u8(fr, rows, buf.draw, S, 1, aug.erase_mode, mix=m, rng=buf.rng, seed=aug.seed)
    kernels = dict(patchify_aug_u8=(lambda: aug_call(None), crop_bytes, fr.numel()),
                   patchify_aug_u8_mixup=(lambda: aug_call(mix.clip), crop_bytes, fr.numel()),
                   patchify_u8_224=(lambda: ops.patchify_u8(fr224, rows, 1), fr224.numel(), fr224.numel()),
                   patchify_mix_u8_224_mixup=(lambda: ops.patchify_mix_u8(fr224, rows, mix.clip, 1), fr224.numel(), fr224.numel()))
    us = {k: [] for k in kernels}
    for fn, _, _ in kernels.values():
        for _ in range(10):
            fn()
    for _ in range(args.rounds):
        for name, (fn, _, _) in kernels.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.launches):
                fn()
            e1.record()
            torch.cuda.synchronize()
            us[name].append(e0.elapsed_time(e1) * 1e3 / args.launches)
    out = {}
    for name, (_, in_bytes, frame_bytes) in kernels.items():
        best = min(us[name])
        moved = in_bytes + out_bytes
        out[name] = dict(us_per_launch=[round(t, 2) for t in us[name]], bytes=moved, bytes_frames=frame_bytes + out_bytes,
                         tb_s_best=round(moved / (best * 1e-6) / 1e12, 3), hbm_fraction_best=round(moved / (best * 1e-6) / 1e12 / HBM_TBS, 3))
    erased = int(p[:, 5].sum())
    return dict(batch=B, frames=[T, H, W], crop=S, tubelet=1, launches=args.launches, rounds=args.rounds, remode=aug.remode,
                clips_erased=erased, crop_area_mean=round(float((p[:, 2] * p[:, 3]).mean()) / (H * W), 3),
                l2="the 63 MB of 256x320 frames and the 39 MB of 224^2 frames fit the 126 MB L2", **out)


def step_times(args, dev):
    import numpy as np
    import torch
    import bench
    from unite_b200 import modeling_finetune  # noqa: F401  (registers the factories)
    from unite_b200.augment import SpatialAugment
    from unite_b200.engine_for_finetuning import Stage2Engine
    from unite_b200.optim_factory import LayerDecayValueAssigner, create_optimizer
    from unite_b200.registry import create_model
    B, C = args.batch, 12
    torch.manual_seed(0)
    model = create_model("vit_base_patch16_224", pretrained=False, num_classes=C, all_frames=8, tubelet_size=1, drop_rate=0.0,
                         drop_path_rate=bench.DROP_PATH, attn_drop_rate=0.0, drop_block_rate=None, use_mean_pooling=True,
                         init_scale=0.001, fc_drop_rate=0.0, use_checkpoint=False, checkpoint_num=0).to(dev).train()
    L = model.get_num_layers()
    asg = LayerDecayValueAssigner([0.65 ** (L + 1 - i) for i in range(L + 2)])

    class A:
        opt, lr, weight_decay, opt_betas, opt_eps = "adamw", 1e-4, 0.05, (0.9, 0.999), 1e-8
    eng = Stage2Engine(model, create_optimizer(A, model, get_num_layer=asg.get_layer_id, get_layer_scale=asg.get_scale), use_graph=True)
    g = torch.Generator().manual_seed(7)
    f224 = torch.randint(0, 256, (B, 8, 224, 224, 3), generator=g, dtype=torch.uint8).to(dev)
    f320 = torch.randint(0, 256, (B, 8, 256, 320, 3), generator=g, dtype=torch.uint8).to(dev)
    y = torch.randint(0, C, (B,), generator=g).to(dev)
    aug = SpatialAugment()
    random.seed(0)
    np.random.seed(0)
    legs = {"uint8_224_plain": lambda: eng.step(f224, y), "uint8_256x320_spatial_aug": lambda: eng.step(f320, y, aug=aug.draw(f320.shape))}
    for fn in legs.values():
        for _ in range(4):
            fn()
    ms = {k: [] for k in legs}
    for _ in range(args.rounds):
        for name, fn in legs.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(round(e0.elapsed_time(e1) / args.steps, 3))
    out = {k: dict(ms_per_step=v, clips_per_s_best=round(B / (min(v) * 1e-3), 1)) for k, v in ms.items()}
    out["aug_over_plain_best"] = round(min(ms["uint8_256x320_spatial_aug"]) / min(ms["uint8_224_plain"]), 4)
    return dict(model="vit_base_patch16_224, 8 frames, tubelet 1, drop_path %.2f" % bench.DROP_PATH, steps=args.steps,
                rounds=args.rounds, note="device-resident batches; the aug leg's host draw (SpatialAugment.draw) and upload are inside "
                "the timed loop", **out)


def host_cost(args):
    import numpy as np
    import torch
    from tests import augment_ref as R
    from unite_b200.augment import SpatialAugment
    torch.set_num_threads(1)
    T, H, W = 8, 256, 320
    g = torch.Generator().manual_seed(3)
    clips = [torch.randint(0, 256, (T, H, W, 3), generator=g, dtype=torch.uint8) for _ in range(4)]
    mean, std = torch.tensor([0.485, 0.456, 0.406]), torch.tensor([0.229, 0.224, 0.225])
    random.seed(0)
    np.random.seed(0)

    def reference(u8):
        x = u8.float() / 255.0                                                      # ToTensor
        x = (x - mean) / std                                                        # tensor_normalize
        x = x.permute(3, 0, 1, 2)                                                   # T H W C -> C T H W
        return R.loader_tail(x, 224, reprob=1.0, remode="pixel")

    aug = SpatialAugment()
    for u8 in clips:
        reference(u8)
    t0 = time.perf_counter()
    for k in range(args.host_clips):
        reference(clips[k % 4])
    ref_ms = (time.perf_counter() - t0) * 1e3 / args.host_clips
    t0 = time.perf_counter()
    for _ in range(args.host_clips * 20):
        aug.draw((1, T, H, W, 3))
    draw_ms = (time.perf_counter() - t0) * 1e3 / (args.host_clips * 20)
    return dict(measured_on="host CPU (not the GPU)", cpu_count=os.cpu_count(), torch_threads=1, clip=[T, H, W, 3], crop=224,
                reference_float_ms_per_clip=round(ref_ms, 3), uint8_handoff_ms_per_clip=round(draw_ms, 4),
                reference_ops="ToTensor + tensor_normalize + random_resized_crop (bilinear) + horizontal_flip + RandomErasing(pixel, "
                "reprob=1) on [T,C,H,W]", uint8_handoff_ops="SpatialAugment.draw of one clip (the frames are handed over as they are)",
                clips_timed=args.host_clips)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--host-clips", type=int, default=16)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_stage2_aug: no CUDA device")
    dev = torch.device("cuda", 0)
    out = dict(tool="bench_stage2_aug", gpu=gpu_info(0), kernel=kernel_times(args, dev), step=step_times(args, dev), host=host_cost(args),
               n_gpus_end_to_end="not measured (one GPU)")
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
