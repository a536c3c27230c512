#!/usr/bin/env python
"""Stage-1 step with a CLIP ViT-L/14 teacher: clips/s of the whole graph-replayed step, one JSON line.

    python tools/bench_clip_l14.py [--batch 32] [--steps 20] [--warmup 5]

Workload: ViT-B/16 student (8x224^2, tubelet 1, drop_path 0.1, clip_output_dim 768) distilled from clip_l14 built at
input_resolution 196 and returning its last six layers; the teacher's copy of every 224-px clip is resized to 196 px on the
device (ub_resize_patchify), so both sides see 14x14 patches per frame.  80 % mask, synthetic fp32 clips (bench.host_batches).

Besides the step rate the line carries
  f_alg_gflop_per_clip  SURVEY.md §8(d)'s rule applied to these shapes (see f_alg below)
  teacher_forward       resize + teacher tower + mask selection + target projection, CUDA events over an untimed eager pass
  resize_patchify       the kernel alone on the benchmark batch, L2 flushed (256 MB write) before every pass, GB/s over the bytes
                        the algorithm must move (fp32 clip read once, padded bf16 rows written once)
  gpu                   card name, power limit and SM clocks read in the same run
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import ClockSampler, DROP_PATH, NOMINAL_BF16_TFLOPS, host_batches, measured_peaks  # noqa: E402

FRAMES, SIDE, TEACHER_SIDE, PATCH_T, MASK_RATIO = 8, 224, 196, 14, 0.8
RETURN_LAYERS = [18, 19, 20, 21, 22, 23]


def blk(S, D):
    """Forward FLOPs of one pre-LN transformer block (MLP ratio 4) on a sequence of S tokens: QKV, scores, P.V, proj, MLP."""
    return 24 * S * D * D + 4 * S * S * D


def f_alg():
    """GFLOP per clip, SURVEY.md §8(d): no padding, no recompute; the teacher's tower on every token, its projection and the
    student on the visible ones."""
    P = (TEACHER_SIDE // PATCH_T) ** 2                                      # 196 patches per frame
    n_vis = P - int(P * MASK_RATIO)                                         # 40 per frame
    Dt, Ds, C = 1024, 768, 768
    teacher_blocks = 24 * FRAMES * blk(P + 1, Dt)
    teacher_embed = 2 * FRAMES * P * (3 * PATCH_T * PATCH_T) * Dt
    teacher_proj = len(RETURN_LAYERS) * FRAMES * n_vis * 2 * Dt * C
    Nv = FRAMES * n_vis                                                     # 320 visible tokens per clip
    s_embed = 2 * Nv * (3 * 16 * 16) * Ds
    s_fwd = 12 * blk(Nv, Ds) + s_embed + len(RETURN_LAYERS) * 2 * Nv * Ds * C
    s_bwd = 2 * s_fwd - s_embed                                             # no input gradient for the patch embedding
    parts = dict(teacher=teacher_blocks + teacher_embed + teacher_proj, teacher_blocks=teacher_blocks, teacher_embed=teacher_embed,
                 teacher_proj_visible=teacher_proj, student_fwd=s_fwd, student_bwd=s_bwd)
    parts = {k: v / 1e9 for k, v in parts.items()}
    parts["total"] = parts["teacher"] + parts["student_fwd"] + parts["student_bwd"]
    return parts


def gpu_info(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        name, power, sm, sm_max = [x.strip() for x in out.split(",")]
        return dict(name=name, power_limit=power, sm_clock=sm, sm_clock_max=sm_max)
    except Exception as e:                                                  # the JSON line still says what is missing
        return dict(error=f"nvidia-smi: {type(e).__name__}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    import torch
    from unite_b200 import modeling_adaptation  # noqa: F401  (registers the factories)
    from unite_b200 import ops
    from unite_b200.clip import clip_l14
    from unite_b200.engine import Stage1Engine
    from unite_b200.registry import create_model
    if not torch.cuda.is_available():
        raise SystemExit("tools/bench_clip_l14.py needs a CUDA device (there is no CPU path)")
    dev = torch.device("cuda", 0)
    B = args.batch
    torch.manual_seed(0)
    student = create_model("adaptation_umt_base_patch16_224", pretrained=False, drop_path_rate=DROP_PATH, drop_block_rate=None,
                           use_learnable_pos_emb=False, use_checkpoint=False, checkpoint_num=0, clip_decoder_embed_dim=768,
                           clip_output_dim=768, clip_norm_type="l2", num_frames=FRAMES, tubelet_size=1,
                           clip_return_layers=[6, 7, 8, 9, 10, 11], clip_student_return_interval=1, use_cls_token=False)
    teacher = clip_l14(pretrained=False, clip_norm_type="l2", input_resolution=TEACHER_SIDE, return_attn=True, kernel_size=1,
                       clip_return_layers=RETURN_LAYERS)
    student, teacher = student.to(dev).train(), teacher.to(dev).eval()
    eng = Stage1Engine(student, teacher, mask_ratio=MASK_RATIO, lr=1.5e-4 * B / 256, weight_decay=0.05, use_graph=True)
    batches = [(v.to(dev), q.to(dev)) for v, q in host_batches(B, 0)]

    # warm-up: 2 eager steps, then one graph capture per resident batch, all before the timed region
    n_warm = max(args.warmup, 2 + len(batches))
    for i in range(n_warm):
        eng.step(*batches[i % 2])
    torch.cuda.synchronize()
    sampler = ClockSampler(0).start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = eng.step(*batches[i % 2])
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_step = e0.elapsed_time(e1) / args.steps
    clips_s = B / (ms_step * 1e-3)
    F = f_alg()

    # ---- teacher forward alone (untimed above): what the step spends before the student starts -----------------------------
    videos, q = batches[0]
    P = (TEACHER_SIDE // PATCH_T) ** 2
    n_vis = eng.n_visible(P)

    def teacher_forward():
        sel = {}

        def select(attn):
            frames = attn.shape[0]
            sel["mask"] = torch.empty(1, frames * P, device=dev, dtype=torch.uint8)
            sel["vis"] = torch.empty(1, B, FRAMES * n_vis, device=dev, dtype=torch.int32)
            sel["rows"] = torch.empty(1, B, FRAMES * n_vis, device=dev, dtype=torch.int32)
            ops.mask_select(attn, q, sel["mask"], sel["vis"], sel["rows"], FRAMES, 1, n_vis)
            return sel["rows"].view(-1)

        layers, _, _ = teacher.forward_features(videos, None, select=select, resolution=TEACHER_SIDE)
        return teacher.project_rows(layers, sel["rows"].view(-1))

    teacher_forward()
    torch.cuda.synchronize()
    reps = 5
    torch.cuda._sleep(int(0.2 * 1.9e9))            # the host queues the eager passes while the device spins
    e0.record()
    for _ in range(reps):
        teacher_forward()
    e1.record()
    torch.cuda.synchronize()
    ms_teacher = e0.elapsed_time(e1) / reps

    # ---- resize + patchify kernel, L2 flushed before every pass ----------------------------------------------------------
    rows = torch.empty(B * FRAMES * P, teacher.k_pad, device=dev, dtype=torch.bfloat16)
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    times = []
    for _ in range(21):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        ops.resize_patchify(videos, rows, TEACHER_SIDE, PATCH_T, 1)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    times.sort()
    us_rp = times[len(times) // 2] * 1e3
    bytes_rp = videos.numel() * 4 + rows.numel() * 2

    peaks = measured_peaks()
    line = dict(
        metric="clips/sec (stage-1 step, ViT-B/16 student 8x224^2, CLIP ViT-L/14 teacher at 196 px)", value=round(clips_s, 2),
        unit="clips/s", ms_per_step=round(ms_step, 3), batch=B, steps=args.steps, warmup_steps_run=n_warm, cuda_graph=True,
        graphs_captured=len(eng._graphs), drop_path=DROP_PATH, loss=round(loss.item(), 5),
        f_alg_gflop_per_clip={k: round(v, 1) for k, v in F.items()},
        mfu=dict(tflops=round(clips_s * F["total"] / 1e3, 1), of_nominal_2250=round(clips_s * F["total"] / 1e3 / NOMINAL_BF16_TFLOPS, 4)),
        teacher_forward=dict(ms=round(ms_teacher, 3), share_of_step=round(ms_teacher / ms_step, 4),
                             tflops=round(B * F["teacher"] / (ms_teacher * 1e-3) / 1e3, 1),
                             note="eager pass (resize + 24 blocks + mask selection + projection of the visible rows), CUDA events"),
        resize_patchify=dict(us=round(us_rp, 1), alg_bytes=bytes_rp, gb_s=round(bytes_rp / (us_rp * 1e-6) / 1e9, 1),
                             of_hbm_peak=round(bytes_rp / (us_rp * 1e-6) / 1e9 / peaks["hbm"], 4), hbm_peak_gb_s=peaks["hbm"],
                             hbm_peak_source=peaks["source"], passes=len(times), l2="flushed before each pass (256 MB write)"),
        clocks=clocks, gpu=gpu_info(0))
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
