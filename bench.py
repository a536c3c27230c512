#!/usr/bin/env python
"""Headline benchmark: clips/s of one full stage-1 UMT distillation step (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch 32] [--workload stage1|stage2|stage3|vitl]
    (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" = teacher forward + attention-guided mask + DropPath draw + student forward/backward + gradient exchange + AdamW on one
batch of synthetic 8x224^2 clips (ViT-B/16 student with the shipped drop_path 0.1, CLIP ViT-B/16 teacher, 80 % mask, per-GPU batch
32, bf16 operands / fp32 accumulate).  Prints ONE JSON line (rank 0).  Keys follow the driver contract; in addition:
  roofline            tensor-bound GEMM kernel family: algorithmic FLOPs / CUDA-event time of every GEMM launch of one
                      instrumented step (events on the launching stream), against the measured sustained bf16 peak
  cpu_baseline        the reference's model modules (baseline/_ref, kind "reference"; else the oracle port) on this box's host
                      cores, fp32, bounded sample (B=2)
  gpu_eager_baseline  the SAME unmodified reference modules, eager, torch.autocast(bf16), fused torch AdamW, B=32, on this GPU,
                      in a separate process (baseline/reference_runner.py) — the bar the fused path has to beat
  e2e                 the same metric through the public train_one_epoch() API with pinned-host inputs (H2D inside)
  parity_check        first eager step at the benchmarked shapes against a committed oracle fixture (tests/golden/
                      bench_b32_check.json): the line is NOT printed when it disagrees
  ddp_parity (N > 1)  one fused NVLink optimizer step against NCCL all-reduce + ub_adamw_seg on the same gradients
--impl reference times the reference's own CPU implementation (see cpu_baseline) with the optimizer step included.
--workload stage2|stage3|vitl: the other BASELINE.json configs as their own lines (not the driver's headline).
--dump-outputs DIR: after the timed steps, the last step's results as DIR/<name>.npy (see dump_outputs); the inputs depend only on
the arguments, so two builds run with the same arguments can be compared array by array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md §8(d) / BASELINE.md §4: algorithmic GFLOP per clip (no padding / recompute)
F_ALG = dict(stage1=462.2, stage2=1074.7, stage3=2229.0, vitl=902.4)
NOMINAL_BF16_TFLOPS = 2250.0
METRIC = "clips/sec (ViT-B/16 8x224^2 stage-1 step)"
DROP_PATH = 0.1                        # configs/stage1_config.yaml:37 (and stage 2 / 3)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16=d.get("bf16_tflops_sustained", 1341.6), bf16_burst=d.get("bf16_tflops", 1640.4), hbm=d.get("hbm_gbs", 6529.1),
                    source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(bf16=1400.0, bf16_burst=1590.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


def build_models(seed=0, drop_path=DROP_PATH, large=False):
    import torch
    from unite_b200.registry import create_model
    from unite_b200 import modeling_adaptation  # noqa: F401  (registers the factories)
    from unite_b200.clip import clip_b16
    torch.manual_seed(seed)
    # kwargs as run_stage1.py:275-291 passes them with configs/stage1_config.yaml (drop_path: 0.1); BASELINE configs[4] swaps in the
    # large student at 16 frames / tubelet 2 with the teacher's kernel_size 2 (SURVEY.md §8(d))
    student = create_model("adaptation_umt_large_patch16_224" if large else "adaptation_umt_base_patch16_224", pretrained=False,
                           drop_path_rate=drop_path, drop_block_rate=None, use_learnable_pos_emb=False, use_checkpoint=False,
                           checkpoint_num=0, clip_decoder_embed_dim=1024 if large else 768, clip_output_dim=512, clip_norm_type="l2",
                           num_frames=16 if large else 8, tubelet_size=2 if large else 1, clip_return_layers=[6, 7, 8, 9, 10, 11],
                           clip_student_return_interval=1, use_cls_token=False)
    teacher = clip_b16(pretrained=False, clip_norm_type="l2", input_resolution=224, return_attn=True, kernel_size=2 if large else 1,
                       clip_return_layers=[6, 7, 8, 9, 10, 11], clip_return_interval=1)
    return student, teacher


def host_batches(B, rank, n=2, frames=8, tokens_per_frame=1):
    """Seeded on the HOST (so the oracle fixture of tests/golden/bench_b32_check.json sees the same clips), then uploaded."""
    import torch
    g = torch.Generator().manual_seed(1000 + rank)
    return [(torch.randn(B, 3, frames, 224, 224, generator=g), torch.empty(B * frames // tokens_per_frame, 196).exponential_(1, generator=g))
            for _ in range(n)]


# ---------------------------------------------------------------------------------------------------------------------------
# reference arms
# ---------------------------------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, batch=2, seed=0, budget_s=150.0):
    """The reference's stage-1 step on the host cores, fp32, all threads, optimizer included, B=`batch` clips per step.
    baseline/_ref present (the unmodified src/models of the reference, copied by build()): kind 'reference'; else the oracle
    port seeded from oracle/weights.py: kind 'port'.  Neither imports unite_b200."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    from baseline import reference_runner as R
    asked = (steps, warmup)
    reason = None
    if R.available():
        t0 = time.perf_counter()
        R.run_stage1("cpu", batch, 1, 0, seed=seed, drop_path=DROP_PATH, world_batch=32)          # probe: also pages the modules in
        probe = time.perf_counter() - t0
        per_step = max(0.05, probe * 0.6)                                     # the probe includes model construction
        fit = max(1, int(budget_s / per_step))
        if steps + warmup > fit:
            steps, warmup = max(1, min(steps, fit - 1)), max(0, min(warmup, 1))
            reason = f"clamped from steps={asked[0]} warmup={asked[1]}: {per_step:.1f} s per CPU step against a {budget_s:.0f} s budget"
        r = R.run_stage1("cpu", batch, steps, warmup, seed=seed, drop_path=DROP_PATH, world_batch=32)
        kind, what = "reference", ("baseline/_ref: unmodified reference src/models (clip.py, modeling_adaptation.py, modeling_finetune.py) driven by "
                                   "the restated step of run_stage1.py:360-458 + torch.optim.AdamW")
        value, ms, loss = r["value"], r["ms_per_step"], r["loss"]
    else:
        from oracle import unite_oracle as O
        from oracle.weights import seeded_state
        scfg, tcfg = O.StudentCfg(), O.TeacherCfg()
        shapes = json.load(open(os.path.join(ROOT, "tests", "golden", "vitb16_shapes.json")))
        ssd, tsd = seeded_state(shapes["student"], 0), seeded_state(shapes["teacher"], 1)
        g = torch.Generator().manual_seed(seed)
        videos = torch.randn(batch, 3, 8, 224, 224, generator=g)
        q = torch.empty(batch * 8, 196).exponential_(1, generator=g)
        params = [v.clone().requires_grad_() for v in ssd.values()]
        opt = torch.optim.AdamW(params, lr=1.5e-4 * 32 / 256, betas=(0.9, 0.95), weight_decay=0.05)

        def one():
            r_ = O.stage1_step(ssd, tsd, videos, q, scfg, tcfg, mask_ratio=0.8)
            for p_, k_ in zip(params, ssd):
                p_.grad = r_["grads"][k_]
            opt.step()
            return r_
        t0 = time.perf_counter(); one(); per_step = time.perf_counter() - t0
        fit = max(1, int(budget_s / per_step))
        if steps + warmup > fit:
            steps, warmup = max(1, min(steps, fit - 1)), max(0, min(warmup, 1))
            reason = f"clamped from steps={asked[0]} warmup={asked[1]}: {per_step:.1f} s per CPU step against a {budget_s:.0f} s budget"
        for _ in range(warmup):
            one()
        t0 = time.perf_counter()
        for _ in range(steps):
            r_ = one()
        dt = (time.perf_counter() - t0) / steps
        kind, what = "port", "oracle/unite_oracle.stage1_step (fp32 restatement) + torch.optim.AdamW, weights from oracle/weights.py"
        value, ms, loss = batch / dt, dt * 1e3, float(r_["loss"])
    out = dict(value=value, unit="clips/s", cores=cores, kind=kind, ms_per_step=ms, loss=loss, steps=steps, warmup=warmup,
               sample=f"{what}; teacher fwd + mask + student fwd/bwd + grad-norm + AdamW, fp32 torch CPU, {cores} threads, B={batch} clips per "
                      f"step cut from the B=32 workload (clips are independent: clips/s does not depend on the batch), {warmup} warm-up + "
                      f"{steps} timed steps")
    if reason:
        out["reason"] = reason
    return out


def gpu_eager_reference(batch, steps, warmup, local_gpu=0):
    """The unmodified reference modules, eager, bf16 autocast, on this GPU — in a SEPARATE process (own CUDA context, none of this
    repo's kernels loaded), with its own clocks sample."""
    from baseline import reference_runner as R
    if not R.available():
        return dict(unavailable="baseline/_ref missing (build() copies it from /root/reference in the build container)")
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=vis.split(",")[local_gpu] if vis else str(local_gpu))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    sampler = ClockSampler(local_gpu).start()
    try:
        r = subprocess.run([sys.executable, "-m", "baseline.reference_runner", "--device", "cuda", "--batch", str(batch), "--steps", str(steps),
                            "--warmup", str(warmup), "--drop-path", str(DROP_PATH)], capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    finally:
        clocks = sampler.stop()
    if r.returncode != 0:
        return dict(unavailable=f"reference_runner failed: {(r.stderr or r.stdout)[-300:]}")
    d = json.loads(r.stdout.strip().splitlines()[-1])
    return dict(value=round(d["value"], 2), unit="clips/s", ms_per_step=round(d["ms_per_step"], 3), steps=steps, warmup=warmup, batch=batch,
                loss=round(d["loss"], 5), peak_mem_gib=round(d["peak_mem_gib"], 2), clocks=clocks, torch=d["torch"],
                what="unmodified reference src/models (baseline/_ref) + the step of run_stage1.py:360-458, eager, torch.autocast('cuda', "
                     "bfloat16), torch.optim.AdamW(fused=True), drop_path 0.1, CUDA events, separate process")


WORKLOAD = ("BASELINE configs[1]: stage-1 UMT masked distillation, ViT-B/16 student (80% CLIP-attn mask, 320 of 1568 tokens, drop_path 0.1) + "
            "frozen CLIP ViT-B/16 teacher, 8x224^2, tubelet 1, K=6 aligned layers, AdamW")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cb = cpu_reference_run(args.steps, args.warmup)
    line = dict(metric=METRIC, value=cb["value"], unit="clips/s", n_gpus=args.gpus, steps=cb["steps"], warmup=cb["warmup"],
                ms_per_step=cb["ms_per_step"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
                impl="reference",
                config=dict(workload=WORKLOAD, per_gpu_batch=args.batch, global_batch=args.batch * args.gpus, parallelism=f"dp{args.gpus}",
                            cpu_sample=cb["sample"], l2_policy="n/a (CPU)"),
                cpu_baseline=dict(kind=cb["kind"], cores=cb["cores"], sample=cb["sample"], value=cb["value"], unit="clips/s"),
                e2e=dict(value=cb["value"], unit="clips/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0, loss=cb["loss"])
    if "reason" in cb:
        line["reason"] = cb["reason"]
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------------
# parity gates inside the bench
# ---------------------------------------------------------------------------------------------------------------------------
def weights_digest(state_dict):
    """sha256 over the first 4096 values of every tensor (sorted by key): identifies the seed-0 initial weights."""
    import hashlib
    import torch
    w = torch.cat([v.detach().float().flatten()[:4096].cpu() for _, v in sorted(state_dict.items())])
    return hashlib.sha256(w.numpy().tobytes()).hexdigest()[:16]



def parity_check_b32(eng, student, batch0, B, compare=True):
    """One eager step (DropPath off, no optimizer) on resident batch 0 against tests/golden/bench_b32_check.json, which
    oracle/make_bench_fixture.py computed with the fp32 oracle for exactly these weights and clips.  Raises on disagreement."""
    import torch
    p = os.path.join(ROOT, "tests", "golden", "bench_b32_check.json")
    if not os.path.exists(p) or B != 32:
        return dict(skipped=f"no fixture for per-GPU batch {B}" if B != 32 else "fixture missing")
    fix = json.load(open(p))
    if compare:
        # The fixture is only comparable when this host's CPU generator reproduced the fixture's weights and clips bit for bit
        # (same torch build: it does on every box of this pool).  If not, the comparison is reported as skipped — a different
        # random draw is not a kernel error; tests/test_optim_groups_cpu.py catches a stale fixture in the build container.
        digest = weights_digest(student.state_dict())
        in_digest = weights_digest({"videos": batch0[0][:1, :, :1, :64, :64].contiguous(), "q": batch0[1][:8]})
        if digest != fix["weights_sha16"] or in_digest != fix.get("inputs_sha16", in_digest):
            return dict(skipped=f"this host's seed-0 weights / clips ({digest}, {in_digest}) are not the fixture's "
                                f"({fix['weights_sha16']}, {fix.get('inputs_sha16')}): nothing to compare against")
    was_training, gs = student.training, eng.grad_sync
    student.eval()
    if eng.nvls is None:
        eng.grad_sync = None           # a local check: no gradient exchange
    eng.optimizer.zero_grad()
    loss = eng.forward_backward(*batch0)
    torch.cuda.synchronize()
    student.train(was_training)
    eng.grad_sync = gs
    if not compare:                    # ranks > 0 hold other clips; they only keep step counts aligned with rank 0
        eng.optimizer.zero_grad()
        return None
    mask = eng.last["mask"].cpu()
    ref_mask = torch.from_numpy(__import__("numpy").unpackbits(__import__("numpy").frombuffer(bytes.fromhex(fix["mask_hex"]), dtype="uint8"))[:mask.numel()]).view_as(mask).bool()
    agree = float((mask == ref_mask).float().mean())
    rel = abs(loss.item() - fix["loss"]) / abs(fix["loss"])
    res = dict(loss=round(loss.item(), 6), oracle_loss=fix["loss"], loss_rel=float(f"{rel:.2e}"), loss_tol=1e-3,
               mask_agreement=round(agree, 5), visible_tokens=int((~mask).sum()), fixture="tests/golden/bench_b32_check.json")
    if rel > 1e-3 or agree < 0.995 or int((~mask).sum()) != fix["visible_tokens"]:
        raise SystemExit(f"bench parity gate FAILED at B=32: {res}")
    eng.optimizer.zero_grad()
    return res


def ddp_parity_check(eng, batch0, world):
    """N > 1, before any optimizer step (every rank still holds identical fp32 masters, zero moments): one fused NVLink step
    (ub_adamw_nvls: push reduce-scatter + AdamW on the shard + shadow all-gather) against NCCL all-reduce + ub_adamw_seg on the
    SAME per-rank gradients.  Returns {max_abs, n_diff, ...}; raises on mismatch."""
    import torch
    import torch.distributed as dist
    from unite_b200 import ops
    a, o = eng.core.arena, eng.optimizer
    eng.optimizer.zero_grad()
    eng.forward_backward(*batch0)
    g_local = a.grads.clone()
    p0, w0 = a.params.clone(), a.w16.clone()
    o.prepare_step(grad_scale=1.0 / world)
    # reference path on clones
    g_sum = g_local.clone()
    dist.all_reduce(g_sum)
    rp, rm, rv, rw = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0), w0.clone()
    gn = torch.zeros(1, device=p0.device)
    ops.adamw_seg(rp, g_sum, rm, rv, rw, o._seg_end4, o._hyper_dev, gn)
    # fused path
    eng.nvls.step_dev()
    torch.cuda.synchronize()
    eng.nvls.check()
    eng.nvls.consolidate()
    torch.cuda.synchronize()
    d = (a.params - rp).abs()
    tol = 2e-5 + 1e-5 * rp.abs()
    n_diff = int((d > tol).sum())
    w_diff = int((a.w16.view(torch.int16) != rw.view(torch.int16)).sum())
    gn_rel = abs(o.gnorm_sq.item() - gn.item()) / max(gn.item(), 1e-30)
    res = dict(max_abs=float(d.max()), n_diff=n_diff, shadow_bf16_diff=w_diff, numel=a.numel, gnorm_sq_rel=float(f"{gn_rel:.2e}"),
               what="ub_adamw_nvls vs NCCL all-reduce + ub_adamw_seg, one step from identical state, same per-rank gradients")
    flag = torch.tensor([n_diff + (1 if w_diff > a.numel * 1e-5 else 0) + (1 if gn_rel > 1e-4 else 0)], device=p0.device)
    dist.all_reduce(flag)
    if flag.item() != 0:
        raise SystemExit(f"bench ddp_parity FAILED: {res}")
    return res


def dump_outputs(out_dir, eng, student, loss, world, rows=8192, per_param=8192):
    """What the last timed step handed its caller, as float32 DIR/<name>.npy (about 35 MB at B = 32), so that two builds can be
    compared output for output: loss, gradient norm, the teacher's attention and the token mask (1 = masked) in full; the student's
    outputs and the teacher's targets at the same seeded sample of `rows` (layer, clip, token position) triples, zero where the
    token is masked; a seeded sample of up to `per_param` elements of every updated student parameter, taken by name in sorted
    order (independent of the parameter arena's layout).
    Rows are addressed by token position, not by place among the visible rows: a token whose visibility flips between two runs
    (attention values within fp noise of each other, a few of 50 176 tokens) then changes its own row only and shifts no other."""
    import numpy as np
    import torch
    eng.optimizer.consolidate()            # collective: with the optimizer sharded by rank, every rank then holds all weights
    if int(os.environ.get("RANK", "0")) != 0:
        return
    rng = np.random.default_rng(0)
    last = eng.last
    out, vis = last["outputs"], last["vis_idx"].long()                     # [K, B, Nv, C]; [B, Nv] ascending token positions
    K, B, Nv, C = out.shape
    N = last["mask"].shape[1]
    pick = lambda n, k: torch.from_numpy(np.sort(rng.choice(n, min(n, k), replace=False))).to(out.device)
    r = pick(K * B * N, rows)
    k, b, n = r // (B * N), r // N % B, r % N
    row = torch.full((B, N), -1, dtype=torch.long, device=out.device).scatter_(1, vis, torch.arange(Nv, device=out.device).expand(B, Nv))
    j = row[b, n]                                                           # -1: token masked
    at = lambda t: torch.where((j >= 0)[:, None], t.reshape(K, B, Nv, C)[k, b, j.clamp(min=0)], 0)
    params = [p.detach().reshape(-1)[pick(p.numel(), per_param)] for _, p in sorted(student.named_parameters())]
    arrays = dict(loss=loss, grad_norm=eng.optimizer.grad_norm(1.0 / world), teacher_attn=last["attn"], mask=last["mask"],
                  student_outputs=at(out), teacher_targets=at(last["targets"]), student_params=torch.cat(params))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=None, help="clips per GPU per step (default 32; stage3: 8 source + 8 target)")
    ap.add_argument("--workload", default="stage1", choices=["stage1", "stage2", "stage3", "vitl"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--profile-out", default=None, help="write the per-op breakdown of one instrumented step here (json)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float32, stage1 workload)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "stage1"):
        ap.error("--dump-outputs needs --impl ours --workload stage1")
    if args.batch is None:
        args.batch = 8 if args.workload == "stage3" else 32
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from unite_b200 import ops
    from unite_b200.ddp import GradSync, DataParallel, init_distributed_from_env

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path in unite_b200); use --impl reference for the CPU baseline")
    # NCCL prints its version banner on stdout when the communicator is created; the driver wants ONE JSON line there
    sys.stdout.flush()
    saved_fd = os.dup(1)
    os.dup2(2, 1)
    try:
        rank, local, world = init_distributed_from_env()
        dev = torch.device("cuda", local)
        if world > 1:
            warm = torch.ones(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved_fd, 1)
        os.close(saved_fd)
    if args.workload != "stage1":
        from tools.bench_workloads import run_workload
        return run_workload(args, rank, local, world, dev, ClockSampler, measured_peaks, F_ALG, NOMINAL_BF16_TFLOPS)

    from unite_b200.engine import Stage1Engine
    from unite_b200.engine_for_pretraining import train_one_epoch, register_engine
    from unite_b200.synthetic import SyntheticStage1Loader
    B = args.batch
    student, teacher = build_models(seed=0)                       # identical weights on every rank (DDP broadcast equivalent)
    student, teacher = student.to(dev).train(), teacher.to(dev).eval()
    model = DataParallel(student)
    model.grad_sync = GradSync() if world > 1 else None
    use_graph = os.environ.get("UB_NO_GRAPH", "0") != "1"
    eng = Stage1Engine(student, teacher, mask_ratio=0.8, lr=1.5e-4 * B * world / 256, weight_decay=0.05, grad_sync=model.grad_sync,
                       use_graph=use_graph)
    register_engine(student, teacher, eng)                  # train_one_epoch (e2e) drives the same engine / optimizer state

    # ---- device-resident inputs (value) ------------------------------------------------------------------------
    dev_batches = [(v.to(dev), q.to(dev)) for v, q in host_batches(B, rank)]

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- parity gates BEFORE anything is timed -------------------------------------------------------------------
    parity = parity_check_b32(eng, student, dev_batches[0], B, compare=(rank == 0))
    ddp_parity = None
    if world > 1 and eng.nvls is not None:
        ddp_parity = ddp_parity_check(eng, dev_batches[0], world)
    sync_all()

    # untimed warm-up: W steps, and at least 2 eager steps + one CUDA-graph capture per resident input buffer (the engine keeps
    # one graph per buffer pair), so that no capture can fall inside the timed region whatever W the caller asked for
    n_warm = max(args.warmup, 2 + len(dev_batches))
    for i in range(n_warm):
        eng.step(*dev_batches[i % 2])
    sync_all()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ops.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = eng.step(*dev_batches[i % 2])
    e1.record()
    sync_all()
    ms = e0.elapsed_time(e1)
    launches = ops.LAUNCHES - launches0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = t.item() / args.steps
    value = world * B / (ms_per_step * 1e-3)
    loss_value = loss.item()
    graphs_captured = len(eng._graphs)
    if args.dump_outputs:                  # before the end-to-end runs below train further and overwrite eng.last
        dump_outputs(args.dump_outputs, eng, student, loss, world)

    # ---- end to end through the public API: pinned host batches, H2D inside the timed region, loss read back ------
    u8_default = world > 1        # N > 1: one host feeds every GPU — decoded uint8 frames (a quarter of the bytes) are the default feed
    loader = SyntheticStage1Loader(B, steps=args.steps, seed=0, rank=rank, n_distinct=2)
    # warm-up through the SAME pinned buffers, staging allocations and graphs as the timed loop: 2 eager steps + one graph
    # capture per slot of the 3-slot staging ring must all happen before the timed region (first-touch effects of a
    # fresh process / box otherwise land inside the timed region: 1516 vs 1704 clips/s measured back to back)
    warm_loader = SyntheticStage1Loader(B, steps=max(6, args.warmup), seed=0, rank=rank, n_distinct=2)
    warm_loader.batches = loader.batches

    class _Args:
        log_freq = 1          # read the loss back every step: the D2H of the step's result is inside the timed region
        use_cuda_graph = use_graph
        clip_loss_data = "mixed"

    def timed_epoch(ld, warm):
        train_one_epoch(model, warm, None, eng.optimizer, dev, 0, None, teacher_model=teacher, mask_type="attention", mask_ratio=0.8, args=_Args)
        sync_all()
        e0.record()
        st = train_one_epoch(model, ld, None, eng.optimizer, dev, 0, None, teacher_model=teacher, mask_type="attention", mask_ratio=0.8, args=_Args)
        e1.record()
        sync_all()
        tt = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return tt.item() / args.steps, st

    f32_ms, stats = timed_epoch(loader, warm_loader)
    h2d_f32 = B * 3 * 8 * 224 * 224 * 4 + B * 8 * 196 * 4
    e2e_f32 = dict(value=round(world * B / (f32_ms * 1e-3), 2), unit="clips/s", ms_per_step=round(f32_ms, 3), h2d_bytes_per_step=h2d_f32,
                   d2h_bytes_per_step=4, input="fp32 clips [B,3,T,H,W] normalised on the host (what the reference's loader hands over)")
    # ---- the same, fed with DECODED uint8 frames [B,T,H,W,3] (what decord / NVDEC deliver; normalised inside the patchify
    #      kernel, SURVEY.md §8 row f2): 4x fewer H2D bytes per step.
    e2e_u8 = None
    if os.environ.get("UB_BENCH_U8", "1") != "0":
        loader8 = SyntheticStage1Loader(B, steps=args.steps, seed=0, rank=rank, n_distinct=2, uint8=True)
        warm8 = SyntheticStage1Loader(B, steps=max(6, args.warmup), seed=0, rank=rank, n_distinct=1, uint8=True)
        warm8.batches = loader8.batches
        u8_ms, stats8 = timed_epoch(loader8, warm8)
        e2e_u8 = dict(value=round(world * B / (u8_ms * 1e-3), 2), unit="clips/s", ms_per_step=round(u8_ms, 3),
                      h2d_bytes_per_step=B * 8 * 224 * 224 * 3 + B * 8 * 196 * 4, d2h_bytes_per_step=4,
                      input="uint8 frames [B,T,H,W,3], ImageNet-normalised on the device inside the patchify kernel")
    api = "unite_b200.engine_for_pretraining.train_one_epoch (reference run_stage1.py:294 signature), pinned host batches"
    if u8_default and e2e_u8 is not None:
        e2e = dict(e2e_u8, api=api)
        e2e_other = ("e2e_fp32_clips", e2e_f32)
    else:
        e2e = dict(e2e_f32, api=api)
        e2e_other = ("e2e_uint8_frames", e2e_u8)

    # ---- one instrumented step: per-op CUDA-event durations on the launching stream (roofline of the GEMM kernel) --
    roof, breakdown = None, None
    if rank == 0:
        ops.PROFILE = []
    eng.use_graph = False              # the instrumented step runs eagerly (events around every launch)
    # Eagerly, the host needs ~10 us per launch and the GPU would idle INSIDE the event pairs waiting for the next command
    # (that inflated the per-kernel times of earlier rounds' JSON by 3-5 us per launch).  A spin kernel ahead of the step lets
    # the host queue the whole step first, so every event pair brackets device execution only.
    torch.cuda._sleep(int(0.15 * 1.9e9))
    eng.step(*dev_batches[0])          # every rank runs it (the step contains the all-reduce); only rank 0 records
    sync_all()
    if rank == 0:
        peaks = measured_peaks()
        prof, ops.PROFILE = ops.PROFILE, None
        by = {}
        shapes = {}
        gemm_flops = gemm_ms = 0.0
        n_gemm = 0
        for name, info, a, b in prof:
            d = a.elapsed_time(b)
            if name == "gemm":
                sh = shapes.setdefault(str(info), [0, 0.0, 2.0 * info[0] * info[1] * info[2]])
                sh[0] += 1
                sh[1] += d
            by.setdefault(name, [0, 0.0])
            by[name][0] += 1
            by[name][1] += d
            if name == "gemm":
                M, N, K = info[0], info[1], info[2]
                gemm_flops += 2.0 * M * N * K
                gemm_ms += d
                n_gemm += 1
        total_ms = sum(v[1] for v in by.values())
        achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "ncu_step_dram_r02_final.json")          # capture of the final build's launch set
        if not os.path.exists(tp):
            tp = os.path.join(ROOT, "profiles", "ncu_step_dram_r02.json")
        if os.path.exists(tp):
            td = json.load(open(tp))
            fam = td.get("families", {}).get("gemm")
            if fam and fam.get("launches"):
                traffic = int(fam["dram_bytes"] / fam["launches"])
                traffic_src = td.get("source")
        roof = dict(bound="tensor", kernel="ub::gemm_kernel (tcgen05/TMEM/TMA bf16 GEMM family, all launches of one step)",
                    achieved=round(achieved, 1), peak=peaks["bf16"], unit="TFLOP/s", frac=round(achieved / peaks["bf16"], 4),
                    traffic=traffic, traffic_source=traffic_src, peak_source=peaks["source"], launches_per_step=n_gemm,
                    alg_flops_per_launch=gemm_flops / n_gemm, avg_launch_us=round(gemm_ms / n_gemm * 1e3, 2),
                    share_of_step=round(gemm_ms / total_ms, 4))
        breakdown = {k: dict(launches=v[0], ms=round(v[1], 3)) for k, v in sorted(by.items(), key=lambda kv: -kv[1][1])}
        if args.profile_out:
            gs = {k: dict(launches=v[0], ms=round(v[1], 3), us_each=round(v[1] / v[0] * 1e3, 1), tflops=round(v[2] * v[0] / (v[1] * 1e-3) / 1e12, 1))
                  for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][1])}
            json.dump(dict(ms_per_step_sum_of_ops=total_ms, ops=breakdown, gemm_tflops=achieved,
                           gemm_shapes_M_N_K_aT_bT_fp32out=gs), open(args.profile_out, "w"), indent=1)

    def finish():
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            # captured graphs hold references to the process group's communicator: drop them before tearing it down
            eng._graphs.clear()
            torch.cuda.synchronize()
            dist.barrier()
            torch.cuda.synchronize()
            # The fused NVLink step leaves no NCCL call inside the captured graphs, and with the graphs dropped above the process
            # group tears down cleanly (checked at 2 GPUs).  Only the NCCL fallback path (UB_DDP_NVLS=0: all-reduces captured in
            # the graphs) has hung in destroy_process_group(); there the ranks still leave together, hard.
            hard = os.environ.get("UB_BENCH_HARD_EXIT", "") == "1" or (getattr(eng, "nvls", None) is None and use_graph)
            if hard and os.environ.get("UB_BENCH_HARD_EXIT", "") != "0":
                os._exit(0)
            dist.destroy_process_group()

    if rank != 0:
        finish()
        return
    # ---- baselines measured on THIS box, after our own timing so they cannot disturb it ------------------------------------
    del dev_batches
    torch.cuda.empty_cache()
    eager = None
    if world == 1 and not args.no_eager_baseline:
        eager = gpu_eager_reference(B, args.steps, args.warmup, local)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_reference_run(steps=3, warmup=1)
        cpu = dict(value=round(cb["value"], 3), unit="clips/s", cores=cb["cores"], kind=cb["kind"], sample=cb["sample"])
    per_gpu = value / world
    f_alg = F_ALG["stage1"]
    line = dict(
        metric=METRIC, value=round(value, 2), unit="clips/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=round(ms_per_step, 3), higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
        config=dict(workload=WORKLOAD, per_gpu_batch=B, global_batch=B * world, parallelism=f"dp{world}", cuda_graph=use_graph,
                    graphs_captured=graphs_captured, drop_path=DROP_PATH, warmup_steps_run=n_warm,
                    ddp=("fused NVLink step (ub_adamw_nvls)" if getattr(eng, "nvls", None) is not None else ("NCCL all-reduce" if world > 1 else "n/a")),
                    l2_policy="inputs_exceed_l2 (154 MB clip batch + "
                    "multi-GB activations per step vs 126 MB L2; two input batches alternate)", init="random (reference initialisers), seed 0"),
        clocks=clocks, e2e=e2e, gpu_launches=launches, roofline=roof, cpu_baseline=cpu, gpu_eager_baseline=eager,
        mfu=dict(alg_gflop_per_clip=f_alg, tflops_per_gpu=round(per_gpu * f_alg / 1e3, 1),
                 of_nominal_2250=round(per_gpu * f_alg / 1e3 / NOMINAL_BF16_TFLOPS, 4),
                 of_measured_sustained=round(per_gpu * f_alg / 1e3 / measured_peaks()["bf16"], 4)),
        parity_check=parity, ddp_parity=ddp_parity,
        loss=round(loss_value, 5), e2e_loss=round(stats["loss"], 5), op_breakdown_ms=breakdown)
    line[e2e_other[0]] = e2e_other[1]
    if eager and "value" in eager:
        line["speedup_vs_eager"] = dict(value=round(value / eager["value"], 2), e2e=round(e2e["value"] / eager["value"], 2),
                                        note="ours / gpu_eager_baseline on the same GPU in the same run (the eager arm's inputs are device-resident)")
    print(json.dumps(line), flush=True)
    finish()


if __name__ == "__main__":
    main()
