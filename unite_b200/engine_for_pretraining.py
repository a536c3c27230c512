"""`train_one_epoch` for stage 1 with the reference's signature (run_stage1.py:294-303, twin
src/engines/engine_for_pretraining_umt.py:32-40) on top of the fused Stage1Engine.

What changes versus the reference loop body: no per-step `.item()` / `torch.cuda.synchronize()` (run_stage1.py:440-441,
458) — the loss and grad-norm are accumulated on the device and read once per `log_freq` steps and at the end;
non-finite loss is still fatal (run_stage1.py:447-449) but is checked at those read points.
Batches are `(videos, mask_placeholder, labels[, noise])`; without `noise` the Exp(1) draw is made on the device.
`clip_input_resolution` is the side the teacher sees (run_stage1.py:360-377: the teacher's copy of the clip is resized to it,
bicubic, when it differs from the clip's); None (the default here) means the teacher's own input_resolution, the only side its
positional embedding fits.  A CLIP ViT-L/14 teacher behind a 16-pixel student at 224 px needs 196.
"""
import math
import sys
from typing import Iterable, Optional

import torch

from .engine import Stage1Engine, require_fused_optimizer

_IO = {}          # per device: copy stream, device staging ring, pinned loss read-back slots


def register_engine(student, teacher, engine):
    """The engine of a (student, teacher) pair lives ON the student module (not in an id()-keyed global: ids are reused after
    garbage collection), so it is dropped together with the model."""
    student.__dict__["_ub_stage1_engine"] = (teacher, engine)


def _engine_for(model, teacher_model, mask_ratio, optimizer, use_graph=False):
    student = model.module if hasattr(model, "module") else model
    teacher = teacher_model.module if hasattr(teacher_model, "module") else teacher_model
    held = student.__dict__.get("_ub_stage1_engine")
    if held is None or held[0] is not teacher:
        gs = getattr(model, "grad_sync", None)
        if gs is not None:
            gs.arena = student.core().arena
        optimizer = require_fused_optimizer(optimizer, student.core().arena, "train_one_epoch")
        eng = Stage1Engine(student, teacher, mask_ratio=mask_ratio, grad_sync=gs, use_graph=use_graph, optimizer=optimizer)
        register_engine(student, teacher, eng)
        return eng
    eng = held[1]
    if optimizer is not None:
        eng.set_optimizer(require_fused_optimizer(optimizer, eng.core.arena, "train_one_epoch"))
    eng.mask_ratio = mask_ratio
    return eng


def train_one_epoch(model: torch.nn.Module, data_loader: Iterable, data_loader_train_target: Optional[Iterable] = None,
                    optimizer=None, device=None, epoch: int = 0, loss_scaler=None, max_norm: float = 0, log_writer=None,
                    lr_scheduler=None, start_steps=0, lr_schedule_values=None, wd_schedule_values=None, src_classifier=None,
                    teacher_model=None, clip_input_resolution=None, clip_loss_type="l2", clip_loss_ratio=0.5,
                    mask_type="attention", mask_ratio=0.0, use_wandb=False, args=None):
    if mask_type != "attention":
        # the reference itself only runs with mask_type='attention': run_stage1.py:378 reads `attn`, which the other mask
        # types never define (NameError on the first step)
        raise NotImplementedError("stage 1 runs with mask_type='attention' only (configs/stage1_config.yaml; run_stage1.py:378)")
    # src_classifier: run_stage1.py:412-415 then calls model(videos, mask) without clip_only and discards the encoder output —
    # the loss is loss_clip either way (:438), and clip_return_layers ends at the last block, so the compute is identical
    clip_loss_data = getattr(args, "clip_loss_data", "mixed") if args is not None else "mixed"
    if clip_loss_data not in ("source", "target", "mixed"):
        raise NotImplementedError(f"clip_loss_data={clip_loss_data!r}")                  # run_stage1.py:426-427
    if clip_loss_type not in ("l2", "mse", "smooth_l1", "l1"):
        raise NotImplementedError(f"clip_loss_type={clip_loss_type!r}")                  # run_stage1.py:434-435
    model.train()
    eng = _engine_for(model, teacher_model, mask_ratio, optimizer, use_graph=bool(getattr(args, "use_cuda_graph", False)))
    eng.clip_loss_type = clip_loss_type
    eng.teacher_resolution = eng.teacher.input_resolution if clip_input_resolution is None else int(clip_input_resolution)
    eng.clip_loss_data = clip_loss_data
    eng.max_norm = float(max_norm) if max_norm else None       # loss_scaler(..., clip_grad=max_norm, ...), run_stage1.py:451-455
    opt = eng.optimizer
    dev = eng.core.arena.device
    log_freq = getattr(args, "log_freq", 10) if args is not None else 10
    loss_sum = torch.zeros(1, device=dev)
    gn_sum = torch.zeros(1, device=dev)
    n = 0
    it_target = iter(data_loader_train_target) if data_loader_train_target is not None else None
    last_loss = float("nan")
    # Input pipeline: the H2D copy of batch i+1 runs on a side stream while batch i computes (pinned host memory, as
    # DataLoader(pin_memory=True) + .to(device, non_blocking=True) at run_stage1.py:349 intend), and the per-step loss is
    # read back through a pinned buffer one step late, so neither direction stalls the launch queue.
    io = _IO.setdefault(dev, dict(stream=torch.cuda.Stream(device=dev), ring={}, free={}, pos=[0],
                                  pin_loss=[torch.empty(1, pin_memory=True) for _ in range(2)]))
    copy_stream = io["stream"]           # persistent: the caching allocator keeps one pool per stream
    pin_loss = io["pin_loss"]
    pin_err = io.setdefault("pin_err", [torch.zeros(1, dtype=torch.int32).pin_memory() for _ in range(2)])
    loss_ev = [None, None]
    # Device staging ring (3 slots per tensor shape): allocating a fresh 154 MB tensor per step on the copy stream makes the
    # caching allocator cudaMalloc (a device-wide sync) whenever record_stream delays a block's reuse — measured as steps of
    # 32-92 ms between 19 ms ones.  A slot is rewritten only after the step that consumed it has been enqueued AND finished.
    ring, ring_free, ring_pos = io["ring"], io["free"], io["pos"]

    def stage(src):
        key = (tuple(src.shape), src.dtype)
        if key not in ring:
            ring[key] = [torch.empty(src.shape, dtype=src.dtype, device=dev) for _ in range(3)]
            ring_free[key] = [None, None, None]
        k = ring_pos[0] % 3
        if ring_free[key][k] is not None:
            copy_stream.wait_event(ring_free[key][k])
        dst = ring[key][k]
        dst.copy_(src, non_blocking=True)
        return dst, (key, k)

    def fetch(batch):
        videos, noise = batch[0], (batch[3] if len(batch) > 3 else None)
        n_source = videos.shape[0]                                             # B_s, run_stage1.py:342
        nonlocal it_target
        if it_target is not None:                                              # run_stage1.py:343-347
            try:
                tb = next(it_target)
            except StopIteration:
                it_target = iter(data_loader_train_target)
                tb = next(it_target)
            videos = torch.cat([videos, tb[0]], dim=0)
            if noise is not None and len(tb) > 3:
                noise = torch.cat([noise, tb[3]], dim=0)
        with torch.cuda.stream(copy_stream):
            v, slot_v = stage(videos)                                          # run_stage1.py:349 (.to(device, non_blocking=True))
            q, slot_q = (None, None) if noise is None else stage(noise)
            ring_pos[0] += 1
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return v, q, ev, (slot_v, slot_q), n_source

    def check(slot):
        nonlocal last_loss
        if loss_ev[slot] is not None:
            loss_ev[slot].synchronize()
            last_loss = float(pin_loss[slot][0])
            loss_ev[slot] = None
            if eng.nvls is not None:
                eng.nvls.raise_if(int(pin_err[slot][0]))                       # a peer stalled inside the fused data-parallel step
            if not math.isfinite(last_loss):
                print("Loss is {}, stopping training".format(last_loss))
                sys.exit(1)

    it_loader = iter(data_loader)
    nxt = next(it_loader, None)
    staged = fetch(nxt) if nxt is not None else None
    step = 0
    while staged is not None:
        videos, noise, ev, slots, eng.n_source = staged
        nxt = next(it_loader, None)
        it = start_steps + step
        for group in opt.param_groups:                                         # run_stage1.py:326-338
            if lr_schedule_values is not None:
                group["lr"] = lr_schedule_values[min(it, len(lr_schedule_values) - 1)] * group.get("lr_scale", 1.0)
            if wd_schedule_values is not None and group["weight_decay"] > 0:
                group["weight_decay"] = wd_schedule_values[min(it, len(wd_schedule_values) - 1)]
        torch.cuda.current_stream(dev).wait_event(ev)
        if noise is None:
            # fp32 clips are [B,3,T,H,W]; decoded uint8 frames are [B,T,H,W,3]
            T_, H_, W_ = (videos.shape[1:4] if videos.dtype == torch.uint8 else videos.shape[2:5])
            frames = videos.shape[0] * (T_ // eng.teacher.kernel_size)
            R, _ = eng.teacher_view(H_, W_)                                    # the mask is drawn over the teacher's patch grid
            noise = torch.empty(frames, (R // eng.teacher.patch_size) ** 2, device=dev).exponential_(1)
        staged = fetch(nxt) if nxt is not None else None                       # overlaps with this step's compute
        loss = eng.step(videos, noise)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(dev))
        for sl in slots:
            if sl is not None:
                ring_free[sl[0]][sl[1]] = done
        loss_sum += loss
        gn_sum += opt.grad_norm(1.0 / (eng.grad_sync.world if eng.grad_sync is not None else 1))
        n += 1
        if log_freq and (step + 1) % log_freq == 0:
            slot = (step // log_freq) & 1
            check(slot)                                                        # the read issued two log points ago
            pin_loss[slot].copy_(loss, non_blocking=True)                      # D2H of this step's loss (async)
            if eng.nvls is not None:
                eng.nvls.poll_error_async(pin_err[slot])
            loss_ev[slot] = torch.cuda.Event()
            loss_ev[slot].record()
        if lr_scheduler is not None:
            lr_scheduler.step_update(start_steps + step)
        step += 1
    check(0)
    check(1)
    stats = torch.cat([loss_sum, gn_sum]) / max(n, 1)
    if torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
        torch.distributed.all_reduce(stats)                                    # utils.py:239-241 (epoch-end meter sync)
        stats /= torch.distributed.get_world_size()
    loss_avg, gn_avg = stats.tolist()
    if not math.isfinite(loss_avg):
        print("Loss is {}, stopping training".format(loss_avg))
        sys.exit(1)
    lrs = [g["lr"] for g in opt.param_groups]
    wds = [g["weight_decay"] for g in opt.param_groups if g["weight_decay"] > 0]
    return {"loss": loss_avg, "loss_clip": loss_avg, "loss_scale": 1.0, "lr": max(lrs), "min_lr": min(lrs),
            "weight_decay": wds[0] if wds else None, "grad_norm": gn_avg}
