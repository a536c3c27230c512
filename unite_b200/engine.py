"""Fused training-step engines: the bodies of the reference's train_one_epoch loops without autograd or host syncs.

Stage1Engine.step == run_stage1.py:360-456 for mask_type='attention', clip_loss_type='l2', clip_loss_data='mixed',
src_classifier=None:
    teacher forward (no grad)                       run_stage1.py:360-377
    attention-guided mask from Exp(1) noise         :379-387      (ub_mask_select, bit-exact given attn and q)
    gather + project teacher targets                :389-397      (only the visible rows are ever projected)
    student forward on visible tokens, l2 loss      :410-438
    backward                                        :451-455  (utils.py:608-609)
    [gradient all-reduce, unite_b200/ddp.py]        run_stage1.py:809 (DDP)
    grad-norm + AdamW                               utils.py:610-622, optim_factory.py:162-163
Nothing in the step reads a device value on the host: the loss and grad-norm stay on the GPU until the caller asks.
"""
import math
import os
import sys
import warnings
from typing import Optional

import torch

from . import ops
from .modeling_adaptation import AdaptationVisionTransformer
from .clip import VisionTransformer as ClipVisionTransformer

BF16, F32, I32, U8 = torch.bfloat16, torch.float32, torch.int32, torch.uint8


def get_num_layer_for_vit(var_name: str, num_max_layer: int) -> int:
    """Layer id of a parameter for layer-wise lr decay — src/optim_factory.py:45-63 (note: names are matched WITHOUT stripping a
    wrapper prefix, so every `encoder.*` parameter of the adaptation student lands in the last group, as in the reference)."""
    if var_name in ("cls_token", "mask_token", "pos_embed"):
        return 0
    if var_name.startswith("patch_embed"):
        return 0
    if var_name.startswith("rel_pos_bias"):
        return num_max_layer - 1
    if var_name.startswith("blocks"):
        return int(var_name.split(".")[1]) + 1
    if var_name.startswith("transformer.resblocks"):
        return int(var_name.split(".")[2]) + 1
    if var_name in ("class_embedding", "positional_embedding", "temporal_positional_embedding"):
        return 0
    if var_name.startswith("conv1"):
        return 0
    return num_max_layer - 1


class LayerDecayValueAssigner:
    """src/optim_factory.py:66-74; built as run_stage2.py:616-617 does: values = [decay ** (L + 1 - i) for i in range(L + 2)]."""

    def __init__(self, values):
        self.values = list(values)

    def get_scale(self, layer_id):
        return self.values[layer_id]

    def get_layer_id(self, var_name):
        return get_num_layer_for_vit(var_name, len(self.values))


class FusedAdamW:
    """AdamW over a ParamArena, one kernel per step (ub_adamw_seg); also refreshes the bf16 weight shadow and measures the global
    gradient norm (utils.py:631-643) without per-tensor kernels.

    Parameter groups follow src/optim_factory.py:76-118 (get_parameter_groups): "decay" / "no_decay", or with a layer assigner
    (get_num_layer / get_layer_scale, optim_factory.py:66-74) "layer_%d_decay" / "layer_%d_no_decay" with their `lr_scale`;
    parameters with requires_grad=False at construction are left out of every group (:83-84) and are never touched.  Each group
    is one or more contiguous runs of the arena; `param_groups` holds one dict per group exactly like torch's, and the training
    loops write `lr` / `weight_decay` into them every step (run_stage1.py:326-338, engine_for_finetuning.py:76-81)."""

    def __init__(self, arena, lr=1.5e-4, weight_decay=0.05, betas=(0.9, 0.95), eps=1e-8, get_num_layer=None, get_layer_scale=None):
        self.arena = arena
        self.lr, self.weight_decay, self.betas, self.eps = lr, weight_decay, betas, eps
        self.exp_avg = torch.zeros_like(arena.params)
        self.exp_avg_sq = torch.zeros_like(arena.params)
        self.step_count = 0
        self.gnorm_sq = torch.zeros(1, device=arena.device, dtype=F32)
        # ---- groups and their runs in the arena ---------------------------------------------------------------------------
        self.param_groups, index = [], {}
        seg_group, seg_end = [], []
        for i, name in enumerate(arena.names):
            off, numel = arena.offsets[name]
            p = arena._params[name]
            nxt = arena.offsets[arena.names[i + 1]][0] if i + 1 < len(arena.names) else arena.numel
            if not p.requires_grad:
                gi = -1                                                         # frozen: optim_factory.py:83-84
            else:
                decay = off < arena.n_decay
                gname = "decay" if decay else "no_decay"
                scale = 1.0
                if get_num_layer is not None:
                    layer_id = get_num_layer(name)
                    gname = "layer_%d_%s" % (layer_id, gname)
                    if get_layer_scale is not None:
                        scale = float(get_layer_scale(layer_id))
                if gname not in index:
                    index[gname] = len(self.param_groups)
                    self.param_groups.append(dict(name=gname, lr=lr * scale, weight_decay=weight_decay if decay else 0.0,
                                                  lr_scale=scale, params=[]))
                gi = index[gname]
                self.param_groups[gi]["params"].append(p)
            if seg_group and seg_group[-1] == gi:
                seg_end[-1] = nxt
            else:
                seg_group.append(gi)
                seg_end.append(nxt)
        if any(e % 4 for e in seg_end):
            raise RuntimeError("arena parameter offsets must be multiples of 4 elements")
        if not self.param_groups:
            raise ValueError("FusedAdamW: every parameter is frozen")
        self._seg_group = seg_group
        self._seg_end4 = torch.tensor([e // 4 for e in seg_end], dtype=I32, device=arena.device)
        self.n_seg = len(seg_group)
        # the two-group default layout [decay | no-decay] without frozen parameters is what the fused NVLink step understands
        self.plain_two_groups = [g["name"] for g in self.param_groups] in (["decay", "no_decay"], ["decay"]) and \
            -1 not in seg_group and self.n_seg == len(self.param_groups)
        n_h = 8 + 2 * self.n_seg
        self._hyper_dev = torch.zeros(n_h, device=arena.device, dtype=F32)
        self._hyper_pin = None
        self._hyper_ev = None

    def zero_grad(self, set_to_none: bool = False):
        self.arena.grads.zero_()

    # ---- graph-friendly form: scalars live in device memory, refreshed by one small async copy per step ----------------------
    _RING = 8

    def prepare_step(self, grad_scale: float = 1.0):
        """Host side of a (possibly graph-replayed) step: advance the step counter and upload every group's lr / wd and the bias
        corrections.  The upload goes through a ring of pinned slots; a slot is rewritten only after the copy that last read
        it has EXECUTED (an event per slot) — the DMA reads pinned memory when it runs, not when it is enqueued, and a host
        that queues graph replays can be many steps ahead of the device."""
        on_gpu = self._hyper_dev.is_cuda
        if self._hyper_pin is None:
            self._hyper_pin = [torch.zeros_like(self._hyper_dev, device="cpu").pin_memory() if on_gpu else
                               torch.zeros_like(self._hyper_dev, device="cpu") for _ in range(self._RING)]
            self._hyper_ev = [None] * self._RING
        self.step_count += 1
        b1, b2 = self.betas
        k = self.step_count % self._RING
        if self._hyper_ev[k] is not None:
            self._hyper_ev[k].synchronize()
        S = self.n_seg
        vals = [0.0] * (8 + 2 * S)
        g0 = self.param_groups[0]
        vals[0], vals[1] = g0["lr"], g0["weight_decay"]                        # read by ub_adamw_nvls (plain two-group layout)
        vals[2:8] = [b1, b2, self.eps, 1.0 - b1 ** self.step_count, math.sqrt(1.0 - b2 ** self.step_count), grad_scale]
        for s, gi in enumerate(self._seg_group):
            if gi < 0:
                vals[8 + s], vals[8 + S + s] = 0.0, -1.0
            else:
                g = self.param_groups[gi]
                vals[8 + s], vals[8 + S + s] = g["lr"], g["weight_decay"]
        hp = self._hyper_pin[k]
        hp.copy_(torch.tensor(vals, dtype=F32))
        self._hyper_dev.copy_(hp, non_blocking=True)
        if on_gpu:
            self._hyper_ev[k] = torch.cuda.Event()
            self._hyper_ev[k].record()

    def step_dev(self, max_norm: Optional[float] = None):
        """Device side: grad-norm + AdamW reading the scalars uploaded by prepare_step (capturable in a CUDA graph).
        max_norm: utils.py:613-615 (torch.nn.utils.clip_grad_norm_ before the step): the norm must be known before the
        update, so it takes its own sweep (ub_sumsq_seg); the clip coefficient min(1, max_norm / (norm + 1e-6)) is folded into
        the kernel's grad_scale on the device — no host read, the gradients themselves are not rewritten."""
        a = self.arena
        self.gnorm_sq.zero_()
        if not max_norm:
            ops.adamw_seg(a.params, a.grads, self.exp_avg, self.exp_avg_sq, a.w16, self._seg_end4, self._hyper_dev, self.gnorm_sq)
            return
        ops.sumsq_seg(a.grads, self._seg_end4, self._hyper_dev, self.gnorm_sq)
        if not hasattr(self, "_hyper_clip"):
            self._hyper_clip = torch.zeros_like(self._hyper_dev)
        h = self._hyper_clip
        h.copy_(self._hyper_dev)
        norm = self.gnorm_sq.sqrt() * self._hyper_dev[7:8]               # norm of the AVERAGED gradients (the arena holds rank sums)
        h[7:8] = self._hyper_dev[7:8] * (max_norm / (norm + 1e-6)).clamp(max=1.0)
        ops.adamw_seg(a.params, a.grads, self.exp_avg, self.exp_avg_sq, a.w16, self._seg_end4, h, None)

    def step(self, grad_scale: float = 1.0, max_norm: Optional[float] = None):
        self.prepare_step(grad_scale=grad_scale)
        self.step_dev(max_norm=max_norm)

    def consolidate(self):
        """Collective no-op unless the optimizer state is sharded by rank (ddp.NvlsShardedStep attaches itself as `_sharded`):
        afterwards every rank holds all fp32 master weights and Adam moments.  Call it on EVERY rank before state_dict()."""
        sharded = getattr(self, "_sharded", None)
        if sharded is not None:
            sharded.consolidate()

    def grad_norm(self, grad_scale: float = 1.0) -> torch.Tensor:
        return self.gnorm_sq.sqrt() * grad_scale

    def state_dict(self):
        groups = [{k: v for k, v in g.items() if k != "params"} for g in self.param_groups]
        return dict(step=self.step_count, exp_avg=self.exp_avg, exp_avg_sq=self.exp_avg_sq, param_groups=groups)

    def load_state_dict(self, sd):
        self.step_count = sd["step"]
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        if len(sd["param_groups"]) != len(self.param_groups):
            raise ValueError("optimizer state has a different number of parameter groups")
        for g, saved in zip(self.param_groups, sd["param_groups"]):
            g.update({k: v for k, v in saved.items() if k != "params"})


_ASYNC_ZERO = os.environ.get("UB_ASYNC_ZERO", "1") != "0"


class GraphReplay:
    """CUDA-graph plumbing of the step engines: the first two steps of an input signature run eagerly (lazy attribute setting,
    workspace allocation, NCCL initialisation), then the step body is captured once per set of persistent input buffers — callers
    that cycle through a few resident buffers (the staging ring of train_one_epoch, bench.py's resident batches) get one graph per
    buffer set, bound directly to them, and no device-to-device copy into a static input per step; past `max_graphs` sets
    (UB_MAX_GRAPHS, default 6; 0: always) the inputs are copied into one more graph that owns private static inputs.  All graphs
    share one memory pool (they never run concurrently).  The body must be free of host synchronisation and read its per-step
    scalars from device memory (FusedAdamW.prepare_step / step_dev)."""

    def __init__(self, max_graphs: Optional[int] = None):
        self.max_graphs = int(os.environ.get("UB_MAX_GRAPHS", "6")) if max_graphs is None else max_graphs
        self._graphs, self._count, self._eager, self._pool = {}, {}, {}, None

    def clear(self):
        self._graphs.clear(); self._count.clear()

    def run(self, shape_key, inputs, body, state_fn=None, private=False):
        """inputs: tuple of device tensors (None entries are passed through).  body(*inputs) runs one step.  state_fn() -> any
        object describing the tensors the body left behind (captured once per graph, returned on every replay).
        private=True: always replay the graph with private static inputs (for callers whose batches arrive in fresh tensors)."""
        n = self._eager.get(shape_key, 0)
        if n < 2:
            self._eager[shape_key] = n + 1
            body(*inputs)
            return state_fn() if state_fn else None
        ptrs = tuple(t.data_ptr() if t is not None else 0 for t in inputs)
        buf_key = shape_key + (("private",) if private else ptrs)
        if buf_key not in self._graphs:
            private = private or self._count.get(shape_key, 0) >= self.max_graphs
            if private:
                buf_key = shape_key + ("private",)
            if buf_key not in self._graphs:
                static = tuple((torch.empty_like(t) if t is not None else None) for t in inputs) if private else tuple(inputs)
                if private:
                    for s_, t in zip(static, inputs):
                        if t is not None:
                            s_.copy_(t)
                torch.cuda.synchronize()
                g = torch.cuda.CUDAGraph()
                n0 = ops.LAUNCHES
                with torch.cuda.graph(g, pool=self._pool):
                    body(*static)
                if self._pool is None:
                    self._pool = g.pool()
                n_kernels = ops.LAUNCHES - n0           # kernels of ours recorded in the graph (capture executes nothing)
                ops.LAUNCHES = n0
                self._graphs[buf_key] = (g, static, n_kernels, state_fn() if state_fn else None)
                self._count[shape_key] = self._count.get(shape_key, 0) + 1
        g, static, n_kernels, state = self._graphs[buf_key]
        ops.LAUNCHES += n_kernels                       # every replay launches all of them
        for s_, t in zip(static, inputs):
            if t is not None and s_.data_ptr() != t.data_ptr():
                s_.copy_(t, non_blocking=True)
        g.replay()
        return state


def require_fused_optimizer(optimizer, arena, what: str):
    """The engines update the arena with FusedAdamW only.  A foreign optimizer (torch.optim.AdamW from the reference's
    create_optimizer, src/optim_factory.py:120-175) would silently be ignored — refuse it instead."""
    if optimizer is None:
        return None
    if not isinstance(optimizer, FusedAdamW):
        raise TypeError(f"{what}: optimizer must be a unite_b200 FusedAdamW built over the model's parameter arena (see "
                        f"unite_b200.optim_factory.create_optimizer), got {type(optimizer).__name__}; a torch optimizer cannot "
                        "drive the fused step")
    if optimizer.arena is not arena:
        raise ValueError(f"{what}: the optimizer was built over a different parameter arena than this model's")
    return optimizer


class StepEngine:
    """The data-parallel update shared by Stage1Engine, Stage2Engine and Stage3Engine.  Everything is read from the engine's
    attributes when it is called (core, optimizer, grad_sync, nvls, max_norm, graphs), so a caller may swap any of them between
    steps (bench.py's parity gate runs forward_backward with grad_sync = None)."""

    @property
    def grad_scale(self) -> float:
        """The arena holds the SUM of every rank's gradients; AdamW and the reported grad-norm take 1 / world of it."""
        return 1.0 / self.grad_sync.world if self.grad_sync is not None else 1.0

    def _fused_step(self):
        """N > 1: the all-reduce -> AdamW pair becomes ONE kernel over NVSwitch multicast (ddp.NvlsShardedStep) when the box
        offers it; UB_DDP_NVLS=0 (or a box without multicast) keeps NCCL range all-reduces overlapped with backward (None)."""
        gs = self.grad_sync
        if gs is None or getattr(gs, "world", 1) <= 1 or self.core.arena.device.type != "cuda" \
                or os.environ.get("UB_DDP_NVLS", "1") == "0" or not self.optimizer.plain_two_groups:
            return None
        from .ddp import NvlsShardedStep
        try:
            return NvlsShardedStep(self.core.arena, self.optimizer, gs.pg)
        except Exception as e:                          # no multicast / symmetric memory on this box: NCCL path
            if os.environ.get("UB_DDP_NVLS") == "1":
                raise
            warnings.warn(f"unite_b200: NVLS fused optimizer step unavailable ({type(e).__name__}: {e}); using NCCL all-reduce")
            return None

    def set_optimizer(self, optimizer: "FusedAdamW"):
        """Swap in a caller-built FusedAdamW over the same arena (train_one_epoch's `optimizer` argument); the fused data-parallel
        step, if active, is re-bound to it (its gradient-norm accumulator lives in symmetric memory)."""
        if optimizer is self.optimizer:
            return
        require_fused_optimizer(optimizer, self.core.arena, f"{type(self).__name__}.set_optimizer")
        if self.nvls is not None:
            if not optimizer.plain_two_groups:
                raise NotImplementedError("the fused NVLink step updates the plain [decay | no-decay] layout; layer-decay groups or "
                                          "frozen parameters need UB_DDP_NVLS=0 (NCCL all-reduce + ub_adamw_seg)")
            self.nvls.opt = optimizer
            optimizer.gnorm_sq = self.optimizer.gnorm_sq
            optimizer._sharded = self.nvls
        self.optimizer = optimizer
        self.graphs.clear()                     # captured graphs hold the old optimizer's buffers

    def _backward_hook(self):
        """Who is told, block by block, that a prefix of the gradient arena is final: the fused NVLink step (copy-engine pushes
        to the owning ranks) or the NCCL path (range all-reduces); both overlap the rest of backward.  With clip_grad the fused
        step needs the summed gradient first (NvlsShardedStep.step_dev_clipped), so nothing is pushed early."""
        if self.nvls is not None:
            return self.nvls if (self.nvls.early_push and not self.max_norm) else None
        return self.grad_sync

    def _update(self):
        """After backward: reduce-scatter + AdamW + shadow all-gather in one kernel (the fused NVLink step), or the NCCL
        all-reduce followed by grad-norm + AdamW.  Reads the scalars of the optimizer's last prepare_step."""
        if self.nvls is not None:
            if self.max_norm:
                self.nvls.step_dev_clipped(self.max_norm)
            else:
                self.nvls.step_dev()
            return
        if self.grad_sync is not None:
            self.grad_sync.all_reduce(self.core.arena.grads)
        self.optimizer.step_dev(max_norm=self.max_norm)


def apply_schedule(optimizer, it: int, lr_schedule_values=None, wd_schedule_values=None):
    """Step `it` of the per-step lr / weight-decay schedules into the optimizer's param_groups: lr times the group's lr_scale
    (layer decay), weight decay only in the groups that decay."""
    for group in optimizer.param_groups:
        if lr_schedule_values is not None:
            group["lr"] = lr_schedule_values[min(it, len(lr_schedule_values) - 1)] * group.get("lr_scale", 1.0)
        if wd_schedule_values is not None and group["weight_decay"] > 0:
            group["weight_decay"] = wd_schedule_values[min(it, len(wd_schedule_values) - 1)]


def schedule_stats(optimizer) -> dict:
    """The lr / min_lr / weight_decay entries of the dict train_one_epoch returns."""
    lrs = [g["lr"] for g in optimizer.param_groups]
    wds = [g["weight_decay"] for g in optimizer.param_groups if g["weight_decay"] > 0]
    return {"lr": max(lrs), "min_lr": min(lrs), "weight_decay": wds[0] if wds else None}


def frames_rows(frames: torch.Tensor, tubelet: int) -> torch.Tensor:
    """Normalised bf16 im2col rows of decoded uint8 frames [B,T,H,W,3] for a Conv3d of temporal kernel `tubelet` and 16-pixel
    patches (ops.patchify_u8)."""
    B, T, H, W, _ = frames.shape
    out = torch.empty(B * (T // tubelet) * (H // 16) * (W // 16), 3 * tubelet * 256, device=frames.device, dtype=BF16)
    return ops.patchify_u8(frames, out, tubelet)


def frames_carrier(frames: torch.Tensor) -> torch.Tensor:
    """A zero-stride fp32 [B,3,T,H,W] view with the shape of the clip that uint8 frames [B,T,H,W,3] stand for: handed to a tower
    together with the frames' im2col rows, it gives the shapes and never has its values read."""
    B, T, H, W, _ = frames.shape
    return torch.empty(1, device=frames.device, dtype=F32).expand(B, 3, T, H, W)


def exit_if_not_finite(loss: float):
    """A non-finite loss stops training, as the reference's loops do."""
    if not math.isfinite(loss):
        print("Loss is {}, stopping training".format(loss))
        sys.exit(1)


class Stage1Engine(StepEngine):
    def __init__(self, student: AdaptationVisionTransformer, teacher: ClipVisionTransformer, mask_ratio: float = 0.8,
                 lr: float = 1.5e-4, weight_decay: float = 0.05, betas=(0.9, 0.95), eps: float = 1e-8, grad_sync=None,
                 use_graph: bool = False, clip_loss_type: str = "l2", optimizer: Optional[FusedAdamW] = None):
        """use_graph: after two eager steps of a given batch shape, the whole step (teacher, mask, DropPath draw, student
        fwd/bwd, gradient all-reduce, grad-norm, AdamW) is captured once in a CUDA graph and replayed — the ~460 launches of a
        step then cost one launch.  DropPath (drop_path: 0.1 in every shipped config) stays inside the graph: its factors come
        from ub_drop_path_draw, a counter-based generator whose step counter lives in device memory (csrc/rng.cu)."""
        self.student, self.teacher, self.mask_ratio = student, teacher, mask_ratio
        self.use_graph = use_graph
        self.clip_loss_type = clip_loss_type
        self.clip_loss_data = "mixed"         # 'source' / 'target': only the first B_s / the remaining clips enter the loss (:418-423)
        self.n_source = None                  # B_s of the current batch (needed when clip_loss_data != 'mixed')
        self.max_norm = None                  # clip_grad of the reference's loss_scaler call (run_stage1.py:451-455); None / 0 = off
        self.graphs = GraphReplay()
        self._graphs = self.graphs._graphs    # the same dict: bench.py counts and drops a stage-1 engine's graphs through it
        self.core = student.core()
        self.core.sync_shadow(force=True)
        self.optimizer = require_fused_optimizer(optimizer, self.core.arena, "Stage1Engine") or \
            FusedAdamW(self.core.arena, lr, weight_decay, betas, eps)
        self.grad_sync = grad_sync            # unite_b200.ddp.GradSync or None
        self.nvls = self._fused_step()
        # the resolution the teacher sees (train_one_epoch's clip_input_resolution): a clip of another size is resized for the
        # teacher only (bicubic, on the device); the student always patchifies the clip as it comes
        self.teacher_resolution = teacher.input_resolution
        if student.clip_output_dim != teacher.output_dim:
            raise ValueError(f"the student's clip_output_dim {student.clip_output_dim} differs from the teacher's output_dim "
                             f"{teacher.output_dim}: the alignment loss compares the two")
        self.loss = torch.zeros(1, device=self.core.arena.device, dtype=F32)
        self.last = {}
        self.drop_path = self.core.drop_path       # vit_core.DropPathSource: device-side draws, one launch per step

    @property
    def share_patches(self) -> bool:
        """Student and teacher read one im2col of the clip: same temporal kernel, 16-pixel teacher patches, no resize."""
        side = self.student.encoder.patch_embed.img_size
        return (self.student.encoder.patch_embed.tubelet_size == self.teacher.kernel_size and self.teacher.patch_size == 16
                and tuple(side) == (self.teacher_resolution, self.teacher_resolution))

    def teacher_view(self, H: int, W: int):
        """(resolution, resize?) of the teacher for an H x W clip; ValueError when the configuration cannot align the teacher's
        attention map with the student's tokens."""
        R, p = int(self.teacher_resolution), self.teacher.patch_size
        if R % p:
            raise ValueError(f"teacher resolution {R} is not a multiple of the teacher's patch size {p}")
        ps = self.student.encoder.patch_embed.patch_size[0]
        n_t, n_s = (R // p) ** 2, (H // ps) * (W // ps)
        if n_t != n_s:
            raise ValueError(f"the teacher sees {n_t} patches per frame ({R} px / {p}), the student {n_s} ({H}x{W} px / {ps}): "
                             "the attention-guided mask needs the same number")
        return R, (R != H or R != W)

    def n_visible(self, P):
        return P - int(P * self.mask_ratio)                      # run_stage1.py:380

    def forward_backward(self, videos: torch.Tensor, q: torch.Tensor, dp: Optional[torch.Tensor] = None,
                         attn_override: Optional[torch.Tensor] = None, clip_loss_type: Optional[str] = None, grads_ready=None):
        """Everything up to (not including) the optimizer.  videos fp32 [B,3,T,H,W] on the device; q fp32 [B*T',HW]
        Exp(1) noise for the mask sampler.  Returns the device loss tensor [1].
        grads_ready: event after which the gradient arena may be written (its fill runs on a side stream, _step_body_dev)."""
        core, teacher = self.core, self.teacher
        B = videos.shape[0]
        H_, W_ = videos.shape[2:4] if videos.dtype == U8 else videos.shape[3:5]
        R, resize = self.teacher_view(H_, W_)
        share = self.share_patches and not resize
        patches = None
        patches_s = None
        if videos.dtype == U8:
            # decoded frames uint8 [B,T,H,W,3]: normalise + patchify in one pass (SURVEY.md §8 row f2); the fp32 clip the
            # reference materialises never exists — `videos` below is a zero-stride shape carrier
            T_ = videos.shape[1]
            ks, tub, p = teacher.kernel_size, self.student.encoder.patch_embed.tubelet_size, teacher.patch_size
            if p == 16 and not resize:
                patches = frames_rows(videos, ks)
            else:
                patches = ops.resize_patchify(videos, torch.empty(B * (T_ // ks) * (R // p) ** 2, teacher.k_pad, device=videos.device,
                                                                  dtype=BF16), R, p, ks)
            patches_s = patches if share else frames_rows(videos, tub)
            videos = frames_carrier(videos)
        elif share:
            ks = teacher.kernel_size
            n_tok = B * (videos.shape[2] // ks) * (videos.shape[3] // 16) * (videos.shape[4] // 16)
            patches = torch.empty(n_tok, 3 * ks * 256, device=videos.device, dtype=BF16)
            ops.patchify(videos, patches, ks)
        sel = {}

        def select(attn):
            # run_stage1.py:379-387 on the device, called by the teacher as soon as its last block's attention map exists
            frames, P = attn.shape
            Tp = frames // B
            n_vis = self.n_visible(P)
            sel["mask"] = torch.empty(1, frames * P, device=videos.device, dtype=U8)
            sel["vis_idx"] = torch.empty(1, B, Tp * n_vis, device=videos.device, dtype=I32)
            sel["tea_rows"] = torch.empty(1, B, Tp * n_vis, device=videos.device, dtype=I32)
            ops.mask_select(attn if attn_override is None else attn_override, q, sel["mask"], sel["vis_idx"], sel["tea_rows"], Tp, 1,
                            n_vis)
            return sel["tea_rows"].view(-1)

        layers, attn, _ = teacher.forward_features(videos, patches, select=select, resolution=R)
        if not sel:                                                               # teacher without return_attn / last-layer tap
            select(attn)
        frames, P = attn.shape
        Tp = frames // B
        mask, vis_idx, tea_rows = sel["mask"], sel["vis_idx"], sel["tea_rows"]
        targets = teacher.project_rows(layers, tea_rows.view(-1))                 # [K, B*Nv, C]
        if dp is None and self.student.training:
            dp = self.drop_path.draw(B)                                            # None when every rate is 0
        loss_clips = self._loss_clips(B)
        self.loss.zero_()
        if patches_s is None:
            patches_s = patches if share else None
        kind = clip_loss_type or self.clip_loss_type
        if kind == "l2":
            # shipped config: the loss and its gradient are fused into the decoder-tail kernels
            _, x_clip, state = core.run_forward(videos, vis_idx[0], patches_s, dp, True, True,
                                                targets=targets, loss_acc=self.loss, loss_clips=loss_clips)
            if grads_ready is not None:
                torch.cuda.current_stream().wait_event(grads_ready)
            core.run_backward(state, targets=targets, grad_sync=self._backward_hook())
        else:
            # run_stage1.py:403-408,432-433 (nn.MSELoss / nn.SmoothL1Loss / nn.L1Loss, mean reduction): loss value and
            # d loss / d outputs are a few element-wise device ops on the [K,B,Nv,C] outputs; the rest of backward is shared
            _, x_clip, state = core.run_forward(videos, vis_idx[0], patches_s, dp, True, True)
            d = x_clip - targets.view_as(x_clip)
            if loss_clips is not None:                                             # :418-423: slice both tensors along the clip axis
                keep = torch.zeros(1, B, 1, 1, device=d.device, dtype=d.dtype)
                keep[:, loss_clips[0]:loss_clips[1]] = 1.0
                d = d * keep
                n = d[:, loss_clips[0]:loss_clips[1]].numel()
            else:
                keep = None
                n = d.numel()
            if kind == "mse":
                self.loss += (d * d).sum() / n
                g = d * (2.0 / n)
            elif kind == "smooth_l1":
                ad = d.abs()
                self.loss += torch.where(ad < 1.0, 0.5 * d * d, ad - 0.5).sum() / n
                g = d.clamp(-1.0, 1.0) / n
            elif kind == "l1":
                self.loss += d.abs().sum() / n
                g = d.sign() / n                                                   # sign(0) = 0 on the rows outside the slice
            else:
                raise NotImplementedError(f"clip_loss_type={kind!r} (run_stage1.py:430-435 raises for anything else too)")
            if grads_ready is not None:
                torch.cuda.current_stream().wait_event(grads_ready)
            core.run_backward(state, g_clip=g, grad_sync=self._backward_hook())
        self.last = dict(attn=attn, mask=mask.view(B, Tp * P).bool(), vis_idx=vis_idx[0], targets=targets, outputs=x_clip)
        return self.loss

    def _loss_clips(self, B):
        """Clip range [lo, hi) of the batch that enters the alignment loss (run_stage1.py:418-423); None = all ('mixed')."""
        if self.clip_loss_data == "mixed":
            return None
        if self.clip_loss_data not in ("source", "target"):
            raise NotImplementedError(f"clip_loss_data={self.clip_loss_data!r}")   # run_stage1.py:426-427
        if self.n_source is None or not (0 <= self.n_source <= B):
            raise ValueError(f"clip_loss_data={self.clip_loss_data!r} needs n_source (B_s, the number of source clips leading the "
                             f"batch) in [0, {B}]")
        lo, hi = (0, self.n_source) if self.clip_loss_data == "source" else (self.n_source, B)
        if hi <= lo:
            raise ValueError(f"clip_loss_data={self.clip_loss_data!r} selects no clip (B_s={self.n_source}, B={B})")
        return lo, hi

    def _step_body_dev(self, videos, q):
        # The 352 MB fill of the gradient arena runs on a side stream beside the teacher's forward (an HBM-write-bound fill next to
        # L2 / tensor-bound GEMMs) and is joined right before the first gradient is written; inside a CUDA graph this is a fork /
        # join of two branches.  UB_ASYNC_ZERO=0: in line, ahead of the step.
        zeroed = None
        if _ASYNC_ZERO and self.core.arena.device.type == "cuda":
            cur = torch.cuda.current_stream()
            if getattr(self, "_zero_stream", None) is None:
                self._zero_stream = torch.cuda.Stream(device=self.core.arena.device)
            self._zero_stream.wait_stream(cur)
            with torch.cuda.stream(self._zero_stream):
                self.optimizer.zero_grad()
                zeroed = torch.cuda.Event()
                zeroed.record()
        else:
            self.optimizer.zero_grad()
        self.forward_backward(videos, q, None, grads_ready=zeroed)
        self._update()

    def step(self, videos, q, dp=None):
        self.optimizer.prepare_step(grad_scale=self.grad_scale)
        if not self.use_graph or dp is not None:
            # eager (bench.py's instrumented per-op step too): the arena fill stays in line, ahead of the step
            self.optimizer.zero_grad()
            self.forward_backward(videos, q, dp)
            self._update()
            return self.loss
        shape_key = (tuple(videos.shape), videos.dtype, tuple(q.shape), self.clip_loss_type, float(self.max_norm or 0.0),
                     self.clip_loss_data, self.n_source if self.clip_loss_data != "mixed" else None, bool(self.student.training))
        # `last` = the mask / target / output tensors of the graph just replayed
        self.last = self.graphs.run(shape_key, (videos, q), self._step_body_dev, state_fn=lambda: self.last)
        return self.loss
