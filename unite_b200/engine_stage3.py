"""Stage-3 collaborative self-training step (run_stage3.py:427-642) on the fused kernels.

masking_type='clip_attention', selection_strategy='clip_matchORconf', train_masked=True, conf_weighted_loss=True — the
shipped configuration (configs/stage3_config.yaml).  Per step:
    teacher attention on the target clips (no projection needed)                   run_stage3.py:434-451
    student, all 1568 tokens, source clips (grad)  -> mean-pool -> src_classifier   :475-477
    student, all tokens, target clips (no grad)    -> logits_full_t                 :480-483
    greedy round-robin masks for k=2 committee members (ub_mask_select, q=NULL)     :493-497, utils.py:89-120
    student on the masked target views (member k-1 with grad) -> logits_masked      :499-505
    zero-shot CLIP probabilities, MatchOrConf selection, pseudo labels              :556-587   (ub_clip_zero_shot, ub_pseudo_label_fusion)
    loss = src_ratio * CE_s + tgt_ratio * |sel|/B_t * mean_sel(msp * CE(masked[-1], pseudo))    :599-625
    backward through both grad-carrying forwards, AdamW on the student only (src_classifier is frozen, :1193/:1264)
The OpenAI-CLIP image/text towers of `clip_infer` are not available offline: the teacher trunk's CLS embedding
(clip.VisionTransformer.cls_features) and a caller-supplied text matrix [n_classes, 512] stand in (SURVEY.md §8(c)).
No host synchronisation: |sel| never leaves the device — tgt_ratio*|sel|/B_t*mean_sel(w*CE) == tgt_ratio/B_t * sum_b sel_b*w_b*CE_b.
"""
import os
from typing import Iterable, Optional

import torch

from . import ops
from .engine import (FusedAdamW, GraphReplay, StepEngine, apply_schedule, exit_if_not_finite, require_fused_optimizer,
                     schedule_stats)

BF16, F32, I32, U8 = torch.bfloat16, torch.float32, torch.int32, torch.uint8


class Stage3Engine(StepEngine):
    def __init__(self, student, teacher, cls_weight: torch.Tensor, cls_bias: torch.Tensor, text_features: torch.Tensor,
                 mask_ratio: float = 0.8, k: int = 2, clip_threshold: float = 0.5, src_ratio: float = 1.0, tgt_ratio: float = 1.0,
                 conf_weighted: bool = True, lr: float = 1e-4, weight_decay: float = 0.05, betas=(0.9, 0.999), grad_sync=None,
                 optimizer: Optional[FusedAdamW] = None, use_graph: bool = False):
        """use_graph: after two eager steps of a batch signature the whole step (the five forwards, both backwards, the gradient
        exchange and AdamW: ~900 launches) is captured in a CUDA graph and replayed (engine.GraphReplay); nothing in it reads a
        device value on the host, DropPath factors and optimizer scalars come from device memory."""
        if teacher.patch_size != 16:
            # the zero-shot head stands the teacher's CLS embedding in for OpenAI CLIP's image tower against a 512-wide text
            # matrix; which stand-in a ViT-L/14 teacher should provide is not settled
            raise NotImplementedError(f"stage 3 runs a 16-pixel (clip_b16) teacher; got patch size {teacher.patch_size}")
        self.use_graph = use_graph
        self.graphs = GraphReplay()
        self.student, self.teacher = student, teacher
        self.core = student.core()
        self.core.sync_shadow(force=True)
        dev = self.core.arena.device
        self.W = cls_weight.detach().to(dev, F32).contiguous()
        self.b = cls_bias.detach().to(dev, F32).contiguous()
        self.text = text_features.detach().to(dev, F32).contiguous()
        self.mask_ratio, self.k, self.thr = mask_ratio, k, clip_threshold
        self.src_ratio, self.tgt_ratio, self.conf_weighted = src_ratio, tgt_ratio, conf_weighted
        self.optimizer = require_fused_optimizer(optimizer, self.core.arena, "Stage3Engine") or \
            FusedAdamW(self.core.arena, lr, weight_decay, betas)
        self.max_norm = None
        self.grad_sync = grad_sync
        # N > 1: the same fused NVLink step as stage 1 (the student's arena is the same; src_classifier is a separate, frozen
        # module, run_stage3.py:1193/:1264): gradient pushes overlapped with the step's last backward, then ub_adamw_nvls
        self.nvls = self._fused_step()
        self.loss = torch.zeros(1, device=dev, dtype=F32)
        self.loss_s = torch.zeros(1, device=dev, dtype=F32)
        self.loss_t = torch.zeros(1, device=dev, dtype=F32)
        self._full_idx = {}
        self.last = {}

    def _all_visible(self, B, N, dev):
        if (B, N) not in self._full_idx:
            self._full_idx[(B, N)] = torch.arange(N, device=dev, dtype=I32).repeat(B, 1).contiguous()
        return self._full_idx[(B, N)]

    def _classify(self, x_vis):
        B, N, D = x_vis.shape
        pooled = torch.empty(B, D, device=x_vis.device, dtype=F32)
        ops.meanpool_fwd(x_vis, pooled)                                            # pool_outputs, run_stage3.py:333-338
        logits = torch.empty(B, self.W.shape[0], device=x_vis.device, dtype=F32)
        ops.linear_small_fwd(pooled, self.W, self.b, logits)
        return pooled, logits

    def _backward_from_logits(self, state, pooled, dlogits, n_tokens, grad_sync=None):
        B, D = pooled.shape
        d_pooled = torch.empty(B, D, device=pooled.device, dtype=F32)
        ops.linear_small_bwd(pooled, self.W, dlogits, d_pooled, None, None)       # classifier frozen: dx only
        g_vis = torch.empty(B, n_tokens, D, device=pooled.device, dtype=F32)
        ops.meanpool_bwd(d_pooled, g_vis)
        self.core.run_backward(state, g_vis=g_vis, grad_sync=grad_sync)

    def forward_backward(self, videos_s, labels_s, videos_t, videos_t_aug: Optional[torch.Tensor] = None,
                         attn_override: Optional[torch.Tensor] = None, dp_override=None):
        """videos_t_aug: the train-augmented view of the target clips (args.return_aug_for_val, kinetics_sparse.py:174-180):
        the teacher attention and the masked committee views use it (`videos = cat([videos_s, videos_t_aug])`,
        run_stage3.py:413, :434-451, :499), while the full-token target pass and the zero-shot head see the plain view
        (:480, :557).  None = one view for everything.
        dp_override: dict slot -> DropPath factors [depth,2,B] for the four forwards ('s', 't', 0..k-1) (tests)."""
        core, teacher, k = self.core, self.teacher, self.k
        dev = videos_s.device
        Bs, Bt, N = videos_s.shape[0], videos_t.shape[0], core.N
        C = self.W.shape[0]
        dual = videos_t_aug is not None and videos_t_aug is not videos_t
        v_mask = videos_t_aug if dual else videos_t
        training = self.student.training

        def dp_for(slot, B):
            if dp_override is not None:
                return dp_override.get(slot)
            return core.drop_path.draw(B, slot=slot) if training else None          # model.train() covers every pass (:352)

        # ---- teacher on the target clips: attention map (augmented view) + CLS embedding for the zero-shot head (plain view)
        _, attn, patches_m = teacher.forward_features(v_mask)
        frames, P = attn.shape
        T = frames // Bt
        if dual:
            _, _, patches_t = teacher.forward_features(videos_t)
        else:
            patches_t = patches_m
        img = teacher.cls_features(frames, P)                                      # [Bt*T, 512]
        share = core.tubelet == teacher.kernel_size
        # ---- source clips, all tokens, with grad
        self.loss.zero_(); self.loss_s.zero_(); self.loss_t.zero_()
        xs, _, st_s = core.run_forward(videos_s, self._all_visible(Bs, N, dev), None, dp_for("s", Bs), False, True, want_clip=False)
        pooled_s, logits_s = self._classify(xs)
        dl_s = torch.empty_like(logits_s)
        ops.softmax_ce(logits_s, labels_s.to(I32), None, self.src_ratio / Bs, self.loss_s, dl_s)
        self._backward_from_logits(st_s, pooled_s, dl_s, N)
        # ---- target clips, all tokens, no grad
        xt, _, _ = core.run_forward(videos_t, self._all_visible(Bt, N, dev), patches_t if share else None, dp_for("t", Bt), False, False,
                                    want_clip=False)
        _, logits_full_t = self._classify(xt)
        # ---- committee masks and masked views
        n_vis = P - int(P * self.mask_ratio)
        mask = torch.empty(k, frames * P, device=dev, dtype=U8)
        vis = torch.empty(k, Bt, T * n_vis, device=dev, dtype=I32)
        ops.mask_select(attn if attn_override is None else attn_override, None, mask, vis, None, T, k, n_vis)
        logits_masked = torch.empty(k, Bt, C, device=dev, dtype=F32)
        base = (torch.arange(Bt, device=dev, dtype=I32) * N).view(Bt, 1)
        st_m = pooled_m = None
        for m in range(k):
            grad = m == k - 1                                                      # only the last member trains (run_stage3.py:606)
            abs_rows = (vis[m] + base).reshape(-1).contiguous() if share else None
            xm, _, st = core.run_forward(v_mask, vis[m].contiguous(), patches_m if share else None, dp_for(m, Bt), False, grad,
                                         want_clip=False, abs_rows=abs_rows)
            pooled, lg = self._classify(xm)
            logits_masked[m].copy_(lg)
            if grad:
                st_m, pooled_m = st, pooled
        # ---- zero-shot CLIP + MatchOrConf fusion
        clip_probs = torch.empty(Bt, C, device=dev, dtype=F32)
        ops.clip_zero_shot(img, self.text, clip_probs, T)
        msp = torch.empty(Bt, device=dev, dtype=F32)
        pseudo = torch.empty(Bt, device=dev, dtype=I32)
        sel = torch.empty(Bt, device=dev, dtype=U8)
        weight = torch.empty(Bt, device=dev, dtype=F32)
        ops.pseudo_label_fusion(logits_full_t, clip_probs, self.thr, self.conf_weighted, msp, pseudo, sel, weight)
        dl_t = torch.empty(Bt, C, device=dev, dtype=F32)
        ops.softmax_ce(logits_masked[k - 1], pseudo, weight, self.tgt_ratio / Bt, self.loss_t, dl_t)
        # the step's LAST backward: every gradient range it completes is final, so the NCCL range all-reduces overlap it
        self._backward_from_logits(st_m, pooled_m, dl_t, T * n_vis, grad_sync=self._backward_hook())
        self.loss.copy_(self.loss_s + self.loss_t)
        self.last = dict(attn=attn, masks=mask.view(k, frames, P).bool(), logits_s=logits_s, logits_full_t=logits_full_t,
                         logits_masked=logits_masked, clip_probs=clip_probs, sel_mask=sel.bool(), pseudo=pseudo, msp=msp)
        return self.loss

    def _step_body_dev(self, videos_s, labels_s, videos_t, videos_t_aug):
        self.optimizer.zero_grad()
        self.forward_backward(videos_s, labels_s, videos_t, videos_t_aug)
        self._update()

    def step(self, videos_s, labels_s, videos_t, videos_t_aug=None, private_inputs=False):
        """One update.  private_inputs: the batch lives in fresh tensors every step (a loader), so a graph keeps its own inputs."""
        self.optimizer.prepare_step(grad_scale=self.grad_scale)
        if videos_t_aug is videos_t:
            videos_t_aug = None
        if not self.use_graph:
            self._step_body_dev(videos_s, labels_s, videos_t, videos_t_aug)
            return self.loss
        key = (tuple(videos_s.shape), tuple(videos_t.shape), videos_t_aug is not None, labels_s.dtype, float(self.max_norm or 0.0),
               bool(self.student.training), self.mask_ratio)
        self.last = self.graphs.run(key, (videos_s, labels_s, videos_t, videos_t_aug), self._step_body_dev,
                                    state_fn=lambda: self.last, private=private_inputs)
        return self.loss


def _engine_for(model, teacher_model, src_classifier, optimizer, mask_ratio, args):
    student = model.module if hasattr(model, "module") else model
    teacher = teacher_model.module if hasattr(teacher_model, "module") else teacher_model
    cls = src_classifier.module if hasattr(src_classifier, "module") else src_classifier
    text = getattr(args, "text_features", None)
    if text is None:
        raise ValueError("stage 3 ('clip_matchORconf') needs args.text_features: the [n_classes, 512] text matrix that "
                         "utils.setup_clip (run_stage3.py:377-378) computes with the OpenAI-CLIP text tower — that package is not "
                         "part of the reference tree, so the caller supplies the matrix")
    held = student.__dict__.get("_ub_stage3_engine")
    if held is None or held[0] is not teacher or held[1] is not cls:
        gs = getattr(model, "grad_sync", None)
        if gs is not None:
            gs.arena = student.core().arena
        eng = Stage3Engine(student, teacher, cls.weight, cls.bias, text, mask_ratio=mask_ratio, k=2,
                           clip_threshold=float(getattr(args, "clip_threshold", 0.5)),
                           src_ratio=float(getattr(args, "class_loss_src_ratio_pl", 1.0)),
                           tgt_ratio=float(getattr(args, "class_loss_tgt_ratio", 1.0)),
                           conf_weighted=bool(getattr(args, "conf_weighted_loss", True)), grad_sync=gs,
                           optimizer=require_fused_optimizer(optimizer, student.core().arena, "train_one_epoch"),
                           use_graph=os.environ.get("UB_NO_GRAPH", "0") != "1")
        student.__dict__["_ub_stage3_engine"] = (teacher, cls, eng)
        return eng
    eng = held[2]
    if optimizer is not None:
        eng.set_optimizer(require_fused_optimizer(optimizer, eng.core.arena, "train_one_epoch"))
    eng.mask_ratio = mask_ratio
    return eng


def train_one_epoch(model: torch.nn.Module, data_loader: Iterable, data_loader_train_target: Iterable, optimizer=None, device=None,
                    epoch: int = 0, loss_scaler=None, max_norm: float = 0, log_writer=None, lr_scheduler=None, start_steps=None,
                    lr_schedule_values=None, wd_schedule_values=None, src_classifier=None, teacher_model=None,
                    clip_input_resolution=224, clip_loss_type="l2", clip_loss_ratio=0.5, mask_type="tube", mask_ratio=0.0,
                    use_wandb=False, args=None, classwise_thresholds=None, global_threshold=None):
    """Stage-3 `train_one_epoch` with the reference's signature (run_stage3.py:340-350) over Stage3Engine — the shipped
    configuration (configs/stage3_config.yaml): masking_type 'clip_attention', selection_strategy 'clip_matchORconf',
    train_masked, conf_weighted_loss, k = 2 committee members.

    Batches: source loader -> (videos_s, labels_s, ...) (:401-403); target loader -> (vid, vid_aug, label, name) when
    args.return_aug_for_val (kinetics_sparse.py:174-180, run_stage3.py:405-411) else (vid, label, name).  As in stage 1 the loop
    has no per-step `.item()`: loss / loss_class / loss_class_t / grad-norm are accumulated on the device and read at the end
    (non-finite loss is still fatal, :640-642).  args.text_features replaces utils.setup_clip (see _engine_for)."""
    if getattr(args, "masking_type", "clip_attention") != "clip_attention":
        raise NotImplementedError("the fused stage-3 path covers masking_type='clip_attention' (configs/stage3_config.yaml)")
    if getattr(args, "selection_strategy", "clip_matchORconf") != "clip_matchORconf":
        raise NotImplementedError("the fused stage-3 path covers selection_strategy='clip_matchORconf' (configs/stage3_config.yaml)")
    if not getattr(args, "train_masked", True) or getattr(args, "full_oracle", False):
        raise NotImplementedError("train_masked=True / full_oracle=False only (configs/stage3_config.yaml)")
    if getattr(args, "class_loss_src_ratio", 1.0) <= 0 or src_classifier is None:
        raise NotImplementedError("stage 3 trains through src_classifier (class_loss_src_ratio > 0, run_stage3.py:354-356 + :477)")
    if data_loader_train_target is None:
        raise ValueError("stage 3 needs the target-domain loader (run_stage3.py:405)")
    model.train()
    eng = _engine_for(model, teacher_model, src_classifier, optimizer, mask_ratio, args)
    eng.max_norm = float(max_norm) if max_norm else None
    opt = eng.optimizer
    dev = eng.core.arena.device
    start_steps = start_steps or 0
    acc = torch.zeros(4, device=dev)                                             # loss, loss_class (source), loss_class_t, grad_norm
    n = 0
    it_target = iter(data_loader_train_target)
    dual = bool(getattr(args, "return_aug_for_val", True))
    for step, batch in enumerate(data_loader):
        apply_schedule(opt, start_steps + step, lr_schedule_values, wd_schedule_values)   # run_stage3.py:383-396
        videos_s, labels_s = batch[0], batch[1]
        try:
            tb = next(it_target)
        except StopIteration:                                                    # :369-375
            it_target = iter(data_loader_train_target)
            tb = next(it_target)
        videos_t = tb[0].to(dev, non_blocking=True)
        videos_t_aug = tb[1].to(dev, non_blocking=True) if dual else None
        loss = eng.step(videos_s.to(dev, non_blocking=True), labels_s.to(dev, non_blocking=True), videos_t, videos_t_aug,
                        private_inputs=True)
        acc += torch.cat([loss, eng.loss_s, eng.loss_t, opt.grad_norm(eng.grad_scale)])
        n += 1
        if lr_scheduler is not None:
            lr_scheduler.step_update(start_steps + step)
    stats = acc / max(n, 1)
    if torch.distributed.is_initialized() and torch.distributed.get_world_size() > 1:
        torch.distributed.all_reduce(stats)                                      # metric_logger.synchronize_between_processes (:705)
        stats /= torch.distributed.get_world_size()
    loss_avg, ls_avg, lt_avg, gn_avg = stats.tolist()
    exit_if_not_finite(loss_avg)                                                 # :640-642
    return {"loss": loss_avg, "loss_class": ls_avg, "loss_class_t": lt_avg, "loss_scale": 1.0, **schedule_stats(opt),
            "grad_norm": gn_avg}
