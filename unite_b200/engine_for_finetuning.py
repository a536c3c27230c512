"""Stage-2 supervised fine-tuning step with the reference's `train_one_epoch` signature
(src/engines/engine_for_finetuning.py:48-54; non-DeepSpeed branch :116-127).

    samples, targets = mixup_fn(samples, targets)             engine_for_finetuning.py:86-87 (when mixup_fn is given)
    loss = criterion(model(samples), targets) / update_freq   engine_for_finetuning.py:37-40, :119
    backward every micro-step, optimizer every update_freq     :120-126
The loss and its gradient come from one fused kernel: ub_softmax_ce for CrossEntropyLoss(), ub_soft_target_ce for the mixup
and label-smoothing criteria (mixup.resolve_loss).  Mixup / cutmix are drawn on the host exactly as timm draws them and applied
on the device inside the im2col (ub_patchify_mix), so the caller's clip is never written.  The model's backward is the explicit
one in finetune_core.py; gradients accumulate in the parameter arena across micro-steps like `.grad` does in torch.
    model_ema.update(model)                                   engine_for_finetuning.py:126-127 (after every optimizer update)
With `model_ema` (ema.ModelEma or timm's ModelEma) the EMA arena is updated by one fused kernel (ub_ema_update) right after the
optimizer, inside the CUDA graph of the step.
"""
import math
import sys
from typing import Iterable, Optional

import torch

from . import ops
from .ema import resolve_model_ema
from .engine import FusedAdamW, require_fused_optimizer
from .mixup import NO_MIX, MixBuffer, draw, resolve_loss


def train_class_batch(model, samples, target, criterion):
    """engine_for_finetuning.py:37-40, as written there: the model's forward is one autograd node over the fused kernels
    (finetune_core._FinetuneFn), so `loss.backward()` on the returned loss accumulates into the parameter arena like any
    torch module.  train_one_epoch below uses the fused loss+gradient kernel instead (no autograd, no host sync)."""
    outputs = model(samples)
    loss = criterion(outputs, target)
    return loss, outputs


def _default_optimizer(net):
    """Only when the caller passes optimizer=None: one FusedAdamW per model, kept on the model object."""
    opt = net.__dict__.get("_ub_default_optimizer")
    if opt is None:
        opt = FusedAdamW(net.core().arena, lr=1e-3, weight_decay=0.05, betas=(0.9, 0.999))
        net.__dict__["_ub_default_optimizer"] = opt
    return opt


def finetune_step(model, samples, targets, loss_acc, scale=1.0, grad_sync=None, mix=None):
    """One micro-step: forward, CE, backward.  Adds scale * mean CE to loss_acc (fp32 [1]).  Returns logits.
    grad_sync: pass the model's GradSync on the micro-step that is followed by the optimizer step — its range all-reduces then
    overlap this backward.
    mix: None (plain CE), or a mixup.MixBuffer holding this step's draw on the device: the clip is mixed on its way into the
    im2col (mix.clip, None for label smoothing alone) and the loss is the soft-target CE of the mixed, smoothed target."""
    net = model.module if hasattr(model, "module") else model
    core = net.core()
    dp = core.drop_path.draw(samples.shape[0]) if net.training else None       # modeling_finetune.py:42-50 (device-side draws)
    logits, state = core.run_forward(samples, dp, save=True, mix=None if mix is None else mix.clip)
    B = logits.shape[0]
    dlogits = torch.empty_like(logits)
    if mix is None:
        ops.softmax_ce(logits, targets.to(torch.int32), None, scale / B, loss_acc, dlogits)
    else:
        ops.soft_target_ce(logits, targets.to(torch.int32), mix.target, scale / B, loss_acc, dlogits)
    core.run_backward(state, dlogits, grad_sync=grad_sync)
    return logits


class Stage2Engine:
    """One whole stage-2 update (update_freq == 1): zero the gradient arena, forward, CE, backward, gradient all-reduce, grad-norm +
    layer-decay AdamW — engine_for_finetuning.py:116-127 — replayed from a CUDA graph after two eager steps (engine.GraphReplay):
    the ~750 launches of the all-token step then cost one launch.  DropPath draws come from the device-side generator, the
    optimizer's lr / wd / bias corrections from device memory (FusedAdamW.prepare_step), so nothing in the body depends on the
    host.  The running sums train_one_epoch reports (loss, correct predictions, grad-norm) are accumulated on the device inside
    the step.  model_ema (ema.ModelEma or timm's ModelEma): its arena is updated right after AdamW, in the same graph; every rank
    of a data-parallel run updates its own EMA from the same replicated weights."""

    def __init__(self, model, optimizer: FusedAdamW, grad_sync=None, use_graph: bool = False, model_ema=None):
        from .engine import GraphReplay
        self.ema = resolve_model_ema(model_ema, model)
        self.model = model
        self.net = model.module if hasattr(model, "module") else model
        self.core = self.net.core()
        if self.ema is not None:
            self.ema.ema_net.core()                         # the EMA's arena exists before any step is captured
        self.optimizer = require_fused_optimizer(optimizer, self.core.arena, "Stage2Engine")
        self.grad_sync = grad_sync
        self.use_graph = use_graph
        self.max_norm = None
        dev = self.core.arena.device
        self.loss = torch.zeros(1, device=dev)
        self.stats = torch.zeros(3, device=dev)             # running sums: loss, correct predictions, grad-norm
        self.graphs = GraphReplay()
        self.logits = None
        self._mix_bufs = {}                                 # loss kind -> MixBuffer (fixed addresses the graphs read)
        self._mix = None                                    # the buffer of the current step, None for plain CE

    def _body(self, samples, targets):
        self.optimizer.zero_grad()
        self.loss.zero_()
        logits = finetune_step(self.model, samples, targets, self.loss, scale=1.0, grad_sync=self.grad_sync, mix=self._mix)
        if self.grad_sync is not None:
            self.grad_sync.all_reduce(self.core.arena.grads)
        self.optimizer.step_dev(max_norm=self.max_norm)
        if self.ema is not None:
            self.ema.update(self.model)
        scale = 1.0 / self.grad_sync.world if self.grad_sync is not None else 1.0
        self.stats += torch.cat([self.loss, (logits.argmax(-1) == targets).sum().float().view(1), self.optimizer.grad_norm(scale)])
        self.logits = logits

    def step(self, samples, targets, private_inputs=False, mix=None, smoothing=None):
        """samples fp32 [B,3,T,H,W], targets integer [B], both on the device.  Returns the device loss tensor [1].
        private_inputs: the batch lives in fresh tensors every step (a loader), so the graph keeps its own static inputs.
        smoothing None: plain CE.  smoothing s: soft-target CE with label smoothing s, and with mix (a mixup.MixDraw, NO_MIX for a
        batch the draw left unmixed) the clip is mixed as drawn.  The draw is uploaded to device memory before the step, so every
        replay of the one graph per loss kind reads its own draw."""
        if mix is not None and smoothing is None:
            raise ValueError("Stage2Engine.step: a mixup draw needs the soft-target loss (pass smoothing=)")
        scale = 1.0 / self.grad_sync.world if self.grad_sync is not None else 1.0
        self.optimizer.prepare_step(grad_scale=scale)
        kind = "ce" if smoothing is None else ("mix" if mix is not None else "smooth")
        self._mix = None
        if kind != "ce":
            if kind not in self._mix_bufs:
                self._mix_bufs[kind] = MixBuffer(self.core.arena.device, mix_clips=kind == "mix")
            self._mix = self._mix_bufs[kind]
            self._mix.upload((mix or NO_MIX).packed(smoothing, self.core.C))
        if not self.use_graph:
            self._body(samples, targets)
            return self.loss
        key = (tuple(samples.shape), samples.dtype, targets.dtype, float(self.max_norm or 0.0), bool(self.net.training), kind)
        if self.ema is not None:
            key += (("ema", self.ema.decay),)               # the decay is a launch argument recorded in the graph
        self.logits = self.graphs.run(key, (samples, targets), self._body, state_fn=lambda: self.logits, private=private_inputs)
        return self.loss


def _stage2_engine(model, net, optimizer, gs, model_ema=None):
    held = net.__dict__.get("_ub_stage2_engine")
    held_ema = None if held is None or held.ema is None else held.ema.source
    if held is None or held.optimizer is not optimizer or held.grad_sync is not gs or held_ema is not model_ema:
        import os
        held = Stage2Engine(model, optimizer, grad_sync=gs, use_graph=os.environ.get("UB_NO_GRAPH", "0") != "1", model_ema=model_ema)
        net.__dict__["_ub_stage2_engine"] = held
    return held


def train_one_epoch(model: torch.nn.Module, criterion=None, data_loader: Iterable = (), optimizer=None, device=None, epoch: int = 0,
                    loss_scaler=None, max_norm: float = 0, model_ema=None, mixup_fn=None, log_writer=None, start_steps=None,
                    lr_schedule_values=None, wd_schedule_values=None, num_training_steps_per_epoch=None, update_freq=None,
                    num_epochs=None, train_head_only=False, wandb_run=None, args=None):
    """mixup_fn: a mixup.Mixup (or the reference's timm Mixup) in batch mode, drawn once per loader batch; criterion: see
    mixup.resolve_loss.  With mixup_fn the returned dict has no class_acc (the reference logs None there).
    model_ema: an ema.ModelEma (or the reference's timm ModelEma) of this model, updated once per optimizer update (see
    ema.resolve_model_ema for what is refused)."""
    ema = resolve_model_ema(model_ema, model)
    if train_head_only:
        raise NotImplementedError("head-only training is not implemented in the fused stage-2 loop")
    smoothing = resolve_loss(criterion, mixup_fn)
    model.train(True)
    net = model.module if hasattr(model, "module") else model
    core = net.core()
    dev = core.arena.device
    if mixup_fn is not None and mixup_fn.num_classes != core.C:
        raise ValueError(f"mixup_fn.num_classes={mixup_fn.num_classes} differs from the model's {core.C} classes")
    update_freq = update_freq or 1
    start_steps = start_steps or 0
    optimizer = require_fused_optimizer(optimizer, core.arena, "train_one_epoch") or _default_optimizer(net)
    gs = getattr(model, "grad_sync", None)
    if update_freq == 1:
        return _train_one_epoch_graphed(model, net, data_loader, optimizer, gs, max_norm, start_steps, lr_schedule_values,
                                        wd_schedule_values, num_training_steps_per_epoch, mixup_fn, smoothing, model_ema)
    mix = None if smoothing is None else MixBuffer(dev, mix_clips=mixup_fn is not None)
    loss_sum = torch.zeros(1, device=dev)
    loss_acc = torch.zeros(1, device=dev)
    correct = torch.zeros(1, device=dev)
    gn_sum = torch.zeros(1, device=dev)
    seen = 0
    n_updates = 0
    data_iter_step = -1
    optimizer.zero_grad()
    for data_iter_step, batch in enumerate(data_loader):
        samples, targets = batch[0], batch[1]
        step = data_iter_step // update_freq
        if num_training_steps_per_epoch is not None and step >= num_training_steps_per_epoch:
            continue                                                               # engine_for_finetuning.py:71-72
        it = start_steps + step
        if data_iter_step % update_freq == 0:
            for group in optimizer.param_groups:                                   # engine_for_finetuning.py:76-81
                if lr_schedule_values is not None:
                    group["lr"] = lr_schedule_values[min(it, len(lr_schedule_values) - 1)] * group.get("lr_scale", 1.0)
                if wd_schedule_values is not None and group["weight_decay"] > 0:
                    group["weight_decay"] = wd_schedule_values[min(it, len(wd_schedule_values) - 1)]
        if mix is not None:
            mix.upload((draw(mixup_fn, samples.shape) if mixup_fn is not None else NO_MIX).packed(smoothing, core.C))
        samples = samples.to(dev, non_blocking=True)
        targets = targets.to(dev, non_blocking=True)
        loss_acc.zero_()
        last_micro = (data_iter_step + 1) % update_freq == 0
        logits = finetune_step(model, samples, targets, loss_acc, scale=1.0 / update_freq, grad_sync=gs if last_micro else None,
                               mix=mix)
        loss_sum += loss_acc * update_freq
        correct += (logits.argmax(-1) == targets).sum()
        seen += samples.shape[0]
        if (data_iter_step + 1) % update_freq == 0:
            scale = gs.all_reduce(core.arena.grads) if gs is not None else 1.0
            optimizer.step(grad_scale=scale, max_norm=float(max_norm) if max_norm else None)   # loss_scaler(..., clip_grad=max_norm)
            gn_sum += optimizer.grad_norm(scale)
            n_updates += 1
            optimizer.zero_grad()
            if ema is not None:
                ema.update(model)                                                  # engine_for_finetuning.py:126-127
    n = max(1, data_iter_step + 1)
    loss_avg = (loss_sum / n).item()
    if not math.isfinite(loss_avg):
        print("Loss is {}, stopping training".format(loss_avg))
        sys.exit(1)
    lrs = [g["lr"] for g in optimizer.param_groups]
    wds = [g["weight_decay"] for g in optimizer.param_groups if g["weight_decay"] > 0]
    stats = {"loss": loss_avg, "class_acc": (correct / max(seen, 1)).item(), "loss_scale": 1.0, "lr": max(lrs), "min_lr": min(lrs),
             "weight_decay": wds[0] if wds else None, "grad_norm": (gn_sum / max(1, n_updates)).item()}
    if mixup_fn is not None:
        del stats["class_acc"]
    return stats


def _train_one_epoch_graphed(model, net, data_loader, optimizer, gs, max_norm, start_steps, lr_schedule_values, wd_schedule_values,
                             num_training_steps_per_epoch, mixup_fn=None, smoothing=None, model_ema=None):
    """update_freq == 1 (the shipped stage-2 recipe): every loader batch is one whole update, run through Stage2Engine (CUDA-graph
    replay).  Same schedule handling and return dict as the general loop above."""
    eng = _stage2_engine(model, net, optimizer, gs, model_ema)
    eng.max_norm = float(max_norm) if max_norm else None
    eng.stats.zero_()
    dev = eng.core.arena.device
    seen = n = 0
    for data_iter_step, batch in enumerate(data_loader):
        if num_training_steps_per_epoch is not None and data_iter_step >= num_training_steps_per_epoch:
            continue                                                               # engine_for_finetuning.py:71-72
        it = start_steps + data_iter_step
        for group in optimizer.param_groups:                                       # engine_for_finetuning.py:76-81
            if lr_schedule_values is not None:
                group["lr"] = lr_schedule_values[min(it, len(lr_schedule_values) - 1)] * group.get("lr_scale", 1.0)
            if wd_schedule_values is not None and group["weight_decay"] > 0:
                group["weight_decay"] = wd_schedule_values[min(it, len(wd_schedule_values) - 1)]
        mix = draw(mixup_fn, batch[0].shape) if mixup_fn is not None else None
        eng.step(batch[0].to(dev, non_blocking=True), batch[1].to(dev, non_blocking=True), private_inputs=True, mix=mix,
                 smoothing=smoothing)
        seen += batch[0].shape[0]
        n += 1
    loss_sum, correct, gn_sum = eng.stats.tolist()
    loss_avg = loss_sum / max(1, n)
    if not math.isfinite(loss_avg):
        print("Loss is {}, stopping training".format(loss_avg))
        sys.exit(1)
    lrs = [g["lr"] for g in optimizer.param_groups]
    wds = [g["weight_decay"] for g in optimizer.param_groups if g["weight_decay"] > 0]
    stats = {"loss": loss_avg, "class_acc": correct / max(seen, 1), "loss_scale": 1.0, "lr": max(lrs), "min_lr": min(lrs),
             "weight_decay": wds[0] if wds else None, "grad_norm": gn_sum / max(1, n)}
    if mixup_fn is not None:
        del stats["class_acc"]                                                     # the reference's class_acc = None under mixup
    return stats


# ---------------------------------------------------------------------------------------------------------------------
# Evaluation path (SURVEY.md §8 row f4): all-token inference + multi-crop / multi-segment score merge
# (src/engines/engine_for_finetuning.py:175-351).  The forward is the inference form of the same kernels (S = all
# tokens, no activations kept); metrics stay on the device until the end of the loop (one sync per loader, not per batch).
# ---------------------------------------------------------------------------------------------------------------------
def accuracy(output: torch.Tensor, target: torch.Tensor, topk=(1,)):
    """timm.utils.accuracy (timm 0.4.12, pinned by environment.yaml; the package is not under /root/reference): top-k
    precision in percent over the batch."""
    maxk = min(max(topk), output.shape[1])
    pred = output.topk(maxk, 1, True, True).indices.t()
    correct = pred.eq(target.reshape(1, -1).expand_as(pred))
    return [correct[:min(k, maxk)].reshape(-1).float().sum(0) * 100.0 / target.shape[0] for k in topk]


def compute_ece(softmaxes: torch.Tensor, labels: torch.Tensor, n_bins: int = 15) -> float:
    """Expected calibration error.  The reference imports it from src/knn.py, which is missing from the tree (SURVEY.md
    §0.1): this is the standard equal-width 15-bin estimator sum_b |acc_b - conf_b| * n_b / n."""
    conf, pred = softmaxes.max(dim=1)
    acc = pred.eq(labels).float()
    edges = torch.linspace(0, 1, n_bins + 1, device=softmaxes.device)
    ece = torch.zeros((), device=softmaxes.device)
    for lo, hi in zip(edges[:-1], edges[1:]):
        m = (conf > lo) & (conf <= hi)
        n = m.float().sum()
        if n > 0:
            ece = ece + (acc[m].mean() - conf[m].mean()).abs() * n / conf.numel()
    return float(ece)


def _gather_all(t: torch.Tensor) -> torch.Tensor:
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return t
    parts = [torch.zeros_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(parts, t.contiguous())
    return torch.cat(parts)


@torch.no_grad()
def validation_one_epoch(data_loader, model, device, save_preds_path=None):
    """engine_for_finetuning.py:175-236: returns ({loss, acc1, acc5}, ece)."""
    model.eval()
    net = model.module if hasattr(model, "module") else model
    dev = net.core().arena.device
    probs, labels, losses = [], [], []
    for batch in data_loader:
        videos, target = batch[0].to(dev, non_blocking=True), batch[1].to(dev, non_blocking=True)
        output = model(videos)
        losses.append(torch.nn.functional.cross_entropy(output, target.long(), reduction="sum"))
        probs.append(torch.softmax(output, dim=1))
        labels.append(target.long())
    probs, labels = _gather_all(torch.cat(probs)), _gather_all(torch.cat(labels))
    loss = _gather_all(torch.stack(losses).sum().reshape(1)).sum() / labels.numel()
    acc1, acc5 = accuracy(probs, labels, topk=(1, 5))
    ece = compute_ece(probs, labels)
    print(f"Expected Calibration Error (ECE): {ece:.4f}")
    if save_preds_path is not None:
        import os
        import numpy as np
        os.makedirs(save_preds_path, exist_ok=True)
        np.save(os.path.join(save_preds_path, "preds.npy"), probs.argmax(1).cpu().numpy())
        np.save(os.path.join(save_preds_path, "labels.npy"), labels.cpu().numpy())
    stats = {"loss": loss.item(), "acc1": acc1.item(), "acc5": acc5.item()}
    print("* Acc@1 {acc1:.3f} Acc@5 {acc5:.3f} loss {loss:.3f}".format(**stats))
    return stats, ece


@torch.no_grad()
def final_test(data_loader, model, device, file):
    """engine_for_finetuning.py:241-296: per-view logits written as `<id> <logits list> <label> <chunk> <split>` lines (the
    format `merge` parses), first line `<acc1>, <acc5>` of the last batch like the reference.  batch = (videos, target,
    ids, chunk_nb, split_nb)."""
    model.eval()
    net = model.module if hasattr(model, "module") else model
    dev = net.core().arena.device
    lines, probs, labels, losses = [], [], [], []
    acc1 = acc5 = torch.zeros(())
    for batch in data_loader:
        videos, target, ids, chunk_nb, split_nb = batch[0], batch[1], batch[2], batch[3], batch[4]
        videos, target = videos.to(dev, non_blocking=True), target.to(dev, non_blocking=True)
        output = model(videos)
        losses.append(torch.nn.functional.cross_entropy(output, target.long(), reduction="sum"))
        out_host, tgt_host = output.float().cpu(), target.cpu()
        for i in range(out_host.shape[0]):
            lines.append("{} {} {} {} {}\n".format(ids[i], str(out_host[i].numpy().tolist()), str(int(tgt_host[i])),
                                                   str(int(chunk_nb[i])), str(int(split_nb[i]))))
        acc1, acc5 = accuracy(output, target.long(), topk=(1, 5))
        probs.append(torch.softmax(output, dim=1))
        labels.append(target.long())
    probs, labels = torch.cat(probs), torch.cat(labels)
    ece = compute_ece(probs, labels)
    print(f"Expected Calibration Error (ECE): {ece:.4f}")
    with open(file, "w") as f:
        f.write("{}, {}\n".format(acc1, acc5))
        f.writelines(lines)
    a1, a5 = accuracy(probs, labels, topk=(1, 5))
    stats = {"loss": (torch.stack(losses).sum() / labels.numel()).item(), "acc1": a1.item(), "acc5": a5.item()}
    print("* Acc@1 {acc1:.3f} Acc@5 {acc5:.3f} loss {loss:.3f}".format(**stats))
    return stats, ece


def compute_video(item):
    """engine_for_finetuning.py:343-351: mean of the per-view softmax scores of one video -> (pred, top1, top5, label)."""
    import numpy as np
    _, _, data, label = item
    feat = np.mean(np.stack(data), axis=0)
    pred = int(np.argmax(feat))
    return [pred, float(pred == int(label)), float(int(label) in np.argsort(-feat)[:5]), int(label)]


def merge(eval_path, num_tasks):
    """engine_for_finetuning.py:299-341: read the per-rank `<rank>.txt` files of final_test, softmax each view, drop repeated
    (chunk, split) views of a video, average the rest, return (top-1 %, top-5 %)."""
    import os
    import numpy as np
    feats, label_of, seen = {}, {}, {}
    for r in range(num_tasks):
        with open(os.path.join(eval_path, str(r) + ".txt")) as f:
            rows = f.readlines()[1:]
        for line in rows:
            line = line.strip()
            name, rest = line.rsplit("[", maxsplit=1)
            vec, tail = rest.rsplit("]", maxsplit=1)
            _, label, chunk_nb, split_nb = tail.split(" ")[:4]
            x = np.array([float(t) for t in vec.split(",")], dtype=np.float64)
            e = np.exp(x - x.max())
            view = chunk_nb + split_nb
            if view in seen.setdefault(name, []):
                continue
            seen[name].append(view)
            feats.setdefault(name, []).append(e / e.sum())
            label_of[name] = label
    ans = [compute_video([i, n, feats[n], label_of[n]]) for i, n in enumerate(feats)]
    return float(np.mean([a[1] for a in ans])) * 100, float(np.mean([a[2] for a in ans])) * 100
