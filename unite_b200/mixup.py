"""Stage-2 mixup / cutmix and label smoothing (run_stage2.py: Mixup when mixup, cutmix or cutmix_minmax is set, then
SoftTargetCrossEntropy / LabelSmoothingCrossEntropy / CrossEntropyLoss around :702; engine_for_finetuning.py:86-87).

The reference takes these from timm 0.4.12 (pinned by environment.yaml).  The host side here is timm's: the same numpy global-RNG
draws in the same order, so with the same np.random.seed the package draws exactly what the reference draws.  The mixing itself
runs on the device, fused into the stage-2 im2col (ub_patchify_mix), and the soft target is built inside the loss kernel
(ub_soft_target_ce): neither the mixed clip nor the [B, C] target is ever stored, and the caller's clip is never written.

Only batch mode (one draw per batch, clip b mixed with clip B-1-b) is supported; it is timm's default and the mode every
recipe of the lineage uses.
"""
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

__all__ = ["Mixup", "SoftTargetCrossEntropy", "LabelSmoothingCrossEntropy", "MixDraw", "draw", "clip_box", "cutmix_bbox_and_lam",
           "rand_bbox", "rand_bbox_minmax", "resolve_loss", "MixBuffer"]


# ---- timm 0.4.12 timm/data/mixup.py: box draws ------------------------------------------------------------------------------------
def rand_bbox(img_shape, lam, margin=0., count=None):
    ratio = np.sqrt(1 - lam)
    img_h, img_w = img_shape[-2:]
    cut_h, cut_w = int(img_h * ratio), int(img_w * ratio)
    margin_y, margin_x = int(margin * cut_h), int(margin * cut_w)
    cy = np.random.randint(0 + margin_y, img_h - margin_y, size=count)
    cx = np.random.randint(0 + margin_x, img_w - margin_x, size=count)
    yl = np.clip(cy - cut_h // 2, 0, img_h)
    yh = np.clip(cy + cut_h // 2, 0, img_h)
    xl = np.clip(cx - cut_w // 2, 0, img_w)
    xh = np.clip(cx + cut_w // 2, 0, img_w)
    return yl, yh, xl, xh


def rand_bbox_minmax(img_shape, minmax, count=None):
    assert len(minmax) == 2
    img_h, img_w = img_shape[-2:]
    cut_h = np.random.randint(int(img_h * minmax[0]), int(img_h * minmax[1]), size=count)
    cut_w = np.random.randint(int(img_w * minmax[0]), int(img_w * minmax[1]), size=count)
    yl = np.random.randint(0, img_h - cut_h, size=count)
    xl = np.random.randint(0, img_w - cut_w, size=count)
    yu = yl + cut_h
    xu = xl + cut_w
    return yl, yu, xl, xu


def cutmix_bbox_and_lam(img_shape, lam, ratio_minmax=None, correct_lam=True, count=None):
    if ratio_minmax is not None:
        yl, yu, xl, xu = rand_bbox_minmax(img_shape, ratio_minmax, count=count)
    else:
        yl, yu, xl, xu = rand_bbox(img_shape, lam, count=count)
    if correct_lam or ratio_minmax is not None:
        bbox_area = (yu - yl) * (xu - xl)
        lam = 1. - bbox_area / float(img_shape[-2] * img_shape[-1])
    return (yl, yu, xl, xu), lam


class Mixup:
    """timm 0.4.12 Mixup, batch mode: constructor, attributes and _params_per_batch as there.  Mixing is not done here but inside
    engine_for_finetuning.train_one_epoch (draw() below, then ub_patchify_mix); the loop accepts any object with these attributes,
    the reference's own Mixup included."""

    def __init__(self, mixup_alpha=1., cutmix_alpha=0., cutmix_minmax=None, prob=1.0, switch_prob=0.5, mode='batch', correct_lam=True,
                 label_smoothing=0.1, num_classes=1000):
        if mode != 'batch':
            raise NotImplementedError(f"Mixup mode {mode!r}: only 'batch' mode (one draw per batch) is implemented")
        self.mixup_alpha = mixup_alpha
        self.cutmix_alpha = cutmix_alpha
        self.cutmix_minmax = cutmix_minmax
        if self.cutmix_minmax is not None:
            assert len(self.cutmix_minmax) == 2
            self.cutmix_alpha = 1.0            # timm: cutmix alpha forced to 1.0 when minmax is active
        self.mix_prob = prob
        self.switch_prob = switch_prob
        self.label_smoothing = label_smoothing
        self.num_classes = num_classes
        self.mode = mode
        self.correct_lam = correct_lam
        self.mixup_enabled = True

    def _params_per_batch(self):
        lam = 1.
        use_cutmix = False
        if self.mixup_enabled and np.random.rand() < self.mix_prob:
            if self.mixup_alpha > 0. and self.cutmix_alpha > 0.:
                use_cutmix = np.random.rand() < self.switch_prob
                lam_mix = np.random.beta(self.cutmix_alpha, self.cutmix_alpha) if use_cutmix else \
                    np.random.beta(self.mixup_alpha, self.mixup_alpha)
            elif self.mixup_alpha > 0.:
                lam_mix = np.random.beta(self.mixup_alpha, self.mixup_alpha)
            elif self.cutmix_alpha > 0.:
                use_cutmix = True
                lam_mix = np.random.beta(self.cutmix_alpha, self.cutmix_alpha)
            else:
                assert False, "One of mixup_alpha > 0., cutmix_alpha > 0., cutmix_minmax not None should be true."
            lam = float(lam_mix)
        return lam, use_cutmix

    def __call__(self, x, target):
        raise NotImplementedError("unite_b200 mixes clips on the device inside engine_for_finetuning.train_one_epoch: pass this "
                                  "object there as mixup_fn")


# ---- timm 0.4.12 timm/loss/cross_entropy.py: the criterion modules (train_class_batch goes through their forward) ---------------
class LabelSmoothingCrossEntropy(nn.Module):
    def __init__(self, smoothing=0.1):
        super().__init__()
        assert smoothing < 1.0
        self.smoothing = smoothing
        self.confidence = 1. - smoothing

    def forward(self, x, target):
        logprobs = F.log_softmax(x, dim=-1)
        nll_loss = -logprobs.gather(dim=-1, index=target.unsqueeze(1))
        nll_loss = nll_loss.squeeze(1)
        smooth_loss = -logprobs.mean(dim=-1)
        loss = self.confidence * nll_loss + self.smoothing * smooth_loss
        return loss.mean()


class SoftTargetCrossEntropy(nn.Module):
    def __init__(self):
        super().__init__()

    def forward(self, x, target):
        loss = torch.sum(-target * F.log_softmax(x, dim=-1), dim=-1)
        return loss.mean()


# ---- the draw of one batch, mapped onto the clip --------------------------------------------------------------------------------
Box = Tuple[Tuple[int, int], Tuple[int, int], Tuple[int, int]]


def clip_box(shape, yl, yh, xl, xh) -> Box:
    """Half-open (T, H, W) ranges of a [B,C,T,H,W] clip that timm's `x[:, :, yl:yh, xl:xh] = x.flip(0)[:, :, yl:yh, xl:xh]`
    overwrites.  timm draws (yl, yh) from H and (xl, xh) from W (img_shape[-2:]), but on a 5-D clip the slice indexes the T axis
    with the H range and the H axis with the W range, and keeps W whole; Python clamps each range to its axis.  The reference's
    stage-2 loop runs exactly this on its [B,3,T,H,W] clips, so the package reproduces it (DESIGN.md §8).  This is the only
    place that knows the mapping; the kernel takes any box on the three axes."""
    _, _, T, H, W = shape

    def rng(lo, hi, n):
        lo, hi = min(int(lo), n), min(int(hi), n)
        return lo, max(lo, hi)
    return rng(yl, yh, T), rng(xl, xh, H), (0, W)


@dataclass(frozen=True)
class MixDraw:
    """One batch's draw.  lam: the Beta draw (1.0 when nothing is mixed); target_lam: the weight of each clip's own label in the
    target (the box-corrected lam under cutmix, else lam)."""
    apply: bool
    lam: float
    use_cutmix: bool
    box: Box
    target_lam: float

    def packed(self, smoothing: float, num_classes: int):
        """The 16 fp32 of the device buffer: ub_patchify_mix's {apply, lam, 1 - lam, use_cutmix, t0, t1, h0, h1, w0, w1}, then
        ub_soft_target_ce's {lam, on, off}, padding.  1 - lam and the smoothing values are computed in double, as timm does."""
        off = smoothing / num_classes
        on = 1. - smoothing + off
        lam = self.target_lam
        (t0, t1), (h0, h1), (w0, w1) = self.box
        return [float(self.apply), lam, 1. - lam, float(self.use_cutmix), t0, t1, h0, h1, w0, w1, lam, on, off, 0., 0., 0.]


NO_MIX = MixDraw(False, 1.0, False, ((0, 0), (0, 0), (0, 0)), 1.0)


def draw(mixup_fn, shape) -> MixDraw:
    """timm Mixup._mix_batch's draws for a clip batch of `shape` [B,C,T,H,W]: mixup_fn._params_per_batch(), then the box through
    cutmix_bbox_and_lam under cutmix.  Raises (before any draw) for an odd batch or a mode other than 'batch'."""
    if getattr(mixup_fn, "mode", "batch") != "batch":
        raise NotImplementedError(f"mixup mode {mixup_fn.mode!r}: only 'batch' mode is implemented")
    if len(shape) != 5:
        raise ValueError(f"mixup: a [B,C,T,H,W] clip batch expected, got shape {tuple(shape)}")
    if shape[0] % 2:
        raise ValueError(f"mixup: the batch size must be even (clip b is mixed with clip B-1-b), got {shape[0]}")
    lam, use_cutmix = mixup_fn._params_per_batch()
    if lam == 1.:
        return NO_MIX
    if use_cutmix:
        (yl, yh, xl, xh), lam_c = cutmix_bbox_and_lam(shape, lam, ratio_minmax=mixup_fn.cutmix_minmax, correct_lam=mixup_fn.correct_lam)
        return MixDraw(True, lam, True, clip_box(shape, yl, yh, xl, xh), float(lam_c))
    return MixDraw(True, lam, False, ((0, 0), (0, 0), (0, 0)), lam)


def resolve_loss(criterion, mixup_fn) -> Optional[float]:
    """Which stage-2 loss the fused step runs for (criterion, mixup_fn), as run_stage2.py:702 pairs them.  None: plain CE
    (ub_softmax_ce, the path without mixup / smoothing); a float s: soft-target CE with label smoothing s (ub_soft_target_ce).
    The criterion modules are recognised by class name, so timm's own classes are accepted too; their forward is never called."""
    if mixup_fn is not None and getattr(mixup_fn, "mode", "batch") != "batch":
        raise NotImplementedError(f"mixup mode {mixup_fn.mode!r}: only 'batch' mode is implemented")
    name = type(criterion).__name__
    plain = criterion is None or (isinstance(criterion, nn.CrossEntropyLoss) and criterion.label_smoothing == 0.0
                                  and criterion.weight is None and criterion.reduction == "mean")
    if mixup_fn is not None:
        if plain or name == "SoftTargetCrossEntropy":          # torch >= 1.10 CE on probability targets is the same loss
            return float(mixup_fn.label_smoothing)
        raise NotImplementedError(f"with mixup_fn the fused stage-2 loss is SoftTargetCrossEntropy (or CrossEntropyLoss()), got {name}")
    if plain:
        return None
    if name == "LabelSmoothingCrossEntropy":
        return float(criterion.smoothing)
    if isinstance(criterion, nn.CrossEntropyLoss) and criterion.weight is None and criterion.reduction == "mean":
        return float(criterion.label_smoothing)
    raise NotImplementedError("without mixup_fn the fused stage-2 loss is CrossEntropyLoss() or label smoothing "
                              f"(LabelSmoothingCrossEntropy(s), CrossEntropyLoss(label_smoothing=s)), got {name}")


class MixBuffer:
    """Device copy of one step's packed draw (MixDraw.packed): `clip` feeds ub_patchify_mix, `target` ub_soft_target_ce.  Each
    upload is one async copy from a ring of pinned slots, as FusedAdamW.prepare_step uploads its scalars: a slot is rewritten
    only after the copy that last read it has executed, since a host that queues graph replays can be many steps ahead of the
    device.  Both views keep their addresses, so a captured step reads each fresh draw on replay.  mix_clips=False (label
    smoothing without mixup_fn): `clip` is None and the clip is patchified as it comes."""
    _RING = 8

    def __init__(self, device, mix_clips: bool = True):
        self.dev = torch.zeros(16, device=device, dtype=torch.float32)
        self.clip, self.target = (self.dev[:10] if mix_clips else None), self.dev[10:13]
        self._pin = [torch.zeros(16, dtype=torch.float32).pin_memory() for _ in range(self._RING)]
        self._ev = [None] * self._RING
        self._k = 0

    def upload(self, values):
        self._k = (self._k + 1) % self._RING
        k = self._k
        if self._ev[k] is not None:
            self._ev[k].synchronize()
        self._pin[k].copy_(torch.tensor(values, dtype=torch.float32))
        self.dev.copy_(self._pin[k], non_blocking=True)
        self._ev[k] = torch.cuda.Event()
        self._ev[k].record()
