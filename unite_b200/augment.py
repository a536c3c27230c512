"""Stage-2 training crop, flip and random erasing of decoded uint8 frames: drawn on the host, applied on the device.

The reference's training transform (kinetics_sparse.py `_aug_frame`, VideoMAE / UMT) runs, per clip:
    RandAugment on uint8 PIL frames -> ToTensor + tensor_normalize -> permute to [C,T,H,W]
    -> spatial_sampling(crop_size, random_horizontal_flip=True, aspect_ratio=(0.75, 1.3333), scale=(0.08, 1.0))
       (random_resized_crop with bilinear interpolation, then horizontal_flip)
    -> RandomErasing(reprob, mode=remode, max_count=recount, num_splits=recount) on the [T,C,H,W] permute.
Only RandAugment needs PIL.  A loader that stops after it hands over the uint8 frames [B,T,H,W,3] with a SpatialAugment: the
per-clip crop box, flip and erasing box are drawn here, call for call as the reference draws them (Python's `random` and numpy's
global generator, the SlowFast functions VideoMAE copies), and ub_patchify_aug_u8 applies them inside the normalising im2col.  The
fill values of 'rand' / 'pixel' erasing come from a device-side Philox generator instead of torch.normal_ on the host.

Each of the three decisions lives in one function below (crop_params, flip_draw, erase_box); a reference copy that differs changes
only that function.
"""
import math
import random
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import torch

from .mixup import PinnedUpload
from .ops import IMAGENET_MEAN, IMAGENET_STD

__all__ = ["SpatialAugment", "AugDraw", "AugBuffer", "crop_params", "flip_draw", "erase_box", "ERASE_MODES"]

ERASE_MODES = {"const": 0, "rand": 1, "pixel": 2}


# ---- SlowFast video_transforms / random_erasing, as VideoMAE and UMT copy them ----------------------------------------------------
def crop_params(scale, ratio, height, width, num_repeat=10):
    """video_transforms._get_param_spatial_crop(scale, ratio, height, width) with log_scale=True, switch_hw=False: (i, j, h, w).
    Each attempt also draws np.random.uniform() (the `np.random.uniform() < 0.5 and switch_hw` test evaluates its left side
    first); after `num_repeat` misses, the central crop of the nearest admissible aspect ratio."""
    for _ in range(num_repeat):
        area = height * width
        target_area = random.uniform(*scale) * area
        log_ratio = (math.log(ratio[0]), math.log(ratio[1]))
        aspect_ratio = math.exp(random.uniform(*log_ratio))
        w = int(round(math.sqrt(target_area * aspect_ratio)))
        h = int(round(math.sqrt(target_area / aspect_ratio)))
        np.random.uniform()
        if 0 < w <= width and 0 < h <= height:
            i = random.randint(0, height - h)
            j = random.randint(0, width - w)
            return i, j, h, w
    in_ratio = float(width) / float(height)
    if in_ratio < min(ratio):
        w = width
        h = int(round(w / min(ratio)))
    elif in_ratio > max(ratio):
        h = height
        w = int(round(h * max(ratio)))
    else:
        w = width
        h = height
    i = (height - h) // 2
    j = (width - w) // 2
    return i, j, h, w


def flip_draw(prob=0.5):
    """video_transforms.horizontal_flip(prob, images): flipped when np.random.uniform() < prob."""
    return bool(np.random.uniform() < prob)


def erase_box(reprob, img_h, img_w, min_area=0.02, max_area=1 / 3, min_aspect=0.3, attempts=100) -> Optional[Tuple[int, int, int, int]]:
    """random_erasing.RandomErasing(reprob, max_count=1, num_splits=1, cube=True)._erase_cube's draws on [T,C,img_h,img_w]: None
    when `random.random() > reprob` or no attempt fits, else the (top, left, h, w) box every frame is erased in."""
    if random.random() > reprob:
        return None
    area = img_h * img_w
    log_aspect_ratio = (math.log(min_aspect), math.log(1 / min_aspect))
    count = 1
    for _ in range(attempts):
        target_area = random.uniform(min_area, max_area) * area / count
        aspect_ratio = math.exp(random.uniform(*log_aspect_ratio))
        h = int(round(math.sqrt(target_area * aspect_ratio)))
        w = int(round(math.sqrt(target_area / aspect_ratio)))
        if w < img_w and h < img_h:
            top = random.randint(0, img_h - h)
            left = random.randint(0, img_w - w)
            return top, left, h, w
    return None


# ---- the configuration and one batch's draws -----------------------------------------------------------------------------------
@dataclass(frozen=True)
class AugDraw:
    """Per-clip draws of one batch: `params` int32 [B, 10] = {i, j, h, w, flip, erase, top, left, eh, ew} per clip (the layout
    ub_patchify_aug_u8 reads), drawn for frames of `frames_hw` pixels by `aug`."""
    aug: "SpatialAugment"
    frames_hw: Tuple[int, int]
    params: np.ndarray


@dataclass(frozen=True)
class SpatialAugment:
    """The stage-2 training loader's spatial augmentation, applied on the device to decoded uint8 frames (see the module doc).
    Pass it as `spatial_aug` to engine_for_finetuning.train_one_epoch; `seed` keys the device generator of the erasing noise."""
    crop_size: int = 224
    scale: Tuple[float, float] = (0.08, 1.0)
    ratio: Tuple[float, float] = (0.75, 1.3333)
    hflip: bool = True
    reprob: float = 0.25
    remode: str = "pixel"
    recount: int = 1
    mean: Tuple[float, float, float] = IMAGENET_MEAN
    std: Tuple[float, float, float] = IMAGENET_STD
    seed: int = 0

    def __post_init__(self):
        if self.remode not in ERASE_MODES:
            raise ValueError(f"SpatialAugment: remode {self.remode!r} is not one of {sorted(ERASE_MODES)}")
        if self.recount != 1:
            raise ValueError(f"SpatialAugment: recount={self.recount}: only one erasing box per clip (recount=1) is implemented")
        if self.crop_size <= 0 or self.crop_size % 16:
            raise ValueError(f"SpatialAugment: crop_size {self.crop_size} must be a positive multiple of the 16-pixel patch")
        if not (0 < self.scale[0] <= self.scale[1]) or not (0 < self.ratio[0] <= self.ratio[1]):
            raise ValueError(f"SpatialAugment: scale {self.scale} and ratio {self.ratio} must be positive, increasing ranges")
        if len(self.mean) != 3 or len(self.std) != 3 or 0.0 in tuple(self.std):
            raise ValueError("SpatialAugment: mean and std take three values, std non-zero")
        object.__setattr__(self, "scale", tuple(float(v) for v in self.scale))
        object.__setattr__(self, "ratio", tuple(float(v) for v in self.ratio))
        object.__setattr__(self, "mean", tuple(float(v) for v in self.mean))
        object.__setattr__(self, "std", tuple(float(v) for v in self.std))

    @property
    def erase_mode(self) -> int:
        return ERASE_MODES[self.remode]

    def draw(self, shape) -> AugDraw:
        """The draws of a batch of frames of `shape` [B,T,H,W,3], clip by clip in the reference loader's order: crop, flip, erase.
        With reprob == 0 the reference builds no RandomErasing, so nothing is drawn for it."""
        B, _, H, W, _ = shape
        S = self.crop_size
        p = np.zeros((B, 10), dtype=np.int32)
        for b in range(B):
            p[b, 0:4] = crop_params(self.scale, self.ratio, H, W)
            p[b, 4] = flip_draw() if self.hflip else 0
            box = erase_box(self.reprob, S, S) if self.reprob > 0 else None
            if box is not None:
                p[b, 5:10] = (1, *box)
        return AugDraw(self, (H, W), p)


class AugBuffer(PinnedUpload):
    """Device copy of one batch's AugDraw (`draw`, int32 [B, 10], fixed address) and the counter of the erasing noise generator
    (`rng`, int64 [2], advanced by every launch), for one batch size and one SpatialAugment."""

    def __init__(self, aug: SpatialAugment, batch: int, device):
        super().__init__((batch, 10), torch.int32, device)
        self.aug, self.batch = aug, batch
        self.draw = self.dev
        self.rng = torch.zeros(2, dtype=torch.int64, device=device)

    def upload(self, d: AugDraw):
        H, W = d.frames_hw
        p = d.params
        S = self.aug.crop_size
        i, j, h, w, top, left, eh, ew = (p[:, k] for k in (0, 1, 2, 3, 6, 7, 8, 9))
        if p.shape != (self.batch, 10) or (h < 1).any() or (w < 1).any() or (i < 0).any() or (j < 0).any() or (i + h > H).any() \
                or (j + w > W).any() or (top < 0).any() or (left < 0).any() or (top + eh > S).any() or (left + ew > S).any():
            raise ValueError(f"AugBuffer: draws out of range of {H}x{W} frames / the {S}x{S} crop")
        super().upload(torch.from_numpy(p))
