"""The reference's stage-2 training augmentation after RandAugment, restated as the SlowFast code VideoMAE / UMT copy it
(slowfast/datasets/transform.py, video_transforms.py, random_erasing.py): the oracle of unite_b200.augment's host draws and of
ub_patchify_aug_u8's rows."""
import math
import random

import numpy as np
import torch


def _get_param_spatial_crop(scale, ratio, height, width, num_repeat=10, log_scale=True, switch_hw=False):
    for _ in range(num_repeat):
        area = height * width
        target_area = random.uniform(*scale) * area
        if log_scale:
            log_ratio = (math.log(ratio[0]), math.log(ratio[1]))
            aspect_ratio = math.exp(random.uniform(*log_ratio))
        else:
            aspect_ratio = random.uniform(*ratio)

        w = int(round(math.sqrt(target_area * aspect_ratio)))
        h = int(round(math.sqrt(target_area / aspect_ratio)))

        if np.random.uniform() < 0.5 and switch_hw:
            w, h = h, w

        if 0 < w <= width and 0 < h <= height:
            i = random.randint(0, height - h)
            j = random.randint(0, width - w)
            return i, j, h, w

    # Fallback to central crop
    in_ratio = float(width) / float(height)
    if in_ratio < min(ratio):
        w = width
        h = int(round(w / min(ratio)))
    elif in_ratio > max(ratio):
        h = height
        w = int(round(h * max(ratio)))
    else:  # whole image
        w = width
        h = height
    i = (height - h) // 2
    j = (width - w) // 2
    return i, j, h, w


def random_resized_crop(images, target_height, target_width, scale=(0.8, 1.0), ratio=(3.0 / 4.0, 4.0 / 3.0)):
    """images [C,T,H,W]."""
    height = images.shape[2]
    width = images.shape[3]
    i, j, h, w = _get_param_spatial_crop(scale, ratio, height, width)
    cropped = images[:, :, i:i + h, j:j + w]
    return torch.nn.functional.interpolate(cropped, size=(target_height, target_width), mode="bilinear", align_corners=False)


def horizontal_flip(prob, images):
    if np.random.uniform() < prob:
        images = images.flip((-1))
    return images


def _get_pixels(per_pixel, rand_color, patch_size, dtype=torch.float32, device="cpu"):
    if per_pixel:
        return torch.empty(patch_size, dtype=dtype, device=device).normal_()
    elif rand_color:
        return torch.empty((patch_size[0], 1, 1), dtype=dtype, device=device).normal_()
    else:
        return torch.zeros((patch_size[0], 1, 1), dtype=dtype, device=device)


class RandomErasing:
    def __init__(self, probability=0.5, min_area=0.02, max_area=1 / 3, min_aspect=0.3, max_aspect=None, mode="const", min_count=1,
                 max_count=None, num_splits=0, device="cuda", cube=True):
        self.probability = probability
        self.min_area = min_area
        self.max_area = max_area
        max_aspect = max_aspect or 1 / min_aspect
        self.log_aspect_ratio = (math.log(min_aspect), math.log(max_aspect))
        self.min_count = min_count
        self.max_count = max_count or min_count
        self.num_splits = num_splits
        mode = mode.lower()
        self.rand_color = False
        self.per_pixel = False
        self.cube = cube
        if mode == "rand":
            self.rand_color = True
        elif mode == "pixel":
            self.per_pixel = True
        else:
            assert not mode or mode == "const"
        self.device = device

    def _erase_cube(self, img, batch_start, batch_size, chan, img_h, img_w, dtype):
        if random.random() > self.probability:
            return
        area = img_h * img_w
        count = self.min_count if self.min_count == self.max_count else random.randint(self.min_count, self.max_count)
        for _ in range(count):
            for _ in range(100):
                target_area = random.uniform(self.min_area, self.max_area) * area / count
                aspect_ratio = math.exp(random.uniform(*self.log_aspect_ratio))
                h = int(round(math.sqrt(target_area * aspect_ratio)))
                w = int(round(math.sqrt(target_area / aspect_ratio)))
                if w < img_w and h < img_h:
                    top = random.randint(0, img_h - h)
                    left = random.randint(0, img_w - w)
                    for i in range(batch_start, batch_size):
                        img_instance = img[i]
                        img_instance[:, top:top + h, left:left + w] = _get_pixels(self.per_pixel, self.rand_color, (chan, h, w),
                                                                                  dtype=dtype, device=self.device)
                    break

    def __call__(self, input):
        batch_size, chan, img_h, img_w = input.size()
        batch_start = batch_size // self.num_splits if self.num_splits > 1 else 0
        self._erase_cube(input, batch_start, batch_size, chan, img_h, img_w, input.dtype)
        return input


def loader_tail(clip_cthw, crop_size=224, scale=(0.08, 1.0), ratio=(0.75, 1.3333), hflip=True, reprob=0.25, remode="pixel", recount=1):
    """kinetics_sparse._aug_frame after tensor_normalize and the permute: spatial_sampling(spatial_idx=-1) with aspect_ratio and
    scale, then RandomErasing on the [T,C,H,W] permute.  clip_cthw: the normalised fp32 clip [C,T,H,W]."""
    x = random_resized_crop(clip_cthw, crop_size, crop_size, scale=scale, ratio=ratio)
    if hflip:
        x = horizontal_flip(0.5, x)
    if reprob > 0:
        erase = RandomErasing(reprob, mode=remode, max_count=recount, num_splits=recount, device=str(x.device))
        x = erase(x.permute(1, 0, 2, 3)).permute(1, 0, 2, 3)
    return x
