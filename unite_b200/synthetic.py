"""Synthetic clip generator — stands in for src/datasets/* (decord decode + augmentation), which needs data files.

Only the BATCH CONTRACT of the reference loaders is reproduced (SURVEY.md §2 row 20):
  stage 1  (videos [B,3,T,224,224] fp32 ImageNet-normalised, mask placeholder, label)     mae.py:220-222, build.py:63-69
  stage 2  (clip, label, index, {})                                                       kinetics_sparse.py:159
  stage 3  target (vid, vid_aug, label, name)                                             kinetics_sparse.py:174-180
Batches live in PINNED host memory (like DataLoader(pin_memory=True), run_stage1.py:700-708) and are seeded by
`seed + rank` (run_stage1.py:613).  `noise` is the Exp(1) draw the attention mask sampler consumes
(torch.multinomial's internal noise made explicit, run_stage1.py:382).
"""
import torch


def _clips(batch_size, num_frames, img_size, g, uint8):
    if uint8:
        return torch.randint(0, 256, (batch_size, num_frames, img_size, img_size, 3), generator=g, dtype=torch.uint8)
    return torch.randn(batch_size, 3, num_frames, img_size, img_size, generator=g)


class SyntheticStage1Loader:
    def __init__(self, batch_size, num_frames=8, img_size=224, steps=10, seed=0, rank=0, n_distinct=2, num_classes=12,
                 frames_per_token=1, pin=True, uint8=False):
        """uint8=True: batches carry DECODED frames uint8 [B,T,H,W,3] (what decord / NVDEC hand over, kinetics_sparse.py:
        loadvideo_decord) instead of the normalised fp32 clip; the engine normalises on the device (ops.patchify_u8)."""
        g = torch.Generator().manual_seed(seed + rank)
        self.steps = steps
        self.batches = []
        pin = pin and torch.cuda.is_available()
        HW = (img_size // 16) ** 2
        for _ in range(n_distinct):
            v = _clips(batch_size, num_frames, img_size, g, uint8)
            q = torch.empty(batch_size * (num_frames // frames_per_token), HW).exponential_(1, generator=g)
            y = torch.randint(0, num_classes, (batch_size,), generator=g)
            if pin:
                v, q = v.pin_memory(), q.pin_memory()
            self.batches.append((v, -1, y, q))

    def __len__(self):
        return self.steps

    def __iter__(self):
        for i in range(self.steps):
            yield self.batches[i % len(self.batches)]


class SyntheticStage2Loader:
    """(clip, label, index, {}) batches of kinetics_sparse.py:159 (train mode), pinned.  uint8=True: the clip is DECODED frames
    uint8 [B,T,H,W,3], as in SyntheticStage1Loader; the engine normalises them on the device."""

    def __init__(self, batch_size, num_frames=8, img_size=224, steps=10, seed=0, rank=0, n_distinct=2, num_classes=12, pin=True,
                 uint8=False):
        g = torch.Generator().manual_seed(seed + rank)
        pin = pin and torch.cuda.is_available()
        self.steps, self.batches = steps, []
        for _ in range(n_distinct):
            v = _clips(batch_size, num_frames, img_size, g, uint8)
            y = torch.randint(0, num_classes, (batch_size,), generator=g)
            self.batches.append((v.pin_memory() if pin else v, y, torch.arange(batch_size), {}))

    def __len__(self):
        return self.steps

    def __iter__(self):
        for i in range(self.steps):
            yield self.batches[i % len(self.batches)]


class SyntheticStage3Loader:
    """Stage-3 loaders: `.source` yields (clip, label, index, {}) (kinetics_sparse.py:159, train mode) and `.target` yields the
    dual-view batch (vid, vid_aug, label, name) of validation mode with return_aug_for_val (kinetics_sparse.py:174-180) — the
    plain view feeds the full-token pass and the zero-shot head, the augmented one the teacher attention and the masked
    committee (run_stage3.py:405-413).  vid_aug = vid + small noise (a stand-in for RandAugment: a different tensor of the same
    distribution).  uint8=True: every view is DECODED frames uint8 [B,T,H,W,3], as in SyntheticStage1Loader."""

    class _Iter:
        def __init__(self, batches, steps):
            self.batches, self.steps = batches, steps

        def __len__(self):
            return self.steps

        def __iter__(self):
            for i in range(self.steps):
                yield self.batches[i % len(self.batches)]

    def __init__(self, batch_size_s, batch_size_t=None, num_frames=8, img_size=224, steps=10, seed=0, rank=0, n_distinct=2,
                 num_classes=12, pin=True, uint8=False):
        g = torch.Generator().manual_seed(seed + rank)
        bt = batch_size_t or batch_size_s
        pin = pin and torch.cuda.is_available()
        src, tgt = [], []
        for i in range(n_distinct):
            vs = _clips(batch_size_s, num_frames, img_size, g, uint8)
            ys = torch.randint(0, num_classes, (batch_size_s,), generator=g)
            vt = _clips(bt, num_frames, img_size, g, uint8)
            if uint8:
                va = (vt.short() + torch.randint(-8, 9, vt.shape, generator=g, dtype=torch.int16)).clamp_(0, 255).to(torch.uint8)
            else:
                va = vt + 0.1 * torch.randn(bt, 3, num_frames, img_size, img_size, generator=g)
            yt = torch.randint(0, num_classes, (bt,), generator=g)
            if pin:
                vs, vt, va = vs.pin_memory(), vt.pin_memory(), va.pin_memory()
            src.append((vs, ys, torch.arange(batch_size_s), {}))
            tgt.append((vt, va, yt, [f"synthetic_{i}_{j}" for j in range(bt)]))
        self.source = self._Iter(src, steps)
        self.target = self._Iter(tgt, steps)
        self.num_classes = num_classes
