"""Checkpoint interop for the B200 modules (SURVEY.md §8 row f3).

The modules keep the reference's state_dict keys and shapes, so real checkpoints (UMT `b16_ptk710_f8_res224.pth`, the
OpenAI-CLIP visual tower `vit_b16.pth`) load once the reference's adapters have been applied.  This file restates those
adapters as small composable steps; `load_student_from_ckpt` / `load_from_ckpt` assemble them in the reference's order.

    select_state       pick the sub-dict named by `model_key` ("model|module")          run_stage1.py:522-533, run_stage2.py:358-365
    remap_keys         strip `backbone.` (and, for the fine-tune ViT, `encoder.`)       run_stage1.py:535-544, run_stage2.py:383-392
    adapt_head         drop / slice / re-index the K710 classifier rows                 run_stage2.py:367-381
    resize_pos_embed   temporal linear + spatial bicubic interpolation of `pos_embed`   run_stage1.py:553-588, run_stage2.py:394-434
    load_state_dict    prefix-aware, non-strict load with the reference's report        src/utils.py:554-599
    save_model / auto_load_model   `checkpoint-<tag>.pth` with model / optimizer / epoch  src/utils.py:689-776
                                   (+ `model_ema`, the EMA model's state_dict, when a model EMA is given)
The CLIP teacher's adapter (2-D -> 3-D conv inflation, positional-grid resize, clip.py:191-231) lives next to the
teacher in unite_b200/clip.py.
"""
import glob
import os
from collections import OrderedDict
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F


def select_state(checkpoint: Dict, model_key: str = "model|module") -> Tuple[Dict, Optional[str]]:
    """First of the `|`-separated keys present in `checkpoint` wins; otherwise the checkpoint itself is the state dict."""
    for key in model_key.split("|"):
        if key in checkpoint:
            return checkpoint[key], key
    return checkpoint, None


def remap_keys(state: Dict, strip: Sequence[str] = ("backbone.",), add_prefix: str = "") -> "OrderedDict":
    """Drop the first matching prefix in `strip` from every key, then prepend `add_prefix`."""
    out = OrderedDict()
    for k, v in state.items():
        for s in strip:
            if k.startswith(s):
                k = k[len(s):]
                break
        out[add_prefix + k] = v
    return out


def adapt_head(state: Dict, nb_classes: int, delete_head: bool = False, label_map: Optional[Sequence[int]] = None) -> Dict:
    """K710-pretrained classifier -> the target label space (run_stage2.py:367-381): delete it, keep the first 400 rows
    (K400 is a prefix of K710), or gather the rows listed in `label_map` (K600 / K700)."""
    if "head.weight" not in state:
        return state
    if delete_head:
        del state["head.weight"], state["head.bias"]
    elif state["head.weight"].shape[0] == 710:
        if nb_classes == 400:
            state["head.weight"], state["head.bias"] = state["head.weight"][:400], state["head.bias"][:400]
        elif nb_classes in (600, 700):
            if label_map is None:
                raise FileNotFoundError(f"k710/label_mixto{nb_classes}.json is needed to map the K710 head to {nb_classes} classes")
            idx = torch.as_tensor(list(label_map), dtype=torch.long)
            state["head.weight"], state["head.bias"] = state["head.weight"][idx], state["head.bias"][idx]
    return state


def resize_pos_embed(pos: torch.Tensor, num_patches: int, num_extra_tokens: int, tubelet_size: int, num_frames: int,
                     pretrain_frames: int = 8) -> torch.Tensor:
    """pos [1, extra + t0*s0*s0, C] -> [1, extra + t1*s1*s1, C].

    Time first (linear along t per (position, channel), run_stage1.py:566-573), then space (bicubic, align_corners=False, on
    each frame's s0 x s0 grid, :576-588).  Extra (class / dist) tokens pass through.  Mirrors the reference's quirk that the
    temporal pass is written for num_extra_tokens == 0 (it views the whole tensor as [t0, s0*s0])."""
    C = pos.shape[-1]
    t0, t1 = pretrain_frames // tubelet_size, num_frames // tubelet_size
    s0 = int(((pos.shape[-2] - num_extra_tokens) // t0) ** 0.5)
    s1 = int((num_patches // t1) ** 0.5)
    if t0 != t1:
        x = pos.view(1, t0, -1, C).permute(0, 2, 3, 1).reshape(-1, C, t0)          # [(1*s0*s0), C, t0]
        x = F.interpolate(x, size=t1, mode="linear")
        pos = x.view(1, -1, C, t1).permute(0, 3, 1, 2).reshape(1, -1, C)
    if s0 != s1:
        extra, grid = pos[:, :num_extra_tokens], pos[:, num_extra_tokens:]
        grid = grid.reshape(-1, s0, s0, C).permute(0, 3, 1, 2)                      # [t1, C, s0, s0]
        grid = F.interpolate(grid, size=(s1, s1), mode="bicubic", align_corners=False)
        grid = grid.permute(0, 2, 3, 1).reshape(-1, t1, s1, s1, C).flatten(1, 3)
        pos = torch.cat((extra, grid), dim=1)
    return pos


def load_state_dict(model: torch.nn.Module, state: Dict, prefix: str = "", ignore_missing: str = "relative_position_index",
                    verbose: bool = True) -> Tuple[List[str], List[str], List[str]]:
    """Non-strict load of the keys under `prefix` (src/utils.py:554-599).  Returns (missing, unexpected, ignored-missing);
    shape mismatches are reported and skipped, like `_load_from_state_dict(strict=True)` collecting error_msgs."""
    own = model.state_dict()
    sub = {k[len(prefix):]: v for k, v in state.items() if k.startswith(prefix)} if prefix else dict(state)
    errors, loadable = [], {}
    for k, v in sub.items():
        if k in own:
            if tuple(own[k].shape) != tuple(v.shape):
                errors.append(f"size mismatch for {k}: checkpoint {tuple(v.shape)} vs model {tuple(own[k].shape)}")
            else:
                loadable[k] = v
    res = model.load_state_dict(loadable, strict=False)
    unexpected = [k for k in sub if k not in own]
    pats = ignore_missing.split("|") if ignore_missing else []
    missing = [k for k in res.missing_keys if not any(p in k for p in pats)]
    ignored = [k for k in res.missing_keys if any(p in k for p in pats)]
    if verbose:
        name = model.__class__.__name__
        if missing:
            print("Weights of {} not initialized from pretrained model: {}".format(name, missing))
        if unexpected:
            print("Weights from pretrained model not used in {}: {}".format(name, unexpected))
        if ignored:
            print("Ignored weights of {} not initialized from pretrained model: {}".format(name, ignored))
        if errors:
            print("\n".join(errors))
    core = getattr(model, "_core", None)            # the bf16 GEMM shadow of the arena must follow the new fp32 values
    if core is not None and hasattr(core, "sync_shadow"):
        core.sync_shadow(force=True)
    return missing, unexpected, ignored


def _maybe_resize_pos(state: Dict, patch_embed, pos_embed, num_frames: int):
    if "pos_embed" in state:
        n_patches = patch_embed.num_patches
        extra = pos_embed.shape[-2] - n_patches
        state["pos_embed"] = resize_pos_embed(state["pos_embed"], n_patches, extra, patch_embed.tubelet_size, num_frames)


def load_student_from_ckpt(args, model: torch.nn.Module) -> torch.nn.Module:
    """Stage-1 / stage-3 student initialisation (run_stage1.py:518-602): the encoder of a UMT checkpoint goes under
    `encoder.`, optional pre-trained alignment decoders are merged in, `clip_decoder.*` can be frozen.
    args: student_init, model_key, student_prefix, num_frames, clip_decoder_init (optional), freeze_clip_decoders."""
    ckpt = torch.load(args.student_init, map_location="cpu", weights_only=False)
    state, key = select_state(ckpt, args.model_key)
    if key is not None:
        state = {f"encoder.{k}": v for k, v in state.items()}
    state = remap_keys(state, strip=("backbone.",))
    if getattr(args, "clip_decoder_init", None):
        dec = torch.load(args.clip_decoder_init, map_location="cpu", weights_only=False)
        state.update({k: v for k, v in dec.items() if k.startswith("clip_decoder.")})
    enc = getattr(model, "encoder", model)
    _maybe_resize_pos(state, enc.patch_embed, enc.pos_embed, args.num_frames)
    load_state_dict(model, state, prefix=getattr(args, "student_prefix", ""))
    if getattr(args, "freeze_clip_decoders", False):
        for n, p in model.named_parameters():
            if n.startswith("clip_decoder."):
                p.requires_grad = False
    return model


def load_from_ckpt(args, model: torch.nn.Module, label_map: Optional[Sequence[int]] = None) -> torch.nn.Module:
    """Stage-2 fine-tune initialisation (run_stage2.py:349-438).  args: finetune, model_key, model_prefix, nb_classes,
    delete_head, num_frames."""
    ckpt = torch.load(args.finetune, map_location="cpu", weights_only=False)
    state, _ = select_state(ckpt, args.model_key)
    state = adapt_head(dict(state), args.nb_classes, getattr(args, "delete_head", False), label_map)
    state = remap_keys(state, strip=("backbone.", "encoder."))
    _maybe_resize_pos(state, model.patch_embed, model.pos_embed, args.num_frames)
    load_state_dict(model, state, prefix=getattr(args, "model_prefix", ""))
    return model


# ---- training checkpoints (src/utils.py:689-776, torch.amp branch) -------------------------------------------------
def _is_master() -> bool:
    import torch.distributed as dist
    return not (dist.is_available() and dist.is_initialized()) or dist.get_rank() == 0


def _ema_model(model_ema):
    """The EMA's own model (timm's get_state_dict(model_ema) unwraps ModelEma.ema and a `.module` wrapper)."""
    m = model_ema.ema if hasattr(model_ema, "ema") else model_ema
    return m.module if hasattr(m, "module") else m


def save_model(output_dir: str, epoch, model_without_ddp, optimizer, loss_scaler=None, args=None, tag: Optional[str] = None,
               model_ema=None) -> str:
    """`checkpoint-<epoch or tag>.pth` = {model, optimizer, epoch, scaler, args}, plus `model_ema` (the EMA model's state_dict)
    when model_ema is given; written by rank 0 only."""
    path = os.path.join(output_dir, "checkpoint-%s.pth" % (tag if tag is not None else str(epoch)))
    if hasattr(optimizer, "consolidate"):
        optimizer.consolidate()        # collective: gathers the rank-sharded fp32 master weights / Adam moments (ddp.NvlsShardedStep)
    if _is_master():
        os.makedirs(output_dir, exist_ok=True)
        to_save = {"model": model_without_ddp.state_dict(), "optimizer": optimizer.state_dict(), "epoch": epoch, "args": args,
                   "scaler": loss_scaler.state_dict() if loss_scaler is not None and hasattr(loss_scaler, "state_dict") else {}}
        if model_ema is not None:
            to_save["model_ema"] = _ema_model(model_ema).state_dict()
        torch.save(to_save, path)
    return path


def auto_load_model(output_dir: str, model_without_ddp, optimizer=None, loss_scaler=None, resume: str = "", auto_resume: bool = True,
                    model_ema=None):
    """Resume order of the reference: checkpoint-latest.pth, checkpoint-best.pth, the highest numbered checkpoint-<n>.pth.
    model_ema: restored from the checkpoint's `model_ema` entry when there is one (its bf16 shadow refreshed).
    Returns the epoch to start from (0 when nothing was found)."""
    if not resume:
        for name in ("checkpoint-latest.pth", "checkpoint-best.pth"):
            if os.path.exists(os.path.join(output_dir, name)):
                resume = os.path.join(output_dir, name)
                break
        else:
            if auto_resume:
                nums = [int(t) for t in (p.split("-")[-1].split(".")[0] for p in glob.glob(os.path.join(output_dir, "checkpoint-*.pth")))
                        if t.isdigit()]
                if nums:
                    resume = os.path.join(output_dir, "checkpoint-%d.pth" % max(nums))
    if not resume:
        return 0
    ckpt = torch.load(resume, map_location="cpu", weights_only=False)
    model_without_ddp.load_state_dict(ckpt["model"])
    core = getattr(model_without_ddp, "_core", None)
    if core is not None and hasattr(core, "sync_shadow"):
        core.sync_shadow(force=True)
    if model_ema is not None and "model_ema" in ckpt:
        ema = _ema_model(model_ema)
        ema.load_state_dict(ckpt["model_ema"])
        core = getattr(ema, "_core", None)
        if core is not None and hasattr(core, "sync_shadow"):
            core.sync_shadow(force=True)
    start = 0
    if optimizer is not None and "optimizer" in ckpt and "epoch" in ckpt:
        optimizer.load_state_dict(ckpt["optimizer"])
        start = ckpt["epoch"] + 1
        if loss_scaler is not None and ckpt.get("scaler") and hasattr(loss_scaler, "load_state_dict"):
            loss_scaler.load_state_dict(ckpt["scaler"])
    print("Resume checkpoint %s" % resume)
    return start
