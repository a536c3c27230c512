"""Model EMA of the stage-2 loop: timm 0.4.12's `ModelEma` (the V1 class VideoMAE / UMT fine-tuning builds with --model_ema,
run_stage2.py's `model_ema` argument of train_one_epoch), updated on the device by one fused kernel.

    ModelEma(model, decay, device, resume)   timm.utils.ModelEma: deepcopy, eval, requires_grad off, optional state_dict_ema
    update(model)                            ema = ema * decay + (1 - decay) * p over every state_dict entry — here every
                                             parameter of the fp32 arena (the model has no buffers), frozen ones included:
                                             ub_ema_update, bit-identical to torch's fp32 arithmetic, which also rewrites the
                                             EMA's bf16 shadow so that the EMA model is always ready to evaluate
    resolve_model_ema(model_ema, model)      what the fused loop accepts: this class, or the reference's own timm ModelEma
                                             (duck-typed), whose update() the fused kernel stands in for
The EMA copy is an ordinary stage-2 model with its own parameter arena (VisionTransformer.__deepcopy__ never carries the
source's); it evaluates through validation_one_epoch / final_test like any model.
"""
from collections import OrderedDict
from copy import deepcopy

import torch

from . import ops


def _unwrap(m):
    return m.module if hasattr(m, "module") else m


def ema_update(ema_model, model, decay: float):
    """One fused EMA update of ema_model's arena from model's, on the current stream (capturable in a CUDA graph).  Both are
    stage-2 models (or wrappers with `.module`); their arenas must have the same layout."""
    ema_arena, arena = _unwrap(ema_model).core().arena, _unwrap(model).core().arena
    if ema_arena.offsets != arena.offsets or ema_arena.numel != arena.numel:
        raise ValueError("model EMA: the EMA model's parameter arena has a different layout from the model's (another "
                         "architecture or parameter set)")
    ops.ema_update(ema_arena.params, ema_arena.w16, arena.params, decay)


class ModelEma:
    """timm 0.4.12 timm.utils.ModelEma (the V1 class): keeps `ema`, an eval-mode deepcopy of the model whose parameters follow
    ema = decay * ema + (1 - decay) * param after every optimizer update.  `device='cpu'` builds the copy on the host as timm does,
    but the fused loop refuses it (the update runs on the GPU, next to the arena)."""

    def __init__(self, model, decay=0.9999, device="", resume=""):
        self.ema = deepcopy(model)
        self.ema.eval()
        self.decay = decay
        self.device = device
        if self.device:
            self.ema.to(device=device)
        self.ema_has_module = hasattr(self.ema, "module")
        if resume:
            self._load_checkpoint(resume)
        for p in self.ema.parameters():
            p.requires_grad_(False)

    def _load_checkpoint(self, checkpoint_path):
        """timm ModelEma._load_checkpoint: `state_dict_ema` of a checkpoint file (or file object), `module.` added when the EMA is
        wrapped; without that key the EMA keeps the model's weights."""
        checkpoint = torch.load(checkpoint_path, map_location="cpu", weights_only=False)
        assert isinstance(checkpoint, dict)
        if "state_dict_ema" not in checkpoint:
            print("Failed to find state_dict_ema, starting from loaded model weights")
            return
        state = OrderedDict()
        for k, v in checkpoint["state_dict_ema"].items():
            state[("module." + k if not k.startswith("module") else k) if self.ema_has_module else k] = v
        self.ema.load_state_dict(state)
        core = getattr(_unwrap(self.ema), "_core", None)
        if core is not None:
            core.sync_shadow(force=True)
        print("Loaded state_dict_ema")

    def update(self, model):
        ema_update(self.ema, model, self.decay)


class ResolvedEma:
    """The EMA the fused stage-2 step updates: the caller's object (this module's ModelEma or timm's), its unwrapped EMA model, and
    the decay read from the object at every step."""

    def __init__(self, source, ema_net):
        self.source, self.ema_net = source, ema_net

    @property
    def decay(self) -> float:
        return float(self.source.decay)

    def update(self, model):
        ema_update(self.ema_net, model, self.decay)


def resolve_model_ema(model_ema, model):
    """None, or the ResolvedEma of `model_ema` for `model` (a stage-2 model or its DataParallel wrapper).  Accepts this module's
    ModelEma and the reference's timm.utils.ModelEma (recognised by its `ema`, `decay` and `device` attributes).  Raises
    NotImplementedError for anything else (before looking at any other argument) and for an EMA kept on the host
    (--model_ema_force_cpu), ValueError for an EMA model of another architecture."""
    if model_ema is None:
        return None
    if not isinstance(model_ema, ModelEma) and not all(hasattr(model_ema, a) for a in ("ema", "decay", "device")):
        raise NotImplementedError(f"model EMA: the fused stage-2 loop takes a unite_b200.ema.ModelEma or timm's ModelEma, got "
                                  f"{type(model_ema).__name__}")
    if str(model_ema.device).startswith("cpu"):
        raise NotImplementedError("model EMA on the host (device='cpu', --model_ema_force_cpu) is not supported: the EMA is updated "
                                  "on the GPU next to the parameter arena; a host EMA would copy the whole arena to the host every "
                                  "update")
    from .modeling_finetune import VisionTransformer
    ema_net, net = _unwrap(model_ema.ema), _unwrap(model)
    shapes = lambda m: [(n, tuple(p.shape)) for n, p in m.named_parameters()]
    if not isinstance(ema_net, VisionTransformer) or type(ema_net) is not type(net) or shapes(ema_net) != shapes(net):
        raise ValueError(f"model EMA: the EMA model ({type(ema_net).__name__}) does not have the architecture of the trained model "
                         f"({type(net).__name__}): build it with ModelEma(model) from the same model")
    return ResolvedEma(model_ema, ema_net)
