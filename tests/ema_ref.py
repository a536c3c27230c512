"""timm 0.4.12 `timm.utils.ModelEma` (timm/utils/model_ema.py, the V1 class VideoMAE's fine-tuning builds with --model_ema),
restated: timm is not a dependency of the package.  The update is torch's own fp32 arithmetic, so it is the reference the fused
kernel is checked against bit for bit.  `update_tensor` applies the same formula to one tensor (e.g. a recorded weight arena)."""
from collections import OrderedDict
from copy import deepcopy

import torch


class ModelEma:
    def __init__(self, model, decay=0.9999, device='', resume=''):
        # make a copy of the model for accumulating moving average of weights
        self.ema = deepcopy(model)
        self.ema.eval()
        self.decay = decay
        self.device = device  # perform ema on different device from model if set
        if device:
            self.ema.to(device=device)
        self.ema_has_module = hasattr(self.ema, 'module')
        if resume:
            self._load_checkpoint(resume)
        for p in self.ema.parameters():
            p.requires_grad_(False)

    def _load_checkpoint(self, checkpoint_path):
        checkpoint = torch.load(checkpoint_path, map_location='cpu', weights_only=False)
        assert isinstance(checkpoint, dict)
        if 'state_dict_ema' in checkpoint:
            new_state_dict = OrderedDict()
            for k, v in checkpoint['state_dict_ema'].items():
                # ema model may have been wrapped by DataParallel, and need module prefix
                if self.ema_has_module:
                    name = 'module.' + k if not k.startswith('module') else k
                else:
                    name = k
                new_state_dict[name] = v
            self.ema.load_state_dict(new_state_dict)

    def update(self, model):
        # correct a mismatch in state dict keys
        needs_module = hasattr(model, 'module') and not self.ema_has_module
        with torch.no_grad():
            msd = model.state_dict()
            for k, ema_v in self.ema.state_dict().items():
                if needs_module:
                    k = 'module.' + k
                model_v = msd[k].detach()
                if self.device:
                    model_v = model_v.to(device=self.device)
                ema_v.copy_(ema_v * self.decay + (1. - self.decay) * model_v)


def update_tensor(ema_v: torch.Tensor, model_v: torch.Tensor, decay: float) -> torch.Tensor:
    """The body of ModelEma.update for one entry, in place."""
    with torch.no_grad():
        ema_v.copy_(ema_v * decay + (1. - decay) * model_v)
    return ema_v
