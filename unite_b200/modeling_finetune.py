"""Student ViT building blocks and the stage-2 classifier — parameter containers with the reference's names.

Mirrors the public surface of reference src/models/modeling_finetune.py (Block :122, Attention :76, Mlp :56,
PatchEmbed :153, VisionTransformer :237, factories :386-415): same constructor kwargs, attribute names and
state_dict keys/shapes, so checkpoints and driver code (`model.patch_embed.patch_size`, `get_num_layers()`,
`no_weight_decay()`) carry over.  The modules hold parameters only — the arithmetic is in vit_core.ViTTrunk
and runs on the CUDA kernels; calling forward without a GPU raises.
"""
from copy import deepcopy
from functools import partial

import numpy as np
import torch
import torch.nn as nn

from .registry import register_model


def to_2tuple(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (v, v)


def get_sinusoid_encoding_table(n_position, d_hid):
    """fp64 table -> fp32 [1, n, d]: angle = pos / 10000^(2*(j//2)/d), sin on even / cos on odd columns
    (reference modeling_finetune.py:225-235, modeling_adaptation.py:41-51)."""
    j = np.arange(d_hid)
    ang = np.arange(n_position, dtype=np.float64)[:, None] / np.power(10000, 2 * (j // 2) / d_hid)[None, :]
    ang[:, 0::2] = np.sin(ang[:, 0::2])
    ang[:, 1::2] = np.cos(ang[:, 1::2])
    return torch.tensor(ang, dtype=torch.float).unsqueeze(0)


class _ParamsOnly(nn.Module):
    def forward(self, *a, **k):
        raise RuntimeError(f"{type(self).__name__} only stores parameters; the owning model runs the fused CUDA path")


class DropPath(_ParamsOnly):
    def __init__(self, drop_prob=None):
        super().__init__()
        self.drop_prob = drop_prob

    def extra_repr(self):
        return "p={}".format(self.drop_prob)


class Mlp(_ParamsOnly):
    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, drop=0.0):
        super().__init__()
        self.fc1 = nn.Linear(in_features, hidden_features or in_features)
        self.fc2 = nn.Linear(hidden_features or in_features, out_features or in_features)


class Attention(_ParamsOnly):
    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_scale=None, attn_drop=0.0, proj_drop=0.0, attn_head_dim=None):
        super().__init__()
        if attn_drop or proj_drop:
            raise NotImplementedError("attention / projection dropout are 0 in every shipped UNITE config")
        head_dim = attn_head_dim or dim // num_heads
        self.num_heads = num_heads
        self.scale = qk_scale or head_dim ** -0.5
        self.qkv = nn.Linear(dim, head_dim * num_heads * 3, bias=False)
        if not qkv_bias:
            raise NotImplementedError("qkv_bias=False is not used by any UNITE factory")
        self.q_bias = nn.Parameter(torch.zeros(head_dim * num_heads))
        self.v_bias = nn.Parameter(torch.zeros(head_dim * num_heads))
        self.proj = nn.Linear(head_dim * num_heads, dim)


class Block(_ParamsOnly):
    def __init__(self, dim, num_heads, mlp_ratio=4.0, qkv_bias=False, qk_scale=None, drop=0.0, attn_drop=0.0, drop_path=0.0,
                 init_values=None, act_layer=nn.GELU, norm_layer=nn.LayerNorm, attn_head_dim=None):
        super().__init__()
        if init_values:
            raise NotImplementedError("layer-scale (init_values > 0) is off in every UNITE config (modeling_finetune.py:137-141)")
        if drop:
            raise NotImplementedError("dropout is 0 in every shipped UNITE config")
        self.norm1 = norm_layer(dim)
        self.attn = Attention(dim, num_heads=num_heads, qkv_bias=qkv_bias, qk_scale=qk_scale, attn_drop=attn_drop,
                              proj_drop=drop, attn_head_dim=attn_head_dim)
        self.drop_path = DropPath(drop_path) if drop_path > 0.0 else nn.Identity()
        self.norm2 = norm_layer(dim)
        self.mlp = Mlp(in_features=dim, hidden_features=int(dim * mlp_ratio), act_layer=act_layer, drop=drop)
        self.gamma_1, self.gamma_2 = None, None


class PatchEmbed(_ParamsOnly):
    """Conv3d(3, D, (tubelet,16,16), stride=same) parameters; applied as patchify + GEMM."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=768, num_frames=16, tubelet_size=2):
        super().__init__()
        img_size, patch_size = to_2tuple(img_size), to_2tuple(patch_size)
        if patch_size != (16, 16) or in_chans != 3:
            raise NotImplementedError("the patchify kernel is specialised for 3-channel 16x16 patches")
        self.tubelet_size = int(tubelet_size)
        self.img_size, self.patch_size = img_size, patch_size
        self.num_patches = (img_size[1] // patch_size[1]) * (img_size[0] // patch_size[0]) * (num_frames // self.tubelet_size)
        self.proj = nn.Conv3d(in_chans, embed_dim, kernel_size=(self.tubelet_size, 16, 16), stride=(self.tubelet_size, 16, 16))


def drop_path_factors(rates, B, device, generator=None):
    """Per-sample DropPath factors floor(keep + u)/keep (timm 0.4.12 drop_path) for every block and both
    branches: fp32 [depth, 2, B]; None if every rate is 0."""
    if not any(r > 0 for r in rates):
        return None
    keep = 1.0 - torch.tensor(rates, dtype=torch.float32, device=device).view(-1, 1, 1)
    u = torch.rand(len(rates), 2, B, device=device, generator=generator)
    return (torch.floor(keep + u) / keep).contiguous()


# --------------------------------------------------------------------------------------------------------------
# Stage-2 classifier: all tokens -> mean-pool -> fc_norm -> head   (reference modeling_finetune.py:237-383)
# --------------------------------------------------------------------------------------------------------------
def _trunc_init(m):
    """modeling_finetune.py:332-339."""
    if isinstance(m, nn.Linear):
        nn.init.trunc_normal_(m.weight, std=0.02)
        if m.bias is not None:
            nn.init.constant_(m.bias, 0)
    elif isinstance(m, nn.LayerNorm):
        nn.init.constant_(m.bias, 0)
        nn.init.constant_(m.weight, 1.0)


class VisionTransformer(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=768, depth=12, num_heads=12,
                 mlp_ratio=4.0, qkv_bias=False, qk_scale=None, fc_drop_rate=0.0, drop_rate=0.0, attn_drop_rate=0.0, drop_path_rate=0.0,
                 norm_layer=nn.LayerNorm, init_values=0.0, use_learnable_pos_emb=False, init_scale=0.0, all_frames=16, tubelet_size=2,
                 use_checkpoint=False, checkpoint_num=0, use_mean_pooling=True, classifier_type="linear", classifier_hidden_dim=256):
        super().__init__()
        if not use_mean_pooling or use_learnable_pos_emb or classifier_type != "linear" or fc_drop_rate:
            raise NotImplementedError("the shipped stage-2 config uses mean pooling, sinusoid positions and a linear head "
                                      "(configs/stage2_config.yaml)")
        self.num_classes = num_classes
        self.num_features = self.embed_dim = embed_dim
        self.tubelet_size = tubelet_size
        self.patch_embed = PatchEmbed(img_size=img_size, patch_size=patch_size, in_chans=in_chans, embed_dim=embed_dim,
                                      num_frames=all_frames, tubelet_size=tubelet_size)
        self.use_checkpoint, self.checkpoint_num, self.classifier_type = use_checkpoint, checkpoint_num, classifier_type
        self.pos_embed = get_sinusoid_encoding_table(self.patch_embed.num_patches, embed_dim)
        self.drop_path_rates = [x.item() for x in torch.linspace(0, drop_path_rate, depth)]
        self.blocks = nn.ModuleList([
            Block(dim=embed_dim, num_heads=num_heads, mlp_ratio=mlp_ratio, qkv_bias=qkv_bias, qk_scale=qk_scale, drop=drop_rate,
                  attn_drop=attn_drop_rate, drop_path=self.drop_path_rates[i], norm_layer=norm_layer, init_values=init_values)
            for i in range(depth)])
        self.norm = nn.Identity()
        self.fc_norm = norm_layer(embed_dim)
        self.fc_dropout = nn.Identity()
        self.head = nn.Linear(embed_dim, num_classes)
        self.apply(_trunc_init)
        self.head.weight.data.mul_(init_scale)
        self.head.bias.data.mul_(init_scale)
        self.num_heads, self.mlp_hidden = num_heads, int(embed_dim * mlp_ratio)
        self._core = None

    def get_num_layers(self):
        return len(self.blocks)

    @torch.jit.ignore
    def no_weight_decay(self):
        return {"pos_embed", "cls_token"}

    def get_classifier(self):
        return self.head

    def core(self):
        if self._core is None:
            dev = next(self.parameters()).device
            if dev.type != "cuda":
                raise RuntimeError("unite_b200 models compute on CUDA only: call model.cuda() first (there is no CPU path)")
            from .finetune_core import FinetuneCore
            self._core = FinetuneCore(self, dev)
        return self._core

    def __deepcopy__(self, memo):
        """A copy with its own parameters and no compute core (timm's ModelEma deep-copies the model, often after its arena
        exists): the copy builds its own arena on first use and never shares the source's arena, bf16 shadow, tensor maps or
        the engine / optimizer cached on the model (`_ub_*`).  Each parameter is cloned on its own (nn.Parameter.__deepcopy__),
        so a parameter that is a view into the source's arena becomes a standalone tensor."""
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        state = {k: (None if k == "_core" else deepcopy(v, memo)) for k, v in self.__dict__.items() if not k.startswith("_ub_")}
        new.__setstate__(state)
        return new

    def _apply(self, fn, *a, **k):
        if self._core is not None:
            raise RuntimeError("the model's parameters already live in its device arena; move it before the first forward")
        return super()._apply(fn, *a, **k)

    def forward(self, x, drop_path_factors_=None):
        """x [B,3,T,H,W] fp32 -> logits [B, num_classes] (modeling_finetune.py:356-383)."""
        from .finetune_core import _FinetuneFn
        core = self.core()
        dp = drop_path_factors_
        if dp is None and self.training:
            dp = core.drop_path.draw(x.shape[0])
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            anchor = torch.empty(0, device=x.device, requires_grad=True)
            return _FinetuneFn.apply(anchor, core, x, dp)
        return core.run_forward(x, dp, save=False)[0]


def _build_vit(embed_dim, depth, heads, img_size, pretrained, kwargs):
    if pretrained:
        raise NotImplementedError("pretrained weights need network access; load a state_dict instead")
    return VisionTransformer(img_size=img_size, patch_size=16, embed_dim=embed_dim, depth=depth, num_heads=heads, mlp_ratio=4,
                             qkv_bias=True, norm_layer=partial(nn.LayerNorm, eps=1e-6), **kwargs)


@register_model
def vit_base_patch16_224(pretrained=False, **kwargs):
    return _build_vit(768, 12, 12, 224, pretrained, kwargs)


@register_model
def vit_large_patch16_224(pretrained=False, **kwargs):
    return _build_vit(1024, 24, 16, 224, pretrained, kwargs)
