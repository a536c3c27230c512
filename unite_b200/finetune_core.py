"""Compute core of the stage-2 classifier (modeling_finetune.VisionTransformer): all 1568 tokens through the trunk,
mean-pool, fc_norm, linear head — forward and explicit backward on the C-ABI kernels."""
from typing import Dict

import torch

from . import ops
from .arena import ParamArena
from .vit_core import DropPathSource, ViTTrunk

BF16, F32, U8 = torch.bfloat16, torch.float32, torch.uint8


class _FinetuneFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, core, x, dp):
        logits, state = core.run_forward(x, dp, save=True)
        ctx.core, ctx.state = core, state
        return logits

    @staticmethod
    def backward(ctx, g_logits):
        ctx.core.run_backward(ctx.state, g_logits)
        return (None,) * 4


class FinetuneCore:
    def __init__(self, model, dev):
        from .modeling_adaptation import student_order_key, no_decay_rule
        self.model = model
        self.D, self.depth = model.embed_dim, len(model.blocks)
        self.N = model.patch_embed.num_patches
        self.tubelet = model.patch_embed.tubelet_size
        self.eps = model.fc_norm.eps
        self.C = model.num_classes
        self.arena = ParamArena(model, dev, student_order_key(self.depth), no_decay_rule(model.no_weight_decay()),
                                gap_after=lambda n, p: p.numel() if n.endswith("attn.q_bias") else 0)
        self.trunk = ViTTrunk(self.arena, "", self.D, self.depth, model.num_heads, model.mlp_hidden, self.eps)
        self.pos = model.pos_embed[0].to(dev).contiguous()
        self._pos_full: Dict[int, torch.Tensor] = {}
        self._shadow_version = None
        import os
        self.drop_path = DropPathSource(model.drop_path_rates, dev, seed=int(os.environ.get("UB_DROP_PATH_SEED", "0")))

    def sync_shadow(self, force=False):
        v = self.arena.params_version()
        if force or v != self._shadow_version:
            ops.cast_bf16(self.arena.params, self.arena.w16)
            self._shadow_version = v

    def _pos_rows(self, B):
        if B not in self._pos_full:
            self._pos_full[B] = self.pos.repeat(B, 1).contiguous()
        return self._pos_full[B]

    def run_forward(self, x, dp, save, mix=None, aug=None):
        """x: the fp32 clip [B,3,T,H,W], or decoded uint8 frames [B,T,H,W,3], normalised on the device (ops.patchify_u8).
        mix: None, or the device draw of batch-mode mixup / cutmix (mixup.MixBuffer.clip): the trunk then sees the mixed clip,
        mixed on the way into the im2col (x itself is not written).
        aug: None, or an augment.AugBuffer holding this batch's crop / flip / erasing draws: uint8 frames of any size are augmented
        to the crop_size x crop_size clip on the way into the im2col (ops.patchify_aug_u8), then mixed by `mix`."""
        u8 = x.dtype == U8
        if aug is not None:
            S = aug.aug.crop_size
            if not u8 or x.dim() != 5:
                raise ValueError("run_forward: the spatial augmentation takes decoded uint8 frames [B,T,H,W,3]")
            n = (x.shape[1] // self.tubelet) * (S // 16) ** 2
            if n != self.N:
                raise ValueError(f"run_forward: a {S}x{S} crop of {x.shape[1]} frames gives {n} tokens, the model has {self.N} "
                                 "(num_patches follows the crop size)")
            if aug.batch != x.shape[0]:
                raise ValueError(f"run_forward: draws for {aug.batch} clips, batch of {x.shape[0]}")
        self.sync_shadow()
        B, dev, a = x.shape[0], x.device, self.arena
        patches = torch.empty(B * self.N, 3 * self.tubelet * 256, device=dev, dtype=BF16)
        if aug is not None:
            g = aug.aug
            ops.patchify_aug_u8(x, patches, aug.draw, g.crop_size, self.tubelet, g.erase_mode, mix=mix, rng=aug.rng, seed=g.seed,
                                mean=g.mean, std=g.std)
        elif u8 and mix is None:
            ops.patchify_u8(x, patches, self.tubelet)
        elif u8:
            ops.patchify_mix_u8(x, patches, mix, self.tubelet)
        elif mix is None:
            ops.patchify(x.contiguous(), patches, self.tubelet)
        else:
            ops.patchify_mix(x.contiguous(), patches, mix, self.tubelet)
        ws = self.trunk.forward(patches, self._pos_rows(B), B, self.N, self.depth, save, dp)
        pooled = torch.empty(B, self.D, device=dev, dtype=F32)
        ops.meanpool_fwd(ws.x_at(self.depth).view(B, self.N, self.D), pooled)                     # x.mean(1)
        normed = torch.empty(B, self.D, device=dev, dtype=F32)
        ops.layernorm_fwd(pooled, a.p32("fc_norm.weight"), a.p32("fc_norm.bias"), self.eps, normed)
        logits = torch.empty(B, self.C, device=dev, dtype=F32)
        ops.linear_small_fwd(normed, a.p32("head.weight"), a.p32("head.bias"), logits)
        state = dict(ws=ws, pooled=pooled, normed=normed, B=B) if save else None
        return logits, state

    def block_grad_hi(self, l):
        """End of the decay-segment prefix that is final once block l's backward has run (head + blocks >= l)."""
        return self.arena.range_of([f"blocks.{l}.mlp.fc2.weight", f"blocks.{l}.attn.qkv.weight"])[1]

    def run_backward(self, state, g_logits, grad_sync=None):
        """grad_sync (ddp.GradSync, world > 1): told block by block which prefix of the gradient arena is final, so that its range
        all-reduces overlap the rest of backward (the role of DDP's buckets, run_stage2.py:641).  Only valid on the LAST
        micro-step of an update (gradients of earlier micro-steps are already in the arena and are summed with it)."""
        a = self.arena
        a.attach_grads()
        ws, B, dev = state["ws"], state["B"], g_logits.device
        g = g_logits.contiguous().float()
        d_normed = torch.empty(B, self.D, device=dev, dtype=F32)
        ops.linear_small_bwd(state["normed"], a.p32("head.weight"), g, d_normed, a.g32("head.weight"), a.g32("head.bias"))
        dy = torch.empty(B, self.D, device=dev, dtype=BF16)
        ops.cast_scale_bf16(d_normed, dy)
        d_pooled = torch.empty(B, self.D, device=dev, dtype=F32)
        ops.layernorm_bwd(dy, state["pooled"], a.p32("fc_norm.weight"), self.eps, None, d_pooled, None, None, 0,
                          a.g32("fc_norm.weight"), a.g32("fc_norm.bias"))
        ops.meanpool_bwd(d_pooled, ws.dx.view(B, self.N, self.D))
        on_done = None
        if grad_sync is not None and grad_sync.world > 1:
            on_done = lambda l: grad_sync.range_ready(a.grads, self.block_grad_hi(l))
        self.trunk.backward(ws, {}, dx_init=True, on_block_done=on_done)
        ws.busy = False
