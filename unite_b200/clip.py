"""Frozen CLIP ViT teacher — inference only, on the CUDA kernels.

Drop-in surface of reference src/models/clip.py: `VisionTransformer` :106 (same constructor kwargs, OpenAI-CLIP
state_dict names: class_embedding, positional_embedding, proj, conv1.weight, ln_pre.*,
transformer.resblocks.{i}.{attn.in_proj_weight,attn.in_proj_bias,attn.out_proj.*,ln_1.*,mlp.c_fc.*,mlp.c_proj.*,ln_2.*},
ln_post.*), `forward(x, mask=None)` returning (feat [K,B,T*HW,C], attn [B*T,HW]) when return_attn, and the
factories clip_b16 / clip_l14 / clip_l14_336 :234-295 plus the checkpoint adapter load_state_dict :191-231.

B200-first differences behind that surface: per-frame sequences are processed batch-first from one im2col
matrix shared with the student; layers 6..11 are kept in fp32 and ln_post + projection + L2-normalise run ONLY on
the visible rows once the mask is known (`project_rows`), instead of on all 1568 tokens of which 80 % are thrown
away (run_stage1.py:393); the last layer's attention map is produced from the CLS query row alone.
"""
from collections import OrderedDict
from typing import Dict, List, Optional

import torch
import torch.nn as nn

from . import ops
from .modeling_finetune import _ParamsOnly

BF16, F32, I32 = torch.bfloat16, torch.float32, torch.int32
# Residual stream of the (frozen, inference-only) teacher: fp16, which is what the reference's torch.cuda.amp.autocast region
# keeps it in (run_stage1.py:360-377 runs the teacher under autocast; clip.LayerNorm casts to fp32 and back, clip.py:20-26).
# Against the fp32 oracle it costs 7.7e-4 mean / 1.0e-3 max per-token feature error (simulated on the CPU oracle, ViT-B/16)
# next to the 5e-3 the bf16 GEMM operands cost; it halves the bytes of every LayerNorm read and residual epilogue.
# UB_TEACHER_STREAM=fp32 restores the fp32 stream.
import os as _os
STREAM = F32 if _os.environ.get("UB_TEACHER_STREAM", "fp16") == "fp32" else torch.float16
# ln_1 / ln_2 folded into the QKV / c_fc GEMMs (needs the fp16 stream): the GEMM reads the raw residual stream x as its fp16 A
# operand against B = fp16(gamma o W); its epilogue applies rstd_m * (acc - mu_m * c_n) + (beta W^T + b)_n with the row
# statistics the producer of x accumulated in ITS epilogue.  Algebraically identical to Linear(LayerNorm(x)); 24 LayerNorm
# launches and their 154 MB each disappear, and the operands carry 11 instead of 8 mantissa bits.  UB_TEACHER_LNFOLD=0: off.
LNFOLD = STREAM == torch.float16 and _os.environ.get("UB_TEACHER_LNFOLD", "1") != "0"


class LayerNorm(nn.LayerNorm):
    """fp32 LayerNorm parameters (clip.py:20-26); statistics are always fp32 in the kernels."""


class QuickGELU(_ParamsOnly):
    pass


class ResidualAttentionBlock(_ParamsOnly):
    def __init__(self, d_model, n_head, attn_mask=None):
        super().__init__()
        if attn_mask is not None:
            raise NotImplementedError("attn_mask is never used by the vision tower")
        self.attn = nn.MultiheadAttention(d_model, n_head)   # parameter holder: in_proj_weight/bias, out_proj
        self.ln_1 = LayerNorm(d_model)
        self.mlp = nn.Sequential(OrderedDict([("c_fc", nn.Linear(d_model, d_model * 4)), ("gelu", QuickGELU()),
                                              ("c_proj", nn.Linear(d_model * 4, d_model))]))
        self.ln_2 = LayerNorm(d_model)


class Transformer(_ParamsOnly):
    def __init__(self, width, layers, heads, return_attn=False, clip_return_layers=[6, 7, 8, 9, 10, 11], clip_return_interval=1,
                 return_cls=False):
        super().__init__()
        self.layers, self.return_attn, self.return_cls = layers, return_attn, return_cls
        self.resblocks = nn.ModuleList([ResidualAttentionBlock(width, heads) for _ in range(layers)])
        self.return_index = list(clip_return_layers)


class VisionTransformer(nn.Module):
    def __init__(self, input_resolution, patch_size, width, layers, heads, output_dim, clip_norm_type="l2", kernel_size=1,
                 return_attn=False, clip_return_layers=[6, 7, 8, 9, 10, 11], clip_return_interval=1, return_cls=False):
        super().__init__()
        if clip_norm_type != "l2":
            raise NotImplementedError("clip_norm_type must be 'l2'")
        if patch_size not in (14, 16):
            raise NotImplementedError(f"patch_size {patch_size}: the teacher runs 14x14 (clip_l14) or 16x16 (clip_b16) patches")
        if width // heads != 64:
            raise NotImplementedError("the attention kernels are specialised for head_dim 64")
        self.clip_norm_type, self.return_attn, self.return_cls = clip_norm_type, return_attn, return_cls
        self.output_dim, self.width, self.heads, self.kernel_size = output_dim, width, heads, kernel_size
        self.input_resolution, self.patch_size = input_resolution, patch_size
        # conv1 runs as a GEMM over im2col rows of 3*ks*p*p features, padded to a multiple of 64 (588 for a 14-pixel patch)
        self.k_pad = ops.padded_k(3 * kernel_size * patch_size * patch_size)
        self.conv1 = nn.Conv3d(3, width, (kernel_size, patch_size, patch_size), (kernel_size, patch_size, patch_size), (0, 0, 0),
                               bias=False)
        scale = width ** -0.5
        self.class_embedding = nn.Parameter(scale * torch.randn(width))
        self.positional_embedding = nn.Parameter(scale * torch.randn((input_resolution // patch_size) ** 2 + 1, width))
        self.ln_pre = LayerNorm(width)
        self.transformer = Transformer(width, layers, heads, return_attn=return_attn, clip_return_layers=clip_return_layers,
                                       clip_return_interval=clip_return_interval, return_cls=return_cls)
        self.ln_post = LayerNorm(width)
        self.proj = nn.Parameter(scale * torch.randn(width, output_dim))
        self._w16: Optional[Dict[str, torch.Tensor]] = None
        self._w_version = None
        self._bufs: Dict = {}

    # ---- weights ---------------------------------------------------------------------------
    def _weights(self):
        """bf16 GEMM operands, refreshed when a parameter changed (the teacher is frozen: normally once)."""
        v = (sum(p._version for p in self.parameters()), self.proj.data_ptr())
        dev = self.proj.device
        if dev.type != "cuda":
            raise RuntimeError("unite_b200 models compute on CUDA only: call teacher.cuda() first (there is no CPU path)")
        if self._w16 is None or v != self._w_version or self._w16["proj_t"].device != dev:
            W = self.width
            conv1 = self.conv1.weight.detach().reshape(W, -1)
            w = {"conv1": torch.nn.functional.pad(conv1, (0, self.k_pad - conv1.shape[1])).to(BF16).contiguous(),
                 "proj_t": self.proj.detach().t().to(BF16).contiguous()}
            for i, blk in enumerate(self.transformer.resblocks):
                w[f"{i}.in_proj"] = blk.attn.in_proj_weight.detach().to(BF16).contiguous()
                w[f"{i}.out_proj"] = blk.attn.out_proj.weight.detach().to(BF16).contiguous()
                w[f"{i}.c_fc"] = blk.mlp.c_fc.weight.detach().to(BF16).contiguous()
                w[f"{i}.c_proj"] = blk.mlp.c_proj.weight.detach().to(BF16).contiguous()
                if LNFOLD:
                    for name, ln, lin_w, lin_b in ((f"{i}.in_proj", blk.ln_1, blk.attn.in_proj_weight, blk.attn.in_proj_bias),
                                                   (f"{i}.c_fc", blk.ln_2, blk.mlp.c_fc.weight, blk.mlp.c_fc.bias)):
                        Wf = lin_w.detach().float()
                        wg = (Wf * ln.weight.detach().float()[None, :]).to(torch.float16).contiguous()      # gamma o W
                        w[name + ".fold"] = wg
                        w[name + ".fold_c"] = wg.float().sum(dim=1).contiguous()                            # c_n = sum_k B[n,k]
                        w[name + ".fold_d"] = (Wf @ ln.bias.detach().float() + lin_b.detach().float()).contiguous()
            self._w16, self._w_version = w, v
        return self._w16

    def _work_buffers(self, frames, P):
        key = (frames, P)
        if key not in self._bufs:
            dev, W = self.proj.device, self.width
            R = frames * (P + 1)
            K = len(self.transformer.return_index)
            self._bufs[key] = dict(
                E=torch.empty(frames * P, W, device=dev, dtype=F32),
                x=[torch.empty(R, W, device=dev, dtype=STREAM) for _ in range(K + 2)],   # work, mid, K snapshots
                stats=torch.zeros(2 * len(self.transformer.resblocks), R, 2, device=dev, dtype=F32),   # LN fold: row (sum, sumsq)
                h=torch.empty(R, W, device=dev, dtype=BF16), qkv=torch.empty(R, 3 * W, device=dev, dtype=BF16),
                o=torch.empty(R, W, device=dev, dtype=BF16), u=torch.empty(R, 4 * W, device=dev, dtype=BF16))
        return self._bufs[key]

    # ---- compute ---------------------------------------------------------------------------
    @torch.no_grad()
    def forward_features(self, x, patches=None, select=None, resolution=None):
        """Runs the tower on the clip x fp32 [B,3,T,H,W] seen at `resolution` x `resolution` (None: H).  When that differs
        from H or W the clip is resized on the device (bicubic, as the reference's engine does before its teacher call);
        `patches` (bf16 im2col rows [frames*P, k_pad] of the clip at that resolution) are used as they are.
        Returns (layers: list of K fp32 [B*T'*(HW+1), W] residual-stream snapshots after the blocks in clip_return_layers,
        attn fp32 [B*T', HW] or None, patches bf16 im2col rows).

        select: optional callable(attn) -> int32 row indices (into the [frames*(HW+1)] token stream) of the tokens whose
        features will be used.  The LAST block's attention map only needs its QKV projection, and nothing after it reads
        the other tokens, so when the last block is a returned layer its out_proj / MLP run on the selected rows only
        (80 % fewer rows in stage 1); that snapshot is then [n_selected, W] and `self.last_gathered` is True."""
        w = self._weights()
        B, _, T, H, Wd = x.shape
        ks, W, p = self.kernel_size, self.width, self.patch_size
        R = H if resolution is None else int(resolution)
        resize = R != H or R != Wd
        if R % p or (not resize and Wd % p):
            raise ValueError(f"teacher resolution {R}x{R if resize else Wd} is not a multiple of its patch size {p}")
        Tp, P = T // ks, (R // p) * ((R if resize else Wd) // p)
        if P + 1 != self.positional_embedding.shape[0]:
            raise ValueError(f"the teacher sees {P} patches per frame at {R} px, but its positional embedding holds "
                             f"{self.positional_embedding.shape[0] - 1} (input_resolution {self.input_resolution}, patch size {p})")
        frames = B * Tp
        if patches is None:
            patches = torch.empty(frames * P, self.k_pad, device=x.device, dtype=BF16)
            if p == 16 and not resize:
                ops.patchify(x.contiguous(), patches, ks)
            else:
                ops.resize_patchify(x.contiguous(), patches, R, p, ks)
        bufs = self._work_buffers(frames, P)
        S = P + 1
        ops.gemm(patches, w["conv1"], bufs["E"])
        xs = bufs["x"]
        work, mid, snaps = xs[0], xs[1], xs[2:]
        cur = work
        stats = bufs["stats"] if LNFOLD else None
        if LNFOLD:
            stats.zero_()
        ops.teacher_embed_ln(bufs["E"], self.class_embedding.detach(), self.positional_embedding.detach(), self.ln_pre.weight.detach(),
                             self.ln_pre.bias.detach(), self.ln_pre.eps, cur, frames, P, W, stats=stats[0] if LNFOLD else None)
        keep: List[torch.Tensor] = []
        attn = None
        ret = self.transformer.return_index
        nblk = len(self.transformer.resblocks)
        scale = 64 ** -0.5
        self.last_gathered = False
        for i, blk in enumerate(self.transformer.resblocks):
            if LNFOLD:
                ops.gemm(cur, w[f"{i}.in_proj.fold"], bufs["qkv"], bias=w[f"{i}.in_proj.fold_d"], ln_stats=stats[2 * i],
                         ln_c=w[f"{i}.in_proj.fold_c"], ln_eps=blk.ln_1.eps)
            else:
                ops.layernorm_fwd(cur, blk.ln_1.weight.detach(), blk.ln_1.bias.detach(), blk.ln_1.eps, bufs["h"])
                ops.gemm(bufs["h"], w[f"{i}.in_proj"], bufs["qkv"], bias=blk.attn.in_proj_bias.detach())
            if i == nblk - 1 and self.return_attn:
                attn = torch.empty(frames, P, device=x.device, dtype=F32)
                ops.cls_attn(bufs["qkv"], attn, frames, S, self.heads, scale)
            ops.attn_fwd(bufs["qkv"], bufs["o"], None, frames, S, self.heads, scale)
            if i == nblk - 1 and select is not None and attn is not None and i in ret:
                rows = select(attn)
                n = rows.numel()
                tb = self._tail_buffers(n)
                ops.gather_rows(bufs["o"], rows, tb["o"])
                ops.gather_rows(cur, rows, tb["x"])
                if LNFOLD:
                    tb["stats"].zero_()
                    ops.gemm(tb["o"], w[f"{i}.out_proj"], tb["mid"], bias=blk.attn.out_proj.bias.detach(), residual=tb["x"],
                             stats_out=tb["stats"])
                    ops.gemm(tb["mid"], w[f"{i}.c_fc.fold"], tb["u"], bias=w[f"{i}.c_fc.fold_d"], act=ops.UB_ACT_QUICKGELU,
                             ln_stats=tb["stats"], ln_c=w[f"{i}.c_fc.fold_c"], ln_eps=blk.ln_2.eps)
                else:
                    ops.gemm(tb["o"], w[f"{i}.out_proj"], tb["mid"], bias=blk.attn.out_proj.bias.detach(), residual=tb["x"])
                    ops.layernorm_fwd(tb["mid"], blk.ln_2.weight.detach(), blk.ln_2.bias.detach(), blk.ln_2.eps, tb["h"])
                    ops.gemm(tb["h"], w[f"{i}.c_fc"], tb["u"], bias=blk.mlp.c_fc.bias.detach(), act=ops.UB_ACT_QUICKGELU)
                ops.gemm(tb["u"], w[f"{i}.c_proj"], tb["out"], bias=blk.mlp.c_proj.bias.detach(), residual=tb["mid"])
                keep.append(tb["out"])
                self.last_gathered = True
                self.last_stream = None
                return keep, attn, patches
            if LNFOLD:
                ops.gemm(bufs["o"], w[f"{i}.out_proj"], mid, bias=blk.attn.out_proj.bias.detach(), residual=cur, stats_out=stats[2 * i + 1])
                ops.gemm(mid, w[f"{i}.c_fc.fold"], bufs["u"], bias=w[f"{i}.c_fc.fold_d"], act=ops.UB_ACT_QUICKGELU,
                         ln_stats=stats[2 * i + 1], ln_c=w[f"{i}.c_fc.fold_c"], ln_eps=blk.ln_2.eps)
            else:
                ops.gemm(bufs["o"], w[f"{i}.out_proj"], mid, bias=blk.attn.out_proj.bias.detach(), residual=cur)
                ops.layernorm_fwd(mid, blk.ln_2.weight.detach(), blk.ln_2.bias.detach(), blk.ln_2.eps, bufs["h"])
                ops.gemm(bufs["h"], w[f"{i}.c_fc"], bufs["u"], bias=blk.mlp.c_fc.bias.detach(), act=ops.UB_ACT_QUICKGELU)
            # a returned layer gets its own snapshot buffer (never written again); others go to the work buffer
            dst = snaps[len(keep)] if i in ret else work
            ops.gemm(bufs["u"], w[f"{i}.c_proj"], dst, bias=blk.mlp.c_proj.bias.detach(), residual=mid,
                     stats_out=stats[2 * i + 2] if (LNFOLD and i + 1 < nblk) else None)
            cur = dst
            if i in ret:
                keep.append(cur)
        self.last_stream = cur        # residual stream after the final block (CLS rows feed the stage-3 zero-shot head)
        return keep, attn, patches

    def _tail_buffers(self, n):
        key = ("tail", n)
        if key not in self._bufs:
            dev, W = self.proj.device, self.width
            self._bufs[key] = dict(o=torch.empty(n, W, device=dev, dtype=BF16), x=torch.empty(n, W, device=dev, dtype=STREAM),
                                   mid=torch.empty(n, W, device=dev, dtype=STREAM), h=torch.empty(n, W, device=dev, dtype=BF16),
                                   u=torch.empty(n, 4 * W, device=dev, dtype=BF16), out=torch.empty(n, W, device=dev, dtype=STREAM),
                                   stats=torch.zeros(n, 2, device=dev, dtype=F32))
        return self._bufs[key]

    @torch.no_grad()
    def project_rows(self, layers: List[torch.Tensor], rows: torch.Tensor) -> torch.Tensor:
        """ln_post -> @proj -> L2-normalise (clip.py:168-173) on the given residual-stream rows only.
        rows int32 [n] (row index into each layer snapshot; a snapshot that already holds exactly those n rows — the
        truncated last block of forward_features(select=...) — is used as is).  Returns fp32 [K, n, output_dim]."""
        w = self._weights()
        K, n = len(layers), rows.numel()
        dev = rows.device
        z = torch.empty(K * n, self.width, device=dev, dtype=BF16)
        for k, xk in enumerate(layers):
            gathered = getattr(self, "last_gathered", False) and k == K - 1 and xk.shape[0] == n
            ops.layernorm_fwd(xk, self.ln_post.weight.detach(), self.ln_post.bias.detach(), self.ln_post.eps, z[k * n:(k + 1) * n],
                              src_rows=None if gathered else rows)
        out = torch.empty(K * n, self.output_dim, device=dev, dtype=F32)
        ops.gemm(z, w["proj_t"], out)
        ops.l2norm_rows(out)
        return out.view(K, n, self.output_dim)

    @torch.no_grad()
    def cls_features(self, frames: int, P: int) -> torch.Tensor:
        """ln_post(CLS) @ proj, L2-normalised, of the last forward_features call: fp32 [frames, output_dim] — the image
        embedding OpenAI CLIP's encode_image returns (stand-in for the stage-3 zero-shot tower, utils.py:55-68)."""
        key = ("cls_rows", frames, P)
        if key not in self._bufs:
            self._bufs[key] = (torch.arange(frames, device=self.proj.device) * (P + 1)).to(I32).contiguous()
        return self.project_rows([self.last_stream], self._bufs[key])[0]

    def _all_patch_rows(self, B, Tp, P, dev):
        key = ("rows", B, Tp, P)
        if key not in self._bufs:
            f = torch.arange(B * Tp, device=dev).view(-1, 1) * (P + 1) + 1 + torch.arange(P, device=dev).view(1, -1)
            self._bufs[key] = f.reshape(-1).to(I32).contiguous()
        return self._bufs[key]

    @torch.no_grad()
    def forward(self, x, mask=None):
        """Reference-compatible call: (feat [K,B,T'*HW,C], attn [B*T',HW]) if return_attn else feat."""
        if mask is not None:
            raise NotImplementedError("the teacher `mask` argument is never passed by any UNITE driver (clip.py:154-160)")
        if self.return_cls:
            raise NotImplementedError("return_cls is off in every shipped config")
        B, _, T, H, Wd = x.shape
        p = self.patch_size
        P = (H // p) * (Wd // p)
        if H % p or Wd % p or P + 1 != self.positional_embedding.shape[0]:
            raise ValueError(f"a {H}x{Wd} clip does not match the teacher's patch grid: {p}-pixel patches and a positional embedding "
                             f"for {self.positional_embedding.shape[0] - 1} patches per frame (input_resolution {self.input_resolution}); "
                             "forward() does not resize, resize the clip to input_resolution first")
        Tp = T // self.kernel_size
        layers, attn, _ = self.forward_features(x)
        feat = self.project_rows(layers, self._all_patch_rows(B, Tp, P, x.device)).view(len(layers), B, Tp * P, self.output_dim)
        return (feat, attn) if self.return_attn else feat


def inflate_weight(weight_2d, time_dim, center=True):
    """2D -> 3D conv kernel inflation for kernel_size > 1 (clip.py:191-201)."""
    if center:
        w3 = torch.zeros(*weight_2d.shape).unsqueeze(2).repeat(1, 1, time_dim, 1, 1)
        w3[:, :, time_dim // 2, :, :] = weight_2d
        return w3
    return weight_2d.unsqueeze(2).repeat(1, 1, time_dim, 1, 1) / time_dim


def load_state_dict(model, state_dict, input_resolution=224, patch_size=16, center=True):
    """Checkpoint adapter (clip.py:203-231): inflate 2-D conv kernels, bicubic-resize the positional grid."""
    target = model.state_dict()
    state_dict = dict(state_dict)
    for k in list(state_dict.keys()):
        if k in target and state_dict[k].shape != target[k].shape:
            if len(target[k].shape) <= 2:
                continue
            state_dict[k] = inflate_weight(state_dict[k], target[k].shape[2], center=center)
    pos = state_dict["positional_embedding"]
    new_size = input_resolution // patch_size
    orig_size = int((pos.shape[-2] - 1) ** 0.5)
    if orig_size != new_size:
        grid = pos[1:].reshape(-1, orig_size, orig_size, pos.shape[-1]).permute(0, 3, 1, 2)
        grid = torch.nn.functional.interpolate(grid, size=(new_size, new_size), mode="bicubic", align_corners=False)
        state_dict["positional_embedding"] = torch.cat((pos[:1], grid.permute(0, 2, 3, 1).flatten(0, 2)), dim=0)
    model.load_state_dict(state_dict, strict=True)


def _factory(width, layers, heads, output_dim, patch_size):
    def build(pretrained=True, clip_norm_type="l2", input_resolution=224, kernel_size=1, return_attn=False, center=True,
              clip_return_layers=[6, 7, 8, 9, 10, 11], clip_return_interval=1, return_cls=False, checkpoint=None):
        model = VisionTransformer(input_resolution=input_resolution, patch_size=patch_size, width=width, layers=layers, heads=heads,
                                  output_dim=output_dim, clip_norm_type=clip_norm_type, kernel_size=kernel_size,
                                  return_attn=return_attn, clip_return_layers=clip_return_layers,
                                  clip_return_interval=clip_return_interval, return_cls=return_cls)
        if pretrained:
            if checkpoint is None:
                raise FileNotFoundError("pretrained CLIP weights are not available offline; pass pretrained=False (random init) or "
                                        "checkpoint=<path to the extracted visual-tower state_dict>")
            load_state_dict(model, torch.load(checkpoint, map_location="cpu"), input_resolution=input_resolution,
                            patch_size=patch_size, center=center)
        return model.eval()
    return build


clip_b16 = _factory(768, 12, 12, 512, 16)
clip_l14 = _factory(1024, 24, 16, 768, 14)
clip_l14_336 = _factory(1024, 24, 16, 768, 14)
