"""Explicit forward / backward of the student ViT trunk on the C-ABI kernels (no autograd inside).

This is the compute behind modeling_finetune.Block / Attention / Mlp / PatchEmbed (reference
src/models/modeling_finetune.py:56-175) and AdaptationVisionTransformerEncoder.forward_features
(src/models/modeling_adaptation.py:131-169) plus their backward.  The nn.Modules in modeling_*.py only hold
parameters (views into a ParamArena); every FLOP of the step runs through `ops` -> libunite_b200.so.

Data layout in HBM (M = B * N_tokens rows, D = embed dim):
    residual stream x[l]      fp32 [M, D]      one buffer per layer boundary (kept for LayerNorm backward)
    LN outputs h1/h2, attn o  bf16 [M, D]      GEMM A operands (and wgrad B operands)
    qkv                       bf16 [M, 3D]     per row q|k|v, heads x 64
    MLP pre-activation / act  bf16 [M, 4D]
    lse                       fp32 [B, H, N]
Weights are read from the arena's bf16 shadow; gradients are red.add-ed into the arena's fp32 grad buffer.
"""
import math
import os
from typing import Dict, List, Optional, Sequence

import torch

from . import ops
from .arena import ParamArena

BF16, F32 = torch.bfloat16, torch.float32


# fc1 bias gradient accumulated by the epilogue of the GEMM that produces d_pre (ub_gemm_epilogue.colsum_out) instead of a
# separate column-sum pass over d_pre: 12 launches and 12 x 63 MB of reads fewer per ViT-B step
_FUSE_COLSUM = os.environ.get("UB_FUSE_COLSUM", "0") == "1"
# q_bias / v_bias gradients accumulated by the attention backward kernels while they store dq / dv (ub_attn_bwd's dbias) instead
# of a separate column-sum pass over dqkv: 12 launches fewer per ViT-B step.  UB_FUSE_QKV_BIAS=0 restores the separate pass.
_FUSE_QKV_BIAS = os.environ.get("UB_FUSE_QKV_BIAS", "1") == "1"
# The four weight gradients of a block (fc2, fc1, proj, qkv: same tokens, different widths) as ONE multi-problem launch at the end
# of the block's backward (ub_gemm_wgrad_multi) instead of four: one prologue / pipeline fill / drain and one wave quantisation
# on the 74 CTA pairs (108 pair tiles x split-K 2 = 216 items = 2.9 waves) instead of four.  UB_MULTI_WGRAD=0: separate launches.
_MULTI_WGRAD = os.environ.get("UB_MULTI_WGRAD", "1") == "1"
# D = rowsum(dO o O) of the attention backward from the epilogue of the GEMM that produces dO (ub_gemm_epilogue.dot_out) instead of
# a separate pass over O and dO per layer.  UB_FUSE_DPREP=0: separate pre-pass inside ub_attn_bwd.
_FUSE_DPREP = os.environ.get("UB_FUSE_DPREP", "1") == "1"
_FORCE_WGRAD_SPLIT = int(os.environ.get("UB_WGRAD_SPLIT", "0"))      # experiments: fixed split-K factor of the multi-problem launch


def _multi_splits(problems, units):
    """split-K factor for a multi-problem weight-gradient launch: the SMALLEST one that fills the waves of `units` CTA pairs to
    >= 93 % (every extra split is another fp32 reduce-add pass over the weight-gradient tiles), >= 32 k-blocks per item."""
    if _FORCE_WGRAD_SPLIT > 0:
        return _FORCE_WGRAD_SPLIT
    tiles = sum(((gw.shape[0] + 255) // 256) * ((gw.shape[1] + 255) // 256) for _, _, gw in problems)
    kb = (problems[0][0].shape[0] + 63) // 64
    best, best_eff = 1, 0.0
    for s_ in range(1, 9):
        if s_ > 1 and kb // s_ < 32:
            break
        items = tiles * s_
        eff = items / (((items + units - 1) // units) * units)
        if eff >= 0.93:
            return s_
        if eff > best_eff + 1e-9:
            best, best_eff = s_, eff
    return best


def _splits_for(out_rows: int, out_cols: int, sms: int) -> int:
    tiles = ((out_rows + 127) // 128) * ((out_cols + 255) // 256)
    return max(1, min(32, sms // max(1, tiles)))


class DropPathSource:
    """Per-step DropPath factors [depth, 2, B] from the device generator (ops.drop_path_draw): one launch per step, no host
    random numbers, replayable in a CUDA graph.  `step` (device int64) counts the draws made; oracle/philox.py reproduces the
    factors of any (seed, step) on the host."""

    def __init__(self, rates, device, seed=0):
        self.rates = [float(r) for r in rates]
        self.active = any(r > 0 for r in self.rates)
        self.seed = seed
        self.device = device
        if self.active:
            self.rates_dev = torch.tensor(self.rates, dtype=F32, device=device)
            self.step = torch.zeros(1, dtype=torch.int64, device=device)
        self._out = {}

    def draw(self, B, slot=0):
        """`slot` distinguishes buffers that must stay alive together (several forwards before one backward, stage 3)."""
        if not self.active:
            return None
        key = (B, slot)
        if key not in self._out:
            self._out[key] = torch.empty(len(self.rates), 2, B, dtype=F32, device=self.device)
        return ops.drop_path_draw(self.rates_dev, self._out[key], self.seed, self.step)


class _LayerBufs:
    __slots__ = ("h1", "qkv", "o", "lse", "x_mid", "h2", "pre", "act")


class TrunkWorkspace:
    """Activation storage for one (B, N) shape.  `save=True` keeps every layer's activations for backward;
    `save=False` reuses one layer's buffers for all layers (inference)."""

    def __init__(self, dev, M, B, N, D, H, hidden, depth, save):
        self.M, self.B, self.N, self.save = M, B, N, save
        self.busy = False
        n_x = depth + 1 if save else 2
        self.x = [torch.empty(M, D, device=dev, dtype=F32) for _ in range(n_x)]
        self.layers: List[_LayerBufs] = []
        for _ in range(depth if save else 1):
            L = _LayerBufs()
            L.h1 = torch.empty(M, D, device=dev, dtype=BF16)
            L.qkv = torch.empty(M, 3 * D, device=dev, dtype=BF16)
            L.o = torch.empty(M, D, device=dev, dtype=BF16)
            L.lse = torch.empty(B, H, N, device=dev, dtype=F32)
            L.x_mid = torch.empty(M, D, device=dev, dtype=F32)
            L.h2 = torch.empty(M, D, device=dev, dtype=BF16)
            L.pre = torch.empty(M, hidden, device=dev, dtype=BF16)
            L.act = torch.empty(M, hidden, device=dev, dtype=BF16)
            self.layers.append(L)
        if save:  # backward temporaries, shared by all layers
            self.dx = torch.empty(M, D, device=dev, dtype=F32)
            # two copies (layer parity): block l's weight gradients are one launch at the END of its backward (UB_MULTI_WGRAD), and
            # before it runs, block l's norm1 LayerNorm backward writes dxs_m of layer l-1, while the launch still reads layer l's
            self.dxs_m = [torch.empty(M, D, device=dev, dtype=BF16) for _ in range(2)]     # gradient entering the MLP branch
            self.dxs_a = [torch.empty(M, D, device=dev, dtype=BF16) for _ in range(2)]     # ... the attention branch
            self.d_pre2 = [torch.empty(M, hidden, device=dev, dtype=BF16) for _ in range(2)]
            self.dqkv2 = [torch.empty(M, 3 * D, device=dev, dtype=BF16) for _ in range(2)]
            self.dxs, self.d_pre, self.dqkv = self.dxs_m[0], self.d_pre2[0], self.dqkv2[0]
            self.d_h = torch.empty(M, D, device=dev, dtype=BF16)
            self.d_o = torch.empty(M, D, device=dev, dtype=BF16)
            self.d_ws = torch.empty(B, H, N, device=dev, dtype=F32)

    def layer(self, l):
        return self.layers[l if self.save else 0]

    def x_at(self, l):
        return self.x[l if self.save else l & 1]


class ViTTrunk:
    """patch-embed GEMM + `depth` pre-LN transformer blocks, forward and backward."""

    def __init__(self, arena: ParamArena, prefix: str, D: int, depth: int, heads: int, hidden: int, eps: float):
        assert D % heads == 0 and D // heads == 64, "the attention kernels are specialised for head_dim 64"
        self.arena, self.prefix = arena, prefix
        self.D, self.depth, self.H, self.hidden, self.eps = D, depth, heads, hidden, eps
        self.scale = 64 ** -0.5
        self.sms = ops.lib.ub_sm_count() if torch.cuda.is_available() else 148
        self._ws: Dict = {}

    # -- parameter access ---------------------------------------------------------------------
    def w(self, name):       # bf16 shadow (GEMM operand)
        return self.arena.b16(self.prefix + name)

    def p(self, name):       # fp32 master (biases, LN affine)
        return self.arena.p32(self.prefix + name)

    def g(self, name):       # fp32 gradient
        return self.arena.g32(self.prefix + name)

    def qkv_bias(self, l):   # [q_bias | 0 | v_bias], contiguous in the arena by construction
        o, k = self.arena.offsets[f"{self.prefix}blocks.{l}.attn.q_bias"]
        return self.arena.params[o:o + 3 * k]

    def qkv_bias_grad(self, l):
        o, k = self.arena.offsets[f"{self.prefix}blocks.{l}.attn.q_bias"]
        return self.arena.grads[o:o + 3 * k]

    def workspace(self, B, N, save) -> TrunkWorkspace:
        """Workspaces holding saved activations stay `busy` until their backward ran, so a second graph-attached
        forward of the same shape (stage 3 runs several before one backward) gets its own buffers."""
        pool = self._ws.setdefault((B, N, save), [])
        for ws in pool:
            if not ws.busy:
                break
        else:
            ws = TrunkWorkspace(self.arena.device, B * N, B, N, self.D, self.H, self.hidden, self.depth, save)
            pool.append(ws)
        ws.busy = save
        return ws

    # -- forward ------------------------------------------------------------------------------
    def forward(self, patches: torch.Tensor, pos_rows: torch.Tensor, B: int, N: int, n_layers: int, save: bool,
                dp: Optional[torch.Tensor] = None, after_layer=None) -> TrunkWorkspace:
        """patches bf16 [B*N, 3*tub*256] (rows already gathered), pos_rows fp32 [B*N, D].
        dp: optional DropPath factors fp32 [depth, 2, B] (attn branch, mlp branch).
        after_layer(l, x_out): called right after block l (its output buffer is only guaranteed to survive
        until the next block when save=False)."""
        ws = self.workspace(B, N, save)
        D = self.D
        x = ws.x_at(0)
        ops.gemm(patches, self.w("patch_embed.proj.weight").view(D, -1), x, bias=self.p("patch_embed.proj.bias"),
                 residual=pos_rows)
        for l in range(n_layers):
            L = ws.layer(l)
            b = f"blocks.{l}."
            ops.layernorm_fwd(x, self.p(b + "norm1.weight"), self.p(b + "norm1.bias"), self.eps, L.h1)
            ops.gemm(L.h1, self.w(b + "attn.qkv.weight"), L.qkv, bias=self.qkv_bias(l))
            ops.attn_fwd(L.qkv, L.o, L.lse, B, N, self.H, self.scale)
            ops.gemm(L.o, self.w(b + "attn.proj.weight"), L.x_mid, bias=self.p(b + "attn.proj.bias"), residual=x,
                     row_scale=None if dp is None else dp[l, 0], rows_per_scale=N)
            ops.layernorm_fwd(L.x_mid, self.p(b + "norm2.weight"), self.p(b + "norm2.bias"), self.eps, L.h2)
            ops.gemm(L.h2, self.w(b + "mlp.fc1.weight"), L.act, bias=self.p(b + "mlp.fc1.bias"), act=ops.UB_ACT_GELU,
                     aux_out=L.pre if save else None)
            xn = ws.x_at(l + 1)
            ops.gemm(L.act, self.w(b + "mlp.fc2.weight"), xn, bias=self.p(b + "mlp.fc2.bias"), residual=L.x_mid,
                     row_scale=None if dp is None else dp[l, 1], rows_per_scale=N)
            x = xn
            if after_layer is not None:
                after_layer(l, x)
        ws.n_layers = n_layers
        ws.patches = patches
        ws.dp = dp
        return ws

    # -- backward -----------------------------------------------------------------------------
    def _wgrad(self, dy, x_in, gw):
        """gw[out,in] += dy[M,out]^T @ x_in[M,in]  (contraction over tokens, both operands MN-major)."""
        ops.gemm(dy, x_in, gw, a_t=True, b_t=True, accumulate=True, split_k=_splits_for(gw.shape[0], gw.shape[1], self.sms))

    def backward(self, ws: TrunkWorkspace, tap_grads: Dict[int, callable], dx_init: bool = False, on_block_done=None):
        """Back-propagates through blocks n_layers-1 .. 0 and the patch embedding.

        tap_grads[l](dx_in, dxs_out, row_scale, dsum) must add the gradient arriving at the OUTPUT of block l into the
        residual-gradient buffer ws.dx (dx_in is None when nothing has been accumulated yet), emit
        dxs_out = bf16(ws.dx * row_scale) and accumulate its column sums (block l's fc2 bias gradient) into dsum.  If dx_init is True, ws.dx already holds the gradient wrt the last
        block's output."""
        N, D = ws.N, self.D
        dp = ws.dp
        have_dx = dx_init
        nl = ws.n_layers
        multi = _MULTI_WGRAD and ws.dx.is_cuda
        pending = []                                    # this block's (dy, x, gw) triples, issued as one launch at its end

        def wgrad(dy, x_in, gw):
            if multi:
                pending.append((dy, x_in, gw))
            else:
                self._wgrad(dy, x_in, gw)

        for l in reversed(range(nl)):
            L = ws.layer(l)
            b = f"blocks.{l}."
            par = l & 1
            dxs_m, dxs_a, d_pre, dqkv = ws.dxs_m[par], ws.dxs_a[par], ws.d_pre2[par], ws.dqkv2[par]
            s_mlp = None if dp is None else dp[l, 1]
            s_att = None if dp is None else dp[l, 0]
            # the producer of dxs also accumulates its column sums = the bias gradient of the Linear it feeds
            if l in tap_grads:
                tap_grads[l](ws.dx if have_dx else None, dxs_m, s_mlp, self.g(b + "mlp.fc2.bias"))
                have_dx = True
            elif l == nl - 1:
                assert have_dx, "no gradient reaches the last block"
                ops.cast_scale_bf16(ws.dx, dxs_m, s_mlp, N)
                ops.colsum_bf16(dxs_m, self.g(b + "mlp.fc2.bias"))
            # ---- MLP branch: x_out = x_mid + s * (gelu(h2 W1^T + b1) W2^T + b2)
            # with _FUSE_COLSUM the fc1 bias gradient (column sums of d_pre) is accumulated by this GEMM's epilogue
            ops.gemm(dxs_m, self.w(b + "mlp.fc2.weight"), d_pre, b_t=True, act=ops.UB_ACT_DGELU, aux_in=L.pre,
                     colsum_out=self.g(b + "mlp.fc1.bias") if _FUSE_COLSUM else None)
            wgrad(dxs_m, L.act, self.g(b + "mlp.fc2.weight"))
            ops.gemm(d_pre, self.w(b + "mlp.fc1.weight"), ws.d_h, b_t=True)
            wgrad(d_pre, L.h2, self.g(b + "mlp.fc1.weight"))
            if not _FUSE_COLSUM:
                ops.colsum_bf16(d_pre, self.g(b + "mlp.fc1.bias"))
            ops.layernorm_bwd(ws.d_h, L.x_mid, self.p(b + "norm2.weight"), self.eps, ws.dx, ws.dx, dxs_a, s_att, N,
                              self.g(b + "norm2.weight"), self.g(b + "norm2.bias"), dsum=self.g(b + "attn.proj.bias"))
            # ---- attention branch: x_mid = x_in + s * (attn(h1) Wp^T + bp)
            if _FUSE_DPREP:
                # the proj dgrad GEMM that produces dO also leaves D = rowsum(dO o O) per (token, head) for the attention backward
                ops.gemm(dxs_a, self.w(b + "attn.proj.weight"), ws.d_o, b_t=True, act=ops.UB_ACT_DOT_AUX, aux_in=L.o, dot_out=ws.d_ws,
                         dot_seq_len=N)
            else:
                ops.gemm(dxs_a, self.w(b + "attn.proj.weight"), ws.d_o, b_t=True)
            wgrad(dxs_a, L.o, self.g(b + "attn.proj.weight"))
            # q_bias | (always-zero k gap) | v_bias are one contiguous 3D span of the gradient arena; the attention backward adds the
            # column sums of dq and dv into it as it stores them (the key bias is structurally zero, modeling_finetune.py:104)
            ops.attn_bwd(L.qkv, None if _FUSE_DPREP else L.o, ws.d_o, L.lse, ws.d_ws, dqkv, ws.B, N, self.H, self.scale,
                         dbias=self.qkv_bias_grad(l) if _FUSE_QKV_BIAS else None)
            ops.gemm(dqkv, self.w(b + "attn.qkv.weight"), ws.d_h, b_t=True)
            wgrad(dqkv, L.h1, self.g(b + "attn.qkv.weight"))
            if not _FUSE_QKV_BIAS:
                ops.colsum_bf16(dqkv, self.qkv_bias_grad(l), skip=(D, 2 * D))
            # next consumer of dxs: block l-1's MLP branch (unless a tap re-emits it) or the patch embedding
            emit = (l - 1) not in tap_grads
            s_next = None if (dp is None or l == 0) else dp[l - 1, 1]
            next_bias = self.g("patch_embed.proj.bias") if l == 0 else self.g(f"blocks.{l - 1}.mlp.fc2.bias")
            ops.layernorm_bwd(ws.d_h, ws.x_at(l), self.p(b + "norm1.weight"), self.eps, ws.dx, ws.dx,
                              ws.dxs_m[(l - 1) & 1] if emit else None, s_next, N, self.g(b + "norm1.weight"),
                              self.g(b + "norm1.bias"), dsum=next_bias if emit else None)
            if multi:
                ops.gemm_wgrad_multi(pending, split_k=_multi_splits(pending, max(1, self.sms // 2)))
                pending.clear()
            if on_block_done is not None:
                on_block_done(l)     # every gradient of block l is final: its arena range can be all-reduced
        # ---- patch embedding (Conv3d as GEMM): only weight and bias gradients exist
        gw = self.g("patch_embed.proj.weight")
        self._wgrad(ws.dxs_m[1], ws.patches, gw.view(D, -1))
