"""fp64 reference of the attention entry points (ub_attn_fwd / ub_attn_bwd, head_dim 64, non-causal), the per-row error bounds
the kernels are judged by, and seeded input builders, including inputs that put rows on each kernel's slow path.

Layouts are the library's: qkv bf16 [n_seq*S, 3*H*64] (per token q|k|v, each H heads x 64), o / d_o bf16 [n_seq*S, H*64],
lse / D [n_seq, H, S].  The reference works per item (sequence, head) as [n_seq*H, S, 64] and processes items in chunks, so memory
stays bounded (S^2 * 8 B is 19.7 MB per item at S = 1568).  It runs on whatever device its inputs are on.

Error bounds are per (sequence, head, row), against a scale that row's own math sets (P is the fp64 softmax, s the softmax scale):
    O_i     2^-7 max_d sum_j P_ij |v_jd|          bf16 P (2^-9) + bf16 output (2^-9), times 2 for margin
    lse_i   2^-8 + 2^-20 |lse_i|                  the kernels sum the bf16-rounded P: up to 2^-9 of the row sum
    dV_j    2^-7 max_d sum_i P_ij |dO_id|         bf16 P + bf16 output, times 2
    dQ_i    2^-6 s max_d sum_j P_ij (|dP_ij| + |D_i|) |k_jd|     bf16 dS + bf16 output + the lse the backward is given, times 4
    dK_j    the same as dQ, with q in place of k
Every bound has an absolute floor of 2^-20 times the item's largest scale of that output, for rows whose exact value is 0
(S = 1 gives dQ = dK = 0; a zero dO row gives dQ_i = 0).
"""
import math

import torch

LOG2E = 1.0 / math.log(2.0)
HD = 64
O_C, DV_C, DQK_C = 2.0 ** -7, 2.0 ** -7, 2.0 ** -6
LSE_ABS, LSE_REL = 2.0 ** -8, 2.0 ** -20
FLOOR = 2.0 ** -20

# the kernels' slow-path thresholds, in log2 units of the scores (score * scale * log2 e)
TC208_SPLIT, TC208_THRESHOLD = 96, 60.0          # attention_tc.cu, NK = 208: keys [0, 96) set the reference, redo above 2^60
FWD_LSE_SPLIT, FWD_LSE_THRESHOLD = 160, 64.0     # attention_fwd_lse_tc.cu: second 160-key chunk, move above 2^64
LONG_CHUNK, LONG_THRESHOLD = 64, 40.0            # attention_long_tc.cu forward: 64-key chunks, move above 2^40
WARP_ROWS = 32                                   # the kernels decide a slow path per warp, i.e. per 32-row block of a sequence


# ---------------------------------------------------------------------------------------------------------------- layouts
def heads(x, n_seq, S, H, part=None):
    """qkv (part 0 / 1 / 2 = q / k / v) or o-shaped rows -> fp64 [n_seq*H, S, 64]."""
    if part is None:
        return x.view(n_seq, S, H, HD).permute(0, 2, 1, 3).reshape(n_seq * H, S, HD).double()
    return x.view(n_seq, S, 3, H, HD)[:, :, part].permute(0, 2, 1, 3).reshape(n_seq * H, S, HD).double()


def _chunks(n_items, S, budget=1 << 24):
    step = max(1, budget // (S * S))
    for a in range(0, n_items, step):
        yield slice(a, min(n_items, a + step))


# ---------------------------------------------------------------------------------------------------------------- reference
def forward(qkv, n_seq, S, H, scale):
    """Exact attention of the bf16 qkv: dict of o [I,S,64], lse [I,S] and o_scale [I,S] (max_d sum_j P_ij |v_jd|), fp64."""
    q, k, v = (heads(qkv, n_seq, S, H, i) for i in range(3))
    o, lse, osc = torch.empty_like(q), q.new_empty(q.shape[:2]), q.new_empty(q.shape[:2])
    for c in _chunks(q.shape[0], S):
        s = scale * (q[c] @ k[c].transpose(1, 2))
        m = s.amax(-1, keepdim=True)
        e = torch.exp(s - m)
        l = e.sum(-1, keepdim=True)
        p = e / l
        o[c] = p @ v[c]
        lse[c] = (m + torch.log(l)).squeeze(-1)
        osc[c] = (p @ v[c].abs()).amax(-1)
    return dict(o=o, lse=lse, o_scale=osc)


def backward(qkv, d_o, n_seq, S, H, scale, o=None):
    """Exact gradients of the bf16 qkv under the bf16 d_o, from the explicit formulas
        D = rowsum(dO o O), dV = P^T dO, dP = dO V^T, dS = P o (dP - D), dQ = s dS K, dK = s dS^T Q.
    o: the O that D is formed from (the kernel's bf16 output, which is what the backward is given); None = the exact O.
    Returns fp64 dq / dk / dv [I,S,64], D [I,S] and the bound scales dq_scale / dk_scale / dv_scale [I,S]."""
    q, k, v = (heads(qkv, n_seq, S, H, i) for i in range(3))
    g = heads(d_o, n_seq, S, H)
    oo = heads(o, n_seq, S, H) if o is not None else None
    out = {n: torch.empty_like(q) for n in ("dq", "dk", "dv")}
    out.update({n: q.new_empty(q.shape[:2]) for n in ("D", "dq_scale", "dk_scale", "dv_scale")})
    for c in _chunks(q.shape[0], S):
        s = scale * (q[c] @ k[c].transpose(1, 2))
        p = torch.softmax(s, -1)
        D = ((oo[c] if oo is not None else p @ v[c]) * g[c]).sum(-1)
        dp = g[c] @ v[c].transpose(1, 2)
        ds = p * (dp - D[..., None])
        w = p * (dp.abs() + D.abs()[..., None])
        out["D"][c] = D
        out["dv"][c] = p.transpose(1, 2) @ g[c]
        out["dq"][c] = scale * (ds @ k[c])
        out["dk"][c] = scale * (ds.transpose(1, 2) @ q[c])
        out["dv_scale"][c] = (p.transpose(1, 2) @ g[c].abs()).amax(-1)
        out["dq_scale"][c] = scale * (w @ k[c].abs()).amax(-1)
        out["dk_scale"][c] = scale * (w.transpose(1, 2) @ q[c].abs()).amax(-1)
    return out


def row_ratio(got, ref, row_scale, c):
    """Per-row error / bound for a [I,S,64] output: max_d |got - ref| over c * row_scale + 2^-20 * (the item's largest row_scale).
    A row whose bound is 0 (its exact value is 0 and so is every row of its item) must be exact."""
    err = (got.double() - ref).abs().amax(-1)
    bound = c * row_scale + FLOOR * row_scale.amax(-1, keepdim=True)
    return ratio(err, bound)


def lse_ratio(got, ref):
    return ratio((got.double() - ref).abs(), LSE_ABS + LSE_REL * ref.abs())


def ratio(err, bound):
    r = err / bound.clamp_min(torch.finfo(torch.float64).tiny)
    return torch.where(bound > 0, r, torch.where(err > 0, torch.full_like(r, math.inf), torch.zeros_like(r)))


# ---------------------------------------------------------------------------------------------------------------- inputs
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def normal_qkv(n_seq, S, H, seed, amp=0.7):
    """randn * amp, bf16 [n_seq*S, 3*H*64] (CPU)."""
    return (torch.randn(n_seq * S, 3 * H * HD, generator=_gen(seed)) * amp).bfloat16()


def mixed_qkv(n_seq, S, H, seed):
    """Items of three kinds, by item index (sequence * H + head) mod 3:
    0  normal rows (randn * 0.7);
    1  one-hot rows: every second query row scores one key j (which one varies with the item) more than 2^100 above every
       other key, so its softmax is that one key and o = v_j exactly; the other rows see key j only mildly;
    2  uniform rows: every key of the item is the same vector, so P = 1/S."""
    x = normal_qkv(n_seq, S, H, seed).float().view(n_seq, S, 3, H, HD)
    for item in range(n_seq * H):
        seq, h = divmod(item, H)
        kind = item % 3
        if kind == 1:
            x[seq, :, :2, h, 0] = 0.0
            x[seq, 0::2, 0, h, 0] = 64.0
            x[seq, (seq * 7 + h * 13) % S, 1, h, 0] = 32.0     # 64 * 32 * s log2 e > 140 for s >= 0.05
        elif kind == 2:
            x[seq, :, 1, h] = x[seq, 0, 1, h].clone()
    return x.view(n_seq * S, 3 * H * HD).bfloat16()


def d_o_rows(n_seq, S, H, seed, amp=1.0, zero_every=5):
    """randn * amp, bf16 [n_seq*S, H*64], with every zero_every-th (row, head) all zero (D = 0 and dQ_i = 0 there)."""
    g = torch.randn(n_seq * S, H, HD, generator=_gen(seed)) * amp
    if zero_every:
        idx = torch.arange(n_seq * S * H).view(n_seq * S, H)
        g[(idx % zero_every) == 3] = 0.0
    return g.view(n_seq * S, H * HD).bfloat16()


def _place_spikes(x, scale, spikes, row_targets):
    """Make key j's score exceed the maximum over keys [0, split) by exactly `target` log2 units (of the bf16-rounded inputs, up
    to the rounding of one q element) for the rows given.  spikes: list of (channel, key j, split).  row_targets[i]: one target
    per spike, or None (the row keeps its normal scores).  x: fp32 [n_seq, S, 3, H, 64], modified in place."""
    n_seq, S, _, H, _ = x.shape
    B = 8.0
    for ch, j, _ in spikes:
        x[:, :, 1, :, ch] = 0.0
        x[:, :, 0, :, ch] = 0.0
        x[:, j, 1, :, ch] = B
    xb = x.bfloat16().double()
    q, k = xb[:, :, 0], xb[:, :, 1]                                    # [n_seq, S, H, 64]
    base = torch.einsum("sihd,sjhd->shij", q, k) * scale * LOG2E       # log2 units, spike channels are zero
    for i, tg in enumerate(row_targets):
        if tg is None:
            continue
        prev = None
        for (ch, j, split), t in zip(spikes, tg):
            # target relative to the maximum of keys [0, split) (which include the earlier spikes)
            m0 = base[:, :, i, :split].amax(-1)
            if prev is not None:
                m0 = torch.maximum(m0, prev)
            want = m0 + t - base[:, :, i, j]
            x[:, i, 0, :, ch] = (want / (scale * LOG2E * B)).float()
            prev = want + base[:, :, i, j]
    return x


def _blocks(S, classes):
    """Row classes by 32-row block (one warp of the kernels): block b gets classes[b % len(classes)]."""
    return [classes[(i // WARP_ROWS) % len(classes)] for i in range(S)]


def tc208_spike_qkv(n_seq, S, H, seed, scale=0.125):
    """attention_tc<208> (193 <= S <= 208, no LSE): key S - 1 (in the masked tail block) scores above the maximum of the first
    96 keys by 64..124 log2 units in some 32-row blocks (the first-half redo), by 50..58 in others (just below 2^60: P up to
    2^58 against the first-half reference) and normally in the rest."""
    x = normal_qkv(n_seq, S, H, seed).float().view(n_seq, S, 3, H, HD)
    cls = _blocks(S, ["redo", "below", "normal"])
    tg = [None if c == "normal" else ((64.0 + (i % 31) * 2.0,) if c == "redo" else (50.0 + (i % 9),)) for i, c in enumerate(cls)]
    _place_spikes(x, scale, [(0, S - 1, TC208_SPLIT)], tg)
    return x.view(n_seq * S, 3 * H * HD).bfloat16()


def fwd_lse_spike_qkv(n_seq, S, H, seed, scale=0.125):
    """attention_fwd_lse_tc (160 < S <= 320, LSE kept): key 160 + (S - 161) // 2 of the second chunk scores above the first
    chunk's maximum by 68..128 log2 units in some 32-row blocks (the reference move), by 33..62 in others (the fast path with P
    between 2^32 and 2^62) and normally in the rest."""
    x = normal_qkv(n_seq, S, H, seed).float().view(n_seq, S, 3, H, HD)
    j = FWD_LSE_SPLIT + (S - FWD_LSE_SPLIT - 1) // 2
    cls = _blocks(S, ["move", "between", "normal"])
    tg = [None if c == "normal" else ((68.0 + (i % 31) * 2.0,) if c == "move" else (33.0 + (i % 30),)) for i, c in enumerate(cls)]
    _place_spikes(x, scale, [(0, j, FWD_LSE_SPLIT)], tg)
    return x.view(n_seq * S, 3 * H * HD).bfloat16()


def long_spike_qkv(n_seq, S, H, seed, scale=0.125):
    """attention_long_tc forward (S > 240 without LSE, S > 320 with): key 64 + 5 (second chunk) scores above the first chunk's
    maximum by 44..104 log2 units in some 32-row blocks (one reference move); in others key S - 1 (the ragged last chunk) then
    scores another 44..74 above that key (two moves); others stay 30..38 above (no move, P up to 2^38); the rest are normal."""
    assert S > 2 * LONG_CHUNK + 6
    x = normal_qkv(n_seq, S, H, seed).float().view(n_seq, S, 3, H, HD)
    j1, j2 = LONG_CHUNK + 5, S - 1
    cls = _blocks(S, ["once", "twice", "below", "normal"])
    tg = []
    for i, c in enumerate(cls):
        t1 = 44.0 + (i % 31) * 2.0
        tg.append(None if c == "normal" else (t1, -200.0) if c == "once" else (t1, 44.0 + (i % 31)) if c == "twice" else (30.0 + (i % 9), -200.0))
    _place_spikes(x, scale, [(0, j1, LONG_CHUNK), (1, j2, LONG_CHUNK)], tg)
    return x.view(n_seq * S, 3 * H * HD).bfloat16()


# ---------------------------------------------------------------------------------------------------------------- path arithmetic
def scores_log2(qkv, n_seq, S, H, scale):
    """fp64 scores of the bf16 inputs in log2 units, [n_seq*H, S, S]."""
    q, k = heads(qkv, n_seq, S, H, 0), heads(qkv, n_seq, S, H, 1)
    return scale * LOG2E * (q @ k.transpose(1, 2))


def split_excess(qkv, n_seq, S, H, scale, split):
    """Per row: max over keys [split, S) minus max over keys [0, split), in log2 units, [n_seq*H, S]."""
    s = scores_log2(qkv, n_seq, S, H, scale)
    return s[..., split:].amax(-1) - s[..., :split].amax(-1)


def long_moves(qkv, n_seq, S, H, scale):
    """Reference moves of the long forward per row, [n_seq*H, S] (ints), and per row the largest step a chunk maximum took
    above the reference without moving it.  The kernel moves a warp's references when any row of the warp exceeds the threshold;
    rows here are evaluated on their own, which matches it for the builders' warp-uniform row classes."""
    s = scores_log2(qkv, n_seq, S, H, scale)
    ref = s[..., :LONG_CHUNK].amax(-1)
    moves = torch.zeros_like(ref, dtype=torch.long)
    stay = torch.full_like(ref, -math.inf)
    for c0 in range(LONG_CHUNK, S, LONG_CHUNK):
        mx = s[..., c0:c0 + LONG_CHUNK].amax(-1)
        mv = (mx - ref) > LONG_THRESHOLD
        stay = torch.where(mv, stay, torch.maximum(stay, mx - ref))
        moves += mv.long()
        ref = torch.where(mv, torch.maximum(ref, mx), ref)
    return moves, stay
