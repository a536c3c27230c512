"""Every attention kernel against the fp64 reference of tests/attention_ref.py, per (sequence, head, row), through ub_attn_fwd /
ub_attn_bwd / ub_cls_attn:
  - at each edge of the dispatch (S = 1 and 2, the 16-key padding, the 128-row tiles, the one / two-chunk boundary of the LSE
    forward at S = 160 / 161, the 240 / 320 kernel bounds, ragged 32- and 64-row chunks of the long kernel), H = 1 .. 16 and
    softmax scales 0.05 .. 1.0;
  - at the shipped shapes, where every CTA of the persistent kernels walks many items;
  - on inputs that put rows on each kernel's slow path (and just below it), one-hot rows, uniform rows and zero dO rows;
  - on grids of 2, 10 and all SMs, which must give bit-identical results;
Outputs are slices of larger NaN-filled buffers: every element must be written and finite, the guard rows around them untouched."""
import math

import pytest
import torch

from tests import attention_ref as R

pytestmark = pytest.mark.gpu

G = 128                                   # guard rows before and after every output
DEV = "cuda"
BF16_SENTINEL = 0x7FA5                    # a NaN no kernel produces
F32_SENTINEL = 0x7FA5A5A5
WORST = {}                                # (path, output) -> worst error / bound seen, printed at the end of the module


def _guarded(rows, cols, dtype):
    it, bits = (torch.int16, BF16_SENTINEL) if dtype == torch.bfloat16 else (torch.int32, F32_SENTINEL)
    buf = torch.full((rows + 2 * G, cols), bits, dtype=it, device=DEV).view(dtype)
    return buf, buf[G:G + rows]


def _guards_intact(buf, rows):
    it, bits = (torch.int16, BF16_SENTINEL) if buf.dtype == torch.bfloat16 else (torch.int32, F32_SENTINEL)
    b = buf.view(it)
    return bool((b[:G] == bits).all()) and bool((b[G + rows:] == bits).all())


def _bits(t):
    return t.view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32)


def _path(S, lse):
    if not lse:
        return "tc" if S <= 240 and (S + 15) // 16 * 16 != 208 else "tc208" if S <= 240 else "long_fwd"
    return "fwd_lse+bwd_tc" if S <= 320 else "long_fwd+long_bwd"


def _note(path, name, r):
    w = float(r.max()) if r.numel() else 0.0
    WORST[(path, name)] = max(WORST.get((path, name), 0.0), w)
    return w


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    print("\nworst error / bound per path and output:")
    for (path, name), w in sorted(WORST.items()):
        print(f"  {path:20s} {name:6s} {w:.3f}")


def _dbias_preset(H, seed):
    n = 3 * H * 64
    g = torch.Generator().manual_seed(seed)
    sign = torch.where(torch.arange(n) % 2 == 0, 1.0, -1.0)
    return ((torch.rand(n, generator=g) + 0.5) * sign).to(DEV)


def run(n_seq, S, H, scale, qkv, lse=True, bwd=True, d_o=None, check=True, tag=""):
    """Forward (and backward) of the library on guarded, sentinel-filled outputs; with check, every output is compared per row
    with the fp64 reference.  Returns the outputs."""
    from unite_b200 import ops
    qkv = qkv.to(DEV)
    rows, path = n_seq * S, _path(S, lse)
    ob, o = _guarded(rows, H * 64, torch.bfloat16)
    lb, l = _guarded(n_seq * H, S, torch.float32) if lse else (None, None)
    ops.attn_fwd(qkv, o, l, n_seq, S, H, scale)
    out = dict(o=o, lse=l)
    if bwd:
        d_o = (d_o if d_o is not None else R.d_o_rows(n_seq, S, H, seed=S * 3 + H)).to(DEV)
        db, dws = _guarded(n_seq * H, S, torch.float32)
        qb, dqkv = _guarded(rows, 3 * H * 64, torch.bfloat16)
        dbias0 = _dbias_preset(H, S + H)
        dbias = dbias0.clone()
        ops.attn_bwd(qkv, o, d_o, l, dws, dqkv, n_seq, S, H, scale, dbias=dbias)
        # the same backward without o: D is taken from D_ws as the first call left it
        qb2, dqkv2 = _guarded(rows, 3 * H * 64, torch.bfloat16)
        ops.attn_bwd(qkv, None, d_o, l, dws, dqkv2, n_seq, S, H, scale)
        out.update(dqkv=dqkv, D=dws, dbias=dbias)
    torch.cuda.synchronize()
    if not check:
        return out
    ratios = {}
    assert _guards_intact(ob, rows), "o: guard rows overwritten"
    assert bool(torch.isfinite(o.float()).all()), "o: an element is unwritten or not finite"
    fw = R.forward(qkv, n_seq, S, H, scale)
    ratios["o"] = R.row_ratio(R.heads(o, n_seq, S, H), fw["o"], fw["o_scale"], R.O_C)
    if lse:
        assert _guards_intact(lb, n_seq * H), "lse: guard rows overwritten"
        assert bool(torch.isfinite(l).all()), "lse: an element is unwritten or not finite"
        ratios["lse"] = R.lse_ratio(l.view(n_seq * H, S), fw["lse"])
    if bwd:
        assert torch.equal(_bits(dqkv2), _bits(dqkv)), "dqkv differs between o given and o = None with the same D_ws"
        assert _guards_intact(qb, rows) and _guards_intact(qb2, rows), "dqkv: guard rows overwritten"
        assert _guards_intact(db, n_seq * H), "D_ws: guard rows overwritten"
        assert bool(torch.isfinite(dqkv.float()).all()), "dqkv: an element is unwritten or not finite"
        assert bool(torch.isfinite(dws).all()), "D_ws: an element is unwritten or not finite"
        bw = R.backward(qkv, d_o, n_seq, S, H, scale, o=o)
        # D: fp32 sum of 64 exact bf16 products, against the fp64 sum of the same products
        od = R.heads(o, n_seq, S, H) * R.heads(d_o, n_seq, S, H)
        ratios["D"] = R.ratio((dws.view(n_seq * H, S).double() - bw["D"]).abs(), 2.0 ** -17 * od.abs().sum(-1))
        for name, part, c in (("dq", 0, R.DQK_C), ("dk", 1, R.DQK_C), ("dv", 2, R.DV_C)):
            ratios[name] = R.row_ratio(R.heads(dqkv, n_seq, S, H, part), bw[name], bw[name + "_scale"], c)
        # dbias: the key third untouched, the q / v thirds += the column sums of the dqkv the kernel wrote.  Each column receives
        # n_seq * ceil(S / 32) fp32 red.adds of partial sums over <= 32 rows; the bound is that many roundings (times 2).
        HD = H * 64
        assert torch.equal(_bits(dbias[HD:2 * HD]), _bits(dbias0[HD:2 * HD])), "dbias: key third written"
        col = dqkv.double().sum(0) + dbias0.double()
        mag = dqkv.double().abs().sum(0) + dbias0.double().abs()
        n_add = 33 + n_seq * math.ceil(S / 32)
        for lo in (0, 2 * HD):
            sl = slice(lo, lo + HD)
            r = R.ratio((dbias[sl].double() - col[sl]).abs(), n_add * 2.0 ** -23 * mag[sl])
            ratios["dbias"] = torch.maximum(ratios["dbias"], r) if "dbias" in ratios else r
    worst = {k: _note(path, k, v) for k, v in ratios.items()}
    print(f"[{path}] n_seq={n_seq} S={S} H={H} scale={scale} {tag} " + " ".join(f"{k}={v:.3f}" for k, v in worst.items()))
    for k, v in ratios.items():
        bad = (v > 1).nonzero()
        assert bad.numel() == 0, f"{k}: {bad.shape[0]} rows over their bound, worst {worst[k]:.3g} (first at {bad[0].tolist()})"
    return out


# ---------------------------------------------------------------------------------------------------------------- dispatch table
FWD_ONLY = [1, 2, 16, 17, 128, 129, 192, 209, 240,        # attention_tc, generic
            193, 197, 208,                                # attention_tc<208>
            241, 257, 320, 577]                           # long forward without LSE
FWD_BWD = [1, 2, 64, 127, 128, 129, 160, 161, 255, 256, 257, 319, 320,    # fwd_lse + bwd_tc
           321, 333, 384, 577, 1568, 1569]                                # long forward + DKV + DQ


@pytest.mark.parametrize("S", FWD_ONLY)
def test_forward_without_lse(S):
    run(2, S, 3, 0.125, R.mixed_qkv(2, S, 3, seed=S), lse=False, bwd=False)


@pytest.mark.parametrize("S", FWD_BWD)
def test_forward_with_lse_and_backward(S):
    run(2, S, 3, 0.125, R.mixed_qkv(2, S, 3, seed=S))


# other head counts, other scales, and the shapes the retired long-kernel check ran (n_seq, S, H)
@pytest.mark.parametrize("n_seq,S,H,scale,lse", [
    (3, 1, 1, 0.125, False), (2, 197, 1, 0.125, False), (2, 257, 1, 0.125, False), (3, 1569, 1, 0.125, True),
    (2, 129, 12, 0.125, False), (2, 320, 12, 0.125, True), (1, 577, 12, 0.125, True),
    (2, 2, 16, 0.125, True), (2, 208, 16, 0.125, False), (2, 321, 16, 0.125, True), (1, 1568, 16, 0.125, True),
    (2, 129, 3, 0.05, False), (2, 17, 3, 1.0, False),
    (2, 197, 3, 0.05, False), (2, 208, 3, 1.0, False),
    (2, 257, 3, 0.05, False), (2, 400, 3, 1.0, False),
    (2, 255, 3, 1.0, True), (2, 161, 3, 0.05, True),
    (2, 333, 3, 1.0, True), (2, 1000, 4, 0.05, True),
    (2, 384, 2, 0.125, True), (1, 333, 3, 0.125, True), (2, 1000, 4, 0.125, True), (3, 1568, 12, 0.125, True),
    (2, 400, 2, 0.125, False),
])
def test_heads_and_scales(n_seq, S, H, scale, lse):
    run(n_seq, S, H, scale, R.mixed_qkv(n_seq, S, H, seed=S + H), lse=lse, bwd=lse)


# ---------------------------------------------------------------------------------------------------------------- slow paths
@pytest.mark.parametrize("n_seq,S,H", [(2, 193, 3), (2, 197, 3), (2, 208, 3)])
def test_tc208_first_half_redo(n_seq, S, H):
    run(n_seq, S, H, 0.125, R.tc208_spike_qkv(n_seq, S, H, seed=S + H), lse=False, bwd=False)


@pytest.mark.parametrize("n_seq,S,H", [(2, 161, 3), (2, 255, 3), (3, 320, 4), (2, 300, 3), (2, 320, 2)])
def test_fwd_lse_reference_move(n_seq, S, H):
    run(n_seq, S, H, 0.125, R.fwd_lse_spike_qkv(n_seq, S, H, seed=S + H))


@pytest.mark.parametrize("n_seq,S,H,lse", [(2, 257, 3, False), (2, 512, 2, False), (2, 333, 3, True), (2, 512, 2, True),
                                           (2, 1569, 2, True)])
def test_long_forward_reference_moves(n_seq, S, H, lse):
    run(n_seq, S, H, 0.125, R.long_spike_qkv(n_seq, S, H, seed=S + H), lse=lse, bwd=lse)


# ---------------------------------------------------------------------------------------------------------------- shipped shapes
@pytest.mark.parametrize("name,n_seq,S,H,lse", [
    ("B/16 teacher", 256, 197, 12, False),
    ("L/14 teacher 224 px", 64, 257, 16, False),
    ("L/14 teacher 336 px", 16, 577, 16, False),
    ("stage-1 student B/16", 32, 320, 12, True),
    ("stage-1 student ViT-L", 16, 320, 16, True),
    ("stage 2", 8, 1568, 12, True),
])
def test_shipped_shapes(name, n_seq, S, H, lse):
    from unite_b200 import _cabi
    units = n_seq * H * (1 if (S <= 240 or (lse and S <= 320)) else ((S + 127) // 128 + 1) // 2)
    grid = min(units, _cabi.lib.ub_sm_count())
    print(f"\n{name}: {units} work items on {grid} CTAs, {units // grid}..{-(-units // grid)} per CTA")
    run(n_seq, S, H, 0.125, R.normal_qkv(n_seq, S, H, seed=S * 5 + H), lse=lse, bwd=lse, tag=name)


# ---------------------------------------------------------------------------------------------------------------- grid independence
@pytest.fixture
def sm_limit():
    """Sets the library's persistent-grid size (ub_set_sm_limit rounds down to even; 0 = the whole device) and restores it."""
    from unite_b200 import _cabi
    lib = _cabi.lib
    full = lib.ub_set_sm_limit(0)

    def set_limit(n):
        got = lib.ub_set_sm_limit(n)
        assert got == (n if n else full), f"ub_set_sm_limit({n}) gave {got}"
    try:
        yield set_limit
    finally:
        lib.ub_set_sm_limit(0)


@pytest.mark.parametrize("kind,n_seq,S,H,lse", [
    ("tc", 16, 150, 3, False),                  # 48 items
    ("tc208", 16, 197, 4, False),               # 64 items, first-half redo rows
    ("fwd_lse", 16, 289, 4, True),              # 64 items of 3 query tiles (odd: warpgroups alternate across items), moves
    ("long", 8, 577, 6, True),                  # 48 items, 144 units, moves once and twice
])
def test_results_do_not_depend_on_the_grid(sm_limit, kind, n_seq, S, H, lse):
    build = dict(tc=R.mixed_qkv, tc208=R.tc208_spike_qkv, fwd_lse=R.fwd_lse_spike_qkv, long=R.long_spike_qkv)[kind]
    qkv = build(n_seq, S, H, seed=S + H)
    runs = []
    for limit in (2, 10, 0):
        sm_limit(limit)
        for rep in range(2):
            runs.append((limit, rep, run(n_seq, S, H, 0.125, qkv, lse=lse, bwd=lse, check=(limit == 2 and rep == 0),
                                         tag=f"sm_limit={limit}")))
    _, _, first = runs[0]
    for limit, rep, r in runs[1:]:
        for name in ("o", "lse", "dqkv", "D"):
            if r.get(name) is not None:
                assert torch.equal(_bits(r[name]), _bits(first[name])), f"{name} differs at sm_limit={limit} (launch {rep})"
        if lse:
            # dbias is accumulated with fp32 red.adds whose order follows the grid: equal within that summation order
            mag = first["dqkv"].double().abs().sum(0) + 2.0
            n_add = 33 + n_seq * math.ceil(S / 32)
            assert bool(((r["dbias"].double() - first["dbias"].double()).abs() <= 2 * n_add * 2.0 ** -23 * mag).all())


# ---------------------------------------------------------------------------------------------------------------- cls_attn
@pytest.mark.parametrize("S", [2, 197, 257, 577])
@pytest.mark.parametrize("H", [12, 16])
def test_cls_attn(S, H):
    from unite_b200 import ops
    n_seq, scale = 4, 0.125
    qkv = R.normal_qkv(n_seq, S, H, seed=S + H).to(DEV)
    buf, out = _guarded(n_seq, S - 1, torch.float32)
    ops.cls_attn(qkv, out, n_seq, S, H, scale)
    torch.cuda.synchronize()
    assert _guards_intact(buf, n_seq)
    q, k = R.heads(qkv, n_seq, S, H, 0), R.heads(qkv, n_seq, S, H, 1)
    p = torch.softmax(scale * (q[:, :1] @ k.transpose(1, 2)), -1)[:, 0, 1:]          # [n_seq*H, S-1]
    ref = p.view(n_seq, H, S - 1).mean(1)
    rel = ((out.double() - ref).abs() / ref).max().item()
    print(f"cls_attn S={S} H={H}: worst relative error {rel:.2e}")
    assert rel <= 1e-4


def test_cls_attn_refuses_a_row_set_over_48_kb():
    from unite_b200 import _cabi, ops
    n_seq, S, H = 2, 800, 16                    # 16 heads x 800 fp32 probabilities = 51,200 B of shared memory
    qkv = R.normal_qkv(n_seq, S, H, seed=1).to(DEV)
    buf, out = _guarded(n_seq, S - 1, torch.float32)
    with pytest.raises(_cabi.UBError, match="too long"):
        ops.cls_attn(qkv, out, n_seq, S, H, 0.125)
    torch.cuda.synchronize()
    assert bool((_bits(buf) == F32_SENTINEL).all()), "the refused call wrote its output"
