"""The attention reference (tests/attention_ref.py) without a GPU: its explicit fp64 backward against torch.autograd, and the input
builders against the slow-path thresholds of the kernels, checked on the bf16-rounded inputs at the scales the GPU tests use."""
import pytest
import torch

from tests import attention_ref as R


@pytest.mark.parametrize("n_seq,S,H,scale", [(2, 1, 3, 0.125), (1, 2, 2, 0.125), (2, 17, 2, 1.0), (1, 70, 3, 0.05), (1, 161, 1, 0.125)])
def test_explicit_backward_matches_autograd(n_seq, S, H, scale):
    qkv = R.mixed_qkv(n_seq, S, H, seed=S + H)
    d_o = R.d_o_rows(n_seq, S, H, seed=S * 3 + H)
    ref = R.backward(qkv, d_o, n_seq, S, H, scale)
    fw = R.forward(qkv, n_seq, S, H, scale)
    q, k, v = (R.heads(qkv, n_seq, S, H, i).requires_grad_() for i in range(3))
    s = scale * (q @ k.transpose(1, 2))
    o = torch.softmax(s, -1) @ v
    o.backward(R.heads(d_o, n_seq, S, H))
    assert torch.allclose(fw["o"], o.detach(), rtol=1e-12, atol=1e-12)
    assert torch.allclose(fw["lse"], torch.logsumexp(s, -1).detach(), rtol=1e-12, atol=1e-12)
    for name, t in (("dq", q), ("dk", k), ("dv", v)):
        assert torch.allclose(ref[name], t.grad, rtol=1e-9, atol=1e-12), name
    if S == 1:     # a single key: P = 1, dP = D, so dQ = dK = 0 exactly
        assert ref["dq"].abs().max() < 1e-12 and ref["dk"].abs().max() < 1e-12
    # the bound scales cover the values they bound
    assert (ref["dv"].abs().amax(-1) <= ref["dv_scale"] * (1 + 1e-12)).all()
    assert (ref["dq"].abs().amax(-1) <= ref["dq_scale"] * (1 + 1e-12)).all()
    assert (ref["dk"].abs().amax(-1) <= ref["dk_scale"] * (1 + 1e-12)).all()
    assert (fw["o"].abs().amax(-1) <= fw["o_scale"] * (1 + 1e-12)).all()


def test_one_hot_and_uniform_items():
    n_seq, S, H, scale = 2, 200, 3, 0.05
    qkv = R.mixed_qkv(n_seq, S, H, seed=5)
    s = R.scores_log2(qkv, n_seq, S, H, scale)
    top2 = s.topk(2, -1).values
    for item in range(n_seq * H):
        if item % 3 == 1:       # every second row: one key more than 2^100 above all others
            assert (top2[item, 0::2, 0] - top2[item, 0::2, 1] > 100).all()
        if item % 3 == 2:       # identical keys
            assert (s[item] == s[item, :, :1]).all()
    fw = R.forward(qkv, n_seq, S, H, scale)
    v = R.heads(qkv, n_seq, S, H, 2)
    j = [(seq * 7 + h * 13) % S for seq in range(n_seq) for h in range(H)]
    for item in range(1, n_seq * H, 3):
        assert torch.equal(fw["o"][item, 0::2], v[item, j[item]].expand(S // 2, -1))
    for item in range(2, n_seq * H, 3):
        assert torch.allclose(fw["o"][item], v[item].mean(0).expand(S, -1), rtol=0, atol=1e-12)


def _blocks(x, S):
    """[I, S] -> per 32-row block (one warp of the kernels) the rows' min and max."""
    out = []
    for b in range(0, S, R.WARP_ROWS):
        blk = x[:, b:b + R.WARP_ROWS]
        out.append((blk.amin(), blk.amax()))
    return out


# the spike cases of test_attention_kernels_gpu.py (n_seq, S, H); all at scale 0.125
@pytest.mark.parametrize("n_seq,S,H", [(2, 193, 3), (2, 197, 3), (2, 208, 3), (16, 197, 4)])
def test_tc208_spike_rows_on_and_below_the_redo_threshold(n_seq, S, H):
    qkv = R.tc208_spike_qkv(n_seq, S, H, seed=S + H)
    ex = R.split_excess(qkv, n_seq, S, H, 0.125, R.TC208_SPLIT)
    blocks = _blocks(ex, S)
    thr = R.TC208_THRESHOLD
    assert any(lo > thr + 2 for lo, _ in blocks), "no warp on the redo path"
    assert any(thr - 12 < lo and hi < thr - 1 for lo, hi in blocks), "no warp just below the threshold"
    assert any(hi < 20 for _, hi in blocks), "no warp of normal rows"


@pytest.mark.parametrize("n_seq,S,H", [(2, 161, 3), (2, 255, 3), (3, 320, 4), (2, 300, 3), (2, 320, 2), (16, 289, 4)])
def test_fwd_lse_spike_rows_on_and_below_the_move_threshold(n_seq, S, H):
    qkv = R.fwd_lse_spike_qkv(n_seq, S, H, seed=S + H)
    ex = R.split_excess(qkv, n_seq, S, H, 0.125, R.FWD_LSE_SPLIT)
    blocks = _blocks(ex, S)
    thr = R.FWD_LSE_THRESHOLD
    assert any(lo > thr + 2 for lo, _ in blocks), "no warp on the reference move"
    assert any(32 < lo and hi < thr - 1 for lo, hi in blocks), "no warp with P between 2^32 and 2^64"
    assert any(hi < 20 for _, hi in blocks), "no warp of normal rows"


@pytest.mark.parametrize("n_seq,S,H", [(2, 257, 3), (2, 333, 3), (2, 512, 2), (2, 1569, 2), (8, 577, 6)])
def test_long_spike_rows_move_once_twice_or_stay_below(n_seq, S, H):
    qkv = R.long_spike_qkv(n_seq, S, H, seed=S + H)
    moves, stay = R.long_moves(qkv, n_seq, S, H, 0.125)
    mv, st = _blocks(moves.double(), S), _blocks(stay, S)
    thr = R.LONG_THRESHOLD
    assert any(lo == hi == 1 for lo, hi in mv), "no warp whose reference moves once"
    assert any(lo == hi == 2 for lo, hi in mv), "no warp whose reference moves twice"
    assert any(m == (0, 0) and thr - 12 < s[0] and s[1] < thr - 1 for m, s in zip(mv, st)), "no warp just below the threshold"
    # no row of any block sits within 1 log2 unit of the threshold, where fp32 scores could decide either way
    s2 = stay[moves == 0]
    assert ((s2 < thr - 1) | (s2 > thr + 1)).all()
