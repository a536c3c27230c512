"""Stage-2 model EMA without a GPU: what the fused loop refuses, ModelEma against timm 0.4.12's (tests/ema_ref.py) at
construction and resume, deepcopy of a stage-2 model, and the checkpoint keys with and without an EMA."""
import copy
import os
from functools import partial

import pytest
import torch
import torch.nn as nn

from tests import ema_ref as R


def _vit(depth=2, num_classes=5, seed=0):
    from unite_b200.modeling_finetune import VisionTransformer
    torch.manual_seed(seed)
    return VisionTransformer(img_size=32, embed_dim=64, depth=depth, num_heads=2, qkv_bias=True, num_classes=num_classes, all_frames=4,
                             tubelet_size=2, init_scale=0.1, norm_layer=partial(nn.LayerNorm, eps=1e-6), drop_path_rate=0.1)


class _Wrapped(nn.Module):
    def __init__(self, m):
        super().__init__()
        self.module = m


def test_refusals():
    from unite_b200.ema import ModelEma, resolve_model_ema
    from unite_b200.engine_for_finetuning import train_one_epoch
    model = _vit()
    # anything that is not a ModelEma: refused first, before the (CPU) model or any other argument is looked at
    with pytest.raises(NotImplementedError, match="EMA"):
        train_one_epoch(torch.nn.Linear(2, 2), None, [], None, "cpu", 0, model_ema=object())
    with pytest.raises(NotImplementedError, match="EMA"):
        train_one_epoch(model, torch.nn.MSELoss(), [], object(), "cpu", 0, model_ema=object(), train_head_only=True)
    with pytest.raises(NotImplementedError, match="EMA"):
        resolve_model_ema(object(), model)
    # --model_ema_force_cpu
    for cls in (ModelEma, R.ModelEma):
        with pytest.raises(NotImplementedError, match="host"):
            resolve_model_ema(cls(model, decay=0.999, device="cpu"), model)
        with pytest.raises(NotImplementedError, match="host"):
            train_one_epoch(model, None, [], None, "cpu", 0, model_ema=cls(model, device="cpu"))
    with pytest.raises(NotImplementedError, match="head-only"):
        train_one_epoch(model, None, [], None, "cpu", 0, train_head_only=True)
    # an EMA of another architecture
    for other in (_vit(depth=3), _vit(num_classes=7), torch.nn.Linear(2, 2)):
        for cls in (ModelEma, R.ModelEma):
            with pytest.raises(ValueError, match="architecture"):
                resolve_model_ema(cls(other), model)
    assert resolve_model_ema(None, model) is None


def test_reference_and_package_model_ema_are_both_accepted():
    from unite_b200.ema import ModelEma, resolve_model_ema
    model = _vit()
    for cls in (ModelEma, R.ModelEma):
        ema = cls(model, decay=0.99996)
        r = resolve_model_ema(ema, model)
        assert r.source is ema and r.ema_net is ema.ema and r.decay == 0.99996
        ema.decay = 0.5                                                  # read from the object at every step
        assert r.decay == 0.5
        wrapped = cls(_Wrapped(model))
        assert wrapped.ema_has_module and resolve_model_ema(wrapped, _Wrapped(model)).ema_net is wrapped.ema.module


def test_model_ema_construction_matches_timm():
    from unite_b200.ema import ModelEma
    model = _vit().train()
    for p in model.blocks[0].parameters():
        p.requires_grad_(False)                                          # a frozen part stays frozen in the source
    mine, ref = ModelEma(model, decay=0.9998), R.ModelEma(model, decay=0.9998)
    for ema in (mine, ref):
        assert ema.decay == 0.9998 and ema.device == "" and ema.ema_has_module is False
        assert not ema.ema.training and model.training
        assert all(not p.requires_grad for p in ema.ema.parameters())
        assert ema.ema._core is None
        for (n, p), (n2, q) in zip(model.named_parameters(), ema.ema.named_parameters()):
            assert n == n2 and torch.equal(p, q) and p.data_ptr() != q.data_ptr()
    assert [p.requires_grad for p in model.parameters()].count(True) == sum(1 for n, _ in model.named_parameters()
                                                                              if not n.startswith("blocks.0."))
    assert list(mine.ema.state_dict()) == list(ref.ema.state_dict()) == list(model.state_dict())
    assert ModelEma(model).decay == 0.9999


def test_model_ema_resume_reads_state_dict_ema(tmp_path):
    from unite_b200.ema import ModelEma
    model, other = _vit(seed=0), _vit(seed=1)
    path = os.path.join(tmp_path, "ema.pth")
    torch.save({"state_dict_ema": other.state_dict()}, path)
    for cls in (ModelEma, R.ModelEma):
        ema = cls(model, resume=path)
        assert all(torch.equal(a, b) for a, b in zip(ema.ema.state_dict().values(), other.state_dict().values()))
        assert all(not p.requires_grad for p in ema.ema.parameters())
    torch.save({"model": other.state_dict()}, path)
    ema = ModelEma(model, resume=path)                                   # no state_dict_ema: the model's weights stay
    assert all(torch.equal(a, b) for a, b in zip(ema.ema.state_dict().values(), model.state_dict().values()))


def test_deepcopy_before_the_core_exists():
    model = _vit()
    model.eval()
    c = copy.deepcopy(model)
    assert type(c) is type(model) and c._core is None and not c.training
    assert c.drop_path_rates == model.drop_path_rates and c.num_heads == model.num_heads and c.mlp_hidden == model.mlp_hidden
    assert torch.equal(c.pos_embed, model.pos_embed) and c.pos_embed is not model.pos_embed
    assert list(c.state_dict()) == list(model.state_dict())
    for p, q in zip(model.parameters(), c.parameters()):
        assert torch.equal(p, q) and p is not q and p.data_ptr() != q.data_ptr()
    with torch.no_grad():
        next(c.parameters()).add_(1.0)
    assert not torch.equal(next(c.parameters()), next(model.parameters()))
    c.to(torch.float64)                                                  # no core: the copy can still be moved
    assert next(c.parameters()).dtype == torch.float64


def test_deepcopy_drops_the_core_and_the_cached_engine():
    """A model whose parameters already are views into one flat buffer (what the arena makes of them): the copy gets standalone
    parameters, no core and none of the engine / optimizer objects cached on the model."""
    model = _vit()
    flat = torch.zeros(sum(p.numel() for p in model.parameters()))
    off = 0
    for p in model.parameters():
        v = flat[off:off + p.numel()].view(p.shape)
        v.copy_(p.detach())
        p.data = v
        p.grad = torch.zeros_like(v)
        off += p.numel()
    model._core = object()
    model.__dict__["_ub_stage2_engine"] = object()
    model.__dict__["_ub_default_optimizer"] = object()
    c = copy.deepcopy(model)
    assert c._core is None and not any(k.startswith("_ub_") for k in c.__dict__)
    for p, q in zip(model.parameters(), c.parameters()):
        assert torch.equal(p, q) and q.grad is None
        assert q.untyped_storage().data_ptr() != flat.untyped_storage().data_ptr() and q.untyped_storage().nbytes() == q.numel() * 4
    assert model._core is not None and "_ub_stage2_engine" in model.__dict__


def test_save_model_keys_with_and_without_ema(tmp_path):
    from unite_b200.checkpoint import auto_load_model, save_model
    from unite_b200.ema import ModelEma
    model = _vit(seed=0)
    opt = torch.optim.SGD(model.parameters(), lr=0.1)
    path = save_model(str(tmp_path), 3, model, opt)
    assert set(torch.load(path, weights_only=False)) == {"model", "optimizer", "epoch", "args", "scaler"}
    ema = ModelEma(model, decay=0.9)
    with torch.no_grad():
        for p in ema.ema.parameters():
            p.mul_(0.5)
    path = save_model(str(tmp_path), 4, model, opt, model_ema=ema)
    ck = torch.load(path, weights_only=False)
    assert set(ck) == {"model", "optimizer", "epoch", "args", "scaler", "model_ema"}
    assert list(ck["model_ema"]) == list(ema.ema.state_dict())
    for cls in (ModelEma, R.ModelEma):                                   # timm's object: its .ema is saved the same way
        fresh, fresh_ema = _vit(seed=5), cls(_vit(seed=6))
        assert auto_load_model(str(tmp_path), fresh, torch.optim.SGD(fresh.parameters(), lr=0.1), model_ema=fresh_ema) == 5
        assert all(torch.equal(a, b) for a, b in zip(fresh_ema.ema.state_dict().values(), ema.ema.state_dict().values()))
        assert all(torch.equal(a, b) for a, b in zip(fresh.state_dict().values(), model.state_dict().values()))
    os.remove(path)                                                      # checkpoint-3.pth has no model_ema: the EMA is left alone
    keep = ModelEma(_vit(seed=7))
    before = [t.clone() for t in keep.ema.state_dict().values()]
    assert auto_load_model(str(tmp_path), _vit(seed=8), model_ema=keep) == 0
    assert all(torch.equal(a, b) for a, b in zip(keep.ema.state_dict().values(), before))
