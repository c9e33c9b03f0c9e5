"""Aggregate-first input gradient of the hidden layers: the two-segment tensor-core projection at the hidden layer's
square shape, and the trainer step in both input-gradient orders."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
from conftest import TOL, rel_err
from gnn_tableextraction_b200 import layers as L, ops, synth
from gnn_tableextraction_b200.graph import batch_pages_host
from oracle import sage_oracle as so

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _padded(t):
    out = ops.empty_padded(t.shape[0], t.shape[1], DEV)
    out.copy_(t)
    return out


def _models(seed, cfg=(13, 218, 9, 3), dropout=0):
    torch.manual_seed(seed)
    om = so.OracleGcnSAGE(*cfg, F.relu, dropout)
    cm = gte.GcnSAGE(*cfg, F.relu, dropout)
    cm.load_state_dict(om.state_dict())
    return cm.to(DEV)


def _spy(monkeypatch, names):
    calls = {n: 0 for n in names}
    for n in names:
        f = getattr(ops, n)

        def wrap(*a, _f=f, _n=n, **kw):
            calls[_n] += 1
            return _f(*a, **kw)

        monkeypatch.setattr(ops, n, wrap)
    return calls


def test_umma_bwd_data2_hidden_shape(umma_kernel):
    """dh = dz Ws + G Wn at fo = fin = 218 (K = 2 x 7 k-blocks: the split-accumulator path) against fp64"""
    n, fin, fo = 3001, 218, 218
    gen = torch.Generator().manual_seed(9)
    W = (torch.rand(fo, 2 * fin, generator=gen) - 0.5) * (2 / (2 * fin) ** 0.5)
    pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
    dz, g = torch.randn(n, fo, generator=gen), torch.randn(n, fo, generator=gen) * 3.0
    dx = ops.umma_linear_bwd_data2(_padded(dz), _padded(g), pack, fin)
    assert dx.shape == (n, fin)
    assert rel_err(dx, dz.double() @ W.double()[:, :fin] + g.double() @ W.double()[:, fin:]) < 3e-6


def test_config2_step_agg_first_matches_layer_order_and_replays(monkeypatch):
    """one config-2 train step (512 pages, N = 153 600) with the aggregate-first input gradient against the per-layer
    order: statistics within 1e-6, every gradient within 1e-5; the captured step replays the eager step bit for bit"""
    hb = batch_pages_host(synth.make_pages(512, distinct=48))
    res = {}
    for order in ("layer", "agg"):
        monkeypatch.setattr(L, "DH_ORDER", order)
        cm = _models(31)
        tr = gte.SageTrainer(cm)
        st = tr.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        res[order] = (st, {k: p.grad.clone() for k, p in cm.named_parameters()}, tr.flat_param.clone())
    assert rel_err(res["agg"][0], res["layer"][0]) < 1e-6
    for k, gl in res["layer"][1].items():
        assert rel_err(res["agg"][1][k], gl) < TOL, k
    tc = gte.SageTrainer(_models(31))
    tc.capture(hb)
    tc.load_batch(hb)
    assert torch.equal(tc.replay(), res["agg"][0])
    assert torch.equal(tc.flat_param, res["agg"][2])


def test_trainer_step_launch_count_and_order(monkeypatch):
    """the default model's eager step stays at 28 launches; its hidden layer takes the two-segment projection"""
    calls = _spy(monkeypatch, ["umma_linear_bwd_data", "umma_linear_bwd_data2"])
    hb = batch_pages_host(synth.make_pages(4, n=300, k=10))
    tr = gte.SageTrainer(_models(101))
    lib = gte.lib()
    c0 = lib.gte_launch_count()
    tr.train_step(gte.PageGraphBatch.from_host(hb, DEV))
    assert lib.gte_launch_count() - c0 == 28
    assert calls == {"umma_linear_bwd_data": 0, "umma_linear_bwd_data2": 1}
    monkeypatch.setattr(L, "DH_ORDER", "layer")
    c0 = lib.gte_launch_count()
    tr.train_step(gte.PageGraphBatch.from_host(hb, DEV))
    assert lib.gte_launch_count() - c0 == 28
    assert calls == {"umma_linear_bwd_data": 1, "umma_linear_bwd_data2": 1}


def test_dropout_layer_keeps_layer_order(monkeypatch):
    """with dropout the mask sits between the projection and A_hat^T: the hidden layer keeps dz W first"""
    calls = _spy(monkeypatch, ["umma_linear_bwd_data", "umma_linear_bwd_data2"])
    hb = batch_pages_host(synth.make_pages(4, n=300, k=10))
    cm = _models(102, dropout=0.3)
    tr = gte.SageTrainer(cm)
    assert cm.training and tr._drop_p[2] > 0  # the hidden layer's dropout is active
    st = tr.train_step(gte.PageGraphBatch.from_host(hb, DEV)).cpu()
    assert calls["umma_linear_bwd_data2"] == 0 and calls["umma_linear_bwd_data"] >= 1
    assert np.isfinite(st.numpy()).all()
