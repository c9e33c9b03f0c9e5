"""Every kernel route of the layer forward and backward against a float64 reference, at the shapes where
``layers.sage_layer_forward`` / ``sage_layer_backward`` change their dispatch (UMMA_MIN_ROWS, SKINNY_MIN_ROWS, COMB_W,
fout <= 16 / 32, fin % 32 / % 128, widths above 256, unaligned rows, bias / LayerNorm / ReLU presence, GCN vs MEAN).

Each row of the route table names the ``ops`` functions its forward and its backward must call, derived by hand from
the rules in layers.py.  The CPU test at the end checks that every ``ops`` call of those two functions is named by at
least one row, so a branch added later without a row fails ``pytest -m "not gpu"``."""
import ast
import dataclasses
import functools
import os
import warnings
from typing import FrozenSet, NamedTuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT, TOL, rel_err

DEV = "cuda"
GCN, MEAN = "gcn", "mean"

# ``ops`` functions layers.py asks a question of; they launch nothing, so no route is told apart by them
_PREDICATES = {"_aligned_mat", "umma_supported", "wide_out_supported", "gram_stream_supported"}


def route_ops():
    """Every ``ops.<name>(...)`` call inside sage_layer_forward and sage_layer_backward, predicates excluded."""
    with open(os.path.join(ROOT, "gnn_tableextraction_b200", "layers.py")) as f:
        tree = ast.parse(f.read())
    names = set()
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef) and fn.name in ("sage_layer_forward", "sage_layer_backward"):
            for node in ast.walk(fn):
                if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute)
                        and isinstance(node.func.value, ast.Name) and node.func.value.id == "ops"):
                    names.add(node.func.attr)
    return names - _PREDICATES


# ------------------------------------------------------------------------------------------------ route table ---
class Row(NamedTuple):
    id: str
    fin: int                  # input width of the layer (use_pp: the width of the pre-propagated input)
    fout: int
    n: int
    fwd: FrozenSet[str]
    bwd: FrozenSet[str]
    ln: bool = False
    relu: bool = False
    bias: bool = True
    agg: str = GCN
    pp: bool = False
    drop: float = 0.0
    graph: str = "pages"      # "pages": synthetic pages summing to n (paged kernels); "multi": no page table
    aligned: bool = True      # False: the input has unaligned rows (stride fin), as a user's [n, fin] tensor does


def _s(*names):
    return frozenset(names)


COMB_FWD = _s("comb_from", "comb_views", "umma_pack_weights", "umma_linear_fwd_comb")
UMMA_FWD = _s("umma_pack_weights", "umma_linear_fwd")
STACKED_FWD = _s("umma_pack_weights", "umma_linear_fwd_stacked")
CLASS_COMB_BWD = _s("comb_from", "comb_views", "umma_linear_bwd_weight2_comb", "umma_linear_bwd_data_comb")

ROWS = [
    # comb: fin <= COMB_W at n >= UMMA_MIN_ROWS, [h | ah] in one [n, 32] operand
    Row("comb-13-218-ln", 13, 218, 1025, COMB_FWD, _s("layernorm_act_bwd", "umma_linear_bwd_weight_comb", "umma_linear_bwd_data"),
        ln=True, relu=True, aligned=False),
    # fin == COMB_W with a bias: the bias gradient has no free column in the combined operand
    Row("comb-16-64-bias", 16, 64, 1024, COMB_FWD, _s("umma_linear_bwd_weight", "umma_linear_bwd_data")),
    Row("comb-1-256-ln", 1, 256, 1153, COMB_FWD, _s("layernorm_act_bwd", "umma_linear_bwd_weight_comb", "umma_linear_bwd_data"),
        ln=True, relu=True),
    # tensor-core aggregate-first
    Row("umma-64-64-ln-multi", 64, 64, 1279, UMMA_FWD, _s("layernorm_act_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_data"),
        ln=True, relu=True, graph="multi"),
    Row("umma-256-256-ln", 256, 256, 1024, UMMA_FWD, _s("layernorm_act_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_data"),
        ln=True, relu=True),
    Row("umma-33-100-relu-unaligned", 33, 100, 1153, _s("empty_padded") | UMMA_FWD,
        _s("relu_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_data"), relu=True, aligned=False),
    Row("umma-100-255-ln-nobias", 100, 255, 1100, UMMA_FWD, _s("layernorm_act_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_data"),
        ln=True, relu=True, bias=False),
    # exact-fp32 narrow input: wide_out forward, gram_stream weight gradient
    Row("wide-13-218-256", 13, 218, 256, _s("wide_out"), _s("layernorm_act_bwd", "gram_stream", "linear_bwd_data"),
        ln=True, relu=True),
    Row("wide-13-218-1023", 13, 218, 1023, _s("wide_out"), _s("layernorm_act_bwd", "gram_stream", "linear_bwd_data"),
        ln=True, relu=True),
    # generic FFMA aggregate-first
    Row("gen-13-20-255-multi", 13, 20, 255, _s("linear_fwd", "layernorm_act_fwd"),
        _s("layernorm_act_bwd", "linear_bwd_weight", "linear_bwd_data"), ln=True, relu=True, graph="multi"),
    Row("gen-64-300-ln", 64, 300, 1100, _s("linear_fwd", "layernorm_act_fwd"),
        _s("layernorm_act_bwd", "linear_bwd_weight", "linear_bwd_data"), ln=True, relu=True),
    Row("gen-8-32-relu", 8, 32, 600, _s("linear_fwd", "relu_fwd"), _s("relu_bwd", "linear_bwd_weight", "linear_bwd_data"),
        relu=True),
    # WeightedMean: a bias with k1 % 32 == 0 refuses the tensor-core weight gradient
    Row("mean-32-64", 32, 64, 1100, UMMA_FWD, _s("linear_bwd_weight", "umma_linear_bwd_data"), agg=MEAN),
    # project-then-aggregate (class layers)
    Row("proj-218-9-1025", 218, 9, 1025, STACKED_FWD, CLASS_COMB_BWD),
    Row("proj-256-9-1100", 256, 9, 1100, STACKED_FWD, _s("gram_stream", "umma_linear_bwd_data2")),
    Row("proj-218-9-600", 218, 9, 600, _s("linear_fwd"), _s("gram_stream", "wide_out")),
    Row("proj-218-20-1100", 218, 20, 1100, _s("linear_fwd"), _s("umma_linear_bwd_weight2", "linear_bwd_data2")),
    Row("proj-128-32-bias", 128, 32, 1100, _s("linear_fwd"), _s("linear_bwd_weight2", "linear_bwd_data2")),
    Row("proj-128-32-nobias", 128, 32, 1100, _s("linear_fwd"), _s("umma_linear_bwd_weight2", "linear_bwd_data2"), bias=False),
    Row("proj-300-40", 300, 40, 1100, _s("linear_fwd"), _s("linear_bwd_weight2", "linear_bwd_data2")),
    Row("proj-300-200-ln", 300, 200, 1100, _s("linear_fwd", "layernorm_act_fwd"),
        _s("layernorm_act_bwd", "linear_bwd_weight2", "linear_bwd_data2"), ln=True, relu=True),
    # pre-propagated input (plain linear), here with unaligned rows
    Row("pp-26-64", 26, 64, 1200, _s("empty_padded", "linear_fwd", "layernorm_act_fwd"),
        _s("layernorm_act_bwd", "linear_bwd_weight", "linear_bwd_data"), ln=True, relu=True, pp=True, aligned=False),
    # dropout on [h | ah]: the comb-buffer branch and the pre-propagated branch
    Row("drop-comb-13-64", 13, 64, 1100, COMB_FWD | _s("comb_buffer", "dropout_concat"),
        _s("layernorm_act_bwd", "umma_linear_bwd_weight_comb", "umma_linear_bwd_data", "dropout_concat"),
        ln=True, relu=True, drop=0.5, aligned=False),
    Row("drop-pp-26-64", 26, 64, 600, _s("dropout_concat", "linear_fwd", "layernorm_act_fwd"),
        _s("layernorm_act_bwd", "linear_bwd_weight", "linear_bwd_data", "dropout_concat"), ln=True, relu=True, pp=True,
        drop=0.3),
]

# whole models (the sets are unions over their layers)
MEAN_MODELS = [
    # 13 -> 64 comb (bias, fin < 16: bias on the combined operand), 64 -> 64 tensor cores (bias, fin % 32 == 0: FFMA
    # dW), 64 -> 9 stacked forward with gram_stream(qsum).  The caller's gradient of the [n, 9] output has unaligned
    # rows, so the class layer's input gradient is the FFMA two-term one.
    ((13, 64, 9, 2), 1100, COMB_FWD | _s("umma_linear_fwd", "umma_linear_fwd_stacked"),
     _s("umma_linear_bwd_weight_comb", "umma_linear_bwd_data", "linear_bwd_weight", "gram_stream", "linear_bwd_data2")),
    # 16 -> 20 wide_out, 20 -> 20 FFMA, 20 -> 9 FFMA forward with gram_stream
    ((16, 20, 9, 3), 600, _s("wide_out", "linear_fwd"), _s("linear_bwd_weight", "linear_bwd_data", "gram_stream", "linear_bwd_data2")),
]

# SageTrainer steps: (in, hidden, classes, layers), n, forward set, backward set.  Every layer the trainer packs
# arrives with its pack (one batched launch), so the layers themselves pack nothing.
TRAINER = [
    ((13, 64, 2, 2), 1025, _s("comb_from", "comb_views", "umma_linear_fwd_comb", "umma_linear_fwd_stacked"),
     _s("gram_stream", "umma_linear_bwd_data2", "layernorm_act_bwd", "umma_linear_bwd_weight_comb")),
    ((13, 256, 9, 3), 1279, _s("comb_from", "comb_views", "umma_linear_fwd_comb", "umma_linear_fwd", "umma_linear_fwd_stacked"),
     _s("gram_stream", "umma_linear_bwd_data2", "layernorm_act_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_weight_comb")),
    ((16, 100, 20, 3), 1153, _s("comb_from", "comb_views", "umma_linear_fwd_comb", "umma_linear_fwd", "linear_fwd"),
     _s("umma_linear_bwd_weight2", "linear_bwd_data2", "layernorm_act_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_data2",
        "umma_linear_bwd_weight_comb")),
    ((17, 300, 33, 3), 1100, _s("empty_padded", "linear_fwd", "layernorm_act_fwd"),
     _s("linear_bwd_weight2", "linear_bwd_data2", "layernorm_act_bwd", "linear_bwd_weight", "linear_bwd_data")),
    ((13, 128, 16, 4), 40000, _s("comb_from", "comb_views", "umma_linear_fwd_comb", "umma_linear_fwd", "umma_linear_fwd_stacked"),
     _s("gram_stream", "umma_linear_bwd_data2", "layernorm_act_bwd", "umma_linear_bwd_weight", "umma_linear_bwd_weight_comb")),
    # fout == COMB_W class layer: the loss backward writes the class layer's combined gradient operand (dy_comb)
    ((13, 100, 16, 3), 1025, _s("comb_from", "comb_views", "umma_linear_fwd_comb", "umma_linear_fwd", "umma_linear_fwd_stacked"),
     _s("comb_views", "umma_linear_bwd_weight2_comb", "umma_linear_bwd_data_comb", "layernorm_act_bwd", "umma_linear_bwd_weight",
        "umma_linear_bwd_data2", "umma_linear_bwd_weight_comb")),
]


def _tensor_core(fwd, bwd):
    return any(name.startswith("umma_") for name in fwd | bwd)


# ------------------------------------------------------------------------------------------- fp64 reference ---
class RefGraph(NamedTuple):
    src: torch.Tensor
    dst: torch.Tensor
    w: torch.Tensor
    deg: torch.Tensor


def ref_graph(src, dst, w, n):
    dst = torch.as_tensor(np.asarray(dst)).long()
    return RefGraph(torch.as_tensor(np.asarray(src)).long(), dst, torch.as_tensor(np.asarray(w)).double(),
                    torch.bincount(dst, minlength=n).double())


def ref_layer(G, h, W, b, gamma, beta, *, agg=GCN, pp=False, ln=False, relu_mask=None, drop_mask=None, eps=1e-5):
    """z = [h | norm * sum_{u->v} w_e h[u]] W^T + b, LayerNorm, ReLU under a given on/off mask; all float64.
    Returns (out, pre-activation)."""
    x = h
    if not pp:
        s = torch.zeros_like(h).index_add(0, G.dst, G.w[:, None] * h[G.src])
        if agg == GCN:
            norm = torch.where(G.deg > 0, 1.0 / G.deg.clamp(min=1), torch.zeros_like(G.deg))
        else:
            norm = 1.0 / G.deg.clamp(min=1)
        x = torch.cat([h, s * norm[:, None]], 1)
    if drop_mask is not None:
        x = x * drop_mask
    z = x @ W.t()
    if b is not None:
        z = z + b
    if ln:
        z = F.layer_norm(z, (z.shape[1],), gamma, beta, eps)
    return (z if relu_mask is None else z * relu_mask), z


def check_flips(pre, mask):
    """The CUDA ReLU pattern may differ from the float64 one only at pre-activations within fp32 noise of 0."""
    diff = (pre > 0) != mask
    if diff.any():
        assert pre[diff].abs().max().item() <= 1e-5 * pre.abs().max().item(), "activation pattern differs away from 0"
    assert int(diff.sum()) <= 1e-5 * mask.numel() + 2


def _log(tag, errs):
    print(f"{tag}: " + " ".join(f"{k}={v:.2e}" for k, v in errs.items()))  # error levels, shown by pytest -rP


def _check(tag, errs):
    _log(tag, errs)
    for k, e in errs.items():
        assert e < TOL, (tag, k, e)


def _param_blocks(prefix, fin, pp, dW, ref_W, db, ref_b, dg, ref_g, dbe, ref_be):
    """each gradient block against its own maximum: a neighbour block or a bias gradient written at small scale must not
    hide under the self block's magnitude"""
    errs = {}
    if pp:
        errs[prefix + "dW"] = rel_err(dW, ref_W.grad)
    else:
        errs[prefix + "dWs"] = rel_err(dW[:, :fin], ref_W.grad[:, :fin])
        errs[prefix + "dWn"] = rel_err(dW[:, fin:], ref_W.grad[:, fin:])
    if db is not None:
        errs[prefix + "db"] = rel_err(db, ref_b.grad)
    if dg is not None:
        errs[prefix + "dgamma"] = rel_err(dg, ref_g.grad)
        errs[prefix + "dbeta"] = rel_err(dbe, ref_be.grad)
    return errs


# -------------------------------------------------------------------------------------------------- inputs ---
@functools.lru_cache(maxsize=None)
def _page(seed, n, k):
    from gnn_tableextraction_b200 import synth

    return synth.make_page(seed, n=n, k=k)


def make_pages(n, k=6, feat_w=None, classes=None, seed=0):
    """synthetic pages of at most 300 nodes whose sizes sum to exactly n; optional random features / labels"""
    sizes = [300] * (n // 300) + ([n % 300] if n % 300 else [])
    pages = [_page(i % 8, s, k) for i, s in enumerate(sizes)]
    rng = np.random.default_rng(seed)
    if feat_w is not None:
        pages = [dataclasses.replace(p, feat=rng.standard_normal((p.num_nodes, feat_w)).astype(np.float32)) for p in pages]
    if classes is not None:
        pages = [dataclasses.replace(p, label=rng.integers(0, classes, p.num_nodes).astype(np.float32)) for p in pages]
    return pages


def make_graph(kind, n, seed=0):
    """(CUDA graph, float64 reference graph) with exactly n nodes"""
    import gnn_tableextraction_b200 as gte
    from gnn_tableextraction_b200 import synth
    from helpers import cuda_graph_from_arrays
    from oracle.csx import batch_coo

    if kind == "multi":  # duplicates, self loops, zero in-degree rows; no page table
        src, dst, w = synth.random_multigraph(seed, n, 6 * n, with_isolated=True)
        return cuda_graph_from_arrays(src, dst, n, w), ref_graph(src, dst, w, n)
    pages = make_pages(n)
    src, dst, w, noff, _ = batch_coo(pages)
    assert int(noff[-1]) == n
    return gte.PageGraphBatch.from_pages(pages, DEV), ref_graph(src, dst, w, n)


def _padded(t):
    from gnn_tableextraction_b200 import ops

    out = ops.empty_padded(t.shape[0], t.shape[1], DEV)
    out.copy_(t)
    return out


def _dropout_mask(n, f, p, seed, offset):
    """the scaled keep mask [n, f] a dropout call site with these Philox coordinates applies"""
    from gnn_tableextraction_b200 import ops

    ones = ops.empty_padded(n, f, DEV)
    ones.fill_(1.0)
    return ops.dropout_concat(ones, None, p, seed=seed, offset=offset)[0].cpu().double()


class OpsSpy:
    """Stands in for the ``ops`` module inside layers.py and records which route functions layers.py calls, per phase.
    Only the calls made by layers.py count (ops functions that call each other, e.g. for an output buffer, do not)."""

    def __init__(self, names):
        from gnn_tableextraction_b200 import ops

        self._ops, self._names = ops, names
        self.calls = {"fwd": set(), "bwd": set()}
        self.phase = "fwd"

    def __getattr__(self, name):
        f = getattr(self._ops, name)
        if name not in self._names:
            return f

        def wrap(*a, **kw):
            self.calls[self.phase].add(name)
            return f(*a, **kw)

        return wrap


def _spy(monkeypatch):
    from gnn_tableextraction_b200 import layers as L

    spy = OpsSpy(route_ops())
    monkeypatch.setattr(L, "ops", spy)
    backward = L.sage_layer_backward

    def tagged_backward(*a, **kw):
        spy.phase = "bwd"
        return backward(*a, **kw)

    monkeypatch.setattr(L, "sage_layer_backward", tagged_backward)
    return spy


def _leaf(t):
    return t.detach().double().clone().requires_grad_(True)


# ----------------------------------------------------------------------------------------------- layer rows ---
def _run_row(row: Row, monkeypatch):
    from gnn_tableextraction_b200 import layers as L

    n, fin, fo = row.n, row.fin, row.fout
    g, G = (None, None) if row.pp else make_graph(row.graph, n)
    K = fin if row.pp else 2 * fin
    gen = torch.Generator().manual_seed(n * 1000 + fin * 7 + fo)
    h0 = torch.randn(n, fin, generator=gen)
    W = (torch.rand(fo, K, generator=gen) - 0.5) * (2.0 / K ** 0.5)
    b = torch.randn(fo, generator=gen) * 0.1 if row.bias else None
    gamma = torch.rand(fo, generator=gen) + 0.5 if row.ln else None
    beta = torch.randn(fo, generator=gen) * 0.1 if row.ln else None
    up = torch.randn(n, fo, generator=gen)
    dev = lambda t: None if t is None else t.to(DEV)
    h = h0.to(DEV) if not row.aligned else _padded(h0.to(DEV))
    assert (h.stride(0) % 4 == 0) == row.aligned or n <= 1
    drop, M = None, None
    if row.drop:
        drop = L.DropoutSpec(row.drop, seed=1234, offset=64)
        M = _dropout_mask(n, K, row.drop, 1234, 64)
    w_edge = None if row.pp else g.edata["feat"]

    spy = _spy(monkeypatch)
    out, ctx = L.sage_layer_forward(g, h, w_edge, W.to(DEV), dev(b), dev(gamma), dev(beta), ln=row.ln, relu=row.relu,
                                    agg=row.agg, use_pp=row.pp, dropout=drop)
    spy.phase = "bwd"
    nan = lambda *s: torch.full(s, float("nan"), device=DEV)  # every block must be written
    dW = nan(fo, K)
    db = nan(fo) if row.bias else None
    dg, dbe = (nan(fo), nan(fo)) if row.ln else (None, None)
    dh = L.sage_layer_backward(g, ctx, _padded(up.to(DEV)), W.to(DEV), dev(gamma), dev(beta), dW, db, dg, dbe, need_dh=True)
    torch.cuda.synchronize()
    assert spy.calls["fwd"] == row.fwd, (row.id, "forward", sorted(spy.calls["fwd"]))
    assert spy.calls["bwd"] == row.bwd, (row.id, "backward", sorted(spy.calls["bwd"]))

    out_c = out.cpu()
    mask = (out_c > 0).double() if row.relu else None
    rh, rW, rb, rg, rbe = _leaf(h0), _leaf(W), *(None if t is None else _leaf(t) for t in (b, gamma, beta))
    ref, pre = ref_layer(G, rh, rW, rb, rg, rbe, agg=row.agg, pp=row.pp, ln=row.ln, relu_mask=mask, drop_mask=M)
    if row.relu:
        check_flips(pre.detach(), mask.bool())
    (ref * up.double()).sum().backward()
    errs = {"out": rel_err(out_c, ref.detach()), "dh": rel_err(dh, rh.grad)}
    errs.update(_param_blocks("", fin, row.pp, dW, rW, db, rb, dg, rg, dbe, rbe))
    return errs


TC_ROWS = [r for r in ROWS if _tensor_core(r.fwd, r.bwd)]
FFMA_ROWS = [r for r in ROWS if not _tensor_core(r.fwd, r.bwd)]


@pytest.mark.gpu
@pytest.mark.parametrize("row", TC_ROWS, ids=[r.id for r in TC_ROWS])
def test_layer_route_tensor_core(row, monkeypatch, umma_kernel):
    _check(f"{row.id} [{umma_kernel}]", _run_row(row, monkeypatch))


@pytest.mark.gpu
@pytest.mark.parametrize("row", FFMA_ROWS, ids=[r.id for r in FFMA_ROWS])
def test_layer_route_fp32(row, monkeypatch):
    _check(row.id, _run_row(row, monkeypatch))


# ------------------------------------------------------------------------------------------- MeanSAGE models ---
@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n,fwd,bwd", MEAN_MODELS, ids=[f"{c}@{n}" for c, n, _, _ in MEAN_MODELS])
def test_meansage_routes_end_to_end(cfg, n, fwd, bwd, monkeypatch, umma_kernel):
    """MeanSAGE through nn autograd (ReluL2Norm between the layers) against float64, every gradient block on its own"""
    import gnn_tableextraction_b200 as gte

    g, G = make_graph("pages", n)
    torch.manual_seed(3)
    model = gte.MeanSAGE(*cfg)
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    model = model.to(DEV)
    gen = torch.Generator().manual_seed(n)
    h0 = torch.randn(n, cfg[0], generator=gen)
    up = torch.randn(n, cfg[2], generator=gen)
    w = g.edata["feat"]
    pre_acts = [None] * len(model.layers)
    hooks = [layer.register_forward_hook(lambda m, i, o, j=j: pre_acts.__setitem__(j, o.detach().cpu()))
             for j, layer in enumerate(model.layers)]
    spy = _spy(monkeypatch)
    h = h0.to(DEV).requires_grad_(True)
    y = model(g, h, w)
    spy.phase = "bwd"
    (y * up.to(DEV)).sum().backward()
    torch.cuda.synchronize()
    for hk in hooks:
        hk.remove()
    assert spy.calls["fwd"] == fwd, sorted(spy.calls["fwd"])
    assert spy.calls["bwd"] == bwd, sorted(spy.calls["bwd"])

    rh = _leaf(h0)
    params = {k: _leaf(v) for k, v in sd.items()}
    x = rh
    nl = len(model.layers)
    for j in range(nl):
        x, pre = ref_layer(G, x, params[f"layers.{j}.linear.weight"], params[f"layers.{j}.linear.bias"], None, None, agg=MEAN)
        if j != nl - 1:
            mask = pre_acts[j] > 0
            check_flips(pre.detach(), mask)
            x = F.normalize(x * mask.double(), p=2.0, dim=1, eps=1e-12)
    (x * up.double()).sum().backward()
    errs = {"out": rel_err(y, x.detach()), "dh": rel_err(h.grad, rh.grad)}
    for j, layer in enumerate(model.layers):
        fin = layer.linear.weight.shape[1] // 2
        errs.update(_param_blocks(f"l{j}.", fin, False, layer.linear.weight.grad, params[f"layers.{j}.linear.weight"],
                                  layer.linear.bias.grad, params[f"layers.{j}.linear.bias"], None, None, None, None))
    _check(f"MeanSAGE{cfg}@{n} [{umma_kernel}]", errs)


# ------------------------------------------------------------------------------------------------ trainer ---
@pytest.mark.gpu
@pytest.mark.parametrize("cfg,n,fwd,bwd", TRAINER, ids=[f"{c}@{n}" for c, n, _, _ in TRAINER])
def test_trainer_step_routes(cfg, n, fwd, bwd, monkeypatch):
    """One SageTrainer step (batched weight packs, the loss backward's combined operand, the aggregate-first input
    gradient) against float64: loss, #correct, logits and every gradient block; the captured replay on a fresh trainer
    from the same weights equals the eager step bit for bit"""
    import gnn_tableextraction_b200 as gte
    from gnn_tableextraction_b200.graph import batch_pages_host
    from oracle.csx import batch_coo

    fin0, hid, C, nl = cfg
    pages = make_pages(n, feat_w=None if fin0 == 13 else fin0, classes=C, seed=C)
    hb = batch_pages_host(pages)
    src, dst, w, _, _ = batch_coo(pages)
    G = ref_graph(src, dst, w, n)
    torch.manual_seed(11)
    sd = {k: v.clone() for k, v in gte.GcnSAGE(fin0, hid, C, nl, F.relu, 0).state_dict().items()}

    def trainer():
        m = gte.GcnSAGE(fin0, hid, C, nl, F.relu, 0)
        m.load_state_dict(sd)
        return gte.SageTrainer(m.to(DEV))

    tr = trainer()
    g = gte.PageGraphBatch.from_host(hb, DEV)
    outs = []
    logits, _ = tr.forward(g, keep_ctx=False, layer_outputs=outs)
    masks = [o.cpu() > 0 for o in outs[:-1]]
    logits = logits.cpu()
    del outs
    with monkeypatch.context() as mp:
        spy = _spy(mp)
        st = tr.train_step(g).clone()
        torch.cuda.synchronize()
    assert spy.calls["fwd"] == fwd, sorted(spy.calls["fwd"])
    assert spy.calls["bwd"] == bwd, sorted(spy.calls["bwd"])
    grads = {k: p.grad.clone() for k, p in tr.model.named_parameters()}
    flat_grad, flat_param = tr.flat_grad.clone(), tr.flat_param.clone()

    tc = trainer()
    tc.capture(hb)
    tc.load_batch(hb)
    assert torch.equal(tc.replay(), st)
    assert torch.equal(tc.flat_grad, flat_grad) and torch.equal(tc.flat_param, flat_param)

    params = {k: _leaf(v) for k, v in sd.items()}
    x = torch.from_numpy(hb["feat"].numpy()).double()
    for j in range(nl):
        p = lambda s: params.get(f"layers.{j}.{s}")
        hidden = j < nl - 1
        x, pre = ref_layer(G, x, p("linear.weight"), p("linear.bias"), p("lynorm.weight"), p("lynorm.bias"), ln=hidden,
                           relu_mask=masks[j].double() if hidden else None)
        if hidden:
            check_flips(pre.detach(), masks[j])
    labels = torch.from_numpy(hb["label"].numpy()).long()
    loss = F.cross_entropy(x, labels)
    loss.backward()
    st = st.cpu()
    assert abs(st[0].item() / st[1].item() - loss.item()) < TOL * max(1.0, abs(loss.item()))
    assert abs(st[2].item() - (x.argmax(1) == labels).sum().item()) <= 2  # near-tied logits may flip
    errs = {"logits": rel_err(logits, x.detach())}
    for j, layer in enumerate(tr.model.layers):
        q = f"layers.{j}."
        fin = layer.linear.weight.shape[1] // 2
        errs.update(_param_blocks(f"l{j}.", fin, False, grads[q + "linear.weight"], params[q + "linear.weight"],
                                  grads[q + "linear.bias"], params[q + "linear.bias"], grads.get(q + "lynorm.weight"),
                                  params.get(q + "lynorm.weight"), grads.get(q + "lynorm.bias"), params.get(q + "lynorm.bias")))
    _check(f"trainer{cfg}@{n}", errs)


# ---------------------------------------------------------------------------------------- kernel identity ---
def cuda_kernel_names(fn):
    """names of the CUDA kernels ``fn`` launches (torch.profiler, CUDA activity only)"""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with warnings.catch_warnings():  # one profiling cycle: that events() forgets earlier cycles does not matter here
        warnings.simplefilter("ignore", UserWarning)
        return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


@pytest.mark.gpu
@pytest.mark.parametrize("fin,split", [(32, "false"), (33, "true")])
def test_umma_fixture_runs_the_kernel_it_names(fin, split, umma_kernel):
    """two-segment forward at n = 1279, fo = 64: 2 k-blocks keep two accumulators (SPLIT = false), 4 k-blocks split; the
    `pair` mode runs the CTA-pair kernel and only that, the `single` mode the single-CTA kernel"""
    from gnn_tableextraction_b200 import ops

    n, fo = 1279, 64
    x1, x2 = _padded(torch.randn(n, fin, device=DEV)), _padded(torch.randn(n, fin, device=DEV))
    pack = ops.umma_pack_weights(torch.randn(fo, 2 * fin, device=DEV) * 0.1, fin, 2)
    names = cuda_kernel_names(lambda: ops.umma_linear_fwd(x1, x2, fin, pack, None, fo))
    gemm = {s for s in names if "k_umma_gemm" in s}
    if umma_kernel == "pair":
        assert gemm and all(f"k_umma_gemm_pair<{split}>" in s for s in gemm), names
    else:
        assert gemm and all(f"k_umma_gemm<{split}>" in s for s in gemm), names


# ------------------------------------------------------------------------------------------------ CPU guard ---
def test_every_layer_route_op_has_a_row():
    """every ops function sage_layer_forward / sage_layer_backward can call is expected by at least one table row"""
    names = route_ops()
    assert {"linear_fwd", "umma_linear_fwd", "gram_stream", "wide_out"} <= names  # the parse found the two functions
    covered = set()
    for r in ROWS:
        covered |= r.fwd | r.bwd
    for _, _, fwd, bwd in MEAN_MODELS + TRAINER:
        covered |= fwd | bwd
    assert names - covered == set(), f"no route-table row expects {sorted(names - covered)}"
    assert covered <= names, f"rows expect functions layers.py never calls: {sorted(covered - names)}"
