"""MeanSAGE in the fused trainer: the ReLU + L2-normalise epilogue of the tensor-core projection (fuse_ln = 2), the
ReLU + L2-normalise backward that also emits the bias gradient, and ``SageTrainer(MeanSAGE(...))`` with its captured,
capacity, resident, validation, predict, data-parallel and checkpoint paths, against float64, the reference's golden
vectors, the oracle and the autograd path.

Bounds (u = 2^-24, K = test_gpu_contraction_numerics.K):
  * z has the per-element bound of the projection, E = K u (G S + Gb |b|) (test_gpu_contraction_numerics.BOUNDS).
  * y = r / max(||r||, eps), r = relu(z): relu is exact and 1-Lipschitz, | ||r~|| - ||r|| | <= ||E||, so against the
    float64 y of the exact operands
        |y~ - y| <= E_i / nrm + |y_i| ||E|| / nrm + K u (f / 2 + 2) |y_i|
    the last term being the rounding of the epilogue itself: the fp32 sum of f squares (relative f u; the split
    accumulator adds one merge), halved by the square root, + 1 for the root and + 1 for the division.
  * Against the float64 y of the kernel's OWN z (same bits as the z it stored) only that last term remains.
  * dz_colsum: the fixed-order reduction of the kernel's own dz over the rows: |got - sum dz| <= K u G sum |dz| with
    G = rows per warp + 8 warps + the blocks + 1, plus u |old| when accumulating.
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
import test_gpu_contraction_numerics as cn
from conftest import TOL, load_golden, rel_err, sub
from helpers import cuda_graph_from_arrays, oracle_graph_from_pages
from gnn_tableextraction_b200 import _lib, ops, synth
from gnn_tableextraction_b200.engine import LayerSpec, model_spec
from gnn_tableextraction_b200.graph import batch_pages_host
from oracle import sage_oracle as so

DEV = "cuda"
U = cn.U
K = cn.K
L2_EPS = 1e-12
BIG_ROW = 7          # this row of every operand is scaled by 1e13
ZERO_ROW = 61        # rows r % ZERO_ROW == 5 are zero: z = b < 0, so every z <= 0 and y must be exactly 0


def _bits(t):
    return t.contiguous().view(torch.int32).clone()


# ------------------------------------------------------------------------------------------------ 1. epilogue ---
def _raw_fwd(form, xs, fin, pack, b, fo, mode, z, y, n):
    """gte_umma_linear_fwd(_comb) on caller-owned outputs (pre-filled with NaN), with the epilogue selector"""
    l = _lib.lib()
    zp, ldz = (None, 0) if z is None else (z.data_ptr(), z.stride(0))
    yp, ldy = (None, 0) if y is None else (y.data_ptr(), y.stride(0))
    if form == "comb":
        rc = l.gte_umma_linear_fwd_comb(xs.data_ptr(), xs.stride(0), fin, pack.data_ptr(), b.data_ptr(), None, None,
                                        L2_EPS, 0, mode, zp, ldz, yp, ldy, None, None, n, fo, ops._stream())
    else:
        x1, x2 = xs
        rc = l.gte_umma_linear_fwd(x1.data_ptr(), x1.stride(0), x2.data_ptr(), x2.stride(0), fin, pack.data_ptr(),
                                   b.data_ptr(), None, None, L2_EPS, 0, mode, zp, ldz, yp, ldy, None, None, n, fo,
                                   ops._stream())
    _lib.check(rc, "umma forward")


def _nan(n, f):
    return ops.empty_padded(n, f, torch.device(DEV)).fill_(float("nan"))


def _operands(n, fin, fo, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    h = torch.randn(n, fin, device=DEV, generator=g)
    ah = torch.randn(n, fin, device=DEV, generator=g)
    for x in (h, ah):
        x[5::ZERO_ROW] = 0.0
        if n > BIG_ROW:
            x[BIG_ROW] *= 1e13
    W = (torch.rand(fo, 2 * fin, device=DEV, generator=g) - 0.5) * (2.0 / (2 * fin) ** 0.5)
    b = -(torch.rand(fo, device=DEV, generator=g) * 0.1 + 0.01)  # negative: a zero row has every z < 0
    return h, ah, W, b


def _ref(h, ah, W, b):
    X = torch.cat([h, ah], 1).double()
    W64 = W.double()
    return X @ W64.T + b.double(), X.abs() @ W64.abs().T


def _y64(z64):
    r = z64.clamp_min(0)
    return r / r.norm(dim=1, keepdim=True).clamp_min(L2_EPS)


def _ratio(got, ref, bound):
    err = (got.double() - ref).abs()
    assert not torch.isnan(err).any(), "NaN in the output (an element was not written)"
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(r.max().item()) if r.numel() else 0.0


EPI_N = (1024, 1100, 153600)
EPI_FO = (32, 64, 96, 218, 224, 256)


@pytest.mark.gpu
@pytest.mark.parametrize("n", EPI_N)
@pytest.mark.parametrize("fo", EPI_FO)
@pytest.mark.parametrize("form", ("comb", "two_segments"))
def test_relu_l2norm_epilogue_per_element(form, fo, n, umma_kernel):
    """fuse_ln = 2 on both kernels: z within its projection bound and bit-identical to mode 0; y within the propagated
    float64 bound, within the rounding of the epilogue of the kernel's own z, the same bits without z (predict), the
    same bits on a repeated call, exactly 0 on rows whose z are all <= 0; every output element written"""
    fin = 13 if form == "comb" else 218
    h, ah, W, b = _operands(n, fin, fo, seed=n + 7 * fo + fin)
    pack = ops.umma_pack_weights(W, fin, 2)
    if form == "comb":
        xs = ops.comb_buffer(n, torch.device(DEV))
        xs[:, :fin] = h
        xs[:, 16:16 + fin] = ah
        G, Gb = cn.BOUNDS["umma_linear_fwd_comb"]()
    else:
        x1, x2 = ops.empty_padded(n, fin, torch.device(DEV)), ops.empty_padded(n, fin, torch.device(DEV))
        x1.copy_(h)
        x2.copy_(ah)
        xs = (x1, x2)
        G, Gb = cn.BOUNDS["umma_linear_fwd"](fin, 2)

    def call(mode, want_z=True, want_y=True):
        z = _nan(n, fo) if want_z else None
        y = _nan(n, fo) if want_y else None
        _raw_fwd(form, xs, fin, pack, b, fo, mode, z, y, n)
        return z, y

    z, y = call(2)
    torch.cuda.synchronize()
    z64, s64 = _ref(h, ah, W, b)
    E = K * U * (G * s64 + Gb * b.double().abs())
    rz = _ratio(z[:, :fo] if z.shape[1] != fo else z, z64, E)
    assert rz <= 1.0, f"z breaks its bound: {rz}"
    y64 = _y64(z64)
    nrm = z64.clamp_min(0).norm(dim=1, keepdim=True).clamp_min(L2_EPS)
    live = (z64 > 0).any(1)
    eps_epi = K * U * (fo / 2 + 3)
    by = E / nrm + y64.abs() * (E.norm(dim=1, keepdim=True) / nrm) + eps_epi * y64.abs()
    ry = _ratio(y[live], y64[live], by[live])
    assert ry <= 1.0, f"y breaks the propagated bound: {ry}"
    yo = _y64(z.double())
    ro = _ratio(y, yo, eps_epi * yo.abs())
    assert ro <= 1.0, f"y breaks the epilogue's own rounding bound: {ro}"
    zero_rows = torch.arange(5, n, ZERO_ROW, device=DEV)
    assert torch.equal(y[zero_rows], torch.zeros_like(y[zero_rows])), "a row with every z <= 0 must give exactly 0"
    if n > BIG_ROW:
        assert y[BIG_ROW].abs().max().item() > 0 and torch.isfinite(y[BIG_ROW]).all()
    print(f"l2 epilogue {form} [{umma_kernel}] fo={fo} n={n}: z {rz:.3e} y {ry:.3e} y(own z) {ro:.3e}")
    z0, _ = call(0, want_y=False)
    assert torch.equal(_bits(z0), _bits(z)), "the z bits depend on the epilogue"
    _, yp = call(2, want_z=False)
    assert torch.equal(_bits(yp), _bits(y)), "want_z=False changed y"
    z2, y2 = call(2)
    assert torch.equal(_bits(z2), _bits(z)) and torch.equal(_bits(y2), _bits(y)), "a repeated call changed bits"


@pytest.mark.gpu
@pytest.mark.parametrize("form", ("comb", "two_segments"))
def test_relu_l2norm_epilogue_empty_batch_writes_nothing(form):
    fin, fo = (13, 218) if form == "comb" else (218, 218)
    W = torch.randn(fo, 2 * fin, device=DEV)
    b = torch.zeros(fo, device=DEV)
    pack = ops.umma_pack_weights(W, fin, 2)
    z, y = _nan(4, fo), _nan(4, fo)
    before = (_bits(z), _bits(y))
    x = ops.empty_padded(0, 32 if form == "comb" else fin, torch.device(DEV))
    _raw_fwd(form, x if form == "comb" else (x, x), fin, pack, b, fo, 2, z, y, 0)
    torch.cuda.synchronize()
    assert torch.equal(_bits(z), before[0]) and torch.equal(_bits(y), before[1])


@pytest.mark.gpu
def test_epilogue_selector_refusals():
    fin, fo, n = 218, 218, 1024
    x = ops.empty_padded(n, fin, torch.device(DEV)).normal_()
    pack = ops.umma_pack_weights(torch.randn(fo, 2 * fin, device=DEV), fin, 2)
    b = torch.zeros(fo, device=DEV)
    with pytest.raises(gte.GteError, match="fuse_ln must be"):
        _raw_fwd("two_segments", (x, x), fin, pack, b, fo, 3, _nan(n, fo), _nan(n, fo), n)
    with pytest.raises(gte.GteError, match="needs y"):
        _raw_fwd("two_segments", (x, x), fin, pack, b, fo, 2, _nan(n, fo), None, n)
    with pytest.raises(gte.GteError, match="two different epilogues"):
        ops.umma_linear_fwd(x, x, fin, pack, b, fo, fuse_ln=True, l2=True)


# ------------------------------------------------------------------------------- 2. backward with colsum ---
BWD_ROWS = (1, 255, 4097, 153600)


@pytest.mark.gpu
@pytest.mark.parametrize("n", BWD_ROWS)
@pytest.mark.parametrize("f", (9, 64, 218, 1024))
def test_relu_l2norm_bwd_colsum(f, n):
    """dz bits equal gte_relu_l2norm_bwd's; dz_colsum within the bound of a fixed-order reduction of that dz, with and
    without accumulate; the same bits on a repeated call"""
    g = torch.Generator(device=DEV).manual_seed(f * 7 + n)
    z = torch.randn(n, f, device=DEV, generator=g)
    z[3::17] *= 1e13
    z[5::ZERO_ROW] = -1.0  # every z <= 0: dz = 0
    dy = torch.randn(n, f, device=DEV, generator=g)
    ref_dz = ops.relu_l2norm_bwd(dy, z, L2_EPS)
    cs = torch.full((f,), float("nan"), device=DEV)
    dz = ops.relu_l2norm_bwd_colsum(dy, z, L2_EPS, dz_colsum=cs)
    assert torch.equal(_bits(dz), _bits(ref_dz)), "dz bits differ from gte_relu_l2norm_bwd"
    d64 = dz.double()
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    grid = max(1, min(-(-n // 8), 2 * sm))
    G = -(-n // (8 * grid)) + 8 + grid + 1
    bound = K * U * G * d64.abs().sum(0)
    r = _ratio(cs, d64.sum(0), bound)
    assert r <= 1.0, r
    old = torch.randn(f, device=DEV, generator=g) * 1e3
    acc = old.clone()
    dz2 = ops.relu_l2norm_bwd_colsum(dy, z, L2_EPS, dz_colsum=acc, accumulate=True)
    ra = _ratio(acc, d64.sum(0) + old.double(), bound + U * old.double().abs() * 2)
    assert ra <= 1.0, ra
    cs2 = torch.full((f,), float("nan"), device=DEV)
    ops.relu_l2norm_bwd_colsum(dy, z, L2_EPS, dz_colsum=cs2)
    assert torch.equal(_bits(cs2), _bits(cs)) and torch.equal(_bits(dz2), _bits(dz)), "repeated call changed bits"
    print(f"relu_l2norm_bwd_colsum f={f} n={n}: colsum {r:.3e} accumulate {ra:.3e}")


@pytest.mark.gpu
def test_relu_l2norm_bwd_colsum_empty_batch():
    f = 64
    cs = torch.full((f,), float("nan"), device=DEV)
    x = torch.empty((0, f), device=DEV)
    ops.relu_l2norm_bwd_colsum(x, x, L2_EPS, dz_colsum=cs)
    assert torch.equal(cs, torch.zeros_like(cs)), "n = 0 writes zeros"
    old = torch.randn(f, device=DEV)
    acc = old.clone()
    ops.relu_l2norm_bwd_colsum(x, x, L2_EPS, dz_colsum=acc, accumulate=True)
    assert torch.equal(acc, old), "n = 0 with accumulate leaves dz_colsum unchanged"


# --------------------------------------------------------------------------------------- trainer helpers ---
def _models(seed, cfg):
    torch.manual_seed(seed)
    om = so.OracleMeanSAGE(*cfg)
    cm = gte.MeanSAGE(*cfg)
    cm.load_state_dict(om.state_dict())
    return om, cm.to(DEV)


def _model(seed, cfg=(13, 218, 9, 2)):
    return _models(seed, cfg)[1]


def _masks(tr, g):
    """the ReLU on/off pattern of every hidden layer of the trainer's forward (y > 0 exactly where z > 0)"""
    outs = []
    logits, _ = tr.forward(g, keep_ctx=False, layer_outputs=outs)
    return logits.clone(), [(o > 0).cpu() for o in outs[:-1]]


def _check_flips(pre, mask):
    """DESIGN.md (c): the trainer's ReLU pattern may differ from the oracle's only within fp32 noise of 0"""
    diff = (pre > 0) != mask
    if diff.any():
        assert pre[diff].abs().max().item() <= 1e-5 * pre.abs().max().item(), "activation pattern differs away from 0"
    assert int(diff.sum()) <= 1e-5 * mask.numel() + 2


def _oracle_forward(om, og, masks):
    """``OracleMeanSAGE.forward`` (models.py:164-170) with each hidden layer's F.relu evaluated under a GIVEN on/off
    pattern (h * mask) -- the ReLU caveat of DESIGN.md (c): fp32 implementations may disagree on elements within rounding
    noise of 0, so the gradients are compared under the same pattern"""
    h, w = og.ndata["feat"], og.edata["feat"]
    last = len(om.layers) - 1
    for l, layer in enumerate(om.layers):
        h = layer(og, h, w)
        if l != last:
            _check_flips(h.detach(), masks[l])
            h = F.normalize(h * masks[l].to(h.dtype))
    return h


def _oracle_step(om, og, masks, opt=None):
    if opt is not None:
        opt.zero_grad()
    logits = _oracle_forward(om, og, masks)
    loss = torch.nn.CrossEntropyLoss()(logits, og.ndata["label"].long())
    loss.backward()
    if opt is not None:
        opt.step()
    return logits.detach(), loss.detach()


# ----------------------------------------------------------------------------------------- 3. golden -------
@pytest.mark.gpu
def test_trainer_reproduces_the_reference_golden():
    d = load_golden("meansage")
    inf, hid, ncls, nl = (int(v) for v in d["config"])
    model = gte.MeanSAGE(inf, hid, ncls, nl)
    model.load_state_dict(sub(d, "state"))
    tr = gte.SageTrainer(model.to(DEV))
    g = cuda_graph_from_arrays(d["src"], d["dst"], int(d["num_nodes"]), d["weight"], d["feat"])
    logits, ctxs = tr.forward(g)
    assert rel_err(logits, d["out"]) < TOL
    tr.backward(g, ctxs, torch.from_numpy(d["upstream"]).float().to(DEV).contiguous())
    grads = sub(d, "grad")
    for k, p in model.named_parameters():
        assert rel_err(p.grad, grads[k]) < TOL, k


# ------------------------------------------------------------------------------------------ 4. oracle -------
class _Counter:
    def __init__(self, monkeypatch, names):
        self.calls = []
        for name in names:
            fn = getattr(ops, name)

            def wrapped(*a, _fn=fn, _name=name, **kw):
                self.calls.append((_name, a[0].shape[1], a[1].shape[1]))
                return _fn(*a, **kw)
            monkeypatch.setattr(ops, name, wrapped)


@pytest.mark.gpu
@pytest.mark.parametrize("pages", (8, 512))
@pytest.mark.parametrize("cfg", ((13, 218, 9, 2), (13, 64, 9, 2)))
def test_train_step_matches_the_oracle(cfg, pages, monkeypatch, umma_kernel):
    """logits, loss and every gradient within 1e-5 under the trainer's ReLU pattern; the 64-wide hidden layer
    (fin % 32 == 0) takes the tensor-core weight gradient now that the bias gradient comes from the L2 backward"""
    pg = synth.make_pages(pages)
    om, cm = _models(5, cfg)
    tr = gte.SageTrainer(cm, lr=0.0, weight_decay=0.0)
    g = gte.PageGraphBatch.from_pages(pg, DEV)
    logits, masks = _masks(tr, g)
    og = oracle_graph_from_pages(pg)
    ologits, oloss = _oracle_step(om, og, masks)
    assert rel_err(logits, ologits) < TOL
    cnt = _Counter(monkeypatch, ("umma_linear_bwd_weight", "linear_bwd_weight", "gram_stream"))
    stats = tr.train_step(g).cpu()
    monkeypatch.undo()
    assert abs(stats[0].item() / stats[1].item() - oloss.item()) <= TOL * abs(oloss.item())
    for (k, p), (_, q) in zip(cm.named_parameters(), om.named_parameters()):
        assert rel_err(p.grad, q.grad) < TOL, k
    hid = cfg[1]
    hidden_dw = [c for c in cnt.calls if c[1] == hid and c[2] == hid]
    assert hidden_dw and all(c[0] == "umma_linear_bwd_weight" for c in hidden_dw), cnt.calls


# --------------------------------------------------------------------------------------- 5. Adam steps ------
@pytest.mark.gpu
def test_three_adam_steps_match_torch_adam_on_the_oracle():
    """the setting of test_gpu_model.test_trainer_three_steps_match_oracle_adam: gradients of every step within 5e-5
    (steps > 0 see drifted parameters), parameters after three steps within 1e-4 (Adam's 1 / sqrt(v) amplifies the
    gradients' last-bit noise)"""
    pg = synth.make_pages(6, n=80, k=6)
    om, cm = _models(9, (13, 48, 9, 2))
    tr = gte.SageTrainer(cm, lr=0.01, weight_decay=5e-4)
    opt = so.make_optimizer(om, lr=0.01, weight_decay=5e-4)
    g = gte.PageGraphBatch.from_pages(pg, DEV)
    og = oracle_graph_from_pages(pg)
    for step in range(3):
        _, masks = _masks(tr, g)
        tr.train_step(g)
        opt.zero_grad()
        _oracle_step(om, og, masks)
        for (k, p), (_, q) in zip(cm.named_parameters(), om.named_parameters()):
            assert rel_err(p.grad, q.grad) < 5e-5, (step, k)
        opt.step()
    for (k, p), (_, q) in zip(cm.named_parameters(), om.named_parameters()):
        assert rel_err(p.data, q.data) < 1e-4, k


# ------------------------------------------------------------------------------ 6. captured and derived ------
def _groups(sizes, seed, k=6):
    pool = synth.make_pages(sum(sizes), base_seed=seed, ragged=True, k=k)
    out, i = [], 0
    for s in sizes:
        out.append(pool[i:i + s])
        i += s
    return out


def _capacity_of(hbs, slack=(37, 101, 1)):
    return gte.BatchCapacity(nodes=max(int(h["num_nodes"]) for h in hbs) + slack[0],
                             edges=max(int(h["src"].numel()) for h in hbs) + slack[1],
                             pages=max(len(h["batch_num_nodes"]) for h in hbs) + slack[2],
                             page_nodes=max(max(h["batch_num_nodes"]) for h in hbs),
                             page_edges=max(max(h["batch_num_edges"]) for h in hbs))


@pytest.mark.gpu
def test_captured_replay_is_bit_identical_to_eager():
    hb = batch_pages_host(synth.make_pages(8, base_seed=3, ragged=True, k=6))
    te, tc = gte.SageTrainer(_model(21)), gte.SageTrainer(_model(21))
    tc.capture(hb)
    for i in range(3):
        se = te.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        tc.load_batch(hb)
        sc = tc.replay().clone()
        assert torch.equal(se, sc), i
        assert torch.equal(te.flat_param, tc.flat_param) and torch.equal(te.exp_avg_sq, tc.exp_avg_sq), i


@pytest.mark.gpu
def test_capacity_capture_on_ragged_batches_trains_like_eager():
    groups = _groups((5, 6, 4, 7, 5, 6), seed=7)
    hbs = [batch_pages_host(p) for p in groups]
    assert min(int(h["num_nodes"]) for h in hbs) >= 1024  # both sides take the tensor-core routes
    cap = _capacity_of(hbs)
    te, tc = gte.SageTrainer(_model(31)), gte.SageTrainer(_model(31))
    tc.capture(hbs[2], capacity=cap)
    for i, hb in enumerate(hbs):
        se = te.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone().cpu()
        if i == 0:
            ge = te.flat_grad[:te._flat_len].clone()
        tc.load_batch(hb)
        sc = tc.replay().clone().cpu()
        if i == 0:
            assert rel_err(tc.flat_grad[:tc._flat_len], ge) < TOL
        assert se[1].item() == sc[1].item() == hb["num_nodes"] and se[2].item() == sc[2].item(), i
        assert abs(se[0].item() - sc[0].item()) <= TOL * abs(se[0].item()), i
    assert rel_err(tc.flat_param, te.flat_param) < 1e-4


@pytest.mark.gpu
def test_resident_replay_is_bit_identical_to_host_fed_capacity_replay():
    pages = synth.make_pages(23, base_seed=17, ragged=True, k=6)
    pool = gte.PagePool(pages, DEV)
    b = 5
    perm = np.random.default_rng(9).permutation(len(pages))
    slices = [perm[i:i + b] for i in range(0, len(perm), b)]
    hbs = [batch_pages_host([pages[j] for j in s]) for s in slices]
    cap = _capacity_of(hbs[:-1], slack=(0, 0, 0))
    th, tr = gte.SageTrainer(_model(5)), gte.SageTrainer(_model(5))
    first = next(i for i, h in enumerate(hbs) if cap.fits(h["batch_num_nodes"], h["batch_num_edges"]))
    th.capture(hbs[first], capacity=cap)
    tr.capture(pool, capacity=cap)
    for x, hb in zip(tr.plan_epoch(perm, b), hbs):
        if x.fits:
            th.load_batch(hb)
            sh, sr = th.replay().clone(), tr.replay().clone()
        else:
            sh = th.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
            sr = tr.train_step(pool.batch(x.ids)).clone()
        assert torch.equal(sh, sr), x.ids
    assert torch.equal(th.flat_param, tr.flat_param)


@pytest.mark.gpu
def test_capture_eval_totals_equal_evaluate():
    hb = batch_pages_host(synth.make_pages(8, base_seed=5, ragged=True, k=6))
    tr = gte.SageTrainer(_model(11))
    ev = tr.capture_eval(hb)
    ref = tr.evaluate(gte.PageGraphBatch.from_host(hb, DEV))
    assert torch.equal(ev.replay(), ref)
    assert ref[1].item() == hb["num_nodes"]


@pytest.mark.gpu
def test_capture_predict_equals_predict_pages_and_the_autograd_argmax():
    pg = synth.make_pages(8, base_seed=13, ragged=True, k=6)
    hb = batch_pages_host(pg)
    model = _model(13)
    tr = gte.SageTrainer(model)
    g = gte.PageGraphBatch.from_host(hb, DEV)
    preds, acc = tr.predict_pages(g)
    tr.capture_predict(hb)
    tr.load_batch(hb)
    cp, cc = tr.replay()
    assert torch.equal(cp, preds)
    with torch.no_grad():
        ref = model(g, g.ndata["feat"], g.edata["feat"])
    top2 = ref.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > 1e-4 * top2[:, 0].abs().clamp_min(1.0)
    assert clear.float().mean().item() > 0.9
    assert torch.equal(preds.long()[clear], ref.argmax(1)[clear])
    sizes = torch.tensor(hb["batch_num_nodes"], dtype=torch.float64, device=DEV)
    assert torch.equal(acc, cc.to(torch.float64) / sizes)


# --------------------------------------------------------------------------------------- 7. data parallel ----
@pytest.mark.gpu
def test_data_parallel_form_on_one_gpu_equals_the_plain_step(monkeypatch):
    hb = batch_pages_host(synth.make_pages(6, ragged=True, k=6))
    t1 = gte.SageTrainer(_model(11, (13, 48, 9, 2)))
    monkeypatch.setenv("GTE_DP_FUSED", "1")
    t2 = gte.SageTrainer(_model(11, (13, 48, 9, 2)))
    t3 = gte.SageTrainer(_model(11, (13, 48, 9, 2)))
    monkeypatch.delenv("GTE_DP_FUSED")
    assert t2.dp_fused and not t1.dp_fused
    t3.capture(hb, split=True)
    for step in range(3):
        s1 = t1.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        s2 = t2.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        t3.load_batch(hb)
        s3 = t3.replay().clone()
        assert rel_err(s2, s1) < 1e-6 and torch.equal(s2, s3), step
        n = t1._flat_len
        assert rel_err(t2.flat_grad[:n] / s2[1], t1.flat_grad[:n]) < 2e-6
        assert rel_err(t2.flat_param, t1.flat_param) < 2e-6 and torch.equal(t2.flat_param, t3.flat_param)


# ------------------------------------------------------------------------------------------ 8. checkpoints ---
@pytest.mark.gpu
def test_plain_adam_checkpoint_loads_and_round_trips():
    pg = synth.make_pages(4)
    model = _model(3)
    g = gte.PageGraphBatch.from_pages(pg, DEV)
    opt = torch.optim.Adam(model.parameters(), lr=0.01, weight_decay=5e-4)
    for _ in range(2):
        opt.zero_grad()
        logits = model(g, g.ndata["feat"], g.edata["feat"])
        gte.cross_entropy(logits, g.ndata["label"]).backward()
        opt.step()
    sd = opt.state_dict()
    twin = _model(3)
    twin.load_state_dict(model.state_dict())
    tr = gte.SageTrainer(twin)
    tr.optimizer.load_state_dict(sd)
    back = tr.optimizer.state_dict()
    assert back["param_groups"][0]["lr"] == 0.01
    for i, st in sd["state"].items():
        assert float(back["state"][i]["step"]) == float(st["step"])
        for k in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(back["state"][i][k].to(st[k].device), st[k]), (i, k)
    tr.train_step(g)
    assert int(tr.step_dev.item()) == 3


# --------------------------------------------------------------------------------------------- 9. refusals ---
@pytest.mark.gpu
def test_refusals_at_construction():
    with pytest.raises(gte.GteError, match="hidden width 1025"):
        gte.SageTrainer(gte.MeanSAGE(13, 1025, 9, 1).to(DEV))

    class Other(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = torch.nn.Linear(4, 4)

    with pytest.raises(gte.GteError, match="Other is not supported"):
        gte.SageTrainer(Other().to(DEV))


# ------------------------------------------------------------------------------------------ 10. CPU spec -----
def test_model_spec_of_both_model_classes():
    drop, spec = model_spec(gte.GcnSAGE(13, 218, 9, 3, F.relu, 0))
    assert drop == 0.0
    hid = LayerSpec(agg="gcn", ln=True, relu=True, l2=False, eps=1e-5, drop_p=0.0, use_pp=False)
    assert spec == [hid, hid, LayerSpec(agg="gcn", ln=False, relu=False, l2=False, eps=1e-5, drop_p=0.0, use_pp=False)]
    drop, spec = model_spec(gte.GcnSAGE(13, 40, 9, 2, F.relu, 0.3, use_pp=True))
    assert drop == pytest.approx(0.3)
    assert [(s.drop_p, s.use_pp, s.ln, s.relu) for s in spec] == [(pytest.approx(0.3), True, True, True),
                                                                   (0.0, False, False, False)]
    for n_layers, count in ((0, 2), (1, 2), (2, 3)):
        drop, spec = model_spec(gte.MeanSAGE(13, 218, 9, n_layers))
        assert drop == 0.0 and len(spec) == count
        assert [s.l2 for s in spec] == [True] * (count - 1) + [False]
        assert all(s.agg == "mean" and not s.ln and not s.relu and s.drop_p == 0.0 and not s.use_pp for s in spec)
        assert all(s.eps == 1e-12 for s in spec)
    with pytest.raises(gte.GteError, match="hidden width 1025"):
        model_spec(gte.MeanSAGE(13, 1025, 9, 1))
    with pytest.raises(gte.GteError, match="not supported"):
        model_spec(torch.nn.Linear(2, 2))


def test_relu_l2norm_helpers_call_only_bounded_kernels():
    """the layer's ReLU + L2-normalise calls sit in layers.relu_l2norm_forward / _backward, outside the functions the
    contraction and gradient bound tests parse: every ops call there must be one whose bound is checked per element
    (gte_relu_l2norm_fwd / _bwd: test_gpu_contraction_numerics; the colsum form: this file)"""
    import ast

    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gnn_tableextraction_b200",
                           "layers.py")) as fh:
        tree = ast.parse(fh.read())
    calls = set()
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef) and fn.name in ("relu_l2norm_forward", "relu_l2norm_backward"):
            for node in ast.walk(fn):
                if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute)
                        and isinstance(node.func.value, ast.Name) and node.func.value.id == "ops"):
                    calls.add(node.func.attr)
    assert calls == {"relu_l2norm_fwd", "relu_l2norm_bwd", "relu_l2norm_bwd_colsum"}, calls
