"""GPU tests of resident passes: a pass captured on a PagePool plans each batch of an epoch and gathers it from the pool
on the device (gte_gather_plan + gte_gather_pages), then pads it as a host-fed capacity pass does.  The static inputs
it builds must equal the host-fed ones bit for bit, so training, prediction and evaluation must too."""
import dataclasses

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
from gnn_tableextraction_b200 import ops, synth
from gnn_tableextraction_b200.engine import _plan_words, padded_page_table
from gnn_tableextraction_b200.graph import batch_pages_host

pytestmark = pytest.mark.gpu
DEV = "cuda"
SENT = 7


def _model(seed, cfg=(13, 218, 9, 3), dropout=0):
    torch.manual_seed(seed)
    return gte.GcnSAGE(*cfg, F.relu, dropout).to(DEV)


def _i32(a):
    return torch.as_tensor(np.asarray(a, dtype=np.int32), device=DEV)


def _capacity_for(pool, slices, refuse_largest=False):
    """a capacity every slice fits, except the one with the most nodes when ``refuse_largest``"""
    n = [int(pool.n_i[s].sum()) for s in slices]
    refuse = [int(np.argmax(n))] if refuse_largest else []
    keep = [i for i in range(len(slices)) if i not in refuse]
    cap = gte.BatchCapacity(nodes=max(n[i] for i in keep), edges=int(max(pool.e_i[s].sum() for s in slices)),
                            pages=max(len(s) for s in slices), page_nodes=int(pool.n_i.max()),
                            page_edges=int(pool.e_i.max()))
    assert [cap.fits(pool.n_i[s], pool.e_i[s]) for s in slices] == [i not in refuse for i in range(len(slices))]
    return cap, refuse


def _slices(ids, b):
    return [np.asarray(ids[i:i + b]) for i in range(0, len(ids), b)]


# ------------------------------------------------------------------------- gte_gather_plan -------------------------
def _run_plan(words, n_i, e_i, cap, meta_init):
    plan = torch.full((ops.PLAN_HEADER + 2 * len(n_i) + SENT,), -9, dtype=torch.int32, device=DEV)
    plan[:words.size] = _i32(words)
    meta = _i32(meta_init)
    n_cap, e_cap, p_cap = cap.shape
    ops.gather_plan(plan[:ops.PLAN_HEADER + 2 * len(n_i)], _i32(n_i), _i32(e_i), cap, meta[:4 + 2 * (p_cap + 1)])
    torch.cuda.synchronize()
    return plan, meta


def _expected_meta(cap, n_i, e_i, ids, start):
    po, eo = padded_page_table(cap, n_i[ids], e_i[ids])
    return [int(n_i[ids].sum()), int(e_i[ids].sum()), len(ids), start] + po.tolist() + eo.tolist()


def test_gather_plan_writes_the_padded_page_table_of_every_batch():
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    n_cap, e_cap, p_cap = cap.shape
    rng = np.random.default_rng(3)
    special = [  # (page nodes, page edges) of batches at the edges of the capacity
        ([100, 200, 150, 50], [800, 900, 700, 100]),  # P == pages
        ([400, 400, 200], [10, 20, 30]),  # n == nodes
        ([100, 100, 100], [3000, 3000, 2000]),  # e == edges
        ([7], [20]),  # one page
        ([400, 300], [3000, 3000]),  # pages at the caps
        ([1], [0]),  # one node, no edge
    ]
    n_i = np.concatenate([np.array(bn) for bn, _ in special] + [rng.integers(1, 401, size=200)]).astype(np.int64)
    e_i = np.concatenate([np.array(be) for _, be in special] + [rng.integers(0, 3001, size=200)]).astype(np.int64)
    batches, o = [], 0
    for bn, _ in special:
        batches.append(np.arange(o, o + len(bn)))
        o += len(bn)
    while len(batches) < 60:  # random batches that fit, including repeated pages
        ids = rng.integers(0, len(n_i), size=int(rng.integers(1, cap.pages + 1)))
        if cap.fits(n_i[ids], e_i[ids]):
            batches.append(ids)
    sentinel = list(range(-50, -50 + 4 + 2 * (p_cap + 1) + SENT))
    for ids in batches:
        words = _plan_words(ids.astype(np.int64), np.zeros(1, dtype=np.int64), len(ids))
        plan, meta = _run_plan(words, n_i, e_i, cap, sentinel)
        m = meta.cpu().numpy()
        assert m[:-SENT].tolist() == _expected_meta(cap, n_i, e_i, ids, 0), ids
        assert m[-SENT:].tolist() == sentinel[-SENT:]
        assert plan[:2].tolist() == [1, 0]  # cursor advanced, no flag


def test_gather_plan_cursor_walks_the_plan_and_flags_what_it_cannot_run():
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    n_cap, e_cap, p_cap = cap.shape
    rng = np.random.default_rng(4)
    n_i = rng.integers(50, 300, size=40).astype(np.int64)
    e_i = rng.integers(0, 2000, size=40).astype(np.int64)
    n_i[7] = 450  # above page_nodes: the batch holding page 7 does not fit
    ids = rng.permutation(40)[:27]
    if 7 not in ids:
        ids[5] = 7
    b = 3
    fit = [s for s in range(0, len(ids), b) if cap.fits(n_i[ids[s:s + b]], e_i[ids[s:s + b]])]
    words = _plan_words(ids.astype(np.int64), np.array(fit, dtype=np.int64), b)
    plan = torch.zeros(ops.PLAN_HEADER + 2 * len(n_i) + SENT, dtype=torch.int32, device=DEV)
    plan[:words.size] = _i32(words)
    plan[ops.PLAN_HEADER + 2 * len(n_i):] = -9
    meta = torch.full((4 + 2 * (p_cap + 1) + SENT,), -3, dtype=torch.int32, device=DEV)
    view = plan[:ops.PLAN_HEADER + 2 * len(n_i)]
    for k, s in enumerate(fit):
        ops.gather_plan(view, _i32(n_i), _i32(e_i), cap, meta[:-SENT])
        assert plan[:2].tolist() == [k + 1, 0]
        assert meta[:-SENT].tolist() == _expected_meta(cap, n_i, e_i, ids[s:s + b], s)
    before = meta.clone()
    ops.gather_plan(view, _i32(n_i), _i32(e_i), cap, meta[:-SENT])  # past the plan
    assert plan[:2].tolist() == [len(fit) + 1, 1] and torch.equal(meta, before)
    # a slice that does not fit, planned as if it did
    bad = next(s for s in range(0, len(ids), b) if s not in fit)
    words = _plan_words(ids.astype(np.int64), np.array([bad], dtype=np.int64), b)
    plan[:words.size] = _i32(words)
    ops.gather_plan(view, _i32(n_i), _i32(e_i), cap, meta[:-SENT])
    assert plan[:2].tolist() == [1, 2] and torch.equal(meta, before)
    # a page id outside the pool
    words = _plan_words(np.array([3, 40], dtype=np.int64), np.array([0], dtype=np.int64), 2)
    plan[:words.size] = _i32(words)
    ops.gather_plan(view, _i32(n_i), _i32(e_i), cap, meta[:-SENT])
    assert plan[:2].tolist() == [1, 2] and torch.equal(meta, before)
    assert (plan[-SENT:] == -9).all()


# ------------------------------------------------------------------------- gte_gather_pages + gte_pad_batch --------
def _static(rng, cap, f):
    """capacity-shaped buffers with SENT sentinel elements after them; the region itself holds garbage"""
    n_cap, e_cap, p_cap = cap.shape
    return {
        "src": torch.from_numpy(rng.integers(-5, 10 ** 6, size=e_cap + SENT).astype(np.int32)).to(DEV),
        "dst": torch.from_numpy(rng.integers(-5, 10 ** 6, size=e_cap + SENT).astype(np.int32)).to(DEV),
        "weight": torch.from_numpy(rng.standard_normal(e_cap + SENT).astype(np.float32)).to(DEV),
        "feat": torch.from_numpy(rng.standard_normal((n_cap + SENT, f)).astype(np.float32)).to(DEV),
        "label": torch.from_numpy(rng.integers(0, 9, size=n_cap + SENT).astype(np.float32)).to(DEV),
        "meta": torch.full((4 + 2 * (p_cap + 1) + SENT,), -3, dtype=torch.int32, device=DEV),
    }


def _pad(st, cap):
    n_cap, e_cap, p_cap = cap.shape
    meta = st["meta"]
    bad = ops.pad_batch(meta[:4], meta[4:5 + p_cap], meta[5 + p_cap:5 + 2 * p_cap + 1], st["src"][:e_cap],
                        st["dst"][:e_cap], st["weight"][:e_cap], st["feat"][:n_cap], st["label"][:n_cap])
    assert int(bad.item()) == 0


@pytest.mark.parametrize("f", [13, 64])
def test_gathered_batch_equals_the_host_fed_batch(f):
    rng = np.random.default_rng(f)
    pages = synth.make_pages(37, base_seed=100 + f, ragged=True, k=6)
    if f != 13:
        pages = [dataclasses.replace(p, feat=rng.standard_normal((p.num_nodes, f)).astype(np.float32)) for p in pages]
    pool = gte.PagePool(pages, DEV)
    ids = rng.permutation(37)
    b = 6
    slices = _slices(ids, b)
    cap, refused = _capacity_for(pool, slices, refuse_largest=True)
    n_cap, e_cap, p_cap = cap.shape
    words = _plan_words(ids.astype(np.int64), np.array([i * b for i in range(len(slices)) if i not in refused]), b)
    plan = torch.zeros(ops.PLAN_HEADER + 2 * pool.num_pages, dtype=torch.int32, device=DEV)
    plan[:words.size] = _i32(words)
    host = _static(np.random.default_rng(1), cap, f)
    res = _static(np.random.default_rng(1), cap, f)
    sent = {k: v[-SENT:].clone() for k, v in host.items()}
    for i, s in enumerate(slices):
        if i in refused:
            continue
        hb = batch_pages_host([pages[j] for j in s], pin=False)
        n, e = int(hb["num_nodes"]), int(hb["src"].numel())
        for k in ("src", "dst", "weight", "feat", "label"):
            host[k][:hb[k].shape[0]].copy_(hb[k])
        po, eo = padded_page_table(cap, hb["batch_num_nodes"], hb["batch_num_edges"])
        host["meta"][:-SENT] = _i32([n, e, len(s), 0] + po.tolist() + eo.tolist())
        _pad(host, cap)
        ops.gather_plan(plan, pool.n_dev, pool.e_dev, cap, res["meta"][:-SENT])
        ops.gather_pages(plan, res["meta"][:-SENT], cap, pool.node_off, pool.edge_off, pool.coo[0], pool.coo[1],
                         pool.w_coo, pool.feat, pool.label, res["src"][:e_cap], res["dst"][:e_cap],
                         res["weight"][:e_cap], res["feat"][:n_cap], res["label"][:n_cap])
        _pad(res, cap)
        for k in ("src", "dst", "weight", "feat", "label"):
            assert torch.equal(host[k], res[k]), (i, k)
        assert torch.equal(host["meta"][:3], res["meta"][:3]) and int(res["meta"][3]) == i * b
        assert torch.equal(host["meta"][4:], res["meta"][4:]), i
        for k, v in sent.items():
            assert torch.equal(res[k][-SENT:], v), k
    assert plan[1].item() == 0


# ------------------------------------------------------------------------- passes -----------------------------------
def _train_pool(seed=17, pages=23):
    return synth.make_pages(pages, base_seed=seed, ragged=True, k=6)


@pytest.mark.parametrize("dropout", [0.0, 0.3])
def test_resident_epochs_train_bit_identically_to_the_host_fed_capacity_loop(dropout):
    pages = _train_pool()
    pool = gte.PagePool(pages, DEV)
    rng = np.random.default_rng(9)
    b = 5
    epochs = [rng.permutation(len(pages)) for _ in range(2)]
    cap, _ = _capacity_for(pool, _slices(epochs[0], b), refuse_largest=True)
    cfg = (13, 218, 9, 3) if dropout == 0 else (13, 40, 9, 3)
    th = gte.SageTrainer(_model(5, cfg, dropout))
    tr = gte.SageTrainer(_model(5, cfg, dropout))
    assert tr.has_dropout == (dropout > 0)
    first = next(s for s in _slices(epochs[0], b) if cap.fits(pool.n_i[s], pool.e_i[s]))
    th.capture(batch_pages_host([pages[j] for j in first]), capacity=cap)
    tr.capture(pool, capacity=cap)
    assert torch.equal(th.flat_param, tr.flat_param) and torch.equal(th.rng_dev, tr.rng_dev)
    eager = 0
    for perm in epochs:
        plan = tr.plan_epoch(perm, b)
        assert [len(x.ids) for x in plan] == [len(s) for s in _slices(perm, b)]
        for x in plan:
            hb = batch_pages_host([pages[j] for j in x.ids])
            assert x.fits == th.fits(hb) and x.nodes == hb["num_nodes"] and x.pages == len(x.ids)
            if x.fits:
                th.load_batch(hb)
                sh = th.replay().clone()
                sr = tr.replay().clone()
            else:
                eager += 1
                sh = th.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
                sr = tr.train_step(pool.batch(x.ids)).clone()
            assert torch.equal(sh, sr), x.ids
            assert sr[1].item() == x.nodes
        with pytest.raises(gte.GteError, match="call plan_epoch"):
            tr.replay()
    assert eager >= 1
    assert torch.equal(th.flat_param, tr.flat_param)
    assert torch.equal(th.exp_avg, tr.exp_avg) and torch.equal(th.exp_avg_sq, tr.exp_avg_sq)
    assert torch.equal(th.step_dev, tr.step_dev) and torch.equal(th.rng_dev, tr.rng_dev)


def test_resident_predict_streams_the_pool_with_a_short_last_batch():
    pages = _train_pool(seed=29, pages=22)
    pool = gte.PagePool(pages, DEV)
    b = 4
    order = np.arange(len(pages))
    slices = _slices(order, b)
    assert len(slices[-1]) == 2
    cap, _ = _capacity_for(pool, slices)
    m1, m2 = _model(7, (13, 64, 9, 3)), _model(7, (13, 64, 9, 3))
    m1.eval(), m2.eval()
    th, tr = gte.SageTrainer(m1), gte.SageTrainer(m2)
    th.capture_predict(batch_pages_host([pages[j] for j in slices[0]]), capacity=cap)
    tr.capture_predict(pool, capacity=cap)
    plan = tr.plan_epoch(order, b)
    assert all(x.fits for x in plan)
    for x in plan:
        hb = batch_pages_host([pages[j] for j in x.ids])
        preds, corr = (t.clone() for t in tr.replay())
        assert preds.numel() == x.nodes and corr.numel() == x.pages
        th.load_batch(hb)
        hp, hc = th.replay()
        assert torch.equal(preds, hp) and torch.equal(corr, hc)  # the same padded batch, the same graph
        g = gte.PageGraphBatch.from_host(hb, DEV)
        p2, acc = tr.predict_pages(g, g.ndata["label"])
        diff = int((preds != p2).sum().item())
        assert diff <= 2, diff  # argmax may flip only at near-ties (tensor-core vs FFMA route at small n)
        if diff == 0:
            sizes = torch.tensor(hb["batch_num_nodes"], dtype=torch.float64, device=DEV)
            assert torch.equal(corr.to(torch.float64) / sizes, acc)


def test_resident_eval_totals_equal_the_host_fed_eval_capture():
    pages = _train_pool(seed=41, pages=19)
    pool = gte.PagePool(pages, DEV)
    b = 4
    order = np.random.default_rng(2).permutation(len(pages))
    slices = _slices(order, b)
    cap, refused = _capacity_for(pool, slices, refuse_largest=True)
    tr = gte.SageTrainer(_model(11))
    eh = tr.capture_eval(batch_pages_host([pages[j] for j in slices[0]]), capacity=cap)
    er = tr.capture_eval(pool, capacity=cap)
    for _ in range(2):  # a second epoch after reset() gives the same totals
        eh.reset(), er.reset()
        plan = er.plan_epoch(order, b)
        assert [not x.fits for x in plan] == [i in refused for i in range(len(slices))]
        for x in plan:
            hb = batch_pages_host([pages[j] for j in x.ids])
            if x.fits:
                eh.load_batch(hb)
                eh.replay()
                er.replay()
            else:
                eh.run(gte.PageGraphBatch.from_host(hb, DEV))
                er.run(pool.batch(x.ids))
        assert torch.equal(eh.totals, er.totals) and er.totals[1].item() > 0


def test_resident_step_launches_at_most_two_kernels_more_than_the_capacity_step():
    lib = gte.lib()
    pages = synth.make_pages(8, n=300, k=10)
    pool = gte.PagePool(pages, DEV)
    cap = gte.BatchCapacity(nodes=1200, edges=12000, pages=4, page_nodes=300, page_edges=3000)
    th, tr = gte.SageTrainer(_model(101)), gte.SageTrainer(_model(101))
    hb = batch_pages_host(pages[:4])
    th.capture(hb, capacity=cap)
    tr.capture(pool, capacity=cap)
    th.load_batch(hb)
    tr.plan_epoch([0, 1, 2, 3], 4)
    c0 = lib.gte_launch_count()
    th._train.run_eager(th._static)
    host_fed = lib.gte_launch_count() - c0
    c0 = lib.gte_launch_count()
    tr._train.run_eager(tr._static)
    resident = lib.gte_launch_count() - c0
    assert resident == host_fed + 2, (host_fed, resident)  # gte_gather_plan + gte_gather_pages


def test_resident_pass_refusals():
    pages = _train_pool(seed=53, pages=12)
    pool = gte.PagePool(pages, DEV)
    cap, _ = _capacity_for(pool, _slices(np.arange(12), 4))
    tr = gte.SageTrainer(_model(13))
    with pytest.raises(gte.GteError, match="needs a capacity"):
        tr.capture(pool)
    with pytest.raises(gte.GteError, match="needs a capacity"):
        tr.capture_eval(pool)
    wide = gte.PagePool([dataclasses.replace(p, feat=np.zeros((p.num_nodes, 16), np.float32)) for p in pages], DEV)
    with pytest.raises(gte.GteError, match="16 wide, the model takes 13"):
        tr.capture_predict(wide, capacity=cap)
    tr.capture(pool, capacity=cap)
    with pytest.raises(gte.GteError, match="fitting batches of the plan have run"):
        tr.replay()  # nothing planned yet
    hb = batch_pages_host(pages[:4])
    for call in (tr.load_batch, tr.prefetch_batch, tr.fits):
        with pytest.raises(gte.GteError, match="gathers its batches from a PagePool"):
            call(hb)
    with pytest.raises(gte.GteError, match="gathers its batches from a PagePool"):
        tr.replay_set(0)
    with pytest.raises(gte.GteError, match=r"\[0, 12\)"):
        tr.plan_epoch([0, 12], 4)
    with pytest.raises(gte.GteError, match="13 page ids > the pool's 12"):
        tr.plan_epoch(list(range(12)) + [0], 4)
    plan = tr.plan_epoch([3, 1, 2], 4)
    assert len(plan) == 1 and plan[0].fits
    s = tr.replay()
    assert s[1].item() == pool.n_i[[3, 1, 2]].sum()
    with pytest.raises(gte.GteError, match="all 1 fitting batches"):
        tr.replay()
    th = gte.SageTrainer(_model(13))
    th.capture(hb, capacity=cap)
    with pytest.raises(gte.GteError, match="captured on a host batch"):
        th.plan_epoch([0, 1], 2)


def test_page_pool_builds_its_sparse_formats_on_first_batch():
    pages = _train_pool(seed=61, pages=6)
    pool = gte.PagePool(pages, DEV)
    assert pool._formats is None
    g = pool.batch([4, 0, 2])
    assert pool._formats is not None
    ref = gte.PageGraphBatch.from_pages([pages[i] for i in (4, 0, 2)], DEV)
    for a, b in zip(g.csc(), ref.csc()):
        assert torch.equal(a, b)
    assert torch.equal(g.ndata["feat"], ref.ndata["feat"]) and torch.equal(g.edges()[0], ref.edges()[0])


def _host_fed_and_resident(pages, pool, cap, mode, seed=71):
    """the same pass captured on the first page (host-fed) and on the pool (resident), on identical models"""
    cfg = (13, 40, 9, 3)
    m1, m2 = _model(seed, cfg), _model(seed, cfg)
    if mode != "train":
        m1.eval(), m2.eval()
    th, tr = gte.SageTrainer(m1), gte.SageTrainer(m2)
    hb = batch_pages_host(pages[:1])
    if mode == "eval":
        return th, tr, th.capture_eval(hb, capacity=cap), tr.capture_eval(pool, capacity=cap)
    capture = "capture" if mode == "train" else "capture_predict"
    getattr(th, capture)(hb, capacity=cap)
    getattr(tr, capture)(pool, capacity=cap)
    return th, tr, th, tr


@pytest.mark.parametrize("mode", ["train", "predict", "eval"])
@pytest.mark.parametrize("pool_pages", [1, 5])
def test_resident_passes_with_one_page_warmups(mode, pool_pages):
    """a capacity of one page per batch (the page-by-page loops of the reference), and a pool of one page: the warm-up
    batch then holds one page, and one-page plans must run like the host-fed pass"""
    pages = _train_pool(seed=83, pages=pool_pages)
    pool = gte.PagePool(pages, DEV)
    cap = gte.BatchCapacity(nodes=int(pool.n_i.max()), edges=int(pool.e_i.max()), pages=1,
                            page_nodes=int(pool.n_i.max()), page_edges=int(pool.e_i.max()))
    th, tr, ph, pr = _host_fed_and_resident(pages, pool, cap, mode)
    order = np.arange(pool_pages)[::-1].copy()
    for epoch in range(2):
        plan = pr.plan_epoch(order, 1)
        assert [x.pages for x in plan] == [1] * pool_pages and all(x.fits for x in plan)
        if mode == "eval":
            ph.reset(), pr.reset()
        for x in plan:
            ph.load_batch(batch_pages_host([pages[j] for j in x.ids]))
            oh, orr = ph.replay(), pr.replay()
            if mode == "predict":
                assert torch.equal(oh[0], orr[0]) and torch.equal(oh[1], orr[1]) and orr[0].numel() == x.nodes
            else:
                assert torch.equal(oh, orr), (epoch, x.ids)
    if mode == "train":
        assert torch.equal(th.flat_param, tr.flat_param) and torch.equal(th.exp_avg_sq, tr.exp_avg_sq)


def test_capture_runs_with_the_cyclic_garbage_collector_paused():
    """a capture must not be interrupted by the cyclic collector freeing another pass's CUDA graph: it is paused while
    the graph captures and restored afterwards (warm-up runs eagerly, with the collector as it was)"""
    import gc

    from gnn_tableextraction_b200.engine import _CapturedPass

    tr = gte.SageTrainer(_model(5, (13, 40, 9, 3)))
    seen = []

    def body(g, labels):
        seen.append(gc.isenabled())
        return tr._step_impl(g, labels)

    assert gc.isenabled()
    _CapturedPass(tr.device, batch_pages_host(synth.make_pages(3, n=200, k=6)), None, body)
    assert seen == [True, True, False] and gc.isenabled()  # two warm-up runs, then the capture
    gc.disable()
    try:  # a caller that runs with the collector off keeps it off
        _CapturedPass(tr.device, batch_pages_host(synth.make_pages(3, n=200, k=6)), None, body)
        assert not gc.isenabled()
    finally:
        gc.enable()
