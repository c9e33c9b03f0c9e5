"""GPU tests of capacity capture: one CUDA graph trains / predicts on ragged page batches of varying size, padded on
the device by gte_pad_batch.  Padding must change nothing but the summation order of batch-wide reductions."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
from conftest import TOL, rel_err
from helpers import oracle_graph_from_pages
from gnn_tableextraction_b200 import ops, synth
from gnn_tableextraction_b200.engine import padded_page_table
from gnn_tableextraction_b200.graph import batch_pages_host
from oracle import sage_oracle as so

pytestmark = pytest.mark.gpu
DEV = "cuda"
SENT = 7


def _models(seed, cfg=(13, 218, 9, 3), dropout=0):
    torch.manual_seed(seed)
    om = so.OracleGcnSAGE(*cfg, F.relu, dropout)
    cm = gte.GcnSAGE(*cfg, F.relu, dropout)
    cm.load_state_dict(om.state_dict())
    return om, cm.to(DEV)


def _groups(sizes=(3, 5, 2, 6, 4, 1), seed=7, k=6):
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


def _padded_graph(tr, cap, hb, which=0):
    """the padded batch as the captured step saw it, read back from static input set ``which``"""
    st = tr._statics[which] if getattr(tr, "_statics", None) else tr._static
    n_cap, _, _ = cap.shape
    po, eo = padded_page_table(cap, hb["batch_num_nodes"], hb["batch_num_edges"])
    g = gte.PageGraphBatch(st["src"].clone(), st["dst"].clone(), n_cap, np.diff(po).tolist(), np.diff(eo).tolist())
    g.edata["feat"] = st["weight"].clone()
    g.ndata["feat"] = st["feat"].clone()
    g.ndata["label"] = st["label"].clone()
    return g


# ------------------------------------------------------------------------- gte_pad_batch ---------------------------
def _ref_pad(po, eo, n, e, src, dst, w, feat, label):
    src, dst, w, feat, label = src.copy(), dst.copy(), w.copy(), feat.copy(), label.copy()
    feat[n:] = 0.0
    label[n:] = -1.0
    w[e:] = 0.0
    for i in range(e, src.size):
        p = int(np.searchsorted(eo, i, side="right")) - 1
        v = po[p] + (i - eo[p]) % (po[p + 1] - po[p])
        src[i] = dst[i] = v
    return src, dst, w, feat, label


def _buffers(rng, n_cap, e_cap, f, ld):
    """device buffers with SENT sentinel elements (and ld - f sentinel columns) around the capacity region; the
    padding region holds garbage the kernel must overwrite"""
    src = torch.from_numpy(rng.integers(-5, 10 ** 6, size=e_cap + SENT).astype(np.int32))
    dst = torch.from_numpy(rng.integers(-5, 10 ** 6, size=e_cap + SENT).astype(np.int32))
    w = torch.from_numpy(rng.standard_normal(e_cap + SENT).astype(np.float32))
    feat = torch.from_numpy(rng.standard_normal((n_cap + SENT, ld)).astype(np.float32))
    label = torch.from_numpy(rng.integers(0, 9, size=n_cap + SENT).astype(np.float32))
    return [t.to(DEV) for t in (src, dst, w, feat, label)]


def _run_pad(cap, word, po, eo, bufs, f):
    n_cap, e_cap, p_cap = cap.shape
    src, dst, w, feat, label = bufs
    table = torch.from_numpy(np.concatenate([po, eo]).astype(np.int32)).to(DEV)
    wd = torch.tensor(list(word) + [0], dtype=torch.int32, device=DEV)
    bad = ops.pad_batch(wd, table[:p_cap + 1], table[p_cap + 1:], src[:e_cap], dst[:e_cap], w[:e_cap],
                        feat[:n_cap, :f], label[:n_cap])
    torch.cuda.synchronize()
    return int(bad.item())


@pytest.mark.parametrize("f,ld", [(13, 13), (64, 64), (13, 16)])
@pytest.mark.parametrize("bn,be", [
    ([100, 200, 150, 50], [800, 900, 700, 100]),  # P == pages
    ([400, 400, 200], [10, 20, 30]),  # n == nodes
    ([100, 100, 100], [3000, 3000, 2000]),  # e == edges: no padding edges
    ([7], [20]),  # one real page
    ([400, 300], [3000, 3000]),  # pages exactly at the caps
])
def test_pad_batch_matches_numpy_reference(f, ld, bn, be):
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    n_cap, e_cap, p_cap = cap.shape
    rng = np.random.default_rng(len(bn) * 1000 + f)
    bufs = _buffers(rng, n_cap, e_cap, f, ld)
    before = [b.cpu().numpy() for b in bufs]
    po, eo = padded_page_table(cap, bn, be)
    n, e = sum(bn), sum(be)
    assert _run_pad(cap, (n, e, len(bn)), po, eo, bufs, f) == 0
    after = [b.cpu().numpy() for b in bufs]
    rs, rd, rw, rf, rl = _ref_pad(po, eo, n, e, before[0][:e_cap], before[1][:e_cap], before[2][:e_cap],
                                  before[3][:n_cap, :f], before[4][:n_cap])
    assert np.array_equal(after[0][:e_cap], rs) and np.array_equal(after[1][:e_cap], rd)
    assert np.array_equal(after[2][:e_cap], rw) and np.array_equal(after[3][:n_cap, :f], rf)
    assert np.array_equal(after[4][:n_cap], rl)
    # the real prefix is untouched, padding self-loops stay inside padding pages, sentinels are untouched
    assert np.array_equal(after[0][:e], before[0][:e]) and np.array_equal(after[3][:n], before[3][:n])
    assert (rs[e:] >= n).all() and (rs[e:] < n_cap).all()
    for a, b in zip(after, before):
        assert np.array_equal(a[-SENT:], b[-SENT:])
    assert np.array_equal(after[3][:, f:], before[3][:, f:])


def test_pad_batch_flags_a_word_outside_the_capacity_and_stays_in_bounds():
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    n_cap, e_cap, p_cap = cap.shape
    po, eo = padded_page_table(cap, [300, 200], [2000, 1000])
    for word, flag in (((n_cap + 50, 3000, 2), 1), ((500, e_cap + 9, 2), 1), ((500, 3000, p_cap + 1), 1),
                       ((-3, -4, 2), 1), ((500, 3000, 2), 0)):
        rng = np.random.default_rng(5)
        bufs = _buffers(rng, n_cap, e_cap, 13, 13)
        before = [b.cpu().numpy() for b in bufs]
        got = _run_pad(cap, word, po, eo, bufs, 13)
        assert (got & 1) == flag and (flag or got == 0), (word, got)  # bit 1 may join: clamping strands padding edges
        after = [b.cpu().numpy() for b in bufs]
        for a, b in zip(after, before):
            assert np.array_equal(a[-SENT:], b[-SENT:]), word
        ids = after[0][:e_cap]
        assert ((ids[min(max(word[1], 0), e_cap):] >= 0) & (ids[min(max(word[1], 0), e_cap):] < n_cap)).all()
    # a page table that gives padding edges no padding node: flag 2, ids still inside [0, n_cap)
    bufs = _buffers(np.random.default_rng(6), n_cap, e_cap, 13, 13)
    broken = po.copy()
    broken[3:] = broken[2]  # padding pages without nodes
    assert _run_pad(cap, (500, 3000, 2), broken, eo, bufs, 13) == 2
    ids = bufs[0][:e_cap].cpu().numpy()
    assert (ids[3000:] >= 0).all() and (ids[3000:] < n_cap).all()


# ------------------------------------------------------------------------- training ---------------------------------
@pytest.mark.parametrize("pipeline", [False, True])
@pytest.mark.parametrize("split", [False, True])
def test_capacity_step_trains_like_eager_steps_on_unpadded_batches(split, pipeline, monkeypatch):
    """six ragged batches, every one of >= 1024 rows: the padded and the unpadded step take the same tensor-core
    routes and differ only in the order of batch-wide sums (shorter batches, whose unpadded step takes the FFMA
    routes, are covered bit for bit by the padded-batch test below)"""
    groups = _groups(sizes=(5, 6, 4, 7, 5, 6))
    hbs = [batch_pages_host(p) for p in groups]
    assert len({int(h["num_nodes"]) for h in hbs}) == len(hbs) and min(int(h["num_nodes"]) for h in hbs) >= 1024
    cap = _capacity_of(hbs)
    om, m1 = _models(51)
    _, m2 = _models(51)
    t1 = gte.SageTrainer(m1)
    if split:
        monkeypatch.setenv("GTE_DP_FUSED", "1")  # the data-parallel step on one GPU (un-normalised gradient + tail)
    t2 = gte.SageTrainer(m2)
    monkeypatch.delenv("GTE_DP_FUSED", raising=False)
    t2.capture(hbs[2], capacity=cap, split=split)
    # oracle step 0 under the CUDA model's ReLU patterns
    g0 = gte.PageGraphBatch.from_host(hbs[0], DEV)
    outs = []
    t1.forward(g0, keep_ctx=False, layer_outputs=outs)
    masks = [(o > 0).cpu() if layer.activation is not None else None for o, layer in zip(outs, m1.layers)]
    og = oracle_graph_from_pages(groups[0])
    torch.nn.CrossEntropyLoss()(om(og, relu_masks=masks), og.ndata["label"].long()).backward()
    if pipeline:
        t2.prefetch_batch(hbs[0])
    for i, hb in enumerate(hbs):
        assert t2.fits(hb)
        s1 = t1.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        if pipeline:
            if i + 1 < len(hbs):
                t2.prefetch_batch(hbs[i + 1])
            s2 = t2.replay_prefetched().clone()
        else:
            t2.load_batch(hb)
            s2 = t2.replay().clone()
        s1, s2 = s1.cpu(), s2.cpu()
        assert s1[1].item() == s2[1].item() == hb["num_nodes"] and s1[2].item() == s2[2].item(), i
        assert abs(s1[0].item() - s2[0].item()) <= 1e-5 * abs(s1[0].item()), i
        if i == 0:
            scale = s2[1].item() if split else 1.0
            for (k, p), (_, q) in zip(m2.named_parameters(), om.named_parameters()):
                assert rel_err(p.grad / scale, q.grad) < TOL, k
    for (k, p), (_, q) in zip(m1.named_parameters(), m2.named_parameters()):
        assert rel_err(q.data, p.data) < 1e-4, k


@pytest.mark.parametrize("cfg", [(13, 218, 9, 3), (13, 24, 9, 3)])
def test_capacity_replay_is_bit_identical_to_eager_on_the_padded_batch(cfg):
    """the padded batch is a valid batch: an eager step of a second trainer on it (read back from the static input
    set) computes exactly what the replay computed; (13, 24, ...) runs the generic gte_spmm route (16 < F <= 32)"""
    hbs = [batch_pages_host(p) for p in _groups(seed=11)]
    cap = _capacity_of(hbs)
    _, m1 = _models(61, cfg)
    _, m2 = _models(61, cfg)
    tc, te = gte.SageTrainer(m1), gte.SageTrainer(m2)
    tc.capture(hbs[0], capacity=cap)
    n_cap, _, _ = cap.shape
    for i, hb in enumerate(hbs):
        tc.load_batch(hb)
        s = tc.replay().clone()
        g = _padded_graph(tc, cap, hb)
        n = int(hb["num_nodes"])
        assert (g.ndata["label"][n:] == -1).all() and (g.ndata["feat"][n:] == 0).all()
        se = te.train_step(g).clone()
        g.check_page_structure()
        assert torch.equal(s, se), i
        assert torch.equal(tc.flat_param, te.flat_param), i
    assert n_cap == g.num_nodes()


def test_capacity_predict_on_a_ragged_stream_with_a_short_last_batch():
    groups = _groups(sizes=(5, 4, 6, 5, 2), seed=23)
    hbs = [batch_pages_host(p) for p in groups]
    cap = _capacity_of(hbs[:-1], slack=(0, 0, 0))  # the full batches define the capacity; the last one is short
    assert int(hbs[-1]["num_nodes"]) < min(int(h["num_nodes"]) for h in hbs[:-1])
    _, cm = _models(71, (13, 64, 9, 3))
    cm.eval()
    tr = gte.SageTrainer(cm)
    tr.capture_predict(hbs[0], capacity=cap)
    tr.prefetch_batch(hbs[0])
    for i, hb in enumerate(hbs):
        preds, corr = tr.replay_prefetched()
        preds, corr = preds.clone(), corr.clone()
        if i + 1 < len(hbs):
            tr.prefetch_batch(hbs[i + 1])
        assert preds.numel() == hb["num_nodes"] and corr.numel() == len(hb["batch_num_nodes"])
        g = gte.PageGraphBatch.from_host(hb, DEV)
        p2, acc = tr.predict_pages(g, g.ndata["label"])
        diff = int((preds != p2).sum().item())
        assert diff <= 2, (i, diff)  # argmax may flip only at near-ties (tensor-core vs FFMA route at small n)
        if diff == 0:
            sizes = torch.tensor(hb["batch_num_nodes"], dtype=torch.float64, device=DEV)
            assert torch.equal(corr.to(torch.float64) / sizes, acc), i


def test_capacity_capture_with_dropout_equals_eager_under_the_same_rng_state():
    hbs = [batch_pages_host(p) for p in _groups(sizes=(4, 2, 5), seed=31)]
    cap = _capacity_of(hbs)
    _, m1 = _models(81, (13, 40, 9, 3), dropout=0.3)
    _, m2 = _models(81, (13, 40, 9, 3), dropout=0.3)
    m1.train(), m2.train()
    tc = gte.SageTrainer(m1, lr=0.0, weight_decay=0.0)
    te = gte.SageTrainer(m2, lr=0.0, weight_decay=0.0)
    assert tc.has_dropout
    tc.capture(hbs[0], capacity=cap)
    losses = []
    for hb in (hbs[0], hbs[0], hbs[1], hbs[2]):
        te.rng_dev.copy_(tc.rng_dev)
        tc.load_batch(hb)
        s = tc.replay().clone()
        se = te.train_step(_padded_graph(tc, cap, hb)).clone()
        assert torch.equal(s, se)
        assert torch.equal(tc.rng_dev, te.rng_dev)
        losses.append(s[0].item())
    assert losses[0] != losses[1]  # same batch, next replay: new masks


def test_capacity_refusals_leave_the_trainer_usable():
    cap = gte.BatchCapacity(nodes=2000, edges=12600, pages=8, page_nodes=500, page_edges=3000)
    ok = [batch_pages_host(synth.make_pages(s, base_seed=40 + s, n=n, k=6)) for s, n in ((4, 300), (6, 320), (2, 450))]
    refused = [
        (synth.make_pages(9, base_seed=1, n=20, k=4), "pages=8"),
        (synth.make_pages(5, base_seed=2, n=450, k=6), "nodes=2000"),
        (synth.make_pages(4, base_seed=3, n=480, k=7), "edges=12600"),
        ([synth.make_page(4, n=600, k=4)], "page_nodes=500"),
        ([synth.make_page(5, n=450, k=7)], "page_edges=3000"),
    ]
    _, m1 = _models(91, (13, 48, 9, 3))
    _, m2 = _models(91, (13, 48, 9, 3))
    t1, t2 = gte.SageTrainer(m1), gte.SageTrainer(m2)
    t1.capture(ok[0], capacity=cap)
    t2.capture(ok[0], capacity=cap)
    t1.prefetch_batch(ok[0])
    t1.replay_prefetched()
    t2.load_batch(ok[0])
    t2.replay()
    for i, (pages, limit) in enumerate(refused):
        hb = batch_pages_host(pages)
        assert not t1.fits(hb)
        with pytest.raises(gte.GteError, match=limit):
            t1.load_batch(hb)
        with pytest.raises(gte.GteError, match=limit):
            t1.prefetch_batch(hb)
        # the route for such a batch: the eager step (both trainers, to stay in lockstep)
        s1 = t1.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        s2 = t2.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
        assert torch.equal(s1, s2)
        good = ok[(i + 1) % len(ok)]
        t1.prefetch_batch(good)
        s1 = t1.replay_prefetched().clone()
        t2.load_batch(good)
        s2 = t2.replay().clone()
        assert torch.equal(s1, s2), i
    assert torch.equal(t1.flat_param, t2.flat_param)
    with pytest.raises(gte.GteError, match="nodes=2000"):
        gte.SageTrainer(_models(92, (13, 48, 9, 3))[1]).capture(batch_pages_host(refused[1][0]), capacity=cap)


def test_capture_without_capacity_is_unchanged():
    """the default model: 28 launches per eager step, capacity capture adds exactly gte_pad_batch to each step body,
    and the fixed-shape replay stays bit-identical to the eager step"""
    lib = gte.lib()
    hb = batch_pages_host(synth.make_pages(4, n=300, k=10))
    _, m0 = _models(101)
    _, m1 = _models(101)
    _, m2 = _models(101)
    t0, t1, t2 = gte.SageTrainer(m0), gte.SageTrainer(m1), gte.SageTrainer(m2)
    c0 = lib.gte_launch_count()
    s0 = t0.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
    assert lib.gte_launch_count() - c0 == 28
    c0 = lib.gte_launch_count()
    t1.capture(hb)
    fixed = lib.gte_launch_count() - c0
    cap = gte.BatchCapacity(nodes=1200, edges=12000, pages=4, page_nodes=300, page_edges=3000)
    c0 = lib.gte_launch_count()
    t2.capture(hb, capacity=cap)
    assert lib.gte_launch_count() - c0 == fixed + 3  # two warm-up steps + the captured body
    t1.load_batch(hb)
    assert torch.equal(t1.replay(), s0)
    assert torch.equal(t1.flat_param, t0.flat_param)
