"""GPU tests of the validation pass: gte_eval_accumulate (weighted CE statistics + confusion matrix of torch.argmax,
added to float64 totals), SageTrainer.evaluate, and the captured evaluation pass (capture_eval) that lives beside
the captured train step without changing anything the train step reads or writes."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
from conftest import load_golden, sub
from gnn_tableextraction_b200 import ops, synth
from gnn_tableextraction_b200.engine import padded_page_table
from gnn_tableextraction_b200.graph import batch_pages_host

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _ref_totals(logits, labels, c, w=None):
    """float64 numpy reference of gte_eval_accumulate"""
    x = logits.astype(np.float64)
    y = np.trunc(labels.astype(np.float64)).astype(np.int64) if labels.dtype == np.float32 else labels.astype(np.int64)
    ok = (y >= 0) & (y < c)
    x, y = x[ok], y[ok]
    wv = np.ones(c) if w is None else w.astype(np.float64)
    t = np.zeros(2 + c * c)
    if y.size:
        m = x.max(axis=1)
        nll = m + np.log(np.exp(x - m[:, None]).sum(axis=1)) - x[np.arange(y.size), y]
        t[0] = (wv[y] * nll).sum()
        t[1] = wv[y].sum()
        nan = np.isnan(x)
        p = np.where(nan.any(axis=1), nan.argmax(axis=1), x.argmax(axis=1))  # torch.argmax: the first NaN wins
        t[2:] = np.bincount(y * c + p, minlength=c * c)
    return t


def _labels(rng, n, c, dtype):
    y = rng.integers(0, c, size=n)
    y[rng.random(n) < 0.1] = -1  # gte_pad_batch padding
    y[rng.random(n) < 0.03] = c  # out of range
    y[rng.random(n) < 0.02] = c + 7
    if dtype == torch.float32:
        return (y + np.where(y >= 0, 0.7, 0.0)).astype(np.float32)  # `.long()` truncation
    return y.astype(np.int64 if dtype == torch.int64 else np.int32)


@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("dtype", [torch.float32, torch.int32, torch.int64])
@pytest.mark.parametrize("c", [2, 9, 16, 64])
def test_eval_accumulate_matches_a_float64_reference(c, dtype, weighted):
    rng = np.random.default_rng(c * 10 + weighted)
    w = rng.uniform(0.2, 3.0, size=c).astype(np.float32) if weighted else None
    wd = None if w is None else torch.from_numpy(w).to(DEV)
    batches = []
    for n in (90001, 777):  # more rows than 296 CTAs x 256 threads; a short batch
        x = rng.standard_normal((n, c + 3)).astype(np.float32) * 3
        x[: n // 50, 1] = x[: n // 50, 0]  # exact ties: the first maximal index
        batches.append((x, _labels(rng, n, c, dtype)))
    totals = torch.zeros(2 + c * c, dtype=torch.float64, device=DEV)
    ref = np.zeros(2 + c * c)
    for x, y in batches:  # two calls accumulate; the logits are a [n, c] view of a wider matrix (ld > c)
        ops.eval_accumulate(torch.from_numpy(x).to(DEV)[:, :c], torch.from_numpy(y).to(DEV), wd, totals)
        ref += _ref_totals(x[:, :c], y, c, w)
    got = totals.cpu().numpy()
    assert np.array_equal(got[2:], ref[2:])
    assert abs(got[0] - ref[0]) <= 1e-5 * abs(ref[0]) and abs(got[1] - ref[1]) <= 1e-5 * abs(ref[1])
    # deterministic: a second run is bit-identical
    again = torch.zeros_like(totals)
    for x, y in batches:
        ops.eval_accumulate(torch.from_numpy(x).to(DEV)[:, :c], torch.from_numpy(y).to(DEV), wd, again)
    assert torch.equal(totals, again)
    # n = 0 adds nothing
    ops.eval_accumulate(torch.zeros((0, c), device=DEV), torch.zeros(0, dtype=dtype, device=DEV), wd, again)
    assert torch.equal(totals, again)


def test_eval_accumulate_nan_rows_take_the_first_nan():
    c, n = 9, 4000
    rng = np.random.default_rng(3)
    x = rng.standard_normal((n, c)).astype(np.float32)
    rows = rng.choice(n, size=40, replace=False)
    x[rows, rng.integers(0, c, size=40)] = np.nan
    x[rows[:10], c - 1] = np.nan  # two NaNs in some rows
    y = rng.integers(0, c, size=n).astype(np.int64)
    totals = ops.eval_accumulate(torch.from_numpy(x).to(DEV), torch.from_numpy(y).to(DEV), None,
                                 torch.zeros(2 + c * c, dtype=torch.float64, device=DEV)).cpu().numpy()
    ref = _ref_totals(x, y, c)
    assert np.array_equal(totals[2:], ref[2:]) and totals[1] == ref[1]
    assert np.isnan(totals[0]) and np.isnan(ref[0])
    preds, _ = ops.page_predictions(torch.from_numpy(x).to(DEV), torch.tensor([0, n], dtype=torch.int32, device=DEV), 1)
    assert np.array_equal(np.bincount(y * c + preds.cpu().numpy(), minlength=c * c), totals[2:])


def test_eval_accumulate_refuses_more_than_64_classes():
    x = torch.zeros((10, 65), device=DEV)
    y = torch.zeros(10, dtype=torch.int64, device=DEV)
    with pytest.raises(gte.GteError, match="c <= 64"):
        ops.eval_accumulate(x, y, None, torch.zeros(2 + 65 * 65, dtype=torch.float64, device=DEV))
    with pytest.raises(gte.GteError, match="totals"):
        ops.eval_accumulate(x[:, :9], y, None, torch.zeros(10, dtype=torch.float64, device=DEV))


# ------------------------------------------------------------------------- eager evaluate -------------------------------
def _page_counts(d):
    bn = [int(v) for v in d["batch_num_nodes"]]
    off = np.concatenate([[0], np.cumsum(bn)])
    page_of_edge = np.searchsorted(off, d["src"], side="right") - 1
    return bn, [int(v) for v in np.bincount(page_of_edge, minlength=len(bn))]


def _confusion(y, p, c):
    return torch.bincount(y.long() * c + p.long(), minlength=c * c).view(c, c).cpu()


def test_evaluate_matches_the_reference_on_the_golden_batch():
    skm = pytest.importorskip("sklearn.metrics")
    d = load_golden("gcnsage_default_2400")
    inf, hid, ncls, nl = (int(v) for v in d["config"])
    model = gte.GcnSAGE(inf, hid, ncls, nl, F.relu, 0)
    model.load_state_dict(sub(d, "state"))
    model = model.to(DEV)
    cw = torch.from_numpy(d["class_w"]).to(DEV)
    tr = gte.SageTrainer(model, class_weights=cw)
    bn, be = _page_counts(d)
    t = lambda a, dt: torch.as_tensor(np.asarray(a)).to(dt).to(DEV)
    g = gte.PageGraphBatch(t(d["src"], torch.int32), t(d["dst"], torch.int32), int(d["num_nodes"]), bn, be)
    g.edata["feat"], g.ndata["feat"], g.ndata["label"] = t(d["weight"], torch.float32), t(d["feat"], torch.float32), \
        t(d["label"], torch.float32)
    totals = tr.evaluate(g)
    ev_loss = (totals[0] / totals[1]).item()
    assert abs(ev_loss - float(d["loss"])) <= 1e-5 * abs(float(d["loss"]))
    cm = totals[2:].view(ncls, ncls).to(torch.int64).cpu()
    # exactly the confusion matrix of torch.argmax of the trainer's own logits
    pred = tr.predict(g).argmax(1)
    assert torch.equal(cm, _confusion(g.ndata["label"], pred, ncls))
    # sklearn on the reference's logits, rows at a near-tie aside
    ref_logits = d["logits"]
    top2 = np.sort(ref_logits, axis=1)[:, -2:]
    far = (top2[:, 1] - top2[:, 0]) >= 1e-5 * np.abs(ref_logits).max()
    y = d["label"].astype(np.int64)
    near = torch.from_numpy(~far).to(DEV)
    cm_far = cm - _confusion(g.ndata["label"][near], pred[near], ncls)
    assert np.array_equal(cm_far.numpy(), skm.confusion_matrix(y[far], ref_logits[far].argmax(1), labels=range(ncls)))
    # the accumulated form: a second batch adds
    tr.evaluate(g, totals=totals)
    assert torch.equal(totals[2:].view(ncls, ncls).to(torch.int64).cpu(), 2 * cm)


# ------------------------------------------------------------------------- captured evaluation -------------------------
def _model(seed, cfg=(13, 218, 9, 3), dropout=0):
    torch.manual_seed(seed)
    return gte.GcnSAGE(*cfg, F.relu, dropout).to(DEV)


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


def _padded_graph(st, cap, hb):
    """the padded batch as the captured pass saw it, read back from its static input set ``st``"""
    n_cap, _, _ = cap.shape
    po, eo = padded_page_table(cap, hb["batch_num_nodes"], hb["batch_num_edges"])
    g = gte.PageGraphBatch(st["src"].clone(), st["dst"].clone(), n_cap, np.diff(po).tolist(), np.diff(eo).tolist())
    g.edata["feat"] = st["weight"].clone()
    g.ndata["feat"] = st["feat"].clone()
    g.ndata["label"] = st["label"].clone()
    return g


def test_captured_eval_of_a_resident_batch_equals_eager_evaluate():
    hb = batch_pages_host(synth.make_pages(8, base_seed=5, ragged=True, k=6))
    tr = gte.SageTrainer(_model(11), class_weights=torch.linspace(0.5, 2.0, 9))
    ev = tr.capture_eval(hb)
    assert torch.equal(ev.totals, torch.zeros_like(ev.totals))  # the warm-up leaves nothing behind
    ref = tr.evaluate(gte.PageGraphBatch.from_host(hb, DEV))
    assert torch.equal(ev.replay(), ref)
    ev.replay()
    assert torch.equal(ev.totals, 2 * ref)
    ev.reset()
    ev.replay()
    loss, acc, cm = ev.result()
    assert torch.equal(ev.totals, ref) and cm.dtype == torch.int64 and cm.shape == (9, 9)
    assert cm.sum().item() == hb["num_nodes"]
    assert loss.item() == (ref[0] / ref[1]).item() and acc.item() == cm.trace().item() / hb["num_nodes"]


def test_captured_eval_with_capacity_over_a_ragged_stream():
    groups = _groups((5, 4, 6, 5, 9, 2), seed=29)
    hbs = [batch_pages_host(p) for p in groups]
    cap = _capacity_of(hbs[:4] + hbs[5:], slack=(0, 0, 0))  # the last batch is short, the 9-page one does not fit
    assert int(hbs[-1]["num_nodes"]) < min(int(h["num_nodes"]) for h in hbs[:4])
    tr = gte.SageTrainer(_model(21, (13, 64, 9, 3)))
    te = gte.SageTrainer(_model(21, (13, 64, 9, 3)))
    ev = tr.capture_eval(hbs[0], capacity=cap)
    assert not ev.fits(hbs[4]) and all(ev.fits(h) for i, h in enumerate(hbs) if i != 4)
    epoch = torch.zeros_like(ev.totals)
    for i, hb in enumerate(hbs):
        ev.reset()
        if ev.fits(hb):
            ev.load_batch(hb)
            ev.replay()
            # bit-identical to an eager evaluation of the padded batch the pass saw
            assert torch.equal(ev.totals, te.evaluate(_padded_graph(ev._pass.statics[0], cap, hb))), i
        else:
            ev.run(gte.PageGraphBatch.from_host(hb, DEV))
        epoch += ev.totals
    # one epoch into the same totals equals the sum of eager evaluations of the unpadded batches
    ev.reset()
    ref = torch.zeros_like(ev.totals)
    near = 0
    for hb in hbs:
        if ev.fits(hb):
            ev.load_batch(hb)
            ev.replay()
        else:
            ev.run(gte.PageGraphBatch.from_host(hb, DEV))
        g = gte.PageGraphBatch.from_host(hb, DEV)
        te.evaluate(g, totals=ref)
        top2 = te.predict(g).topk(2, dim=1).values
        near += int(((top2[:, 0] - top2[:, 1]) < 1e-5 * top2.abs().max()).sum().item())
    assert torch.equal(ev.totals, epoch)
    assert ev.totals[1].item() == ref[1].item() == sum(int(h["num_nodes"]) for h in hbs)
    assert abs(ev.totals[0].item() - ref[0].item()) <= 1e-5 * abs(ref[0].item())
    assert (ev.totals[2:] - ref[2:]).abs().sum().item() <= 2 * near
    # the prefetch pipeline gives the same totals
    ev2 = tr.capture_eval(hbs[0], capacity=cap)
    fit = [h for h in hbs if ev2.fits(h)]
    ev2.prefetch_batch(fit[0])
    for i in range(len(fit)):
        if i + 1 < len(fit):
            ev2.prefetch_batch(fit[i + 1])
        ev2.replay_prefetched()
    ev2.run(gte.PageGraphBatch.from_host(hbs[4], DEV))
    ev.reset()
    for hb in fit:
        ev.load_batch(hb)
        ev.replay()
    ev.run(gte.PageGraphBatch.from_host(hbs[4], DEV))
    assert torch.equal(ev2.totals, ev.totals)


def _state(tr):
    return [t.clone() for t in (tr.flat_param, tr.exp_avg, tr.exp_avg_sq, tr.step_dev, tr.rng_dev, tr.step_stats())]


@pytest.mark.parametrize("eval_first", [False, True])
def test_eval_pass_leaves_the_captured_train_step_untouched(eval_first):
    """sequence A: train replays, eval replay (+ eager evaluate), train replays; sequence B: the same train replays on
    a twin trainer without evaluation.  Optimiser state, dropout RNG and loss statistics stay bit-identical."""
    hbs = [batch_pages_host(p) for p in _groups((4, 3, 5, 4), seed=37)]
    val = batch_pages_host(synth.make_pages(6, base_seed=91, ragged=True, k=6))
    cap = _capacity_of(hbs)
    ma, mb = _model(41, (13, 40, 9, 3), dropout=0.3), _model(41, (13, 40, 9, 3), dropout=0.3)
    ma.train(), mb.train()
    ta, tb = gte.SageTrainer(ma), gte.SageTrainer(mb)
    assert ta.has_dropout
    if eval_first:
        ev = ta.capture_eval(val)
        ta.capture(hbs[0], capacity=cap)
    else:
        ta.capture(hbs[0], capacity=cap)
        ev = ta.capture_eval(val)
    tb.capture(hbs[0], capacity=cap)
    assert all(torch.equal(a, b) for a, b in zip(_state(ta), _state(tb)))
    seq = hbs + hbs[:2]
    seen = []
    for i, hb in enumerate(seq):
        for t in (ta, tb):
            t.load_batch(hb)
            t.replay()
        if i in (1, 3):
            ev.reset()
            seen.append(ev.replay().clone())
            # the eval replay sees the updated parameters
            assert torch.equal(seen[-1], ta.evaluate(gte.PageGraphBatch.from_host(val, DEV))), i
        assert all(torch.equal(a, b) for a, b in zip(_state(ta), _state(tb))), i
    assert not torch.equal(seen[0], seen[1])


def test_eval_leaves_the_flat_gradient_tail_untouched(monkeypatch):
    """the data-parallel trainer keeps its loss statistics in the tail of the all-reduced flat gradient buffer"""
    hb = batch_pages_host(synth.make_pages(4, base_seed=3, ragged=True, k=6))
    monkeypatch.setenv("GTE_DP_FUSED", "1")
    tr = gte.SageTrainer(_model(51, (13, 48, 9, 3)))
    monkeypatch.delenv("GTE_DP_FUSED", raising=False)
    assert tr.dp_fused
    g = gte.PageGraphBatch.from_host(hb, DEV)
    tr.train_step(g)
    before = (tr.flat_grad.clone(), tr.step_stats().clone())
    tr.evaluate(g)
    ev = tr.capture_eval(hb)
    ev.replay()
    torch.cuda.synchronize()
    assert torch.equal(tr.flat_grad, before[0]) and torch.equal(tr.step_stats(), before[1])
    assert ev.totals[1].item() == hb["num_nodes"]


def test_eval_capture_refuses_batches_it_cannot_run_and_copies_nothing():
    hbs = [batch_pages_host(p) for p in _groups((3, 4), seed=43)]
    cap = _capacity_of(hbs[:1], slack=(0, 0, 0))
    tr = gte.SageTrainer(_model(61, (13, 48, 9, 3)))
    ev = tr.capture_eval(hbs[0], capacity=cap)
    narrow = dict(hbs[0], feat=hbs[0]["feat"][:, :12].contiguous())
    big = hbs[1]
    assert ev.fits(hbs[0]) and not ev.fits(big) and not ev.fits(narrow)
    st = ev._pass.statics[0]
    before = {k: v.clone() for k, v in st.items()}
    for hb in (big, narrow):
        with pytest.raises(gte.GteError):
            ev.load_batch(hb)
        with pytest.raises(gte.GteError):
            ev.prefetch_batch(hb)
    torch.cuda.synchronize()
    assert all(torch.equal(st[k], v) for k, v in before.items())
    # a fixed-shape pass refuses a different feature width too
    fixed = tr.capture_eval(hbs[0])
    assert not fixed.fits(narrow)
    with pytest.raises(gte.GteError, match="features"):
        fixed.load_batch(narrow)
