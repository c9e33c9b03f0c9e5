"""GPU tests of Adam's hyper-parameters on the device and of SageTrainer.optimizer: the *_dev kernels against their
by-value forms and torch.optim.Adam, learning-rate changes reaching every captured pass, schedules giving the same
trajectory on every route, exact resume from a checkpoint, checkpoints exchanged with the reference's optimizer, and
the refusals."""
import io
import warnings

import numpy as np
import pytest
import torch
import torch.nn.functional as F
from torch.optim.lr_scheduler import ReduceLROnPlateau, StepLR

import gnn_tableextraction_b200 as gte
from conftest import rel_err
from helpers import oracle_graph_from_pages
from gnn_tableextraction_b200 import ops, synth
from gnn_tableextraction_b200.engine import padded_page_table
from gnn_tableextraction_b200.graph import batch_pages_host
from oracle import sage_oracle as so

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _models(seed, cfg=(13, 40, 9, 3)):
    torch.manual_seed(seed)
    om = so.OracleGcnSAGE(*cfg, F.relu, 0)
    cm = gte.GcnSAGE(*cfg, F.relu, 0)
    cm.load_state_dict(om.state_dict())
    return om, cm.to(DEV)


def _model(seed, cfg=(13, 40, 9, 3)):
    return _models(seed, cfg)[1]


def _state(tr):
    return [t.clone() for t in (tr.flat_param, tr.exp_avg, tr.exp_avg_sq, tr.step_dev)]


def _assert_same_state(a, b):
    for x, y in zip(_state(a), _state(b)):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------- kernels ---------------------------------
SCHEDULES = {
    "fixed": [(0.01, 0.9, 0.999, 1e-8, 5e-4)] * 5,
    "changing": [(0.01, 0.9, 0.999, 1e-8, 5e-4), (0.005, 0.9, 0.999, 1e-8, 5e-4), (0.005, 0.8, 0.99, 1e-6, 1e-3),
                 (0.0025, 0.8, 0.99, 1e-6, 1e-3), (0.0, 0.9, 0.999, 1e-8, 0.0)],
}


@pytest.mark.parametrize("schedule", ["fixed", "changing"])
def test_adam_step_dev_is_bit_identical_to_the_by_value_entry_and_matches_torch(schedule):
    n = 10007
    p0 = torch.randn(n)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref])
    pa, pb = p0.to(DEV), p0.to(DEV)
    ma, mb, va, vb = (torch.zeros(n, device=DEV) for _ in range(4))
    sa, sb = torch.zeros(1, dtype=torch.int64, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV)
    hp = torch.zeros(5, device=DEV)
    for t, (lr, b1, b2, eps, wd) in enumerate(SCHEDULES[schedule], start=1):
        g = torch.randn(n, generator=torch.Generator().manual_seed(t))
        opt.param_groups[0].update(lr=lr, betas=(b1, b2), eps=eps, weight_decay=wd)
        ref.grad = g.clone()
        opt.step()
        gd = g.to(DEV)
        ops.adam_step(pa, gd, ma, va, lr=lr, beta1=b1, beta2=b2, eps=eps, weight_decay=wd, step_dev=sa)
        hp.copy_(torch.tensor([lr, b1, b2, eps, wd]))
        if t % 2:
            ops.adam_step(pb, gd, mb, vb, hparams=hp, step_dev=sb)
        else:  # the host step count works with device hyper-parameters too
            ops.adam_step(pb, gd, mb, vb, hparams=hp, step=t)
            sb += 1
        assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), t
        assert rel_err(pb, ref.data) < 2e-6, t
    assert sa.item() == sb.item() == 5


def test_adam_wrappers_validate_the_hyper_parameters():
    n = 64
    p, g, m, v = (torch.zeros(n, device=DEV) for _ in range(4))
    with pytest.raises(gte.GteError, match="hparams"):
        ops.adam_step(p, g, m, v, hparams=torch.zeros(4, device=DEV), step=1)
    with pytest.raises(gte.GteError, match="hparams"):
        ops.adam_step(p, g, m, v, hparams=torch.zeros(5, dtype=torch.float64, device=DEV), step=1)
    with pytest.raises(gte.GteError, match="CPU"):
        ops.adam_step(p, g, m, v, hparams=torch.zeros(5), step=1)
    with pytest.raises(gte.GteError, match="not both"):
        ops.adam_step(p, g, m, v, lr=0.01, hparams=torch.zeros(5, device=DEV), step=1)
    with pytest.raises(gte.GteError, match="required"):
        ops.adam_step(p, g, m, v, step=1)


def test_dp_allreduce_adam_dev_single_rank_is_bit_identical_to_the_by_value_entry():
    n = 4096 * 3 + 8
    gen = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=gen)
    ranks = []
    for _ in range(2):  # one world-1 setup per entry, each its own only peer
        grad = torch.zeros(n + 4, device=DEV)
        pad = torch.zeros(64, dtype=torch.int32, device=DEV)
        ranks.append(dict(p=p0.clone().to(DEV), m=torch.zeros(n, device=DEV), v=torch.zeros(n, device=DEV),
                          step=torch.zeros(1, dtype=torch.int64, device=DEV), grad=grad,
                          ptrs=torch.tensor([grad.data_ptr()], dtype=torch.int64, device=DEV), pad=pad,
                          pads=torch.tensor([pad.data_ptr()], dtype=torch.int64, device=DEV),
                          local=torch.zeros(4, dtype=torch.int32, device=DEV), stats=torch.zeros(4, device=DEV)))
    hp = torch.zeros(5, device=DEV)
    for it, (lr, b1, b2, eps, wd) in enumerate(SCHEDULES["changing"][:3]):
        g = torch.randn(n, generator=gen) * 100.0
        hp.copy_(torch.tensor([lr, b1, b2, eps, wd]))
        for r in ranks:
            r["grad"][:n] = g.to(DEV)
            r["grad"][n:n + 3] = torch.tensor([321.0, 153600.0 + it, 777.0], device=DEV)
        a, b = ranks
        ops.dp_allreduce_adam(a["ptrs"].data_ptr(), a["pads"].data_ptr(), 0, 1, n, n, a["p"], a["m"], a["v"], a["stats"],
                              lr=lr, beta1=b1, beta2=b2, eps=eps, weight_decay=wd, step_dev=a["step"],
                              local_words=a["local"])
        ops.dp_allreduce_adam(b["ptrs"].data_ptr(), b["pads"].data_ptr(), 0, 1, n, n, b["p"], b["m"], b["v"], b["stats"],
                              hparams=hp, step_dev=b["step"], local_words=b["local"])
        for k in ("p", "m", "v", "step", "stats", "local"):
            assert torch.equal(a[k], b[k]), (it, k)
    assert ranks[1]["step"].item() == 3


# ----------------------------------------------------------------- a change reaches captured replays ---------------
def _fixed_batches(count=3, n=64):
    return [batch_pages_host(synth.make_pages(4, base_seed=1 + 50 * i, n=n, k=5)) for i in range(count)]


def _zero_lr_leaves_parameters(tr, replay):
    replay()
    torch.cuda.synchronize()
    p, m = tr.flat_param.clone(), tr.exp_avg.clone()
    tr.lr = 0.0
    replay()
    assert torch.equal(tr.flat_param, p)  # with the captured learning rate the parameters would move
    assert not torch.equal(tr.exp_avg, m)  # the moments still follow the gradients
    tr.lr = 0.01
    replay()
    assert not torch.equal(tr.flat_param, p)


@pytest.mark.parametrize("split", [False, True])
def test_learning_rate_change_reaches_fixed_shape_replays(split):
    hbs = _fixed_batches(2)
    tr = gte.SageTrainer(_model(3))
    tr.capture(hbs[0], split=split)
    tr.load_batch(hbs[0])
    _zero_lr_leaves_parameters(tr, tr.replay)
    tr.prefetch_batch(hbs[1])

    def prefetched():
        tr.prefetch_batch(hbs[1])
        tr.replay_prefetched()

    _zero_lr_leaves_parameters(tr, prefetched)
    _zero_lr_leaves_parameters(tr, lambda: tr.replay_set(1))


def test_learning_rate_change_reaches_capacity_and_resident_replays():
    pages = synth.make_pages(12, base_seed=5, ragged=True, k=6)
    pool = gte.PagePool(pages, DEV)
    cap = gte.BatchCapacity(nodes=int(pool.n_i.sum()), edges=int(pool.e_i.sum()), pages=4,
                            page_nodes=int(pool.n_i.max()), page_edges=int(pool.e_i.max()))
    tc = gte.SageTrainer(_model(4))
    tc.capture(batch_pages_host(pages[:4]), capacity=cap)
    tc.load_batch(batch_pages_host(pages[4:8]))
    _zero_lr_leaves_parameters(tc, tc.replay)
    tr = gte.SageTrainer(_model(4))
    tr.capture(pool, capacity=cap)
    tr.plan_epoch(np.arange(12), 4)
    _zero_lr_leaves_parameters(tr, tr.replay)


# ----------------------------------------------------------------- schedules on every route ------------------------
PLATEAU_METRICS = [1.0, 0.9, 0.95, 0.97, 0.8, 0.99]


def _scheduler(kind, tr):
    if kind == "plateau":
        return ReduceLROnPlateau(tr.optimizer, factor=0.5, patience=0)
    return StepLR(tr.optimizer, step_size=1, gamma=0.5)


def _end_epoch(sched, epoch):
    if isinstance(sched, ReduceLROnPlateau):
        sched.step(PLATEAU_METRICS[epoch])
    else:
        sched.step()


@pytest.mark.parametrize("kind", ["plateau", "step"])
@pytest.mark.parametrize("split", [False, True])
def test_schedule_gives_eager_and_fixed_shape_replays_the_same_trajectory(kind, split):
    hbs = _fixed_batches(3)
    te, tc = gte.SageTrainer(_model(6)), gte.SageTrainer(_model(6))
    tc.capture(hbs[0], split=split)
    se, sc = _scheduler(kind, te), _scheduler(kind, tc)
    lrs = []
    with warnings.catch_warnings():
        warnings.simplefilter("error")  # no "lr_scheduler.step() before optimizer.step()"
        for epoch in range(len(PLATEAU_METRICS)):
            for hb in hbs:
                s1 = te.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
                tc.load_batch(hb)
                s2 = tc.replay().clone()
                assert torch.equal(s1, s2), epoch
            _end_epoch(se, epoch)
            _end_epoch(sc, epoch)
            assert te.lr == tc.lr
            lrs.append(tc.lr)
    assert len(set(lrs)) >= 3  # at least two reductions
    _assert_same_state(te, tc)


def _padded_graph(tr, cap, hb):
    """the padded batch the last capacity replay ran, read back from its static input set"""
    st = tr._static
    n_cap, _, _ = cap.shape
    po, eo = padded_page_table(cap, hb["batch_num_nodes"], hb["batch_num_edges"])
    g = gte.PageGraphBatch(st["src"].clone(), st["dst"].clone(), n_cap, np.diff(po).tolist(), np.diff(eo).tolist())
    g.edata["feat"] = st["weight"].clone()
    g.ndata["feat"] = st["feat"].clone()
    g.ndata["label"] = st["label"].clone()
    return g


def _pool_epochs(seed=17, b=5, epochs=4):
    """25 pages cut into the same 5 batches every epoch, visited in a new order each time; the capacity refuses the
    batch with the most nodes, so every epoch has one eager batch"""
    pages = synth.make_pages(5 * b, base_seed=seed, ragged=True, k=6)
    pool = gte.PagePool(pages, DEV)
    rng = np.random.default_rng(9)
    base = rng.permutation(len(pages))
    slices = [base[i:i + b] for i in range(0, len(pages), b)]
    perms = [np.concatenate([slices[j] for j in rng.permutation(len(slices))]) for _ in range(epochs)]
    n = [int(pool.n_i[s].sum()) for s in slices]
    assert sorted(n)[-1] > sorted(n)[-2]
    cap = gte.BatchCapacity(nodes=sorted(n)[-2], edges=int(max(pool.e_i[s].sum() for s in slices)), pages=b,
                            page_nodes=int(pool.n_i.max()), page_edges=int(pool.e_i.max()))
    return pages, pool, perms, cap


@pytest.mark.parametrize("kind", ["plateau", "step"])
def test_schedule_gives_host_fed_and_resident_epochs_the_same_trajectory(kind):
    pages, pool, perms, cap = _pool_epochs()
    th, tr = gte.SageTrainer(_model(5, (13, 218, 9, 3))), gte.SageTrainer(_model(5, (13, 218, 9, 3)))
    first = next(x for x in gte.engine.plan_slices(cap, pool.n_i, pool.e_i, perms[0], 5)[0] if x.fits)
    th.capture(batch_pages_host([pages[j] for j in first.ids]), capacity=cap)
    tr.capture(pool, capacity=cap)
    sh, sr = _scheduler(kind, th), _scheduler(kind, tr)
    eager = 0
    for epoch, perm in enumerate(perms):
        for x in tr.plan_epoch(perm, 5):
            hb = batch_pages_host([pages[j] for j in x.ids])
            if x.fits:
                th.load_batch(hb)
                a, b = th.replay().clone(), tr.replay().clone()
            else:
                eager += 1
                a = th.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
                b = tr.train_step(pool.batch(x.ids)).clone()
            assert torch.equal(a, b), (epoch, x.ids)
        _end_epoch(sh, epoch)
        _end_epoch(sr, epoch)
    assert eager == len(perms) and th.lr == tr.lr < 0.01 / 2
    _assert_same_state(th, tr)


@pytest.mark.parametrize("kind", ["plateau", "step"])
def test_eager_fallback_batch_takes_the_learning_rate_of_the_replays(kind):
    """every epoch has a batch above the capacity; the captured trainer's replays and its eager fallback both follow
    the schedule when they equal an eager trainer fed the same (padded) batches"""
    pages, pool, perms, cap = _pool_epochs(seed=23)
    tc, te = gte.SageTrainer(_model(8, (13, 218, 9, 3))), gte.SageTrainer(_model(8, (13, 218, 9, 3)))
    first = next(x for x in gte.engine.plan_slices(cap, pool.n_i, pool.e_i, perms[0], 5)[0] if x.fits)
    tc.capture(batch_pages_host([pages[j] for j in first.ids]), capacity=cap)
    sc, se = _scheduler(kind, tc), _scheduler(kind, te)
    for epoch, perm in enumerate(perms):
        fallbacks = 0
        for s in range(0, len(perm), 5):
            hb = batch_pages_host([pages[j] for j in perm[s:s + 5]])
            if tc.fits(hb):
                tc.load_batch(hb)
                a = tc.replay().clone()
                b = te.train_step(_padded_graph(tc, cap, hb)).clone()
            else:
                fallbacks += 1
                a = tc.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
                b = te.train_step(gte.PageGraphBatch.from_host(hb, DEV)).clone()
            assert torch.equal(a, b), (epoch, s)
        assert fallbacks == 1
        _end_epoch(sc, epoch)
        _end_epoch(se, epoch)
    _assert_same_state(tc, te)


# ----------------------------------------------------------------- resume ------------------------------------------
def test_resume_from_a_checkpoint_is_exact():
    hbs = _fixed_batches(3)
    k, m = 4, 3
    ta = gte.SageTrainer(_model(9))
    ta.capture(hbs[0])
    mb = _model(9)
    tb = gte.SageTrainer(mb)
    tb.capture(hbs[0])
    for i in range(k):
        for t in (ta, tb):
            if i == k - 1:
                t.lr = 0.004  # the checkpoint carries the learning rate
            t.load_batch(hbs[i % 3])
            t.replay()
    buf = io.BytesIO()
    torch.save({"epoch": 1, "state_dict": mb.state_dict(), "optimizer": tb.optimizer.state_dict()}, buf)
    del tb, mb
    buf.seek(0)
    mc = _model(99)  # other initial parameters, overwritten by the checkpoint
    tc = gte.SageTrainer(mc)
    tc.capture(hbs[0])
    ckpt = torch.load(buf, map_location=DEV)
    mc.load_state_dict(ckpt["state_dict"])
    tc.optimizer.load_state_dict(ckpt["optimizer"])
    assert tc.lr == 0.004 and tc.step_dev.item() == k
    for i in range(k, k + m):
        for t in (ta, tc):
            t.load_batch(hbs[i % 3])
            t.replay()
        assert torch.equal(ta.step_stats(), tc.step_stats()), i
    _assert_same_state(ta, tc)


# ----------------------------------------------------------------- interchange with the reference ------------------
def _oracle_setup():
    pages = synth.make_pages(6, n=80, k=6)
    cw = torch.tensor([1.0] * 6 + [2.0] + [1.0] * 2)
    return pages, oracle_graph_from_pages(pages), gte.PageGraphBatch.from_pages(pages, DEV), cw


def _roundtrip(obj, map_location):
    buf = io.BytesIO()
    torch.save(obj, buf)
    buf.seek(0)
    return torch.load(buf, map_location=map_location)


def test_reference_checkpoint_resumes_in_the_trainer():
    _, og, g, cw = _oracle_setup()
    om, _ = _models(3, (13, 48, 9, 3))
    opt = so.make_optimizer(om, lr=0.01, weight_decay=5e-4)
    for _ in range(2):
        so.train_step(om, og, og.ndata["label"], opt, class_weights=cw)
    ckpt = _roundtrip({"state_dict": om.state_dict(), "optimizer": opt.state_dict()}, None)
    _, cm = _models(77, (13, 48, 9, 3))
    tr = gte.SageTrainer(cm, class_weights=cw.to(DEV))
    cm.load_state_dict(ckpt["state_dict"])
    tr.optimizer.load_state_dict(ckpt["optimizer"])
    assert tr.step_dev.item() == 2
    for _ in range(2):
        so.train_step(om, og, og.ndata["label"], opt, class_weights=cw)
        tr.train_step(g)
    for (k, p), (_, q) in zip(cm.named_parameters(), om.named_parameters()):
        assert rel_err(p.data, q.data) < 1e-4, k


def test_trainer_checkpoint_resumes_in_the_reference_optimizer():
    _, og, g, cw = _oracle_setup()
    om, cm = _models(3, (13, 48, 9, 3))
    tr = gte.SageTrainer(cm, class_weights=cw.to(DEV))
    for _ in range(2):
        tr.train_step(g)
    ckpt = _roundtrip({"state_dict": cm.state_dict(), "optimizer": tr.optimizer.state_dict()}, "cpu")
    om.load_state_dict(ckpt["state_dict"])
    opt = so.make_optimizer(om, lr=0.5, weight_decay=0.0)  # the checkpoint's param group replaces these
    opt.load_state_dict(ckpt["optimizer"])
    assert opt.param_groups[0]["lr"] == 0.01 and opt.state_dict()["state"][0]["step"].item() == 2
    for _ in range(2):
        so.train_step(om, og, og.ndata["label"], opt, class_weights=cw)
        tr.train_step(g)
    for (k, p), (_, q) in zip(cm.named_parameters(), om.named_parameters()):
        assert rel_err(p.data, q.data) < 1e-4, k


def test_trainer_state_dict_structure_equals_a_plain_adam_after_one_step():
    _, og, g, cw = _oracle_setup()
    om, cm = _models(3, (13, 48, 9, 3))
    opt = so.make_optimizer(om)
    so.train_step(om, og, og.ndata["label"], opt, class_weights=cw)
    tr = gte.SageTrainer(cm, class_weights=cw.to(DEV))
    assert tr.optimizer.state_dict()["state"] == {}
    tr.train_step(g)
    ref, got = opt.state_dict(), tr.optimizer.state_dict()
    assert got.keys() == ref.keys() and got["param_groups"] == ref["param_groups"]
    assert got["state"].keys() == ref["state"].keys()
    for k, st in got["state"].items():
        assert list(st.keys()) == list(ref["state"][k].keys())
        assert st["step"].dtype == ref["state"][k]["step"].dtype and st["step"].device == ref["state"][k]["step"].device
        assert st["step"].item() == 1 and st["exp_avg"].shape == ref["state"][k]["exp_avg"].shape
        assert rel_err(st["exp_avg"], ref["state"][k]["exp_avg"]) < 1e-4


# ----------------------------------------------------------------- refusals ----------------------------------------
def test_refusals_raise_before_any_launch():
    lib = gte.lib()
    hb = _fixed_batches(1)[0]
    cm = _model(12)
    tr = gte.SageTrainer(cm)
    tr.capture(hb)
    tr.load_batch(hb)
    g = gte.PageGraphBatch.from_host(hb, DEV)
    tr.train_step(g)
    torch.cuda.synchronize()
    state = _state(tr)
    group = dict(tr.optimizer.param_groups[0])

    def refused(call, match=None):
        c0 = lib.gte_launch_count()
        with pytest.raises(gte.GteError, match=match):
            call()
        assert lib.gte_launch_count() == c0
        torch.cuda.synchronize()
        for a, b in zip(_state(tr), state):
            assert torch.equal(a, b)

    refused(tr.optimizer.step)
    refused(tr.optimizer.zero_grad)
    refused(lambda: tr.optimizer.zero_grad(set_to_none=False))
    assert all(p.grad is not None for p in cm.parameters())
    refused(lambda: tr.optimizer.add_param_group({"params": [torch.zeros(4, device=DEV, requires_grad=True)]}),
            "one param group")
    for change, match in (({"amsgrad": True}, "amsgrad"), ({"maximize": True}, "maximize"),
                          ({"decoupled_weight_decay": True}, "decoupled_weight_decay"),
                          ({"lr": torch.tensor(0.01)}, "tensor"), ({"lr": -0.1}, "learning rate")):
        tr.optimizer.param_groups[0].update(change)
        for call in (lambda: tr.train_step(g), tr.replay, lambda: tr.capture(hb)):
            refused(call, match)
        tr.optimizer.param_groups[0].update(group)
    tr.optimizer.param_groups.append(dict(group, params=[]))
    refused(lambda: tr.train_step(g), "one param group")
    tr.optimizer.param_groups.pop()
    # loaded state dicts that do not match the model
    good = tr.optimizer.state_dict()
    bad = []
    sd = _roundtrip(good, None)
    sd["param_groups"][0]["amsgrad"] = True
    bad.append((sd, "amsgrad"))
    sd = _roundtrip(good, None)
    sd["param_groups"][0]["params"].pop()
    bad.append((sd, "parameters, the model has"))
    sd = _roundtrip(good, None)
    sd["state"][0]["exp_avg"] = sd["state"][0]["exp_avg"][:1]
    bad.append((sd, "shape"))
    sd = _roundtrip(good, None)
    sd["state"][3]["step"] = torch.tensor(7.0)
    bad.append((sd, "different step counts"))
    for sd, match in bad:
        refused(lambda: tr.optimizer.load_state_dict(sd), match)
    assert tr.optimizer.param_groups[0]["lr"] == group["lr"]
    # a change of the hyper-parameters while a graph is being captured
    tr.lr = 0.02
    graph = torch.cuda.CUDAGraph()
    c0 = lib.gte_launch_count()
    with pytest.raises(gte.GteError, match="captured"):
        with torch.cuda.graph(graph):
            tr.train_step(g)
    assert lib.gte_launch_count() == c0
    tr.lr = group["lr"]
    tr.replay()  # still usable
    assert not torch.equal(tr.flat_param, state[0])


# ----------------------------------------------------------------- launch counts -----------------------------------
def test_launch_counts_with_device_hyper_parameters():
    lib = gte.lib()
    pages = synth.make_pages(8, n=300, k=10)
    hb = batch_pages_host(pages[:4])
    cap = gte.BatchCapacity(nodes=1200, edges=12000, pages=4, page_nodes=300, page_edges=3000)
    t0, t1, t2 = (gte.SageTrainer(_model(101, (13, 218, 9, 3))) for _ in range(3))
    t1.capture(hb, capacity=cap)
    pool = gte.PagePool(pages, DEV)
    t2.capture(pool, capacity=cap)
    t1.load_batch(hb)
    t2.plan_epoch([0, 1, 2, 3], 4)
    for t in (t0, t1, t2):
        t.lr = 0.005  # a changed learning rate costs a copy, not a launch
    counts = []
    for run in (lambda: t0.train_step(gte.PageGraphBatch.from_host(hb, DEV)), lambda: t1._train.run_eager(t1._static),
                lambda: t2._train.run_eager(t2._static)):
        t0._sync_hparams(), t1._sync_hparams(), t2._sync_hparams()
        c0 = lib.gte_launch_count()
        run()
        counts.append(lib.gte_launch_count() - c0)
    assert counts == [28, 29, 31]
    assert torch.equal(t0.hparams.cpu(), torch.tensor([0.005, 0.9, 0.999, 1e-8, 5e-4], dtype=torch.float32))


# ----------------------------------------------------------------- the INTEGRATION.md loop ---------------------------
@pytest.mark.filterwarnings("error")
def test_integration_loop_with_scheduler_validation_and_resume():
    """INTEGRATION.md section 3, short: capacity-captured train step, captured validation pass, ReduceLROnPlateau on
    the validation loss, a checkpoint every epoch, and a resume that continues exactly"""
    pages = synth.make_pages(14, base_seed=3, ragged=True, k=6)
    train, val = pages[:12], pages[12:]
    batches = [batch_pages_host(train[i:i + 4]) for i in range(0, 12, 4)]
    cap = gte.BatchCapacity(nodes=max(int(b["num_nodes"]) for b in batches) + 16,
                            edges=max(int(b["src"].numel()) for b in batches) + 64, pages=5,
                            page_nodes=max(max(b["batch_num_nodes"]) for b in batches),
                            page_edges=max(max(b["batch_num_edges"]) for b in batches))

    def setup(seed):
        model = _model(seed)
        trainer = gte.SageTrainer(model, lr=0.01, weight_decay=5e-4)
        scheduler = ReduceLROnPlateau(trainer.optimizer, mode="min", factor=0.5, patience=0)
        trainer.capture(batches[0], capacity=cap)
        ev = trainer.capture_eval(batch_pages_host(val))
        return model, trainer, scheduler, ev

    def epoch(trainer, scheduler, ev):
        for hb in batches:
            trainer.prefetch_batch(hb)
            trainer.replay_prefetched()
        ev.reset()
        ev.replay()
        loss, acc, cm = ev.result()
        scheduler.step(loss.item())
        return loss.item()

    model, trainer, scheduler, ev = setup(21)
    ckpts = []
    for e in range(4):
        loss = epoch(trainer, scheduler, ev)
        buf = io.BytesIO()  # the reference's checkpoint (model_train.py:411-419), plus the plateau's counters
        torch.save({"epoch": e, "state_dict": model.state_dict(), "optimizer": trainer.optimizer.state_dict(),
                    "metrics": {"val_loss": loss}, "scheduler": scheduler.state_dict()}, buf)
        ckpts.append(buf)
    assert trainer.lr < 0.01
    ckpts[1].seek(0)
    ckpt = torch.load(ckpts[1], map_location=DEV, weights_only=False)
    model2, trainer2, scheduler2, ev2 = setup(22)
    model2.load_state_dict(ckpt["state_dict"])
    trainer2.optimizer.load_state_dict(ckpt["optimizer"])
    scheduler2.load_state_dict(ckpt["scheduler"])
    for _ in range(2):
        epoch(trainer2, scheduler2, ev2)
    assert trainer2.lr == trainer.lr
    _assert_same_state(trainer, trainer2)
