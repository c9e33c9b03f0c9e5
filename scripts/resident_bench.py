"""Whole epochs with host batching included: the host-fed capacity loop against the resident loop over a PagePool.

The workload is the one of varbatch_bench.py: a pool of ragged synthetic pages (sizes ~ clip(N(300, 80), 40, 900),
k = 10), reshuffled every epoch into batches of B pages, the last short batch dropped (model_train.py:279-297), a
capacity at the --quantile of the batch totals, the default model, and the step statistics copied to the host after
every batch (the reference reads the loss every batch).  Per B it times whole epochs of
  (a) today's loop: batch_pages_host (the host-side dgl.batch) + prefetch_batch / replay_prefetched, the eager step
      on batches above the capacity -- the host batching of batch i+1 runs while step i is on the GPU;
  (b) the resident loop: plan_epoch once per epoch, then replay() per fitting batch, train_step(pool.batch(ids)) for
      the others (counted as eager fallbacks);
and the predict stream over the whole pool (the last batch short) fed both ways.  It also reports the device time of
gte_gather_plan and gte_gather_pages (CUDA events around replays of a CUDA graph of many launches), and the GPU's name
and power limit.
The captured-step bound of varbatch_bench.py (fixed shape at N_cap) comes from that script, run beside this one.
Prints one JSON line; --out also writes it to a file.
"""
import argparse
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gnn_tableextraction_b200 as gte  # noqa: E402
from gnn_tableextraction_b200 import ops, synth  # noqa: E402
from gnn_tableextraction_b200.engine import _plan_words  # noqa: E402
from gnn_tableextraction_b200.graph import batch_pages_host  # noqa: E402
from varbatch_bench import MODEL_CFG, fresh_trainer, gpu_identity, make_capacity  # noqa: E402


def epoch_ids(rng, num_pages, b):
    perm = rng.permutation(num_pages)
    return perm[:len(perm) // b * b]  # the train loop drops the short last batch


def timed_epochs(run_epoch, warm, work):
    """ms per batch over the epochs in `work` after running those in `warm`; host clock around work that ends in a
    device synchronise"""
    for ids in warm:
        run_epoch(ids)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    batches = sum(run_epoch(ids) for ids in work)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / batches


def graph_us(launch, k, reps=5, prepare=None):
    """device time per launch: ``k`` launches captured in one CUDA graph, the graph replayed ``reps`` times (after one
    untimed replay) between CUDA events, so the host's enqueue cost stays out of the window.  ``prepare`` runs before
    each replay, outside the timed window"""
    if prepare:
        prepare()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(k):
            launch()
    tot = 0.0
    for r in range(reps + 1):
        if prepare:
            prepare()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        if r:
            tot += e0.elapsed_time(e1) * 1e3
    return tot / (k * reps)


def gather_kernels_us(tr, pool, cap, ids):
    """device time of one gte_gather_plan and one gte_gather_pages launch on the batch ``ids`` (which fits), on the
    pass's own plan buffer and static set.  The plan kernel runs a plan of that batch repeated len(ids) times (the most
    one plan holds), uploaded again before every replay"""
    p = tr._train
    st = p.statics[0]
    k = len(ids)
    words = _plan_words(np.asarray(ids, dtype=np.int64), np.zeros(k, dtype=np.int64), k)
    plan = graph_us(lambda: ops.gather_plan(p.plan, pool.n_dev, pool.e_dev, cap, st["meta"]), k,
                    prepare=lambda: p._upload_plan(words))
    if int(p.plan[1].item()) != 0:
        raise SystemExit("resident_bench.py: the plan kernel flagged the timing plan")
    gather = graph_us(lambda: ops.gather_pages(p.plan, st["meta"], cap, pool.node_off, pool.edge_off, pool.coo[0],
                                               pool.coo[1], pool.w_coo, pool.feat, pool.label, st["src"], st["dst"],
                                               st["weight"], st["feat"], st["label"]), 100)
    n, e, f = int(st["meta"][0]), int(st["meta"][1]), pool.feat_width
    moved = 2 * (4 * n * (f + 1) + 12 * e)  # read from the pool + written to the static set
    return {"plan_kernel_us": plan, "gather_kernel_us": gather, "gather_bytes": moved,
            "gather_gb_per_s": moved / (gather * 1e-6) / 1e9}


def bench_train(pages, pool, b, args, dev, rng):
    cap = make_capacity(pages, b, args.quantile, rng)
    epochs = [epoch_ids(rng, len(pages), b) for _ in range(args.warmup + args.epochs)]
    warm, work = epochs[:args.warmup], epochs[args.warmup:]
    stats_host = torch.zeros(3, dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream()
    fallbacks = {"a": 0, "b": 0}  # over the warm-up and the timed epochs

    # (a) host batching + prefetch pipeline, as users run the capacity-captured step today
    th = fresh_trainer(dev)
    first = next(s for s in (epochs[0][i:i + b] for i in range(0, len(epochs[0]), b))
                 if cap.fits(pool.n_i[s], pool.e_i[s]))
    th.capture(batch_pages_host([pages[j] for j in first]), capacity=cap)
    slices = [e[i:i + b] for e in epochs for i in range(0, len(e), b)]
    big = max(slices, key=lambda s: int(pool.n_i[s].sum()))
    th.train_step(gte.PageGraphBatch.from_host(batch_pages_host([pages[j] for j in big]), dev))  # warm the eager route

    def host_fed(ids):
        slices = [ids[i:i + b] for i in range(0, len(ids), b)]
        hb = batch_pages_host([pages[j] for j in slices[0]])
        pending = th.fits(hb)
        if pending:
            th.prefetch_batch(hb)
        for i in range(len(slices)):
            if pending:
                st = th.replay_prefetched()
            else:
                fallbacks["a"] += 1
                st = th.train_step(gte.PageGraphBatch.from_host(hb, dev))
            if i + 1 < len(slices):
                hb = batch_pages_host([pages[j] for j in slices[i + 1]])
                pending = th.fits(hb)
                if pending:
                    th.prefetch_batch(hb)
            stats_host.copy_(st, non_blocking=True)
            stream.synchronize()
        return len(slices)

    ms_a = timed_epochs(host_fed, warm, work)
    del th

    # (b) resident: one plan upload per epoch, one replay per fitting batch
    tr = fresh_trainer(dev)
    tr.capture(pool, capacity=cap)
    tr.train_step(pool.batch(big))  # warm the eager route (the first pool.batch builds the pool's CSC / CSR)

    def resident(ids):
        plan = tr.plan_epoch(ids, b)
        for x in plan:
            if x.fits:
                st = tr.replay()
            else:
                fallbacks["b"] += 1
                st = tr.train_step(pool.batch(x.ids))
            stats_host.copy_(st, non_blocking=True)
            stream.synchronize()
        return len(plan)

    ms_b = timed_epochs(resident, warm, work)
    fit_ids = next(x.ids for x in tr.plan_epoch(epochs[0], b) if x.fits)
    kern = gather_kernels_us(tr, pool, cap, fit_ids)
    del tr
    n_cap, e_cap, p_cap = cap.shape
    return {
        "batch_pages": b, "batches_per_epoch": len(epochs[0]) // b, "epochs": args.epochs,
        "capacity": {"nodes": cap.nodes, "edges": cap.edges, "pages": cap.pages, "page_nodes": cap.page_nodes,
                     "page_edges": cap.page_edges, "N_cap": n_cap, "E_cap": e_cap, "P_cap": p_cap,
                     "quantile": args.quantile},
        "host_fed_ms": ms_a, "host_fed_graphs_per_s": b / ms_a * 1e3,
        "resident_ms": ms_b, "resident_graphs_per_s": b / ms_b * 1e3, "speedup_resident_vs_host_fed": ms_a / ms_b,
        "eager_fallbacks_per_epoch_host_fed": fallbacks["a"] / len(epochs),
        "eager_fallbacks_per_epoch_resident": fallbacks["b"] / len(epochs), **kern,
    }


def bench_predict(pages, pool, b, args, dev, rng):
    cap = make_capacity(pages, b, args.quantile, rng)
    order = rng.permutation(len(pages))  # the stream ends with a short batch
    slices = [order[i:i + b] for i in range(0, len(order), b)]
    preds_host = torch.zeros(max(cap.shape[0], max(int(pool.n_i[s].sum()) for s in slices)),
                             dtype=torch.int32).pin_memory()
    stream = torch.cuda.current_stream()
    fallbacks = {"a": 0, "b": 0}

    th = fresh_trainer(dev, train=False)
    first = next(s for s in slices if cap.fits(pool.n_i[s], pool.e_i[s]))
    th.capture_predict(batch_pages_host([pages[j] for j in first]), capacity=cap)
    big = max(slices, key=lambda s: int(pool.n_i[s].sum()))
    th.predict_pages(gte.PageGraphBatch.from_host(batch_pages_host([pages[j] for j in big]), dev))  # warm the eager route

    def host_fed(_):
        hb = batch_pages_host([pages[j] for j in slices[0]])
        pending = th.fits(hb)
        if pending:
            th.prefetch_batch(hb)
        for i in range(len(slices)):
            if pending:
                preds, _ = th.replay_prefetched()
            else:
                fallbacks["a"] += 1
                g = gte.PageGraphBatch.from_host(hb, dev)
                preds, _ = th.predict_pages(g, g.ndata["label"])
            if i + 1 < len(slices):
                hb = batch_pages_host([pages[j] for j in slices[i + 1]])
                pending = th.fits(hb)
                if pending:
                    th.prefetch_batch(hb)
            preds_host[:preds.numel()].copy_(preds, non_blocking=True)
            stream.synchronize()
        return len(slices)

    ms_a = timed_epochs(host_fed, [None] * args.warmup, [None] * args.epochs)
    del th
    tr = fresh_trainer(dev, train=False)
    tr.capture_predict(pool, capacity=cap)
    tr.predict_pages(pool.batch(big))

    def resident(_):
        plan = tr.plan_epoch(order, b)
        for x in plan:
            if x.fits:
                preds, _ = tr.replay()
            else:
                fallbacks["b"] += 1
                g = pool.batch(x.ids)
                preds, _ = tr.predict_pages(g, g.ndata["label"])
            preds_host[:preds.numel()].copy_(preds, non_blocking=True)
            stream.synchronize()
        return len(plan)

    ms_b = timed_epochs(resident, [None] * args.warmup, [None] * args.epochs)
    return {
        "batch_pages": b, "batches": len(slices), "last_batch_pages": len(slices[-1]), "N_cap": cap.shape[0],
        "host_fed_ms": ms_a, "resident_ms": ms_b, "speedup_resident_vs_host_fed": ms_a / ms_b,
        "host_fed_graphs_per_s": len(pages) / (ms_a * len(slices)) * 1e3,
        "resident_graphs_per_s": len(pages) / (ms_b * len(slices)) * 1e3,
        "eager_fallbacks_per_pass_host_fed": fallbacks["a"] / (args.warmup + args.epochs),
        "eager_fallbacks_per_pass_resident": fallbacks["b"] / (args.warmup + args.epochs),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[100, 512], help="pages per training batch")
    ap.add_argument("--pool", type=int, default=2048, help="pages in the pool (reshuffled every epoch)")
    ap.add_argument("--distinct", type=int, default=256, help="distinct synthetic pages in the pool")
    ap.add_argument("--quantile", type=float, default=0.99, help="capacity = this quantile of the batch totals")
    ap.add_argument("--epochs", type=int, default=5, help="timed epochs per loop")
    ap.add_argument("--warmup", type=int, default=1, help="untimed epochs per loop before them")
    ap.add_argument("--predict-batch", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resident_bench.py: no CUDA device -- nothing here runs on the host")
    if args.epochs < 1 or args.warmup < 1:
        raise SystemExit("--epochs and --warmup must be >= 1")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = gpu_identity()
    pages = synth.make_pages(args.pool, base_seed=1234, k=10, ragged=True, distinct=args.distinct)
    pool = gte.PagePool(pages, dev)
    rng = np.random.default_rng(0)
    res = {"metric": "resident", "gpu": name, "power_limit_w": power, "model": list(MODEL_CFG),
           "pool_pages": args.pool, "distinct_pages": args.distinct, "train": [], "predict": None}
    for b in args.batch:
        res["train"].append(bench_train(pages, pool, b, args, dev, rng))
    res["predict"] = bench_predict(pages, pool, args.predict_batch, args, dev, rng)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
