"""Captured steps on batches of varying size: what capacity capture is worth.

The workload mimics the reference loops: a pool of ragged synthetic pages (sizes ~ clip(N(300, 80), 40, 900), k = 10)
is reshuffled every epoch into batches of B pages (model_train.py:279-297), and the predict pass streams the pool in
batches of B pages ending with a short batch (model_predict.py:130-154).  The capacity is B pages at the --quantile of
the batch totals over many shuffles of the pool; a batch above it runs the eager step (SageTrainer.fits).

Reports, per B (train) and for the predict stream, ms per batch and graphs/s of
  (a) the eager step on each batch (H2D + train_step / predict_pages),
  (b) the capacity-captured step through prefetch_batch / replay_prefetched,
  (c) the fixed-shape captured step on one batch of the capacity's padded shape (the bound (b) should approach),
with the results copied to the host every batch (the reference reads the loss / predictions every batch), the mean
padding fraction (N_cap - n) / n, and the device time of gte_pad_batch (CUDA events over many launches).
Prints one JSON line; --out also writes it to a file.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import gnn_tableextraction_b200 as gte  # noqa: E402
from gnn_tableextraction_b200 import ops, synth  # noqa: E402
from gnn_tableextraction_b200.engine import padded_page_table  # noqa: E402
from gnn_tableextraction_b200.graph import batch_pages_host  # noqa: E402

MODEL_CFG = (13, 218, 9, 3)  # GcnSAGE(13, 218, 9, 3) of the reference's config


def gpu_identity():
    name = torch.cuda.get_device_name()
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        power = float(out.stdout.strip().splitlines()[0])
    except Exception:  # the number is reported without it rather than guessed
        power = None
    return name, power


def epoch_batches(rng, num_pages, b, drop_last):
    perm = rng.permutation(num_pages)
    cut = len(perm) // b * b if drop_last else len(perm)
    return [perm[i:i + b] for i in range(0, cut, b)]


def make_capacity(pool, b, quantile, rng, shuffles=400):
    pn = np.array([p.num_nodes for p in pool])
    pe = np.array([p.num_edges for p in pool])
    ns, es = [], []
    for _ in range(shuffles):
        for idx in epoch_batches(rng, len(pool), b, True):
            ns.append(int(pn[idx].sum()))
            es.append(int(pe[idx].sum()))
    return gte.BatchCapacity(nodes=int(np.ceil(np.quantile(ns, quantile))), edges=int(np.ceil(np.quantile(es, quantile))),
                             pages=b, page_nodes=int(pn.max()), page_edges=int(pe.max()))


def fresh_trainer(dev, train=True):
    torch.manual_seed(0)
    model = gte.GcnSAGE(*MODEL_CFG[:3], MODEL_CFG[3], F.relu, 0).to(dev)
    if not train:
        model.eval()
    return gte.SageTrainer(model, lr=0.01, weight_decay=5e-4)


def timed(fn, warm, work):
    """ms per item of fn over `work` after running it over `warm`; host clock around work that ends in a sync"""
    fn(warm)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn(work)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / len(work)


def padded_host_batch(tr, cap, hb):
    """the capacity-shaped padded batch of `hb`, read back from the trainer's static input set, as a host batch"""
    st = tr._static
    po, eo = padded_page_table(cap, hb["batch_num_nodes"], hb["batch_num_edges"])
    out = {k: st[k].cpu().pin_memory() for k in ("src", "dst", "weight", "feat", "label")}
    out["page_off"], out["edge_off"] = torch.from_numpy(po).pin_memory(), torch.from_numpy(eo).pin_memory()
    out["num_nodes"] = cap.shape[0]
    out["batch_num_nodes"], out["batch_num_edges"] = np.diff(po).tolist(), np.diff(eo).tolist()
    return out


def pad_kernel_us(tr, iters=500):
    st = tr._static
    args = (st["word"], st["page_off"], st["edge_off"], st["src"], st["dst"], st["weight"], st["feat"], st["label"])
    for _ in range(10):
        ops.pad_batch(*args, bad=st["pad_bad"])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        ops.pad_batch(*args, bad=st["pad_bad"])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters


def bench_train(pool, b, args, dev, rng):
    cap = make_capacity(pool, b, args.quantile, rng)
    n_cap, e_cap, p_cap = cap.shape
    need = args.warmup + args.steps
    idx = []
    while len(idx) < need:
        idx += epoch_batches(rng, len(pool), b, True)
    hbs = [batch_pages_host([pool[j] for j in ix], pin=True) for ix in idx[:need]]
    warm, work = hbs[:args.warmup], hbs[args.warmup:]
    stats_host = torch.zeros(3, dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream()

    te = fresh_trainer(dev)

    def eager(batches):
        for hb in batches:
            stats_host.copy_(te.train_step(gte.PageGraphBatch.from_host(hb, dev)), non_blocking=True)
            stream.synchronize()

    ms_a = timed(eager, warm, work)
    del te

    tc = fresh_trainer(dev)
    first = next(h for h in hbs if cap.fits(h["batch_num_nodes"], h["batch_num_edges"]))
    tc.capture(first, capacity=cap)
    big = max(hbs, key=lambda h: int(h["num_nodes"]))
    tc.train_step(gte.PageGraphBatch.from_host(big, dev))  # the eager route for batches above the capacity: warm
    fallbacks = [0]

    def captured(batches):
        pending = tc.fits(batches[0])
        if pending:
            tc.prefetch_batch(batches[0])
        for i, hb in enumerate(batches):
            if pending:
                st = tc.replay_prefetched()
            else:
                fallbacks[0] += 1
                st = tc.train_step(gte.PageGraphBatch.from_host(hb, dev))
            pending = i + 1 < len(batches) and tc.fits(batches[i + 1])
            if pending:
                tc.prefetch_batch(batches[i + 1])
            stats_host.copy_(st, non_blocking=True)
            stream.synchronize()

    ms_b = timed(captured, warm, work)
    fallback_timed = fallbacks[0]
    tc.load_batch(first)
    tc.replay()
    torch.cuda.synchronize()
    pad_us = pad_kernel_us(tc)
    hb_cap = padded_host_batch(tc, cap, first)
    del tc

    tf = fresh_trainer(dev)
    tf.capture(hb_cap)

    def fixed(batches):
        tf.prefetch_batch(hb_cap)
        for i in range(len(batches)):
            st = tf.replay_prefetched()
            if i + 1 < len(batches):
                tf.prefetch_batch(hb_cap)
            stats_host.copy_(st, non_blocking=True)
            stream.synchronize()

    ms_c = timed(fixed, warm, work)
    del tf
    ns = np.array([int(h["num_nodes"]) for h in work])
    fit = np.array([cap.fits(h["batch_num_nodes"], h["batch_num_edges"]) for h in work])
    return {
        "batch_pages": b, "capacity": {"nodes": cap.nodes, "edges": cap.edges, "pages": cap.pages,
                                       "page_nodes": cap.page_nodes, "page_edges": cap.page_edges,
                                       "N_cap": n_cap, "E_cap": e_cap, "P_cap": p_cap, "quantile": args.quantile},
        "steps": len(work), "mean_nodes": float(ns.mean()), "min_nodes": int(ns.min()), "max_nodes": int(ns.max()),
        "eager_ms": ms_a, "eager_graphs_per_s": b / ms_a * 1e3,
        "capacity_captured_ms": ms_b, "capacity_captured_graphs_per_s": b / ms_b * 1e3,
        "fixed_captured_ms_at_N_cap": ms_c, "fixed_captured_graphs_per_s": b / ms_c * 1e3,
        "speedup_capacity_vs_eager": ms_a / ms_b, "capacity_over_fixed": ms_b / ms_c,
        "padding_fraction_mean": float(((n_cap - ns[fit]) / ns[fit]).mean()) if fit.any() else None,
        "eager_fallbacks": int(fallback_timed), "pad_kernel_us": pad_us,
    }


def bench_predict(pool, b, args, dev, rng):
    cap = make_capacity(pool, b, args.quantile, rng)
    order = rng.permutation(len(pool))
    stream_idx = [order[i:i + b] for i in range(0, len(order), b)]  # the last batch is short
    hbs = [batch_pages_host([pool[j] for j in ix], pin=True) for ix in stream_idx]
    warm, work = hbs[:2], hbs
    preds_host = torch.zeros(max([cap.shape[0]] + [int(h["num_nodes"]) for h in hbs]), dtype=torch.int32).pin_memory()
    stream = torch.cuda.current_stream()

    te = fresh_trainer(dev, train=False)

    def eager(batches):
        for hb in batches:
            g = gte.PageGraphBatch.from_host(hb, dev)
            preds, _ = te.predict_pages(g, g.ndata["label"])
            preds_host[:preds.numel()].copy_(preds, non_blocking=True)
            stream.synchronize()

    ms_a = timed(eager, warm, work)
    first = next(h for h in hbs if cap.fits(h["batch_num_nodes"], h["batch_num_edges"]))
    tc = fresh_trainer(dev, train=False)
    tc.capture_predict(first, capacity=cap)
    big = max(hbs, key=lambda h: int(h["num_nodes"]))
    tc.predict_pages(gte.PageGraphBatch.from_host(big, dev))  # the eager route for batches above the capacity: warm
    fallbacks = [0]

    def captured(batches):
        pending = tc.fits(batches[0])
        if pending:
            tc.prefetch_batch(batches[0])
        for i, hb in enumerate(batches):
            if pending:
                preds, _ = tc.replay_prefetched()
            else:
                fallbacks[0] += 1
                g = gte.PageGraphBatch.from_host(hb, dev)
                preds, _ = tc.predict_pages(g, g.ndata["label"])
            pending = i + 1 < len(batches) and tc.fits(batches[i + 1])
            if pending:
                tc.prefetch_batch(batches[i + 1])
            preds_host[:preds.numel()].copy_(preds, non_blocking=True)
            stream.synchronize()

    ms_b = timed(captured, warm, work)
    fallback_timed = fallbacks[0]
    tc.load_batch(first)
    tc.replay()
    torch.cuda.synchronize()
    hb_cap = padded_host_batch(tc, cap, first)
    tf = fresh_trainer(dev, train=False)
    tf.capture_predict(hb_cap)

    def fixed(batches):
        tf.prefetch_batch(hb_cap)
        for i in range(len(batches)):
            preds, _ = tf.replay_prefetched()
            if i + 1 < len(batches):
                tf.prefetch_batch(hb_cap)
            preds_host[:preds.numel()].copy_(preds, non_blocking=True)
            stream.synchronize()

    ms_c = timed(fixed, warm, work)
    ns = np.array([int(h["num_nodes"]) for h in work])
    return {
        "batch_pages": b, "batches": len(work), "last_batch_pages": len(work[-1]["batch_num_nodes"]),
        "N_cap": cap.shape[0], "mean_nodes": float(ns.mean()),
        "eager_ms": ms_a, "capacity_captured_ms": ms_b, "fixed_captured_ms_at_N_cap": ms_c,
        "eager_graphs_per_s": len(pool) / (ms_a * len(work)) * 1e3,
        "capacity_captured_graphs_per_s": len(pool) / (ms_b * len(work)) * 1e3,
        "speedup_capacity_vs_eager": ms_a / ms_b, "eager_fallbacks": int(fallback_timed),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, nargs="+", default=[100, 512], help="pages per batch")
    ap.add_argument("--pool", type=int, default=2048, help="pages in the pool (reshuffled every epoch)")
    ap.add_argument("--distinct", type=int, default=256, help="distinct synthetic pages in the pool")
    ap.add_argument("--quantile", type=float, default=0.99, help="capacity = this quantile of the batch totals")
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--predict-batch", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("varbatch_bench.py: no CUDA device -- nothing here runs on the host")
    if args.steps < 1 or args.warmup < 1:
        raise SystemExit("--steps and --warmup must be >= 1")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = gpu_identity()
    pool = synth.make_pages(args.pool, base_seed=1234, k=10, ragged=True, distinct=args.distinct)
    rng = np.random.default_rng(0)
    res = {"metric": "varbatch", "gpu": name, "power_limit_w": power, "model": list(MODEL_CFG),
           "pool_pages": args.pool, "distinct_pages": args.distinct, "train": [], "predict": None}
    for b in args.batch:
        res["train"].append(bench_train(pool, b, args, dev, rng))
    res["predict"] = bench_predict(pool, args.predict_batch, args, dev, rng)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
