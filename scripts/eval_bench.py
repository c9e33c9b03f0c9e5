"""The validation pass of the reference's epoch loop (model_train.py:242-249,349-370) in three forms.

Workload: one seeded validation batch of --val-pages ragged synthetic pages (config 2: GcnSAGE 13 -> 218 -> 218 -> 9,
class weights from the batch's label frequencies), resident on the device as the reference keeps it
(`dgl.batch(val_graphs).to(device)` once).  Each form ends with the validation loss, accuracy and per-class
precision / recall / F1 on the host:
  (a) captured:  ev.reset(); ev.replay(); ev.result(), one D2H of the 2 + C*C totals, metrics.precision_recall_f1;
  (b) eager:     SageTrainer.evaluate into the same totals, the same D2H and host scores;
  (c) reference: model.eval(); model(g) through the nn.Module path, F.cross_entropy(weight), argmax, a D2H of the
                 predictions and labels, sklearn precision_recall_fscore_support.
Times are CUDA events around --steps passes, each ending with its results on the host (so host work is included).

Epoch: --train-batches capacity-captured train steps over batches of --batch pages reshuffled from a ragged pool,
then the validation pass.  `eval capture` keeps one train capture and one eval capture for the whole run; `recapture`
is what a trainer offered before the eval capture: capture_predict(val) + replay + D2H of the predictions + sklearn,
then capture(train, capacity) again before the next epoch's train steps (and no validation loss at all).
Prints one JSON line; --out also writes it to a file.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import gnn_tableextraction_b200 as gte  # noqa: E402
from gnn_tableextraction_b200 import synth  # noqa: E402
from gnn_tableextraction_b200.graph import batch_pages_host  # noqa: E402

from varbatch_bench import MODEL_CFG, epoch_batches, gpu_identity  # noqa: E402


def events_ms(fn, steps, warmup):
    """ms per call of fn (which ends with its results on the host) from CUDA events around `steps` calls"""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def trainer(dev, class_w, train=True):
    torch.manual_seed(0)
    model = gte.GcnSAGE(*MODEL_CFG, F.relu, 0).to(dev)
    model.train(train)
    return gte.SageTrainer(model, lr=0.01, weight_decay=5e-4, class_weights=class_w)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--val-pages", type=int, default=512)
    ap.add_argument("--steps", type=int, default=50, help="timed validation passes per form")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=100, help="pages per train batch")
    ap.add_argument("--train-batches", type=int, default=20, help="train batches per epoch")
    ap.add_argument("--epochs", type=int, default=5, help="timed epochs per epoch form (after one warm-up epoch)")
    ap.add_argument("--pool", type=int, default=2048)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("eval_bench.py: no CUDA device -- nothing here runs on the host")
    if min(args.steps, args.warmup, args.epochs, args.train_batches) < 1:
        raise SystemExit("--steps, --warmup, --epochs and --train-batches must be >= 1")
    from sklearn.metrics import precision_recall_fscore_support

    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = gpu_identity()
    c = MODEL_CFG[2]
    val_host = batch_pages_host(synth.make_pages(args.val_pages, base_seed=777, k=10, ragged=True))
    counts = np.bincount(val_host["label"].numpy().astype(np.int64), minlength=c).astype(np.float64)
    class_w = torch.tensor(counts.sum() / (c * np.maximum(counts, 1)), dtype=torch.float32, device=dev)
    g = gte.PageGraphBatch.from_host(val_host, dev)
    labels = g.ndata["label"]
    res = {"metric": "eval_pass", "gpu": name, "power_limit_w": power, "model": list(MODEL_CFG),
           "val_pages": args.val_pages, "val_nodes": int(val_host["num_nodes"]), "val_edges": int(val_host["src"].numel())}

    # ---- one validation pass, three forms ----
    tr = trainer(dev, class_w, train=False)
    ev = tr.capture_eval(val_host)
    out = {}

    def to_host(loss, acc, cm):
        """one D2H of 2 + C*C words"""
        h = torch.cat([loss.view(1), acc.view(1), cm.view(-1).to(torch.float64)]).cpu()
        return float(h[0]), gte.precision_recall_f1(h[2:].view(c, c))

    def captured():
        ev.reset()
        ev.replay()
        out["a"] = to_host(*ev.result())

    totals = tr.eval_totals()

    def eager():
        totals.zero_()
        tr.evaluate(g, totals=totals)
        cm = totals[2:].view(c, c).to(torch.int64)
        out["b"] = to_host(totals[0] / totals[1], cm.trace().to(torch.float64) / cm.sum(), cm)

    model = tr.model

    def reference():
        model.eval()
        with torch.no_grad():
            logits = model(g)
            loss = F.cross_entropy(logits, labels.long(), weight=class_w)
            preds = logits.argmax(1)
        y, p = labels.long().cpu().numpy(), preds.cpu().numpy()
        out["c"] = (loss.item(), precision_recall_fscore_support(y, p, labels=range(c), zero_division=0))

    res["captured_ms"] = events_ms(captured, args.steps, args.warmup)
    res["eager_ms"] = events_ms(eager, args.steps, args.warmup)
    res["reference_ms"] = events_ms(reference, args.steps, args.warmup)
    res["speedup_captured_vs_reference"] = res["reference_ms"] / res["captured_ms"]
    res["speedup_captured_vs_eager"] = res["eager_ms"] / res["captured_ms"]
    res["loss"] = {k: v[0] for k, v in out.items()}
    res["f1_max_abs_diff_vs_reference"] = {k: float(np.abs(out[k][1][2] - out["c"][1][2]).max()) for k in ("a", "b")}
    res["captured_equals_eager"] = bool(out["a"][0] == out["b"][0] and all(
        np.array_equal(x, y) for x, y in zip(out["a"][1], out["b"][1])))
    del ev, tr

    # ---- one epoch: T capacity-captured train batches + validation ----
    pool = synth.make_pages(args.pool, base_seed=1234, k=10, ragged=True, distinct=256)
    rng = np.random.default_rng(0)
    epochs = []
    for _ in range(args.epochs + 1):
        idx = epoch_batches(rng, len(pool), args.batch, True)[:args.train_batches]
        epochs.append([batch_pages_host([pool[j] for j in ix], pin=True) for ix in idx])
    every = [h for e in epochs for h in e]  # the capacity holds every batch: no eager fallbacks in either form
    cap = gte.BatchCapacity(nodes=max(int(h["num_nodes"]) for h in every), edges=max(int(h["src"].numel()) for h in every),
                            pages=args.batch, page_nodes=max(p.num_nodes for p in pool),
                            page_edges=max(p.num_edges for p in pool))

    def train_batches(t, hbs):
        t.prefetch_batch(hbs[0])
        for i in range(len(hbs)):
            t.replay_prefetched()
            if i + 1 < len(hbs):
                t.prefetch_batch(hbs[i + 1])

    def epoch_ms(run_epoch):
        run_epoch(epochs[0])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for hbs in epochs[1:]:
            run_epoch(hbs)
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) / args.epochs

    ta = trainer(dev, class_w)
    ta.capture(epochs[0][0], capacity=cap)
    eva = ta.capture_eval(val_host)

    def with_eval_capture(hbs):
        train_batches(ta, hbs)
        eva.reset()
        eva.replay()
        t = eva.totals.cpu()
        gte.precision_recall_f1(t[2:].view(c, c))

    res["epoch_eval_capture_ms"] = epoch_ms(with_eval_capture)
    del eva, ta

    tb = trainer(dev, class_w)

    def recapture(hbs):
        tb.capture(hbs[0], capacity=cap)
        train_batches(tb, hbs)
        tb.capture_predict(val_host)
        preds, _ = tb.replay()
        p = preds.cpu().numpy()
        precision_recall_fscore_support(val_host["label"].numpy().astype(np.int64), p, labels=range(c), zero_division=0)

    res["epoch_recapture_ms"] = epoch_ms(recapture)
    res.update({"epoch_train_batches": args.train_batches, "batch_pages": args.batch,
                "capacity": {"nodes": cap.nodes, "edges": cap.edges, "pages": cap.pages, "N_cap": cap.shape[0]},
                "epoch_speedup_eval_capture_vs_recapture": res["epoch_recapture_ms"] / res["epoch_eval_capture_ms"]})
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
