"""Timing of the train step's aggregation-side launches at config-2 shapes (512 pages of 300 nodes, N = 153 600,
E = 1.536 M, hidden width 218), with CUDA events, the variants alternating round by round:

  * hidden input gradient, ``layer`` order: dz W -> [d_self | d_ah], then A_hat^T d_ah + d_self
    (gte_umma_linear_bwd_data + the CSR SpMM with addend)
  * hidden input gradient, ``agg`` order:   G = A_hat^T dz, then [dz | G] W (the CSR SpMM without addend +
    gte_umma_linear_bwd_data2)
  * the three narrow packed SpMMs of the step, each alone: the 13-wide input forward, the 9-wide class-layer forward
    with addend and the 9-wide class-layer backward (column views of combined [n, 32] operands)

Every launch (pair) is timed on its own between two events, after a 256 MB write that evicts the 126 MB L2.  Run it from
two builds to compare them.  Writes one JSON object (card name and power limit included) to --out and prints it.

    python scripts/agg_order_bench.py --rounds 10 --per-round 25 --out /tmp/agg_order.json
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import gnn_tableextraction_b200 as gte  # noqa: E402
from gnn_tableextraction_b200 import layers as L, ops, synth  # noqa: E402
from gnn_tableextraction_b200.graph import batch_pages_host  # noqa: E402


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = (v.strip() for v in q.stdout.splitlines()[0].split(","))
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pages", type=int, default=512)
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--per-round", type=int, default=25, help="timed launch pairs of each variant per round")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("agg_order_bench.py needs a CUDA device")
    dev = torch.device("cuda")
    hb = batch_pages_host(synth.make_pages(args.pages, distinct=48))
    g = gte.PageGraphBatch.from_host(hb, dev)
    w = g.edata["feat"]
    g.prepare(w)
    n, fin = g.ndata["feat"].shape[0], 218
    gen = torch.Generator(device=dev).manual_seed(0)

    def mat(f):
        return ops.empty_padded(n, f, dev).copy_(torch.randn(n, f, device=dev, generator=gen))

    W = (torch.rand(fin, 2 * fin, device=dev, generator=gen) - 0.5) * 0.1
    pack = ops.umma_pack_weights(W, fin, 2)
    dz = mat(fin)

    def comb():
        return ops.comb_buffer(n, dev).copy_(torch.randn(n, 32, device=dev, generator=gen))

    xc, sp, dc = comb(), comb(), comb()
    h13, ah13 = ops.comb_views(xc, 13)
    s9, p9 = sp[:, :9], sp[:, 16:25]
    dz9, gq9 = ops.comb_views(dc, 9)

    def dh_layer():
        d_self, d_ah = ops.umma_linear_bwd_data(dz, pack, fin, 2)
        return L.aggregate_backward(g, d_ah, w, addend=d_self)

    def dh_agg():
        return ops.umma_linear_bwd_data2(dz, L.aggregate_backward(g, dz, w), pack, fin)

    variants = {"dh_layer": dh_layer, "dh_agg": dh_agg,
                "input_fwd_f13": lambda: L.aggregate_forward(g, h13, w, L.GCN, out=ah13),
                "class_fwd_f9_addend": lambda: L.aggregate_forward(g, p9, w, L.GCN, addend=s9),
                "class_bwd_f9": lambda: L.aggregate_backward(g, dz9, w, out=gq9)}
    # the two orders agree (different summation order)
    ref, new = dh_layer(), dh_agg()
    rel = ((new - ref).abs().max() / ref.abs().max()).item()
    flush = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)  # 256 MB
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.per_round)]
    times = {k: [] for k in variants}
    for fn in variants.values():  # warm-up of every shape
        fn()
    for _ in range(args.rounds):
        for k, fn in variants.items():
            for a, b in ev:
                flush.zero_()
                a.record()
                fn()
                b.record()
            torch.cuda.synchronize()
            times[k] += [a.elapsed_time(b) * 1e3 for a, b in ev]
    res = {"card": card(), "pages": args.pages, "n": n, "launches_per_variant": args.rounds * args.per_round,
           "dh_agg_vs_layer_rel_err": rel, "us": {}}
    for k, t in times.items():
        t = sorted(t)
        res["us"][k] = {"median": round(statistics.median(t), 2), "p10": round(t[len(t) // 10], 2),
                        "p90": round(t[(9 * len(t)) // 10], 2)}
    res["saved_us"] = round(res["us"]["dh_layer"]["median"] - res["us"]["dh_agg"]["median"], 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
