"""MeanSAGE(13, 218, 9, 2) (13 -> 218 -> 218 -> 9) on the config-2 batch (512 synthetic pages, 153600 nodes).

Times, with CUDA events around every pass, the L2 cache overwritten (a 256 MB write) before every pass, and the two
arms of each comparison alternating pass by pass:
  (a) step:    the captured SageTrainer step (replay of one CUDA graph: forward, loss, backward, Adam) against the
               autograd path (MeanSAGE nn.Module, gte.cross_entropy, loss.backward(), torch.optim.Adam.step()) on
               the same batch;
  (b) forward: the hidden layer's projection 218 -> 218 (two segments, [h | A_hat h]) with ReLU + L2-normalise fused
               into the tensor-core epilogue (fuse_ln = 2) against the projection followed by gte_relu_l2norm_fwd, in
               train form (z and y written) and predict form (y only; the unfused arm still writes z).
Records the card name and power limit in the same run, the launches of one step, the algorithmic bytes of (b), and
the largest difference between the fused and unfused y.  Prints one JSON line; --out also writes it to a file.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import gnn_tableextraction_b200 as gte  # noqa: E402
from gnn_tableextraction_b200 import ops, synth  # noqa: E402
from gnn_tableextraction_b200.graph import batch_pages_host  # noqa: E402

from varbatch_bench import gpu_identity  # noqa: E402

MODEL_CFG = (13, 218, 9, 2)


def alternate(arms, passes, warmup, flush):
    """{name: [ms per pass]}: every pass of every arm timed by its own pair of events after an L2 flush, arms in turn"""
    for _ in range(warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(passes):
        for k, fn in arms.items():
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1))
    return times


def summary(ts):
    a = np.asarray(ts)
    return {"median_ms": float(np.median(a)), "p10_ms": float(np.percentile(a, 10)),
            "p90_ms": float(np.percentile(a, 90)), "passes": int(a.size)}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--pages", type=int, default=512)
    ap.add_argument("--passes", type=int, default=40, help="timed passes per arm")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("meansage_bench.py: no CUDA device -- nothing here runs on the host")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = gpu_identity()
    scratch = torch.empty(64 * 1024 * 1024, dtype=torch.float32, device=dev)  # 256 MB > the 126 MB L2

    def flush():
        scratch.fill_(1.0)

    hb = batch_pages_host(synth.make_pages(args.pages))
    n = int(hb["num_nodes"])
    res = {"card": name, "power_limit_w": power, "model": "MeanSAGE(13, 218, 9, 2)", "pages": args.pages, "nodes": n,
           "method": "CUDA events per pass, L2 overwritten (256 MB) before every pass, arms alternating"}

    # ---- (a) the step
    torch.manual_seed(0)
    m_tr = gte.MeanSAGE(*MODEL_CFG).to(dev)
    m_ag = gte.MeanSAGE(*MODEL_CFG).to(dev)
    m_ag.load_state_dict(m_tr.state_dict())
    tr = gte.SageTrainer(m_tr, lr=0.01, weight_decay=5e-4)
    g = gte.PageGraphBatch.from_host(hb, dev)
    before = gte.lib().gte_launch_count()
    tr.train_step(g)
    torch.cuda.synchronize()
    res["launches_per_step"] = int(gte.lib().gte_launch_count() - before)
    tr.capture(hb)
    tr.load_batch(hb)
    opt = torch.optim.Adam(m_ag.parameters(), lr=0.01, weight_decay=5e-4)
    g_ag = gte.PageGraphBatch.from_host(hb, dev)
    h, w, labels = g_ag.ndata["feat"], g_ag.edata["feat"], g_ag.ndata["label"]

    def autograd_step():
        opt.zero_grad()
        loss = gte.cross_entropy(m_ag(g_ag, h, w), labels)
        loss.backward()
        opt.step()

    t = alternate({"captured_trainer": tr.replay, "autograd_torch_adam": autograd_step}, args.passes, args.warmup, flush)
    res["step"] = {k: summary(v) for k, v in t.items()}
    res["step"]["speedup"] = res["step"]["autograd_torch_adam"]["median_ms"] / res["step"]["captured_trainer"]["median_ms"]

    # ---- (b) the hidden layer's forward
    fin = fo = MODEL_CFG[1]
    gen = torch.Generator(device=dev).manual_seed(1)
    x1, x2 = ops.empty_padded(n, fin, dev), ops.empty_padded(n, fin, dev)
    x1.copy_(torch.randn(n, fin, device=dev, generator=gen))
    x2.copy_(torch.randn(n, fin, device=dev, generator=gen))
    W = (torch.rand(fo, 2 * fin, device=dev, generator=gen) - 0.5) * (2.0 / (2 * fin) ** 0.5)
    b = torch.randn(fo, device=dev, generator=gen) * 0.1
    pack = ops.umma_pack_weights(W, fin, 2)

    def fused(want_z):
        return ops.umma_linear_fwd(x1, x2, fin, pack, b, fo, eps=1e-12, l2=True, want_z=want_z)[1]

    def unfused():
        z = ops.umma_linear_fwd(x1, x2, fin, pack, b, fo)[0]
        return ops.relu_l2norm_fwd(z, 1e-12)

    yf, yu = fused(True), unfused()
    res["forward_max_abs_diff_fused_vs_unfused_y"] = float((yf - yu).abs().max().item())
    t = alternate({"fused_train": lambda: fused(True), "unfused_train": unfused,
                   "fused_predict": lambda: fused(False)}, args.passes, args.warmup, flush)
    mat = n * 224 * 4  # one [N, 218] fp32 matrix at ld 224
    res["forward"] = {k: summary(v) for k, v in t.items()}
    res["forward"]["bytes_per_matrix"] = mat
    res["forward"]["algorithmic_bytes"] = {
        "fused_train": 2 * mat + 2 * mat,          # read h, ah; write z, y
        "unfused_train": 2 * mat + 2 * mat + mat,  # + read z again for the normalise
        "fused_predict": 2 * mat + mat,            # read h, ah; write y
        "unfused_predict": 2 * mat + 2 * mat + mat,  # the projection still writes z, the normalise reads it
    }
    res["forward"]["unfused_over_fused_train"] = (res["forward"]["unfused_train"]["median_ms"]
                                                  / res["forward"]["fused_train"]["median_ms"])
    res["forward"]["unfused_over_fused_predict"] = (res["forward"]["unfused_train"]["median_ms"]
                                                    / res["forward"]["fused_predict"]["median_ms"])
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
