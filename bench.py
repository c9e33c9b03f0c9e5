#!/usr/bin/env python
"""Headline benchmark: page-graphs/sec of the GNN train step (fwd + CE + bwd + Adam)
on synthetic PubLayNet-shaped page-graph batches, B200-native path.

    python bench.py --gpus N --steps K --warmup W            # our arm
    python bench.py --impl reference --gpus N --steps K ...  # reference CPU path (oracle port)

Workload (BASELINE.json configs[1]): repo-default GcnSAGE 13->218->218->9, fp32,
512 page graphs per GPU per step (300 nodes, directed k-NN k=10 => N=153600,
E=1536000), weak scaling over GPUs (pages are independent; one gradient
all-reduce per step).  One "step" = one pass of the hot path over one batch:
CSC/CSR build from the batched COO, 3 conv layers forward, weighted-CE,
backward, Adam.  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "page-graphs/sec (fwd+bwd train step)"
UNIT = "graphs/s"
NODES_PER_PAGE, KNN = 300, 10
MODEL_CFG = (13, 218, 9, 3)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pages", type=int, default=512, help="page graphs per GPU per step (config 2: 512)")
    ap.add_argument("--no-graph", action="store_true", help="do not replay the step from a CUDA graph")
    ap.add_argument("--cpu-pages", type=int, default=32, help="pages per step of the CPU baseline sample (config 1)")
    ap.add_argument("--ref-pages", type=int, default=0,
                    help="pages per step of --impl reference (0 = the workload's own --pages, i.e. the exact config)")
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="train: configs[1] train step (the headline); infer: configs[2] batched inference over --infer-pages")
    ap.add_argument("--global-pages", type=int, default=0,
                    help="fixed GLOBAL batch (strong scaling, configs[3]: 4096): pages per GPU = global / world")
    ap.add_argument("--infer-pages", type=int, default=100_000, help="configs[2]: page graphs of the whole inference job")
    ap.add_argument("--infer-batch", type=int, default=4096, help="configs[2]: pages per batched predict pass")
    ap.add_argument("--no-extras", action="store_true", help="skip the ragged-page and sustained-clock extras")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-op-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed train step hands its caller (loss statistics, updated parameters, "
                         "their gradients) to DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs is not None and (args.impl != "ours" or args.mode != "train"):
        ap.error("--dump-outputs applies to the train step of --impl ours")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained":
                d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0,
            "source": "fallback (B200_PROFILING.md)"}


# ------------------------------------------------------------ clocks -------
class ClockSampler:
    """Samples SM clock + throttle reasons during the timed region (pynvml, every 10 ms)."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self._stop.wait(0.01)

    def __enter__(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------ per-op profile -----
class OpTimer:
    """Wraps the tensor-level ops with CUDA events on the launching stream."""

    NAMES = ["csx_from_coo", "gather_f32", "degree_norm", "spmm", "spmm_packed", "paged_pack_edges", "build_page_formats", "gram_stream", "wide_out", "linear_fwd", "linear_bwd_data",
             "linear_bwd_weight", "layernorm_act_fwd", "layernorm_act_bwd", "cross_entropy_fwd",
             "cross_entropy_bwd", "adam_step", "umma_pack_weights", "umma_linear_fwd", "umma_linear_bwd_data", "linear_bwd_data2", "linear_bwd_weight2", "umma_linear_bwd_weight", "umma_linear_bwd_weight2", "umma_linear_fwd_stacked", "umma_linear_bwd_data2",
             "umma_linear_fwd_comb", "umma_linear_bwd_data_comb", "umma_linear_bwd_weight_comb", "umma_linear_bwd_weight2_comb",
             "comb_from", "cross_entropy_bwd_comb"]

    def __init__(self, ops, torch):
        self.ops, self.torch, self.rec, self.orig = ops, torch, [], {}

    def _key(self, name, a, kw):
        if name == "spmm":
            x = a[3]
            return (name, int(a[0].numel() - 1), int(x.shape[1]), int(a[1].numel()), kw.get("addend") is not None)
        if name == "spmm_packed":  # (indptr, packed edges, x, pages)
            return ("spmm", int(a[0].numel() - 1), int(a[2].shape[1]), int(a[1].indices.numel()), kw.get("addend") is not None)
        if name == "gram_stream":  # (P wide, Q1, Q2, ...)
            return (name, int(a[0].shape[0]), int(a[0].shape[1]), int(a[1].shape[1]) + (int(a[2].shape[1]) if a[2] is not None else 0))
        if name == "wide_out":  # (A1, A2, B1, B2, sj, sc, c, ...)
            return (name, int(a[0].shape[0]), int(a[0].shape[1]) + (int(a[1].shape[1]) if a[1] is not None else 0), int(a[6]))
        if name == "linear_fwd":
            k = a[0].shape[1] + (a[1].shape[1] if a[1] is not None else 0)
            return (name, int(a[0].shape[0]), int(k), int(a[2].shape[0]))
        if name == "linear_bwd_data":
            return (name, int(a[0].shape[0]), int(a[0].shape[1]), int(a[3]))
        if name == "umma_linear_fwd_stacked":  # (x, fin, pack, bias, fo)
            return (name, int(a[0].shape[0]), int(a[1]), 2 * int(a[4]))
        if name == "umma_linear_bwd_data2":  # (dz1, dz2, pack, fin)
            return (name, int(a[0].shape[0]), 2 * int(a[0].shape[1]), int(a[3]))
        if name == "umma_linear_bwd_weight2":
            return (name, int(a[0].shape[0]), 2 * int(a[0].shape[1]), int(a[2].shape[1]))
        if name in ("linear_bwd_weight", "umma_linear_bwd_weight"):
            k = a[1].shape[1] + (a[2].shape[1] if a[2] is not None else 0)
            return (name, int(a[0].shape[0]), int(a[0].shape[1]), int(k))
        if name in ("layernorm_act_fwd", "layernorm_act_bwd"):
            return (name, int(a[0].shape[0]), int(a[0].shape[1]))
        if name == "linear_bwd_data2":  # (dz1, col1, dz2, col2, W, k)
            return (name, int(a[0].shape[0]), 2 * int(a[0].shape[1]), int(a[5]))
        if name == "linear_bwd_weight2":  # (dz1, dz2, x, ...)
            return (name, int(a[0].shape[0]), 2 * int(a[0].shape[1]), int(a[2].shape[1]))
        if name == "umma_linear_fwd":
            return (name, int(a[0].shape[0]), int(a[2]) * (2 if a[1] is not None else 1), int(a[5]))
        if name == "umma_linear_fwd_comb":  # (xc, fin, pack, bias, fo)
            return (name, int(a[0].shape[0]), 32, int(a[4]))
        if name == "umma_linear_bwd_data_comb":  # (dc, fo, pack, fin)
            return (name, int(a[0].shape[0]), 32, int(a[3]))
        if name == "umma_linear_bwd_weight_comb":  # (dz, xc, w, ...)
            return (name, int(a[0].shape[0]), int(a[0].shape[1]), 32)
        if name == "umma_linear_bwd_weight2_comb":  # (dc, fo, x, ...)
            return (name, int(a[0].shape[0]), 32, int(a[2].shape[1]))
        if name == "umma_linear_bwd_data":
            return (name, int(a[0].shape[0]), int(a[0].shape[1]), int(a[2]) * int(a[3]))
        return (name,)

    def __enter__(self):
        for n in self.NAMES:
            f = getattr(self.ops, n)
            self.orig[n] = f

            def wrap(*a, _f=f, _n=n, **kw):
                e0 = self.torch.cuda.Event(enable_timing=True)
                e1 = self.torch.cuda.Event(enable_timing=True)
                e0.record()
                out = _f(*a, **kw)
                e1.record()
                self.rec.append((self._key(_n, a, kw), e0, e1))
                return out

            setattr(self.ops, n, wrap)
        return self

    def __exit__(self, *a):
        for n, f in self.orig.items():
            setattr(self.ops, n, f)

    def table(self, steps):
        self.torch.cuda.synchronize()
        agg = {}
        for key, e0, e1 in self.rec:
            ms = e0.elapsed_time(e1)
            t = agg.setdefault(key, [0.0, 0])
            t[0] += ms
            t[1] += 1
        return {k: (v[0] / v[1], v[1] / steps) for k, v in agg.items()}  # avg ms per launch, launches per step


def op_cost(key):
    """(algorithmic bytes, flops) per launch -- DESIGN.md section 4."""
    n = key[0]
    if n == "spmm":
        _, N, F, E, add = key
        return 8 * N * F + 8 * E + 4 * N + (4 * N * F if add else 0), 2 * E * F + N * F
    if n == "linear_fwd":
        _, N, K, Fo = key
        return 4 * N * K + 4 * N * Fo + 4 * K * Fo, 2 * N * K * Fo
    if n == "umma_linear_fwd_stacked":
        _, N, K, Fo = key
        return 4 * N * K + 4 * N * 32, 2 * N * K * Fo
    if n == "umma_linear_fwd_comb":  # reads the [n, 32] operand, writes z and y
        _, N, K, Fo = key
        return 4 * N * K + 8 * N * Fo + 4 * K * Fo, 2 * N * K * Fo
    if n in ("umma_linear_bwd_data_comb", "umma_linear_bwd_weight_comb", "umma_linear_bwd_weight2_comb"):
        _, N, a, b = key
        return 4 * N * (a + b) + 4 * a * b, 2 * N * a * b
    if n == "umma_linear_fwd":  # reads [h | ah], writes z and y
        _, N, K, Fo = key
        return 4 * N * K + 8 * N * Fo + 4 * K * Fo, 2 * N * K * Fo
    if n in ("linear_bwd_data", "umma_linear_bwd_data", "linear_bwd_data2", "linear_bwd_weight2", "umma_linear_bwd_data2"):
        _, N, Fo, K = key
        return 4 * N * Fo + 4 * N * K + 4 * K * Fo, 2 * N * K * Fo
    if n in ("linear_bwd_weight", "umma_linear_bwd_weight", "umma_linear_bwd_weight2"):
        _, N, Fo, K = key
        return 4 * N * Fo + 4 * N * K + 4 * K * Fo, 2 * N * K * Fo
    if n in ("gram_stream", "wide_out"):
        _, N, a, b = key
        return 4 * N * (a + b), 2 * N * a * b
    if n == "layernorm_act_fwd":
        return 8 * key[1] * key[2], 10 * key[1] * key[2]
    if n == "layernorm_act_bwd":
        return 12 * key[1] * key[2], 16 * key[1] * key[2]
    return 0, 0


def ncu_traffic(op_key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel behind an op, from the committed
    `ncu --set full` summary (profiles/r02_kernel_metrics.json, written by scripts/summarize_profiles.py from a
    capture of one step of this same workload).  None when no capture of that kernel at this size is on file."""
    path = os.path.join(ROOT, "profiles", "r02_kernel_metrics.json")
    if not os.path.exists(path):
        return None
    try:
        m = json.load(open(path))
    except Exception:
        return None

    def recs(prefix):
        return sorted((r for k, v in m.items() if k.startswith(prefix) for r in v), key=lambda r: -r.get("time_us", 0))

    name, want = op_key[0], None
    if name == "umma_linear_bwd_weight" and op_key[3] > 64:
        r = recs("k_umma_dw<4>") or recs("k_umma_dw grid")
        want = r[0] if r else None
    elif name == "umma_linear_fwd" and op_key[2] > 64:  # hidden layer: the longest launch of the pair kernel
        r = recs("k_umma_gemm_pair<1>")
        want = r[0] if r else None
    elif name == "umma_linear_bwd_data" and op_key[2] > 64:  # second longest (the stacked class forward is far shorter)
        r = recs("k_umma_gemm_pair<1>")
        want = r[1] if len(r) > 1 else None
    elif name == "spmm" and op_key[2] > 64:
        r = sorted(recs("k_spmm_paged_pk<8, 2"), key=lambda q: q.get("dram_bytes", 0))
        want = (r[-1] if op_key[4] else r[0]) if r else None  # with addend = the larger traffic
    return None if want is None else {"bytes": want["dram_bytes"], "capture": "profiles/r02_kernel_metrics.json: " + want["capture"]}


# ------------------------------------------------------------- CPU arm -----
def cpu_oracle_run(pages_per_step: int, steps: int, warmup: int, budget_s: float):
    """Times the oracle port (torch-only restatement of the reference's DGL CPU path:
    index_add aggregation + MKL sgemm + autograd + Adam) on the host cores."""
    import numpy as np
    import torch
    import torch.nn.functional as F

    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant to use every host core it can
    torch.set_num_threads(max(1, os.cpu_count() or 1))

    from gnn_tableextraction_b200 import synth
    from oracle import sage_oracle as so
    from oracle.csx import OracleGraph, batch_coo

    pages = synth.make_pages(pages_per_step, base_seed=42, n=NODES_PER_PAGE, k=KNN, distinct=min(pages_per_step, 32))
    src, dst, w, noff, _ = batch_coo(pages)
    g = OracleGraph(src, dst, int(noff[-1]), w, np.concatenate([p.feat for p in pages]))
    labels = torch.from_numpy(np.concatenate([p.label for p in pages]))
    torch.manual_seed(0)
    model = so.OracleGcnSAGE(*MODEL_CFG[:3], MODEL_CFG[3], F.relu, 0)
    opt = so.make_optimizer(model)
    for _ in range(warmup):
        so.train_step(model, g, labels, opt)
    times = []
    t_start = time.perf_counter()
    for _ in range(steps):
        t0 = time.perf_counter()
        so.train_step(model, g, labels, opt)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s:
            break
    total = sum(times)
    return {"value": pages_per_step * len(times) / total, "ms_per_step": 1e3 * total / len(times),
            "steps": len(times), "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(),
            "torch": torch.__version__}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref_pages = args.ref_pages if args.ref_pages > 0 else args.pages
    r = cpu_oracle_run(ref_pages, args.steps, max(args.warmup, 1), budget_s=150.0)
    sample = (f"{ref_pages} pages/step x {r['steps']} steps (the workload's batch is {args.pages} pages), fwd+CE+bwd+Adam, "
              f"oracle PORT, not DGL (DGL is not installable here: torch-only restatement of the reference CPU path -- "
              f"index_add aggregation + MKL sgemm + autograd + Adam; a DGL OpenMP SpMM would likely be faster than "
              f"index_add), torch {r['torch']}, {r['cores']} threads of {r['host_cpus']} host cpus")
    cfg = workload_config(args, 1)
    cfg["reference_arm"] = {"pages_per_step": ref_pages, "same_batch_as_workload": ref_pages == args.pages,
                            "kind": "port (torch-only restatement, not DGL)", "torch_threads": r["cores"],
                            "host_cpus": r["host_cpus"]}
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": max(args.warmup, 1), "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {
        "workload": f"configs[1]: GcnSAGE 13-218-218-9 train step, {args.pages} synthetic PubLayNet-shaped page graphs "
                    f"per GPU (300 nodes, directed kNN k=10, edge weights), fp32",
        "pages_per_gpu": args.pages, "global_pages": args.pages * world, "nodes_per_page": NODES_PER_PAGE, "knn": KNN,
        "parallelism": f"dp{world} by graph", "step": "CSC+CSR build, fwd, weighted CE, bwd, Adam",
        "l2": "working set per step > 1 GB (activations of 153600 x 218 fp32 = 134 MB each) exceeds the 126 MB L2; "
              "two (resident leg) / three (e2e leg) different input batches alternate",
    }


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(trainer, model):
    """Host copies of what a caller holds after a train step: [sum w*nll, sum w, #correct], every updated parameter and
    its gradient (the model is 105957 fp32 values, so everything is stored in full)."""
    out = {"stats": trainer.step_stats().cpu().numpy()}
    for name, p in model.named_parameters():
        out["param." + name] = p.detach().cpu().numpy()
        out["grad." + name] = p.grad.detach().cpu().numpy()
    return out


def write_outputs(dirname, outputs):
    import numpy as np

    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: {total} bytes of outputs exceed the {DUMP_LIMIT_BYTES}-byte dump limit")
    os.makedirs(dirname, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


# ------------------------------------------------------------- our arm -----
def run_ours(args):
    import numpy as np
    import torch
    import torch.nn.functional as F

    import gnn_tableextraction_b200 as gte
    from gnn_tableextraction_b200 import ops, synth
    from gnn_tableextraction_b200.graph import batch_pages_host

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = torch.distributed
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gte.lib()
    pk = peaks()

    # synthetic batches (host, pinned); 3 different page orders to rotate through
    base = synth.make_pages(args.pages, base_seed=42 + 1000 * rank, n=NODES_PER_PAGE, k=KNN, distinct=min(args.pages, 64))
    rng = np.random.default_rng(rank)
    host_batches = []
    for i in range(3):
        order = np.arange(args.pages) if i == 0 else rng.permutation(args.pages)
        host_batches.append(batch_pages_host([base[j] for j in order], pin=True))
    n_nodes, n_edges = int(host_batches[0]["num_nodes"]), int(host_batches[0]["src"].numel())

    torch.manual_seed(0)
    model = gte.GcnSAGE(*MODEL_CFG[:3], MODEL_CFG[3], F.relu, 0).to(dev)
    trainer = gte.SageTrainer(model, lr=0.01, weight_decay=5e-4)
    use_graph = not args.no_graph
    lib = gte.lib()

    dev_batches = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in hb.items()} for hb in host_batches]

    def eager_step(db):
        g = gte.PageGraphBatch(db["src"], db["dst"], n_nodes, db["batch_num_nodes"], db["batch_num_edges"])
        g.edata["feat"] = db["weight"]
        g.ndata["feat"] = db["feat"]
        return trainer.train_step(g, db["label"])

    c0 = lib.gte_launch_count()
    eager_step(dev_batches[0])
    launches_per_step = lib.gte_launch_count() - c0
    if use_graph:
        try:
            trainer.capture(host_batches[0])  # data parallel: two graphs around the eager NCCL all-reduces
        except Exception as exc:  # e.g. a NCCL build that cannot be captured: keep the eager step
            if world == 1:
                raise
            print(f"[bench] rank {rank}: CUDA-graph capture failed ({type(exc).__name__}: {exc}); eager step", file=sys.stderr)
            use_graph = False
        if world > 1:  # all ranks must agree
            flag = torch.tensor([1 if use_graph else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            use_graph = bool(flag.item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = torch.tensor([e0.elapsed_time(e1), wall * 1e3], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms[0].item(), ms[1].item()

    stats_host = torch.zeros(3, dtype=torch.float32).pin_memory()
    stream = torch.cuda.current_stream()

    # --- leg 1: inputs resident in HBM ---------------------------------------------------------
    if use_graph:
        # two different batches sit in the trainer's two static input sets; the step alternates between them
        trainer.prefetch_batch(host_batches[0])
        trainer.prefetch_batch(host_batches[1])
        torch.cuda.synchronize()

        def resident(i):
            trainer.replay_set(i % 2)
    else:
        def resident(i):
            eager_step(dev_batches[i % 3])

    # --- leg 2: end to end through the public API with HOST buffers ---------------------------------
    if use_graph:
        trainer.replay_prefetched()  # consume the two resident batches of leg 1, then start the pipeline afresh
        trainer.replay_prefetched()
        trainer.prefetch_batch(host_batches[0])

        def e2e(i):
            # every step: the captured step on the current batch (launched first, so the GPU never waits for the
            # host to queue copies), H2D of the NEXT batch from pinned memory (side stream, overlaps this step's
            # kernels; it lands in the other static input set, no staging copy), D2H of [sum w*nll, sum w, #correct]
            trainer.replay_prefetched()
            trainer.prefetch_batch(host_batches[(i + 1) % 3])
            stats_host.copy_(trainer.step_stats(), non_blocking=True)
            stream.synchronize()  # the caller reads the loss every step (model_train.py:328 .item())
    else:
        def e2e(i):
            g = gte.PageGraphBatch.from_host(host_batches[i % 3], dev)
            stats_host.copy_(trainer.train_step(g), non_blocking=True)
            stream.synchronize()

    with ClockSampler(local) as clk:
        ms_res, _ = timed(resident, args.steps, args.warmup)
        # the legs below keep training the same model: take the headline leg's results before they do
        outputs = step_outputs(trainer, model) if args.dump_outputs and rank == 0 else None
        ms_e2e, wall_e2e = timed(e2e, args.steps, max(3, args.warmup // 2))
    loss = float(stats_host[0] / stats_host[1])
    hb = host_batches[0]
    h2d = sum(int(hb[k].numel() * hb[k].element_size()) for k in ("src", "dst", "weight", "feat", "label"))
    d2h = 12

    total_pages = args.pages * world
    value = total_pages * args.steps / (ms_res / 1e3)
    e2e_value = total_pages * args.steps / (max(ms_e2e, wall_e2e) / 1e3)

    # --- per-op device times (eager, events on the launching stream) --------------------------------
    roofline, conv, ops_table = None, None, None
    if not args.no_op_profile:
        prof_steps = max(3, min(args.steps, 10))
        for i in range(2):
            eager_step(dev_batches[i % 3])
        with OpTimer(ops, torch) as ot:
            for i in range(prof_steps):
                eager_step(dev_batches[i % 3])
            tab = ot.table(prof_steps)
        step_ms = sum(ms * cnt for ms, cnt in tab.values())
        rows = []
        for key, (ms, cnt) in sorted(tab.items(), key=lambda kv: -kv[1][0] * kv[1][1]):
            b, fl = op_cost(key)
            rows.append({"op": "/".join(str(x) for x in key), "ms": round(ms, 4), "per_step": cnt,
                         "share": round(ms * cnt / step_ms, 4),
                         "GBs": round(b / ms / 1e6, 1) if b else None, "TFLOPs": round(fl / ms / 1e9, 2) if fl else None})
        ops_table = rows[:14]
        # dominant kernel
        dkey, (dms, dcnt) = max(tab.items(), key=lambda kv: kv[1][0] * kv[1][1])
        b, fl = op_cost(dkey)
        hbm_t, tensor_peak = b / (pk["hbm_gbs"] * 1e9), pk["bf16_tflops_sustained"] / 2.0  # TF32 dense = bf16 / 2
        # The tensor-core kernels are 3xTF32: every fp32 product of the contraction is THREE tf32 MMAs (hi*hi, hi*lo,
        # lo*hi) -- that is what holds the 1e-5 fp32 parity bar.  So the tensor pipe has 3x the algorithmic flops to
        # execute, and that executed work is what its roofline bounds.
        mma_fl = 3 * fl if dkey[0].startswith("umma_") else fl
        if "linear" in dkey[0] and mma_fl / (tensor_peak * 1e12) > hbm_t:
            roofline = {"kernel": "/".join(str(x) for x in dkey), "bound": "tensor", "achieved": mma_fl / dms / 1e9,
                        "peak": tensor_peak, "unit": "TFLOP/s", "frac": mma_fl / dms / 1e9 / tensor_peak, "traffic": None,
                        "alg_flops": fl, "executed_mma_flops": mma_fl,
                        "hbm_frac_on_alg_bytes": b / dms / 1e6 / pk["hbm_gbs"],
                        "peak_source": pk["source"] + " bf16 sustained / 2 (TF32 dense rate); executed flops = 3 x "
                                                      "algorithmic (3xTF32 split: three tf32 MMAs per fp32 product)"}
        else:
            roofline = {"kernel": "/".join(str(x) for x in dkey), "bound": "hbm", "achieved": b / dms / 1e6,
                        "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": b / dms / 1e6 / pk["hbm_gbs"], "traffic": None,
                        "peak_source": pk["source"]}
        roofline["share_of_step"] = round(dms * dcnt / step_ms, 4)
        tr = ncu_traffic(dkey)
        if tr:
            roofline["traffic"], roofline["traffic_source"] = tr["bytes"], tr["capture"]
            roofline["alg_bytes"] = b
        # the conv (aggregation) kernel of the hidden layer: the HBM-roofline number north_star asks for
        sp = [(k, v) for k, v in tab.items() if k[0] == "spmm" and k[2] == MODEL_CFG[1]]
        if sp:
            k, (ms, cnt) = max(sp, key=lambda kv: kv[1][0])
            b, _ = op_cost(k)
            conv = {"kernel": "/".join(str(x) for x in k), "bound": "hbm", "achieved": b / ms / 1e6, "peak": pk["hbm_gbs"],
                    "unit": "GB/s", "frac": b / ms / 1e6 / pk["hbm_gbs"], "frac_of_8TBs_nominal": b / ms / 1e6 / 8000.0,
                    "ms": ms, "alg_bytes": b, "traffic": None}
            tr = ncu_traffic(k)
            if tr:
                conv["traffic"], conv["traffic_source"] = tr["bytes"], tr["capture"]

    # --- extras (N=1): ragged pages (SURVEY 8d second distribution) and a sustained-clock run -------------------
    extras = None
    if world == 1 and not args.no_extras:
        extras = {}
        try:
            # >= 2 s of back-to-back steps on the resident batches: the clock the GPU holds under this load
            n_sus = max(200, int(2000.0 / max(ms_res / args.steps, 1e-3)))
            with ClockSampler(local) as clk2:
                ms_sus, _ = timed(resident, n_sus, 3)
            extras["sustained"] = {"steps": n_sus, "ms_per_step": ms_sus / n_sus, "seconds": ms_sus / 1e3,
                                   "value": total_pages * n_sus / (ms_sus / 1e3), "unit": UNIT, "clocks": clk2.summary()}
            # ragged batch: page sizes ~ clip(N(300, 80), 40, 900) (builder.py:240-292 produces such pages), same model
            rp = synth.make_pages(args.pages, base_seed=7, k=KNN, ragged=True, distinct=min(args.pages, 96))
            rhb = batch_pages_host(rp, pin=True)
            torch.manual_seed(0)
            m2 = gte.GcnSAGE(*MODEL_CFG[:3], MODEL_CFG[3], F.relu, 0).to(dev)
            t2 = gte.SageTrainer(m2, lr=0.01, weight_decay=5e-4)
            t2.capture(rhb)
            t2.load_batch(rhb)
            ms_rag, _ = timed(lambda i: t2.replay(), args.steps, args.warmup)
            sizes = rhb["batch_num_nodes"]
            extras["ragged"] = {"pages": args.pages, "nodes": int(rhb["num_nodes"]), "edges": int(rhb["src"].numel()),
                                "page_nodes_min_max": [int(min(sizes)), int(max(sizes))], "ms_per_step": ms_rag / args.steps,
                                "value": args.pages * args.steps / (ms_rag / 1e3), "unit": UNIT,
                                "nodes_per_s": int(rhb["num_nodes"]) * args.steps / (ms_rag / 1e3),
                                "note": "same step, page sizes ~ clip(N(300,80),40,900), in-degree 10; resident inputs"}
            del t2, m2
        except Exception as exc:  # extras never take the headline line down
            extras["error"] = f"{type(exc).__name__}: {exc}"

    # --- CPU baseline (rank 0, N=1 only) -------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = cpu_oracle_run(args.cpu_pages, 10, 2, budget_s=20.0)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": f"configs[0]: {args.cpu_pages} pages/step x {r['steps']} steps, fwd+CE+bwd+Adam, oracle port "
                         f"(DGL absent: torch-only restatement of the reference CPU path), {r['ms_per_step']:.1f} ms/step, "
                         f"host_cpus={r['host_cpus']}"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_res / args.steps, "higher_is_better": True,
            "scaling": "strong" if args.global_pages else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": max(ms_e2e, wall_e2e) / args.steps},
            "gpu_launches": int(launches_per_step * args.steps), "launches_per_step": int(launches_per_step),
            "cuda_graph": bool(use_graph), "clocks": clk.summary(), "roofline": roofline, "conv_roofline": conv,
            "cpu_baseline": cpu, "ops": ops_table, "loss": loss, "nodes_per_step_per_gpu": n_nodes,
            "edges_per_step_per_gpu": n_edges, "lib": os.path.relpath(gte.LIB_PATH, ROOT), "extras": extras,
        }
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------- configs[2] --
def run_infer(args):
    """BASELINE.json configs[2]: inference on --infer-pages synthetic page graphs sharded by graph across the GPUs of one
    box (model_predict.py:130-154 does one forward per page; here: batched predict passes).  Every rank takes pages
    [r*P/W, (r+1)*P/W) and streams them in batches of --infer-batch pages from pinned host memory: the captured predict
    pass (format build, 3 layers without saved activations, argmax, per-page correct counts) of batch i runs while the
    copy engine brings batch i+1 into the other static input set; predictions stay on the device (all_pred buffer).
    No collective on the data path; one all-reduce of the accuracy counters at the end.  One "step" = the whole job."""
    import numpy as np
    import torch
    import torch.nn.functional as F

    import gnn_tableextraction_b200 as gte
    from gnn_tableextraction_b200 import synth
    from gnn_tableextraction_b200.graph import batch_pages_host

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = torch.distributed
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = gte.lib()
    lo, hi = rank * args.infer_pages // world, (rank + 1) * args.infer_pages // world
    mine = hi - lo
    # equal batches: nb = ceil(mine / infer_batch) captured predict passes of bsz = ceil(mine / nb) pages each; the last one
    # is filled up with repeated pages whose predictions are dropped (they are not counted in the metric either)
    nb = max(1, -(-mine // max(1, args.infer_batch)))
    bsz = -(-mine // nb)
    last_real = mine - (nb - 1) * bsz
    base = synth.make_pages(bsz, base_seed=42 + 1000 * rank, n=NODES_PER_PAGE, k=KNN, distinct=min(bsz, 64))
    rng = np.random.default_rng(rank)
    hbs = [batch_pages_host([base[j] for j in (np.arange(bsz) if i == 0 else rng.permutation(bsz))], pin=True) for i in range(3)]
    n_nodes = int(hbs[0]["num_nodes"])
    torch.manual_seed(0)
    model = gte.GcnSAGE(*MODEL_CFG[:3], MODEL_CFG[3], F.relu, 0).to(dev).eval()
    tr = gte.SageTrainer(model)
    tr.capture_predict(hbs[0])
    all_pred = torch.empty(mine * NODES_PER_PAGE, dtype=torch.int32, device=dev)
    correct_pages = torch.zeros(1, dtype=torch.float64, device=dev)
    sizes_full = torch.tensor(hbs[0]["batch_num_nodes"], dtype=torch.float64, device=dev)
    acc_host = torch.zeros(1, dtype=torch.float64).pin_memory()

    def consume(b, preds, corr, off):
        real = bsz if b + 1 < nb else last_real  # pages of this batch that belong to the job
        all_pred[off:off + real * NODES_PER_PAGE].copy_(preds[:real * NODES_PER_PAGE])
        correct_pages.add_((corr[:real].to(torch.float64) / sizes_full[:real]).sum())  # page permutations keep size 300
        return off + real * NODES_PER_PAGE

    def pass_e2e():
        """host buffers: H2D of every batch inside the timed region, overlapped with the previous batch's pass"""
        correct_pages.zero_()
        off = 0
        tr.prefetch_batch(hbs[0])
        for b in range(nb):
            preds, corr = tr.replay_prefetched()
            if b + 1 < nb:
                tr.prefetch_batch(hbs[(b + 1) % 3])
            off = consume(b, preds, corr, off)
        acc_host.copy_(correct_pages, non_blocking=True)  # the job's metric reaches the host every pass
        torch.cuda.current_stream().synchronize()
        return off

    def pass_resident():
        """inputs already in HBM: the two static input sets hold two different batches and alternate"""
        correct_pages.zero_()
        off = 0
        for b in range(nb):
            preds, corr = tr.replay_set(b % 2)
            off = consume(b, preds, corr, off)
        return off

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_passes(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        ms = torch.tensor([max(e0.elapsed_time(e1), 0.0), wall * 1e3], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms[0].item(), ms[1].item()

    c0 = lib.gte_launch_count()
    nw = max(1, min(args.warmup, 2))
    for _ in range(nw):
        pass_e2e()
    launches_per_pass = (lib.gte_launch_count() - c0) // nw
    steps = args.steps
    with ClockSampler(local) as clk:
        ms_e2e, wall_e2e = timed_passes(pass_e2e, steps)
        # resident leg: both static input sets hold a batch (the e2e leg left two of them there)
        tr.prefetch_batch(hbs[0])
        tr.prefetch_batch(hbs[1])
        tr.replay_prefetched()
        tr.replay_prefetched()
        pass_resident()
        ms_res, _ = timed_passes(pass_resident, steps)
    acc = correct_pages.clone()
    if world > 1:
        dist.all_reduce(acc)
    ms = [ms_res, max(ms_e2e, wall_e2e)]
    h2d = sum(int(hbs[0][k].numel() * hbs[0][k].element_size()) for k in ("src", "dst", "weight", "feat", "label"))
    if rank == 0:
        value = args.infer_pages * steps / (ms[0] / 1e3)
        line = {
            "metric": "page-graphs/sec (batched inference)", "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": nw, "ms_per_step": ms[0] / steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"configs[2]: GcnSAGE 13-218-218-9 inference on {args.infer_pages} synthetic page graphs "
                                   f"(300 nodes, directed kNN k=10) sharded by graph over {world} GPU(s), batches of {bsz} pages",
                       "pages_total": args.infer_pages, "pages_per_gpu": mine, "batch_pages": bsz, "parallelism": f"dp{world} by graph",
                       "step": "one step = the whole job: H2D of every batch (pinned, overlapped), CSC build, 3 layers, argmax, "
                               "per-page accuracy; predictions stay on the device",
                       "l2": "every batch is > 1 GB of activations; three different page orders alternate"},
            "e2e": {"value": args.infer_pages * steps / (ms[1] / 1e3), "unit": UNIT, "ms_per_step": ms[1] / steps,
                    "h2d_bytes_per_step": h2d * nb, "d2h_bytes_per_step": 8,
                    "note": "host buffers every batch; H2D inside the timed region (52.8 KB per page: PCIe / host-memory bound)"},
            "gpu_launches": int(launches_per_pass * steps), "launches_per_step": int(launches_per_pass), "cuda_graph": True,
            "clocks": clk.summary(), "mean_page_accuracy": acc.item() / args.infer_pages, "lib": os.path.relpath(gte.LIB_PATH, ROOT),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.global_pages:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if args.global_pages % world:
            raise SystemExit("--global-pages must be divisible by the number of GPUs")
        args.pages = args.global_pages // world
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "infer":
        run_infer(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
