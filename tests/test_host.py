"""CPU tests of the host layer: the C-ABI library loads and exports every symbol
declared in include/gte.h, the Python mirror keeps the reference's module
surface, and CPU tensors are rejected (there is no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import gnn_tableextraction_b200 as gte
from gnn_tableextraction_b200 import _lib, synth
from gnn_tableextraction_b200.graph import batch_pages_host

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "gte.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gte_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_header_symbol():
    names = _header_functions()
    assert len(names) >= 24
    l = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(l, n), f"{n} declared in include/gte.h but not exported by libgte_b200.so"
    assert sorted(_lib.SIGNATURES.keys()) == names  # ctypes table mirrors the header one to one


def test_abi_version_and_error_string():
    l = gte.lib()
    assert l.gte_abi_version() == _lib.ABI_VERSION == 3
    assert isinstance(l.gte_last_error_string(), bytes)
    # argument validation happens before any CUDA call: usable without a GPU
    assert l.gte_spmm(None, None, None, None, None, 7, None, 0, None, 0, None, 0, 4, 4, None) == -1
    assert b"bad mode" in l.gte_last_error_string()
    assert l.gte_csx_from_coo_workspace_bytes(10, 100) >= 2 * 100 * 4 + 11 * 4
    assert l.gte_csx_from_coo(None, None, 4, 2, None, None, None, None, 0, None) == -1
    assert l.gte_linear_bwd_weight_workspace_bytes(1000, 218, 218, 218) > 0


def test_module_surface_matches_reference():
    m = gte.GcnSAGE(13, 218, 9, 3, F.relu, 0)
    keys = list(m.state_dict().keys())
    assert keys == [
        "layers.0.linear.weight", "layers.0.linear.bias", "layers.0.lynorm.weight", "layers.0.lynorm.bias",
        "layers.1.linear.weight", "layers.1.linear.bias", "layers.1.lynorm.weight", "layers.1.lynorm.bias",
        "layers.2.linear.weight", "layers.2.linear.bias",
    ]
    assert m.layers[0].linear.weight.shape == (218, 26) and m.layers[2].linear.weight.shape == (9, 436)
    assert sum(p.numel() for p in m.parameters()) == 105957  # SURVEY section 8d
    assert m.layers[2].activation is None and not isinstance(m.layers[2].lynorm, torch.nn.LayerNorm)
    assert m.layers[0].dropout == 0.0 and isinstance(m.dropout, torch.nn.Dropout)
    ms = gte.MeanSAGE(13, 20, 9, 2)
    assert len(ms.layers) == 3 and list(ms.state_dict().keys())[0] == "layers.0.linear.weight"
    lay = gte.GcnSAGELayer(4, 8, F.relu, 0.5, bias=False, use_pp=True, use_lynorm=False)
    assert lay.linear.bias is None and lay.use_pp and isinstance(lay.dropout, torch.nn.Dropout)
    for meth in ("reset_parameters", "concat", "get_norm", "forward"):
        assert hasattr(lay, meth)


def test_cpu_inputs_are_rejected_not_computed():
    src = torch.zeros(3, dtype=torch.int32)
    with pytest.raises(gte.GteError):
        gte.PageGraphBatch(src, src, 2)
    with pytest.raises(gte.GteError):
        gte.ops.spmm(torch.zeros(3, dtype=torch.int32), src, None, torch.zeros(2, 4))
    with pytest.raises(gte.GteError):
        gte.ops.linear_fwd(torch.zeros(2, 4), None, torch.zeros(3, 4), None)
    from oracle.csx import OracleGraph

    g = OracleGraph([0], [1], 2, [1.0], np.zeros((2, 13), np.float32))
    with pytest.raises(gte.GteError):
        gte.GcnSAGE(13, 8, 3, 3, F.relu, 0)(g)


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libgte_b200.so")
    with pytest.raises(gte.GteError, match="no CPU fallback"):
        _lib.lib()


def test_batch_pages_host_is_dgl_batch():
    pages = [synth.make_page(1, n=20, k=3), synth.make_page(2, n=30, k=3)]
    hb = batch_pages_host(pages, pin=False)
    assert hb["num_nodes"] == 50 and hb["batch_num_nodes"] == [20, 30] and hb["batch_num_edges"] == [60, 90]
    assert hb["src"].dtype == torch.int32 and hb["feat"].shape == (50, 13) and hb["label"].dtype == torch.float32
    assert torch.equal(hb["src"][60:], torch.from_numpy(pages[1].src) + 20)
    assert torch.equal(hb["dst"][:60], torch.from_numpy(pages[0].dst))


def test_strategy_choice():
    from gnn_tableextraction_b200.layers import pick_strategy

    assert pick_strategy(13, 218, False) == "agg"
    assert pick_strategy(218, 218, False) == "agg"
    assert pick_strategy(218, 9, False) == "proj"  # aggregate 9 columns instead of 218
    assert pick_strategy(13, 9, True) == "pp"


def test_narrow_layer_policy_and_cpu_rejection():
    """host logic of the combined-operand route (layers.py): which layers pre-pack their weights / take the combined
    [n, 32] operands, and that its producers refuse CPU tensors instead of computing"""
    from gnn_tableextraction_b200 import layers as L, ops

    n = 153600
    assert L.wants_pack(n, 13, 218, False) and L.wants_pack(n, 218, 218, False) and L.wants_pack(n, 218, 9, False)
    assert not L.wants_pack(n, 13, 218, True)        # pre-propagated input: plain linear, no tensor-core pack
    assert not L.wants_pack(100, 218, 218, False)    # below the tensor-core row threshold
    assert not L.wants_pack(n, 300, 218, False)      # wider than the tensor-core tiles
    ctx = L.LayerCtx(strategy="proj", agg=L.GCN, h=None, ln=False, relu=False, fin=218, fout=9)
    assert not L.wants_class_grad_comb(ctx, n)       # no packed weights on the context: the layer ran on CUDA cores
    with pytest.raises(gte.GteError):
        ops.comb_from(torch.zeros(4, 13))
    with pytest.raises(gte.GteError):
        ops.umma_linear_fwd_comb(torch.zeros(4, 32), 13, torch.zeros(8), torch.zeros(218), 218)
    assert ops.COMB_W == 16 and ops.COMB_LD == 32


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver times beside ours) runs without a GPU and prints ONE JSON
    line with the agreed keys; under torchrun only rank 0 prints."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-pages", "2"]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "graphs/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "graphs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("configs[1]") and d["vs_baseline"] is None and d["dtype"] == "f32"
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out2 = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=root, env=env)
    assert out2.returncode == 0 and not [l for l in out2.stdout.splitlines() if l.startswith("{")]


@pytest.mark.gpu
def test_bench_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    """`bench.py --dump-outputs DIR`: the same arguments write the same arrays; one more timed step changes them"""
    import json
    import subprocess
    import sys

    def run(steps, tag):
        d = tmp_path / tag
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
               "--pages", "8", "--no-extras", "--no-cpu-baseline", "--no-op-profile", "--dump-outputs", str(d)]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == steps
        return {f.name: np.load(f) for f in sorted(d.iterdir())}

    a, b, c = run(2, "a"), run(2, "b"), run(3, "c")
    m = gte.GcnSAGE(13, 218, 9, 3, F.relu, 0)
    names = {"stats.npy"} | {f"{kind}.{k}.npy" for kind in ("param", "grad") for k, _ in m.named_parameters()}
    assert set(a) == set(b) == set(c) == names
    for k in names:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all()
        assert np.array_equal(a[k], b[k]), k
    assert a["stats.npy"][1] == 8 * 300  # sum of the label weights: one per node
    assert not np.array_equal(a["param.layers.0.linear.weight.npy"], c["param.layers.0.linear.weight.npy"])
