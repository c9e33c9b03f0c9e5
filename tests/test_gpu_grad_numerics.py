"""Per-element float64 bounds of every gradient reduction over the batch: dW, db, dgamma, dbeta and the column sums of dz.

The parity tests elsewhere measure max|a-b| / max|b| over a whole tensor.  The input layer reads the raw BBOX features,
whose columns differ by three to four orders of magnitude (w*h around 1e3-1e4, the four histogram columns in [0, 1]),
so that metric lets the small columns of dW carry an error 1000 times larger than fp32 allows.  Here every output
element is checked against float64 computed on the device from the exact fp32 operands the kernel read:

    |got - ref| <= K u G S            (+ u |old| with accumulate = 1)

with S the element's sum of absolute terms (|A|^T |B|; for a bias gradient the column sum of |dz|; for dgamma / dbeta
the column sums of |dy g x_hat| / |dy g|, g the ReLU gate) and G the number of rounded additions on the element's path,
read from the kernel's own plan (BOUNDS below).  Each test prints its worst bound ratio per entry, shape and kind
(pytest -rP).

The same calls check the operand contracts: outputs start as NaN (every element is written), the shared eager
workspace is filled with NaN (no partial is read that this launch did not write), the padding columns [f, ld) of every
operand hold NaN and then +-Inf (bit-identical results: padding is never interpreted), accumulate = 1 adds onto values
of another magnitude, and a repeated call gives the same bits.  n = 0 writes zeros, or leaves an accumulated output as
it was.

Operand kinds: "bbox" (the synthetic BBOX features and their GCN aggregation against a positive gradient), "positive"
(nearly constant positive columns: every rounding of a chain errs the same way and nothing cancels, the worst case of
chain growth), "cancel" (zero-mean gradient columns and cross-entropy gradient rows, which sum to zero and include rows
of class weight 0) and "spread" (rows and columns scaled by powers of two across +-40 binades).  Subnormal operands are
out of scope: the tensor-core split flushes them, and no layer of the model produces them.

The CPU tests at the end emulate, in numpy fp32, the defects these bounds exist to reject -- 1xTF32 products, one
sequential chain over all rows, a dropped chunk of rows, 1xTF32 error confined to the histogram columns -- and assert
that each breaks the bound while the two-level chunked sum and a 3xTF32 emulation stay within it.
"""
import ast
import functools
import os

import numpy as np
import pytest
import torch

DEV = "cuda"
U = 2.0 ** -24  # unit roundoff of fp32
# Constant of every bound in this file.  On an NVIDIA B200 (1000 W power limit) the worst ratio of the GPU tests is 0.91
# with K = 4, reached where u |old| dominates the accumulate bound; the worst ratio of any tensor-core entry is 0.81.
# The CPU tests below show the defects each bound targets clear it by 7x (one sequential chain against the loosest
# entry) to 95x (a dropped chunk against a tensor-core entry) at this K.
K = 4.0
EPS = float(np.float32(1e-5))
SMS_B200 = 148
ROWS = (0, 1, 255, 256, 257, 511, 513, 1023, 1024, 4097, 153600)  # 153600: config 2 (512 pages of 300 nodes)
KINDS = ("bbox", "positive", "cancel", "spread")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _log_ratio(tag, ratio):
    print(f"{tag}: worst bound ratio {ratio:.3e}")  # shown by pytest -rP


def _ratio(err, bound):
    """max(err / bound) with 0/0 = 0; NaN anywhere (error or bound) counts as a violation"""
    err = np.asarray(err, np.float64)
    bound = np.asarray(bound, np.float64)
    if np.isnan(err).any() or np.isnan(bound).any():
        return float("inf")
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / bound)  # err > 0 = bound: inf
    return float(np.max(r)) if r.size else 0.0


def _cdiv(a, b):
    return -(-a // b)


# ---------------------------------------------------------------------------------------- G of every entry ---
# Each function mirrors the host-side plan of one kernel (same constants, same rounding) and returns
# (rows of the first-level chain, G).  The GPU tests pass the device's SM count; the CPU tests use the B200's 148.
REP_3XTF32 = 32  # in units of u: the dropped lo*lo product (2^-20 S) and the tf32 rounding of both low parts (2 * 2^-21 S)


def _red(nb):
    """reduce_partials_block (gte_common.cuh): slice s adds partials s, s + 32, ... (ceil(nb / 32) additions), slice 0
    adds the 32 slice sums; + 1 for the accumulate add"""
    return _cdiv(nb, 32) + 32 + 1


def g_umma_dw(n, ipc, sms):
    """k_umma_dw + k_umma_dw_reduce (gte_umma_dw.cu).  dw_launch picks 384..640 rows per chunk (24..40 stages of 16
    rows, first minimum of rounds * stages); a chunk is rows / 8 MMA K-steps of 8 products each (3 levels) into a
    TMEM accumulator that truncates: doubled; + 1 for main + cross accumulator; + the chunks one CTA adds into its
    partial tile; then k_umma_dw_reduce: ceil(partials / 32) per accumulator, 2 to merge the four, 8 slices, accumulate;
    + the 3xTF32 representation term"""
    lanes = max(sms // ipc, 1)
    best_kb, best_cost = 32, -1
    for kb in range(384 // 16, 640 // 16 + 1):
        cost = _cdiv(_cdiv(n, kb * 16), lanes) * kb
        if best_cost < 0 or cost < best_cost:
            best_kb, best_cost = kb, cost
    rows = best_kb * 16
    nchunks = max(_cdiv(n, rows), 1)
    peers = _cdiv(min(sms, nchunks * ipc), ipc)  # partial tiles of one output tile
    return rows, 2 * (rows // 8 + 3) + 1 + _cdiv(nchunks, peers) + _cdiv(peers, 32) + 2 + 8 + 1 + REP_3XTF32


def ipc_umma_bwd_weight(fo, k1, k2):
    """(group, m-tile) items per chunk of gte_umma_linear_bwd_weight: one group while both segments fit 8 boxes"""
    nb = _cdiv(k1, 32) + _cdiv(k2, 32)
    return (1 if nb <= 8 else 2) * _cdiv(fo, 128)


def plan_split(rows, M, N):
    """plan_split (gte_dense.cu): (splits, rows per split)"""
    nt = 16 if N <= 16 else (32 if N <= 32 else (64 if N <= 64 else 128))
    want = min(_cdiv(592, _cdiv(M, 128) * _cdiv(N, nt)), 256)
    chunk = _cdiv(max(_cdiv(rows, want), 256), 16) * 16
    return max(_cdiv(rows, chunk), 1), chunk


def g_splitk(n, M, N):
    """FFMA split-K GEMM (one FMA chain per split) + k_splitk_reduce"""
    splits, chunk = plan_split(n, M, N)
    return chunk, min(chunk, max(n, 1)) + _red(splits)


def g_colsum(n):
    """k_colsum_partial (one chain per split of plan_split(n, 128, 128)) + k_splitk_reduce"""
    return g_splitk(n, 128, 128)


def g_gram_tall(n, wide):
    """k_gram_tall[_v4] (gte_gram.cuh): one FMA chain per row chunk of gram_plan, + k_gram_reduce / k_gram_qsum_reduce"""
    chunks = max(1184 // _cdiv(wide, 256), 1)
    rpc = _cdiv(max(_cdiv(max(n, 1), chunks), 64), 16) * 16
    return rpc, min(rpc, max(n, 1)) + _red(_cdiv(max(n, 1), rpc))


def g_gram_stream(n, sms):
    """k_gram_stream (gte_skinny.cu): one FMA chain per CTA over gs_grid's rows, + k_gram_stream_reduce"""
    rows = max(_cdiv(_cdiv(max(n, 1), 3 * sms), 32) * 32, 32)
    return rows, min(rows, max(n, 1)) + _red(_cdiv(max(n, 1), rows))


def g_ln_bwd(n, sms):
    """k_layernorm_act_bwd[_v4] (gte_rowops.cu): a warp walks rows w, w + 8 grid, ... (one chain), 8 warps add in a
    fixed order, + k_reduce_partials3 over the ln_bwd_grid partials"""
    grid = min(max(_cdiv(n, 8), 1), 2 * sms)
    rows = _cdiv(max(n, 1), 8 * grid)
    return rows, rows + 8 + _red(grid)


def g_linear_bwd_weight(n, fo, k1, k2, db):
    """G of (dW[:, :k1], dW[:, k1:], db) along gte_linear_bwd_weight's routes (gram_tall for narrow blocks, split-K
    otherwise, k_colsum_partial for a bias gradient no pass produced)"""
    if k1 > 0 and k2 > 0 and k1 + k2 + db <= 32:
        g = g_gram_tall(n, fo)[1]
        return g, g, g

    def block(k, with_db):
        if k + with_db <= 32:
            return g_gram_tall(n, fo)[1], with_db
        if fo <= 32:
            return g_gram_tall(n, k)[1], False
        return g_splitk(n, max(fo, k), min(fo, k))[1], False

    g1, did1 = block(k1, db)
    g2, did2 = block(k2, db and not did1)
    return g1, g2, (g1 if did1 else g2 if did2 else g_colsum(n)[1])


def g_linear_bwd_weight2(n, fo, k, x_aligned):
    """G of (dW[:, col1:], dW[:, col2:], db) along gte_linear_bwd_weight2's routes: one gram_tall pass over x when
    2 fo <= 32 (db from the same pass on aligned x), else two blocks and k_colsum_partial"""
    if 2 * fo <= 32:
        g = g_gram_tall(n, k)[1]
        return g, g, (g if x_aligned else g_colsum(n)[1])
    g = g_linear_bwd_weight(n, fo, k, 0, False)[0]
    return g, g, g_colsum(n)[1]


# Every weight-, bias- and LayerNorm-parameter-gradient entry of layers.sage_layer_backward and the function giving
# the G of its outputs (n, shape..., sms) -> G per output; the CPU test below fails when the layer calls a reduction
# that is not listed here.
BOUNDS = {
    "umma_linear_bwd_weight_comb": lambda n, fo, sms: [g_umma_dw(n, 1, sms)[1]] * 3,
    "umma_linear_bwd_weight": lambda n, fo, k1, k2, sms: [g_umma_dw(n, ipc_umma_bwd_weight(fo, k1, k2), sms)[1]] * 3,
    "umma_linear_bwd_weight2_comb": lambda n, fo, k, sms: [g_umma_dw(n, 1, sms)[1]] * 3,
    "umma_linear_bwd_weight2": lambda n, fo, k, db, sms: [g_umma_dw(n, _cdiv(k + db, 128), sms)[1]] * 3,
    "gram_stream": lambda n, sms: [g_gram_stream(n, sms)[1]] * 3,
    "linear_bwd_weight": lambda n, fo, k1, k2, db, sms: list(g_linear_bwd_weight(n, fo, k1, k2, db)),
    "linear_bwd_weight2": lambda n, fo, k, aligned, sms: list(g_linear_bwd_weight2(n, fo, k, aligned)),
    "layernorm_act_bwd": lambda n, sms: [g_ln_bwd(n, sms)[1] + 2, g_ln_bwd(n, sms)[1], g_ln_bwd(n, sms)[1]],
}
# ops calls of sage_layer_backward that reduce over no batch axis: input gradients, element-wise and layout kernels
NOT_BATCH_REDUCTIONS = {"relu_bwd", "linear_bwd_data", "linear_bwd_data2", "umma_linear_bwd_data",
                        "umma_linear_bwd_data2", "umma_linear_bwd_data_comb", "wide_out", "dropout_concat",
                        "comb_from", "comb_views", "_aligned_mat", "gram_stream_supported", "wide_out_supported"}
GRAD_ARGS = {"dW", "db", "dgamma", "dbeta"}


# ------------------------------------------------------------------------------------------------ operands ---
@functools.lru_cache(maxsize=1)
def bbox_features():
    """(h, A_hat h) [153600, 13] float32: the synthetic BBOX features of 512 pages and their GCN aggregation
    (in-degree-normalised weighted sum over in-edges)"""
    from gnn_tableextraction_b200 import synth

    hs, ahs = [], []
    for p in synth.make_pages(512, n=300, distinct=16):
        x = p.feat.astype(np.float64)
        agg = np.zeros_like(x)
        np.add.at(agg, p.dst, p.weight[:, None].astype(np.float64) * x[p.src])
        deg = np.bincount(p.dst, minlength=p.num_nodes).astype(np.float64)
        hs.append(p.feat)
        ahs.append((agg / np.maximum(deg, 1.0)[:, None]).astype(np.float32))
    return np.concatenate(hs), np.concatenate(ahs)


def positive_cols(rng, n, f):
    """nearly constant positive columns: s_c (1 + j 2^-18), j in [0, 16)"""
    s = rng.uniform(0.5, 2.0, f)
    return (s[None, :] * (1.0 + rng.integers(0, 16, (n, f)) * 2.0 ** -18)).astype(np.float32)


def truncate_tf32(x):
    """what kind::tf32 reads of an fp32 word: the low 13 mantissa bits cleared"""
    return (np.asarray(x, np.float32).view(np.uint32) & np.uint32(0xFFFFE000)).view(np.float32)


def round_tf32(x):
    """round to nearest (ties away) at 10 mantissa bits: the kernels' tf32_rna"""
    b = np.asarray(x, np.float32).view(np.uint32)
    return ((b + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _spread(rng, n, f):
    er = rng.integers(-20, 21, n).astype(np.float64)
    ec = rng.integers(-20, 21, f).astype(np.float64)
    return (rng.standard_normal((n, f)) * np.exp2(er[:, None] + ec[None, :])).astype(np.float32)


def grad_side(kind, n, f, seed):
    """fp32 [n, f] gradient operand (dz, A_hat^T dz, dy) of one kind, on the device"""
    from gnn_tableextraction_b200 import ops

    rng = np.random.default_rng(seed)
    if kind in ("bbox", "positive"):
        return _t(positive_cols(rng, n, f))
    if kind == "spread":
        return _t(_spread(rng, n, f))
    x = rng.standard_normal((n, f))
    x = (x - x.mean(0)[None, :] if n > 1 else x).astype(np.float32)
    rows = np.arange(0, n, 3)
    if len(rows):
        # cross-entropy gradient rows: sum to zero, scaled by w_y / den; class weight 0 and label -1 give zero rows
        c = min(f, 32)
        logits = _t((rng.standard_normal((len(rows), c)) * 3).astype(np.float32))
        y = rng.integers(0, c, len(rows))
        y[::7] = -1
        w = rng.uniform(0.25, 2.0, c).astype(np.float32)
        w[::3] = 0.0
        den = torch.tensor([max(len(rows) * 0.75, 1.0)], dtype=torch.float32, device=DEV)
        d = ops.cross_entropy_bwd(logits, _t(y), _t(w), den).cpu().numpy()
        x[rows] = 0.0
        x[rows, :c] = d
    return _t(x)


def act_side(kind, n, f, seed, agg=False):
    """fp32 [n, f] activation operand (h, A_hat h, x) of one kind; "bbox" tiles the 13 feature columns"""
    rng = np.random.default_rng(seed)
    if kind == "bbox":
        h = bbox_features()[1 if agg else 0][:n]
        return _t(h[:, np.arange(f) % 13])
    if kind == "positive":
        return _t(positive_cols(rng, n, f))
    if kind == "spread":
        return _t(_spread(rng, n, f))
    return _t(rng.standard_normal((n, f)).astype(np.float32))


def place(t, aligned):
    """(operand view, padding view or None): aligned = rows 16-byte aligned with ld = ops.padded_cols(f) (the tensor-core
    and 128-bit kernels); unaligned = ld = f + 1 starting 4 bytes past a 16-byte boundary (the scalar kernels)"""
    from gnn_tableextraction_b200 import ops

    n, f = t.shape
    if aligned:
        full = torch.zeros((n, ops.padded_cols(f)), dtype=torch.float32, device=DEV)
    else:
        full = torch.zeros(n * (f + 1) + 1, dtype=torch.float32, device=DEV)[1:].view(n, f + 1)
    v = full[:, :f]
    v.copy_(t)
    return v, (full[:, f:] if full.shape[1] > f else None)


def comb_place(a, b):
    """combined [n, 32] operand [a | b] (columns [0, w) and [16, 16 + w)) and its unused columns"""
    from gnn_tableextraction_b200 import ops

    n, w = a.shape
    xc = ops.comb_buffer(n, DEV)
    xc[:, :w] = a
    xc[:, 16:16 + w] = b
    pads = [xc[:, w:16]] + ([xc[:, 16 + w:]] if w < 16 else [])
    return xc, pads


# ------------------------------------------------------------------------------------- the checks of a call ---
WS_BYTES = 256 << 20


def _workspace():
    """the shared eager workspace, grown once so that every call of this file uses (and sees the poison of) it"""
    from gnn_tableextraction_b200 import ops

    return ops.workspace(WS_BYTES, torch.device(DEV))


def _bits(t):
    return t.contiguous().view(torch.int32).clone()


def _dev_ratio(got, ref, bound):
    err = (got.double() - ref).abs()
    if torch.isnan(err).any() or torch.isnan(bound).any():
        return float("inf")
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(r.max().item()) if r.numel() else 0.0


def check_call(call, outs, pads, seed=0):
    """call(accumulate) writes the tensors of outs = [(out, ref64, S64, G)].  Runs it with a zeroed and then a
    NaN-filled workspace (same bits), with NaN and then +-Inf operand padding (same bits), and with accumulate = 1
    onto values of another magnitude; returns the worst bound ratio.  n = 0 (ref None): zeros, or old values kept."""
    ws = _workspace()
    nan = float("nan")
    if outs[0][1] is None:
        for o, *_ in outs:
            o.fill_(nan)
        ws.fill_(255)
        call(False)
        for o, *_ in outs:
            assert torch.all(o == 0), "n = 0 must write zeros"
        olds = [_bits(torch.randn_like(o)) for o, *_ in outs]
        for (o, *_), old in zip(outs, olds):
            o.copy_(old.view(torch.float32).view_as(o))
        call(True)
        for (o, *_), old in zip(outs, olds):
            assert torch.equal(_bits(o), old), "n = 0 with accumulate must leave the output untouched"
        return 0.0

    def run(ws_fill, acc=False):
        if ws_fill is None:
            ws.zero_()
        else:
            ws.fill_(ws_fill)
        if not acc:
            for o, *_ in outs:
                o.fill_(nan)
        call(acc)
        return [_bits(o) for o, *_ in outs]

    first = run(None)
    again = run(255)  # 0xFFFFFFFF: NaN in every float of the workspace
    for k, (a, b) in enumerate(zip(first, again)):
        assert torch.equal(a, b), f"output {k}: a NaN workspace or a repeated call changed the bits"
    worst = 0.0
    for o, ref, S, G in outs:
        worst = max(worst, _dev_ratio(o, ref, K * U * G * S))
    for fill in ("nan", "inf"):
        for p in pads:
            if fill == "nan":
                p.fill_(nan)
            else:
                p.fill_(float("inf"))
                p[:, ::2].fill_(float("-inf"))
        got = run(255)
        for k, (a, b) in enumerate(zip(first, got)):
            assert torch.equal(a, b), f"output {k}: {fill} in the operand padding changed the result"
    for p in pads:
        p.zero_()
    g = torch.Generator(device=DEV).manual_seed(seed)
    olds = []
    for o, ref, S, G in outs:
        mag = torch.pow(10.0, torch.empty(o.shape, device=DEV, dtype=torch.float64).uniform_(-3, 3, generator=g))
        old = (torch.randn(o.shape, device=DEV, dtype=torch.float64, generator=g) * mag * (ref.abs() + S * 1e-3)).float()
        olds.append(old)
        o.copy_(old)
    run(255, acc=True)
    for (o, ref, S, G), old in zip(outs, olds):
        worst = max(worst, _dev_ratio(o, ref + old.double(), K * U * G * S + U * old.double().abs()))
    return worst


def _mm(a, b):
    """(a^T b, |a|^T |b|) in float64 on the device"""
    a64, b64 = a.double(), b.double()
    return a64.t() @ b64, a64.abs().t() @ b64.abs()


def _colsum(a):
    a64 = a.double()
    return a64.sum(0), a64.abs().sum(0)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _finish(tag, per_kind):
    for kind, r in per_kind.items():
        _log_ratio(f"{tag} kind={kind}", r)
    worst = max(per_kind.values())
    assert worst <= 1.0, f"{tag}: worst bound ratio {worst:.3e}"


def _skip_refused(name, n):
    """the tensor-core entries and gram_stream refuse n <= 1 in their argument checks (a one-row view reports ld = f,
    an empty operand a null pointer); sage_layer_backward dispatches them from 1024 and 256 rows on"""
    if n <= 1 and (name.startswith("umma_") or name == "gram_stream"):
        pytest.skip(f"{name} refuses n = {n}")


# ---------------------------------------------------------------------------------------------- input layer ---
FIN, FH = 13, 218
INPUT_ENTRIES = ("umma_linear_bwd_weight_comb", "gram_stream:aligned", "gram_stream:unaligned",
                 "linear_bwd_weight:aligned", "linear_bwd_weight:unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("entry", INPUT_ENTRIES)
def test_input_layer_weight_grad_per_element(entry, n):
    """dW = dz^T [h | A_hat h] (fin = 13, fo = 218) and db = colsum(dz) where the entry produces it"""
    from gnn_tableextraction_b200 import ops

    name, _, form = entry.partition(":")
    _skip_refused(name, n)
    sms = _sms()
    per_kind = {}
    for i, kind in enumerate(KINDS):
        dz0 = grad_side(kind, n, FH, 10 * i + n)
        h0, ah0 = act_side(kind, n, FIN, 10 * i + n + 1), act_side(kind, n, FIN, 10 * i + n + 2, agg=True)
        dz, pdz = place(dz0, True)  # dz is the wide P operand of gram_stream: aligned on every form
        dW = torch.empty((FH, 2 * FIN), device=DEV)
        db = torch.empty(FH, device=DEV)
        refs = None
        if n > 0:
            r1, s1 = _mm(dz0, h0)
            r2, s2 = _mm(dz0, ah0)
            refs = (torch.cat([r1, r2], 1), torch.cat([s1, s2], 1)) + _colsum(dz0)
        if name == "umma_linear_bwd_weight_comb":
            xc, pads = comb_place(h0, ah0)
            G = BOUNDS[name](n, FH, sms)
            call = lambda acc: ops.umma_linear_bwd_weight_comb(dz, xc, FIN, dW, db, acc)
            with_db = True
        elif name == "gram_stream":
            h, ph = place(h0, form == "aligned")
            ah, pah = place(ah0, form == "aligned")
            pads = [ph, pah]
            G = BOUNDS[name](n, sms)
            call = lambda acc: ops.gram_stream(dz, h, ah, dW, dW.stride(0), 1, dW[:, FIN:], dW.stride(0), 1, accumulate=acc)
            with_db = False
        else:
            dz, pdz = place(dz0, form == "aligned")
            h, ph = place(h0, form == "aligned")
            ah, pah = place(ah0, form == "aligned")
            pads = [ph, pah]
            G = BOUNDS[name](n, FH, FIN, FIN, True, sms)
            call = lambda acc: ops.linear_bwd_weight(dz, h, ah, dW, db, acc)
            with_db = True
        pads = [p for p in pads + [pdz] if p is not None]
        if refs is None:
            outs = [(dW, None, None, None)] + ([(db, None, None, None)] if with_db else [])
        else:
            Gw = torch.tensor([G[0]] * FIN + [G[1]] * FIN, dtype=torch.float64, device=DEV)[None, :]
            outs = [(dW, refs[0], refs[1], Gw)] + ([(db, refs[2], refs[3], G[2])] if with_db else [])
        per_kind[kind] = check_call(call, outs, pads, seed=i)
    _finish(f"input {entry} n={n}", per_kind)


# --------------------------------------------------------------------------------------------- hidden layer ---
HIDDEN_ENTRIES = ("umma_linear_bwd_weight:db", "umma_linear_bwd_weight:nodb", "linear_bwd_weight:aligned",
                  "linear_bwd_weight:unaligned", "linear_bwd_weight2:aligned", "linear_bwd_weight2:unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("entry", HIDDEN_ENTRIES)
@pytest.mark.parametrize("k", (218, 256, 255))
def test_hidden_layer_weight_grad_per_element(k, entry, n):
    """dW = dz^T [h | A_hat h] (k -> k) with db = colsum(dz), on the tensor-core kernel (with and without the all-ones
    column; db needs k % 32 != 0) and the FFMA kernels; linear_bwd_weight2: dW = [dz^T h | gq^T h]"""
    from gnn_tableextraction_b200 import ops

    name, _, form = entry.partition(":")
    if name == "umma_linear_bwd_weight" and form == "db" and k % 32 == 0:
        pytest.skip("the tensor-core bias gradient needs a free padding column (k % 32 != 0)")
    _skip_refused(name, n)
    aligned = form != "unaligned"
    sms = _sms()
    per_kind = {}
    for i, kind in enumerate(KINDS):
        dz0 = grad_side(kind, n, k, 10 * i + n + k)
        h0 = act_side(kind, n, k, 10 * i + n + k + 1)
        b0 = grad_side(kind, n, k, 10 * i + n + k + 2) if name == "linear_bwd_weight2" else \
            act_side(kind, n, k, 10 * i + n + k + 2, agg=True)
        dz, pdz = place(dz0, aligned)
        h, ph = place(h0, aligned)
        b, pb = place(b0, aligned)
        with_db = form != "nodb"
        dW = torch.empty((k, 2 * k), device=DEV)
        db = torch.empty(k, device=DEV) if with_db else None
        if name == "umma_linear_bwd_weight":
            G = BOUNDS[name](n, k, k, k, sms)
            call = lambda acc: ops.umma_linear_bwd_weight(dz, h, b, dW, db, acc)
        elif name == "linear_bwd_weight":
            G = BOUNDS[name](n, k, k, k, True, sms)
            call = lambda acc: ops.linear_bwd_weight(dz, h, b, dW, db, acc)
        else:
            G = BOUNDS[name](n, k, k, aligned, sms)
            call = lambda acc: ops.linear_bwd_weight2(dz, b, h, dW, 0, k, db, acc)
        pads = [p for p in (pdz, ph, pb) if p is not None]
        if n == 0:
            outs = [(dW, None, None, None)] + ([(db, None, None, None)] if with_db else [])
        else:
            if name == "linear_bwd_weight2":
                (r1, s1), (r2, s2) = _mm(dz0, h0), _mm(b0, h0)
            else:
                (r1, s1), (r2, s2) = _mm(dz0, h0), _mm(dz0, b0)
            Gw = torch.tensor([G[0]] * k + [G[1]] * k, dtype=torch.float64, device=DEV)[None, :]
            outs = [(dW, torch.cat([r1, r2], 1), torch.cat([s1, s2], 1), Gw)]
            if with_db:
                outs.append((db, *_colsum(dz0), G[2]))
        per_kind[kind] = check_call(call, outs, pads, seed=i)
    _finish(f"hidden k={k} {entry} n={n}", per_kind)


# ---------------------------------------------------------------------------------------------- class layer ---
CLASS_ENTRIES = ("umma_linear_bwd_weight2_comb", "umma_linear_bwd_weight2", "gram_stream:aligned",
                 "gram_stream:unaligned", "linear_bwd_weight2:aligned", "linear_bwd_weight2:unaligned")


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("entry", CLASS_ENTRIES)
@pytest.mark.parametrize("fo", (9, 16, 17, 32))
def test_class_layer_weight_grad_per_element(fo, entry, n):
    """dW = [dz^T h | (A_hat^T dz)^T h] (218 -> fo) and db = colsum(dz): the combined-operand and plain tensor-core
    kernels (db through the all-ones column / row), gram_stream with qsum = db, and the FFMA kernel"""
    from gnn_tableextraction_b200 import ops

    name, _, form = entry.partition(":")
    if name in ("umma_linear_bwd_weight2_comb", "gram_stream") and fo > 16:
        pytest.skip(f"{name} takes at most 16 classes")
    _skip_refused(name, n)
    aligned = form != "unaligned"
    sms = _sms()
    per_kind = {}
    for i, kind in enumerate(KINDS):
        dz0, gq0 = grad_side(kind, n, fo, 10 * i + n + fo), grad_side(kind, n, fo, 10 * i + n + fo + 1)
        h0 = act_side(kind, n, FH, 10 * i + n + fo + 2)
        h, ph = place(h0, True)  # the wide operand: aligned on every form (gram_stream's P)
        dW = torch.empty((fo, 2 * FH), device=DEV)
        db = torch.empty(fo, device=DEV)
        if name == "umma_linear_bwd_weight2_comb":
            dc, pads = comb_place(dz0, gq0)
            G = BOUNDS[name](n, fo, FH, sms)
            call = lambda acc: ops.umma_linear_bwd_weight2_comb(dc, fo, h, dW, 0, FH, db, acc)
        elif name == "umma_linear_bwd_weight2":
            dz, pdz = place(dz0, True)
            gq, pgq = place(gq0, True)
            pads = [pdz, pgq]
            G = BOUNDS[name](n, fo, FH, True, sms)
            call = lambda acc: ops.umma_linear_bwd_weight2(dz, gq, h, dW, 0, FH, db, acc)
        elif name == "gram_stream":
            dz, pdz = place(dz0, aligned)
            gq, pgq = place(gq0, aligned)
            pads = [pdz, pgq]
            G = BOUNDS[name](n, sms)
            call = lambda acc: ops.gram_stream(h, dz, gq, dW, 1, dW.stride(0), dW[:, FH:], 1, dW.stride(0), qsum=db,
                                               accumulate=acc)
        else:
            dz, pdz = place(dz0, aligned)
            gq, pgq = place(gq0, aligned)
            h, ph = place(h0, aligned)
            pads = [pdz, pgq]
            G = BOUNDS[name](n, fo, FH, aligned, sms)
            call = lambda acc: ops.linear_bwd_weight2(dz, gq, h, dW, 0, FH, db, acc)
        pads = [p for p in pads + [ph] if p is not None]
        if n == 0:
            outs = [(dW, None, None, None), (db, None, None, None)]
        else:
            (r1, s1), (r2, s2) = _mm(dz0, h0), _mm(gq0, h0)
            Gw = torch.tensor([G[0]] * FH + [G[1]] * FH, dtype=torch.float64, device=DEV)[None, :]
            outs = [(dW, torch.cat([r1, r2], 1), torch.cat([s1, s2], 1), Gw), (db, *_colsum(dz0), G[2])]
        per_kind[kind] = check_call(call, outs, pads, seed=i)
    _finish(f"class fo={fo} {entry} n={n}", per_kind)


# -------------------------------------------------------------------------------------- LayerNorm backward ---
def ln_bwd_ref(z, dy, mean, rstd, gamma, beta, relu):
    """float64 backward from the fp32 operands the kernel reads (its own mean and rstd): (ReLU gate g, x_hat, dz,
    per-element dz scale Sz = rstd (|a| + mean|a| + |x_hat| (mean|a x_hat| + |c2|)))"""
    z64, dy64 = z.double(), dy.double()
    xh = (z64 - mean.double()[:, None]) * rstd.double()[:, None]
    g = torch.ones_like(xh)
    if relu:
        g = (xh * gamma.double() + beta.double() > 0).double()
    a = dy64 * g * gamma.double()
    c1 = a.mean(1, keepdim=True)
    c2 = (a * xh).mean(1, keepdim=True)
    r = rstd.double()[:, None]
    dz = r * (a - c1 - xh * c2)
    sz = r * (a.abs() + a.abs().mean(1, keepdim=True) + xh.abs() * ((a * xh).abs().mean(1, keepdim=True) + c2.abs()))
    return g, xh, dz, sz


def ln_case(kind, n, f, seed):
    """(z, dy, mean, rstd, gamma, beta, relu) of one kind; dy is 0 where the ReLU kink is within 2^-12 of y's scale, so
    the fp32 gate of the kernel and the float64 gate agree wherever they matter"""
    rng = np.random.default_rng(seed)
    z = act_side(kind, n, f, seed)
    dy = grad_side(kind, n, f, seed + 1)
    z64 = z.double()
    mean = z64.mean(1)
    rstd = 1.0 / torch.sqrt(((z64 - mean[:, None]) ** 2).mean(1) + EPS)
    mean, rstd = mean.float(), rstd.float()
    gamma = (rng.random(f) + 0.5).astype(np.float32)
    gamma[::7] = 0.0
    gamma[1::5] *= -1
    beta = (rng.standard_normal(f) * 0.5).astype(np.float32)
    gamma, beta = _t(gamma), _t(beta)
    relu = KINDS.index(kind) % 2 == 0
    if relu and n > 0:
        xh = (z64 - mean.double()[:, None]) * rstd.double()[:, None]
        t = xh * gamma.double() + beta.double()
        near = t.abs() <= 2.0 ** -12 * ((xh * gamma.double()).abs() + beta.double().abs())
        dy = torch.where(near, torch.zeros_like(dy), dy)
    return z, dy, mean, rstd, gamma, beta, relu


@pytest.mark.gpu
@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("aligned", (True, False), ids=("v4", "scalar"))
@pytest.mark.parametrize("f", (9, 218, 256, 481, 1000))
def test_layernorm_bwd_param_grads_per_element(f, aligned, n):
    """layernorm_act_bwd under a general upstream dy: dgamma, dbeta and the column sums of dz per element (the
    latter against float64 sums of the kernel's own dz), dz per element; the 128-bit kernel takes aligned rows up to
    f = 480, the scalar kernel the rest"""
    from gnn_tableextraction_b200 import ops

    sms = _sms()
    per_kind = {}
    for i, kind in enumerate(KINDS):
        z0, dy0, mean, rstd, gamma, beta, relu = ln_case(kind, n, f, 100 * i + n + f)
        z, pz = place(z0, aligned)
        dy, pdy = place(dy0, aligned)
        dz = place(torch.zeros((n, f), device=DEV), aligned)[0]
        dgamma, dbeta, dcol = (torch.empty(f, device=DEV) for _ in range(3))
        call = lambda acc: ops.layernorm_act_bwd(dy, z, mean, rstd, gamma, beta, relu, dgamma, dbeta, acc, out=dz,
                                                 dz_colsum=dcol)
        pads = [p for p in (pz, pdy) if p is not None]
        if n == 0:
            per_kind[kind] = check_call(call, [(dgamma, None, None, None), (dbeta, None, None, None),
                                               (dcol, None, None, None)], pads, seed=i)
            continue
        g, xh, dz64, sz = ln_bwd_ref(z0, dy0, mean, rstd, gamma, beta, relu)
        gdg, gdb, gcol = BOUNDS["layernorm_act_bwd"](n, sms)
        gz = max(_cdiv(f, 32), 4 * _cdiv(f, 128)) + 5 + 6  # lane chain, warp_sum, the element's own roundings
        # dz: the kernel's output, checked once, then the column sums against float64 sums of that output
        dz.fill_(float("nan"))
        call(False)
        got_dz = dz.clone()
        rz = _dev_ratio(got_dz, dz64, K * U * gz * sz)
        t = dy0.double() * g
        outs = [(dgamma, (t * xh).sum(0), (t * xh).abs().sum(0), gdg), (dbeta, t.sum(0), t.abs().sum(0), gdb),
                (dcol, *_colsum(got_dz), gcol)]
        per_kind[kind] = max(rz, check_call(call, outs, pads, seed=i))
        assert torch.equal(_bits(dz), _bits(got_dz)), "dz changed between identical calls"
    _finish(f"layernorm_act_bwd f={f} {'v4' if aligned else 'scalar'} n={n}", per_kind)


# ------------------------------------------------------------------------------ every reduction has a bound ---
def _backward_calls():
    """[(ops function, names of its arguments)] of every ops call in layers.sage_layer_backward"""
    with open(os.path.join(ROOT, "gnn_tableextraction_b200", "layers.py")) as fh:
        tree = ast.parse(fh.read())
    calls = []
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef) and fn.name == "sage_layer_backward":
            for node in ast.walk(fn):
                if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute)
                        and isinstance(node.func.value, ast.Name) and node.func.value.id == "ops"):
                    args = list(node.args) + [kw.value for kw in node.keywords]
                    names = {a.id for arg in args for a in ast.walk(arg) if isinstance(a, ast.Name)}
                    calls.append((node.func.attr, names))
    return calls


def test_every_backward_reduction_has_a_bound():
    """every ops call of sage_layer_backward that receives dW, db, dgamma or dbeta has a G in BOUNDS (and a GPU test
    above), and every other call is a known non-reduction: a new reduction entry without a bound fails here"""
    calls = _backward_calls()
    assert {"layernorm_act_bwd", "umma_linear_bwd_weight", "gram_stream"} <= {c for c, _ in calls}
    for name, args in calls:
        if args & GRAD_ARGS:
            assert name in BOUNDS, f"sage_layer_backward reduces into {sorted(args & GRAD_ARGS)} with ops.{name}, " \
                                   f"which has no per-element bound"
        else:
            assert name in BOUNDS or name in NOT_BATCH_REDUCTIONS, f"unclassified ops.{name} in sage_layer_backward"
    assert {c for c, a in calls if a & GRAD_ARGS} == set(BOUNDS), "BOUNDS lists an entry the layer no longer calls"


# -------------------------------------------------------------------------------- sharpness of the bounds ---
N2 = 153600
ELEMS = 36  # emulated output elements per kind


def _sharp_operands(kind):
    """ELEMS (a, b) column pairs of length N2 in fp32: a a positive gradient column, b a positive column ("positive")
    or a BBOX feature column, the four histogram columns included ("bbox")"""
    rng = np.random.default_rng(7)
    a = positive_cols(rng, N2, ELEMS)
    if kind == "positive":
        b = positive_cols(rng, N2, ELEMS)
    else:
        h, ah = bbox_features()
        b = np.concatenate([h, ah], 1)[:, np.arange(ELEMS) % 26]
    return a, b


def _exact(a, b):
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    return (a64 * b64).sum(0), (np.abs(a64) * np.abs(b64)).sum(0)


def _planned_fp32(p, rows, group=1):
    """fp32 sum of each column of p in the shape of a kernel's plan: sequential chains of `rows` rows, `group`
    consecutive chain sums added in order (the warps of a CTA, the chunks of a CTA's partial tile), then the
    reduce_partials_block order over those partials (32 slices, then the slice sums)"""
    n, m = p.shape
    pad = _cdiv(n, rows * group) * rows * group - n
    q = np.concatenate([p, np.zeros((pad, m), np.float32)]).reshape(-1, rows, m)
    part = np.add.accumulate(q, axis=1, dtype=np.float32)[:, -1]
    part = np.add.accumulate(part.reshape(-1, group, m), axis=1, dtype=np.float32)[:, -1]
    slices = np.zeros((32, m), np.float32)
    for s in range(32):
        if len(part[s::32]):
            slices[s] = np.add.accumulate(part[s::32], axis=0, dtype=np.float32)[-1]
    return np.add.accumulate(slices, axis=0, dtype=np.float32)[-1].astype(np.float64)


def _entries_at(n):
    """(tensor-core entries, FFMA entries) at n rows on a 148-SM B200, for the shapes of the GPU tests: (entry, chain
    rows, chains per partial, G)"""
    s = SMS_B200

    def umma(name, ipc):
        rows, G = g_umma_dw(n, ipc, s)
        nchunks = _cdiv(n, rows)
        return name, rows, _cdiv(nchunks, _cdiv(min(s, nchunks * ipc), ipc)), G

    tc = [umma("umma_linear_bwd_weight_comb", 1), umma("umma_linear_bwd_weight", ipc_umma_bwd_weight(218, 218, 218)),
          umma("umma_linear_bwd_weight2", 2)]
    ffma = [("gram_stream", *g_gram_stream(n, s)), ("gram_tall", *g_gram_tall(n, 218)),
            ("linear_bwd_weight split-K", *g_splitk(n, 218, 218)), ("colsum", *g_colsum(n)),
            ("layernorm_act_bwd", *g_ln_bwd(n, s))]
    ffma = [(name, rows, 8 if name == "layernorm_act_bwd" else 1, G) for name, rows, G in ffma]
    return tc, ffma


def _log_margin(tag, margin):
    print(f"{tag}: bound ratio {margin:.3e} (the worst element)")


@pytest.mark.parametrize("kind", ("positive", "bbox"))
def test_tf32_single_pass_breaks_the_tensor_core_bound(kind):
    """(a) 1xTF32 (both operands truncated as kind::tf32 reads them) breaks the tensor-core bounds by at least 10x;
    (d) a 3xTF32 emulation summed in each plan's chunks stays within them"""
    a, b = _sharp_operands(kind)
    ref, S = _exact(a, b)
    one = _exact(truncate_tf32(a), truncate_tf32(b))[0]
    ah, bh = truncate_tf32(a), truncate_tf32(b)
    al, bl = round_tf32(a - ah), round_tf32(b - bh)
    p3 = (ah * bh + (ah * bl + al * bh)).astype(np.float32)
    for name, rows, group, G in _entries_at(N2)[0]:
        margin = _ratio(np.abs(one - ref), K * U * G * S)
        _log_margin(f"1xTF32 {name} {kind} N={N2}", margin)
        assert margin >= 10.0, (name, margin)
        r3 = _ratio(np.abs(_planned_fp32(p3, rows, group) - ref), K * U * G * S)
        _log_ratio(f"3xTF32 {name} {kind} N={N2}", r3)
        assert r3 <= 1.0, (name, r3)


@pytest.mark.parametrize("kind", ("positive", "bbox"))
def test_dropped_chunk_breaks_every_bound_and_the_planned_sum_keeps_it(kind):
    """(c) leaving out one chunk of rows of an entry's own plan breaks that entry's bound (by at least 10x for the
    tensor-core entries); (d) the fp32 sum in the shape of the plan (chains, partials, fixed-order reduction) stays
    within it"""
    a, b = _sharp_operands(kind)
    ref, S = _exact(a, b)
    tc, ffma = _entries_at(N2)
    p = (a * b).astype(np.float32)
    for entry in tc + ffma:
        name, rows, group, G = entry
        bound = K * U * G * S
        dropped = ref - (a[:rows].astype(np.float64) * b[:rows]).sum(0)
        margin = _ratio(np.abs(dropped - ref), bound)
        _log_margin(f"drop one chunk of {rows} rows, {name} {kind}", margin)
        assert margin > (10.0 if entry in tc else 1.0), (name, margin)
        planned = _ratio(np.abs(_planned_fp32(p, rows, group) - ref), bound)
        _log_ratio(f"fp32 sum in the plan's order, {name} {kind}", planned)
        assert planned <= 1.0, (name, planned)


def test_sequential_chain_breaks_every_bound():
    """(b) one sequential fp32 chain over all N rows breaks the bound of every entry on the positive kind, whose
    nearly equal terms make the roundings of a chain err the same way; the margin against the loosest entry (the FFMA
    split-K weight gradient, G about 1100) is the smallest"""
    a, b = _sharp_operands("positive")
    ref, S = _exact(a, b)
    seq = np.add.accumulate((a * b).astype(np.float32), axis=0, dtype=np.float32)[-1].astype(np.float64)
    tc, ffma = _entries_at(N2)
    for name, rows, group, G in tc + ffma:
        margin = _ratio(np.abs(seq - ref), K * U * G * S)
        _log_margin(f"one fp32 chain of {N2} rows against {name} (G = {G})", margin)
        assert margin > 1.0, (name, margin)


def test_histogram_columns_at_tf32_pass_rel_err_but_break_the_bound():
    """(e) a dW of the input layer whose four histogram columns alone carry 1xTF32 error, on BBOX x and positive dz:
    within the whole-tensor rel_err < 1e-5 of the parity tests, far outside the per-element bound"""
    h, _ = bbox_features()
    rng = np.random.default_rng(3)
    dz = positive_cols(rng, N2, 16)
    dz64, h64 = dz.astype(np.float64), h.astype(np.float64)
    ref, S = dz64.T @ h64, np.abs(dz64).T @ np.abs(h64)  # [16, 13]
    bad = ref.copy()
    hist = slice(9, 13)
    bad[:, hist] = truncate_tf32(dz).astype(np.float64).T @ truncate_tf32(h[:, hist]).astype(np.float64)
    rel = np.abs(bad - ref).max() / np.abs(ref).max()
    G = max(entry[3] for entry in _entries_at(N2)[0])
    margin = _ratio(np.abs(bad - ref), K * U * G * S)
    _log_margin(f"1xTF32 histogram columns: rel_err {rel:.2e}, per-element", margin)
    assert rel < 1e-5 and margin > 10.0, (rel, margin)
