"""Per-element float64 bounds of every sum that produces the layer's values: the forward projections
z = [h | ah] W^T + b, the input gradients dx = dz W, the neighbour aggregations A_hat h / A_hat^T dz, and the
ReLU + L2-normalise row op of MeanSAGE.

The parity tests measure max|a-b| / max|b| over a whole tensor.  That metric cannot see a defect confined to rows of
small magnitude while other rows are 2^20 times larger: one segment (the neighbour block) computed at 1xTF32, the last
partial k-block dropped, a missing edge, the source scale of the backward aggregation read at the destination.  Such
rows are common (zero-size boxes, isolated nodes, rows whose terms cancel, the cross-entropy gradient rows of
well-classified nodes).  Here every output element is checked against float64 computed on the device from the exact
fp32 operands the kernel read:

    |got - ref| <= K u (G S + Gb |b|)        (+ u |old| with accumulate = 1)

with S the element's sum of absolute terms (|X| |W|^T for a projection; post * sum_e |w_e pre_c x_c| + |addend| for an
aggregation), b the bias and G, Gb the number of rounded operations on the element's path, read from the kernel's own
plan (BOUNDS below).  Each test prints its worst bound ratio per entry, shape and kind (pytest -rP).

The same calls check the operand contracts: outputs passed as out= start as NaN (every element is written), a repeated
call gives the same bits, NaN and then +-Inf in the padding columns [f, ld) of every operand give the same bits
(padding is never interpreted), accumulate = 1 adds onto values of another magnitude, rows of zeros give exactly the
bias, n = 0 writes nothing, and the predict path (want_z=False) gives the same y bits as the training path.  Combined
[n, 32] operands need finite padding instead (ops.comb_buffer): their builders must leave zeros there.

Operand kinds: "bbox" (the synthetic BBOX features and their GCN aggregation against positive gradients), "spread"
(rows and columns scaled across +-20 binades, so S varies by about 2^40 between elements), "cancel" (x2 = -x1 against
equal weight blocks, and cross-entropy gradient rows: z is about b while S is not) and "positive" (nearly constant
terms: every rounding of a chain errs the same way).

The CPU tests at the end parse the layer functions (every kernel call they make has a bound somewhere) and emulate in
numpy fp32 the defects these bounds exist to reject, reporting by how much each one clears its bound.
"""
import ast
import functools
import os

import numpy as np
import pytest
import torch

import test_gpu_grad_numerics as gn  # operand kinds, TF32 emulation and the reduction bounds of the backward pass

DEV = "cuda"
U = 2.0 ** -24  # unit roundoff of fp32
# Constant of every bound in this file.  On an NVIDIA B200 (1000 W power limit) the worst ratio of the GPU tests is 0.98
# with K = 4, reached where u |old| dominates the accumulate bound of the FFMA input gradient; without accumulation the
# worst is 0.25 (FFMA), 0.19 (tensor cores), 0.16 (aggregations), 0.06 (ReLU + L2 normalise).  The CPU tests below show
# the defects each bound targets clear it by 24x (1xTF32 on the neighbour block only) and more at this K.
K = 4.0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KINDS = ("bbox", "spread", "cancel", "positive")
ROWS = (1, 255, 256, 257, 1023, 1024, 1153, 1279, 4097, 153600)
# (fin, fo) at the dispatch edges of every entry: the model's layers (13 -> 218 -> 218 -> 9), both sides of the
# 16-wide combined operand, of one, two and more 32-float k-blocks per segment (the split-accumulator threshold is
# more than two k-blocks in all: fin 32 | 33 with two segments, 64 | 65 with one), and of the 256-wide limit
SHAPES = ((13, 218), (218, 218), (218, 9), (16, 17), (17, 33), (32, 64), (33, 17), (64, 16), (65, 13), (250, 255),
          (255, 256), (256, 250))
BIG = ((13, 218), (218, 218), (218, 9))  # the shapes run at 153600 rows (config 2: 512 pages of 300 nodes)
ZERO_ROW = 61  # rows r % ZERO_ROW == 5 are all zero in every operand


def _log_ratio(tag, ratio):
    print(f"{tag}: worst bound ratio {ratio:.3e}")  # shown by pytest -rP


def _ratio(err, bound):
    """max(err / bound) with 0/0 = 0; NaN anywhere (error or bound) counts as a violation"""
    err = np.asarray(err, np.float64)
    bound = np.asarray(bound, np.float64)
    if np.isnan(err).any() or np.isnan(bound).any():
        return float("inf")
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / bound)
    return float(np.max(r)) if r.size else 0.0


def _dev_ratio(got, ref, bound):
    err = (got.double() - ref).abs()
    if torch.isnan(err).any() or torch.isnan(bound).any():
        return float("inf")
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    return float(r.max().item()) if r.numel() else 0.0


def _cdiv(a, b):
    return -(-a // b)


# ---------------------------------------------------------------------------------------- G of every entry ---
# Each function mirrors the plan of one kernel and returns (G, Gb): G multiplies S, Gb the bias magnitude.
REP_3XTF32 = gn.REP_3XTF32  # the 3xTF32 representation term, in units of u S


def g_ffma(k, accumulate=False):
    """k_gemm_ffma (gte_gemm.cuh): one FMA chain over all k terms of both segments, * row_scale, + bias, + old"""
    return k + 1 + int(accumulate), 1


def g_wide_out(k, row_scale=False):
    """k_wide_out (gte_skinny.cu): one FMA chain that starts from the bias, over k1 + k2 <= 32 terms, * row_scale"""
    return k + 1 + int(row_scale), k + 1 + int(row_scale)


def g_umma(kblocks):
    """k_umma_gemm / k_umma_gemm_pair: per 32-float k-block 4 K-steps x 3 MMAs (hi hi, hi lo, lo hi) of 8 products
    (3 levels) into a TMEM accumulator that truncates (doubled); with more than 2 k-blocks the cross terms go to a
    separate accumulator merged by 1 add (launch_umma_single / launch_umma_pair); + bias; + the 3xTF32 term"""
    return 2 * (12 * kblocks + 3) + int(kblocks > 2) + 1 + REP_3XTF32, 1


def g_spmm(deg, rounded_scale):
    """k_spmm_rows / k_spmm_paged / k_spmm_paged_pk (and its MG variant): one FMA chain over the row's in-page and
    then out-of-page edges; + 1 when w * pre_scale is rounded (generic kernels at load, the packed kernel at pack
    time); post (* norm, or / max(deg, 1)); + addend"""
    return deg + int(rounded_scale) + 2


# Every contraction entry of sage_layer_forward, aggregate_forward, aggregate_backward and the dh half of
# sage_layer_backward, and the function giving its (G, Gb); the CPU test below fails when the layer calls a kernel that
# is neither here, nor in test_gpu_grad_numerics.BOUNDS, nor in EXEMPT.
BOUNDS = {
    "linear_fwd": lambda fin, nseg: g_ffma(nseg * fin),
    "linear_bwd_data": lambda fo, acc: g_ffma(fo, acc),
    "linear_bwd_data2": lambda fo, acc: g_ffma(2 * fo, acc),
    "wide_out": lambda k, row_scale: g_wide_out(k, row_scale),
    "umma_linear_fwd": lambda fin, nseg: g_umma(nseg * _cdiv(fin, 32)),
    "umma_linear_fwd_stacked": lambda fin: g_umma(_cdiv(fin, 32)),
    "umma_linear_fwd_comb": lambda: g_umma(1),
    "umma_linear_bwd_data": lambda fo: g_umma(_cdiv(fo, 32)),
    "umma_linear_bwd_data2": lambda fo: g_umma(2 * _cdiv(fo, 32)),
    "umma_linear_bwd_data_comb": lambda: g_umma(1),
    "spmm": g_spmm,
    "spmm_packed": g_spmm,
}
# ops calls of the four layer functions bounded elsewhere or not sums at all
EXEMPT = {
    "layernorm_act_fwd",    # per-row bounds on y, mean and rstd: test_gpu_numerics.py
    "relu_fwd",             # element-wise max(z, 0), exact
    "relu_bwd",             # element-wise mask, exact
    "dropout_concat",       # element-wise mask and 1 / (1 - p); mask bits: test_gpu_kernels.py
    "umma_pack_weights",    # the tf32 hi/lo split of W: its error is REP_3XTF32 of every tensor-core bound here
    "comb_from",            # layout copy; its zero padding is checked below
    "comb_buffer",          # zeroed allocation
    "comb_views",           # column views
    "empty_padded",         # allocation
    "_aligned_mat",         # predicate
    "umma_supported",       # predicate
    "wide_out_supported",   # predicate
    "gram_stream_supported",  # predicate
}
LAYER_FUNCTIONS = ("sage_layer_forward", "sage_layer_backward", "aggregate_forward", "aggregate_backward")
MAY_REFUSE = {"umma_linear_fwd", "umma_linear_fwd_stacked", "umma_linear_fwd_comb", "umma_linear_bwd_data",
              "umma_linear_bwd_data2", "umma_linear_bwd_data_comb", "wide_out", "spmm_packed"}


# ------------------------------------------------------------------------------------------------ operands ---
def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def place(t, aligned):
    """(view, padding view): aligned = 16-byte aligned rows with at least 4 padding columns (the tensor-core, 128-bit
    and wide_out kernels); unaligned = ld = f + 1, starting 4 bytes past a 16-byte boundary (the scalar paths)"""
    from gnn_tableextraction_b200 import ops

    n, f = t.shape
    if aligned:
        ld = ops.padded_cols(f)
        ld = ld if ld > f else f + 4
        full = torch.zeros((max(n, 1), ld), dtype=torch.float32, device=DEV)[:n]
    else:
        full = torch.zeros(n * (f + 1) + 1, dtype=torch.float32, device=DEV)[1:].view(n, f + 1)
    v = full[:, :f]
    v.copy_(t)
    return v, full[:, f:]


def zero_rows(n):
    return torch.arange(5, max(n, 5), ZERO_ROW, device=DEV)


def act(kind, n, f, seed, agg=False):
    x = gn.act_side(kind, n, f, seed, agg=agg)
    x[zero_rows(n)] = 0.0
    return x


def grad(kind, n, f, seed):
    x = gn.grad_side(kind, n, f, seed)
    x[zero_rows(n)] = 0.0
    return x


def weights(kind, fo, k, seed):
    """fp32 [fo, k] weights; "spread" spreads the columns across +-8 binades"""
    rng = np.random.default_rng(seed)
    w = rng.standard_normal((fo, k)) / np.sqrt(k)
    if kind == "positive":
        w = np.abs(w) + 0.1
    if kind == "spread":
        w *= np.exp2(rng.integers(-8, 9, k))[None, :]
    return _t(w.astype(np.float32))


def bias(fo, seed):
    return _t(np.random.default_rng(seed).standard_normal(fo).astype(np.float32))


def _mm(a, w):
    """(a w^T, |a| |w|^T) in float64 on the device"""
    a64, w64 = a.double(), w.double()
    return a64 @ w64.t(), a64.abs() @ w64.abs().t()


def _bits(t):
    return t.contiguous().view(torch.int32).clone()


def _fill_pads(pads, how):
    for p in pads:
        if how == "nan":
            p.fill_(float("nan"))
        elif how == "inf":
            p.fill_(float("inf"))
            p[:, ::2].fill_(float("-inf"))
        else:
            p.zero_()


def check(call, expect, pads, acc_call=None, seed=0, zero_rows_exact=True):
    """call() returns the output tensors; expect = [(ref64, bound64)] per output.  Checks a repeated call (same bits),
    NaN and +-Inf padding (same bits), rows of zeros (exactly ref there) and, with acc_call(olds), accumulate = 1
    onto values of another magnitude; returns the worst bound ratio"""
    first = [_bits(o) for o in call()]
    outs = call()
    for k, o in enumerate(outs):
        assert torch.equal(first[k], _bits(o)), f"output {k}: a repeated call changed the bits"
    worst = 0.0
    for o, (ref, bound) in zip(outs, expect):
        worst = max(worst, _dev_ratio(o, ref, bound))
        zr = zero_rows(o.shape[0]) if zero_rows_exact else ()
        if len(zr):
            assert torch.equal(o[zr].double(), ref[zr]), "a row of zeros must give exactly the bias (or zero)"
    for how in ("nan", "inf"):
        _fill_pads(pads, how)
        for k, o in enumerate(call()):
            assert torch.equal(first[k], _bits(o)), f"output {k}: {how} in the operand padding changed the result"
    _fill_pads(pads, "zero")
    if acc_call is not None:
        g = torch.Generator(device=DEV).manual_seed(seed)
        olds = []
        for ref, bound in expect:
            mag = torch.pow(10.0, torch.empty(ref.shape, device=DEV, dtype=torch.float64).uniform_(-3, 3, generator=g))
            scale = ref.abs() + bound / (K * U) * 1e-3
            olds.append((torch.randn(ref.shape, device=DEV, dtype=torch.float64, generator=g) * mag * scale).float())
        for o, (ref, bound), old in zip(acc_call(olds), expect, olds):
            worst = max(worst, _dev_ratio(o, ref + old.double(), bound + U * old.double().abs()))
    return worst


def _refused(name, fn):
    """run fn(); an entry that refuses the shape in its argument check raises GteError: skip the combination"""
    from gnn_tableextraction_b200._lib import GteError

    try:
        return fn()
    except GteError as e:
        if name not in MAY_REFUSE:
            raise
        pytest.skip(f"{name} refuses this shape: {e}")


def _finish(tag, per_kind):
    for kind, r in per_kind.items():
        _log_ratio(f"{tag} kind={kind}", r)
    worst = max(per_kind.values())
    assert worst <= 1.0, f"{tag}: worst bound ratio {worst:.3e}"


def _bound(G, S, Gb=0, b=None):
    out = K * U * G * S
    if b is not None:
        out = out + K * U * Gb * b.double().abs()
    return out


def _shapes(n):
    return BIG if n == 153600 else SHAPES


def _cases():
    return [(fin, fo, n) for n in ROWS for fin, fo in _shapes(n)]


# ------------------------------------------------------------------------------------- operands of one case ---
class Case:
    """the operands of one (kind, n, fin, fo): forward x1 = h, x2 = ah, W = [Ws | Wn], b; backward dz1 = dz,
    dz2 = A_hat^T dz; kind "cancel" makes x2 = -x1, dz2 = -dz1 and Wn = Ws"""

    def __init__(self, kind, n, fin, fo, seed):
        self.kind, self.n, self.fin, self.fo = kind, n, fin, fo
        self.x1 = act(kind, n, fin, seed)
        self.x2 = -self.x1 if kind == "cancel" else act(kind, n, fin, seed + 1, agg=True)
        self.dz1 = grad(kind, n, fo, seed + 2)
        self.dz2 = -self.dz1 if kind == "cancel" else grad(kind, n, fo, seed + 3)
        w = weights(kind, fo, 2 * fin, seed + 4)
        if kind == "cancel":
            w[:, fin:] = w[:, :fin]
        self.W, self.pW = place(w, True)
        self.b = bias(fo, seed + 5)
        self.rs = _t(np.random.default_rng(seed + 6).uniform(0.0, 2.0, n).astype(np.float32))

    def w1(self):
        return self.W[:, :self.fin]

    def w2(self):
        return self.W[:, self.fin:]


# ------------------------------------------------------------------------------------------ FFMA + wide_out ---
FFMA_FWD = ("linear_fwd:agg", "linear_fwd:proj", "wide_out:fwd", "wide_out:fwd_rs_ln")
FFMA_BWD = ("linear_bwd_data", "linear_bwd_data2", "wide_out:bwd")


@pytest.mark.gpu
@pytest.mark.parametrize("fin,fo,n", _cases())
@pytest.mark.parametrize("entry", FFMA_FWD)
def test_exact_fp32_projection_per_element(entry, fin, fo, n):
    """z = [h | ah] W^T + b on the FFMA GEMM (two segments, or the proj route's two one-segment calls) and on
    wide_out (bias, optional row_scale and fused LayerNorm + ReLU, whose y must only repeat bit for bit: it is bounded
    against the kernel's own z in test_gpu_numerics.py)"""
    from gnn_tableextraction_b200 import ops

    name, _, form = entry.partition(":")
    if name == "wide_out" and fin > 16:
        x, _ = place(torch.zeros(4, fin, device=DEV), True)
        W = torch.zeros(fo, 2 * fin, device=DEV)
        with pytest.raises(ops.GteError):
            ops.wide_out(x, x, W.data_ptr(), W.data_ptr() + 4 * fin, 1, W.stride(0), fo)
        pytest.skip("wide_out takes fin <= 16")
    per_kind = {}
    for i, kind in enumerate(KINDS):
        c = Case(kind, n, fin, fo, 1000 * i + n + 7 * fin + fo)
        aligned = name == "wide_out" or i % 2 == 0
        x1, p1 = place(c.x1, aligned)
        x2, p2 = place(c.x2, aligned)
        pads = [p1, p2, c.pW]
        r1, s1 = _mm(c.x1, c.w1())
        r2, s2 = _mm(c.x2, c.w2())
        b64 = c.b.double()
        if entry == "linear_fwd:agg":
            out = torch.empty((n, fo), device=DEV)
            G, Gb = BOUNDS[name](fin, 2)

            def call():
                out.fill_(float("nan"))
                return [ops.linear_fwd(x1, x2, c.W, c.b, out=out)]
            expect = [(r1 + r2 + b64, _bound(G, s1 + s2, Gb, c.b))]
        elif entry == "linear_fwd:proj":
            outs = torch.empty((n, fo), device=DEV), torch.empty((n, fo), device=DEV)
            G, Gb = BOUNDS[name](fin, 1)
            pads = [p1, c.pW]

            def call():
                for o in outs:
                    o.fill_(float("nan"))
                return [ops.linear_fwd(x1, None, c.W, c.b, out=outs[0], w_col0=0),
                        ops.linear_fwd(x1, None, c.W, None, out=outs[1], w_col0=fin)]
            ra, sa = _mm(c.x1, c.w2())
            expect = [(r1 + b64, _bound(G, s1, Gb, c.b)), (ra, _bound(G, sa))]
        else:
            ln = form == "fwd_rs_ln"
            rs = c.rs if ln else None
            G, _ = BOUNDS[name](2 * fin, rs is not None)
            gamma, beta = torch.rand(fo, device=DEV) + 0.5, torch.randn(fo, device=DEV)

            def call():
                z, y, _, _ = _refused(name, lambda: ops.wide_out(x1, x2, c.W.data_ptr(), c.W.data_ptr() + 4 * fin, 1,
                                                                 c.W.stride(0), fo, c.b, gamma=gamma, beta=beta,
                                                                 relu=True, fuse_ln=ln, row_scale=rs))
                return [z] + ([y] if ln else [])
            rsc = c.rs.double()[:, None] if ln else 1.0
            ref = (r1 + r2 + b64) * rsc
            if ln:  # a row of zeros leaves the chain at b, then one fp32 rounding of b * row_scale
                zr = zero_rows(n)
                ref[zr] = (c.b[None, :] * c.rs[zr, None]).double()
            expect = [(ref, K * U * G * (s1 + s2 + b64.abs()) * (rsc.abs() if ln else 1.0))]
        per_kind[kind] = check(call, expect, pads)
    _finish(f"{entry} fin={fin} fo={fo} n={n}", per_kind)


@pytest.mark.gpu
@pytest.mark.parametrize("fin,fo,n", _cases())
@pytest.mark.parametrize("entry", FFMA_BWD)
def test_exact_fp32_input_gradient_per_element(entry, fin, fo, n):
    """dx = dz W[:, blk] (* row_scale) (+ old) on the FFMA GEMM, dx = dz Ws + gq Wn in one chain, and wide_out's
    class-layer form (B read through the sj / sc strides of W, fo <= 16)"""
    from gnn_tableextraction_b200 import ops

    if entry == "wide_out:bwd" and fo > 16:
        pytest.skip("the input-gradient form of wide_out takes fo <= 16")
    per_kind = {}
    for i, kind in enumerate(KINDS):
        c = Case(kind, n, fin, fo, 2000 * i + n + 7 * fin + fo)
        aligned = entry == "wide_out:bwd" or i % 2 == 0
        d1, p1 = place(c.dz1, aligned)
        d2, p2 = place(c.dz2, aligned)
        rs = c.rs if i % 2 == 1 else None
        rsc = rs.double()[:, None] if rs is not None else 1.0
        rsa = rsc.abs() if rs is not None else 1.0
        r1, s1 = c.dz1.double() @ c.w1().double(), c.dz1.double().abs() @ c.w1().double().abs()
        r2, s2 = c.dz2.double() @ c.w2().double(), c.dz2.double().abs() @ c.w2().double().abs()
        acc_call = None
        if entry == "linear_bwd_data":
            outs = [place(torch.zeros(n, fin, device=DEV), i % 2 == 0)[0] for _ in range(2)]
            pads = [p1, c.pW]
            G = BOUNDS[entry](fo, True)[0]

            def run(acc, olds=None):
                for k, o in enumerate(outs):
                    o.copy_(olds[k]) if acc else o.fill_(float("nan"))
                return [ops.linear_bwd_data(d1, c.W, 0, fin, row_scale=rs, out=outs[0], accumulate=acc),
                        ops.linear_bwd_data(d1, c.W, fin, fin, row_scale=rs, out=outs[1], accumulate=acc)]
            ra, sa = c.dz1.double() @ c.w2().double(), c.dz1.double().abs() @ c.w2().double().abs()
            expect = [(r1 * rsc, _bound(G, s1 * rsa)), (ra * rsc, _bound(G, sa * rsa))]
            acc_call = lambda olds: run(True, olds)
        elif entry == "linear_bwd_data2":
            out = place(torch.zeros(n, fin, device=DEV), i % 2 == 0)[0]
            pads = [p1, p2, c.pW]
            G = BOUNDS[entry](fo, True)[0]

            def run(acc, olds=None):
                out.copy_(olds[0]) if acc else out.fill_(float("nan"))
                return [ops.linear_bwd_data2(d1, 0, d2, fin, c.W, fin, row_scale=rs, out=out, accumulate=acc)]
            expect = [((r1 + r2) * rsc, _bound(G, (s1 + s2) * rsa))]
            acc_call = lambda olds: run(True, olds)
        else:
            pads = [p1, p2, c.pW]
            G = BOUNDS["wide_out"](2 * fo, False)[0]

            def run(acc, olds=None):
                return [_refused("wide_out", lambda: ops.wide_out(d1, d2, c.W.data_ptr(), c.W.data_ptr() + 4 * fin,
                                                                  c.W.stride(0), 1, fin))[0]]
            expect = [(r1 + r2, _bound(G, s1 + s2))]
        per_kind[kind] = check(lambda: run(False), expect, pads, acc_call, seed=i)
    _finish(f"{entry} fin={fin} fo={fo} n={n}", per_kind)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ("linear_fwd", "linear_bwd_data", "linear_bwd_data2", "wide_out", "spmm"))
def test_empty_batch_writes_nothing(name):
    """n = 0: the call succeeds and leaves every byte of the output buffer as it was"""
    from gnn_tableextraction_b200 import ops

    fin, fo = 13, 16
    W = torch.randn(fo, 2 * fin, device=DEV)
    buf = torch.full((4, 32), float("nan"), device=DEV)
    before = _bits(buf)
    x = torch.empty((0, 16), device=DEV)
    if name == "linear_fwd":
        ops.linear_fwd(x[:, :fin], x[:, :fin], W, torch.zeros(fo, device=DEV), out=buf[:0, :fo])
    elif name == "linear_bwd_data":
        ops.linear_bwd_data(x[:, :fo], W, 0, fin, out=buf[:0, :fin], accumulate=True)
    elif name == "linear_bwd_data2":
        ops.linear_bwd_data2(x[:, :fo], 0, x[:, :fo], fin, W, fin, out=buf[:0, :fin])
    elif name == "wide_out":
        z = ops.wide_out(x[:, :fin], x[:, :fin], W.data_ptr(), W.data_ptr() + 4 * fin, 1, W.stride(0), fo)[0]
        assert z.shape == (0, fo)
    else:
        indptr = torch.zeros(1, dtype=torch.int32, device=DEV)
        e = torch.zeros(0, dtype=torch.int32, device=DEV)
        ops.spmm(indptr, e, torch.zeros(0, device=DEV), x, out=buf[:0, :16])
    torch.cuda.synchronize()
    assert torch.equal(_bits(buf), before), "n = 0 wrote into the output"


# ---------------------------------------------------------------------------------------------- tensor cores ---
UMMA_FWD = ("umma_linear_fwd", "umma_linear_fwd:ln", "umma_linear_fwd_stacked", "umma_linear_fwd_comb",
            "umma_linear_fwd_comb:ln")
UMMA_BWD = ("umma_linear_bwd_data", "umma_linear_bwd_data2", "umma_linear_bwd_data_comb")


@pytest.mark.gpu
@pytest.mark.parametrize("fin,fo,n", _cases())
@pytest.mark.parametrize("entry", UMMA_FWD)
def test_tensor_core_projection_per_element(entry, fin, fo, n, umma_kernel):
    """z = [h | ah] W^T + b on the 3xTF32 kernels (both kernels via umma_kernel): two segments, the stacked class-layer
    form [h Ws^T + b | h Wn^T] and the combined [n, 32] operand; ":ln" fuses LayerNorm + ReLU, whose y must be the
    same bits with want_z=False (the predict path)"""
    from gnn_tableextraction_b200 import ops

    name, _, form = entry.partition(":")
    if name == "umma_linear_fwd_stacked" and fo > 16:
        pytest.skip("the stacked form takes fo <= 16")
    if name == "umma_linear_fwd_comb" and fin > 16:
        pytest.skip("the combined operand holds fin <= 16")
    ln = form == "ln"
    per_kind = {}
    for i, kind in enumerate(KINDS):
        c = Case(kind, n, fin, fo, 3000 * i + n + 7 * fin + fo)
        x1, p1 = place(c.x1, True)
        x2, p2 = place(c.x2, True)
        gamma = (torch.rand(fo, device=DEV) + 0.5) if ln else None
        beta = torch.randn(fo, device=DEV) if ln else None
        b64 = c.b.double()
        r1, s1 = _mm(c.x1, c.w1())
        r2, s2 = _mm(c.x2, c.w2())
        if name == "umma_linear_fwd":
            pads = [p1, p2, c.pW]
            G, Gb = BOUNDS[name](fin, 2)

            def fwd(want_z):
                pack = ops.umma_pack_weights(c.W, fin, 2)
                z, y, _, _ = _refused(name, lambda: ops.umma_linear_fwd(x1, x2, fin, pack, c.b, fo, gamma=gamma,
                                                                        beta=beta, relu=ln, fuse_ln=ln, want_z=want_z))
                return [z, y]
            expect = [(r1 + r2 + b64, _bound(G, s1 + s2, Gb, c.b))]
        elif name == "umma_linear_fwd_comb":
            pads = [c.pW]
            G, Gb = BOUNDS[name]()

            def fwd(want_z):
                xc = ops.comb_from(c.x1)
                assert torch.all(xc[:, fin:] == 0), "comb_from must leave zeros in the unused columns"
                xc[:, 16:16 + fin] = c.x2
                pack = ops.umma_pack_weights(c.W, fin, 2)
                z, y, _, _ = _refused(name, lambda: ops.umma_linear_fwd_comb(xc, fin, pack, c.b, fo, gamma=gamma,
                                                                             beta=beta, relu=ln, fuse_ln=ln,
                                                                             want_z=want_z))
                return [z, y]
            expect = [(r1 + r2 + b64, _bound(G, s1 + s2, Gb, c.b))]
        else:
            pads = [p1, c.pW]
            G, Gb = BOUNDS[name](fin)
            ra, sa = _mm(c.x1, c.w2())

            def fwd(want_z):
                pack = ops.umma_pack_weights(c.W, fin, 2)
                sp = _refused(name, lambda: ops.umma_linear_fwd_stacked(x1, fin, pack, c.b, fo))
                return [sp[:, :fo], sp[:, 16:16 + fo]]
            expect = [(r1 + b64, _bound(G, s1, Gb, c.b)), (ra, _bound(G, sa))]
        # outputs: z (and y with ":ln", which must only repeat), or the two blocks of the stacked form
        per_kind[kind] = check(lambda: [o for o in fwd(True) if o is not None], expect, pads)
        if ln:
            assert torch.equal(_bits(fwd(True)[1]), _bits(fwd(False)[1])), "want_z=False changed y"
    _finish(f"{entry} [{umma_kernel}] fin={fin} fo={fo} n={n}", per_kind)


@pytest.mark.gpu
@pytest.mark.parametrize("fin,fo,n", _cases())
@pytest.mark.parametrize("entry", UMMA_BWD)
def test_tensor_core_input_gradient_per_element(entry, fin, fo, n, umma_kernel):
    """dx = dz W on the 3xTF32 kernels: (dz Ws, dz Wn), dz Ws + gq Wn in one contraction, and the combined [dz | gq]
    operand of the class layer, built by cross_entropy_bwd_comb / comb_from, which must leave zeros in its unused
    columns"""
    from gnn_tableextraction_b200 import ops

    if entry == "umma_linear_bwd_data_comb" and fo > 16:
        pytest.skip("the combined operand holds fo <= 16")
    per_kind = {}
    for i, kind in enumerate(KINDS):
        c = Case(kind, n, fin, fo, 4000 * i + n + 7 * fin + fo)
        d1, p1 = place(c.dz1, True)
        d2, p2 = place(c.dz2, True)
        w1, w2 = c.w1().double(), c.w2().double()
        r1, s1 = c.dz1.double() @ w1, c.dz1.double().abs() @ w1.abs()
        r2, s2 = c.dz2.double() @ w2, c.dz2.double().abs() @ w2.abs()
        if entry == "umma_linear_bwd_data":
            pads = [p1, c.pW]
            G = BOUNDS[entry](fo)[0]

            def call():
                pack = ops.umma_pack_weights(c.W, fin, 2)
                return list(_refused(entry, lambda: ops.umma_linear_bwd_data(d1, pack, fin, 2)))
            ra, sa = c.dz1.double() @ w2, c.dz1.double().abs() @ w2.abs()
            expect = [(r1, _bound(G, s1)), (ra, _bound(G, sa))]
        elif entry == "umma_linear_bwd_data2":
            pads = [p1, p2, c.pW]
            G = BOUNDS[entry](fo)[0]

            def call():
                pack = ops.umma_pack_weights(c.W, fin, 2)
                return [_refused(entry, lambda: ops.umma_linear_bwd_data2(d1, d2, pack, fin))]
            expect = [(r1 + r2, _bound(G, s1 + s2))]
        else:
            pads = [c.pW]
            G = BOUNDS[entry]()[0]

            def call():
                dc = ops.comb_from(c.dz1)
                assert torch.all(dc[:, fo:] == 0), "comb_from must leave zeros in the unused columns"
                dc[:, 16:16 + fo] = c.dz2
                pack = ops.umma_pack_weights(c.W, fin, 2)
                return [_refused(entry, lambda: ops.umma_linear_bwd_data_comb(dc, fo, pack, fin))]
            expect = [(r1 + r2, _bound(G, s1 + s2))]
        per_kind[kind] = check(call, expect, pads)
    _finish(f"{entry} [{umma_kernel}] fin={fin} fo={fo} n={n}", per_kind)


@pytest.mark.gpu
@pytest.mark.parametrize("c", (1, 9, 13, 16))
def test_cross_entropy_comb_leaves_zero_padding(c):
    """cross_entropy_bwd_comb writes d logits as the self block of an [n, 32] operand and zeros everywhere else: the
    tensor-core kernels read those columns against zero weights, so they must be finite"""
    from gnn_tableextraction_b200 import ops

    n = 1279
    logits = torch.randn(n, c, device=DEV) * 3
    labels = torch.randint(-1, c, (n,), device=DEV)
    w = torch.rand(c, device=DEV) + 0.25
    den = torch.tensor([n * 0.75], device=DEV)
    dc = ops.cross_entropy_bwd_comb(logits, labels, w, den)
    assert torch.all(dc[:, c:] == 0), "cross_entropy_bwd_comb must leave zeros in the unused columns"
    ref = ops.cross_entropy_bwd(logits, labels, w, den)
    assert torch.equal(_bits(dc[:, :c]), _bits(ref)), "the self block must be the plain kernel's d logits"


# ------------------------------------------------------------------------------------------------ aggregation ---
def _graph(kind):
    """(src, dst, w, n, page sizes or None) int32 / float32 numpy arrays of one aggregation case; edge weights
    include 0"""
    from gnn_tableextraction_b200 import synth

    if kind == "multi":  # a hub row of about 3600 in-edges, zero-in-degree rows, duplicates, self loops; no pages
        n = 4097
        src, dst, w = synth.random_multigraph(11, n, 6 * n, with_isolated=True)
        rng = np.random.default_rng(12)
        hub_src = rng.integers(0, n, 3600).astype(np.int32)
        src = np.concatenate([src, hub_src])
        dst = np.concatenate([dst, np.full(3600, 17, np.int32)])
        w = np.concatenate([w, rng.random(3600).astype(np.float32)])
        sizes = None
    else:
        if kind.startswith("pages7"):
            pages = synth.make_pages(37, k=7, ragged=True)
        else:
            pages = synth.make_pages(512, n=300, k=int(kind[5:]), distinct=8)
        off = np.cumsum([0] + [p.num_nodes for p in pages])
        src = np.concatenate([p.src + o for p, o in zip(pages, off)]).astype(np.int32)
        dst = np.concatenate([p.dst + o for p, o in zip(pages, off)]).astype(np.int32)
        w = np.concatenate([p.weight for p in pages]).astype(np.float32)
        n = int(off[-1])
        sizes = [p.num_nodes for p in pages]
    w = w.copy()
    w[::11] = 0.0
    return src, dst, w, n, sizes


def _page_table(indptr_h, sizes, cut):
    """(page_off, P, max page nodes, max page edges) over the rows of one direction; cut = each page split in two at
    a third of its rows, so that edges leave the (smaller) pages"""
    if cut:
        sizes = [s for p in sizes for s in (max(p // 3, 1), p - max(p // 3, 1)) if s > 0]
    off = np.cumsum([0] + list(sizes)).astype(np.int32)
    edges = indptr_h[off[1:]] - indptr_h[off[:-1]]
    return torch.from_numpy(off).to(DEV), len(sizes), int(max(sizes)), int(edges.max())


@functools.lru_cache(maxsize=1)
def _graph_dev(kind):
    from gnn_tableextraction_b200 import ops

    src, dst, w, n, sizes = _graph(kind)
    s, d, we = _t(src), _t(dst), _t(w)
    out = {"n": n, "sizes": sizes}
    for which, key, other in (("csc", d, s), ("csr", s, d)):
        indptr, indices, eid = ops.csx_from_coo(key, other, n)
        out[which] = (indptr, indices, ops.gather_f32(we, eid))
    out["norm"] = ops.degree_norm(out["csc"][0])
    return out


AGG_GRAPHS = ("pages7", "multi", "pages7cut", "pages45", "pages40")
AGG_WIDTHS = (1, 3, 4, 9, 13, 16, 17, 32, 33, 64, 218, 256, 512)
AGG_WIDTHS_BIG = (9, 33, 218, 512)
AGG_MODES = ("sum_norm", "mean", "sum_pre_addend")
AGG_KERNELS = ("rows", "rows_unaligned", "paged", "packed")


def _agg_cases():
    out = []
    for gk in AGG_GRAPHS:
        for f in (AGG_WIDTHS_BIG if gk.startswith("pages4") else AGG_WIDTHS):
            for kern in AGG_KERNELS:
                if gk == "multi" and kern in ("paged", "packed"):
                    continue
                out.append((gk, f, kern))
    return out


def spmm_ref(indptr, indices, w, x, post, pre=None, addend=None):
    """(y, S) in float64 on the device: y = post * sum_e w_e pre_c x_c (+ addend), S = post * sum |...| + |addend|"""
    n = indptr.numel() - 1
    vals = w.double() * (pre.double()[indices.long()] if pre is not None else 1.0)
    A = torch.sparse_csr_tensor(indptr.long(), indices.long(), vals, size=(n, x.shape[0]))
    Aa = torch.sparse_csr_tensor(indptr.long(), indices.long(), vals.abs(), size=(n, x.shape[0]))
    y = (A @ x.double()) * post[:, None]
    S = (Aa @ x.double().abs()) * post.abs()[:, None]
    if addend is not None:
        y = y + addend.double()
        S = S + addend.double().abs()
    return y, S


@pytest.mark.gpu
@pytest.mark.parametrize("graph,f,kernel", _agg_cases())
def test_aggregation_per_element(graph, f, kernel):
    """A_hat h (GCN: sum * norm; mean: sum / max(deg, 1)) on the CSC and A_hat^T dz (sum of w_e norm[src] dz with an
    addend) on the CSR, on the generic row kernel (aligned and scalar), the page-staged kernel and the packed page
    kernel (staged or edges through L1); the reference uses the kernel's own fp32 norm"""
    from gnn_tableextraction_b200 import _lib, ops

    gd = _graph_dev(graph)
    n = gd["n"]
    per = {}
    for i, xkind in enumerate(("spread", "cancel", "positive")):
        for mode in AGG_MODES:
            which = "csr" if mode == "sum_pre_addend" else "csc"
            indptr, indices, w = gd[which]
            aligned = kernel != "rows_unaligned"
            x, px = place(grad(xkind, n, f, 100 * i + f), aligned)
            pads = [px]
            addend = pre = row_norm = None
            deg = (indptr[1:] - indptr[:-1]).double()
            if mode == "sum_norm":
                kmode, row_norm, post = _lib.GTE_AGG_SUM_NORM, gd["norm"], gd["norm"].double()
            elif mode == "mean":
                kmode, post = _lib.GTE_AGG_MEAN, 1.0 / deg.clamp_min(1.0)
            else:
                kmode, pre, post = _lib.GTE_AGG_SUM, gd["norm"], torch.ones(n, dtype=torch.float64, device=DEV)
                a0 = act(xkind, n, f, 100 * i + f + 1)
                addend, pa = place(a0, aligned)
                pads.append(pa)
            out = place(torch.zeros(n, f, device=DEV), aligned)[0]
            pages = None
            if kernel in ("paged", "packed"):
                pages = _page_table(indptr.cpu().numpy(), gd["sizes"], graph.endswith("cut"))
            if kernel == "packed":
                pk = ops.paged_pack_edges(indptr, indices, w, pages, pre_scale=pre)

                def call():
                    out.fill_(float("nan"))
                    return [_refused("spmm_packed", lambda: ops.spmm_packed(indptr, pk, x, pages, mode=kmode,
                                                                            row_norm=row_norm, addend=addend, out=out))]
            else:
                def call():
                    out.fill_(float("nan"))
                    return [ops.spmm(indptr, indices, w, x, mode=kmode, row_norm=row_norm, pre_scale=pre,
                                     addend=addend, out=out, pages=pages)]
            ref, S = spmm_ref(indptr, indices, w, x, post, pre, addend)
            G = BOUNDS["spmm"](deg, pre is not None)[:, None]
            per[f"{xkind}/{mode}"] = _check_agg(call, ref, K * U * G * S, pads)
    _finish(f"spmm {kernel} graph={graph} f={f}", per)


def _check_agg(call, ref, bound, pads):
    """check() without the zero-row rule (an aggregated row is zero only where its sources are)"""
    first = [_bits(o) for o in call()]
    outs = call()
    assert torch.equal(first[0], _bits(outs[0])), "a repeated call changed the bits"
    worst = _dev_ratio(outs[0], ref, bound)
    for how in ("nan", "inf"):
        _fill_pads(pads, how)
        assert torch.equal(first[0], _bits(call()[0])), f"{how} in the operand padding changed the result"
    _fill_pads(pads, "zero")
    return worst


# ------------------------------------------------------------------------------- ReLU + L2 normalise ---
EPS_L2 = float(np.float32(1e-12))  # the kernel's fp32 eps; torch's fp32 clamp_min compares against the same value


def l2_rows(f, seed):
    """(z, dy) fp32 [rows, f]: random mixed-sign rows whose ReLU part has norm 10^s, s from -11.5 to 18 (plus one row
    below eps), a row of norm exactly fp32(eps), a row at norm 1e13, all-negative rows, and rows with dy parallel to y.
    Rows whose sum of squares overflows fp32 (|z| >~ 1.8e19) follow torch's fp32 behaviour and are out of scope."""
    rng = np.random.default_rng(seed)
    scales = [10.0 ** s for s in np.arange(-11.5, 18.01, 0.5)] + [1e-13, 1.0, 1e13]
    z = rng.standard_normal((len(scales) * 2, f))
    z[:, 0] = np.abs(z[:, 0]) + 0.1  # at least one positive entry
    rows = []
    for k, s in enumerate(scales):
        for r in (2 * k, 2 * k + 1):
            z[r] *= s / np.linalg.norm(np.maximum(z[r], 0.0))
            rows.append(z[r])
    tie = np.zeros(f)
    tie[0] = EPS_L2
    if f > 2:
        tie[2] = -1.0
    big = -np.ones(f)
    big[:3] = [1e13, 2e13, 5e12][:f]
    neg = -np.abs(rng.standard_normal((2, f))) - 0.1
    z = np.concatenate([np.stack(rows), tie[None], big[None], neg]).astype(np.float32)
    dy = rng.standard_normal(z.shape)
    dy[len(rows):len(rows) + 2] = np.arange(1.0, f + 1.0)  # [1, 2, 3, ...] at the tie and 1e13 rows
    r = np.maximum(z.astype(np.float64), 0)
    par = np.arange(0, len(rows), 5)
    dy[par] = 3.0 * r[par] / np.linalg.norm(r[par], axis=1, keepdims=True)  # dy parallel to y: dz = 0
    return z, dy.astype(np.float32)


def l2_ref(z, dy):
    """float64 of torch's definition F.normalize(F.relu(z), eps) = r / max(|r|, eps), its backward (the clamp passes
    the gradient where |r| >= eps), and the per-element scales |y| and (|g| + |y| sum|y g|) / max(|r|, eps)"""
    r = np.maximum(z.astype(np.float64), 0.0)
    g = dy.astype(np.float64)
    nrm = np.sqrt((r * r).sum(1, keepdims=True))
    nc = np.maximum(nrm, EPS_L2)
    y = r / nc
    live = nrm >= EPS_L2
    dot = (y * g).sum(1, keepdims=True)
    dz = np.where(r > 0, (g - live * y * dot) / nc, 0.0)
    sd = np.where(r > 0, (np.abs(g) + live * np.abs(y) * (np.abs(y * g)).sum(1, keepdims=True)) / nc, 0.0)
    return y, dz, np.abs(y), sd


def g_l2(f):
    """k_relu_l2norm_fwd / _bwd: lane chains of ceil(f / 32) FMAs, 5 butterfly levels, sqrt, the divisions and the
    element's own 3 roundings"""
    return _cdiv(f, 32) + 5 + 6


@pytest.mark.gpu
@pytest.mark.parametrize("f", (1, 31, 32, 33, 218, 1024))
def test_relu_l2norm_per_element(f):
    """y and dz of ReLU + L2-normalise per element against float64 of torch's definition, from norm 1e-13 (clamped)
    to 1e18, at a norm of exactly eps and at 1e13 (where nrm^3 overflows fp32)"""
    from gnn_tableextraction_b200 import ops

    z0, dy0 = l2_rows(f, f)
    y64, dz64, sy, sdz = l2_ref(z0, dy0)
    z, pz = place(_t(z0), True)
    dy, pdy = place(_t(dy0), False)
    G = g_l2(f)
    outs = [place(torch.zeros(z0.shape, device=DEV), True)[0] for _ in range(2)]

    def call():
        for o in outs:
            o.fill_(float("nan"))
        return [ops.relu_l2norm_fwd(z, 1e-12, out=outs[0]), ops.relu_l2norm_bwd(dy, z, 1e-12, out=outs[1])]
    expect = [(_t(y64), _t(K * U * G * sy)), (_t(dz64), _t(K * U * G * sdz))]
    worst = check(call, expect, [pz, pdy], zero_rows_exact=False)
    tie = len(z0) - 4
    got = outs[1][tie:tie + 2].cpu().numpy()
    _log_ratio(f"relu_l2norm f={f} (tie row dz {got[0, 0]:.3e}, 1e13 row dz {got[1, 0]:.3e})", worst)
    assert worst <= 1.0, f"relu_l2norm f={f}: worst bound ratio {worst:.3e}"


@pytest.mark.gpu
def test_relu_l2norm_refuses_wide_rows():
    from gnn_tableextraction_b200 import ops

    z = torch.randn(4, 1025, device=DEV)
    with pytest.raises(ops.GteError):
        ops.relu_l2norm_fwd(z)
    with pytest.raises(ops.GteError):
        ops.relu_l2norm_bwd(z, z)


# ------------------------------------------------------------------- every layer contraction has a bound ---
def _layer_calls():
    """{ops function: [layer functions calling it]} over the four layer functions of layers.py"""
    with open(os.path.join(ROOT, "gnn_tableextraction_b200", "layers.py")) as fh:
        tree = ast.parse(fh.read())
    calls = {}
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef) and fn.name in LAYER_FUNCTIONS:
            for node in ast.walk(fn):
                if (isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute)
                        and isinstance(node.func.value, ast.Name) and node.func.value.id == "ops"):
                    calls.setdefault(node.func.attr, []).append(fn.name)
    return calls


def test_every_layer_kernel_call_has_a_bound():
    """every ops call of the forward, the aggregations and the backward is bounded per element here, in
    test_gpu_grad_numerics.BOUNDS (the reductions over the batch), or is listed in EXEMPT with where it is checked"""
    calls = _layer_calls()
    assert {"spmm", "spmm_packed", "umma_linear_fwd", "linear_bwd_data"} <= set(calls)
    for name, where in sorted(calls.items()):
        assert name in BOUNDS or name in gn.BOUNDS or name in EXEMPT, \
            f"{sorted(set(where))} call ops.{name}, which has no per-element bound"
    assert set(BOUNDS) <= set(calls), f"BOUNDS lists entries the layer no longer calls: {set(BOUNDS) - set(calls)}"


# -------------------------------------------------------------------------------- sharpness of the bounds ---
def _log_margin(tag, margin):
    print(f"{tag}: bound ratio {margin:.3e} (the worst element)")


def _positive(rng, n, f):
    return gn.positive_cols(rng, n, f)


def _spread_rows(rng, n, f, lo, hi):
    return (gn.positive_cols(rng, n, f) * np.exp2(rng.integers(lo, hi + 1, n))[:, None]).astype(np.float32)


def _exact(x, w):
    x64, w64 = x.astype(np.float64), w.astype(np.float64)
    return x64 @ w64.T, np.abs(x64) @ np.abs(w64).T


def _chain_fp32(x, w):
    """fp32 FMA chain over k in order (the FFMA kernels' plan), emulated with float64 products rounded per step"""
    acc = np.zeros((x.shape[0], w.shape[0]), np.float32)
    for k in range(x.shape[1]):
        acc = (acc.astype(np.float64) + np.outer(x[:, k], w[:, k])).astype(np.float32)
    return acc.astype(np.float64)


def _tf32_3x(x, w):
    """3xTF32 per k-step: x split by truncation + rna low part, w by rna + rna low part (gte_umma.cu), the three
    products summed in fp32 per K-step of 8 and accumulated in fp32 (truncation of the accumulator not emulated)"""
    xh = gn.truncate_tf32(x)
    xl = gn.round_tf32(x - xh)
    wh = gn.round_tf32(w)
    wl = gn.round_tf32(w - wh)
    acc = np.zeros((x.shape[0], w.shape[0]), np.float32)
    for k0 in range(0, x.shape[1], 8):
        sl = slice(k0, k0 + 8)
        step = (xh[:, sl].astype(np.float64) @ wh[:, sl].T.astype(np.float64)
                + xh[:, sl].astype(np.float64) @ wl[:, sl].T.astype(np.float64)
                + xl[:, sl].astype(np.float64) @ wh[:, sl].T.astype(np.float64))
        acc = (acc.astype(np.float64) + step.astype(np.float32)).astype(np.float32)
    return acc.astype(np.float64)


def _fwd_operands(seed, n=2048, fin=64, fo=64, ah_binades=(-20, 20)):
    rng = np.random.default_rng(seed)
    h = _spread_rows(rng, n, fin, -20, 20)
    ah = _spread_rows(rng, n, fin, *ah_binades)
    w = (np.abs(rng.standard_normal((fo, 2 * fin))) / np.sqrt(fin) + 0.05).astype(np.float32)
    return np.concatenate([h, ah], 1), w


def test_tf32_single_pass_breaks_the_tensor_core_bound_and_3xtf32_keeps_it():
    """1xTF32 products on both segments break umma_linear_fwd's bound; a 3xTF32 emulation and the FFMA chain keep
    their bounds"""
    x, w = _fwd_operands(1)
    fin = x.shape[1] // 2
    ref, S = _exact(x, w)
    G = BOUNDS["umma_linear_fwd"](fin, 2)[0]
    one = _exact(gn.truncate_tf32(x), gn.truncate_tf32(w))[0]
    margin = _ratio(np.abs(one - ref), K * U * G * S)
    _log_margin(f"1xTF32 on both segments against umma_linear_fwd (G = {G})", margin)
    assert margin >= 10.0, margin
    r3 = _ratio(np.abs(_tf32_3x(x, w) - ref), K * U * G * S)
    _log_ratio("3xTF32 emulation against umma_linear_fwd", r3)
    assert r3 <= 1.0, r3
    Gf = BOUNDS["linear_fwd"](fin, 2)[0]
    rf = _ratio(np.abs(_chain_fp32(x, w) - ref), K * U * Gf * S)
    _log_ratio(f"fp32 FMA chain against linear_fwd (G = {Gf})", rf)
    assert rf <= 1.0, rf


def test_tf32_on_the_neighbour_segment_passes_rel_err_but_breaks_the_bound():
    """1xTF32 on the neighbour block only, on a spread batch whose neighbour rows are at most 2^0 while the self rows
    reach 2^20: within the rel_err < 2e-6 of the parity tests, far outside the per-element bound"""
    x, w = _fwd_operands(2, ah_binades=(-20, 0))
    fin = x.shape[1] // 2
    ref, S = _exact(x, w)
    bad = _exact(x[:, :fin], w[:, :fin])[0] + _exact(gn.truncate_tf32(x[:, fin:]), gn.truncate_tf32(w[:, fin:]))[0]
    rel = np.abs(bad - ref).max() / np.abs(ref).max()
    G = BOUNDS["umma_linear_fwd"](fin, 2)[0]
    margin = _ratio(np.abs(bad - ref), K * U * G * S)
    _log_margin(f"1xTF32 neighbour block: rel_err {rel:.2e}, per-element", margin)
    assert rel < 2e-6 and margin > 10.0, (rel, margin)


def test_dropped_partial_k_block_breaks_the_bound():
    """the last partial k-block (column 32 of fin = 33, both segments: 4 k-blocks, the split accumulator) left out
    breaks umma_linear_fwd's bound, and linear_fwd's"""
    rng = np.random.default_rng(3)
    fin, fo = 33, 17
    x = _positive(rng, 1024, 2 * fin)
    w = (np.abs(rng.standard_normal((fo, 2 * fin))) / np.sqrt(fin) + 0.05).astype(np.float32)
    ref, S = _exact(x, w)
    keep = np.ones(2 * fin, bool)
    keep[[32, fin + 32]] = False
    bad = _exact(x[:, keep], w[:, keep])[0]
    for name in ("umma_linear_fwd", "linear_fwd"):
        G = BOUNDS[name](fin, 2)[0]
        margin = _ratio(np.abs(bad - ref), K * U * G * S)
        _log_margin(f"last partial k-block dropped against {name} (G = {G})", margin)
        assert margin > 10.0, (name, margin)


def _agg_case():
    """CSC of the multigraph (hub row, zero in-degree rows): fp32 norm = 1 / in-degree (0 when isolated) varies from
    row to row, so reading it at the wrong end of an edge changes the sum; positive x"""
    src, dst, w, n, _ = _graph("multi")
    order = np.lexsort((src, dst))
    src, dst, w = src[order], dst[order], w[order]
    deg = np.bincount(dst, minlength=n)
    indptr = np.concatenate([[0], np.cumsum(deg)])
    norm = np.where(deg > 0, (1.0 / np.maximum(deg, 1)).astype(np.float32), 0.0).astype(np.float32)
    x = _positive(np.random.default_rng(4), n, 8)
    return src, dst, w, n, deg, indptr, norm, x


def _agg_sum(src, dst, wt, x, n):
    y = np.zeros((n, x.shape[1]))
    np.add.at(y, dst, wt[:, None].astype(np.float64) * x[src].astype(np.float64))
    return y


def _agg_chain_fp32(indptr, src, wt, x, n):
    """one fp32 FMA chain per row over its edges in CSC order (the kernels' plan)"""
    y = np.zeros((n, x.shape[1]), np.float32)
    for r in range(n):
        acc = np.zeros(x.shape[1], np.float32)
        for e in range(indptr[r], indptr[r + 1]):
            acc = (acc.astype(np.float64) + np.float64(wt[e]) * x[src[e]].astype(np.float64)).astype(np.float32)
        y[r] = acc
    return y.astype(np.float64)


def test_aggregation_defects_break_the_bound_and_the_chain_keeps_it():
    """in A_hat^T dz (sum of w_e norm[src] x[src] per row): one edge dropped per row and the source scale read at the
    destination (norm[dst]) break the bound; the fp32 chain in CSC order with w * norm rounded first keeps it"""
    src, dst, w, n, deg, indptr, norm, x = _agg_case()
    wt = (w * norm[src]).astype(np.float32)  # the rounded w * pre_scale the kernel uses
    ref = _agg_sum(src, dst, wt, x, n)
    S = _agg_sum(src, dst, np.abs(wt), np.abs(x), n)
    G = np.asarray([BOUNDS["spmm"](d, True) for d in deg], np.float64)[:, None]
    bound = K * U * G * S
    chain = _agg_chain_fp32(indptr, src, wt, x, n)
    r = _ratio(np.abs(chain - ref), bound)
    _log_ratio("fp32 chain in CSC order against spmm", r)
    assert r <= 1.0, r
    last = indptr[1:][deg > 0] - 1
    keep = np.ones(len(src), bool)
    keep[last] = False
    keep[w == 0] = True  # a zero-weight edge changes nothing: drop the row's last non-trivial edge instead
    dropped = _agg_sum(src[keep], dst[keep], wt[keep], x, n)
    margin = _ratio(np.abs(dropped - ref), bound)
    _log_margin("one edge dropped per row against spmm", margin)
    assert margin > 10.0, margin
    wdst = (w * norm[dst]).astype(np.float32)
    margin = _ratio(np.abs(_agg_sum(src, dst, wdst, x, n) - ref), bound)
    _log_margin("pre_scale taken at the destination against spmm", margin)
    assert margin > 10.0, margin


def _l2_bwd_fp32(z, dy, old):
    """the backward in fp32 (numpy, sequential sums): old = the former d = g/nrm - r (r.g) / nrm^3 taken only when
    nrm > eps; new = (g - y (y.g)) / nrm taken when nrm >= eps"""
    f32 = np.float32
    r = np.maximum(z, f32(0))
    g = dy
    with np.errstate(over="ignore", invalid="ignore"):
        nrm = np.sqrt((r * r).sum(1, dtype=f32, keepdims=True)).astype(f32)
        eps = f32(EPS_L2)
        if old:
            clamped = ~(nrm > eps)
            nc = np.where(clamped, eps, nrm).astype(f32)
            dot = (r * g).sum(1, dtype=f32, keepdims=True).astype(f32)
            d = (g / nc).astype(f32) - np.where(clamped, f32(0), (r * dot / (nc * nc * nc)).astype(f32))
        else:
            clamped = nrm < eps
            nc = np.where(clamped, eps, nrm).astype(f32)
            y = (r / nc).astype(f32)
            dot = np.where(clamped, f32(0), (y * g).sum(1, dtype=f32, keepdims=True)).astype(f32)
            d = ((g - y * dot) / nc).astype(f32)
    return np.where(r > 0, d, f32(0)).astype(np.float64)


def test_old_relu_l2norm_backward_breaks_the_bound_at_the_tie_and_1e13_rows():
    """the former nrm^3 backward breaks the per-element bound at the row of norm exactly eps (it took the clamped
    branch) and at the row of norm 1e13 (nrm^3 overflows); the formula without powers of the norm keeps it"""
    z = np.array([[EPS_L2, 0.0, -1.0], [1e13, 2e13, 5e12]], np.float32)
    dy = np.array([[1.0, 2.0, 3.0], [1.0, 2.0, 3.0]], np.float32)
    _, dz64, _, sdz = l2_ref(z, dy)
    bound = K * U * g_l2(3) * sdz
    for row, tag in ((0, "norm = eps"), (1, "norm 1e13")):
        margin = _ratio(np.abs(_l2_bwd_fp32(z, dy, True)[row] - dz64[row]), bound[row])
        _log_margin(f"old nrm^3 backward at the {tag} row", margin)
        assert margin > 10.0, (tag, margin)
    zs, dys = l2_rows(33, 5)
    _, dz64, _, sdz = l2_ref(zs, dys)
    r = _ratio(np.abs(_l2_bwd_fp32(zs, dys, False) - dz64), K * U * g_l2(33) * sdz)
    _log_ratio("fp32 emulation of the new backward on every test row", r)
    assert r <= 1.0, r
