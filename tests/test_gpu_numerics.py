"""Per-row float64 error bounds of the cross-entropy and LayerNorm kernels on shifted and ill-conditioned rows.

The parity tests elsewhere feed well-scaled random rows and measure max|a-b| / max|b| over a whole tensor.  That metric
hides an error confined to a few rows, and well-scaled rows never reach the formulas that lose accuracy with a common
offset, a near-zero variance or an extreme logit.  Here every value is checked against float64 computed from the fp32
values the kernel itself read or wrote (for LayerNorm: the kernel's own z, so GEMM rounding is not counted against the
statistics), under a bound derived per row (or per element) from the operation's conditioning.  Each test prints its
worst bound ratio (pytest -rP).

The CPU tests at the end emulate, in numpy fp32, the formulas these bounds exist to reject -- the one-pass variance
E[z^2] - E[z]^2 and the loss (max + log-sum-exp) - x_y -- and assert that they violate the bounds on the same rows, while
the stable forms pass: the bounds are tight enough to catch the defects they target.
"""
import numpy as np
import pytest
import torch

DEV = "cuda"
U = 2.0 ** -24  # unit roundoff of fp32
# Constant of every bound in this file.  The tensor-core epilogues sum a row of up to 256 values sequentially in one
# thread; on rows that repeat one value those rounding errors add up linearly, and the one-accumulator pair kernel's
# one-pass sums around the first chunk's mean amplify them by 1 + (shift - mean)^2 / var: its two-level rows at
# fo = 250 and 256 reach 0.98 to 1.02 times the bounds with K = 32 on a B200.
K = 64.0
EPS = float(np.float32(1e-5))  # the LayerNorm eps as the kernels receive it


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


# ------------------------------------------------------------------------------------------ cross entropy ---
CE_SHIFTS = (0.0, 30.0, -30.0, 1e3, 1e4, -1e4)
CE_CLASSES = (1, 2, 9, 16, 17, 64)
LABEL_DTYPES = (torch.int64, torch.int32, torch.float32)


def ce_rows(c, n, shift, seed=0):
    """fp32 logits [n, c] built from the same base rows for every shift, in four kinds cycling over the rows: plain
    (randn * 3), confident (label logit 10-20 above the rest), hopeless (label logit 150 below the maximum: its exp
    underflows), -inf in some non-label columns; labels int64 with a few -1 (padding) and c (out of range)"""
    rng = np.random.default_rng(seed * 1000 + c)
    base = rng.standard_normal((n, c)) * 3
    y = rng.integers(0, c, n)
    rows = np.arange(n)
    kind = rows % 4
    if c > 1:
        others = base.copy()
        others[rows, y] = -np.inf
        omax = others.max(1)
        conf = kind == 1
        base[rows[conf], y[conf]] = omax[conf] + rng.uniform(10, 20, conf.sum())
        hope = kind == 2
        base[rows[hope], y[hope]] = omax[hope] - 150
    x = (base + shift).astype(np.float32)
    if c > 2:
        for i in rows[kind == 3]:
            cols = rng.choice(np.delete(np.arange(c), y[i]), size=max(1, (c - 1) // 3), replace=False)
            x[i, cols] = -np.inf
    y[rows % 13 == 5] = -1
    y[rows % 17 == 7] = c
    return x, y


def class_weights(c, seed=0):
    w = np.random.default_rng(seed + c).uniform(0.25, 2.0, c).astype(np.float32)
    w[::3] = 0.0  # class weights that include 0
    return w


def ce_ref(x, y, w):
    """float64 per-row nll, its bound K u (1 + log se + |x_y - mx|) (both 0 for labels outside [0, c)), label weight
    (0 for those labels) and softmax of fp32 logits x [n, c]"""
    n, c = x.shape
    x64 = x.astype(np.float64)
    mx = x64.max(1)
    e = np.exp(x64 - mx[:, None])
    se = e.sum(1)
    valid = (y >= 0) & (y < c)
    yc = np.where(valid, y, 0)
    dist = np.where(valid, x64[np.arange(n), yc] - mx, 0.0)
    nll = np.where(valid, np.log(se) - dist, 0.0)  # rows without a label contribute nothing
    bound = np.where(valid, K * U * (1.0 + np.log(se) + np.abs(dist)), 0.0)
    wy = np.where(valid, (np.ones(c) if w is None else w.astype(np.float64))[yc], 0.0)
    return nll, bound, wy, e / se[:, None], valid


def nll_fp32_old(x, y):
    """the former kernel's nll in fp32: (mx + logf(se)) - x_y"""
    mx = x.max(1)
    se = np.exp(x - mx[:, None]).astype(np.float32).sum(1, dtype=np.float32)
    return (mx + np.log(se).astype(np.float32)).astype(np.float32) - x[np.arange(len(y)), y]


def nll_fp32_stable(x, y):
    """the kernel's nll in fp32: logf(se) - (x_y - mx)"""
    mx = x.max(1)
    se = np.exp(x - mx[:, None]).astype(np.float32).sum(1, dtype=np.float32)
    return np.log(se).astype(np.float32) - (x[np.arange(len(y)), y] - mx).astype(np.float32)


def _labels_dev(y, dtype):
    return torch.as_tensor(y).to(dtype).to(DEV)


def _argmax(x):
    """torch.argmax of each row: the first maximal index, NaN counting as maximal"""
    return torch.from_numpy(x).argmax(1).numpy()


N_CE = 1500
SAMPLE = (0, 1, 2, 3, 5, 7, 255, 256, 257, 1022, 1023, N_CE - 1)  # every row kind, both label paddings, block edges


@pytest.mark.gpu
@pytest.mark.parametrize("shift", CE_SHIFTS)
@pytest.mark.parametrize("c", CE_CLASSES)
def test_cross_entropy_fwd_and_eval_per_row_bounds(c, shift):
    """cross_entropy_fwd and eval_accumulate on one-row views and on the whole batch, every label dtype, with and
    without class weights: per-row |w nll - w nll64| <= w K u (1 + log se + |x_y - mx|), the batch at the sum of the
    row bounds; #correct and the confusion counts exact"""
    from gnn_tableextraction_b200 import ops

    x, y = ce_rows(c, N_CE, shift)
    nll64, bnd, _, _, valid = ce_ref(x, y, None)
    pred = _argmax(x)
    xd = torch.from_numpy(x).to(DEV)
    worst = 0.0
    for w in (None, class_weights(c)):
        _, _, wy, _, _ = ce_ref(x, y, w)
        wd = None if w is None else torch.from_numpy(w).to(DEV)
        for dt in LABEL_DTYPES:
            yd = _labels_dev(y, dt)
            # one-row views: the per-row values
            rows = [i for i in SAMPLE if i < N_CE]
            stats = torch.empty((len(rows), 4), dtype=torch.float32, device=DEV)
            totals = torch.zeros((len(rows), 2 + c * c), dtype=torch.float64, device=DEV)
            for k, i in enumerate(rows):
                ops.cross_entropy_fwd(xd[i:i + 1], yd[i:i + 1], wd, stats[k, :3])
                ops.eval_accumulate(xd[i:i + 1], yd[i:i + 1], wd, totals[k])
            st, tt = stats[:, :3].double().cpu().numpy(), totals.cpu().numpy()
            r = np.array(rows)
            for got in (st[:, 0], tt[:, 0]):
                worst = max(worst, _ratio(np.abs(got - wy[r] * nll64[r]), wy[r] * bnd[r]))
                assert np.all(got[wy[r] == 0] == 0.0)
            assert np.array_equal(st[:, 1], wy[r].astype(np.float32)) and np.array_equal(tt[:, 1], wy[r].astype(np.float32))
            assert np.array_equal(st[:, 2], (pred[r] == y[r]).astype(np.float64))
            cm = np.zeros((len(rows), c * c))
            vr = valid[r]
            cm[np.arange(len(rows))[vr], (y[r] * c + pred[r])[vr]] = 1.0
            assert np.array_equal(tt[:, 2:], cm)
            # the whole batch
            s = ops.cross_entropy_fwd(xd, yd, wd).double().cpu().numpy()
            tot = torch.zeros(2 + c * c, dtype=torch.float64, device=DEV)
            ops.eval_accumulate(xd, yd, wd, tot)
            tot = tot.cpu().numpy()
            for got in (s[0], tot[0]):
                worst = max(worst, _ratio(abs(got - np.sum(wy * nll64)), np.sum(wy * bnd)))
            for got in (s[1], tot[1]):
                worst = max(worst, _ratio(abs(got - np.sum(wy)), K * U * np.sum(wy)))
            assert s[2] == np.sum(pred == y)
            assert np.array_equal(tot[2:], np.bincount((y * c + pred)[valid], minlength=c * c).astype(np.float64))
    _log_ratio(f"ce fwd/eval c={c} shift={shift:g}", worst)
    assert worst <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("shift", CE_SHIFTS)
@pytest.mark.parametrize("c", CE_CLASSES)
def test_cross_entropy_bwd_per_element_bounds(c, shift):
    """cross_entropy_bwd and cross_entropy_bwd_comb (k_ce_bwd_comb32 at width 32, the padded kernel at other widths):
    |d - d64| <= K u |w_y / den| (p64_j (1 + |x_j - mx|) + [j = y]) -- fl(x_j - mx) is off by up to u |x_j - mx|, which
    exp turns into a relative error of p_j; rows with a label outside [0, c) and the padding columns are exactly 0; a
    one-row view gives the bits of its row in the batch"""
    from gnn_tableextraction_b200 import ops

    x, y = ce_rows(c, N_CE, shift, seed=1)
    w = class_weights(c, seed=1)
    _, _, wy, p64, valid = ce_ref(x, y, w)
    den = np.float32(max(np.sum(wy), 1.0) * 0.75)  # any positive scalar: a data-parallel step divides by a global sum
    scale = wy / np.float64(den)
    onehot = np.arange(c)[None, :] == y[:, None]
    ref = scale[:, None] * (p64 - onehot)
    dist = np.abs(x.astype(np.float64) - x.max(1).astype(np.float64)[:, None])
    bound = K * U * np.abs(scale)[:, None] * (np.where(p64 > 0, p64 * (1.0 + dist), 0.0) + onehot)
    xd = torch.from_numpy(x).to(DEV)
    wd, dend = torch.from_numpy(w).to(DEV), torch.tensor([den], dtype=torch.float32, device=DEV)
    widths = [None, 12 if c <= 12 else (c + 3) // 4 * 4] + ([32] if c <= 16 else [])  # 32: k_ce_bwd_comb32
    worst = 0.0
    for k, width in enumerate(widths):
        yd = _labels_dev(y, LABEL_DTYPES[k % 3])
        run = (lambda a, b: ops.cross_entropy_bwd(a, b, wd, dend)) if width is None else (
            lambda a, b: ops.cross_entropy_bwd_comb(a, b, wd, dend, width=width))
        out = run(xd, yd)
        d = out[:, :c].double().cpu().numpy()
        worst = max(worst, _ratio(np.abs(d - ref), bound))
        assert np.all(d[~valid] == 0.0)
        if width is not None:
            assert torch.all(out[:, c:] == 0)
        for i in SAMPLE:
            assert torch.equal(run(xd[i:i + 1], yd[i:i + 1]), out[i:i + 1]), (width, i)
    _log_ratio(f"ce bwd c={c} shift={shift:g} widths={widths}", worst)
    assert worst <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("c", (1, 2, 9, 64))
def test_argmax_nan_rows_match_torch(c):
    """#correct of cross_entropy_fwd, the confusion counts of eval_accumulate and page_predictions all take
    torch.argmax: the first maximal index, NaN counting as maximal; ties and NaN in any column"""
    from gnn_tableextraction_b200 import ops

    rng = np.random.default_rng(c)
    n = 700
    x = rng.integers(-3, 4, (n, c)).astype(np.float32)  # small integers: many ties
    nan_rows = rng.random(n) < 0.5
    x[nan_rows, rng.integers(0, c, n)[nan_rows]] = np.nan
    y = rng.integers(0, c, n)
    y[::11] = -1
    pred = _argmax(x)
    valid = y >= 0
    xd = torch.from_numpy(x).to(DEV)
    for dt in LABEL_DTYPES:
        yd = _labels_dev(y, dt)
        assert ops.cross_entropy_fwd(xd, yd)[2].item() == np.sum(pred == y)
        tot = torch.zeros(2 + c * c, dtype=torch.float64, device=DEV)
        ops.eval_accumulate(xd, yd, None, tot)
        assert np.array_equal(tot[2:].cpu().numpy(), np.bincount((y * c + pred)[valid], minlength=c * c))
    page_off = np.array([0, 1, 130, 131, 400, n], np.int32)
    preds, correct = ops.page_predictions(xd, torch.from_numpy(page_off).to(DEV), len(page_off) - 1,
                                          _labels_dev(y, torch.int64))
    assert np.array_equal(preds.cpu().numpy(), pred)
    hit = (pred == y).astype(np.int64)
    assert np.array_equal(correct.cpu().numpy(), [hit[a:b].sum() for a, b in zip(page_off[:-1], page_off[1:])])


@pytest.mark.gpu
@pytest.mark.parametrize("c", CE_CLASSES)
def test_page_predictions_shifted_rows(c):
    """page_predictions on every row kind and shift of the cross-entropy tests (ties of -inf, confident and hopeless
    rows): predictions and per-page counts exact, on one-row pages too"""
    from gnn_tableextraction_b200 import ops

    for shift in CE_SHIFTS:
        x, y = ce_rows(c, N_CE, shift)
        pred = _argmax(x)
        xd = torch.from_numpy(x).to(DEV)
        page_off = np.array([0, 1, 2, 3, 77, 256, 257, 1000, N_CE], np.int32)
        for dt in LABEL_DTYPES:
            preds, correct = ops.page_predictions(xd, torch.from_numpy(page_off).to(DEV), len(page_off) - 1,
                                                  _labels_dev(y, dt))
            assert np.array_equal(preds.cpu().numpy(), pred), (shift, dt)
            hit = (pred == y).astype(np.int64)
            assert np.array_equal(correct.cpu().numpy(), [hit[a:b].sum() for a, b in zip(page_off[:-1], page_off[1:])])


# ---------------------------------------------------------------------------------------------- LayerNorm ---
def ln_ref(z, gamma, beta, relu):
    """float64 LayerNorm of the kernel's fp32 z [n, f]: mean, rstd, x_hat, y and kappa_r = max_k |z_rk| rstd_r"""
    z64 = z.astype(np.float64)
    mean = z64.mean(1)
    rstd = 1.0 / np.sqrt(((z64 - mean[:, None]) ** 2).mean(1) + EPS)
    xh = (z64 - mean[:, None]) * rstd[:, None]
    y = xh * gamma.astype(np.float64) + beta.astype(np.float64)
    if relu:
        y = np.maximum(y, 0.0)
    kappa = np.abs(z64).max(1) * rstd
    return mean, rstd, xh, y, kappa


def ln_ratio(z, y, mean, rstd, gamma, beta, relu):
    """worst ratio over the forward bounds
         |y - y64|          <= K u (|gamma_j| (kappa_r + |x_hat_rj|) + |beta_j|)
         |mean - mean64|    <= K u kappa_r / rstd64_r        (= K u max_k |z_rk|)
         |rstd - rstd64|    <= K u (1 + kappa_r) rstd64_r"""
    m64, r64, xh, y64, kap = ln_ref(z, gamma, beta, relu)
    g, b = np.abs(gamma.astype(np.float64)), np.abs(beta.astype(np.float64))
    ry = _ratio(np.abs(y.astype(np.float64) - y64), K * U * (g * (kap[:, None] + np.abs(xh)) + b))
    rm = _ratio(np.abs(mean.astype(np.float64) - m64), K * U * kap / r64)
    rr = _ratio(np.abs(rstd.astype(np.float64) - r64), K * U * (1.0 + kap) * r64)
    return max(ry, rm, rr)


# Row kinds of the LayerNorm tests.  The offset C of a row is up to 1e4 times its spread; "two" rows hold one level in
# their first m columns and random values at another level in the rest ("mirror": the other way round) -- with m the
# columns of the first half of the pair kernel's split accumulator, whose merge then sees a large delta; "sym" rows are
# pairs C +- t and, in an odd row, C itself: elements at the ReLU kink when beta = 0.
LN_KINDS = (("shift", 0.0, 1.0), ("shift", 3e2, 0.5), ("shift", -5e3, 0.5), ("shift", 1e4, 1.0), ("const", 7e2, 0.0),
            ("const", 0.0, 0.0), ("two", 4e3, 0.5), ("mirror", -2e3, 0.25), ("sym", 1e3, 1.0), ("sym", 0.0, 1.0))


def split_cols(f):
    """columns of the first half of the pair kernel's split accumulator: c_split = ceil(chunks / 2) 32-float chunks"""
    return min(f, ((f + 31) // 32 + 1) // 2 * 32)


def kind_layout(kind, f, level):
    """(per-column offset b [f], random-column mask [f], signs of the random part [f] or None) of a row kind: a row
    is b + sigma * (random part), where the random part of "sym" rows comes in +- pairs"""
    m = split_cols(f)
    b = np.full(f, level)
    rand = np.ones(f, bool)
    if kind == "const":
        rand[:] = False
    elif kind == "two":
        rand[:m] = False
        b[m:] = -level / 2
    elif kind == "mirror":
        rand[m:] = False
        b[m:] = -level / 2 + 1.0
    elif kind == "sym":
        rand[-1] = f % 2 == 0
    return b, rand


def ln_params(f, rng, beta_zero):
    gamma = (rng.random(f) + 0.5).astype(np.float32)
    gamma[::7] = 0.0  # gamma values including 0
    gamma[1::5] *= -1
    beta = np.zeros(f, np.float32) if beta_zero else (rng.standard_normal(f) * 0.5).astype(np.float32)
    return gamma, beta


def ln_rows(kind, level, sigma, n, f, rng):
    """fp32 z [n, f] of one row kind (the row-wise kernel's input)"""
    b, rand = kind_layout(kind, f, level)
    r = rng.standard_normal((n, f))
    if kind == "sym":
        r[:, 1::2] = -r[:, 0:(f // 2) * 2:2]
    return (b[None, :] + sigma * r * rand[None, :]).astype(np.float32)


def ln_fp32_naive(z, gamma, beta, relu):
    """numpy fp32 emulation of the one-pass statistics E[z^2] - E[z]^2 (clamped at 0)"""
    f = np.float32(z.shape[1])
    mean = z.sum(1, dtype=np.float32) / f
    var = np.maximum((z * z).sum(1, dtype=np.float32) / f - mean * mean, np.float32(0))
    rstd = np.float32(1) / np.sqrt(var + np.float32(EPS))
    y = ((z - mean[:, None]) * rstd[:, None] * gamma + beta).astype(np.float32)
    return (np.maximum(y, 0) if relu else y), mean, rstd


def ln_fp32_two_pass(z, gamma, beta, relu):
    """numpy fp32 emulation of the two-pass statistics of the kernels"""
    f = np.float32(z.shape[1])
    mean = z.sum(1, dtype=np.float32) / f
    d = z - mean[:, None]
    rstd = np.float32(1) / np.sqrt((d * d).sum(1, dtype=np.float32) / f + np.float32(EPS))
    y = (d * rstd[:, None] * gamma + beta).astype(np.float32)
    return (np.maximum(y, 0) if relu else y), mean, rstd


def _dev_aligned(a):
    """device copy with 16-byte aligned rows padded to 4 floats (the 128-bit backward kernel takes these)"""
    from gnn_tableextraction_b200 import ops

    t = ops.empty_padded(a.shape[0], a.shape[1], DEV)
    t.copy_(torch.as_tensor(a))
    return t


def _dev_unaligned(a):
    """device copy whose rows are packed and start 4 bytes past a 16-byte boundary (the scalar backward kernel)"""
    n, f = a.shape
    buf = torch.empty(n * f + 1, dtype=torch.float32, device=DEV)
    t = buf[1:].view(n, f)
    t.copy_(torch.as_tensor(a))
    return t


def mask_check(z, y, mean, rstd, gamma, beta, relu):
    """layernorm_act_bwd with dy = 1 on aligned (128-bit kernel up to f = 480) and unaligned (scalar kernel) operands:
    dbeta[j] must equal #(y[:, j] > 0) exactly (ReLU) or n; dz and dgamma against the float64 backward under the CUDA
    mask.  Returns the worst bound ratio of dz / dgamma."""
    from gnn_tableextraction_b200 import ops

    n, f = z.shape
    m64, r64, xh, _, kap = ln_ref(z, gamma, beta, relu)
    g = (y > 0).astype(np.float64) if relu else np.ones((n, f))
    a = g * gamma.astype(np.float64)
    c1, c2 = a.mean(1), (a * xh).mean(1)
    dz64 = r64[:, None] * (a - c1[:, None] - xh * c2[:, None])
    dg64 = (g * xh).sum(0)
    amax, xmax = np.abs(a).max(1), np.abs(xh).max(1)
    bz = K * U * (r64 * amax * (1.0 + kap) * (1.0 + xmax) ** 2)[:, None]
    bg = K * U * (g * (1.0 + kap[:, None]) * (1.0 + np.abs(xh))).sum(0)
    md, rd, gd, bd = (torch.from_numpy(v).to(DEV) for v in (mean, rstd, gamma, beta))
    worst = 0.0
    for place in (_dev_aligned, _dev_unaligned):
        zd, dyd = place(z), place(np.ones((n, f), np.float32))
        dgamma, dbeta = torch.empty(f, device=DEV), torch.empty(f, device=DEV)
        dz = ops.layernorm_act_bwd(dyd, zd, md, rd, gd, bd, relu, dgamma, dbeta).cpu().numpy()
        assert np.array_equal(dbeta.cpu().numpy(), g.sum(0)), f"ReLU mask of the backward differs ({place.__name__})"
        worst = max(worst, _ratio(np.abs(dz - dz64), bz), _ratio(np.abs(dgamma.cpu().numpy() - dg64), bg))
    return worst


def _outputs(*ts):
    return [t.cpu().numpy() for t in ts]


LN_F = (1, 9, 31, 32, 33, 218, 256, 257, 481, 1000, 1024)


@pytest.mark.gpu
@pytest.mark.parametrize("f", LN_F)
def test_layernorm_act_fwd_row_bounds_and_relu_mask(f):
    """layernorm_act_fwd (two-pass statistics) on every row kind, both ReLU settings; the backward's ReLU mask
    recomputed from the saved mean / rstd equals the forward's y > 0 on both backward kernels"""
    from gnn_tableextraction_b200 import ops

    rng = np.random.default_rng(f)
    n = 77
    fw = bw = 0.0
    for i, (kind, level, sigma) in enumerate(LN_KINDS):
        relu = i % 2 == 0 or kind == "sym"
        gamma, beta = ln_params(f, rng, beta_zero=kind in ("sym", "const"))
        z = ln_rows(kind, level, sigma, n, f, rng)
        y, mean, rstd = ops.layernorm_act_fwd(_dev_aligned(z), torch.from_numpy(gamma).to(DEV),
                                              torch.from_numpy(beta).to(DEV), EPS, relu)
        y, mean, rstd = _outputs(y, mean, rstd)
        fw = max(fw, ln_ratio(z, y, mean, rstd, gamma, beta, relu))
        bw = max(bw, mask_check(z, y, mean, rstd, gamma, beta, relu))
    _log_ratio(f"layernorm_act_fwd f={f} forward", fw)
    _log_ratio(f"layernorm_act_bwd f={f} dz/dgamma", bw)
    assert fw <= 1.0 and bw <= 1.0


def linear_case(kind, level, sigma, n, k, f, rng):
    """(X [n, k], W [f, k], b [f]) whose z = X W^T + b has the structure of ln_rows(kind): the offsets come through
    the bias, the random columns through W (zero rows of W give constant columns, negated rows the +- pairs)"""
    b, rand = kind_layout(kind, f, level)
    X = rng.standard_normal((n, k)).astype(np.float32)
    W = rng.standard_normal((f, k)) * (sigma / np.sqrt(k))
    if kind == "sym":
        W[1::2] = -W[0:(f // 2) * 2:2]
    W[~rand] = 0.0
    return X, W.astype(np.float32), b.astype(np.float32)


def _run_linear_cases(tag, f, run, k):
    """run(X, W, b, gamma, beta, relu) -> (z, y, mean, rstd) on every row kind: forward bounds and ReLU mask"""
    rng = np.random.default_rng(f * 7 + k)
    fw = bw = 0.0
    for i, (kind, level, sigma) in enumerate(LN_KINDS):
        relu = i % 2 == 0 or kind == "sym"
        gamma, beta = ln_params(f, rng, beta_zero=kind in ("sym", "const"))
        X, W, b = linear_case(kind, level, sigma, 300, k, f, rng)
        z, y, mean, rstd = _outputs(*run(X, W, b, gamma, beta, relu))
        fw = max(fw, ln_ratio(z, y, mean, rstd, gamma, beta, relu))
        bw = max(bw, mask_check(z, y, mean, rstd, gamma, beta, relu))
    _log_ratio(f"{tag} forward", fw)
    _log_ratio(f"{tag} backward dz/dgamma", bw)
    assert fw <= 1.0 and bw <= 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("f", (17, 96, 218, 256))
def test_wide_out_layernorm_row_bounds_and_relu_mask(f):
    """wide_out(fuse_ln): two-pass statistics in registers after the narrow-contraction product"""
    from gnn_tableextraction_b200 import ops

    k1 = k2 = 13

    def run(X, W, b, gamma, beta, relu):
        Wd = torch.from_numpy(W).to(DEV)  # [f, k1 + k2]: element (j, c) of B at j + c * (k1 + k2)
        z, y, mean, rstd = ops.wide_out(_dev_aligned(X[:, :k1]), _dev_aligned(X[:, k1:]), Wd.data_ptr(),
                                        Wd.data_ptr() + 4 * k1, 1, k1 + k2, f, torch.from_numpy(b).to(DEV),
                                        gamma=torch.from_numpy(gamma).to(DEV), beta=torch.from_numpy(beta).to(DEV),
                                        eps=EPS, relu=relu, fuse_ln=True)
        return z, y, mean, rstd

    _run_linear_cases(f"wide_out f={f}", f, run, k1 + k2)


def _umma_run(ops, fin, nseg, fo):
    def run(X, W, b, gamma, beta, relu):
        pack = ops.umma_pack_weights(torch.from_numpy(W).to(DEV), fin, nseg)
        x1 = _dev_aligned(X[:, :fin])
        x2 = _dev_aligned(X[:, fin:]) if nseg == 2 else None
        return ops.umma_linear_fwd(x1, x2, fin, pack, torch.from_numpy(b).to(DEV), fo,
                                   gamma=torch.from_numpy(gamma).to(DEV), beta=torch.from_numpy(beta).to(DEV), eps=EPS,
                                   relu=relu, fuse_ln=True, want_y=True)
    return run


# one and two segments on both sides of the split-accumulator threshold (more than two 32-float k-blocks in all)
UMMA_K = ((1, 64, False), (1, 65, True), (2, 32, False), (2, 33, True))


@pytest.mark.gpu
@pytest.mark.parametrize("nseg,fin,split", UMMA_K)
@pytest.mark.parametrize("fo", (17, 32, 33, 96, 218, 250, 256))
def test_umma_linear_fwd_layernorm_row_bounds_and_relu_mask(fo, nseg, fin, split, umma_kernel):
    """umma_linear_fwd(fuse_ln): two passes over TMEM (single-CTA kernel), per-half shifted sums merged with the
    parallel-variance formula (pair kernel, split accumulator) or one shifted pass (pair kernel, one accumulator)"""
    from gnn_tableextraction_b200 import ops

    if not ops.umma_supported(fo, fin):
        pytest.skip(f"umma_supported({fo}, {fin}) is false")
    _run_linear_cases(f"umma [{umma_kernel}] fo={fo} nseg={nseg} fin={fin} split={split}", fo,
                      _umma_run(ops, fin, nseg, fo), nseg * fin)


@pytest.mark.gpu
@pytest.mark.parametrize("fin,fo", ((13, 218), (16, 33), (4, 256)))
def test_umma_linear_fwd_comb_layernorm_row_bounds_and_relu_mask(fin, fo, umma_kernel):
    """umma_linear_fwd_comb(fuse_ln): the combined [h | A_hat h] operand of a narrow input layer"""
    from gnn_tableextraction_b200 import ops

    def run(X, W, b, gamma, beta, relu):
        pack = ops.umma_pack_weights(torch.from_numpy(W).to(DEV), fin, 2)
        xc = ops.comb_buffer(X.shape[0], DEV)
        xs, xn = ops.comb_views(xc, fin)
        xs.copy_(torch.from_numpy(X[:, :fin]))
        xn.copy_(torch.from_numpy(X[:, fin:]))
        return ops.umma_linear_fwd_comb(xc, fin, pack, torch.from_numpy(b).to(DEV), fo,
                                        gamma=torch.from_numpy(gamma).to(DEV), beta=torch.from_numpy(beta).to(DEV),
                                        eps=EPS, relu=relu, fuse_ln=True, want_y=True)

    _run_linear_cases(f"umma_comb [{umma_kernel}] fin={fin} fo={fo}", fo, run, 2 * fin)


# -------------------------------------------------------------------------------- sharpness of the bounds ---
def test_nll_bound_rejects_the_offset_sensitive_formula():
    """(mx + logf(se)) - x_y breaks the nll bound on the shifted rows of the GPU tests at s = 1e4, while
    logf(se) - (x_y - mx) in the same fp32 arithmetic stays within it at every shift"""
    c = 9
    worst_old = 0.0
    for shift in CE_SHIFTS:
        x, y = ce_rows(c, N_CE, shift)
        valid = (y >= 0) & (y < c)
        x, y = x[valid & np.isfinite(x).all(1)], y[valid & np.isfinite(x).all(1)]
        nll64, bnd, _, _, _ = ce_ref(x, y, None)
        stable = _ratio(np.abs(nll_fp32_stable(x, y) - nll64), bnd)
        assert stable <= 1.0, (shift, stable)
        old = _ratio(np.abs(nll_fp32_old(x, y) - nll64), bnd)
        if abs(shift) >= 1e4:
            assert old > 1.0, (shift, old)
            worst_old = max(worst_old, old)
    _log_ratio("nll of (mx + logf(se)) - x_y in fp32 at |s| = 1e4", worst_old)


def test_layernorm_bound_rejects_one_pass_variance():
    """E[z^2] - E[z]^2 breaks the LayerNorm bounds on the offset rows of the GPU tests, while the two-pass form in the
    same fp32 arithmetic stays within them"""
    rng = np.random.default_rng(0)
    for f in (218, 256):
        for kind, level, sigma in LN_KINDS:
            gamma, beta = ln_params(f, rng, beta_zero=False)
            z = ln_rows(kind, level, sigma, 64, f, rng)
            two = ln_ratio(z, *ln_fp32_two_pass(z, gamma, beta, False), gamma, beta, False)
            assert two <= 1.0, (f, kind, level, two)
            naive = ln_ratio(z, *ln_fp32_naive(z, gamma, beta, False), gamma, beta, False)
            if kind == "shift" and abs(level) / sigma >= 1e4:
                assert naive > 1.0, (f, kind, level, naive)
                _log_ratio(f"one-pass variance f={f} C/sigma={abs(level) / sigma:g}", naive)
