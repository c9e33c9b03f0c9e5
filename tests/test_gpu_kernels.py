"""GPU parity tests of the individual C-ABI entry points against the CPU oracle
(bit-exact for the integer formats, <= 1e-5 relative -- usually 1e-6 -- for fp32)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import TOL, rel_err
from gnn_tableextraction_b200 import _lib, ops, synth
from oracle import csx
from oracle import sage_oracle as so

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _i32(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.int32, device=DEV)


def _f32(a):
    return torch.as_tensor(np.asarray(a), dtype=torch.float32, device=DEV)


def _padded(t):
    """copy a CPU [n, f] tensor into a 16-byte-aligned padded device view"""
    out = ops.empty_padded(t.shape[0], t.shape[1], DEV)
    out.copy_(t)
    return out


# ----------------------------------------------------------- formats --------
@pytest.mark.parametrize("n,e,seed", [(1, 0, 0), (5, 0, 1), (1, 7, 2), (50, 400, 3), (1000, 20000, 4), (37, 5000, 5),
                                      (200_000, 1_000_000, 6)])
def test_csx_from_coo_bit_exact(n, e, seed):
    src, dst, _ = synth.random_multigraph(seed, n, e) if e else (np.zeros(0, np.int32),) * 2 + (None,)
    for key, other in ((dst, src), (src, dst)):  # CSC and CSR
        ip, ix, ei = csx.csx_from_coo(key, other, n)
        gp, gx, ge = ops.csx_from_coo(_i32(key), _i32(other), n)
        assert np.array_equal(gp.cpu().numpy(), ip)
        assert np.array_equal(gx.cpu().numpy(), ix)
        assert np.array_equal(ge.cpu().numpy(), ei)


def test_csx_hub_rows_longer_than_a_warp():
    rng = np.random.default_rng(0)
    n, e = 64, 6000
    dst = np.where(rng.random(e) < 0.6, 3, rng.integers(0, n, e)).astype(np.int32)  # row 3 has ~3600 entries
    src = rng.integers(0, n, e).astype(np.int32)
    ip, ix, ei = csx.csx_from_coo(dst, src, n)
    gp, gx, ge = ops.csx_from_coo(_i32(dst), _i32(src), n)
    assert np.array_equal(gp.cpu().numpy(), ip) and np.array_equal(gx.cpu().numpy(), ix)
    assert np.array_equal(ge.cpu().numpy(), ei)


def test_csx_batched_pages_and_concat_kernel():
    pages = synth.make_pages(24, ragged=True, k=6)
    s, d, w, noff, eoff = csx.batch_coo(pages)
    n = int(noff[-1])
    for key, other in ((d, s), (s, d)):
        ip, ix, ei = csx.csx_from_coo(key, other, n)
        gp, gx, ge = ops.csx_from_coo(_i32(key), _i32(other), n)
        assert np.array_equal(gp.cpu().numpy(), ip) and np.array_equal(gx.cpu().numpy(), ix)
        assert np.array_equal(ge.cpu().numpy(), ei)
    # device-resident per-page pool -> batch by offset concatenation == stable sort of the batched COO
    from gnn_tableextraction_b200.pool import PagePool

    pool = PagePool(pages, device=DEV)
    order = [5, 0, 23, 7, 7, 11]
    sub = [pages[i] for i in order]
    s2, d2, w2, noff2, _ = csx.batch_coo(sub)
    g = pool.batch(order)
    ip, ix, ei = csx.csx_from_coo(d2, s2, int(noff2[-1]))
    assert np.array_equal(g.csc()[0].cpu().numpy(), ip)
    assert np.array_equal(g.csc()[1].cpu().numpy(), ix)
    assert np.array_equal(g.csc()[2].cpu().numpy(), ei)
    ip, ix, ei = csx.csx_from_coo(s2, d2, int(noff2[-1]))
    assert np.array_equal(g.csr()[0].cpu().numpy(), ip)
    assert np.array_equal(g.csr()[1].cpu().numpy(), ix)
    assert np.array_equal(g.csr()[2].cpu().numpy(), ei)
    assert np.array_equal(g.edges()[0].cpu().numpy(), s2) and np.array_equal(g.edges()[1].cpu().numpy(), d2)
    assert np.array_equal(g.edata["feat"].cpu().numpy(), w2)
    assert np.array_equal(g.weights_csc(g.edata["feat"]).cpu().numpy(), w2[csx.csx_from_coo(d2, s2, int(noff2[-1]))[2]])
    assert np.array_equal(g.ndata["feat"].cpu().numpy(), np.concatenate([p.feat for p in sub]))


def test_degree_norm_and_gather():
    src, dst, w = synth.random_multigraph(1, 300, 2000)
    ip, _, ei = csx.csx_from_coo(dst, src, 300)
    deg = np.diff(ip).astype(np.float32)
    with np.errstate(divide="ignore"):
        n0 = np.where(deg > 0, 1.0 / deg, 0.0).astype(np.float32)
    assert np.array_equal(ops.degree_norm(_i32(ip), _lib.GTE_NORM_INV_DEG_ZERO).cpu().numpy(), n0)
    n1 = (1.0 / np.maximum(deg, 1)).astype(np.float32)
    assert np.array_equal(ops.degree_norm(_i32(ip), _lib.GTE_NORM_INV_DEG_CLAMP).cpu().numpy(), n1)
    assert np.array_equal(ops.gather_f32(_f32(w), _i32(ei)).cpu().numpy(), w[ei])


# -------------------------------------------------------------- spmm --------
@pytest.mark.parametrize("f", [1, 3, 4, 9, 13, 16, 31, 64, 100, 128, 218, 256, 300, 512, 700])
@pytest.mark.parametrize("padded", [True, False])
def test_spmm_matches_oracle(f, padded):
    n, e = 500, 6000
    src, dst, w = synth.random_multigraph(f, n, e)
    h = torch.randn(n, f, generator=torch.Generator().manual_seed(f))
    st, dt, wt = torch.from_numpy(src), torch.from_numpy(dst), torch.from_numpy(w)
    ip, ix, ei = ops.csx_from_coo(_i32(dst), _i32(src), n)
    w_row = ops.gather_f32(_f32(w), ei)
    hd = _padded(h) if padded else h.to(DEV)
    out_pad = None if padded else torch.empty(n, f, device=DEV)
    # GcnSAGE: sum * norm
    norm = ops.degree_norm(ip)
    y = ops.spmm(ip, ix, w_row, hd, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm, out=out_pad)
    deg = so.in_degrees(dt, n).float().unsqueeze(1)
    nrm = torch.where(deg > 0, 1.0 / deg, torch.zeros_like(deg))
    exp = so.u_mul_e_sum(st, dt, wt, h, n) * nrm
    assert rel_err(y, exp) < 2e-6
    assert torch.all(y.cpu()[deg.squeeze(1) == 0] == 0)  # isolated nodes exactly 0
    # mean
    y = ops.spmm(ip, ix, w_row, hd, mode=_lib.GTE_AGG_MEAN)
    assert rel_err(y, so.u_mul_e_mean(st, dt, wt, h, n)) < 2e-6
    # plain sum, unweighted, with addend and source-side scale (the backward form)
    pre = torch.rand(n)
    add = torch.randn(n, f)
    y = ops.spmm(ip, ix, None, hd, mode=_lib.GTE_AGG_SUM, pre_scale=pre.to(DEV), addend=_padded(add) if padded else add.to(DEV))
    exp = so.u_mul_e_sum(st, dt, torch.ones(e), h * pre.unsqueeze(1), n) + add
    assert rel_err(y, exp) < 2e-6


def test_spmm_transposed_is_autograd_of_forward():
    pages = synth.make_pages(4, n=120, k=7)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n, f = int(noff[-1]), 50
    h = torch.randn(n, f, requires_grad=True)
    up = torch.randn(n, f)
    st, dt, wt = torch.from_numpy(s), torch.from_numpy(d), torch.from_numpy(w)
    deg = so.in_degrees(dt, n).float().unsqueeze(1)
    nrm = torch.where(deg > 0, 1.0 / deg, torch.zeros_like(deg))
    ((so.u_mul_e_sum(st, dt, wt, h, n) * nrm) * up).sum().backward()
    ipc, _, _ = ops.csx_from_coo(_i32(d), _i32(s), n)
    ip, ix, ei = ops.csx_from_coo(_i32(s), _i32(d), n)  # CSR: rows = sources
    dh = ops.spmm(ip, ix, ops.gather_f32(_f32(w), ei), _padded(up), mode=_lib.GTE_AGG_SUM, pre_scale=ops.degree_norm(ipc))
    assert rel_err(dh, h.grad) < 2e-6


def test_spmm_large_linearity_and_determinism():
    """Size-independent properties at config-2 scale (512 pages x 300 nodes, F=218)."""
    pages = synth.make_pages(512, distinct=16)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n, f = int(noff[-1]), 218
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    w_row = ops.gather_f32(_f32(w), ei)
    norm = ops.degree_norm(ip)
    a = _padded(torch.randn(n, f))
    b = _padded(torch.randn(n, f))
    run = lambda x: ops.spmm(ip, ix, w_row, x, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    ya, yb = run(a), run(b)
    c = ops.empty_padded(n, f, DEV)
    torch.add(a, b, alpha=2.0, out=c)
    assert rel_err(run(c), ya + 2.0 * yb) < 1e-5
    assert torch.equal(run(a), ya)  # deterministic: fixed summation order, no atomics
    # constant rows: y = norm * sum(w) for every column
    ones = _padded(torch.ones(n, f))
    wsum = torch.zeros(n).index_add(0, torch.from_numpy(d).long(), torch.from_numpy(w)) / 10.0
    assert rel_err(run(ones)[:, 7], wsum) < 2e-6


# ------------------------------------------------------------- dense --------
@pytest.mark.parametrize("n,k1,k2,fo", [(1000, 13, 13, 218), (777, 218, 218, 218), (513, 218, 218, 9), (5, 7, 7, 20),
                                        (300, 64, 0, 33), (129, 100, 100, 130), (0, 13, 13, 8)])
@pytest.mark.parametrize("aligned", [True, False])
def test_linear_fwd_bwd(n, k1, k2, fo, aligned):
    gen = torch.Generator().manual_seed(n + fo)
    x1 = torch.randn(n, k1, generator=gen)
    x2 = torch.randn(n, k2, generator=gen) if k2 else None
    W = torch.randn(fo, k1 + k2, generator=gen) * 0.2
    b = torch.randn(fo, generator=gen)
    dz = torch.randn(n, fo, generator=gen)
    X = torch.cat([x1, x2], 1) if k2 else x1
    mk = _padded if aligned else (lambda t: t.to(DEV))
    x1d, x2d, dzd = mk(x1), (mk(x2) if k2 else None), mk(dz)
    Wd, bd = W.to(DEV), b.to(DEV)
    z = ops.linear_fwd(x1d, x2d, Wd, bd)
    exp = (X.double() @ W.double().t() + b.double())
    assert z.shape == (n, fo)
    if n:
        assert rel_err(z, exp) < 2e-6
    # input gradient, per column block, with row scaling and accumulation
    rs = torch.rand(n)
    dx1 = ops.linear_bwd_data(dzd, Wd, 0, k1)
    if n:
        assert rel_err(dx1, dz.double() @ W.double()[:, :k1]) < 2e-6
    if k2:
        dx2 = ops.linear_bwd_data(dzd, Wd, k1, k2, row_scale=rs.to(DEV))
        if n:
            assert rel_err(dx2, (dz.double() @ W.double()[:, k1:]) * rs.double().unsqueeze(1)) < 2e-6
        if k1 == k2 and n:
            ops.linear_bwd_data(dzd, Wd, k1, k2, out=dx1, accumulate=True)
            assert rel_err(dx1, dz.double() @ (W.double()[:, :k1] + W.double()[:, k1:])) < 2e-6
    # weight / bias gradient (deterministic split reduction)
    dW = torch.full((fo, k1 + k2), 7.0, device=DEV)
    db = torch.full((fo,), 7.0, device=DEV)
    ops.linear_bwd_weight(dzd, x1d, x2d, dW, db)
    expW = dz.double().t() @ X.double()
    assert rel_err(dW, expW) < 2e-6 if n else torch.all(dW == 0)
    assert rel_err(db, dz.double().sum(0)) < 2e-6 if n else torch.all(db == 0)
    dW2 = dW.clone()
    ops.linear_bwd_weight(dzd, x1d, x2d, dW2, db, accumulate=True)
    if n:
        assert rel_err(dW2, 2 * expW) < 2e-6
    dW3 = torch.empty_like(dW)
    ops.linear_bwd_weight(dzd, x1d, x2d, dW3, None)
    assert torch.equal(dW3, dW)  # run-to-run bit-identical


def test_linear_column_offset_views():
    """project-then-aggregate uses the two column blocks of W separately."""
    n, k, fo = 400, 218, 9
    x = torch.randn(n, k)
    W = torch.randn(fo, 2 * k) * 0.1
    b = torch.randn(fo)
    xd, Wd = _padded(x), W.to(DEV)
    s = ops.linear_fwd(xd, None, Wd, b.to(DEV), w_col0=0)
    p = ops.linear_fwd(xd, None, Wd, None, w_col0=k)
    assert rel_err(s, x.double() @ W.double()[:, :k].t() + b.double()) < 2e-6
    assert rel_err(p, x.double() @ W.double()[:, k:].t()) < 2e-6
    dz = torch.randn(n, fo)
    dW = torch.zeros(fo, 2 * k, device=DEV)
    ops.linear_bwd_weight(_padded(dz), xd, None, dW, None, w_col0=k)
    assert torch.all(dW[:, :k] == 0)
    assert rel_err(dW[:, k:], dz.double().t() @ x.double()) < 2e-6


# ----------------------------------------------------------- row ops --------
@pytest.mark.parametrize("n,f", [(1000, 218), (33, 9), (257, 32), (100, 1000), (64, 300), (1, 5)])
@pytest.mark.parametrize("relu", [True, False])
def test_layernorm_act(n, f, relu):
    gen = torch.Generator().manual_seed(f)
    z = (torch.randn(n, f, generator=gen) * 3 + 1).requires_grad_(True)
    gamma = (torch.rand(f, generator=gen) + 0.5).requires_grad_(True)
    beta = (torch.randn(f, generator=gen) * 0.1).requires_grad_(True)
    up = torch.randn(n, f, generator=gen)
    y = F.layer_norm(z, (f,), gamma, beta, 1e-5)
    if relu:
        y = F.relu(y)
    (y * up).sum().backward()
    zd = _padded(z.detach())
    yd, mean, rstd = ops.layernorm_act_fwd(zd, gamma.detach().to(DEV), beta.detach().to(DEV), 1e-5, relu)
    assert rel_err(yd, y) < 2e-6
    dg = torch.empty(f, device=DEV)
    dbt = torch.empty(f, device=DEV)
    dcs = torch.empty(f, device=DEV)
    dz = ops.layernorm_act_bwd(_padded(up), zd, mean, rstd, gamma.detach().to(DEV), beta.detach().to(DEV), relu, dg, dbt,
                               dz_colsum=dcs)
    assert rel_err(dz, z.grad) < 5e-6
    assert (dcs.double().cpu() - z.grad.double().sum(0)).abs().max() < 5e-6 * max(1.0, z.grad.abs().sum(0).max().item())
    assert rel_err(dg, gamma.grad) < 5e-6 and rel_err(dbt, beta.grad) < 5e-6
    dg2 = torch.empty(f, device=DEV)
    dz2 = ops.layernorm_act_bwd(_padded(up), zd, mean, rstd, gamma.detach().to(DEV), beta.detach().to(DEV), relu, dg2,
                                torch.empty(f, device=DEV))
    assert torch.equal(dg2, dg) and torch.equal(dz2, dz)  # deterministic


@pytest.mark.parametrize("n,f", [(500, 20), (100, 218), (7, 3)])
def test_relu_l2norm_and_relu(n, f):
    z = torch.randn(n, f)
    z[0] = -1.0  # a row that relu zeroes completely (norm clamps at eps)
    z = z.requires_grad_(True)
    up = torch.randn(n, f)
    y = F.normalize(F.relu(z))
    (y * up).sum().backward()
    zd = _padded(z.detach())
    assert rel_err(ops.relu_l2norm_fwd(zd), y) < 2e-6
    assert rel_err(ops.relu_l2norm_bwd(_padded(up), zd), z.grad) < 5e-6
    assert torch.equal(ops.relu_fwd(zd).cpu(), F.relu(z.detach()))
    assert torch.equal(ops.relu_bwd(_padded(up), zd).cpu(), up * (z.detach() > 0))


@pytest.mark.parametrize("n,c,weighted,ldt", [(1000, 9, False, torch.float32), (333, 9, True, torch.int64),
                                              (50, 5, True, torch.int32), (1, 3, False, torch.float32)])
def test_cross_entropy(n, c, weighted, ldt):
    gen = torch.Generator().manual_seed(n)
    logits = (torch.randn(n, c, generator=gen) * 3).requires_grad_(True)
    labels = torch.randint(0, c, (n,), generator=gen)
    cw = (torch.rand(c, generator=gen) + 0.5) if weighted else None
    loss = F.cross_entropy(logits, labels, weight=cw)
    loss.backward()
    ld = _padded(logits.detach())
    lab = labels.to(ldt).to(DEV)
    cwd = cw.to(DEV) if weighted else None
    stats = ops.cross_entropy_fwd(ld, lab, cwd)
    s = stats.cpu()
    assert abs(s[0] / s[1] - loss.item()) < 2e-6 * max(1.0, abs(loss.item()))
    assert s[2].item() == (logits.argmax(1) == labels).sum().item()
    dl = ops.cross_entropy_bwd(ld, lab, cwd, stats[1:2])
    assert rel_err(dl, logits.grad) < 2e-6


def test_adam_matches_torch():
    p0 = torch.randn(10007)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=0.01, weight_decay=5e-4)
    p, m, v = p0.to(DEV), torch.zeros(10007, device=DEV), torch.zeros(10007, device=DEV)
    step_dev = torch.zeros(1, dtype=torch.int64, device=DEV)
    for t in range(1, 6):
        g = torch.randn(10007, generator=torch.Generator().manual_seed(t))
        ref.grad = g.clone()
        opt.step()
        if t % 2:
            ops.adam_step(p, g.to(DEV), m, v, lr=0.01, weight_decay=5e-4, step_dev=step_dev)
        else:
            ops.adam_step(p, g.to(DEV), m, v, lr=0.01, weight_decay=5e-4, step=t)
            step_dev += 1
        assert rel_err(p, ref.data) < 2e-6, t
    assert step_dev.item() == 5


# ------------------------------------------------- tensor-core route --------
def _log_err(tag, err):
    print(f"{tag} {err:.3e}")  # error levels of the tensor-core route: shown by pytest -rP


@pytest.mark.parametrize("n,fin,fo,ln,relu,two", [(1000, 218, 218, True, True, True), (129, 64, 64, False, False, True),
                                                  (5000, 100, 130, True, False, True), (128, 32, 16, False, True, False),
                                                  (3001, 256, 256, True, True, True), (40000, 218, 218, True, True, True)])
def test_umma_linear_fwd_3xtf32(n, fin, fo, ln, relu, two, umma_kernel):
    gen = torch.Generator().manual_seed(n)
    x1 = torch.randn(n, fin, generator=gen)
    x2 = torch.randn(n, fin, generator=gen) * 3 if two else None
    nseg = 2 if two else 1
    W = (torch.rand(fo, nseg * fin, generator=gen) - 0.5) * (2.0 / (nseg * fin) ** 0.5)
    b = torch.randn(fo, generator=gen) * 0.1
    gamma = torch.rand(fo, generator=gen) + 0.5
    beta = torch.randn(fo, generator=gen) * 0.1
    X = torch.cat([x1, x2], 1) if two else x1
    z64 = X.double() @ W.double().t() + b.double()
    y64 = F.layer_norm(z64, (fo,), gamma.double(), beta.double(), 1e-5) if ln else z64
    if relu:
        y64 = F.relu(y64)
    pack = ops.umma_pack_weights(W.to(DEV), fin, nseg)
    z, y, mean, rstd = ops.umma_linear_fwd(_padded(x1), _padded(x2) if two else None, fin, pack, b.to(DEV), fo,
                                           gamma=gamma.to(DEV), beta=beta.to(DEV), relu=relu, fuse_ln=ln, want_y=True)
    ez, ey = rel_err(z, z64), rel_err(y, y64)
    # the same product in plain fp32 (FFMA path) for comparison of the error level
    zf = ops.linear_fwd(_padded(x1), _padded(x2) if two else None, W.to(DEV), b.to(DEV))
    _log_err(f"fwd n={n} fin={fin} fo={fo} ln={ln}: umma_z={ez:.2e} umma_y={ey:.2e} ffma_z", rel_err(zf, z64))
    assert ez < 3e-6 and ey < 5e-6
    if ln or relu:  # inference form: no z stores, same y bits
        z2, y2, _, _ = ops.umma_linear_fwd(_padded(x1), _padded(x2) if two else None, fin, pack, b.to(DEV), fo,
                                           gamma=gamma.to(DEV), beta=beta.to(DEV), relu=relu, fuse_ln=ln, want_z=False)
        assert z2 is None and torch.equal(y2, y)
    if ln:
        assert rel_err(mean, z64.mean(1)) < 3e-6
        assert rel_err(rstd, 1.0 / torch.sqrt(z64.var(1, unbiased=False) + 1e-5)) < 3e-6


@pytest.mark.parametrize("n,fin,fo", [(1000, 218, 218), (4097, 64, 96), (257, 256, 16)])
def test_umma_linear_bwd_data_3xtf32(n, fin, fo, umma_kernel):
    gen = torch.Generator().manual_seed(n + 1)
    dz = torch.randn(n, fo, generator=gen)
    W = (torch.rand(fo, 2 * fin, generator=gen) - 0.5) * 0.2
    pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
    d1, d2 = ops.umma_linear_bwd_data(_padded(dz), pack, fin, 2)
    e1 = rel_err(d1, dz.double() @ W.double()[:, :fin])
    e2 = rel_err(d2, dz.double() @ W.double()[:, fin:])
    _log_err(f"bwd_data n={n} fin={fin} fo={fo}: d1={e1:.2e} d2", e2)
    assert e1 < 3e-6 and e2 < 3e-6


@pytest.mark.parametrize("n,k,fo", [(2000, 218, 9), (300, 40, 16), (700, 64, 48), (0, 10, 4)])
def test_linear_two_term_backward(n, k, fo):
    """project-then-aggregate backward: dW blocks against one input, dx from two gradients."""
    gen = torch.Generator().manual_seed(k)
    x = torch.randn(n, k, generator=gen)
    dz1, dz2 = torch.randn(n, fo, generator=gen), torch.randn(n, fo, generator=gen)
    W = torch.randn(fo, 2 * k, generator=gen) * 0.1
    dW = torch.full((fo, 2 * k), 3.0, device=DEV)
    db = torch.full((fo,), 3.0, device=DEV)
    ops.linear_bwd_weight2(_padded(dz1), _padded(dz2), _padded(x), dW, 0, k, db)
    if n:
        assert rel_err(dW[:, :k], dz1.double().t() @ x.double()) < 2e-6
        assert rel_err(dW[:, k:], dz2.double().t() @ x.double()) < 2e-6
        assert rel_err(db, dz1.double().sum(0)) < 2e-6
    else:
        assert torch.all(dW == 0) and torch.all(db == 0)
    dx = ops.linear_bwd_data2(_padded(dz1), 0, _padded(dz2), k, W.to(DEV), k)
    if n:
        assert rel_err(dx, dz1.double() @ W.double()[:, :k] + dz2.double() @ W.double()[:, k:]) < 2e-6
    dW2 = torch.empty_like(dW)
    ops.linear_bwd_weight2(_padded(dz1), _padded(dz2), _padded(x), dW2, 0, k, None)
    assert torch.equal(dW2, dW)


@pytest.mark.parametrize("f", [9, 13, 64, 218, 300])
def test_spmm_paged_equals_generic(f):
    """shared-memory staged kernel (one CTA per page x column slice) == generic kernel, bit for bit"""
    pages = synth.make_pages(9, ragged=True, k=7)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n = int(noff[-1])
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    w_row = ops.gather_f32(_f32(w), ei)
    norm = ops.degree_norm(ip)
    x = _padded(torch.randn(n, f))
    add = _padded(torch.randn(n, f))
    pre = torch.rand(n, device=DEV)
    pg = (_i32(noff), len(pages), int(max(p.num_nodes for p in pages)), int(max(p.num_edges for p in pages)))
    for kw in (dict(mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm), dict(mode=_lib.GTE_AGG_MEAN),
               dict(mode=_lib.GTE_AGG_SUM, pre_scale=pre, addend=add)):
        a = ops.spmm(ip, ix, w_row, x, **kw)
        b = ops.spmm(ip, ix, w_row, x, pages=pg, **kw)
        assert torch.equal(a, b)
    # wrong page table (graph is NOT block diagonal w.r.t. it): the slow path keeps the result correct
    fake = (_i32(np.array([0, n // 3, n])), 2, int(n - n // 3), 64)  # also under-sized edge capacity
    if fake[2] <= 1600:
        b = ops.spmm(ip, ix, w_row, x, pages=fake, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
        assert torch.equal(ops.spmm(ip, ix, w_row, x, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm), b)


@pytest.mark.parametrize("f", [3, 9, 13, 20, 33, 64, 100, 218, 300, 512])
@pytest.mark.parametrize("ragged", [True, False])
def test_spmm_paged_packed_equals_generic(f, ragged):
    """persistent double-buffered kernel on pre-packed edges == generic row kernel, bit for bit
    (forward CSC with norm / mean, backward CSR with norm[dst] folded into the packing + addend)"""
    pages = synth.make_pages(41, ragged=ragged, k=7, n=120)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n = int(noff[-1])
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    wd = _f32(w)
    w_row = ops.gather_f32(wd, ei)
    norm = ops.degree_norm(ip)
    x = _padded(torch.randn(n, f))
    add = _padded(torch.randn(n, f))
    pre = torch.rand(n, device=DEV)
    pg = (_i32(noff), len(pages), int(max(p.num_nodes for p in pages)), int(max(p.num_edges for p in pages)))
    assert ops.paged_packed_supported(pg, f)
    pk = ops.paged_pack_edges(ip, ix, wd, pg, eid=ei)               # weights in edge order + eid
    pk_row = ops.paged_pack_edges(ip, ix, w_row, pg)                # weights already in row order
    e = ix.numel()
    assert torch.equal(pk.packed[:e], pk_row.packed[:e]) and int(pk.page_flag.sum()) == 0
    pk_pre = ops.paged_pack_edges(ip, ix, wd, pg, eid=ei, pre_scale=pre)
    for kw, p_ in ((dict(mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm), pk), (dict(mode=_lib.GTE_AGG_MEAN), pk),
                   (dict(mode=_lib.GTE_AGG_SUM, addend=add), pk_pre)):
        a = ops.spmm(ip, ix, w_row, x, pre_scale=p_.pre_scale, **kw)
        b = ops.spmm_packed(ip, p_, x, pg, **kw)
        assert torch.equal(a, b)
    # unweighted extension (w = None == all ones)
    pk1 = ops.paged_pack_edges(ip, ix, None, pg)
    assert torch.equal(ops.spmm(ip, ix, None, x), ops.spmm_packed(ip, pk1, x, pg))


@pytest.mark.parametrize("f", [13, 64, 218])
def test_spmm_paged_packed_high_degree_reads_edges_through_l1(f):
    """pages whose packed edges do not fit a shared-memory stage next to the x slice (in-degree 45): the kernel
    variant that reads the edge entries from global memory gives the same bits"""
    pages = synth.make_pages(6, k=45, n=300)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n = int(noff[-1])
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    wd = _f32(w)
    w_row = ops.gather_f32(wd, ei)
    norm = ops.degree_norm(ip)
    x, add = _padded(torch.randn(n, f)), _padded(torch.randn(n, f))
    pg = (_i32(noff), len(pages), 300, int(max(p.num_edges for p in pages)))
    assert pg[3] >= 300 * 45 and ops.paged_packed_supported(pg, f)
    pk = ops.paged_pack_edges(ip, ix, wd, pg, eid=ei, pre_scale=norm)
    a = ops.spmm(ip, ix, w_row, x, pre_scale=norm, mode=_lib.GTE_AGG_SUM, addend=add)
    b = ops.spmm_packed(ip, pk, x, pg, mode=_lib.GTE_AGG_SUM, addend=add)
    assert torch.equal(a, b)


def test_spmm_paged_packed_wrong_page_table_and_small_capacity():
    """a page table that does not describe a block-diagonal graph (edges leave their page), and page
    capacities smaller than the real pages: the slow path keeps the result correct"""
    pages = synth.make_pages(9, ragged=True, k=7)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n = int(noff[-1])
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    wd = _f32(w)
    w_row = ops.gather_f32(wd, ei)
    norm = ops.degree_norm(ip)
    x = _padded(torch.randn(n, 70))
    ref = ops.spmm(ip, ix, w_row, x, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    halves = sorted(set(int(v) for v in noff) | set(int((a + b) // 2) for a, b in zip(noff[:-1], noff[1:])))
    cuts = np.array(halves, dtype=np.int32)  # every page cut in two: many edges leave their half page
    ipc = ip.cpu().numpy()
    fake = (_i32(cuts), len(cuts) - 1, int(np.diff(cuts).max()), int(np.diff(ipc[cuts]).max()))
    assert ops.paged_packed_supported(fake, 70)
    pk = ops.paged_pack_edges(ip, ix, wd, fake, eid=ei)
    assert int(pk.page_flag.sum()) > 0
    out = ops.spmm_packed(ip, pk, x, fake, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    assert rel_err(out, ref) < 1e-6  # inside-page edges first, outside edges after: same terms, other order
    # true page table, capacities under-stated: pages that do not fit a stage run from global memory
    pg_small = (_i32(noff), len(pages), int(min(p.num_nodes for p in pages)) + 1, 64)
    pk2 = ops.paged_pack_edges(ip, ix, wd, pg_small, eid=ei)
    out2 = ops.spmm_packed(ip, pk2, x, pg_small, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    assert torch.equal(out2, ref)
    # empty pages in the table
    noff2 = np.concatenate([[0, 0], noff[1:3], [noff[2]], noff[3:]]).astype(np.int32)
    pg2 = (_i32(noff2), len(noff2) - 1, int(np.diff(noff2).max()), int(max(p.num_edges for p in pages)))
    pk3 = ops.paged_pack_edges(ip, ix, wd, pg2, eid=ei)
    assert torch.equal(ops.spmm_packed(ip, pk3, x, pg2, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm), ref)


@pytest.mark.parametrize("n,fo,k1,k2,with_db", [(5000, 218, 218, 218, False), (2000, 218, 13, 13, True), (1000, 64, 100, 0, True),
                                                (513, 256, 256, 256, False), (40000, 218, 218, 218, False), (7, 9, 20, 0, True)])
def test_umma_linear_bwd_weight_3xtf32(n, fo, k1, k2, with_db, umma_kernel):
    gen = torch.Generator().manual_seed(n + fo)
    dz = torch.randn(n, fo, generator=gen)
    x1 = torch.randn(n, k1, generator=gen)
    x2 = torch.randn(n, k2, generator=gen) * 2 if k2 else None
    X = torch.cat([x1, x2], 1) if k2 else x1
    dW = torch.full((fo, k1 + k2), 5.0, device=DEV)
    db = torch.full((fo,), 5.0, device=DEV) if with_db else None
    ops.umma_linear_bwd_weight(_padded(dz), _padded(x1), _padded(x2) if k2 else None, dW, db)
    e = rel_err(dW, dz.double().t() @ X.double())
    dWf = torch.empty_like(dW)
    ops.linear_bwd_weight(_padded(dz), _padded(x1), _padded(x2) if k2 else None, dWf, None)
    _log_err(f"bwd_weight n={n} fo={fo} k={k1}+{k2}: umma={e:.2e} ffma", rel_err(dWf, dz.double().t() @ X.double()))
    assert e < 3e-6
    if with_db:
        assert rel_err(db, dz.double().sum(0)) < 3e-6
    dW2 = torch.empty_like(dW)
    ops.umma_linear_bwd_weight(_padded(dz), _padded(x1), _padded(x2) if k2 else None, dW2, None)
    assert torch.equal(dW2, dW)  # deterministic
    ops.umma_linear_bwd_weight(_padded(dz), _padded(x1), _padded(x2) if k2 else None, dW2, None, accumulate=True)
    assert rel_err(dW2, 2 * (dz.double().t() @ X.double())) < 3e-6


@pytest.mark.parametrize("n,fo,k", [(3000, 9, 218), (1025, 32, 100), (200, 5, 256 - 1)])
def test_umma_linear_bwd_weight2_3xtf32(n, fo, k, umma_kernel):
    gen = torch.Generator().manual_seed(n)
    x = torch.randn(n, k, generator=gen)
    dz1, dz2 = torch.randn(n, fo, generator=gen), torch.randn(n, fo, generator=gen)
    dW = torch.full((fo, 2 * k), 3.0, device=DEV)
    db = torch.full((fo,), 3.0, device=DEV)
    ops.umma_linear_bwd_weight2(_padded(dz1), _padded(dz2), _padded(x), dW, 0, k, db)
    e1, e2 = rel_err(dW[:, :k], dz1.double().t() @ x.double()), rel_err(dW[:, k:], dz2.double().t() @ x.double())
    _log_err(f"bwd_weight2 n={n} fo={fo} k={k}: e1={e1:.2e} e2", e2)
    assert e1 < 3e-6 and e2 < 3e-6
    assert rel_err(db, dz1.double().sum(0)) < 3e-6


def test_umma_class_layer_forms(umma_kernel):
    """stacked forward + two-segment input gradient of the project-then-aggregate class layer"""
    n, fin, fo = 3000, 218, 9
    gen = torch.Generator().manual_seed(5)
    x = torch.randn(n, fin, generator=gen)
    W = (torch.rand(fo, 2 * fin, generator=gen) - 0.5) * 0.1
    b = torch.randn(fo, generator=gen)
    pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
    sp = ops.umma_linear_fwd_stacked(_padded(x), fin, pack, b.to(DEV), fo)
    assert sp.shape == (n, 32)
    assert rel_err(sp[:, :fo], x.double() @ W.double()[:, :fin].t() + b.double()) < 3e-6
    assert rel_err(sp[:, 16:16 + fo], x.double() @ W.double()[:, fin:].t()) < 3e-6
    assert torch.all(sp[:, fo:16] == 0) and torch.all(sp[:, 16 + fo:] == 0)
    dz1, dz2 = torch.randn(n, fo, generator=gen), torch.randn(n, fo, generator=gen)
    dx = ops.umma_linear_bwd_data2(_padded(dz1), _padded(dz2), pack, fin)
    assert rel_err(dx, dz1.double() @ W.double()[:, :fin] + dz2.double() @ W.double()[:, fin:]) < 3e-6


def test_umma_input_layer_narrow_k(umma_kernel):
    """input layer on tensor cores: K = 13 + 13 (raw BBOX magnitudes up to 5e3), fused LayerNorm + ReLU"""
    pages = synth.make_pages(5)
    n = 1500
    feat = torch.from_numpy(np.concatenate([p.feat for p in pages]))
    ah = feat * 0.7 + 3.0
    gen = torch.Generator().manual_seed(2)
    W = (torch.rand(218, 26, generator=gen) - 0.5) * (2 / 26 ** 0.5)
    b = torch.randn(218, generator=gen) * 0.1
    gamma, beta = torch.rand(218, generator=gen) + 0.5, torch.randn(218, generator=gen) * 0.1
    z64 = torch.cat([feat, ah], 1).double() @ W.double().t() + b.double()
    y64 = F.relu(F.layer_norm(z64, (218,), gamma.double(), beta.double(), 1e-5))
    pack = ops.umma_pack_weights(W.to(DEV), 13, 2)
    z, y, mean, rstd = ops.umma_linear_fwd(_padded(feat), _padded(ah), 13, pack, b.to(DEV), 218, gamma=gamma.to(DEV),
                                           beta=beta.to(DEV), relu=True, fuse_ln=True)
    zf = ops.linear_fwd(_padded(feat), _padded(ah), W.to(DEV), b.to(DEV))
    _log_err(f"input layer K=26: umma_z={rel_err(z, z64):.2e} umma_y={rel_err(y, y64):.2e} ffma_z", rel_err(zf, z64))
    assert rel_err(z, z64) < 3e-6 and rel_err(y, y64) < 5e-6


def _comb(a, b):
    """[n, 32] combined operand: a in columns [0, w), b in [16, 16+w), zeros elsewhere"""
    buf = ops.comb_buffer(a.shape[0], DEV)
    va, vb = ops.comb_views(buf, a.shape[1])
    va.copy_(a)
    vb.copy_(b)
    return buf


@pytest.mark.parametrize("n,fin,fo", [(1500, 13, 218), (129, 16, 64), (40000, 13, 218), (7, 1, 256)])
def test_umma_comb_input_layer_forms(n, fin, fo, umma_kernel):
    """combined [h | ah] operand (narrow input): forward = the two-operand forward bit for bit (same products, one
    k-block instead of two); weight gradient + bias gradient vs fp64"""
    gen = torch.Generator().manual_seed(n + fin)
    h = torch.randn(n, fin, generator=gen) * 50
    ah = torch.randn(n, fin, generator=gen) * 30 + 3
    W = (torch.rand(fo, 2 * fin, generator=gen) - 0.5) * (2 / (2 * fin) ** 0.5)
    b = torch.randn(fo, generator=gen) * 0.1
    gamma, beta = torch.rand(fo, generator=gen) + 0.5, torch.randn(fo, generator=gen) * 0.1
    pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
    xc = _comb(h, ah)
    kw = dict(gamma=gamma.to(DEV), beta=beta.to(DEV), relu=True, fuse_ln=True)
    z, y, mean, rstd = ops.umma_linear_fwd_comb(xc, fin, pack, b.to(DEV), fo, **kw)
    z64 = torch.cat([h, ah], 1).double() @ W.double().t() + b.double()
    y64 = F.relu(F.layer_norm(z64, (fo,), gamma.double(), beta.double(), 1e-5))
    assert rel_err(z, z64) < 3e-6 and rel_err(y, y64) < 5e-6
    z2, y2, _, _ = ops.umma_linear_fwd(_padded(h), _padded(ah), fin, pack, b.to(DEV), fo, **kw)
    _log_err(f"fwd_comb n={n} fin={fin} fo={fo}: z={rel_err(z, z64):.2e} two-operand z", rel_err(z2, z64))
    # y only (inference)
    zi, yi, _, _ = ops.umma_linear_fwd_comb(xc, fin, pack, b.to(DEV), fo, want_z=False, **kw)
    assert zi is None and torch.equal(yi, y)
    # weight gradient
    dz = torch.randn(n, fo, generator=gen)
    dW = torch.full((fo, 2 * fin), 5.0, device=DEV)
    db = torch.full((fo,), 5.0, device=DEV) if fin < 16 else None
    ops.umma_linear_bwd_weight_comb(_padded(dz), xc, fin, dW, db)
    ref = dz.double().t() @ torch.cat([h, ah], 1).double()
    assert rel_err(dW, ref) < 3e-6
    if db is not None:
        assert rel_err(db, dz.double().sum(0)) < 3e-6
    dW2 = torch.empty_like(dW)
    ops.umma_linear_bwd_weight_comb(_padded(dz), xc, fin, dW2, None)
    assert torch.equal(dW2, dW)  # deterministic
    ops.umma_linear_bwd_weight_comb(_padded(dz), xc, fin, dW2, None, accumulate=True)
    assert rel_err(dW2, 2 * ref) < 3e-6


@pytest.mark.parametrize("n,fin,fo", [(3000, 218, 9), (40000, 218, 9), (200, 100, 16), (5, 255, 1)])
def test_umma_comb_class_layer_forms(n, fin, fo, umma_kernel):
    """combined [dz | A^T dz] operand (narrow output): input gradient and weight / bias gradients vs fp64"""
    gen = torch.Generator().manual_seed(n + fo)
    x = torch.randn(n, fin, generator=gen)
    W = (torch.rand(fo, 2 * fin, generator=gen) - 0.5) * 0.1
    dz, gq = torch.randn(n, fo, generator=gen), torch.randn(n, fo, generator=gen) * 2
    pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
    dc = _comb(dz, gq)
    dx = ops.umma_linear_bwd_data_comb(dc, fo, pack, fin)
    ref = dz.double() @ W.double()[:, :fin] + gq.double() @ W.double()[:, fin:]
    assert dx.shape == (n, fin) and rel_err(dx, ref) < 3e-6
    dW = torch.full((fo, 2 * fin), 3.0, device=DEV)
    db = torch.full((fo,), 3.0, device=DEV)
    ops.umma_linear_bwd_weight2_comb(dc, fo, _padded(x), dW, 0, fin, db)
    e1, e2 = rel_err(dW[:, :fin], dz.double().t() @ x.double()), rel_err(dW[:, fin:], gq.double().t() @ x.double())
    _log_err(f"bwd_weight2_comb n={n} fo={fo} k={fin}: e1={e1:.2e} e2", e2)
    assert e1 < 3e-6 and e2 < 3e-6
    assert rel_err(db, dz.double().sum(0)) < 3e-6
    dW2 = torch.full_like(dW, 1.0)
    ops.umma_linear_bwd_weight2_comb(dc, fo, _padded(x), dW2, 0, fin, None, accumulate=True)
    assert rel_err(dW2 - 1.0, torch.cat([dz.double().t() @ x.double(), gq.double().t() @ x.double()], 1)) < 1e-5


@pytest.mark.parametrize("n,w", [(1, 13), (1000, 13), (4097, 16), (33, 1), (7, 9)])
def test_comb_fill_and_padded_ce_bwd(n, w):
    """the two native producers of combined [n, 32] operands: self block = the source (bit for bit), every other column 0"""
    gen = torch.Generator().manual_seed(n * 31 + w)
    x = (torch.randn(n, w, generator=gen) * 100).to(DEV)          # unaligned rows (ld = w)
    xc = ops.comb_from(x)
    assert xc.shape == (n, 32) and torch.equal(xc[:, :w], x) and torch.all(xc[:, w:] == 0)
    xs = torch.randn(n, 40, generator=gen).to(DEV)[:, 3:3 + w]     # strided view
    assert torch.equal(ops.comb_from(xs)[:, :w], xs)
    c = min(w, 9)
    logits = _padded(torch.randn(n, c, generator=gen) * 3)
    labels = torch.randint(0, c, (n,), generator=gen).float().to(DEV)
    cw = (torch.rand(c, generator=gen) + 0.5).to(DEV)
    den = torch.tensor([float(n) * 0.7], device=DEV)
    ref = ops.cross_entropy_bwd(logits, labels, cw, den)
    dc = ops.cross_entropy_bwd_comb(logits, labels, cw, den)
    assert dc.shape == (n, 32) and torch.equal(dc[:, :c], ref[:, :c]) and torch.all(dc[:, c:] == 0)
    d12 = ops.cross_entropy_bwd_comb(logits, labels, cw, den, width=12)  # the general padded kernel
    assert d12.shape == (n, 12) and torch.equal(d12[:, :c], ref[:, :c]) and torch.all(d12[:, c:] == 0)


def test_umma_pack_weights_batch_equals_single():
    """one launch for several weight matrices = the per-matrix packs, bit for bit (all planes, incl. the combined ones)"""
    gen = torch.Generator().manual_seed(11)
    shapes = [(218, 13), (218, 218), (9, 218), (64, 100), (256, 256), (16, 16), (1, 1), (130, 7), (33, 250)]
    Ws = [((torch.rand(fo, 2 * fin, generator=gen) - 0.5) * 3).to(DEV) for fo, fin in shapes]
    batch = ops.umma_pack_weights_batch([(W, fin, 2) for W, (_, fin) in zip(Ws, shapes)])  # 9 > GTE_PACK_BATCH_MAX: two launches
    assert len(batch) == len(shapes)
    for W, (fo, fin), pk in zip(Ws, shapes, batch):
        assert torch.equal(pk, ops.umma_pack_weights(W, fin, 2)), (fo, fin)
    one = ops.umma_pack_weights_batch([(Ws[3][:, :100].contiguous(), 100, 1)])[0]
    assert torch.equal(one, ops.umma_pack_weights(Ws[3][:, :100].contiguous(), 100, 1))


def test_umma_split_accumulator_ln_relu_matches_fp64():
    """n = 5000, 218 -> 218 with LayerNorm + ReLU fused: the split accumulator (cross terms in their own TMEM
    accumulator) keeps z within 3e-6 of fp64"""
    n, fin, fo = 5000, 218, 218
    gen = torch.Generator().manual_seed(77)
    h, ah = torch.randn(n, fin, generator=gen), torch.randn(n, fin, generator=gen)
    W = (torch.rand(fo, 2 * fin, generator=gen) - 0.5) * (2 / (2 * fin) ** 0.5)
    b = torch.randn(fo, generator=gen) * 0.1
    gamma, beta = torch.rand(fo, generator=gen) + 0.5, torch.randn(fo, generator=gen) * 0.1
    pack = ops.umma_pack_weights(W.to(DEV), fin, 2)
    z, _, _, _ = ops.umma_linear_fwd(_padded(h), _padded(ah), fin, pack, b.to(DEV), fo, gamma=gamma.to(DEV),
                                     beta=beta.to(DEV), relu=True, fuse_ln=True)
    z64 = torch.cat([h, ah], 1).double() @ W.double().t() + b.double()
    e_split = rel_err(z, z64)
    _log_err(f"accumulator split n={n}: split", e_split)
    assert e_split < 3e-6


# ------------------------------------------------- narrow dense streams ----
@pytest.mark.parametrize("n,wide,nq1,nq2", [(5000, 218, 13, 13), (3001, 218, 9, 9), (2, 7, 3, 0), (777, 256, 16, 16),
                                            (40000, 218, 13, 13), (64, 100, 1, 0), (2049, 33, 5, 2)])
def test_gram_stream_matches_fp64(n, wide, nq1, nq2):
    """C = P^T [Q1|Q2] (+ column sums of Q1), both output orientations, accumulate, run-to-run bit identical"""
    gen = torch.Generator().manual_seed(n + wide)
    P = torch.randn(n, wide, generator=gen)
    Q1 = torch.randn(n, nq1, generator=gen)
    Q2 = torch.randn(n, nq2, generator=gen) if nq2 else None
    Pd, Q1d = _padded(P), _padded(Q1)
    Q2d = _padded(Q2) if nq2 else None
    # orientation 1: out[a, b] row-major [wide, nq1+nq2] (input-layer dW = dz^T [h|ah])
    out = torch.full((wide, nq1 + nq2), 7.0, device=DEV)
    qs = torch.full((nq1,), 7.0, device=DEV)
    ld = nq1 + nq2
    ops.gram_stream(Pd, Q1d, Q2d, out, ld, 1, out[:, nq1:] if nq2 else None, ld, 1, qsum=qs)
    ref = P.double().T @ torch.cat([Q1, Q2], 1).double() if nq2 else P.double().T @ Q1.double()
    assert rel_err(out, ref) < 2e-6
    assert rel_err(qs, Q1.double().sum(0)) < 2e-6
    out_b = torch.full((wide, nq1 + nq2), -1.0, device=DEV)
    ops.gram_stream(Pd, Q1d, Q2d, out_b, ld, 1, out_b[:, nq1:] if nq2 else None, ld, 1)
    assert torch.equal(out, out_b)  # deterministic
    # orientation 2: transposed blocks [nq, 2*wide] (class-layer dW = [dz|G]^T h), accumulate on top of ones
    outT = torch.ones((max(nq1, nq2), 2 * wide), device=DEV)
    ops.gram_stream(Pd, Q1d, Q2d, outT, 1, 2 * wide, outT[:, wide:] if nq2 else None, 1, 2 * wide, accumulate=True)
    assert rel_err(outT[:nq1, :wide] - 1, ref[:, :nq1].T) < 2e-6
    if nq2:
        assert rel_err(outT[:nq2, wide:] - 1, ref[:, nq1:].T) < 2e-6


@pytest.mark.parametrize("n,k1,k2,c,ln,relu", [(5000, 13, 13, 218, True, True), (3001, 9, 9, 218, False, False),
                                               (7, 13, 0, 40, True, False), (40000, 13, 13, 218, True, True),
                                               (1000, 16, 16, 256, True, True), (513, 5, 3, 31, False, False)])
def test_wide_out_matches_fp64(n, k1, k2, c, ln, relu):
    """z = [A1|A2] B + bias (narrow contraction, wide output) with fused LayerNorm + ReLU, both B orientations"""
    gen = torch.Generator().manual_seed(n + c)
    A1 = torch.randn(n, k1, generator=gen) * 30          # large-magnitude inputs like the BBOX features
    A2 = torch.randn(n, k2, generator=gen) if k2 else None
    W = torch.randn(c, k1 + k2, generator=gen) * 0.2     # nn.Linear layout [out, in]
    b = torch.randn(c, generator=gen)
    gam, bet = torch.rand(c, generator=gen) + 0.5, torch.randn(c, generator=gen)
    A1d = _padded(A1)
    A2d = _padded(A2) if k2 else None
    Wd = W.to(DEV)
    x = torch.cat([A1, A2], 1).double() if k2 else A1.double()
    zref = x @ W.double().T + b.double()
    z, y, mean, rstd = ops.wide_out(A1d, A2d, Wd.data_ptr(), Wd.data_ptr() + 4 * k1, 1, k1 + k2, c, b.to(DEV),
                                    gamma=gam.to(DEV), beta=bet.to(DEV), eps=1e-5, relu=relu, fuse_ln=ln)
    assert rel_err(z, zref) < 2e-6
    if ln:
        yref = F.layer_norm(zref, (c,), gam.double(), bet.double(), 1e-5)
        if relu:
            yref = F.relu(yref)
        assert rel_err(y, yref) < 5e-6
        assert rel_err(mean, zref.mean(1)) < 2e-6
        assert rel_err(rstd, 1.0 / torch.sqrt(zref.var(1, unbiased=False) + 1e-5)) < 5e-6
    else:
        assert y is None
    # transposed B (class-layer input gradient: dx = dz Ws + G Wn with W stored [o, 2*c]), row scale
    if k2 == k1:
        W3 = torch.randn(k1, 2 * c, generator=gen) * 0.2
        W3d = W3.to(DEV)
        rs = torch.rand(n, generator=gen)
        z2, _, _, _ = ops.wide_out(A1d, A2d, W3d.data_ptr(), W3d.data_ptr() + 4 * c, 2 * c, 1, c, None, row_scale=rs.to(DEV))
        ref2 = (A1.double() @ W3.double()[:, :c] + A2.double() @ W3.double()[:, c:]) * rs.double()[:, None]
        assert rel_err(z2, ref2) < 2e-6


# ------------------------------------------- either side of the layers ----
def test_bbox_features_bit_exact_vs_reference_golden():
    """gte_bbox_features == the reference's get_shape / get_histogram (golden vectors), bit for bit"""
    import os
    from conftest import GOLDEN
    from gnn_tableextraction_b200 import features

    d = np.load(os.path.join(GOLDEN, "bbox_features.npz"), allow_pickle=True)
    out = features.bbox_features(d["boxes"], d["counts"], DEV)
    assert out.shape == (4000, 13) and out.stride(0) % 4 == 0
    assert np.array_equal(out.cpu().numpy(), d["feat"])
    out2 = features.bbox_features(d["boxes"], [str(t) for t in d["texts"]], DEV)   # from the texts
    assert torch.equal(out, out2)
    assert features.bbox_features(d["boxes"][:0], d["counts"][:0], DEV).shape == (0, 13)


@pytest.mark.parametrize("ldt", [torch.float32, torch.int64, torch.int32])
def test_page_predictions_match_torch_argmax(ldt):
    from oracle import bbox_oracle as bo

    gen = torch.Generator().manual_seed(5)
    sizes = [300, 1, 0, 77, 512, 300]
    n, c = sum(sizes), 9
    logits = torch.randn(n, c, generator=gen)
    logits[5] = torch.tensor([0.0, 3.0, 3.0, 1.0, 3.0, 0.0, 0.0, 0.0, 0.0])  # tie -> first maximal index
    logits[6, 4] = float("nan")                                                 # NaN is maximal (torch.argmax)
    labels = torch.randint(0, c, (n,), generator=gen)
    labels[::3] = logits.argmax(1)[::3]
    off = _i32(np.concatenate([[0], np.cumsum(sizes)]))
    preds, correct = ops.page_predictions(_padded(logits), off, len(sizes), labels.to(ldt).to(DEV))
    assert torch.equal(preds.cpu().long(), logits.argmax(1))
    ref_preds, accs, _ = bo.page_predictions(logits.numpy(), labels.numpy(), sizes)
    want = [int(round(a * s)) for a, s in zip(accs, sizes)]
    assert correct.cpu().tolist() == want
    p2, c2 = ops.page_predictions(_padded(logits), off, len(sizes))
    assert torch.equal(p2, preds) and c2 is None


@pytest.mark.parametrize("ragged,k,bidir", [(False, 10, False), (True, 7, False), (True, 5, True), (False, 45, False)])
def test_build_page_formats_bit_exact(ragged, k, bidir):
    """one-kernel batch assembly == stable argsort oracle (CSC and CSR), == gte_degree_norm, == gte_paged_pack_edges"""
    pages = synth.make_pages(23, ragged=ragged, k=k, bidirectional=bidir, n=300 if k < 40 else 120)
    s, d, w, noff, eoff = csx.batch_coo(pages)
    n = int(noff[-1])
    mx_n, mx_e = int(max(p.num_nodes for p in pages)), int(max(p.num_edges for p in pages))
    sd, dd, wd = _i32(s), _i32(d), _f32(w)
    csc, csr, norm, pk_csc, pk_csr, bad = ops.build_page_formats(sd, dd, wd, _i32(noff), _i32(eoff), len(pages), n, mx_n, mx_e)
    assert int(bad.item()) == 0
    for got, (key, other) in ((csc, (d, s)), (csr, (s, d))):
        ip, ix, ei = csx.csx_from_coo(key, other, n)
        assert np.array_equal(got[0].cpu().numpy(), ip) and np.array_equal(got[1].cpu().numpy(), ix)
        assert np.array_equal(got[2].cpu().numpy(), ei)
    assert torch.equal(norm, ops.degree_norm(csc[0]))
    pg = (_i32(noff), len(pages), mx_n, mx_e)
    e = len(s)
    ref_in = ops.paged_pack_edges(csc[0], csc[1], wd, pg, eid=csc[2])
    ref_out = ops.paged_pack_edges(csr[0], csr[1], wd, pg, eid=csr[2], pre_scale=norm)
    assert torch.equal(pk_csc.packed[:e], ref_in.packed[:e]) and torch.equal(pk_csr.packed[:e], ref_out.packed[:e])
    # broken contract: an edge that leaves its page raises the flag
    s2 = s.copy()
    s2[0] = int(noff[-1]) - 1
    *_, bad2 = ops.build_page_formats(_i32(s2), dd, wd, _i32(noff), _i32(eoff), len(pages), n, mx_n, mx_e)
    assert int(bad2.item()) == 1


# ------------------------------- config-5 sizes: 64-bit row offsets, F = 512, edges-through-L1 at 512 pages -----
def _oracle_rows_for_pages(pages, page_ids, noff, x_dev, f, mode_norm=True, addend_dev=None):
    """so.u_mul_e_sum on the sub-batch made of the sampled pages (pages are independent), rows in batch order"""
    outs = []
    for p_id in page_ids:
        pg = pages[p_id]
        lo = int(noff[p_id])
        xs = x_dev[lo:lo + pg.num_nodes, :f].cpu()
        ah = so.u_mul_e_sum(torch.from_numpy(pg.src), torch.from_numpy(pg.dst), torch.from_numpy(pg.weight), xs, pg.num_nodes)
        if mode_norm:
            deg = so.in_degrees(torch.from_numpy(pg.dst), pg.num_nodes).float().unsqueeze(1)
            norm = 1.0 / deg
            norm[torch.isinf(norm)] = 0
            ah = ah * norm
        if addend_dev is not None:
            ah = ah + addend_dev[lo:lo + pg.num_nodes, :f].cpu()
        outs.append(ah)
    return outs


def test_spmm_paged_packed_row_offsets_beyond_2_31_bytes_f512():
    """3600 pages x 300 nodes x F = 512: N * ld * 4 = 2.2e9 > 2^31 bytes, so every row offset of the last pages needs
    64-bit arithmetic (config 5 reaches 10 M x 512).  Sampled pages (first, around the 2^31-byte mark, last) against
    so.u_mul_e_sum; whole output against the generic row kernel on 8 random column probes."""
    num_pages, f = 3600, 512
    pages = synth.make_pages(num_pages, distinct=24)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n = int(noff[-1])
    assert n * f * 4 > 2 ** 31
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    wd = _f32(w)
    norm = ops.degree_norm(ip)
    gen = torch.Generator(device=DEV).manual_seed(5)
    x = ops.empty_padded(n, f, DEV)
    x.normal_(generator=gen)
    pg = (_i32(noff), num_pages, 300, int(max(p.num_edges for p in pages)))
    assert ops.paged_packed_supported(pg, f)
    pk = ops.paged_pack_edges(ip, ix, wd, pg, eid=ei)
    y = ops.spmm_packed(ip, pk, x, pg, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    mark = (2 ** 31) // (f * 4 * 300)
    sample = [0, 1, mark - 1, mark, mark + 1, num_pages // 2, num_pages - 2, num_pages - 1]
    for p_id, ref in zip(sample, _oracle_rows_for_pages(pages, sample, noff, x, f)):
        lo = int(noff[p_id])
        assert rel_err(y[lo:lo + 300], ref) < 2e-6, p_id
    # generic kernel (global gathers, 64-bit offsets as well) agrees bit for bit on the last 1000 pages
    y2 = ops.spmm(ip, ix, ops.gather_f32(wd, ei), x, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    lo = int(noff[num_pages - 1000])
    assert torch.equal(y[lo:], y2[lo:])
    del y2
    # backward form (CSR, norm[dst] folded in, addend) on the same sizes
    ipr, ixr, eir = ops.csx_from_coo(_i32(s), _i32(d), n)
    pkr = ops.paged_pack_edges(ipr, ixr, wd, pg, eid=eir, pre_scale=norm)
    dh = ops.spmm_packed(ipr, pkr, x, pg, mode=_lib.GTE_AGG_SUM, addend=y)
    for p_id in (0, mark, num_pages - 1):
        pgp = pages[p_id]
        lo = int(noff[p_id])
        xs = x[lo:lo + 300].cpu()
        deg = so.in_degrees(torch.from_numpy(pgp.dst), 300).float().unsqueeze(1)
        nrm = 1.0 / deg
        nrm[torch.isinf(nrm)] = 0
        ref = so.u_mul_e_sum(torch.from_numpy(pgp.dst), torch.from_numpy(pgp.src), torch.from_numpy(pgp.weight), xs * nrm, 300)
        assert rel_err(dh[lo:lo + 300], ref + y[lo:lo + 300].cpu()) < 2e-6, p_id


@pytest.mark.parametrize("f", [218, 512])
def test_spmm_paged_packed_edges_through_l1_at_512_pages(f):
    """in-degree 40 (config 5's densest point) on 512 pages: the page's packed edges do not fit a stage next to the x
    slice, the kernel reads them through L1 -- same bits as the generic kernel, sampled pages against the oracle"""
    num_pages = 512
    pages = synth.make_pages(num_pages, k=40, distinct=12)
    s, d, w, noff, _ = csx.batch_coo(pages)
    n = int(noff[-1])
    ip, ix, ei = ops.csx_from_coo(_i32(d), _i32(s), n)
    wd = _f32(w)
    norm = ops.degree_norm(ip)
    x = ops.empty_padded(n, f, DEV)
    x.normal_(generator=torch.Generator(device=DEV).manual_seed(f))
    pg = (_i32(noff), num_pages, 300, int(max(p.num_edges for p in pages)))
    assert pg[3] == 300 * 40 and ops.paged_packed_supported(pg, f)
    pk = ops.paged_pack_edges(ip, ix, wd, pg, eid=ei)
    y = ops.spmm_packed(ip, pk, x, pg, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm)
    assert torch.equal(y, ops.spmm(ip, ix, ops.gather_f32(wd, ei), x, mode=_lib.GTE_AGG_SUM_NORM, row_norm=norm))
    sample = [0, 137, 511]
    for p_id, ref in zip(sample, _oracle_rows_for_pages(pages, sample, noff, x, f)):
        lo = int(noff[p_id])
        assert rel_err(y[lo:lo + 300], ref) < 2e-6, p_id


# ------------------------------------------------------------- native dropout (models.py:30-33,60-61,113) -----
@pytest.mark.parametrize("p", [0.1, 0.5, 0.8])
def test_dropout_concat_statistics_determinism_and_indexing(p):
    n, f1, f2 = 20000, 218, 218
    x1, x2 = _padded(torch.ones(n, f1)), _padded(torch.ones(n, f2))
    y1, y2 = ops.dropout_concat(x1, x2, p, seed=1234, offset=40)
    y = torch.cat([y1, y2], 1)
    kept = y != 0
    # kept values are x / (1 - p); the keep rate is 1 - p within 5 sigma
    assert torch.allclose(y[kept], torch.full_like(y[kept], 1.0 / (1.0 - p)), rtol=1e-6)
    rate, m = kept.float().mean().item(), n * (f1 + f2)
    assert abs(rate - (1 - p)) < 5 * (p * (1 - p) / m) ** 0.5
    # per-column and per-row keep rates are unbiased as well (no stripe patterns from the counter layout)
    assert (kept.float().mean(0) - (1 - p)).abs().max().item() < 6 * (p * (1 - p) / n) ** 0.5
    assert (kept.float().mean(1) - (1 - p)).abs().max().item() < 6 * (p * (1 - p) / (f1 + f2)) ** 0.5
    # same (seed, offset) => same mask (this is what the backward pass relies on); other offsets / seeds differ
    z1, z2 = ops.dropout_concat(x1, x2, p, seed=1234, offset=40)
    assert torch.equal(z1, y1) and torch.equal(z2, y2)
    assert not torch.equal(ops.dropout_concat(x1, x2, p, seed=1234, offset=41)[0], y1)
    assert not torch.equal(ops.dropout_concat(x1, x2, p, seed=1235, offset=40)[0], y1)
    # the mask is a function of the element index of the concatenation: one [n, f1 + f2] matrix gets the same mask
    xc = _padded(torch.ones(n, f1 + f2))
    assert torch.equal(ops.dropout_concat(xc, None, p, seed=1234, offset=40)[0], y)
    # device-side state (captured steps): same numbers => same mask; advancing the base offset moves the mask
    rng = torch.tensor([1234, 30], dtype=torch.int64, device=DEV)
    assert torch.equal(ops.dropout_concat(x1, x2, p, offset=10, rng_dev=rng)[0], y1)
    ops.rng_advance(rng, 7)
    assert int(rng[1].item()) == 37
    assert not torch.equal(ops.dropout_concat(x1, x2, p, offset=10, rng_dev=rng)[0], y1)
    # in place, and on real data: y = x * mask / (1 - p) with the mask of a single [n, f1] matrix
    xr = _padded(torch.randn(n, f1))
    m1 = ops.dropout_concat(_padded(torch.ones(n, f1)), None, p, seed=1234, offset=40)[0]
    ref = xr * m1
    ops.dropout_concat(xr, None, p, seed=1234, offset=40, inplace=True)
    assert rel_err(xr, ref) < 1e-6


def test_dp_allreduce_adam_single_rank_equals_adam_step():
    """the fused exchange + optimiser kernel with world = 1 (its own buffer as the only peer) == gte_adam_step with the
    device-side denominator: same parameters and moments, step counter advanced, statistics copied out; three calls in a
    row exercise the sequence numbers of the flag protocol"""
    n = 4096 * 3 + 8
    gen = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=gen)
    pa, pb = p0.clone().to(DEV), p0.clone().to(DEV)
    ma, mb = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    va, vb = torch.zeros(n, device=DEV), torch.zeros(n, device=DEV)
    step_a, step_b = torch.zeros(1, dtype=torch.int64, device=DEV), torch.zeros(1, dtype=torch.int64, device=DEV)
    grad = torch.zeros(n + 4, device=DEV)
    ptrs = torch.tensor([grad.data_ptr()], dtype=torch.int64, device=DEV)
    pad = torch.zeros(64, dtype=torch.int32, device=DEV)
    pads = torch.tensor([pad.data_ptr()], dtype=torch.int64, device=DEV)
    local = torch.zeros(4, dtype=torch.int32, device=DEV)
    stats = torch.zeros(4, device=DEV)
    for it in range(3):
        grad[:n] = torch.randn(n, generator=gen).to(DEV) * 100.0
        grad[n:n + 3] = torch.tensor([321.0, 153600.0 + it, 777.0], device=DEV)
        ops.adam_step(pa, grad, ma, va, lr=0.01, weight_decay=5e-4, step_dev=step_a, grad_den=grad[n + 1:n + 2], count=n)
        ops.dp_allreduce_adam(ptrs.data_ptr(), pads.data_ptr(), 0, 1, n, n, pb, mb, vb, stats, lr=0.01, beta1=0.9, beta2=0.999,
                              eps=1e-8, weight_decay=5e-4, step_dev=step_b, local_words=local)
        assert torch.equal(stats[:3], grad[n:n + 3])
    assert step_a.item() == step_b.item() == 3 and local[0].item() == 3 and local[2].item() == 0
    assert rel_err(pb, pa) < 1e-6 and rel_err(mb, ma) < 1e-6 and rel_err(vb, va) < 1e-6
    # a step without weighted labels leaves the replica untouched (and still completes the handshake)
    grad[n + 1] = 0.0
    before = pb.clone()
    ops.dp_allreduce_adam(ptrs.data_ptr(), pads.data_ptr(), 0, 1, n, n, pb, mb, vb, stats, lr=0.01, beta1=0.9, beta2=0.999,
                          eps=1e-8, weight_decay=5e-4, step_dev=step_b, local_words=local)
    assert torch.equal(pb, before) and local[0].item() == 4
