"""CPU tests of capacity capture's host side: the padded page table a batch gets inside a BatchCapacity (the layout
gte_pad_batch fills on the device), the refusals of batches that do not fit, and the validation of the capacity."""
import numpy as np
import pytest

import gnn_tableextraction_b200 as gte
from gnn_tableextraction_b200.engine import padded_page_table


def _check_layout(cap, bn, be):
    """every invariant the padded batch needs to be a valid dgl.batch of the capacity shape"""
    n_cap, e_cap, p_cap = cap.shape
    po, eo = padded_page_table(cap, bn, be)
    assert po.dtype == np.int32 and eo.dtype == np.int32
    assert po.shape == eo.shape == (p_cap + 1,)
    p, n, e = len(bn), sum(bn), sum(be)
    # real pages first, exactly as given
    assert po[:p + 1].tolist() == np.concatenate([[0], np.cumsum(bn)]).tolist()
    assert eo[:p + 1].tolist() == np.concatenate([[0], np.cumsum(be)]).tolist()
    assert po[-1] == n_cap and eo[-1] == e_cap
    pn, pe = np.diff(po.astype(np.int64)), np.diff(eo.astype(np.int64))
    assert (pn >= 0).all() and (pe >= 0).all()
    # no page above the caps: the page kernels were sized for them
    assert pn.max() <= cap.page_nodes and pe.max() <= cap.page_edges
    pad_n, pad_e = pn[p:], pe[p:]
    # a page with edges has a node to carry its self-loops
    assert (pad_n[pad_e > 0] >= 1).all()
    # padding pages, then empty pages at the end only
    used = np.nonzero(pad_n)[0]
    if used.size:
        assert (pad_n[:used[-1] + 1] >= 1).all()
        assert (pad_n[used[-1] + 1:] == 0).all() and (pad_e[used[-1] + 1:] == 0).all()
    else:
        assert n == n_cap and e == e_cap
    return po, eo


def _random_fit(rng, cap):
    p = int(rng.integers(1, cap.pages + 1))
    bn = rng.integers(1, cap.page_nodes + 1, size=p)
    while bn.sum() > cap.nodes:
        bn = np.maximum(bn // 2, 1)
        if bn.sum() > cap.nodes:
            bn = bn[: max(1, len(bn) // 2)]
    be = rng.integers(0, cap.page_edges + 1, size=len(bn))
    while be.sum() > cap.edges:
        be //= 2
    return bn.tolist(), be.tolist()


@pytest.mark.parametrize("cap", [gte.BatchCapacity(3000, 30000, 12, 900, 9000), gte.BatchCapacity(50, 400, 7, 9, 80),
                                 gte.BatchCapacity(10, 0, 3, 2, 1), gte.BatchCapacity(1600, 5000, 2, 1600, 5000),
                                 gte.BatchCapacity(7, 100, 7, 7, 100)])
def test_padded_layout_invariants_on_random_batches(cap):
    rng = np.random.default_rng(cap.nodes + cap.edges)
    for _ in range(300):
        _check_layout(cap, *_random_fit(rng, cap))


def test_padded_layout_edge_cases():
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    n_cap, e_cap, p_cap = cap.shape
    k = max(-(-1000 // 399), -(-8000 // 3000))
    assert (n_cap, e_cap, p_cap) == (1000 + k, 8000, 4 + k)
    _check_layout(cap, [100, 200, 150, 50], [800, 900, 700, 100])  # P == pages
    _check_layout(cap, [400, 400, 200], [10, 20, 30])  # n == nodes
    po, eo = _check_layout(cap, [300, 300], [3000, 3000])  # pages exactly at the caps
    _check_layout(cap, [100, 100, 100], [3000, 3000, 2000])  # e == edges: no padding edges
    _check_layout(cap, [400, 400, 200, 0], [3000, 3000, 2000, 0])  # everything at once, with an empty real page
    _check_layout(cap, [7], [20])  # one real page
    _check_layout(cap, [1], [0])
    # one padding slot per node when free nodes are scarcer than free pages
    tight = gte.BatchCapacity(nodes=6, edges=40, pages=6, page_nodes=2, page_edges=8)
    _check_layout(tight, [2, 2, 2], [8, 8, 8])
    _check_layout(tight, [1], [0])


@pytest.mark.parametrize("bn,be,limit", [
    ([300, 300, 300, 300], [1, 1, 1, 1], "nodes=1000"),
    ([100] * 5, [1] * 5, "pages=4"),
    ([300, 300], [3000, 3000], None),
    ([300, 300, 300], [3000, 3000, 2001], "edges=8000"),
    ([401], [10], "page_nodes=400"),
    ([100, 100], [10, 3001], "page_edges=3000"),
])
def test_batches_over_a_limit_are_refused_by_name(bn, be, limit):
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    if limit is None:
        assert cap.fits(bn, be)
        return
    assert not cap.fits(bn, be)
    with pytest.raises(gte.GteError, match=limit):
        cap.check(bn, be)
    with pytest.raises(gte.GteError, match=limit):
        padded_page_table(cap, bn, be)


def test_malformed_batches_are_refused():
    cap = gte.BatchCapacity(nodes=1000, edges=8000, pages=4, page_nodes=400, page_edges=3000)
    for bn, be in (([], []), ([10, 20], [5]), ([10, -1], [5, 5])):
        with pytest.raises(gte.GteError):
            cap.check(bn, be)


def test_capacity_validation():
    with pytest.raises(gte.GteError, match="page_nodes=1 < 2"):
        gte.BatchCapacity(100, 100, 4, 1, 10)
    with pytest.raises(gte.GteError, match="page_nodes=1601 > 1600"):
        gte.BatchCapacity(10000, 100, 40, 1601, 10)
    with pytest.raises(gte.GteError, match="int32"):
        gte.BatchCapacity(1000, 2 ** 31, 4, 400, 2 ** 30)
    for bad in (dict(nodes=0), dict(pages=0), dict(edges=-1), dict(page_edges=0), dict(nodes=10.5), dict(pages=True)):
        kw = dict(nodes=100, edges=100, pages=4, page_nodes=50, page_edges=50)
        kw.update(bad)
        with pytest.raises(gte.GteError):
            gte.BatchCapacity(**kw)
    cap = gte.BatchCapacity(np.int64(100), 100, 4, 50, 50)
    assert type(cap.nodes) is int and cap.shape == (103, 100, 7)


def test_capacity_check_reads_host_batches():
    """the page lists of batch_pages_host() are what the trainer checks against its capacity"""
    from gnn_tableextraction_b200 import synth
    from gnn_tableextraction_b200.graph import batch_pages_host

    hb = batch_pages_host(synth.make_pages(3, n=60, k=4), pin=False)
    small = gte.BatchCapacity(nodes=150, edges=2000, pages=3, page_nodes=60, page_edges=240)
    with pytest.raises(gte.GteError, match="nodes=150"):
        small.check(hb["batch_num_nodes"], hb["batch_num_edges"])
    assert gte.BatchCapacity(nodes=180, edges=720, pages=3, page_nodes=60, page_edges=240).fits(
        hb["batch_num_nodes"], hb["batch_num_edges"])
