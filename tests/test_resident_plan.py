"""CPU tests of the resident pass's host side: how plan_epoch cuts an epoch over a PagePool into batches and decides
which fit the capacity, the plan words it uploads, the warm-up batch of a capture, and the refusals that need no
kernel."""
from types import SimpleNamespace

import numpy as np
import pytest

import gnn_tableextraction_b200 as gte
from gnn_tableextraction_b200 import ops
from gnn_tableextraction_b200.engine import check_resident_capture, plan_slices, resident_warmup_ids


def _ragged_pool(rng, pages):
    n_i = np.clip(rng.normal(300, 80, size=pages), 40, 900).astype(np.int64)
    e_i = n_i * 10 - rng.integers(0, 40, size=pages)
    return n_i, e_i


@pytest.mark.parametrize("seed", range(6))
def test_plan_decisions_equal_capacity_fits_and_cover_the_ids_in_order(seed):
    rng = np.random.default_rng(seed)
    pages = int(rng.integers(40, 400))
    n_i, e_i = _ragged_pool(rng, pages)
    b = int(rng.integers(1, 40))
    cap = gte.BatchCapacity(nodes=int(300 * b * rng.uniform(0.9, 1.1)), edges=int(3000 * b * rng.uniform(0.9, 1.1)),
                            pages=int(rng.integers(max(1, b - 2), b + 2)), page_nodes=int(rng.integers(500, 901)),
                            page_edges=int(rng.integers(5000, 9001)))
    perm = rng.permutation(pages)[:int(rng.integers(1, pages + 1))]
    batches, words = plan_slices(cap, n_i, e_i, perm, b)
    assert len(batches) == -(-perm.size // b)
    assert np.array_equal(np.concatenate([x.ids for x in batches]), perm)
    assert all(x.pages == b for x in batches[:-1]) and batches[-1].pages == perm.size - b * (len(batches) - 1)
    for x in batches:
        assert x.fits == cap.fits(n_i[x.ids], e_i[x.ids])
        assert x.nodes == int(n_i[x.ids].sum()) and x.pages == x.ids.size
    # [cursor, flag, nfit, B, L, 0, 0, 0 | ids | starts of the fitting batches]
    h = ops.PLAN_HEADER
    fit = [i * b for i, x in enumerate(batches) if x.fits]
    assert words.dtype == np.int32 and words.size == h + perm.size + len(fit)
    assert words[:h].tolist() == [0, 0, len(fit), min(b, perm.size), perm.size, 0, 0, 0]
    assert np.array_equal(words[h:h + perm.size], perm) and words[h + perm.size:].tolist() == fit


def test_plan_mixes_fitting_and_refused_batches():
    n_i = np.array([100, 100, 100, 500, 100, 100, 100], dtype=np.int64)
    e_i = n_i * 10
    cap = gte.BatchCapacity(nodes=450, edges=4500, pages=3, page_nodes=400, page_edges=4000)
    batches, words = plan_slices(cap, n_i, e_i, [0, 1, 2, 3, 4, 5, 6], 3)
    assert [x.fits for x in batches] == [True, False, True]  # the middle batch holds a page above page_nodes
    assert [x.pages for x in batches] == [3, 3, 1] and [x.nodes for x in batches] == [300, 700, 100]
    assert words[ops.PLAN_HEADER + 7:].tolist() == [0, 6]


@pytest.mark.parametrize("ids,batch_pages,match", [
    ([0, 1, 10], 2, r"\[0, 10\)"),
    ([-1, 2], 2, r"\[0, 10\)"),
    (list(range(10)) + [3], 4, "11 page ids > the pool's 10 pages"),
    ([], 4, "non-empty"),
    ([[0, 1], [2, 3]], 2, "1-D"),
    ([0.0, 1.0], 2, "integer"),
    ([0, 1], 0, "positive"),
    ([0, 1], True, "positive"),
])
def test_plan_refusals(ids, batch_pages, match):
    n_i = np.full(10, 100, dtype=np.int64)
    cap = gte.BatchCapacity(nodes=1000, edges=10000, pages=10, page_nodes=100, page_edges=1000)
    with pytest.raises(gte.GteError, match=match):
        plan_slices(cap, n_i, n_i * 10, ids, batch_pages)


def test_resident_capture_refusals():
    cap = gte.BatchCapacity(nodes=1000, edges=10000, pages=10, page_nodes=400, page_edges=4000)
    pool = SimpleNamespace(feat_width=13)
    check_resident_capture(pool, cap, 1, 13)
    with pytest.raises(gte.GteError, match="needs a capacity"):
        check_resident_capture(pool, None, 1, 13)
    with pytest.raises(gte.GteError, match="data parallel"):
        check_resident_capture(pool, cap, 2, 13)
    with pytest.raises(gte.GteError, match="13 wide, the model takes 64"):
        check_resident_capture(pool, cap, 1, 64)


def test_warmup_batch_is_the_first_pages_that_fit():
    cap = gte.BatchCapacity(nodes=1000, edges=10000, pages=3, page_nodes=400, page_edges=4000)
    n_i = np.array([500, 300, 300, 300, 300], dtype=np.int64)
    pool = SimpleNamespace(n_i=n_i, e_i=n_i * 10)
    assert resident_warmup_ids(pool, cap).tolist() == [1, 2, 3]  # page 0 is above page_nodes
    pool = SimpleNamespace(n_i=np.array([300, 400, 350, 10]), e_i=np.array([3000, 4000, 3500, 100]))
    assert resident_warmup_ids(pool, cap).tolist() == [0, 1]  # a third page would pass nodes=1000
    ids = resident_warmup_ids(pool, cap)
    assert cap.fits(pool.n_i[ids], pool.e_i[ids])
    with pytest.raises(gte.GteError, match="no page of the pool fits"):
        resident_warmup_ids(SimpleNamespace(n_i=np.array([500]), e_i=np.array([10])), cap)


def test_page_pool_is_exported():
    assert gte.PagePool is gte.pool.PagePool and "PagePool" in gte.__all__
