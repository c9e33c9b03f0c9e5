"""CPU tests of gnn_tableextraction_b200.metrics: per-class precision / recall / F1 / support from a confusion matrix
equal sklearn's precision_recall_fscore_support(labels=range(C), zero_division=0)."""
import numpy as np
import pytest
import torch

import gnn_tableextraction_b200 as gte

sklearn_metrics = pytest.importorskip("sklearn.metrics")


def _confusion(y, p, c):
    return np.bincount(y * c + p, minlength=c * c).reshape(c, c)


@pytest.mark.parametrize("seed,c,n", [(0, 9, 500), (1, 2, 40), (2, 16, 3000), (3, 64, 200), (4, 5, 1)])
def test_precision_recall_f1_equals_sklearn(seed, c, n):
    rng = np.random.default_rng(seed)
    y = rng.integers(0, c, size=n)
    p = np.where(rng.random(n) < 0.6, y, rng.integers(0, c, size=n))
    if c > 2:
        y[y == 1] = 0  # class 1: no support
        p[p == c - 1] = 0  # class c - 1: never predicted
    cm = _confusion(y, p, c)
    assert np.array_equal(cm, sklearn_metrics.confusion_matrix(y, p, labels=range(c)))
    ref = sklearn_metrics.precision_recall_fscore_support(y, p, labels=range(c), zero_division=0)
    for got in (gte.metrics.precision_recall_f1(cm), gte.precision_recall_f1(torch.from_numpy(cm))):
        for a, b in zip(got, ref):
            assert a.shape == (c,)
            np.testing.assert_array_equal(a, b)


def test_precision_recall_f1_of_an_empty_matrix_is_zero():
    prec, rec, f1, sup = gte.metrics.precision_recall_f1(np.zeros((3, 3), dtype=np.int64))
    for a in (prec, rec, f1, sup):
        assert np.array_equal(a, np.zeros(3))


def test_precision_recall_f1_refuses_a_non_square_matrix():
    with pytest.raises(ValueError):
        gte.metrics.precision_recall_f1(np.zeros((3, 4)))
