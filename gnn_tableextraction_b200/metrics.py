"""Per-class scores of a validation or test pass from its confusion matrix (host side).

The reference scores a pass with sklearn on the host (model_train.py:349-364 ``f1_score``, model_predict.py:159-169
``precision_recall_fscore_support`` / ``confusion_matrix``), which needs every prediction and label copied off the
device.  ``SageTrainer.evaluate`` and ``capture_eval`` count the confusion matrix on the device instead; this module
turns its C x C entries into the same numbers.
"""
from __future__ import annotations

from typing import Tuple

import numpy as np


def _divide(num: np.ndarray, den: np.ndarray) -> np.ndarray:
    """num / den, 0 where den == 0 (sklearn's zero_division=0)"""
    out = np.zeros(num.shape, dtype=np.float64)
    np.divide(num, den, out=out, where=den != 0)
    return out


def precision_recall_f1(cm) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """Per-class (precision, recall, F1, support) of a confusion matrix ``cm[true, predicted]`` (array or tensor,
    [C, C]): float64 arrays [C] and int64 support, equal to sklearn's ``precision_recall_fscore_support(y, p,
    labels=range(C), zero_division=0)`` for the labels and predictions the matrix counts."""
    if hasattr(cm, "detach"):
        cm = cm.detach().cpu().numpy()
    cm = np.asarray(cm)
    if cm.ndim != 2 or cm.shape[0] != cm.shape[1]:
        raise ValueError(f"precision_recall_f1: expected a square [C, C] confusion matrix, got shape {cm.shape}")
    cm = cm.astype(np.int64)
    tp = np.diag(cm)
    true_sum = cm.sum(axis=1)
    pred_sum = cm.sum(axis=0)
    precision = _divide(tp.astype(np.float64), pred_sum.astype(np.float64))
    recall = _divide(tp.astype(np.float64), true_sum.astype(np.float64))
    f1 = _divide(2.0 * tp.astype(np.float64), true_sum.astype(np.float64) + pred_sum.astype(np.float64))
    return precision, recall, f1, true_sum
