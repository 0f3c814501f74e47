"""Oracle (test infrastructure): Keras `AUC()` with its defaults (SURVEY.md App. A19).

`model.compile(..., metrics=[AUC()])` then `model.evaluate` — src/ctr/fm/train.py:50,58,67.
TF >= 2.6 path for evenly spaced thresholds (`_update_confusion_matrix_variables_optimized`):
the fp32 bucket formula, per-bucket counts, tp / fp as suffix sums, then the trapezoid sum.
Counts are int64 and the result fp64 (the documented divergences from Keras' fp32 accumulators).
"""
from __future__ import annotations

import numpy as np


def auc_thresholds(T: int):
    """[-1e-7, 1/(T-1), ..., (T-2)/(T-1), 1+1e-7] (Keras' evenly spaced thresholds)."""
    return np.array([-1e-7] + [i / (T - 1) for i in range(1, T - 1)] + [1.0 + 1e-7])


def auc_buckets(p, T: int):
    """b = max(ceil(fp32(p * fp32(T-1))) - 1, 0): one fp32 multiply, then ceil."""
    p = np.asarray(p, dtype=np.float32)
    prod = (p * np.float32(T - 1)).astype(np.float32)
    return np.maximum(np.ceil(prod).astype(np.int64) - 1, 0)


def auc_counts(y, p, T: int):
    """-> (counts (2, T) int64: row 0 positives, row 1 negatives per bucket, invalid flag).
    Elements with p outside [0, 1] (or NaN) or a label other than 0 / 1 are not counted; Keras
    raises on them, so the flag is set."""
    y = np.asarray(y, dtype=np.float32).reshape(-1)
    p = np.asarray(p, dtype=np.float32).reshape(-1)
    with np.errstate(invalid="ignore"):
        ok = (p >= 0) & (p <= 1) & ((y == 0) | (y == 1))
    b = auc_buckets(np.where(ok, p, 0), T)
    counts = np.zeros((2, T), dtype=np.int64)
    np.add.at(counts[0], b[ok & (y == 1)], 1)
    np.add.at(counts[1], b[ok & (y == 0)], 1)
    return counts, bool((~ok).any())


def auc_confusion(counts):
    """tp[i] = sum_{j>=i} pos[j], fp likewise; fn = P - tp, tn = N - fp (all int64)."""
    tp = np.cumsum(counts[0][::-1])[::-1]
    fp = np.cumsum(counts[1][::-1])[::-1]
    P, N = (tp[0], fp[0]) if len(tp) else (0, 0)
    return tp, fp, P - tp, N - fp


def auc_from_counts(counts) -> float:
    """AUC = sum_{i<T-1} (fpr[i] - fpr[i+1]) (tpr[i] + tpr[i+1]) / 2 in fp64, with
    divide_no_nan: one class only, or no data, gives 0.0."""
    tp, fp, fn, tn = auc_confusion(counts)
    P, N = tp + fn, fp + tn
    tpr = np.divide(tp, P, out=np.zeros(len(tp)), where=P > 0)
    fpr = np.divide(fp, N, out=np.zeros(len(fp)), where=N > 0)
    return float(np.sum((fpr[:-1] - fpr[1:]) * (tpr[:-1] + tpr[1:]) / 2.0))


def auc(y, p, num_thresholds: int = 200) -> float:
    counts, _ = auc_counts(y, p, num_thresholds)
    return auc_from_counts(counts)
