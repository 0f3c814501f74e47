"""Keras AUC(): the oracle's restatement (SURVEY App. A19) and the C-ABI's argument checks, no GPU."""
import ctypes

import numpy as np
import pytest
from scipy.stats import rankdata

from oracle import metrics as O


def _rank_auc(y, p):
    """Exact ROC AUC as the Mann-Whitney statistic, ties counted 1/2 (= sklearn roc_auc_score)."""
    y = np.asarray(y)
    r = rankdata(p)
    P, N = int((y == 1).sum()), int((y == 0).sum())
    return (r[y == 1].sum() - P * (P + 1) / 2.0) / (P * N)


def test_keras_docstring_example():
    counts, bad = O.auc_counts([0, 0, 1, 1], [0, 0.5, 0.3, 0.9], 3)
    tp, fp, fn, tn = O.auc_confusion(counts)
    assert not bad
    assert tp.tolist() == [2, 1, 0] and fp.tolist() == [2, 0, 0]
    assert fn.tolist() == [0, 1, 2] and tn.tolist() == [0, 2, 2]
    assert O.auc_from_counts(counts) == 0.75
    assert O.auc([0, 0, 1, 1], [0, 0.5, 0.3, 0.9], 3) == 0.75


@pytest.mark.parametrize("T", [3, 17, 200, 4096])
def test_bucket_centres_give_the_exact_rank_auc(T):
    """One score per bucket: the threshold curve passes through every ROC vertex, so the
    trapezoid sum is the exact rank statistic (ties within a bucket count 1/2 in both)."""
    rng = np.random.default_rng(T)
    k = rng.integers(0, T - 1, 5000)
    p = ((k + 0.5) / (T - 1)).astype(np.float32)
    assert np.array_equal(O.auc_buckets(p, T), k)
    y = (rng.random(5000) < 0.2 + 0.6 * p).astype(np.float32)
    got = O.auc(y, p, T)
    assert abs(got - _rank_auc(y, p)) < 1e-12
    try:
        from sklearn.metrics import roc_auc_score
    except ImportError:
        return
    assert abs(got - roc_auc_score(y, p)) < 1e-12


def test_one_class_or_no_data_gives_zero():
    assert O.auc([1, 1, 1], [0.1, 0.5, 0.9]) == 0.0
    assert O.auc([0, 0], [0.1, 0.9]) == 0.0
    assert O.auc([], []) == 0.0


def test_fp32_bucket_formula_at_thresholds():
    f = np.float32
    up = lambda x: np.nextafter(f(x), f(2))        # noqa: E731
    down = lambda x: np.nextafter(f(x), f(-1))     # noqa: E731
    assert O.auc_buckets([f(0.5)], 3).tolist() == [0]
    assert O.auc_buckets([up(0.5)], 3).tolist() == [1]
    assert O.auc_buckets([f(0), f(1), up(0), down(1)], 3).tolist() == [0, 1, 0, 1]
    T = 200
    for k in (1, 2, 50, 99, 100, 198):
        t = f(k) / f(T - 1)                    # fp32 threshold k/(T-1) and its neighbours
        for x in (down(t), t, up(t)):
            prod = f(x) * f(T - 1)
            assert O.auc_buckets([x], T)[0] == max(int(np.ceil(prod)) - 1, 0)
    assert O.auc_buckets([f(1.0)], T).tolist() == [T - 2]


def test_invalid_elements_are_flagged_and_skipped():
    counts, bad = O.auc_counts([1, 0, 1, 0.5, 1], [0.9, 1.5, -0.1, 0.5, np.nan], 3)
    assert bad and counts.sum() == 1 and counts[0, 1] == 1


def test_auc_argument_errors_without_gpu():
    import __graft_entry__ as g
    g.build()
    import recommend_tf2_b200 as pkg
    lib = pkg.lib()
    buf = ctypes.c_void_p(0x1000)
    # NULL pointers or n < 0 -> RTF_E_ARG; T outside [2, 4096] -> RTF_E_RANGE; nothing launched
    assert lib.rtf_auc_update(None, buf, 4, 200, buf, buf, None) == -1
    assert lib.rtf_auc_update(buf, buf, 4, 200, None, buf, None) == -1
    assert lib.rtf_auc_update(buf, buf, 4, 200, buf, None, None) == -1
    assert lib.rtf_auc_update(buf, buf, -1, 200, buf, buf, None) == -1
    assert lib.rtf_auc_update(buf, buf, 4, 1, buf, buf, None) == -3
    assert lib.rtf_auc_update(buf, buf, 4, 4097, buf, buf, None) == -3
    assert lib.rtf_auc_update(buf, buf, 0, 200, buf, buf, None) == 0
    assert lib.rtf_auc_result(None, 200, buf, None) == -1
    assert lib.rtf_auc_result(buf, 200, None, None) == -1
    assert lib.rtf_auc_result(buf, 1, buf, None) == -3
    assert lib.rtf_auc_result(buf, 4097, buf, None) == -3


def test_auc_constructor_follows_keras():
    import recommend_tf2_b200 as pkg
    m = pkg.metrics.AUC()
    assert (m.num_thresholds, m.curve, m.summation_method, m.name) == (200, "ROC", "interpolation", "auc")
    for kw in ({"curve": "PR"}, {"summation_method": "majoring"}, {"num_thresholds": 1},
               {"num_thresholds": 4097}):
        with pytest.raises(ValueError):
            pkg.metrics.AUC(**kw)
    import torch
    with pytest.raises(pkg.RtfError):
        m.update_state(torch.zeros(4), torch.zeros(4))
