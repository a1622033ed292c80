"""CPU: exact score curves - the numpy oracle against sklearn's documented examples, metrics.average_precision, and the
checks of cf_curve_* / metrics.score_curve that refuse bad input before any device work."""
import ctypes

import numpy as np
import pytest

from catfish_b200 import _cabi, metrics
import curve_oracle

# sklearn's roc_curve / roc_auc_score / average_precision_score examples
Y = [0, 0, 1, 1]
S = [0.1, 0.4, 0.35, 0.8]


def test_oracle_reproduces_sklearn_examples():
    thresholds, counts, auc, ap = curve_oracle.curve(np.array(S, np.float32), Y)
    fpr, tpr, _, _ = curve_oracle.rates(counts)
    assert fpr.tolist() == [0, 0, 0.5, 0.5, 1]
    assert tpr.tolist() == [0, 0.5, 0.5, 1, 1]
    assert thresholds[0] == np.inf
    assert thresholds[1:].tolist() == pytest.approx([0.8, 0.4, 0.35, 0.1], rel=1e-7)   # float32 scores
    assert auc == 0.75
    assert ap == pytest.approx(0.8333333333333333, rel=1e-15)
    # the rates of the shared helpers are the oracle's
    roc = metrics.roc_curve(counts)
    assert np.array_equal(roc.fpr, fpr) and np.array_equal(roc.tpr, tpr) and roc.area_trapezoid == auc
    assert metrics.average_precision(counts) == pytest.approx(ap, rel=1e-15)


def test_oracle_ties_nan_and_signed_zero():
    s = np.array([0.5, 0.5, np.nan, 0.0, -0.0, 1.0, np.nan], np.float32)
    y = [1, 0, 1, 0, 1, 1, 0]
    thresholds, counts, auc, ap = curve_oracle.curve(s, y)
    assert thresholds.tolist() == [np.inf, 1.0, 0.5, 0.0]                     # -0.0 and +0.0: one threshold
    assert counts.tolist() == [[0, 0, 3, 4], [1, 0, 3, 3], [2, 1, 2, 2], [3, 2, 1, 1]]
    # closing point (3, 4) for the NaN scores: S = 0*1 + 1*3 + 1*5 + 1*7 = 15 over 2 * 3 * 4
    assert auc == 15 / 24
    assert ap == pytest.approx((1 * 1 + 1 * 2 / 3 + 1 * 3 / 5 + 1 * 4 / 7) / 4, rel=1e-15)
    # no positives / no negatives: the areas that divide by them are NaN
    _, _, auc, ap = curve_oracle.curve(np.array([0.2, 0.3], np.float32), [0, 0])
    assert np.isnan(auc) and np.isnan(ap)
    _, _, auc, ap = curve_oracle.curve(np.array([0.2, 0.3], np.float32), [1, 1])
    assert np.isnan(auc) and ap == 1.0


def test_average_precision_of_sweep_rows():
    # rows in any order; the step sum starts at recall 0 and skips rows that add no recall
    _, counts, _, ap = curve_oracle.curve(np.array(S, np.float32), Y)
    rng = np.random.default_rng(1)
    assert metrics.average_precision(counts[rng.permutation(len(counts))]) == pytest.approx(ap, rel=1e-15)
    assert metrics.average_precision(counts[[0, 3]]) == 2 / 3               # one threshold: recall 1 at precision 2/3
    assert np.isnan(metrics.average_precision(np.array([[0, 3, 1, 0]])))    # no positives
    with pytest.raises(ValueError):
        metrics.average_precision(np.zeros((2, 3)))


def _create(device=0, values=None, logits=0, labels=None, n=0, out=True):
    lib = _cabi.load_library()
    h = ctypes.c_void_p()
    return lib.cf_curve_create(device, values, logits, labels, n, None, ctypes.byref(h) if out else None), h


def test_curve_abi_refuses_bad_arguments():
    lib = _cabi.load_library()
    assert _create(out=False)[0] == _cabi.CF_ERR_BAD_ARG
    assert _create(n=-1)[0] == _cabi.CF_ERR_BAD_ARG
    assert _create(n=10)[0] == _cabi.CF_ERR_BAD_ARG                                  # values / labels NULL
    assert _create(values=16, n=10)[0] == _cabi.CF_ERR_BAD_ARG                       # labels NULL
    assert _create(values=16, labels=16, n=2 ** 31)[0] == _cabi.CF_ERR_BAD_ARG       # beyond the int32 row counts
    assert b"cf_curve_create" in lib.cf_last_error()
    assert lib.cf_curve_summary(None, None, None, None, None, None, None) == _cabi.CF_ERR_BAD_ARG
    assert lib.cf_curve_read(None, 0, 1, None, None) == _cabi.CF_ERR_BAD_ARG
    lib.cf_curve_destroy(None)
    status, h = _create()
    assert status == _cabi.CF_OK
    try:
        th = np.zeros(2)
        for first, count in [(0, 2), (1, 1), (2, 0), (-1, 1), (0, -1)]:
            assert lib.cf_curve_read(h, first, count, th.ctypes.data, None) == _cabi.CF_ERR_BAD_ARG, (first, count)
        assert lib.cf_curve_read(h, 1, 0, None, None) == _cabi.CF_OK
    finally:
        lib.cf_curve_destroy(h)


def test_curve_of_nothing_is_one_row():
    lib = _cabi.load_library()
    status, h = _create()
    assert status == _cabi.CF_OK
    try:
        p, n0, n1, nn = ctypes.c_int64(-1), ctypes.c_int64(-1), ctypes.c_int64(-1), ctypes.c_int64(-1)
        auc, ap = ctypes.c_double(), ctypes.c_double()
        assert lib.cf_curve_summary(h, ctypes.byref(p), ctypes.byref(n0), ctypes.byref(n1), ctypes.byref(nn),
                                    ctypes.byref(auc), ctypes.byref(ap)) == _cabi.CF_OK
        assert (p.value, n0.value, n1.value, nn.value) == (1, 0, 0, 0)
        assert np.isnan(auc.value) and np.isnan(ap.value)
        th, counts = np.zeros(1), np.full((1, 4), -7, np.int64)
        assert lib.cf_curve_read(h, 0, 1, th.ctypes.data, counts.ctypes.data) == _cabi.CF_OK
        assert th.tolist() == [np.inf] and not counts.any()
    finally:
        lib.cf_curve_destroy(h)
    c = metrics.score_curve(np.zeros(0, np.float32), np.zeros(0, np.uint8))
    assert c.thresholds.tolist() == [np.inf] and c.counts.tolist() == [[0, 0, 0, 0]]
    assert np.isnan(c.roc_auc) and np.isnan(c.average_precision)
    c = metrics.score_curve([], [], points=False)
    assert c.thresholds is None and c.counts is None and np.isnan(c.roc_auc)


@pytest.mark.parametrize("scores, labels, logits, what", [
    ([0.1, 0.2, 0.3], [0, 2, 1], False, "position 1"),
    ([0.1, 1.5, 0.3], [0, 1, 1], False, "position 1"),
    ([0.1, 0.2, -1e-30], [0, 1, 1], False, "position 2"),
    ([0.1, 0.2, np.inf], [0, 1, 1], False, "position 2"),
    ([5.0, -3.0, 0.3], [0, 1, 7], True, "position 2"),           # logits: only the labels can be bad
])
def test_score_curve_checks_host_arrays_before_upload(scores, labels, logits, what):
    with pytest.raises(ValueError, match=what):
        metrics.score_curve(np.array(scores, np.float32), np.array(labels), logits=logits)


def test_score_curve_checks_lengths():
    with pytest.raises(ValueError):
        metrics.score_curve(np.zeros(3, np.float32), np.zeros(2, np.uint8))
