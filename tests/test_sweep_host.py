"""CPU: threshold sweeps - the pure curve helpers of metrics.py and the argument checks of cf_sweep_thresholds /
cf_validate_windows_sweep, which refuse bad input before any device work."""
import ctypes

import numpy as np
import pytest

from catfish_b200 import _cabi, metrics


def _sweep(th, n=0, values=None, labels=None, counts=True):
    lib = _cabi.load_library()
    th = np.ascontiguousarray(th, dtype=np.float64)
    out = np.full((max(th.size, 1), 4), -7, np.int64)
    status = lib.cf_sweep_thresholds(0, values, 0, labels, n, th.ctypes.data if th.size else None, th.size,
                                     out.ctypes.data_as(_cabi.c_i64_p) if counts else None, None)
    return status, out


@pytest.mark.parametrize("th", [[], np.zeros(4097), [0.5, np.nan]])
def test_sweep_refuses_bad_thresholds(th):
    status, _ = _sweep(th)
    assert status == _cabi.CF_ERR_BAD_ARG
    assert b"threshold" in _cabi.load_library().cf_last_error()
    with pytest.raises(ValueError):
        metrics.confusion_curve(np.zeros(0, np.float32), np.zeros(0, np.uint8), th)


def test_sweep_refuses_null_pointers_and_negative_n():
    assert _sweep([0.5], counts=False)[0] == _cabi.CF_ERR_BAD_ARG
    assert _sweep([0.5], n=-1)[0] == _cabi.CF_ERR_BAD_ARG
    assert _sweep([0.5], n=10)[0] == _cabi.CF_ERR_BAD_ARG                      # values / labels NULL
    lib = _cabi.load_library()
    th = np.array([0.5])
    out = np.zeros((1, 4), np.int64)
    assert lib.cf_sweep_thresholds(0, None, 0, None, 0, None, 1, out.ctypes.data_as(_cabi.c_i64_p), None) \
        == _cabi.CF_ERR_BAD_ARG
    acc, loss = ctypes.c_double(), ctypes.c_double()
    assert lib.cf_validate_windows_sweep(None, None, None, 1, 0, th.ctypes.data, 1, out.ctypes.data_as(_cabi.c_i64_p),
                                         ctypes.byref(acc), ctypes.byref(loss), None) == _cabi.CF_ERR_BAD_ARG


def test_sweep_of_nothing_is_zero_counts_at_every_threshold():
    status, out = _sweep([0.9, 0.1, 0.9, -np.inf, np.inf, 4096.0])
    assert status == _cabi.CF_OK and not out.any() and out.shape == (6, 4)
    got = metrics.confusion_curve(np.zeros(0, np.float32), np.zeros(0, np.uint8), [0.3, 0.2])
    assert got.dtype == np.int64 and got.shape == (2, 4) and not got.any()
    assert metrics.confusion_curve([], [], np.linspace(0, 1, 4096)).shape == (4096, 4)


def test_confusion_curve_checks_lengths():
    with pytest.raises(ValueError):
        metrics.confusion_curve(np.zeros(3, np.float32), np.zeros(2, np.uint8), [0.5])


def test_precision_recall_and_roc_rows():
    counts = np.array([[5, 1, 10, 2],      # t0
                       [3, 0, 11, 4],      # t1
                       [0, 0, 11, 7]])     # t2: nothing predicted positive
    pr = metrics.precision_recall_curve(counts)
    for row, p, r in zip(counts, pr.precision, pr.recall):
        assert (p, r) == pytest.approx(metrics.precision_recall(row[0], row[1], row[3]))
    assert pr.precision[2] == 0.0 and pr.recall[2] == 0.0            # 0 / 0 -> 0, as precision_recall
    roc = metrics.roc_curve(counts)
    assert roc.fpr.tolist() == pytest.approx([1 / 11, 0.0, 0.0])
    assert roc.tpr.tolist() == pytest.approx([5 / 7, 3 / 7, 0.0])
    zero = metrics.roc_curve(np.zeros((3, 4), np.int64))
    assert not zero.fpr.any() and not zero.tpr.any() and zero.area_trapezoid == 0.0
    with pytest.raises(ValueError):
        metrics.roc_curve(np.zeros((3, 3)))


def test_trapezoid_areas():
    # a perfect classifier swept from below every score to above every score: ROC (0,0) (0,1) (1,1) -> area 1
    counts = np.array([[4, 6, 0, 0], [4, 0, 6, 0], [0, 0, 6, 4]])
    roc = metrics.roc_curve(counts)
    assert roc.area_trapezoid == 1.0
    assert metrics.roc_curve(counts[::-1]).area_trapezoid == 1.0          # any row order
    # a chance-level classifier: the diagonal, area 1/2
    diag = np.array([[10, 10, 0, 0], [5, 5, 5, 5], [0, 0, 10, 10]])
    assert metrics.roc_curve(diag).area_trapezoid == pytest.approx(0.5)
    # only the given points count: one point has no area
    assert metrics.roc_curve(diag[1:2]).area_trapezoid == 0.0
    pr = metrics.precision_recall_curve(np.array([[4, 4, 0, 0], [2, 0, 4, 2]]))
    # (recall, precision) = (1, 0.5) and (0.5, 1): trapezoid 0.5 * (0.5 + 1) / 2
    assert pr.area_trapezoid == pytest.approx(0.375)
