"""Host-side scalar metrics of the validation path ("next" row N4).

Reference: /root/reference/networks/trainingDB/metrics.py (``confusion_matrix`` :10-37,
``precision_recall`` :40-55, ``calculate_accuracy`` :58-63, ``weighted_f1`` :95-113, ``f1`` :117-135).
The per-position counting for a forward pass runs on the GPU inside ``RNN.test_network``
(C ABI ``cf_validate_windows``); ``confusion_matrix`` here is the array-level twin for label
lists that already live on the host.  ``confusion_curve`` counts at many thresholds at once on the GPU (K11,
``cf_sweep_thresholds``); ``precision_recall_curve`` / ``roc_curve`` turn those counts into the rates of the
reference's networks/precision_recall_ROC.py.  ``score_curve`` gives the exact curve at every distinct score with its
ROC AUC and average precision (K13, ``cf_curve_create``: a radix sort on the GPU), the numbers sklearn's
``roc_auc_score`` / ``average_precision_score`` give in the reference's networks/metrics.py.  Plotting helpers are out
of scope.
"""

import collections

import numpy as np


def confusion_matrix(true_labels, predicted_labels):
    """(true_pos, false_pos, true_neg, false_neg); predictions other than 0 / 1 are not counted."""
    if len(true_labels) != len(predicted_labels):
        raise ValueError("Length of labels to compare is not equal.")
    t = np.asarray(true_labels)
    p = np.asarray(predicted_labels)
    called, uncalled = p == 1, p == 0
    true_pos = int(np.count_nonzero(called & (t == 1)))
    false_pos = int(np.count_nonzero(called)) - true_pos
    true_neg = int(np.count_nonzero(uncalled & (t == 0)))
    false_neg = int(np.count_nonzero(uncalled)) - true_neg
    return true_pos, false_pos, true_neg, false_neg


def _ratio(num, den, complaint=None):
    if den == 0:
        if complaint:
            print(complaint)
        return 0
    return num / den


def precision_recall(true_pos, false_pos, false_neg):
    precision = _ratio(true_pos, true_pos + false_pos, "Precision could not be calculated.")
    recall = _ratio(true_pos, true_pos + false_neg, "Recall could not be calculated.")
    return precision, recall


def calculate_accuracy(true_pos, false_pos, true_neg, false_neg):
    return _ratio(true_pos + true_neg, true_pos + false_pos + true_neg + false_neg)


def f1(precision, recall):
    return _ratio(2 * (precision * recall), precision + recall,
                  "Precision, recall or both are zero. Unable of calculating weighted F1.")


def weighted_f1(precision, recall, n, N):
    return _ratio(2 * n / N * (precision * recall), precision + recall,
                  "Precision, recall or both are zero. Unable of calculating weighted F1.")


# ------------------------------------------------------------------------------ threshold sweeps
PrecisionRecallCurve = collections.namedtuple("PrecisionRecallCurve", "precision recall area_trapezoid")
RocCurve = collections.namedtuple("RocCurve", "fpr tpr area_trapezoid")


def confusion_curve(scores, labels, thresholds, logits=False):
    """``confusion_matrix(labels, scores >= t)`` for every threshold t: int64 ``[T, 4]`` rows of (tp, fp, tn, fn), in the
    order of ``thresholds`` (unsorted and repeated thresholds are fine; 1 <= T <= 4096, none NaN).

    ``scores`` are float32 probabilities (``logits=True``: logits, turned into probabilities as the network's head
    does), compared as doubles with each threshold - ties count as positive, NaN scores are never positive.  Labels
    other than 0 / 1 count as ``confusion_matrix`` counts them.  Either argument may be a numpy array (staged to the
    GPU; other float dtypes must hold float32 values exactly) or a CUDA tensor (float32 / uint8 contiguous tensors
    are used in place).  One pass over the data on the GPU whatever T is; only the counts come back."""
    from . import _cabi
    th = np.ascontiguousarray(np.asarray(thresholds, dtype=np.float64).reshape(-1))
    counts = np.zeros((th.size, 4), np.int64)
    n_th = min(th.size, 2 ** 31 - 1)
    n = _length(scores)
    if _length(labels) != n:
        raise ValueError("Length of labels to compare is not equal.")
    lib = _cabi.load_library()
    if n == 0:
        _cabi.check(lib.cf_sweep_thresholds(0, None, int(bool(logits)), None, 0, th.ctypes.data, n_th,
                                            counts.ctypes.data_as(_cabi.c_i64_p), None))
        return counts
    import torch
    dev = next((x.device.index for x in (scores, labels) if _is_cuda_tensor(x)), None)
    if dev is None:
        from . import get_device
        dev = get_device()
    with torch.cuda.device(dev):
        s = _device_scores(torch, scores, dev)
        y = _device_labels(torch, labels, dev)
        _cabi.check(lib.cf_sweep_thresholds(dev, s.data_ptr(), int(bool(logits)), y.data_ptr(), n, th.ctypes.data, n_th,
                                            counts.ctypes.data_as(_cabi.c_i64_p),
                                            torch.cuda.current_stream(dev).cuda_stream))
    return counts


def _is_cuda_tensor(x):
    return hasattr(x, "data_ptr") and getattr(x, "is_cuda", False)


def _length(x):
    return int(x.numel()) if _is_cuda_tensor(x) else int(np.asarray(x).size)


def _device_scores(torch, scores, dev):
    if _is_cuda_tensor(scores):
        if scores.device.index != dev:
            raise ValueError("scores and labels are on different devices")
        if scores.dtype != torch.float32:
            raise ValueError("scores must be a float32 tensor")
        return scores.reshape(-1).contiguous()
    s = np.asarray(scores).reshape(-1)
    s32 = np.ascontiguousarray(s, dtype=np.float32)
    if s.dtype != np.float32 and not np.array_equal(s32, s, equal_nan=True):
        raise ValueError("scores must hold float32 values (the library's probabilities are float32)")
    return torch.from_numpy(s32).to("cuda:%d" % dev)


def _device_labels(torch, labels, dev):
    if _is_cuda_tensor(labels):
        if labels.device.index != dev:
            raise ValueError("scores and labels are on different devices")
        y = labels.reshape(-1)
        if y.dtype != torch.uint8:
            if y.is_floating_point() or y.is_complex() or (y.numel() and (int(y.min()) < 0 or int(y.max()) > 255)):
                raise ValueError("labels must be small non-negative integers")
            y = y.to(torch.uint8)
        return y.contiguous()
    y = np.asarray(labels).reshape(-1)
    y8 = y.astype(np.uint8)
    if not np.array_equal(y8, y):
        raise ValueError("labels must be small non-negative integers")
    return torch.from_numpy(np.ascontiguousarray(y8)).to("cuda:%d" % dev)


def _counts_rows(counts):
    c = np.asarray(counts)
    if c.ndim != 2 or c.shape[1] != 4:
        raise ValueError("counts must be [T, 4] rows of (tp, fp, tn, fn)")
    return [c[:, i].astype(np.float64) for i in range(4)]


def _rates(num, den):
    """num / den per row, 0 where den == 0 (the rule of ``_ratio``, without the message)."""
    out = np.zeros(num.shape, np.float64)
    np.divide(num, den, out=out, where=den != 0)
    return out


def _trapezoid(x, y):
    """Area under the points (x, y) by the trapezoid rule, taken in increasing x (ties: increasing y).  Only the
    given points are used: nothing is added at x = 0 or x = 1, so a sparse sweep gives a partial area."""
    order = np.lexsort((y, x))
    x, y = x[order], y[order]
    return float(np.sum((x[1:] - x[:-1]) * (y[1:] + y[:-1]) * 0.5))


def precision_recall_curve(counts):
    """Per row of ``confusion_curve``: precision tp / (tp + fp) and recall tp / (tp + fn), 0 where a denominator is 0
    (as ``precision_recall``), and the trapezoid-rule area under precision over recall at these thresholds."""
    tp, fp, tn, fn = _counts_rows(counts)
    precision, recall = _rates(tp, tp + fp), _rates(tp, tp + fn)
    return PrecisionRecallCurve(precision, recall, _trapezoid(recall, precision))


def roc_curve(counts):
    """Per row of ``confusion_curve``: false-positive rate fp / (fp + tn) and true-positive rate tp / (tp + fn), 0 where
    a denominator is 0, and the trapezoid-rule area under the true-positive rate over the false-positive rate at these
    thresholds (the ROC AUC only when the thresholds reach both corners)."""
    tp, fp, tn, fn = _counts_rows(counts)
    fpr, tpr = _rates(fp, fp + tn), _rates(tp, tp + fn)
    return RocCurve(fpr, tpr, _trapezoid(fpr, tpr))


def average_precision(counts):
    """sklearn's ``average_precision_score`` over the rows of ``confusion_curve`` (or ``score_curve``): the step sum
    ``sum (R_i - R_{i-1}) P_i`` with the rows taken in increasing number of predicted positives (tp + fp) from recall
    0; precision is 0 where nothing is predicted positive.  NaN when no row has a positive label.  Over a sweep it
    covers only the given thresholds; over every row of a ``score_curve`` without NaN scores it is that curve's
    ``average_precision``."""
    tp, fp, tn, fn = _counts_rows(counts)
    positives = tp + fn
    if not positives.size or not positives.any():
        return float("nan")
    order = np.lexsort((tp, tp + fp))
    tp, predicted, positives = tp[order], (tp + fp)[order], positives[order]
    recall = _rates(tp, positives)
    return float(np.sum(np.diff(recall, prepend=0.0) * _rates(tp, predicted)))


# ------------------------------------------------------------------------------ exact curves
ScoreCurve = collections.namedtuple("ScoreCurve", "thresholds counts roc_auc average_precision")


def score_curve(scores, labels, logits=False, points=True):
    """The exact curve at every distinct score (K13, ``cf_curve_create``): ``ScoreCurve(thresholds, counts, roc_auc,
    average_precision)``.

    ``thresholds`` float64 ``[P]`` holds +inf and then every distinct non-NaN score in decreasing order; row i of
    ``counts`` (int64 ``[P, 4]``, tp, fp, tn, fn) is ``confusion_curve(scores, labels, [thresholds[i]])``, so
    ``roc_curve`` and ``precision_recall_curve`` apply to it unchanged - these are the points of sklearn's
    ``roc_curve`` without ``drop_intermediate``.  ``roc_auc`` and ``average_precision`` are sklearn's
    ``roc_auc_score`` and ``average_precision_score``, with NaN scores taken as one tie below every number (they
    close the curve at (1, 1)); NaN when a class they divide by is empty.  Deterministic.

    Labels must be 0 or 1 and scores NaN or in [0, 1] (``logits=True``: logits, mapped as the network's head does).
    Inputs are staged as ``confusion_curve`` stages them: numpy arrays are checked on the host and uploaded, CUDA
    float32 / uint8 tensors are used in place and checked on the device.  The GPU sorts every score; with
    ``points=False`` only the areas come back (``thresholds`` and ``counts`` are None), which saves the copy of a
    curve that can hold as many rows as positions."""
    from . import _cabi
    import ctypes
    n = _length(scores)
    if _length(labels) != n:
        raise ValueError("Length of labels to compare is not equal.")
    lib = _cabi.load_library()
    if not _is_cuda_tensor(labels):
        y = np.asarray(labels).reshape(-1)
        bad = np.flatnonzero((y != 0) & (y != 1))
        if bad.size:
            raise ValueError("score curve: label %r at position %d is not 0 or 1" % (y[bad[0]], bad[0]))
    if not logits and not _is_cuda_tensor(scores):
        s = np.asarray(scores).reshape(-1)
        bad = np.flatnonzero(~np.isnan(s) & ((s < 0) | (s > 1)))
        if bad.size:
            raise ValueError("score curve: score %r at position %d is neither NaN nor in [0, 1]" % (s[bad[0]], bad[0]))
    handle = ctypes.c_void_p()
    if n == 0:
        _cabi.check(lib.cf_curve_create(0, None, int(bool(logits)), None, 0, None, ctypes.byref(handle)))
    else:
        import torch
        dev = next((x.device.index for x in (scores, labels) if _is_cuda_tensor(x)), None)
        if dev is None:
            from . import get_device
            dev = get_device()
        with torch.cuda.device(dev):
            s = _device_scores(torch, scores, dev)
            y = _device_labels(torch, labels, dev)
            _cabi.check(lib.cf_curve_create(dev, s.data_ptr(), int(bool(logits)), y.data_ptr(), n,
                                            torch.cuda.current_stream(dev).cuda_stream, ctypes.byref(handle)))
    try:
        rows = ctypes.c_int64()
        auc, ap = ctypes.c_double(), ctypes.c_double()
        _cabi.check(lib.cf_curve_summary(handle, ctypes.byref(rows), None, None, None, ctypes.byref(auc),
                                         ctypes.byref(ap)))
        thresholds = counts = None
        if points:
            thresholds = np.empty(rows.value, np.float64)
            counts = np.empty((rows.value, 4), np.int64)
            _cabi.check(lib.cf_curve_read(handle, 0, rows.value, thresholds.ctypes.data, counts.ctypes.data))
        return ScoreCurve(thresholds, counts, auc.value, ap.value)
    finally:
        lib.cf_curve_destroy(handle)
