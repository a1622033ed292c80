"""numpy statement of the exact score curve (metrics.score_curve, cf_curve_create): a stable sort, the ends of runs of
distinct scores, cumulative counts; for the areas NaN scores are one tie below every number."""
import numpy as np


def curve(scores, labels):
    """(thresholds float64 [P], counts int64 [P, 4] = tp, fp, tn, fn, roc_auc, average_precision)."""
    s = np.asarray(scores).reshape(-1).astype(np.float64)
    y = np.asarray(labels).reshape(-1).astype(np.int64)
    nan = np.isnan(s)
    order = np.argsort(-s[~nan], kind="stable")
    ss, ys = s[~nan][order], y[~nan][order]
    ends = np.flatnonzero(np.r_[ss[1:] != ss[:-1], True]) if ss.size else np.zeros(0, np.int64)
    tp = np.r_[0, np.cumsum(ys)[ends]].astype(np.int64)
    fp = np.r_[0, ends + 1].astype(np.int64) - tp
    n1 = int(y.sum())
    n0 = y.size - n1
    thresholds = np.r_[np.inf, ss[ends]]
    counts = np.stack([tp, fp, n0 - fp, n1 - tp], axis=1)
    # the closing point (N0, N1): every position positive, NaN scores included
    tpc, fpc = np.r_[tp, n1], np.r_[fp, n0]
    auc = ap = float("nan")
    if n0 and n1:
        auc = int(np.sum(np.diff(fpc) * (tpc[1:] + tpc[:-1]))) / (2.0 * n0 * n1)     # int64: at most n^2 / 2
    if n1:
        dt = np.diff(tpc)
        keep = dt > 0
        ap = float(np.sum(dt[keep] * (tpc[1:][keep] / (tpc[1:][keep] + fpc[1:][keep])))) / n1
    return thresholds, counts, auc, ap


def rates(counts):
    """(fpr, tpr, precision, recall) per row, 0 where a denominator is 0."""
    tp, fp, tn, fn = [counts[:, i].astype(np.float64) for i in range(4)]

    def div(a, b):
        out = np.zeros(a.shape)
        np.divide(a, b, out=out, where=b != 0)
        return out

    return div(fp, fp + tn), div(tp, tp + fn), div(tp, tp + fp), div(tp, tp + fn)
