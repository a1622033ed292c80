"""Exact score curves on the GPU (K13): metrics.score_curve against the numpy oracle row for row, against the merged
threshold sweep (K11) at the curve's own thresholds, and evaluate_reads_curve against score_curve of infer_reads'
scores."""
import ctypes

import numpy as np
import pytest

from helpers import random_labels
import curve_oracle

TILE = 4096                    # keys per tile of the sort and of the run count


def _scores(kind, n, rng):
    if kind == "uniform":
        s = rng.random(n, dtype=np.float32)
    elif kind == "grid":                                     # heavy ties: 257 values
        s = (rng.integers(0, 257, n) / 256.0).astype(np.float32)
    elif kind == "sigmoid":                                  # piles at 0 and 1 (exact 0.0 / 1.0 among them)
        s = (1.0 / (1.0 + np.exp(-rng.normal(0, 4, n) * 8))).astype(np.float32)
    elif kind == "equal":
        s = np.full(n, 0.37, np.float32)
    elif kind == "specials":                                 # 0, 1, -0.0 next to +0.0, subnormals
        pool = np.array([0.0, -0.0, 1.0, 1e-45, 3e-42, np.float32(1.17e-38), 0.5, np.nextafter(np.float32(1), 0)],
                        np.float32)
        s = pool[rng.integers(0, pool.size, n)]
    elif kind == "nan":
        s = rng.random(n, dtype=np.float32)
        s[rng.random(n) < 0.2] = np.nan
    else:
        raise ValueError(kind)
    return s


def _labels(kind, n, rng):
    if kind == "positives":
        return np.ones(n, np.uint8)
    if kind == "negatives":
        return np.zeros(n, np.uint8)
    return (rng.random(n) < 0.3).astype(np.uint8)


def _on_device(torch, s, y, offset):
    """CUDA tensors holding s and y at `offset` elements into larger buffers (offset 1..3: the scalar-load path)."""
    sd = torch.zeros(s.size + 4, dtype=torch.float32, device="cuda")
    yd = torch.zeros(y.size + 4, dtype=torch.uint8, device="cuda")
    sd[offset:offset + s.size] = torch.from_numpy(s).cuda()
    yd[offset:offset + y.size] = torch.from_numpy(y).cuda()
    return sd[offset:offset + s.size], yd[offset:offset + y.size]


def _same_area(got, want):
    if np.isnan(want):
        return np.isnan(got)
    return got == pytest.approx(want, rel=1e-12, abs=0.0)


def _check(s, y, offset, logits=False, rng=None):
    import torch
    from catfish_b200 import metrics
    sd, yd = _on_device(torch, s, y, offset)
    got = metrics.score_curve(sd, yd, logits=logits)
    if not logits:
        th, counts, auc, ap = curve_oracle.curve(s, y)
        assert np.array_equal(got.thresholds, th)
        assert np.array_equal(got.counts, counts)
        assert _same_area(got.roc_auc, auc), (got.roc_auc, auc)
        assert _same_area(got.average_precision, ap), (got.average_precision, ap)
    # pinned to the merged sweep: confusion_curve at up to 4096 of the curve's thresholds gives those rows
    rng = rng or np.random.default_rng(0)
    rows = np.sort(rng.choice(got.counts.shape[0], min(4096, got.counts.shape[0]), replace=False))
    assert np.array_equal(metrics.confusion_curve(sd, yd, got.thresholds[rows], logits=logits), got.counts[rows])
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 31, TILE - 1, TILE, TILE + 1, 3 * TILE + 17])
@pytest.mark.parametrize("kind", ["uniform", "grid", "sigmoid", "equal", "specials", "nan"])
def test_curve_equals_oracle(kind, n):
    rng = np.random.default_rng(n * 7 + len(kind))
    s, y = _scores(kind, n, rng), _labels("mixed", n, rng)
    _check(s, y, offset=n % 4, rng=rng)


@pytest.mark.gpu
@pytest.mark.parametrize("labels", ["positives", "negatives"])
@pytest.mark.parametrize("n", [1, 4097])
def test_curve_of_one_class_has_nan_areas(labels, n):
    rng = np.random.default_rng(n)
    s, y = _scores("nan", n, rng), _labels(labels, n, rng)
    got = _check(s, y, offset=1, rng=rng)
    assert np.isnan(got.roc_auc)
    assert np.isnan(got.average_precision) == (labels == "negatives")


@pytest.mark.gpu
@pytest.mark.parametrize("kind, offset", [("uniform", 0), ("grid", 3), ("sigmoid", 1), ("nan", 2)])
def test_curve_over_many_tiles(kind, offset):
    n = (1 << 25) + 12345                                     # 8195 tiles: runs cross tile boundaries
    rng = np.random.default_rng(25)
    s = _scores(kind, n, rng)
    y = _labels("mixed", n, rng)
    _check(s, y, offset, rng=rng)


@pytest.mark.gpu
def test_curve_of_logits_follows_the_head_sigmoid():
    rng = np.random.default_rng(3)
    n = 3 * TILE + 5
    z = rng.normal(0, 6, n).astype(np.float32)
    z[::101] = np.nan
    z[1::211] = np.inf
    z[2::307] = -np.inf
    got = _check(z, _labels("mixed", n, rng), offset=2, logits=True, rng=rng)
    assert got.thresholds[0] == np.inf and (np.diff(got.thresholds[1:]) < 0).all()
    assert got.thresholds[1] == 1.0 and got.thresholds[-1] == 0.0
    assert (np.diff(got.counts[:, 0] + got.counts[:, 1]) > 0).all()


@pytest.mark.gpu
def test_curve_is_deterministic_and_reads_in_windows():
    import torch
    from catfish_b200 import _cabi, metrics
    rng = np.random.default_rng(9)
    n = 5_000_000
    s, y = _scores("sigmoid", n, rng), _labels("mixed", n, rng)
    sd, yd = _on_device(torch, s, y, 0)
    a, b = metrics.score_curve(sd, yd), metrics.score_curve(sd, yd)
    assert np.array_equal(a.thresholds, b.thresholds) and np.array_equal(a.counts, b.counts)
    assert a.roc_auc == b.roc_auc and a.average_precision == b.average_precision        # bit for bit
    c = metrics.score_curve(sd, yd, points=False)
    assert c.thresholds is None and (c.roc_auc, c.average_precision) == (a.roc_auc, a.average_precision)
    lib = _cabi.load_library()
    h = ctypes.c_void_p()
    _cabi.check(lib.cf_curve_create(0, sd.data_ptr(), 0, yd.data_ptr(), n, torch.cuda.current_stream().cuda_stream,
                                    ctypes.byref(h)))
    try:
        p, nn = ctypes.c_int64(), ctypes.c_int64()
        _cabi.check(lib.cf_curve_summary(h, ctypes.byref(p), None, None, ctypes.byref(nn), None, None))
        assert p.value == a.counts.shape[0] and nn.value == 0
        th, counts = np.empty(p.value), np.empty((p.value, 4), np.int64)
        cuts = [0, 1, 2, 1000, p.value // 2, p.value - 1, p.value]
        for lo, hi in zip(cuts, cuts[1:]):
            _cabi.check(lib.cf_curve_read(h, lo, hi - lo, th[lo:].ctypes.data, counts[lo:].ctypes.data))
        assert np.array_equal(th, a.thresholds) and np.array_equal(counts, a.counts)
        assert lib.cf_curve_read(h, 1, p.value, None, None) == _cabi.CF_ERR_BAD_ARG
    finally:
        lib.cf_curve_destroy(h)


@pytest.mark.gpu
@pytest.mark.parametrize("where, score, label", [(0, 0.5, 2), (4096 + 7, 1.5, 1), (9999, -0.25, 0), (123, np.inf, 0)])
def test_bad_input_on_the_device_names_the_position(where, score, label):
    import torch
    from catfish_b200 import metrics
    rng = np.random.default_rng(4)
    n = 10_000
    s, y = _scores("uniform", n, rng), _labels("mixed", n, rng)
    s[where], y[where] = score, label
    s[where + 1:][:3] = 7.0                                  # later bad positions are not the first
    sd, yd = _on_device(torch, s, y, 1)
    with pytest.raises(ValueError, match="position %d " % where):
        metrics.score_curve(sd, yd)
    ok = s.copy()
    ok[where:where + 4] = 0.5
    y[where] = 1
    sd, yd = _on_device(torch, ok, y, 1)                      # the device still works
    got = metrics.score_curve(sd, yd)
    assert np.array_equal(got.counts, curve_oracle.curve(ok, y)[1])


# ------------------------------------------------------------------------------ read level
@pytest.fixture(scope="module")
def model(shipped_weights):
    from catfish_b200 import neural_network, weights
    m = neural_network.build_model("ResNetRNN", **weights.SHIPPED_HPARAMS)
    m.set_weights(shipped_weights)
    return m


@pytest.mark.gpu
def test_evaluate_reads_curve_equals_score_curve_of_infer_reads(model, monkeypatch):
    from catfish_b200 import infer, metrics, synth
    rng = np.random.default_rng(42)
    reads = synth.synth_reads([9001, 35, 17_777, 4_003, 70, 60_000], base_seed=7)
    reads.append(np.full(1234, 480, np.int16))                # MAD = 0: NaN scores
    labels = [random_labels(rng, r.size).astype(np.uint8) for r in reads]
    _, _, scores = infer.infer_reads(reads, model, return_scores=True)
    want = metrics.score_curve(np.concatenate(scores), np.concatenate(labels))
    got = infer.evaluate_reads_curve(reads, labels, model)
    assert np.array_equal(got.thresholds, want.thresholds) and np.array_equal(got.counts, want.counts)
    assert (got.roc_auc, got.average_precision) == (want.roc_auc, want.average_precision)
    areas = infer.evaluate_reads_curve(reads, labels, model, points=False)
    assert areas.counts is None and (areas.roc_auc, areas.average_precision) == (want.roc_auc, want.average_precision)
    # several groups, each writing its probabilities at its offset
    monkeypatch.setattr(infer, "_GROUP_SAMPLES", 20_000)
    split = infer.evaluate_reads_curve(reads, labels, model)
    assert np.array_equal(split.counts, want.counts) and split.roc_auc == want.roc_auc
    with pytest.raises(ValueError):
        infer.evaluate_reads_curve(reads, [l[:-1] for l in labels], model)
    with pytest.raises(ValueError):
        infer.evaluate_reads_curve(reads[:1], [np.full(reads[0].size, 2, np.uint8)], model)
    with pytest.raises(IndexError):
        infer.evaluate_reads_curve([np.zeros(0, np.int16)], [np.zeros(0, np.uint8)], model)
    empty = infer.evaluate_reads_curve([], [], model)
    assert empty.counts.tolist() == [[0, 0, 0, 0]]
