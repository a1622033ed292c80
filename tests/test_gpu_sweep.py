"""Threshold sweeps on the GPU (K11): cf_validate_windows_sweep against K9 at every threshold, cf_sweep_thresholds
against numpy counting of the library's own probabilities, and evaluate_reads against both."""
import numpy as np
import pytest

from helpers import random_labels


def _model(shipped_weights, engine="auto"):
    from catfish_b200 import neural_network, weights
    m = neural_network.build_model("ResNetRNN", engine=engine, **weights.SHIPPED_HPARAMS)
    m.set_weights(shipped_weights)
    return m


@pytest.fixture(scope="module")
def model(shipped_weights):
    return _model(shipped_weights)


@pytest.fixture(scope="module")
def scored(model):
    """Seeded ragged reads, one of them constant (MAD = 0: NaN scores), their probabilities from infer_reads and
    labels with a few values other than 0 / 1."""
    from catfish_b200 import infer, synth
    rng = np.random.default_rng(42)
    reads = synth.synth_reads([9001, 35, 17_777, 4_003, 70], base_seed=7)
    reads.append(np.full(1234, 480, np.int16))
    _, _, scores = infer.infer_reads(reads, model, return_scores=True)
    labels = [random_labels(rng, r.size).astype(np.uint8) for r in reads]
    labels[2][::97] = 2
    labels[3][5] = 7
    return reads, labels, np.concatenate(scores), np.concatenate(labels)


def _numpy_curve(scores, labels, thresholds):
    from catfish_b200 import metrics
    s = np.asarray(scores).astype(np.float64)
    return np.array([metrics.confusion_matrix(labels, (s >= t).astype(np.int64)) for t in thresholds], np.int64)


def _check_invariants(counts, labels):
    assert (counts.sum(axis=1) == labels.size).all()
    if set(np.unique(labels).tolist()) <= {0, 1}:
        assert (counts[:, 0] + counts[:, 3] == (labels == 1).sum()).all()     # tp + fn: the positives, at every t
    return counts


# ------------------------------------------------------------------------------ (1) against K9, bit for bit
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["auto", "simt"])
def test_validate_sweep_equals_test_network_at_every_threshold(engine, shipped_weights):
    from catfish_b200 import train_validate
    m = _model(shipped_weights, engine)
    rng = np.random.default_rng(11)
    thresholds = np.linspace(0.0, 1.0, 257)
    rng.shuffle(thresholds)
    for n in (35 * 4, 2000, 4513):                # 140, 2030 and 4515 positions: n % 4 = 0, 2, 3
        data = rng.normal(0, 1.5, n)
        labels = (rng.random(n) < 0.3).astype(np.int64)
        x, pad = train_validate.padding(data)
        y, _ = train_validate.padding(labels)
        m.reset_sweep()
        acc_s, loss_s = m.test_network_sweep(x, y, thresholds, pad)
        sweep = m.sweep_counts.copy()
        assert sweep.shape == (257, 4) and sweep.dtype == np.int64
        for i, t in enumerate(thresholds):
            m.tp = m.fp = m.tn = m.fn = 0
            acc, loss = m.test_network(x, y, None, None, pad, threshold=float(t))
            assert [m.tp, m.fp, m.tn, m.fn] == sweep[i].tolist(), (n, t)
            assert acc == acc_s and loss == loss_s
        assert (sweep.sum(axis=1) == x.shape[0] * 35 - pad).all()
    # the accumulator adds over calls and refuses another threshold count until reset
    m.reset_sweep()
    m.test_network_sweep(x, y, thresholds, pad)
    m.test_network_sweep(x, y, thresholds, pad)
    assert np.array_equal(m.sweep_counts, 2 * sweep)
    with pytest.raises(ValueError):
        m.test_network_sweep(x, y, thresholds[:3], pad)
    m.reset_sweep()
    assert m.sweep_counts is None


@pytest.mark.gpu
def test_validate_driver_with_thresholds(model):
    from catfish_b200 import metrics, train_validate
    rng = np.random.default_rng(3)
    reads = [(rng.normal(0, 1.5, n), (rng.random(n) < 0.2).astype(int)) for n in (900, 1500, 300)]
    thresholds = [0.5, 0.2, 0.9]
    acc, prec, rec = train_validate.validate(model, reads, 700, None, validation_start=0, thresholds=thresholds)
    assert model.sweep_counts is None and (model.tp, model.fp, model.tn, model.fn) == (0, 0, 0, 0)
    want = train_validate.validate(model, reads, 700, None, validation_start=0)       # default: threshold 0.5
    assert (acc[0], prec[0], rec[0]) == want
    # every threshold equals test_network's counts at that threshold over the same windows
    for i, t in enumerate(thresholds):
        model.tp = model.fp = model.tn = model.fn = 0
        for data, labels in reads[:2]:
            x, pad = train_validate.padding(data[:700])
            y, _ = train_validate.padding(labels[:700])
            model.test_network(x, y, None, None, pad, threshold=t)
        assert acc[i] == metrics.calculate_accuracy(model.tp, model.fp, model.tn, model.fn)
        assert (prec[i], rec[i]) == metrics.precision_recall(model.tp, model.fp, model.fn)
    model.tp = model.fp = model.tn = model.fn = 0


# ------------------------------------------------------------------------------ (2) against numpy, exact
@pytest.mark.gpu
def test_confusion_curve_equals_numpy(scored):
    from catfish_b200 import metrics
    _, _, scores, labels = scored
    assert np.isnan(scores).sum() == 1234
    real = scores[~np.isnan(scores)]
    rng = np.random.default_rng(1)
    ties = rng.choice(real, 40).astype(np.float64)                 # thresholds equal to some scores' values
    assert ties.size and all((real == t).any() for t in ties)
    special = [0.0, 1.0, -0.25, 1.5, -np.inf, np.inf, 0.5, float(np.nextafter(np.float32(0.5), np.float32(1))),
               0.5 + 1e-12, 1e300, -1e300]
    thresholds = np.concatenate([ties, special, ties[:7], [0.5, 0.0]])     # unsorted, with repeats
    rng.shuffle(thresholds)
    got = metrics.confusion_curve(scores, labels, thresholds)
    assert np.array_equal(got, _numpy_curve(scores, labels, thresholds))
    _check_invariants(got, labels)
    # ties count as positive: at the largest score exactly the scores equal to it are predicted 1
    t = float(real.max())
    top = metrics.confusion_curve(scores, labels, [t])[0]
    assert top[0] + top[1] == (real == real.max()).sum() > 0


@pytest.mark.gpu
def test_confusion_curve_one_and_4096_thresholds(scored):
    from catfish_b200 import metrics
    _, _, scores, labels = scored
    for th in ([0.5], [0.31], np.linspace(-0.1, 1.1, 4096)):
        got = metrics.confusion_curve(scores, labels, th)
        assert got.shape == (len(th), 4)
        assert np.array_equal(got, _numpy_curve(scores, labels, th))
    th = np.sort(np.concatenate([np.random.default_rng(2).choice(scores[~np.isnan(scores)], 4000), np.linspace(0, 1, 96)]))
    got = _check_invariants(metrics.confusion_curve(scores, labels, th), labels)
    assert np.array_equal(got, _numpy_curve(scores, labels, th))
    assert (np.diff(got[:, 0] + got[:, 1]) <= 0).all()             # predicted positives never grow with t
    assert np.array_equal(metrics.confusion_curve(scores, labels, th), got)          # deterministic


@pytest.mark.gpu
def test_confusion_curve_device_tensors_in_place_and_unaligned(scored):
    import torch
    from catfish_b200 import metrics
    _, _, scores, labels = scored
    th = np.linspace(0, 1, 101)
    s = torch.from_numpy(scores).cuda()
    y = torch.from_numpy(labels).cuda()
    want = _numpy_curve(scores, labels, th)
    assert np.array_equal(metrics.confusion_curve(s, y, th), want)
    assert np.array_equal(metrics.confusion_curve(s, labels, th), want)
    assert np.array_equal(metrics.confusion_curve(s, y.to(torch.int64), th), want)
    # odd offsets: the kernel's scalar-load path
    for off in (1, 3):
        assert np.array_equal(metrics.confusion_curve(s[off:], y[off:], th), _numpy_curve(scores[off:], labels[off:], th))
    with pytest.raises(ValueError):
        metrics.confusion_curve(s.double(), y, th)
    with pytest.raises(ValueError):
        metrics.confusion_curve(scores.astype(np.float64) + 1e-12, labels, th)      # not float32 values


@pytest.mark.gpu
def test_confusion_curve_of_logits_follows_the_head_sigmoid():
    import torch
    from catfish_b200 import metrics
    rng = np.random.default_rng(9)
    z = rng.normal(0, 4, 100_003).astype(np.float32)
    y = (rng.random(z.size) < 0.4).astype(np.uint8)
    p = torch.sigmoid(torch.from_numpy(z).cuda())
    th = np.linspace(0.01, 0.99, 99)
    got = metrics.confusion_curve(z, y, th, logits=True)
    _check_invariants(got, y)
    # the head's fp32 sigmoid and torch's may differ in the last bit: counts within the scores that close
    ref = _numpy_curve(p.cpu().numpy(), y, th)
    near = np.array([(np.abs(p.cpu().numpy().astype(np.float64) - t) < 1e-6).sum() for t in th])
    assert (np.abs(got - ref).max(axis=1) <= near).all()


@pytest.mark.gpu
def test_refusals_raise_value_error(scored):
    from catfish_b200 import _cabi, metrics
    _, _, scores, labels = scored
    for th in ([], np.zeros(4097), [0.1, np.nan]):
        with pytest.raises(ValueError):
            metrics.confusion_curve(scores, labels, th)
    lib = _cabi.load_library()
    th = np.array([0.5])
    out = np.zeros((1, 4), np.int64)
    assert lib.cf_sweep_thresholds(0, None, 0, None, 100, th.ctypes.data, 1, out.ctypes.data_as(_cabi.c_i64_p),
                                   None) == _cabi.CF_ERR_BAD_ARG
    assert lib.cf_sweep_thresholds(0, None, 0, None, -5, th.ctypes.data, 1, out.ctypes.data_as(_cabi.c_i64_p),
                                   None) == _cabi.CF_ERR_BAD_ARG


# ------------------------------------------------------------------------------ (3) read level
@pytest.mark.gpu
def test_evaluate_reads_equals_counting_infer_reads_scores(model, scored):
    from catfish_b200 import infer
    reads, labels, scores, flat = scored
    th = np.concatenate([np.linspace(0, 1, 65), [0.5, 0.07]])
    got = infer.evaluate_reads(reads, labels, model, th)
    assert np.array_equal(got, _numpy_curve(scores, flat, th))
    assert np.array_equal(infer.evaluate_reads(reads, labels, model, th), got)
    with pytest.raises(ValueError):
        infer.evaluate_reads(reads, [l[:-1] for l in labels], model, th)
    with pytest.raises(ValueError):
        infer.evaluate_reads(reads, labels, model, [np.nan])
    with pytest.raises(IndexError):
        infer.evaluate_reads([np.zeros(0, np.int16)], [np.zeros(0, np.uint8)], model, th)


@pytest.mark.gpu
def test_evaluate_reads_over_several_engine_passes(model):
    from catfish_b200 import infer, synth
    rng = np.random.default_rng(8)
    lengths = synth.ragged_lengths(90, 100_000, 200_000, seed=8)
    assert lengths.sum() > 1.1 * infer._GROUP_SAMPLES
    reads = synth.synth_reads(lengths, base_seed=80)
    labels = [random_labels(rng, r.size).astype(np.uint8) for r in reads]
    th = np.linspace(0.05, 0.95, 19)
    got = infer.evaluate_reads(reads, labels, model, th)
    _, _, scores = infer.infer_reads(reads, model, return_scores=True)
    want = _numpy_curve(np.concatenate(scores), np.concatenate(labels), th)
    assert np.array_equal(got, want)
    _check_invariants(got, np.concatenate(labels))
