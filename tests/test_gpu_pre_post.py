"""GPU: K1 (median/MAD normalisation) and K6 (interval calling) through the C ABI,
bit-exact against the oracle restatement of infer.py and the golden vectors."""
import numpy as np
import pytest

from helpers import golden, random_labels
from catfish_b200 import infer, synth
from oracle import postprocess

pytestmark = pytest.mark.gpu


def test_normalize_golden_bit_exact():
    g = golden("postprocess.npz")
    for i in range(int(g["n_raws"])):
        raw = g["raw%d" % i]
        got = infer.normalize_raw_signal(raw, "median")
        np.testing.assert_array_equal(got, g["raw%d_norm" % i])       # NaN/inf positions included
    with pytest.raises(ValueError):
        infer.normalize_raw_signal(np.array([1, 2, 3], np.int16), "zscore")


def test_read_stats_ragged_batch_exact():
    rng = np.random.default_rng(1)
    reads = synth.synth_reads([1, 2, 3, 35, 70, 777, 10000, 50001], base_seed=10)
    reads.append(rng.integers(-32768, 32768, size=4001).astype(np.int16))        # wide path, odd n
    reads.append(rng.integers(-32768, 32768, size=4000).astype(np.int16))        # wide path, even n
    reads.append(np.full(100, 7, np.int16))                                      # constant: scale 0
    reads.append(np.array([-32768, -32768, 32767, 32767], np.int16))
    reads.append(rng.integers(0, 8192, size=30000).astype(np.int16))             # exactly fills smem bins
    st = infer.read_stats(reads)
    for r, (shift, scale) in zip(reads, st):
        want_shift = np.median(r)
        want_scale = np.median(np.abs(r - want_shift))
        assert shift == want_shift and scale == want_scale, (len(r), shift, want_shift, scale, want_scale)


def test_read_stats_many_short_reads_one_cta_per_read():
    """>= 296 short reads take the one-CTA-per-read kernel (fewer, longer reads are chunked over CTAs)."""
    rng = np.random.default_rng(2)
    reads = synth.synth_reads(rng.integers(1, 3000, size=400), base_seed=2000)
    reads[7] = rng.integers(-32768, 32768, size=999).astype(np.int16)        # wide path inside the batch
    st = infer.read_stats(reads)
    for r, (shift, scale) in zip(reads, st):
        want_shift = np.median(r)
        assert shift == want_shift and scale == np.median(np.abs(r - want_shift))


def test_read_stats_long_read():
    raw = synth.synth_read(1_000_000, 77)
    st = infer.read_stats([raw])[0]
    shift = np.median(raw)
    assert st[0] == shift and st[1] == np.median(np.abs(raw - shift))


def _call_intervals(probs_list, dtype, lead=0, **kw):
    """cf_call_intervals on a ragged batch of probability arrays, placed after `lead` values that belong to no read
    (lead 1-3 moves the first read's device pointer off 16-byte alignment)."""
    import ctypes
    import torch
    from catfish_b200 import _cabi
    lib = _cabi.load_library()
    offsets = np.full(len(probs_list) + 1, lead, np.int64)
    offsets[1:] += np.cumsum([len(p) for p in probs_list], dtype=np.int64)
    flat = np.concatenate([np.ones(lead)] + list(probs_list)).astype(dtype)
    min_run = kw.get("min_run", 15)
    cap = int(lib.cf_max_intervals(len(flat), len(probs_list), min_run))
    pd = torch.from_numpy(flat).cuda()
    out = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    ioff = torch.empty(len(probs_list) + 1, dtype=torch.int64, device="cuda")
    _cabi.check(lib.cf_call_intervals(0, pd.data_ptr(), 1 if dtype == np.float64 else 0,
                                      offsets.ctypes.data_as(_cabi.c_i64_p), len(probs_list), out.data_ptr(),
                                      ioff.data_ptr(), cap, kw.get("threshold", 0.5), min_run,
                                      kw.get("ext_left", 11), kw.get("ext_right", 16),
                                      torch.cuda.current_stream().cuda_stream))
    ioff = ioff.cpu().numpy()
    out = out.cpu().numpy()
    assert ioff[-1] <= cap
    return [out[ioff[r]:ioff[r + 1]].tolist() for r in range(len(probs_list))]


def _oracle_intervals(p, threshold=0.5, min_run=15, ext_left=11, ext_right=16):
    labels = postprocess.correct_short(postprocess.class_from_threshold(p, threshold), min_run)
    return postprocess.hp_in_pred(labels, ext_left, ext_right)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_call_intervals_ragged_random(dtype):
    rng = np.random.default_rng(3)
    lens = [1, 14, 15, 16, 31, 32, 33, 64, 100, 1000, 8191, 8192, 8193, 20000, 3, 70000]
    probs = []
    for i, n in enumerate(lens):
        lab = random_labels(rng, n, p_switch=[0.03, 0.08, 0.3][i % 3])
        p = np.where(lab == 1, 0.5 + 0.5 * rng.random(n), 0.5 * rng.random(n) - 1e-9).astype(dtype)
        p[rng.integers(0, n, size=max(1, n // 50))] = 0.5                  # exactly on the threshold: counts as 1
        probs.append(p)
    for lead in (0, 1, 2, 3):          # f32 at leads 1-3: the unaligned (ballot) pack kernel
        got = _call_intervals(probs, dtype, lead=lead)
        for p, g in zip(probs, got):
            assert g == _oracle_intervals(p.astype(np.float64))
    # other parameters
    got = _call_intervals(probs, dtype, threshold=0.9, min_run=4, ext_left=0, ext_right=3)
    for p, g in zip(probs, got):
        assert g == _oracle_intervals(p.astype(np.float64), 0.9, 4, 0, 3)


def test_call_intervals_edge_patterns():
    ones = lambda n: np.ones(n, np.float32)
    zeros = lambda n: np.zeros(n, np.float32)
    cases = [ones(1), zeros(1), ones(15), ones(14), ones(100000), zeros(100000),
             np.concatenate([ones(20), zeros(5)]), np.concatenate([zeros(5), ones(20)]),
             np.concatenate([ones(14), zeros(3), ones(15)]), np.concatenate([ones(31), zeros(1), ones(32)]),
             np.concatenate([zeros(17), ones(64), zeros(1), ones(64)]),
             np.full(50, np.nan, np.float32)]
    got = _call_intervals(cases, np.float32)
    for p, g in zip(cases, got):
        assert g == _oracle_intervals(p.astype(np.float64)), len(p)
    # runs must not leak across read boundaries: all-ones neighbours stay separate intervals
    got = _call_intervals([ones(10), ones(10), ones(40), ones(7)], np.float32)
    assert got == [[], [], [[-11, 56]], []]
    # empty reads have no intervals and keep their non-empty neighbours apart
    got = _call_intervals([ones(0), ones(20), ones(0), ones(20), zeros(3), ones(0)], np.float32)
    assert got == [[], [[-11, 36]], [], [[-11, 36]], [], []]
    assert _call_intervals([], np.float32) == [] and _call_intervals([ones(0), ones(0)], np.float32) == [[], []]


def test_python_helpers_match_golden():
    g = golden("postprocess.npz")
    for i in range(int(g["n_patterns"])):
        p = g["pat%d" % i]
        np.testing.assert_array_equal(infer.correct_short(list(p)), g["pat%d_correct_short" % i])
        for lab in (1, 0):
            assert infer.hp_in_pred(list(p), label=lab) == g["pat%d_hp_label%d" % (i, lab)].tolist()
        assert infer.hp_in_pred(p, 3, 0) == g["pat%d_hp_ext" % i].tolist()
    s = g["scores"]
    assert infer.class_from_threshold(s) == g["scores_labels_0.5"].tolist()
    assert infer.class_from_threshold(list(s), 0.9) == g["scores_labels_0.9"].tolist()
    assert infer.hp_in_pred([1] * 20 + [0] * 5) == [[-11, 36]]
    out = infer.correct_short([1] * 14 + [0] * 3 + [1] * 15)
    assert out.tolist() == [0] * 17 + [1] * 15 and out.dtype == np.int64
    with pytest.raises(IndexError):
        infer.hp_in_pred([])
    with pytest.raises(IndexError):
        infer.correct_short([])
    rng = np.random.default_rng(9)
    for n, thr in ((5000, 15), (5000, 1), (777, 40)):
        lab = random_labels(rng, n) * rng.integers(1, 4, size=n)          # multi-valued labels
        np.testing.assert_array_equal(infer.correct_short(lab, thr), postprocess.correct_short(lab, thr))
        assert infer.hp_in_pred(lab, label=2) == postprocess.hp_in_pred(lab, label=2)


def test_interval_calling_property_based():
    """hypothesis: arbitrary small label patterns, thresholds and run lengths against the loop oracle."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=60, deadline=None)
    @given(st.lists(st.lists(st.integers(0, 1), min_size=1, max_size=200), min_size=1, max_size=6),
           st.integers(1, 40), st.integers(0, 20), st.integers(0, 20))
    def check(label_lists, min_run, ext_left, ext_right):
        probs = [np.where(np.array(l) == 1, 0.75, 0.25).astype(np.float32) for l in label_lists]
        got = _call_intervals(probs, np.float32, min_run=min_run, ext_left=ext_left, ext_right=ext_right)
        for l, g in zip(label_lists, got):
            labels = postprocess.correct_short_loops(list(l), min_run)
            assert g == postprocess.hp_in_pred_loops(list(labels), ext_left, ext_right)

    check()
