"""GPU: the read path held bit for bit to the window path, on every kernel variant and across engine passes.

The window path (``model.infer``, cf_infer_windows) is held to float64 at each kernel's own budget by
test_gpu_operand_formats.py and test_gpu_precision_budgets.py.  Users call the read path (``infer_reads``,
``infer_concatenated``), which adds the K1 median / MAD and window table, the int16 gather inside the conv kernels and
k1_fill_windows, the head scatter that cuts the padding, the NaN rule for MAD = 0, the label bits and K6.  Both paths
read their samples through window_input and write through head_output (csrc/window_io.cuh), and the reference's own
pipeline (oracle/postprocess.infer_read) feeds the network exactly what window_input computes: numpy's float64
(raw - median) / MAD rounded to float32, the same zero padding (a whole extra window when 35 divides the length), and
``model.infer`` gives the float32 probabilities widened to float64.  So the read path must equal the window path bit
for bit, and that equality carries the window path's float64 budget over to it.

A. Ragged batches on every kernel variant: scores equal, lengths equal, and the intervals of the label-bit path
   (infer_reads and one infer_concatenated call, default and non-default calling parameters) equal the reference
   post-processing of the window-path scores, with no tolerance band.
B. Engine passes (2368 tiles on the tensor-core engine, 256 on the CUDA-core one): the window path against float64 on
   the tiles at the first pass boundary and the last, partial tile; one infer_concatenated call in which a read
   straddles the boundary at another tile phase than it has alone, bit for bit; one read longer than a group.
C. Label-bit ties on the three head kernels: a threshold equal to an occurring score counts it positive, one a
   quarter ulp above counts it negative although it rounds to the same float.
D. BASELINE config 3 (ResNetRNN, reads of 50k-200k samples) against float64 through the whole infer_reads pipeline.

tests/tools/read_path_mutants.patch holds the faults these tests catch; the measured values are in DESIGN.md
section 4.
"""
import os
import sys
import time

import numpy as np
import pytest

from helpers import allowed_label_flips, bn_weights, build_model, hparams
from catfish_b200 import infer, synth
from oracle import postprocess, tf_graph

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import precision_emulation as pe  # noqa: E402
# the window-path budgets of each variant, worst-tile RMS of p - p64 (the bf16x3 bounds are against the CUDA-core
# engine, which sits three orders of magnitude closer to float64 than they are)
from test_gpu_operand_formats import BF16X3_WMAX_BOUND, RNN_BOUND, SHIPPED_BOUND  # noqa: E402
from test_gpu_precision_budgets import BF16X3_CASES, _wmax_shipped  # noqa: E402

pytestmark = pytest.mark.gpu

WINDOW = 35
TILE = 128
TC_PASS_TILES = 2368             # kTcChunkTiles, csrc/tc_engine.cu
SIMT_PASS_TILES = 256            # kSimtChunkTiles, csrc/simt_engine.cu
K1_CTA_PER_READ = 2 * 148        # from this many reads (of < 64 Ki samples on average) K1 runs one CTA per read

VARIANTS = {
    # id: (kind, hyper-parameters, weights (seed; None: shipped; callable of the shipped ones), engine, operand
    #      format, window-path bound)
    "shipped": ("ResNetRNN", {}, None, "tcgen05", "f16e5", SHIPPED_BOUND),     # tc_conv4 gather, tc_head_kernel
    "rnn64x3": ("RNN", hparams("RNN", h=64, n_layers=3), 11, "tcgen05", "f16e5", RNN_BOUND),   # k1_fill_windows
    "resnet2": ("ResNet", hparams("ResNet", n_res=2), BF16X3_CASES["resnet-2-blocks"][2], "tcgen05", "bf16x3",
                BF16X3_CASES["resnet-2-blocks"][3]),                           # head fused into tc_conv4_kernel
    "resnet1": ("ResNet", hparams("ResNet", n_res=1), BF16X3_CASES["resnet-1-block"][2], "tcgen05", "bf16x3",
                BF16X3_CASES["resnet-1-block"][3]),                            # tc_conv2_kernel, tc_head_conv_kernel
    "resnetrnn1": ("ResNetRNN", hparams("ResNetRNN", n_res=1), BF16X3_CASES["resnetrnn-1-block"][2], "tcgen05",
                   "bf16x3", BF16X3_CASES["resnetrnn-1-block"][3]),            # tc_conv2_kernel, bf16x3 GRU
    "resnetrnn3": ("ResNetRNN", hparams("ResNetRNN", n_res=3), BF16X3_CASES["resnetrnn-3-blocks"][2], "tcgen05",
                   "bf16x3", BF16X3_CASES["resnetrnn-3-blocks"][3]),           # tc_conv_block_kernel
    "padded": ("ResNetRNN", hparams("ResNetRNN", c=16, h=32, n_res=3, n_layers=2), BF16X3_CASES["padded-c16-h32"][2],
               "tcgen05", "bf16x3", BF16X3_CASES["padded-c16-h32"][3]),        # zero-padded weights
    "wmax": ("ResNetRNN", {}, _wmax_shipped, "tcgen05", "bf16x3", BF16X3_WMAX_BOUND),   # bf16x3 GRU at KX = 128
    "simt": ("ResNetRNN", {}, None, "simt", "f32", None),                      # simt_head_kernel
}
TC_VARIANTS = [v for v in VARIANTS if VARIANTS[v][3] == "tcgen05"]
NON_DEFAULT_CALL = dict(threshold=0.3, min_run=7, extension_left=0, extension_right=5)

_MODELS = {}
_CACHE = {}


def _weights(case, shipped):
    kind, hpm, src = VARIANTS[case][:3]
    if src is None:
        return shipped
    if callable(src):
        return src(shipped)
    return bn_weights(kind, src, **hpm)


def _model(case, shipped):
    """(model, weights) of VARIANTS[case], built once per module; its engine and operand format are asserted, so a
    change of format choice cannot silently drop a case."""
    if case not in _MODELS:
        kind, hpm, _, engine, fmt, _ = VARIANTS[case]
        w = _weights(case, shipped)
        m = build_model(kind, engine, w, **hpm)
        assert m.resolved_engine == engine and m.operand_format == fmt, (case, m.resolved_engine, m.operand_format)
        _MODELS[case] = (m, w)
    return _MODELS[case]


def n_windows(length):
    return length // WINDOW + 1          # padding: a whole extra window when 35 divides the length


def mad_is_zero(raw):
    raw = np.asarray(raw)
    return np.median(np.abs(raw - np.median(raw))) == 0


def window_scores(m, raw):
    """The reference pipeline on the window path: float32 scores of one read."""
    return postprocess.infer_read(raw, m.infer)[2].astype(np.float32)


def called(scores, threshold=0.5, min_run=15, extension_left=11, extension_right=16):
    """infer.py's post-processing of one read's scores (float32 widened to float64 against the threshold)."""
    labels = postprocess.correct_short(postprocess.class_from_threshold(scores, threshold), min_run)
    return postprocess.hp_in_pred(labels, extension_left, extension_right)


def assert_read_equal(m, raw, scores, intervals, length=None, want=None):
    """Part A's comparison of one read: read-path scores equal the window path's bit for bit, the intervals equal
    the post-processing of those scores; a read with MAD = 0 has NaN scores and no interval."""
    assert scores.dtype == np.float32 and scores.shape == (len(raw),)
    if length is not None:
        assert length == len(raw)
    if mad_is_zero(raw):
        assert np.isnan(scores).all() and list(intervals) == [], len(raw)
        return
    if want is None:
        want = window_scores(m, raw)
    assert np.isfinite(scores).all(), len(raw)
    assert np.array_equal(scores, want), (
        "read of %d samples: %d positions differ from the window path, max |d| %.3e"
        % (len(raw), int(np.count_nonzero(scores != want)), float(np.abs(scores - want).max())))
    assert list(intervals) == called(want), len(raw)


def ragged_reads(seed, n_short=0):
    """Window edges (1, 2, 34..36, 69..71, 4479..4481, 8960), odd lengths so that later reads start at unaligned
    int16 addresses, a read spanning more than 8192 distinct values (K1's wide path), a spike read whose full-scale
    samples normalise to +-3.2e4 (conv activations far beyond fp16's range), a constant read (MAD = 0), 20k-90k
    synthetic reads and `n_short` short synthetic reads."""
    rng = np.random.default_rng(seed)
    edges = [1, 2, 34, 35, 36, 69, 70, 71, 4479, 4480, 4481, 8960, 3, 1001, 12345]
    reads = synth.synth_reads(edges, base_seed=seed)
    wide = np.rint(rng.normal(0.0, 4000.0, 20011)).astype(np.int16)
    assert np.unique(wide).size > 8192
    spike = (500 + rng.integers(-1, 2, 9001)).astype(np.int16)           # MAD 1
    spike[::97], spike[50::97] = 32767, -32768                           # normalised +-3.2e4
    const = np.full(5003, 487, np.int16)
    longs = synth.synth_reads(rng.integers(20_000, 90_001, 3), base_seed=seed + 100)
    shorts = synth.synth_reads(rng.integers(100, 4001, n_short), base_seed=seed + 200)
    return reads[:8] + [wide] + reads[8:11] + [spike] + longs[:1] + [const] + reads[11:] + longs[1:] + shorts


def _check_label_path(m, reads, want_of, **call):
    """Intervals of the label-bit path (infer_reads without scores, one infer_concatenated call) equal want_of(r)."""
    hps, lengths = infer.infer_reads(reads, m, **call)
    raw, offsets = synth.concat_reads(reads)
    iv, ioff = infer.infer_concatenated(raw, offsets, m, **call)
    for r, read in enumerate(reads):
        want = want_of(r)
        assert lengths[r] == len(read)
        assert hps[r] == want, (r, len(read), call)
        assert iv[ioff[r]:ioff[r + 1]].tolist() == want, (r, len(read), call)


# ---------------------------------------------------------------- A. read path == window path
@pytest.mark.parametrize("case", list(VARIANTS))
def test_read_path_equals_window_path(case, shipped_weights):
    m, _ = _model(case, shipped_weights)
    # fewer than 296 reads: K1's chunked kernel; on `shipped` one group of at least 296 reads: one CTA per read
    reads = ragged_reads(700, n_short=K1_CTA_PER_READ + 4 if case == "shipped" else 0)
    total = sum(len(r) for r in reads)
    assert total < infer._FIRST_GROUP_SAMPLES and (len(reads) >= K1_CTA_PER_READ) == (case == "shipped")
    assert sum(n_windows(len(r)) for r in reads) > TILE * 16
    hps, lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    want = [None if mad_is_zero(r) else window_scores(m, r) for r in reads]
    assert sum(w is None for w in want) == 2                       # the one-sample read and the constant one
    for r, raw in enumerate(reads):
        assert_read_equal(m, raw, scores[r], hps[r], lengths[r], want[r])
    for call in ({}, NON_DEFAULT_CALL):
        _check_label_path(m, reads, lambda r: [] if want[r] is None else called(want[r], **call), **call)


# ---------------------------------------------------------------- B. engine passes
def _pass_windows(case, n):
    """n windows of the window-path input: synthetic-read windows for the shipped weights, N(0, 1.5) samples for
    random ones (the inputs the variant's bound was measured on)."""
    shipped = VARIANTS[case][2] is None or VARIANTS[case][2] is _wmax_shipped
    key = ("windows", shipped, n)
    if key not in _CACHE:
        _CACHE.clear()
        _CACHE[key] = pe.synthetic_windows(n) if shipped else \
            np.random.default_rng(600).normal(0, 1.5, size=(n, WINDOW, 1)).astype(np.float32)
    return _CACHE[key]


def straddling_batch(pass_windows, seed):
    """Reads whose concatenation crosses window `pass_windows`: fillers, one read that ends 1500 windows before it,
    the straddler (3001 windows, from 1500 before to 1501 after), and two reads after it.  Returns (reads, index of
    the straddler, its first window)."""
    rng = np.random.default_rng(seed)
    lengths, win = [], 0
    while True:
        n = int(rng.integers(20_000, 90_001)) | 1
        if win + n_windows(n) > pass_windows - 5000:
            break
        lengths.append(n)
        win += n_windows(n)
    g0 = pass_windows - 1500
    lengths.append((g0 - win - 1) * WINDOW + 17)                  # ends at window g0
    lengths += [3000 * WINDOW + 11, 40_001, 35 * 999]
    reads = synth.synth_reads(lengths, base_seed=seed)
    s = len(lengths) - 3
    assert sum(n_windows(len(r)) for r in reads[:s]) == g0 and g0 + n_windows(len(reads[s])) > pass_windows
    return reads, s, g0


@pytest.mark.parametrize("case", TC_VARIANTS)
def test_pass_edge_window_path(case, shipped_weights):
    """The window path on 2368 x 128 + 200 windows against float64: the two tiles each side of the first pass
    boundary and the last, partial tile, at the variant's budget.  (The CUDA-core engine's pass edge:
    test_gpu_precision_budgets.py::test_simt_chunk_edge_bit_exact.)"""
    m, w = _model(case, shipped_weights)
    n = TC_PASS_TILES * TILE + 200
    x = _pass_windows(case, n)
    p = m.infer(x)
    assert np.isfinite(p).all()
    sel = np.arange((TC_PASS_TILES - 2) * TILE, n)
    pos = (sel[:, None] * WINDOW + np.arange(WINDOW)).reshape(-1)
    tile = pe.tile_rms(p[pos], tf_graph.forward_np(w, x[sel], np.float64))
    bound = VARIANTS[case][5]
    print("%s: worst-tile RMS of p - p64 on tiles %d..%d: %s" % (case, TC_PASS_TILES - 2, TC_PASS_TILES + 1,
                                                                np.array2string(tile, precision=2)))
    assert tile.size == 4 and tile.max() <= bound, (
        "worst-tile RMS of p - p64 at the pass edge: %s (tiles %d.., bound %.1e)"
        % (np.array2string(tile, precision=3), TC_PASS_TILES - 2, bound))


@pytest.mark.parametrize("case", list(VARIANTS))
def test_pass_edge_read_path(case, shipped_weights):
    """One infer_concatenated call over more than one engine pass; the read that straddles the first boundary runs
    at another tile phase than it has alone, and it and its neighbours equal the window path bit for bit."""
    m, _ = _model(case, shipped_weights)
    pass_windows = (TC_PASS_TILES if case != "simt" else SIMT_PASS_TILES) * TILE
    reads, s, g0 = straddling_batch(pass_windows, 710)
    assert g0 % TILE != 0
    raw, offsets = synth.concat_reads(reads)
    if case != "simt":
        assert raw.size > TC_PASS_TILES * TILE * WINDOW
    iv, ioff, scores = infer.infer_concatenated(raw, offsets, m, return_scores=True)
    for r in (s - 1, s, s + 1):
        assert_read_equal(m, reads[r], scores[offsets[r]:offsets[r + 1]], iv[ioff[r]:ioff[r + 1]].tolist())


def test_read_longer_than_a_group(shipped_weights):
    """One read of 11 M samples, longer than infer_reads' groups and than one engine pass."""
    m, _ = _model("shipped", shipped_weights)
    raw = synth.synth_read(11_000_001, 720)
    assert raw.size > infer._GROUP_SAMPLES and n_windows(raw.size) > TC_PASS_TILES * TILE
    hps, lengths, scores = infer.infer_reads([raw], m, return_scores=True)
    assert_read_equal(m, raw, scores[0], hps[0], lengths[0])


# ---------------------------------------------------------------- C. label-bit ties
@pytest.mark.parametrize("case", ["shipped", "resnet1", "simt"])
def test_label_bit_ties(case, shipped_weights):
    """Threshold at an occurring score s (a tie: positive), at s + ulp(s) / 4 in double (negative, though it rounds
    to s in float32) and at 0.9 (float32(0.9) < 0.9): the label bits compare the float32 score widened to double,
    as class_from_threshold does.  min_run 1 and no extension, so one flipped position shows in the intervals."""
    m, _ = _model(case, shipped_weights)
    reads = synth.synth_reads([4481, 20011, 70001], base_seed=730)
    want = [window_scores(m, r) for r in reads]
    every = np.sort(np.concatenate(want))
    s = every[every.size // 2]                                    # the median score: it occurs
    t_tie = float(s)
    t_above = float(s) + float(np.spacing(s)) / 4
    assert np.float32(t_above) == s and t_above > t_tie
    labels = {}
    for t in (t_tie, t_above, 0.9):
        call = dict(threshold=t, min_run=1, extension_left=0, extension_right=0)
        labels[t] = [called(x, **call) for x in want]
        _check_label_path(m, reads, lambda r: labels[t][r], **call)
    assert labels[t_tie] != labels[t_above], "no occurring score separates the two thresholds"


# ---------------------------------------------------------------- D. config 3 against float64
CONFIG3_READS = 256
CONFIG3_CHECKED = 32
CONFIG3_SEED = 3


def test_config3_against_float64(shipped_weights):
    """BASELINE config 3: the shipped ResNetRNN on reads of U{50k..200k} samples, built as bench.make_batch builds
    them, through infer_reads (several groups, two in flight).  Every read's intervals follow from its scores; on a
    seeded subset the scores are held to float64 (max |dp| < 1e-3, label flips only inside the band, worst RMS over
    consecutive 4480-position blocks within the shipped f16e5 budget) and equal the window path bit for bit."""
    m, w = _model("shipped", shipped_weights)
    lengths = synth.ragged_lengths(CONFIG3_READS, 50_000, 200_000, seed=CONFIG3_SEED)
    reads = synth.synth_reads(lengths, base_seed=CONFIG3_SEED * 1_000_003)
    assert sum(lengths) > 2 * infer._GROUP_SAMPLES
    hps, got_lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    assert got_lengths == lengths.tolist()
    for h, s in zip(hps, scores):
        assert h == called(s)
    worst_rms, worst_dp, t0 = 0.0, 0.0, time.monotonic()
    for r in np.sort(np.random.default_rng(CONFIG3_SEED).choice(CONFIG3_READS, CONFIG3_CHECKED, replace=False)):
        raw, s = reads[r], scores[r]
        p64 = postprocess.infer_read(raw, lambda x: tf_graph.forward_np(w, x, np.float64))[2]
        d = np.abs(s.astype(np.float64) - p64)
        flips = (s >= 0.5) != (p64 >= 0.5)
        assert not (flips & ~allowed_label_flips(p64)).any(), (r, int(np.count_nonzero(flips)))
        worst_dp = max(worst_dp, float(d.max()))
        worst_rms = max(worst_rms, float(pe.tile_rms(s, p64).max()))
        assert_read_equal(m, raw, s, hps[r])
    print("config 3, %d of %d reads: max |dp| %.3e, worst 4480-position RMS %.3e, float64 oracle %.1f s"
          % (CONFIG3_CHECKED, CONFIG3_READS, worst_dp, worst_rms, time.monotonic() - t0))
    assert worst_dp < 1e-3 and worst_rms <= SHIPPED_BOUND, (worst_dp, worst_rms)
