"""GPU: network forward and the end-to-end per-read entry points against the oracle.

Contract (BASELINE.json north_star): probabilities within 1e-3 absolute of the
reference's fp32 CPU path; interval calls identical except where the reference
probability lies within 1e-3 of the threshold."""
import numpy as np
import pytest

from helpers import FakeFast5, allowed_label_flips, fake_h5py_module, golden, hpm_from_golden, random_bn_weights
from catfish_b200 import infer, neural_network, synth, weights
from oracle import postprocess, tf_graph

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-3          # north_star tolerance
ENGINES = ["simt", "auto"]


def _model(kind, engine, w=None, **hpm):
    full = dict(weights.SHIPPED_HPARAMS)
    full.update(hpm)
    m = neural_network.build_model(kind, engine=engine, **full)
    m.set_weights(w if w is not None else weights.load_shipped())
    return m


def _check_intervals(got_hps, scores_gpu, p_ref, threshold=0.5):
    """Intervals must equal the oracle's; where they differ, every differing label must sit in the
    allowed band, and the GPU intervals must be the exact post-processing of the GPU labels."""
    ref_labels = postprocess.class_from_threshold(p_ref, threshold)
    want = postprocess.hp_in_pred(postprocess.correct_short(ref_labels))
    if got_hps == want:
        return
    gpu_labels = postprocess.class_from_threshold(scores_gpu.astype(np.float64), threshold)
    diff = gpu_labels != ref_labels
    assert diff.any() and np.all(allowed_label_flips(p_ref, threshold)[diff]), "interval mismatch outside the band"
    assert got_hps == postprocess.hp_in_pred(postprocess.correct_short(gpu_labels))


@pytest.mark.parametrize("engine", ENGINES)
def test_infer_windows_shipped_vs_oracle(engine, shipped_weights):
    rng = np.random.default_rng(0)
    m = _model("ResNetRNN", engine)
    graph = tf_graph.TorchGraph(shipped_weights)
    for n_windows in (1, 127, 128, 129, 300):
        x = rng.normal(0, 1.5, size=(n_windows, 35, 1)).astype(np.float32)
        got = m.infer(x)
        assert got.dtype == np.float64 and got.shape == (n_windows * 35,)
        assert np.abs(got - graph.infer(x)).max() < PROB_TOL
    with pytest.raises(ValueError):
        m.infer(np.zeros((3, 34, 1)))


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["forward_rnn_le64_ns3_seed11.npz", "forward_resnet_ls32_ns2_seed12.npz",
                                  "forward_rnn_le16_ns2_seed13.npz"])
def test_variants_random_init_vs_golden(engine, name):
    g = golden(name)
    hpm = hpm_from_golden(g)
    kind = str(g["kind"])
    w = weights.random_init(kind, seed=int(g["seed"]), **hpm)
    m = _model(kind, engine, w, **hpm)
    got = m.infer(g["x"])
    assert np.abs(got - g["p64"]).max() < PROB_TOL


@pytest.mark.parametrize("engine", ENGINES)
def test_reads_golden_shipped(engine):
    g = golden("forward_resnetrnn_shipped.npz")
    m = _model("ResNetRNN", engine)
    reads = [g["read%d" % i] for i in range(int(g["n_reads"]))]
    hps, lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    for i, r in enumerate(reads):
        assert lengths[i] == len(r)
        assert scores[i].shape == (len(r),)
        assert np.abs(scores[i] - g["read%d_p32" % i]).max() < PROB_TOL
        _check_intervals(hps[i], scores[i], g["read%d_p32" % i].astype(np.float64))
        for a, b in hps[i]:
            assert isinstance(a, int) and isinstance(b, int)
    # single-read entry point returns the same as the batch
    one_hps, one_len = infer.infer_class_from_raw(reads[1], m)
    assert one_hps == hps[1] and one_len == lengths[1]


@pytest.mark.parametrize("engine", ENGINES)
def test_reads_ragged_vs_oracle(engine, shipped_weights):
    """Config-1 style: synthetic reads of ragged lengths incl. the padding edge cases."""
    lengths = [35, 36, 69, 70, 71, 4480, 4481, 10000, 10000, 12345, 1, 34]
    reads = synth.synth_reads(lengths, base_seed=300)
    m = _model("ResNetRNN", engine)
    graph = tf_graph.TorchGraph(shipped_weights)
    hps, lens, scores = infer.infer_reads(reads, m, return_scores=True)
    worst = 0.0
    for i, r in enumerate(reads):
        want_hps, want_len, want_scores = postprocess.infer_read(r, graph.infer)
        assert lens[i] == want_len
        worst = max(worst, float(np.abs(scores[i] - want_scores).max()))
        _check_intervals(hps[i], scores[i], want_scores)
    assert worst < PROB_TOL, worst


def test_degenerate_and_error_cases():
    m = _model("ResNetRNN", "auto")
    with pytest.raises(IndexError):
        infer.infer_reads([np.zeros(0, np.int16)], m)
    const = np.full(200, 512, np.int16)                   # MAD = 0: the reference divides by zero -> NaN
    hps, lens, scores = infer.infer_reads([const, synth.synth_read(500, 1)], m, return_scores=True)
    assert hps[0] == [] and lens == [200, 500] and np.all(np.isnan(scores[0]))
    assert np.all(np.isfinite(scores[1]))
    with pytest.raises(ValueError):
        infer.infer_class_from_signal("/nonexistent/file.fast5", m)
    assert infer.infer_reads([], m) == ([], [])


def test_engine_cross_check_large():
    """tcgen05 engine vs the fp32 SIMT engine on a batch the CPU oracle would take minutes for."""
    fast = _model("ResNetRNN", "auto")
    if fast.resolved_engine == "simt":
        pytest.skip("tcgen05 engine not available for this build")
    slow = _model("ResNetRNN", "simt")
    reads = synth.synth_reads(synth.ragged_lengths(40, 20000, 60000, seed=5), base_seed=900)
    h1, l1, s1 = infer.infer_reads(reads, fast, return_scores=True)
    h2, l2, s2 = infer.infer_reads(reads, slow, return_scores=True)
    assert l1 == l2
    worst = max(float(np.abs(a - b).max()) for a, b in zip(s1, s2))
    assert worst < PROB_TOL, worst
    for a, b, sa, sb in zip(h1, h2, s1, s2):
        _check_intervals(a, sa, sb.astype(np.float64))


@pytest.mark.parametrize("kind,n_res", [("ResNetRNN", 1), ("ResNetRNN", 3), ("ResNet", 1)],
                         ids=["resnetrnn-1-block", "resnetrnn-3-blocks", "resnet-1-block"])
def test_tcgen05_kernel_variants(kind, n_res):
    """Networks off the default path, which run split-bf16 operands in every layer, against the fp32 SIMT engine:
    one residual block (tc_conv2_kernel, then the 32- and 128-wide GRU layers or tc_head_conv_kernel) and three
    (tc_conv4_kernel for blocks 0 and 1, tc_conv_block_kernel for block 2, then the GRU layers).  The longest input
    spans more tiles than the GPU has SMs, so a CTA of every kernel runs several tiles."""
    w = weights.random_init(kind, seed=30 + n_res, n_layers_res=n_res)
    m = _model(kind, "auto", w, n_layers_res=n_res)
    assert m.resolved_engine == "tcgen05" and m.operand_format == "bf16x3"
    ref = _model(kind, "simt", w, n_layers_res=n_res)
    g = golden("forward_resnetrnn_shipped.npz")
    reads = [g["read%d" % i] for i in range(int(g["n_reads"]))] + synth.synth_reads([30000, 4481, 700000], base_seed=77)
    if kind == "ResNet":
        x = np.random.default_rng(31).normal(0, 1.5, size=(20000, 35, 1)).astype(np.float32)
        assert np.abs(m.infer(x) - ref.infer(x)).max() < PROB_TOL
        # tc_head_conv_kernel's label bits: the intervals without scores are those with scores
        assert infer.infer_reads(reads, m)[0] == infer.infer_reads(reads, m, return_scores=True)[0]
    hps, lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    hps2, lengths2, scores2 = infer.infer_reads(reads, ref, return_scores=True)
    assert lengths == lengths2
    for a, b_, sa, sb in zip(hps, hps2, scores, scores2):
        assert np.abs(sa - sb).max() < PROB_TOL
        _check_intervals(a, sa, sb.astype(np.float64))


def test_properties_at_scale():
    """Size-independent properties on a batch too large for the CPU oracle: batch invariance (a read's
    result does not depend on its neighbours in the ragged batch), interval/probability consistency,
    and determinism."""
    m = _model("ResNetRNN", "auto")
    reads = synth.synth_reads(synth.ragged_lengths(64, 50_000, 200_000, seed=11), base_seed=4000)
    hps, lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    hps_again, _, scores_again = infer.infer_reads(reads, m, return_scores=True)
    assert hps == hps_again
    for a, b_ in zip(scores, scores_again):
        np.testing.assert_array_equal(a, b_)                    # deterministic, bit for bit
    # a permuted / partial batch gives every read the same answer (tiles are shared between reads)
    order = [5, 63, 0, 17]
    hps_p, len_p, scores_p = infer.infer_reads([reads[i] for i in order], m, return_scores=True)
    for k, i in enumerate(order):
        assert hps_p[k] == hps[i] and len_p[k] == lengths[i]
        np.testing.assert_array_equal(scores_p[k], scores[i])
    # intervals are exactly the post-processing of the returned probabilities
    for h, s in zip(hps, scores):
        labels = postprocess.correct_short(postprocess.class_from_threshold(s.astype(np.float64)))
        assert h == postprocess.hp_in_pred(labels)
        assert np.all((s >= 0) & (s <= 1))


def test_ultra_long_read_vs_oracle(shipped_weights):
    """BASELINE configs[4]: a 1M-sample read (28 572 windows) end to end against the CPU oracle."""
    m = _model("ResNetRNN", "auto")
    raw = synth.synth_read(1_000_000, 4242)
    hps, lengths, scores = infer.infer_reads([raw], m, return_scores=True)
    graph = tf_graph.TorchGraph(shipped_weights)
    want_hps, want_len, want_scores = postprocess.infer_read(raw, graph.infer)
    assert lengths[0] == want_len == 1_000_000
    assert np.abs(scores[0] - want_scores).max() < PROB_TOL
    _check_intervals(hps[0], scores[0], want_scores)


def test_random_init_resnetrnn_outliers_and_parameters():
    """Different weights (seeded Glorot draw), signal with spikes spanning the int16 range, and the
    non-default post-processing parameters through the batched entry point."""
    w = weights.random_init("ResNetRNN", seed=5)
    m = _model("ResNetRNN", "auto", w)
    graph = tf_graph.TorchGraph(w)
    rng = np.random.default_rng(12)
    reads = synth.synth_reads([5000, 7777, 3500], base_seed=880)
    spiky = reads[1].copy()
    spiky[rng.integers(0, len(spiky), size=40)] = rng.choice([-32768, 32767, 0, 8191], size=40)
    reads[1] = spiky
    hps, lens, scores = infer.infer_reads(reads, m, return_scores=True)
    for r, h, s in zip(reads, hps, scores):
        want_h, _, want_s = postprocess.infer_read(r, graph.infer)
        assert np.abs(s - want_s).max() < PROB_TOL
        _check_intervals(h, s, want_s)
    # non-default threshold / min_run / extensions
    m2 = _model("ResNetRNN", "auto")
    reads2 = synth.synth_reads([9000, 4000], base_seed=41)
    for thr, min_run, el, er in ((0.9, 15, 11, 16), (0.3, 5, 0, 0), (0.5, 40, 3, 7)):
        hps2, _, sc2 = infer.infer_reads(reads2, m2, threshold=thr, min_run=min_run, extension_left=el,
                                         extension_right=er, return_scores=True)
        for h, s in zip(hps2, sc2):
            labels = postprocess.correct_short(postprocess.class_from_threshold(s.astype(np.float64), thr), min_run)
            assert h == postprocess.hp_in_pred(labels, el, er)


def test_rnn_stress_variant_h256_five_layers_simt():
    """The reference's commented "RNN" search setting (train_validate.py:330): H = 256, 5 layers.  Not a
    tcgen05 shape: runs on the fp32 SIMT engine, still through the same C ABI."""
    hpm = dict(layer_size=256, n_layers=5)
    w = weights.random_init("RNN", seed=31, **hpm)
    m = _model("RNN", "auto", w, **hpm)
    assert m.resolved_engine == "simt"
    rng = np.random.default_rng(5)
    x = rng.normal(0, 1.5, size=(70, 35, 1)).astype(np.float32)
    got = m.infer(x)
    want = tf_graph.forward_np(w, x, np.float64)
    assert np.abs(got - want).max() < PROB_TOL


def test_outlier_samples_stay_finite_and_in_contract():
    """Raw spikes thousands of MADs away from the median (the fp16 operand format must not overflow):
    the tcgen05 engine still agrees with the fp32 engine and the CPU oracle."""
    rng = np.random.default_rng(9)
    reads = []
    for k, mad in enumerate((1, 3, 20)):
        raw = (500 + np.rint(rng.normal(0, mad * 1.4826, 6000))).astype(np.int16)
        idx = rng.choice(raw.size, 12, replace=False)
        raw[idx[:6]] = 32767
        raw[idx[6:]] = -32768
        reads.append(raw)
    m = _model("ResNetRNN", "auto")
    ref = _model("ResNetRNN", "simt")
    _, _, s1 = infer.infer_reads(reads, m, return_scores=True)
    _, _, s2 = infer.infer_reads(reads, ref, return_scores=True)
    graph = tf_graph.TorchGraph(weights.load_shipped())
    for raw, a, b in zip(reads, s1, s2):
        assert np.isfinite(a).all()
        assert np.abs(a - b).max() < PROB_TOL
        _, _, want = postprocess.infer_read(raw, graph.infer)
        assert np.abs(a - want).max() < PROB_TOL


def test_outlier_windows_stay_in_contract():
    """Same through the window-level entry point (cf_infer_windows), including a non-finite window."""
    rng = np.random.default_rng(10)
    x = rng.normal(0, 1.5, size=(200, 35, 1)).astype(np.float32)
    x[17, 5, 0] = 4.0e4
    x[90, 30, 0] = -2.5e4
    m, ref = _model("ResNetRNN", "auto"), _model("ResNetRNN", "simt")
    a, b = m.infer(x), ref.infer(x)
    assert np.isfinite(a).all() and np.abs(a - b).max() < PROB_TOL
    assert m.operand_format in ("f16e5", "bf16x3") and ref.operand_format == "f32"
    x[3, 0, 0] = np.inf
    a, b = m.infer(x).reshape(200, 35), ref.infer(x).reshape(200, 35)
    keep = np.arange(200) != 3                       # windows are independent: only window 3 may be non-finite
    assert np.isfinite(a[keep]).all() and np.abs(a[keep] - b[keep]).max() < PROB_TOL


def test_large_batch_in_groups_equals_host_calls():
    """A batch of several engine passes through cf_infer_reads_host: CSR offsets, intervals and probabilities
    equal those of smaller calls over sub-ranges of the same reads (batch invariance at the host boundary), and
    infer_reads, which runs the batch as several groups of reads, gives the same intervals and scores."""
    m = _model("ResNetRNN", "auto")
    lengths = synth.ragged_lengths(300, 60_000, 120_000, seed=3)           # ~27M samples = 5 passes
    reads = synth.synth_reads(lengths, base_seed=9000)
    raw, off = synth.concat_reads(reads)
    iv, ioff, scores = infer.infer_concatenated(raw, off, m, return_scores=True)
    assert ioff[0] == 0 and ioff[-1] == len(iv) and np.all(np.diff(ioff) >= 0)
    for lo, hi in ((0, 40), (130, 170), (260, 300)):
        sub_raw = raw[off[lo]:off[hi]]
        sub_off = off[lo:hi + 1] - off[lo]
        iv2, ioff2, scores2 = infer.infer_concatenated(sub_raw, sub_off, m, return_scores=True)
        assert np.array_equal(ioff2, ioff[lo:hi + 1] - ioff[lo])
        assert np.array_equal(iv2, iv[ioff[lo]:ioff[hi]])
        assert np.array_equal(scores2, scores[off[lo]:off[hi]])
    # the Python entry point runs a batch of this size as several groups of reads (device-side calls overlapped
    # with the host's staging): identical per-read results and scores, list-like and as arrays
    assert len(infer._cut_groups(off, infer._FIRST_GROUP_SAMPLES, infer._GROUP_SAMPLES)) > 1
    hps, lens, scores_py = infer.infer_reads(reads, m, return_scores=True)
    assert lens == [len(r) for r in reads]
    for r in range(len(reads)):
        assert np.array_equal(hps[r].array, iv[ioff[r]:ioff[r + 1]])
        assert np.array_equal(scores_py[r], scores[off[r]:off[r + 1]])
    assert hps[7] == iv[ioff[7]:ioff[8]].tolist() and isinstance(hps[7][0][0], int)
    hps_again, _ = infer.infer_reads(reads, m)                     # the model's pooled buffers reused
    assert all(a == b for a, b in zip(hps, hps_again))


def test_fast5_entry_point_with_stub_h5py(tmp_path, monkeypatch, shipped_weights):
    """infer_class_from_signal / process_signal (infer.py:12-51, 77-93) through a stand-in for h5py: the leading
    first_sample_template samples are dropped, the first Raw/Reads member is read, and the result equals the
    array-level twin and the oracle's driver on the trimmed signal."""
    import sys
    m = _model("ResNetRNN", "auto")
    path = str(tmp_path / "read.fast5")
    open(path, "wb").close()                                   # the entry point checks os.path.exists first
    signal, first = synth.synth_read(3000, 5), 211
    fake = FakeFast5(signal, first, read_names=("Read_42", "Read_43"))
    monkeypatch.setitem(sys.modules, "h5py", fake_h5py_module({path: fake}))
    hps, length = infer.infer_class_from_signal(path, m)
    assert length == len(signal) - first and isinstance(hps, list) and all(type(v) is int for iv in hps for v in iv)
    assert (hps, length) == infer.infer_class_from_raw(signal[first:], m)
    want_hps, want_len, want_scores = postprocess.infer_read(signal[first:], tf_graph.TorchGraph(shipped_weights).infer)
    _, _, scores = infer.infer_reads([signal[first:]], m, return_scores=True)
    assert length == want_len and np.abs(scores[0] - want_scores).max() < PROB_TOL
    _check_intervals(hps, scores[0], want_scores)
    norm = infer.process_signal(fake)
    np.testing.assert_array_equal(norm, postprocess.normalize_raw_signal(signal[first:]))
    with pytest.raises(ValueError):
        infer.infer_class_from_signal(str(tmp_path / "missing.fast5"), m)


def test_random_bn_statistics_vs_reference_graph_golden():
    """Seeded weights with non-trivial batch-norm statistics: the CUDA engines against the reference graph's
    own output (tests/golden/forward_resnetrnn_randbn_seed14.npz, made by the meta-graph executor)."""
    g = golden("forward_resnetrnn_randbn_seed14.npz")
    w = random_bn_weights(int(g["seed"]))
    for engine in ENGINES:
        m = _model("ResNetRNN", engine, w=w)
        got = m.infer(g["x"])
        assert np.abs(got - g["p64"]).max() < PROB_TOL, engine
