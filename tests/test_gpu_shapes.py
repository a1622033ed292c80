"""GPU: the tensor-core engine on hyper-parameters other than the shipped ones.

Narrower networks (conv channels C < 32, GRU units H < 64) run the C = 32 / H = 64 kernels on a copy of the
weights padded with zeros; conv stacks of any depth run on tensor cores (blocks after the second in
tc_conv_block_kernel).  Each shape is checked against the reference graph in float64, the padding against
an explicitly padded network bit for bit, and deep stacks against the fp32 CUDA-core engine at scale."""
import numpy as np
import pytest

from helpers import allowed_label_flips
from catfish_b200 import infer, neural_network, synth, weights
from oracle import postprocess, tf_graph

pytestmark = pytest.mark.gpu

PROB_TOL = 1e-3
PAD_C, PAD_H = 32, 64


def _bn_weights(kind, seed, **hpm):
    """Seeded weights of any shape with non-trivial BN gamma / beta / moving statistics."""
    w = weights.random_init(kind, seed=seed, **hpm)
    rng = np.random.default_rng(seed + 1000)
    for k in sorted(w):
        if k.endswith("moving_mean"):
            w[k] = rng.normal(0, 0.3, size=w[k].shape).astype(np.float32)
        elif k.endswith("moving_variance"):
            w[k] = rng.uniform(0.3, 2.0, size=w[k].shape).astype(np.float32)
        elif k.endswith("beta"):
            w[k] = rng.normal(0, 0.2, size=w[k].shape).astype(np.float32)
        elif k.endswith("gamma"):
            w[k] = rng.uniform(0.5, 1.5, size=w[k].shape).astype(np.float32)
    return w


def _hpm(kind, c=32, h=64, n_res=2, n_layers=3):
    hpm = {}
    if kind != "RNN":
        hpm.update(layer_size_res=c, n_layers_res=n_res)
    if kind != "ResNet":
        hpm.update(layer_size=h, n_layers=n_layers)
    return hpm


def _model(kind, engine, w, **hpm):
    full = dict(weights.SHIPPED_HPARAMS)
    full.update(hpm)
    m = neural_network.build_model(kind, engine=engine, **full)
    m.set_weights(w)
    return m


def _check_intervals(got_hps, scores_gpu, p_ref, threshold=0.5):
    """Intervals equal the reference's, or differ only through labels whose reference probability lies in the
    1e-3 band around the threshold, and are then the exact post-processing of the returned probabilities."""
    ref_labels = postprocess.class_from_threshold(p_ref, threshold)
    want = postprocess.hp_in_pred(postprocess.correct_short(ref_labels))
    if got_hps == want:
        return
    gpu_labels = postprocess.class_from_threshold(scores_gpu.astype(np.float64), threshold)
    diff = gpu_labels != ref_labels
    assert diff.any() and np.all(allowed_label_flips(p_ref, threshold)[diff]), "interval mismatch outside the band"
    assert got_hps == postprocess.hp_in_pred(postprocess.correct_short(gpu_labels))


def _pad_weights(w, kind, c, h, n_res, n_layers):
    """The same network at C = 32 / H = 64: channel c at c, unit j of each gate group at j of its 64-wide group,
    fw unit j of a [fw | bw] input at row j and bw unit j at row 64 + j.  Every added weight and bias is 0 (BN of an
    added channel: gamma 1, beta 0, mean 0, variance 1, so that it folds to zero)."""
    out = {}
    for b in range(n_res if kind != "RNN" else 0):
        for j in range(4):
            i = 4 * b + j
            name = weights.conv_name(i)
            k = w[name + "/kernel"]
            cin = 1 if (b == 0 and j < 2) else PAD_C
            kp = np.zeros((k.shape[0], cin, PAD_C), np.float32)
            kp[:, :k.shape[1], :c] = k
            out[name + "/kernel"] = kp
            v = np.zeros(PAD_C, np.float32)
            v[:c] = w[name + "/bias"]
            out[name + "/bias"] = v
            bn = weights.bn_name(i)
            for leaf, fill in (("gamma", 1.0), ("beta", 0.0), ("moving_mean", 0.0), ("moving_variance", 1.0)):
                v = np.full(PAD_C, fill, np.float32)
                v[:c] = w[bn + "/" + leaf]
                out[bn + "/" + leaf] = v
    if kind == "ResNet":
        head = np.zeros((PAD_C, 1), np.float32)
        head[:c] = w["final_fully_connected/kernel"]
        out["final_fully_connected/kernel"] = head
        out["final_fully_connected/bias"] = w["final_fully_connected/bias"].copy()
        return out
    unit2 = np.concatenate([np.arange(h), PAD_H + np.arange(h)])          # rows of a [fw | bw] input

    def cols(groups):
        return np.concatenate([g * PAD_H + np.arange(h) for g in range(groups)])
    for l in range(n_layers):
        fin = (c if kind == "ResNetRNN" else 1) if l == 0 else 2 * h
        fin_p = (PAD_C if kind == "ResNetRNN" else 1) if l == 0 else 2 * PAD_H
        x_rows = np.arange(fin) if l == 0 else unit2
        for d in ("fw", "bw"):
            p = weights.gru_prefix(l, d)
            for part, groups in (("gates", 2), ("candidate", 1)):
                k = w[p + "/%s/kernel" % part]
                kp = np.zeros((fin_p + PAD_H, groups * PAD_H), np.float32)
                kp[np.ix_(x_rows, cols(groups))] = k[:fin]
                kp[np.ix_(fin_p + np.arange(h), cols(groups))] = k[fin:]
                out[p + "/%s/kernel" % part] = kp
                bp = np.zeros(groups * PAD_H, np.float32)
                bp[cols(groups)] = w[p + "/%s/bias" % part]
                out[p + "/%s/bias" % part] = bp
    head = np.zeros((2 * PAD_H, 1), np.float32)
    head[unit2] = w["final_fully_connected/kernel"]
    out["final_fully_connected/kernel"] = head
    out["final_fully_connected/bias"] = w["final_fully_connected/bias"].copy()
    return out


NEW_SHAPES = [
    ("RNN", dict(h=8, n_layers=2)),
    ("RNN", dict(h=16, n_layers=3)),
    ("RNN", dict(h=32, n_layers=2)),
    ("RNN", dict(h=48, n_layers=3)),
    ("ResNetRNN", dict(c=16, h=32, n_res=2, n_layers=2)),
    ("ResNetRNN", dict(c=32, h=16, n_res=1, n_layers=2)),
    ("ResNetRNN", dict(c=8, h=64, n_res=3, n_layers=2)),
    ("ResNet", dict(c=16, n_res=1)),
    ("ResNet", dict(c=24, n_res=2)),
]


@pytest.mark.parametrize("kind,shape", NEW_SHAPES, ids=["%s-%s" % (k, "-".join("%s%d" % kv for kv in s.items()))
                                                        for k, s in NEW_SHAPES])
def test_new_shapes_vs_reference_graph(kind, shape):
    hpm = _hpm(kind, **shape)
    w = _bn_weights(kind, 40 + NEW_SHAPES.index((kind, shape)), **hpm)
    m = _model(kind, "auto", w, **hpm)
    assert m.resolved_engine == "tcgen05"
    rng = np.random.default_rng(41)
    for n_windows in (1, 129, 300):
        x = rng.normal(0, 1.5, size=(n_windows, 35, 1)).astype(np.float32)
        got = m.infer(x)
        want = tf_graph.forward_np(w, x, np.float64)
        assert np.abs(got - want).max() < PROB_TOL, n_windows


@pytest.mark.parametrize("kind,shape", [("RNN", dict(h=32, n_layers=3)), ("ResNetRNN", dict(c=16, h=32, n_res=2, n_layers=3))],
                         ids=["rnn-h32", "resnetrnn-c16-h32"])
def test_padding_is_exact(kind, shape):
    """The engine's own padding gives bit for bit what the network zero-padded by hand gives."""
    hpm = _hpm(kind, **shape)
    w = _bn_weights(kind, 70, **hpm)
    full = dict(c=shape.get("c", 32), h=shape["h"], n_res=shape.get("n_res", 0), n_layers=shape["n_layers"])
    wp = _pad_weights(w, kind, **full)
    hpm_p = _hpm(kind, c=PAD_C, h=PAD_H, n_res=full["n_res"], n_layers=full["n_layers"])
    narrow, padded = _model(kind, "auto", w, **hpm), _model(kind, "auto", wp, **hpm_p)
    assert narrow.resolved_engine == padded.resolved_engine == "tcgen05"
    assert narrow.operand_format == padded.operand_format
    # the hand-padded network is the same function (float64 reference graph)
    x = np.random.default_rng(71).normal(0, 1.5, size=(40, 35, 1)).astype(np.float32)
    assert np.abs(tf_graph.forward_np(w, x) - tf_graph.forward_np(wp, x)).max() < 1e-12
    reads = synth.synth_reads([1, 34, 35, 36, 4481, 23456, 41000], base_seed=72)
    h1, l1, s1 = infer.infer_reads(reads, narrow, return_scores=True)
    h2, l2, s2 = infer.infer_reads(reads, padded, return_scores=True)
    assert l1 == l2 == [len(r) for r in reads]
    for a, b in zip(h1, h2):
        assert a == b
    for a, b in zip(s1, s2):
        np.testing.assert_array_equal(a, b)


DEEP = [("ResNetRNN", 3), ("ResNetRNN", 4), ("ResNetRNN", 5), ("ResNetRNN", 11), ("ResNet", 3), ("ResNet", 4)]


@pytest.mark.parametrize("kind,n_res", DEEP, ids=["%s-%d-blocks" % d for d in DEEP])
def test_deep_conv_stacks(kind, n_res):
    """Conv stacks of three or more blocks: TK2 runs blocks 0-1, tc_conv_block_kernel each further block."""
    hpm = _hpm(kind, n_res=n_res)
    w = _bn_weights(kind, 80 + n_res, **hpm)
    m = _model(kind, "auto", w, **hpm)
    assert m.resolved_engine == "tcgen05" and m.operand_format == "bf16x3"
    x = np.random.default_rng(81).normal(0, 1.5, size=(300, 35, 1)).astype(np.float32)
    assert np.abs(m.infer(x) - tf_graph.forward_np(w, x, np.float64)).max() < PROB_TOL
    if kind == "ResNet":
        return
    # the longest read spans more tiles than the GPU has SMs: every CTA runs several tiles
    ref = _model(kind, "simt", w, **hpm)
    reads = synth.synth_reads([30000, 4481, 35, 36, 700000], base_seed=82)
    hps, lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    hps2, lengths2, scores2 = infer.infer_reads(reads, ref, return_scores=True)
    assert lengths == lengths2
    for a, b, sa, sb in zip(hps, hps2, scores, scores2):
        assert np.abs(sa - sb).max() < PROB_TOL
        _check_intervals(a, sa, sb.astype(np.float64))


def test_new_shape_deterministic_and_batch_invariant():
    kind, hpm = "ResNetRNN", _hpm("ResNetRNN", c=8, h=48, n_res=3, n_layers=2)
    m = _model(kind, "auto", _bn_weights(kind, 90, **hpm), **hpm)
    assert m.resolved_engine == "tcgen05"
    reads = synth.synth_reads(synth.ragged_lengths(24, 20_000, 90_000, seed=91), base_seed=92)
    hps, lengths, scores = infer.infer_reads(reads, m, return_scores=True)
    hps_again, _, scores_again = infer.infer_reads(reads, m, return_scores=True)
    assert hps == hps_again
    for a, b in zip(scores, scores_again):
        np.testing.assert_array_equal(a, b)
    order = [7, 23, 0, 11]
    hps_p, len_p, scores_p = infer.infer_reads([reads[i] for i in order], m, return_scores=True)
    for k, i in enumerate(order):
        assert hps_p[k] == hps[i] and len_p[k] == lengths[i]
        np.testing.assert_array_equal(scores_p[k], scores[i])


@pytest.mark.parametrize("kind,shape", [("RNN", dict(h=128, n_layers=2)), ("ResNetRNN", dict(c=64, h=64, n_res=2, n_layers=1)),
                                        ("ResNet", dict(c=64, n_res=2))], ids=["rnn-h128", "resnetrnn-c64", "resnet-c64"])
def test_wider_shapes_refused_by_tcgen05(kind, shape):
    hpm = _hpm(kind, **shape)
    w = weights.random_init(kind, seed=95, **hpm)
    with pytest.raises(ValueError, match="tcgen05"):
        _model(kind, "tcgen05", w, **hpm)
    assert _model(kind, "auto", w, **hpm).resolved_engine == "simt"
