"""Training without a GPU: the float64 oracle step against the pinned forward graph and finite differences, the
Philox dropout mask, the checkpoint format with optimizer slots, and the refusals that happen before any device work."""

import os

import numpy as np
import pytest

from catfish_b200 import rnn_class, weights
from oracle import tf_graph, train, validation

SHAPES = [
    ("ResNetRNN", dict(layer_size=64, n_layers=3, layer_size_res=32, n_layers_res=2)),
    ("RNN", dict(layer_size=16, n_layers=2)),
    ("ResNet", dict(layer_size_res=8, n_layers_res=2)),
]


def _batch(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 1.0, size=(n, 35, 1)).astype(np.float32)
    y = (rng.random(n * 35) < 0.3).astype(np.uint8)
    return x, y


@pytest.mark.parametrize("kind,hpm", [("shipped", None)] + SHAPES)
def test_oracle_forward_at_keep_one_is_the_inference_graph(kind, hpm, shipped_weights):
    w = shipped_weights if kind == "shipped" else weights.random_init(kind, seed=5, **hpm)
    x, y = _batch(6, 1)
    z = train.TrainGraph(w).logits(x).detach().numpy()
    ref = tf_graph.forward_np(w, x, np.float64, return_logits=True)
    assert np.max(np.abs(z - ref)) <= 1e-12
    loss = train.loss_of_logits(train.TrainGraph(w).logits(x), y).item()
    assert loss == pytest.approx(validation.test_network(ref, y, 0)[2], rel=1e-12)


@pytest.mark.parametrize("keep_prob", [1.0, 0.8])
def test_oracle_gradients_match_central_differences(keep_prob):
    hpm = dict(layer_size=4, n_layers=1, layer_size_res=4, n_layers_res=1)
    w = weights.random_init("ResNetRNN", seed=3, **hpm)
    rng = np.random.default_rng(4)
    for k in sorted(w):     # non-trivial BN affine and statistics, so gamma / beta gradients are exercised
        if k.endswith("gamma") or k.endswith("moving_variance"):
            w[k] = rng.uniform(0.5, 1.5, size=w[k].shape).astype(np.float32)
        elif k.endswith("beta") or k.endswith("moving_mean") or k.endswith("/bias"):
            w[k] = rng.normal(0, 0.3, size=w[k].shape).astype(np.float32)
    x, y = _batch(3, 2)
    masks = train.dropout_masks(w, 9, 1, 3, keep_prob)
    _, grads, _ = train.step_gradients(w, x, y, keep_prob, masks)
    w64 = {k: v.astype(np.float64) for k, v in w.items()}

    def loss(ws):
        return train.loss_of_logits(train.TrainGraph(ws).logits(x, keep_prob, masks), y).item()

    h = 1e-6
    for name, g in grads.items():
        flat = g.reshape(-1)
        for i in rng.choice(flat.size, size=min(flat.size, 4), replace=False):
            plus, minus = dict(w64), dict(w64)
            plus[name] = w64[name].copy().reshape(-1)
            minus[name] = w64[name].copy().reshape(-1)
            plus[name][i] += h
            minus[name][i] -= h
            plus[name] = plus[name].reshape(w[name].shape)
            minus[name] = minus[name].reshape(w[name].shape)
            fd = (loss(plus) - loss(minus)) / (2 * h)
            assert abs(fd - flat[i]) <= 1e-7 + 1e-5 * abs(fd), (name, i, fd, flat[i])


def test_philox_known_answers_and_kept_fraction():
    # Random123 kat_vectors, philox4x32 10 rounds
    kat = [([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
           ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
           ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
            [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])]
    for ctr, key, want in kat:
        assert [int(v) for v in train.philox4x32_10(ctr, key)] == want
    m = train.dropout_mask(seed=12345, step=7, layer=1, direction=0, n_windows=448, hidden=64, keep_prob=0.8)
    assert m.size >= 10 ** 6
    assert abs(m.mean() - 0.8) <= 0.002
    assert train.dropout_masks({}, 0, 0, 1, 1.0) is None


def test_rmsprop_first_step_from_fresh_slots():
    g = np.array([0.0, 1.0, -3.0, 1e-3])
    var, ms, mom = train.rmsprop(np.zeros(4), np.ones(4), np.zeros(4), g, 0.001)
    assert np.allclose(ms, 0.9 + 0.1 * g * g)
    assert np.allclose(var, -0.001 * g / np.sqrt(0.9 + 0.1 * g * g))


def test_checkpoint_round_trip_carries_the_slots(tmp_path, shipped_weights):
    slots = weights.fresh_slots(shipped_weights)
    rng = np.random.default_rng(0)
    slots = {k: (v + rng.random(v.shape)).astype(np.float32) for k, v in slots.items()}
    out = weights.save_checkpoint(str(tmp_path), 30017, shipped_weights, slots)
    assert os.path.basename(out) == "ckpnt-30017.npz"
    assert rnn_class._latest_checkpoint(str(tmp_path)) == "ckpnt-30017"
    tensors = weights.load_npz(out)
    assert len(shipped_weights) == 74 and len(slots) == 116 and len(tensors) == 190
    inf, got = weights.split_slots(tensors)
    back = weights.check_weights(inf, "ResNetRNN", **{k: weights.SHIPPED_HPARAMS[k] for k in
                                                      ("layer_size", "n_layers", "layer_size_res", "n_layers_res")})
    assert set(back) == set(shipped_weights)
    for k in shipped_weights:
        assert np.array_equal(back[k], shipped_weights[k])
    assert set(got) == set(slots)
    for k in slots:
        assert np.array_equal(got[k], slots[k])
    assert weights.checkpoint_step("ckpnt-30017") == 30017 and weights.checkpoint_step("model") is None


def _model(**over):
    hp = dict(weights.SHIPPED_HPARAMS)
    hp.update(over)
    return rnn_class.RNN(**hp)


@pytest.mark.parametrize("over", [dict(optimizer_choice="Adam"), dict(keep_prob=0.0), dict(keep_prob=1.5)])
def test_training_refusals_before_device_work(over):
    x, y = _batch(2, 0)
    with pytest.raises(ValueError):
        _model(**over).train_network(x, y)


def test_save_true_still_refused():
    with pytest.raises(NotImplementedError):
        rnn_class.RNN(save=True, **weights.SHIPPED_HPARAMS)
