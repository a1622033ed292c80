"""Training on the GPU (K12, cf_trainer): gradients against float64 autograd of oracle/train.py with and without
dropout, RMSProp updates against the float64 optimizer, bit-exact determinism and checkpoint resume, learning on
labelled synthetic reads, and the refusals."""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = {
    "shipped": ("ResNetRNN", dict(layer_size=64, n_layers=3, layer_size_res=32, n_layers_res=2)),
    "rnn64x3": ("RNN", dict(layer_size=64, n_layers=3)),
    "resnet": ("ResNet", dict(layer_size_res=32, n_layers_res=2)),
    "rnn256x2": ("RNN", dict(layer_size=256, n_layers=2)),
    "resnetrnn_c64_b3": ("ResNetRNN", dict(layer_size=32, n_layers=1, layer_size_res=64, n_layers_res=3)),
}
BOUND = 2e-4


def _model(kind, hpm, w, engine="simt", **over):
    from catfish_b200 import neural_network, weights
    hp = dict(weights.SHIPPED_HPARAMS)
    hp.update(layer_size=64, n_layers=1, layer_size_res=32, n_layers_res=1)
    hp.update(hpm)
    hp.update(over)
    m = neural_network.build_model(kind, engine=engine, **hp)
    m.set_weights(w)
    return m


def _weights(name, seed=11, shipped=None):
    from catfish_b200 import weights
    kind, hpm = SHAPES[name]
    if name == "shipped":
        return kind, hpm, shipped
    w = weights.random_init(kind, seed=seed, **hpm)
    if kind != "RNN":     # non-trivial BN statistics and affine, as in the shipped model
        rng = np.random.default_rng(seed)
        for k in sorted(w):
            if k.endswith("gamma") or k.endswith("moving_variance"):
                w[k] = rng.uniform(0.5, 1.5, size=w[k].shape).astype(np.float32)
            elif k.endswith("beta") or k.endswith("moving_mean"):
                w[k] = rng.normal(0, 0.2, size=w[k].shape).astype(np.float32)
    return kind, hpm, w


def _batch(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 1.0, size=(n, 35, 1)).astype(np.float32)
    y = (rng.random(n * 35) < 0.35).astype(np.uint8)
    return x, y


def _worst(got, want):
    """max over tensors of max|got - want| / max|want|."""
    worst = 0.0
    for k, g in want.items():
        scale = np.max(np.abs(g))
        err = np.max(np.abs(got[k].astype(np.float64) - g))
        worst = max(worst, err / scale if scale > 0 else err)
    return worst


@pytest.mark.parametrize("n", [1, 129, 300])
@pytest.mark.parametrize("name", list(SHAPES))
def test_gradients_match_float64_autograd(name, n, shipped_weights):
    from oracle import train
    kind, hpm, w = _weights(name, shipped=shipped_weights)
    x, y = _batch(n, 100 + n)
    m = _model(kind, hpm, w)
    grads, loss = m.compute_gradients(x, y, keep_prob=1.0)
    loss64, g64, _ = train.step_gradients(w, x, y)
    assert set(grads) == set(g64)
    for k in g64:
        scale = np.max(np.abs(g64[k]))
        err = np.max(np.abs(grads[k] - g64[k]))
        assert err <= BOUND * scale, (k, err, scale)
    print("worst ratio %s n=%d: %.3g" % (name, n, _worst(grads, g64)))
    assert loss == pytest.approx(loss64, rel=1e-6)
    _, test_loss = m.test_network(x, y)
    assert float(test_loss) == pytest.approx(loss64, rel=1e-6)


@pytest.mark.parametrize("name", ["shipped", "rnn256x2"])
def test_dropout_gradients_match_the_rebuilt_mask(name, shipped_weights):
    from oracle import train
    kind, hpm, w = _weights(name, shipped=shipped_weights)
    n, seed, step = 129, 0x1234_5678_9ABC, 17
    x, y = _batch(n, 5)
    m = _model(kind, hpm, w)
    m.dropout_seed = seed
    grads, loss = m.compute_gradients(x, y, keep_prob=0.8, step=step)
    masks = train.dropout_masks(w, seed, step, n, 0.8)
    loss64, g64, _ = train.step_gradients(w, x, y, 0.8, masks)
    for k in g64:
        assert np.max(np.abs(grads[k] - g64[k])) <= BOUND * np.max(np.abs(g64[k])), k
    print("worst ratio dropout %s: %.3g" % (name, _worst(grads, g64)))
    assert loss == pytest.approx(loss64, rel=1e-6)
    # another step draws another mask
    other, _ = m.compute_gradients(x, y, keep_prob=0.8, step=step + 1)
    assert any(not np.array_equal(other[k], grads[k]) for k in grads)


RMS_LR = 0.001      # the reference's learning_rate (ResNetRNN.txt)


@pytest.mark.parametrize("steps", [1, 5])
@pytest.mark.parametrize("name", ["shipped", "rnn64x3"])
def test_rmsprop_steps_match_the_float64_optimizer(name, steps, shipped_weights):
    from oracle import train
    kind, hpm, w = _weights(name, shipped=shipped_weights)
    batches = [_batch(200, 300 + i) for i in range(steps)]
    m = _model(kind, hpm, w, keep_prob=1.0, learning_rate=RMS_LR)
    for x, y in batches:
        m.train_network(x, y)
    assert m.global_step == steps
    w64, s64, _ = train.train_steps(w, batches, RMS_LR)
    got, slots = m.get_weights(), m.optimizer_state()
    for k, v in w64.items():
        if not train._is_trainable(k):
            assert np.array_equal(got[k], w[k]), k
            continue
        moved = np.max(np.abs(v - w[k].astype(np.float64)))
        # each step stores the variable in fp32 once: a gate bias near 1.0 that moves by 1e-5 is a few ulps of its
        # value, so the bound also allows one ulp of the tensor's largest value per step
        rounding = steps * float(np.spacing(np.float32(np.max(np.abs(v)))))
        assert np.max(np.abs(got[k] - v)) <= BOUND * moved + rounding, (k, np.max(np.abs(got[k] - v)), moved)
        ms, mom = k + "/RMSProp", k + "/RMSProp_1"
        assert np.max(np.abs(slots[ms] - s64[ms])) <= BOUND * np.max(np.abs(s64[ms] - 1.0)), ms
        assert np.max(np.abs(slots[mom] - s64[mom])) <= BOUND * np.max(np.abs(s64[mom])), mom


def test_steps_are_deterministic_and_resume_bit_for_bit(tmp_path, shipped_weights):
    from catfish_b200 import weights
    kind, hpm, w = _weights("shipped", shipped=shipped_weights)
    batches = [_batch(256, 500 + i) for i in range(20)]

    def run(model, bs):
        for x, y in bs:
            model.train_network(x, y)
        return model.get_weights(), model.optimizer_state()

    a = _model(kind, hpm, w)
    b = _model(kind, hpm, w)
    wa, sa = run(a, batches)
    wb, sb = run(b, batches)
    for k in wa:
        assert np.array_equal(wa[k], wb[k]), k
    for k in sa:
        assert np.array_equal(sa[k], sb[k]), k
    assert any(not np.array_equal(wa[k], w[k]) for k in w)

    k_steps = 3
    first = _model(kind, hpm, w)
    run(first, batches[:k_steps])
    path = first.save_network(str(tmp_path))
    assert path.endswith("ckpnt-%d.npz" % k_steps) and len(weights.load_npz(path)) == 190
    resumed = _model(kind, hpm, weights.random_init(kind, seed=1, **hpm))
    resumed.restore_network(str(tmp_path))
    assert resumed.global_step == k_steps
    wr, sr = run(resumed, batches[k_steps:])
    for k in wa:
        assert np.array_equal(wr[k], wa[k]), k
    for k in sa:
        assert np.array_equal(sr[k], sa[k]), k


# ---------------------------------------------------------------- learning
def _labelled_read(length, seed):
    """synth_read with label 1 inside events of length >= 12 (the event lengths are the read's first draw)."""
    from catfish_b200 import infer, synth
    raw = synth.synth_read(length, seed)
    ev_len = np.random.default_rng(seed).integers(3, 20, size=length // 3 + 2)
    labels = np.repeat((ev_len >= 12).astype(np.uint8), ev_len)[:length]
    return raw, infer.normalize_raw_signal(raw, "median").astype(np.float32), labels


def _windows(reads):
    x = np.concatenate([r[1][: r[1].size // 35 * 35] for r in reads]).reshape(-1, 35, 1)
    y = np.concatenate([r[2][: r[2].size // 35 * 35] for r in reads])
    return x, y


# Step budget of the learning test: the held-out check runs every 50 steps and training stops once the loss has
# halved; DESIGN.md ("Training") gives the step at which a B200 run first met it, well inside this budget.
LEARN_STEPS, LEARN_RATE = 3000, 0.003


@pytest.mark.parametrize("kind", ["RNN", "ResNetRNN"])
def test_training_learns_event_lengths(kind):
    from catfish_b200 import infer, metrics, train_validate, weights
    hpm = dict(layer_size=32, n_layers=2) if kind == "RNN" else \
        dict(layer_size=64, n_layers=3, layer_size_res=32, n_layers_res=2)
    w0 = weights.random_init(kind, seed=3, **hpm)
    m = _model(kind, hpm, w0, engine="auto", keep_prob=0.8, learning_rate=LEARN_RATE)
    train_reads = [_labelled_read(9000, 1000 + i) for i in range(40)]
    held = [_labelled_read(7000, 5000 + i) for i in range(6)]
    tx, ty = _windows(train_reads)
    hx, hy = _windows(held)
    _, loss0 = m.test_network(hx, hy)
    p0, r0 = train_validate.validate(m, [(r[1], r[2]) for r in held], 0, validation_start="complete")[1:]
    rng = np.random.default_rng(0)
    trace = []
    for step in range(LEARN_STEPS):
        idx = rng.integers(0, tx.shape[0], size=256)
        m.train_network(tx[idx], ty.reshape(-1, 35)[idx].reshape(-1))
        if (step + 1) % 50 == 0:
            trace.append(float(m.test_network(hx, hy)[1]))
            if trace[-1] <= 0.5 * loss0:
                break
    _, loss1 = m.test_network(hx, hy)
    p1, r1 = train_validate.validate(m, [(r[1], r[2]) for r in held], 0, validation_start="complete")[1:]
    print("%s: held-out loss %.4f -> %.4f after %d steps, f1 %.4f -> %.4f; every 50 steps: %s"
          % (kind, loss0, loss1, m.global_step, metrics.f1(p0, r0), metrics.f1(p1, r1),
             " ".join("%.3f" % v for v in trace)))
    assert loss1 <= 0.5 * loss0
    assert metrics.f1(p1, r1) > metrics.f1(p0, r0)
    # the trained model infers as a fresh model built from its weights
    fresh = _model(kind, hpm, m.get_weights(), engine="auto")
    raws = [r[0] for r in held]
    hp_a, len_a, s_a = infer.infer_reads(raws, m, return_scores=True)
    hp_b, len_b, s_b = infer.infer_reads(raws, fresh, return_scores=True)
    assert [list(map(list, h)) for h in hp_a] == [list(map(list, h)) for h in hp_b]
    for a, b in zip(s_a, s_b):
        assert np.array_equal(np.asarray(a), np.asarray(b))


# ---------------------------------------------------------------- refusals
def test_training_refusals(shipped_weights):
    kind, hpm, w = _weights("shipped", shipped=shipped_weights)
    x, y = _batch(4, 0)
    with pytest.raises(ValueError):
        _model(kind, hpm, w, optimizer_choice="Adam").train_network(x, y)
    m = _model(kind, hpm, w)
    for keep in (0.0, 1.5):
        m.keep_prob = keep
        with pytest.raises(ValueError):
            m.train_network(x, y)
    m.keep_prob = 0.8
    with pytest.raises(ValueError):
        m.train_network(x[:, :34], y)
    with pytest.raises(ValueError):
        m.train_network(x, y[:-1])
    bad = y.copy()
    bad[3] = 2
    with pytest.raises(ValueError):
        m.train_network(x, bad)
    assert m.global_step == 0


def test_c_abi_bad_arguments(shipped_weights):
    import torch
    from catfish_b200 import _cabi, weights
    lib = _cabi.load_library()
    kind, hpm, w = _weights("shipped", shipped=shipped_weights)
    m = _model(kind, hpm, w)
    names = list(weights.expected_shapes(kind, **hpm))
    arrays = [np.ascontiguousarray(w[n], np.float32) for n in names]
    ptrs = (ctypes.c_void_p * len(names))(*[a.ctypes.data for a in arrays])
    sizes = (ctypes.c_int64 * len(names))(*[a.size for a in arrays])
    desc = m._desc()
    tr = ctypes.c_void_p()
    assert lib.cf_trainer_create(None, ptrs, sizes, len(names), None, None, 0, ctypes.byref(tr)) == _cabi.CF_ERR_BAD_ARG
    assert lib.cf_trainer_create(ctypes.byref(desc), ptrs, sizes, len(names) - 1, None, None, 0,
                                 ctypes.byref(tr)) == _cabi.CF_ERR_BAD_ARG
    bad_sizes = (ctypes.c_int64 * len(names))(*[a.size for a in arrays])
    bad_sizes[3] += 1
    assert lib.cf_trainer_create(ctypes.byref(desc), ptrs, bad_sizes, len(names), None, None, 0,
                                 ctypes.byref(tr)) == _cabi.CF_ERR_BAD_ARG
    _cabi.check(lib.cf_trainer_create(ctypes.byref(desc), ptrs, sizes, len(names), None, None, 0, ctypes.byref(tr)))
    try:
        xd = torch.zeros(4 * 35, device="cuda")
        yd = torch.zeros(4 * 35, dtype=torch.uint8, device="cuda")
        x, y = xd.data_ptr(), yd.data_ptr()

        def step(t=tr, xp=x, yp=y, n=4, lr=1e-3, keep=0.8, s=0):
            return lib.cf_trainer_step(t, xp, yp, n, lr, keep, 0, s, None, None, None)
        assert step(t=None) == _cabi.CF_ERR_BAD_ARG
        assert step(xp=None) == _cabi.CF_ERR_BAD_ARG
        assert step(yp=None) == _cabi.CF_ERR_BAD_ARG
        assert step(n=0) == _cabi.CF_ERR_BAD_ARG
        for keep in (0.0, -0.5, 1.0001, float("nan")):
            assert step(keep=keep) == _cabi.CF_ERR_BAD_ARG
        for lr in (0.0, -1e-3, float("nan"), float("inf")):
            assert step(lr=lr) == _cabi.CF_ERR_BAD_ARG
        assert step(s=-1) == _cabi.CF_ERR_BAD_ARG
        assert lib.cf_trainer_gradients(tr, x, y, 4, 1.0, 0, 0, None, None, None) == _cabi.CF_ERR_BAD_ARG
        assert lib.cf_trainer_read(tr, None, None, None) == _cabi.CF_ERR_BAD_ARG
        assert step() == _cabi.CF_OK
        torch.cuda.synchronize()
    finally:
        lib.cf_trainer_destroy(tr)
