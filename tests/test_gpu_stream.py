"""GPU: streaming inference (infer.infer_stream) and the execution contexts of the C ABI (cf_exec_*).

A stream must give exactly what one infer_reads call on the whole list gives, in input order, whatever the
grouping and the number of groups in flight; it must pull reads lazily, flush early on request, meet a bad read
the way the reference's one-file-at-a-time loop does, and release everything when it ends.  Contexts of one model
must run concurrently without disturbing each other or the model's default context."""
import ctypes
import threading

import numpy as np
import pytest

from catfish_b200 import _cabi, infer, neural_network, synth, weights

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def shipped():
    return neural_network.load_network("ResNetRNN", None, 30000)


def _model(kind, engine="auto", seed=7):
    hpm = {}
    if kind != "RNN":
        hpm.update(layer_size_res=32, n_layers_res=2)
    if kind != "ResNet":
        hpm.update(layer_size=64, n_layers=3)
    full = dict(weights.SHIPPED_HPARAMS)
    full.update(hpm)
    m = neural_network.build_model(kind, engine=engine, **full)
    m.set_weights(weights.random_init(kind, seed=seed, **hpm))
    return m


def _mixed_reads(seed=0):
    """Edge lengths around one window, a 4481-sample read, a 1M-sample read, many 10k reads and U{50k..200k} reads."""
    rng = np.random.default_rng(seed)
    lengths = [1, 34, 35, 36, 4481, 1_000_000] + [10_000] * 40 + synth.ragged_lengths(12, 50_000, 200_000, seed).tolist()
    order = rng.permutation(len(lengths))
    return synth.synth_reads([lengths[i] for i in order], base_seed=1000 * seed + 5)


def _assert_same(got, hps, lengths, scores=None):
    assert len(got) == len(hps)
    for r, item in enumerate(got):
        assert isinstance(item[0], infer.IntervalList)
        assert np.array_equal(item[0].array, hps[r].array), "read %d" % r
        assert item[1] == lengths[r]
        if scores is not None:
            assert len(item) == 3
            assert item[2].dtype == np.float32
            assert np.array_equal(item[2], scores[r], equal_nan=True), "scores of read %d" % r
        else:
            assert len(item) == 2


SETTINGS = [(1, 2), (50_000, 1), (300_000, 3), (None, 2)]     # (group_samples, depth); 1 = one read per group


@pytest.mark.parametrize("kind", ["ResNetRNN", "RNN", "ResNet", "simt"])
def test_stream_equals_infer_reads(kind, shipped):
    model = shipped if kind == "ResNetRNN" else (
        neural_network.load_network("ResNetRNN", None, 30000, engine="simt") if kind == "simt" else _model(kind))
    reads = _mixed_reads(seed=3)
    hps, lengths = infer.infer_reads(reads, model)
    for group_samples, depth in SETTINGS:
        got = list(infer.infer_stream(iter(reads), model, group_samples=group_samples, depth=depth))
        _assert_same(got, hps, lengths)
    hps_s, lengths_s, scores = infer.infer_reads(reads, model, return_scores=True)
    for group_samples, depth in [(1, 3), (300_000, 2)]:
        got = list(infer.infer_stream(reads, model, return_scores=True, group_samples=group_samples, depth=depth))
        _assert_same(got, hps_s, lengths_s, scores)


class _Counting(object):
    """An iterable that counts the reads taken from it."""

    def __init__(self, reads):
        self.reads, self.pulled = reads, 0

    def __iter__(self):
        for r in self.reads:
            self.pulled += 1
            yield r


def test_stream_is_lazy_and_bounded(shipped):
    reads = synth.synth_reads([10_000] * 60, base_seed=77)
    hps, lengths = infer.infer_reads(reads, shipped)
    for depth in (1, 2, 3):
        src = _Counting(reads)
        got = []
        for i, item in enumerate(infer.infer_stream(src, shipped, group_samples=30_000, depth=depth)):
            assert src.pulled - i <= (depth + 1) * 3, (depth, i, src.pulled)      # 3 reads per group
            got.append(item)
        _assert_same(got, hps, lengths)


def test_stream_close_mid_way(shipped):
    reads = synth.synth_reads([10_000] * 60, base_seed=78)
    src = _Counting(reads)
    stream = infer.infer_stream(src, shipped, group_samples=30_000, depth=2)
    got = []
    for item in stream:
        got.append(item)
        if len(got) == 10:
            break
    stream.close()
    pulled = src.pulled
    assert pulled <= 10 + 3 * 3
    hps, lengths = infer.infer_reads(reads, shipped)
    _assert_same(got, hps[:10], lengths[:10])
    assert src.pulled == pulled
    with pytest.raises(StopIteration):
        next(stream)


def test_stream_early_flush(shipped):
    reads = synth.synth_reads([5_000] * 12, base_seed=79)
    for depth in (1, 2):
        src = _Counting(reads)
        stream = infer.infer_stream(src, shipped, max_wait_s=0, depth=depth)
        first = next(stream)
        assert src.pulled <= depth + 1, (depth, src.pulled)
        hps, lengths = infer.infer_reads(reads[:1], shipped)
        _assert_same([first], hps, lengths)
        stream.close()


@pytest.mark.parametrize("bad, exc", [(np.zeros(0, np.int16), IndexError),
                                      (np.full(100, 500.25), ValueError)])
def test_stream_bad_read_mid_stream(bad, exc, shipped):
    k = 7
    reads = synth.synth_reads([3_000] * 12, base_seed=80)
    with pytest.raises(exc):
        infer.infer_reads(reads[:k] + [bad] + reads[k:], shipped)
    hps, lengths = infer.infer_reads(reads[:k], shipped)
    got = []
    with pytest.raises(exc):
        for item in infer.infer_stream(reads[:k] + [bad] + reads[k:], shipped, group_samples=6_000, depth=2):
            got.append(item)
    _assert_same(got, hps, lengths)


def test_stream_window_size_checked_before_pulling(shipped):
    src = _Counting(synth.synth_reads([1000] * 3))
    with pytest.raises(ValueError):
        infer.infer_stream(src, shipped, window_size=36)
    assert src.pulled == 0


# ---------------------------------------------------------------------------------------------- C ABI
def _batch(seed, n):
    reads = synth.synth_reads(synth.ragged_lengths(n, 2_000, 120_000, seed), base_seed=seed)
    raw, offsets = synth.concat_reads(reads)
    return raw, offsets


class _Call(object):
    """Device buffers of one cf_infer_reads / cf_exec_infer_reads call, and its results after a sync."""

    def __init__(self, torch, lib, raw, offsets, min_run=15):
        self.offsets = offsets
        self.n = len(offsets) - 1
        self.cap = int(lib.cf_max_intervals(int(offsets[-1]), self.n, min_run))
        self.raw = torch.from_numpy(raw).cuda()
        self.iv = torch.empty((self.cap, 2), dtype=torch.int64, device="cuda")
        self.ioff = torch.empty(self.n + 1, dtype=torch.int64, device="cuda")
        self.probs = torch.empty(int(offsets[-1]), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()

    def args(self, stream):
        return (self.raw.data_ptr(), self.offsets.ctypes.data_as(_cabi.c_i64_p), self.n, self.probs.data_ptr(),
                self.iv.data_ptr(), self.ioff.data_ptr(), self.cap, 0.5, 15, 11, 16, stream.cuda_stream)

    def result(self):
        ioff = self.ioff.cpu().numpy()
        return ioff, self.iv[:int(ioff[-1])].cpu().numpy(), self.probs.cpu().numpy()


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(a[2], b[2], equal_nan=True)


def test_contexts_overlap_and_match_default_context(shipped):
    import torch
    lib = _cabi.load_library()
    batches = [_batch(11, 40), _batch(12, 25), _batch(13, 60)]
    st = [torch.cuda.Stream() for _ in range(3)]
    # sequential default-context calls
    want = []
    for raw, off in batches:
        c = _Call(torch, lib, raw, off)
        _cabi.check(lib.cf_infer_reads(shipped.handle, *c.args(st[0])))
        st[0].synchronize()
        want.append(c.result())
    ex = [ctypes.c_void_p(), ctypes.c_void_p()]
    for e in ex:
        _cabi.check(lib.cf_exec_create(shipped.handle, ctypes.byref(e)))
    try:
        _cabi.check(lib.cf_exec_reserve(ex[1], 4_000_000, 64))
        for _ in range(2):
            calls = [_Call(torch, lib, raw, off) for raw, off in batches]
            # two contexts on two streams, and the default context on a third, with no sync in between
            _cabi.check(lib.cf_exec_infer_reads(ex[0], *calls[0].args(st[0])))
            _cabi.check(lib.cf_exec_infer_reads(ex[1], *calls[1].args(st[1])))
            _cabi.check(lib.cf_infer_reads(shipped.handle, *calls[2].args(st[2])))
            for s in st:
                s.synchronize()
            for c, w in zip(calls, want):
                _same(c.result(), w)
        # one context, two streams: the second call waits for the first
        calls = [_Call(torch, lib, raw, off) for raw, off in batches[:2]]
        _cabi.check(lib.cf_exec_infer_reads(ex[0], *calls[0].args(st[0])))
        _cabi.check(lib.cf_exec_infer_reads(ex[0], *calls[1].args(st[1])))
        torch.cuda.synchronize()
        for c, w in zip(calls, want):
            _same(c.result(), w)
        # errors come back as for the handle
        bad = np.array([0, 0], np.int64)
        c = calls[0]
        rc = lib.cf_exec_infer_reads(ex[0], c.raw.data_ptr(), bad.ctypes.data_as(_cabi.c_i64_p), 1, None,
                                     c.iv.data_ptr(), c.ioff.data_ptr(), c.cap, 0.5, 15, 11, 16, st[0].cuda_stream)
        assert rc == _cabi.CF_ERR_EMPTY_READ
        _cabi.check(lib.cf_exec_infer_reads(ex[0], *calls[1].args(st[0])))
        st[0].synchronize()
        _same(calls[1].result(), want[1])
    finally:
        for e in ex:
            lib.cf_exec_destroy(e)


def test_context_outlives_model_handle():
    import torch
    lib = _cabi.load_library()
    model = neural_network.load_network("ResNetRNN", None, 30000)
    raw, off = _batch(21, 30)
    s = torch.cuda.Stream()
    c = _Call(torch, lib, raw, off)
    _cabi.check(lib.cf_infer_reads(model.handle, *c.args(s)))
    s.synchronize()
    want = c.result()
    ex, idle = ctypes.c_void_p(), ctypes.c_void_p()
    _cabi.check(lib.cf_exec_create(model.handle, ctypes.byref(ex)))
    _cabi.check(lib.cf_exec_create(model.handle, ctypes.byref(idle)))
    model.close()                                  # cf_model_destroy: the contexts keep the weights alive
    lib.cf_exec_destroy(idle)                      # a context that never ran
    for _ in range(2):
        c = _Call(torch, lib, raw, off)
        _cabi.check(lib.cf_exec_infer_reads(ex, *c.args(s)))
        s.synchronize()
        _same(c.result(), want)
    # the last reference goes while the context's last call is still in flight on another stream: destroying the
    # context waits for that call before it frees the context and the weights
    s2 = torch.cuda.Stream()
    c = _Call(torch, lib, raw, off)
    _cabi.check(lib.cf_exec_infer_reads(ex, *c.args(s2)))
    lib.cf_exec_destroy(ex)
    s2.synchronize()
    _same(c.result(), want)


def test_two_threads_stream_through_one_model(shipped):
    lists = [synth.synth_reads(synth.ragged_lengths(50, 5_000, 150_000, 31), base_seed=31),
             synth.synth_reads(synth.ragged_lengths(70, 1_000, 60_000, 32), base_seed=32)]
    want = [infer.infer_reads(reads, shipped) for reads in lists]
    got, errors = [None, None], []

    def run(i):
        try:
            got[i] = list(infer.infer_stream(lists[i], shipped, group_samples=400_000, depth=2))
        except BaseException as e:      # reported by the main thread
            errors.append(e)

    threads = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for g, (hps, lengths) in zip(got, want):
        _assert_same(g, hps, lengths)


@pytest.mark.parametrize("kind", ["RNN", "simt"])
def test_reserved_context_matches_default_context(kind):
    """cf_exec_reserve and cf_model_reserve size the engine workspaces too (the CUDA-core one for the CUDA-core engine
    and for the tensor-core engine's RNN-only input); a call within the reservation gives the results of a default
    context that was not reserved."""
    import torch
    lib = _cabi.load_library()

    def make():
        return _model("RNN") if kind == "RNN" else neural_network.load_network("ResNetRNN", None, 30000, engine="simt")

    model = make()
    raw, off = _batch(41, 20)
    s = torch.cuda.Stream()
    c = _Call(torch, lib, raw, off)
    _cabi.check(lib.cf_infer_reads(model.handle, *c.args(s)))
    s.synchronize()
    want = c.result()
    ex = ctypes.c_void_p()
    _cabi.check(lib.cf_exec_create(model.handle, ctypes.byref(ex)))
    try:
        _cabi.check(lib.cf_exec_reserve(ex, int(off[-1]), len(off) - 1))
        c = _Call(torch, lib, raw, off)
        _cabi.check(lib.cf_exec_infer_reads(ex, *c.args(s)))
        s.synchronize()
        _same(c.result(), want)
    finally:
        lib.cf_exec_destroy(ex)
    # the default context of a second model with the same weights, reserved before its first call
    reserved = make()
    _cabi.check(lib.cf_model_reserve(reserved.handle, int(off[-1]), len(off) - 1))
    c = _Call(torch, lib, raw, off)
    _cabi.check(lib.cf_infer_reads(reserved.handle, *c.args(s)))
    s.synchronize()
    _same(c.result(), want)
