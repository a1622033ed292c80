"""The group pipeline of infer_reads / evaluate_reads: how a batch is cut into groups of whole reads (no GPU), and,
on the GPU, that concurrent calls never share a buffer and that the model's buffers are freed with the model."""
import threading

import numpy as np
import pytest

from catfish_b200 import infer, neural_network, synth
from helpers import random_labels


def _offsets(lengths):
    off = np.zeros(len(lengths) + 1, np.int64)
    np.cumsum(lengths, out=off[1:])
    return off


def _check_groups(groups, off, first, later):
    n_reads = len(off) - 1
    assert [lo for lo, _ in groups] == [0] + [hi for _, hi in groups[:-1]]         # in order, no gaps
    assert (groups[-1][1] if groups else 0) == n_reads                              # every read
    for g, (lo, hi) in enumerate(groups):
        want = first if g == 0 else later
        assert hi > lo                                                              # never empty
        size = off[hi] - off[lo]
        assert size <= want or hi == lo + 1                                         # over only for a single read
        if hi < n_reads:
            assert off[hi + 1] - off[lo] > want                                     # the next read would not fit


def test_cut_groups_hand_made():
    lengths = [3, 4, 10, 1, 1, 1, 20, 2, 2]
    off = _offsets(lengths)
    groups = infer._cut_groups(off, 5, 8)
    assert groups == [(0, 1), (1, 2), (2, 3), (3, 6), (6, 7), (7, 9)]
    _check_groups(groups, off, 5, 8)
    assert infer._cut_groups(off, 100, 100) == [(0, 9)]
    assert infer._cut_groups(off, 1, 1) == [(r, r + 1) for r in range(9)]
    assert infer._cut_groups(_offsets([]), 5, 8) == []
    assert infer._cut_groups(_offsets([7]), 5, 8) == [(0, 1)]


@pytest.mark.parametrize("seed", range(5))
def test_cut_groups_random(seed):
    rng = np.random.default_rng(seed)
    lengths = rng.integers(1, 5_000, size=int(rng.integers(1, 400)))
    off = _offsets(lengths)
    for first, later in ((1_000, 4_000), (4_000, 4_000), (1, 10), (10 ** 9, 10 ** 9)):
        _check_groups(infer._cut_groups(off, first, later), off, first, later)


def test_first_group_is_a_quarter_pass():
    off = _offsets([10_000] * 3_000)
    groups = infer._cut_groups(off, infer._FIRST_GROUP_SAMPLES, infer._GROUP_SAMPLES)
    assert infer._FIRST_GROUP_SAMPLES * 4 == infer._GROUP_SAMPLES
    assert [hi - lo for lo, hi in groups] == [260, 1040, 1040, 660]


# ---------------------------------------------------------------------------------------------- GPU
def _workload(seed):
    """A batch of several groups with labels, and a small batch."""
    rng = np.random.default_rng(seed)
    big = synth.synth_reads(synth.ragged_lengths(80, 100_000, 200_000, seed=seed), base_seed=100 * seed)
    assert sum(r.size for r in big) > infer._GROUP_SAMPLES             # several groups in both calls
    labels = [random_labels(rng, r.size).astype(np.uint8) for r in big]
    small = synth.synth_reads(synth.ragged_lengths(5, 2_000, 20_000, seed=seed), base_seed=100 * seed + 90)
    return big, labels, small


TH = np.linspace(0.05, 0.95, 19)


def _run(model, work):
    big, labels, small = work
    iv, ioff, _ = infer.infer_reads_arrays(big, model)
    hps, lens = infer.infer_reads(small, model)
    counts = infer.evaluate_reads(big, labels, model, TH)
    return iv, ioff, [h.array for h in hps], lens, counts


def _same(a, b):
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert len(a[2]) == len(b[2]) and all(np.array_equal(x, y) for x, y in zip(a[2], b[2]))
    assert a[3] == b[3] and np.array_equal(a[4], b[4])


@pytest.mark.gpu
@pytest.mark.parametrize("models", ["one model", "two models"])
def test_concurrent_calls_equal_single_threaded(models):
    first = neural_network.load_network("ResNetRNN", None, 30000)
    pair = [first, first if models == "one model" else neural_network.load_network("ResNetRNN", None, 30000)]
    works = [_workload(1), _workload(2)]
    want = [_run(first, w) for w in works]
    got, errors = [[], []], []
    start = threading.Barrier(2)

    def run(i):
        try:
            for _ in range(3):
                start.wait()
                got[i].append(_run(pair[i], works[i]))
        except BaseException as e:      # reported by the main thread
            errors.append(e)
            start.abort()

    threads = [threading.Thread(target=run, args=(i,)) for i in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    for i in range(2):
        assert len(got[i]) == 3
        for res in got[i]:
            _same(res, want[i])


@pytest.mark.gpu
def test_close_returns_the_device_memory():
    import torch
    model = neural_network.load_network("ResNetRNN", None, 30000)
    big, labels, _ = _workload(3)
    dev = torch.device("cuda", model.device)
    torch.cuda.synchronize(dev)
    before = torch.cuda.memory_allocated(dev)
    infer.infer_reads(big, model)
    infer.evaluate_reads(big, labels, model, TH)
    assert torch.cuda.memory_allocated(dev) > before          # the model keeps its buffers between calls
    model.close()
    assert torch.cuda.memory_allocated(dev) == before
