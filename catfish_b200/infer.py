"""Mirror of /root/reference/catfish/infer.py: the per-read inference driver.

Same function names, arguments, defaults and return types as the reference;
the arithmetic runs on the GPU through the C ABI (include/catfish_b200.h):

===========================  ==========================  =========================
reference (catfish/infer.py)  here                        C-ABI entry
===========================  ==========================  =========================
infer_class_from_signal :12   infer_class_from_signal     cf_infer_reads
(array-level twins)           infer_class_from_raw,       cf_infer_reads
                              infer_reads
(the CLI's per-file loop)     infer_stream                cf_exec_infer_reads
(precision_recall_ROC.py)     evaluate_reads              cf_infer_reads + cf_sweep_thresholds
(metrics.py, sklearn curves)  evaluate_reads_curve        cf_infer_reads + cf_curve_create
process_signal :77            process_signal (h5py)       cf_normalize_reads
normalize_raw_signal :96      normalize_raw_signal        cf_normalize_reads
reshape_input :108            reshape_input               (pure reshape, host)
class_from_threshold :128     class_from_threshold        cf_class_from_threshold
hp_in_pred :141               hp_in_pred                  cf_hp_in_pred
correct_short :174            correct_short               cf_correct_short
===========================  ==========================  =========================

PyTorch tensors are used only to hold device buffers and to name the stream.
"""

import collections
import collections.abc
import ctypes
import os
import threading
import time

import numpy as np

from . import _cabi


class IntervalList(collections.abc.Sequence):
    """The ``[[start, end], ...]`` list of one read (infer.py:149-162), backed by the int64 [n, 2] slice of the
    batch result.  Behaves like the reference's list of two-element lists of Python ints (indexing, iteration,
    ``len``, ``==`` with a list), but the Python objects are only built when asked for: a 512-read batch holds
    ~3e5 intervals and eager conversion costs more than the GPU work of the whole batch."""

    __slots__ = ("array",)

    def __init__(self, array):
        self.array = array

    def __len__(self):
        return int(self.array.shape[0])

    def __getitem__(self, i):
        if isinstance(i, slice):
            return self.array[i].tolist()
        return self.array[i].tolist()

    def __iter__(self):
        return iter(self.array.tolist())

    def __eq__(self, other):
        if isinstance(other, IntervalList):
            return np.array_equal(self.array, other.array)
        if isinstance(other, (list, tuple)):
            return self.array.tolist() == [list(x) if isinstance(x, tuple) else x for x in other]
        return NotImplemented

    def __ne__(self, other):
        r = self.__eq__(other)
        return r if r is NotImplemented else not r

    __hash__ = None

    def tolist(self):
        return self.array.tolist()

    def __repr__(self):
        return repr(self.array.tolist())

    def __reduce__(self):
        return (IntervalList, (np.ascontiguousarray(self.array),))


_POOL = None
_POOL_LOCK = threading.Lock()


def _concat_into(stage, arrays, offsets):
    """Ragged concat of the batch into the pinned staging buffer.  Large batches are split into a few
    contiguous groups copied by worker threads (numpy releases the GIL while copying): one thread moves
    ~10 GB/s, which for a 128 MB batch is a tenth of the GPU time of the whole call."""
    global _POOL
    total = int(offsets[-1])
    workers = min(8, os.cpu_count() or 1)
    if total < (1 << 23) or len(arrays) < 2 * workers or workers < 2:
        np.concatenate(arrays, out=stage)
        return
    with _POOL_LOCK:
        if _POOL is None:
            import concurrent.futures
            _POOL = concurrent.futures.ThreadPoolExecutor(max_workers=workers, thread_name_prefix="catfish-stage")
    cuts = np.searchsorted(offsets, np.linspace(0, total, workers + 1)[1:-1]).tolist()
    bounds = [0] + cuts + [len(arrays)]
    jobs = []
    for lo, hi in zip(bounds, bounds[1:]):
        if hi > lo:
            jobs.append(_POOL.submit(np.concatenate, arrays[lo:hi], out=stage[int(offsets[lo]):int(offsets[hi])]))
    for j in jobs:
        j.result()


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise _cabi.CatfishError("catfish_b200 needs a CUDA device (no CPU fallback)")
    return torch


def _device_index(device=None):
    from . import get_device
    return get_device() if device is None else int(device)


def _offsets_ptr(offsets):
    return offsets.ctypes.data_as(_cabi.c_i64_p)


# ------------------------------------------------------------------------------ inference
def infer_class_from_signal(fast5_file, model, label=1, window_size=35):
    """infer.py:12-51: FAST5 path -> (list of [start, end] homopolymer intervals, read length)."""
    if not os.path.exists(fast5_file):
        raise ValueError("path to FAST5 is not correct.")
    import h5py                                   # not a dependency of the array-level API
    with h5py.File(fast5_file, "r") as fast5:
        raw = _trimmed_raw(fast5)
    return infer_class_from_raw(raw, model, label=label, window_size=window_size)


def infer_class_from_raw(raw, model, label=1, window_size=35, threshold=0.5):
    """Array-level twin of infer_class_from_signal: ``raw`` is the int16 signal of one read
    with the leading ``first_sample_template`` samples already dropped (infer.py:87-90)."""
    hps, lengths = infer_reads([raw], model, threshold=threshold, window_size=window_size)
    return hps[0].tolist(), lengths[0]          # a plain list of [int, int], exactly the reference's type


def infer_reads(raws, model, threshold=0.5, min_run=15, extension_left=11, extension_right=16,
                window_size=35, return_scores=False):
    """Batched infer_class_from_signal over a list of int16 reads (ragged).

    Returns ``(hps, lengths)`` - per read the [start, end] intervals (an ``IntervalList``: list-like, Python
    ints on access, as the reference) and ``len(labels)`` - plus the per-position float32 scores when
    ``return_scores`` is set.  The batch runs as groups of whole reads, about one engine pass each (the first a
    quarter pass, so that the device starts early), with two groups in flight: while the device works on one group
    (``cf_infer_reads``: median/MAD normalisation, windowing, network, threshold / short-run removal / interval
    emission), the host concatenates the next one straight into pinned staging and starts its copy."""
    res = infer_reads_arrays(raws, model, threshold, min_run, extension_left, extension_right, window_size,
                             return_scores)
    intervals, ioff, lengths = res[0], res[1], res[2]
    bounds = ioff.tolist()
    hps = [IntervalList(intervals[bounds[r]:bounds[r + 1]]) for r in range(len(lengths))]
    if return_scores:
        return hps, lengths.tolist(), res[3]
    return hps, lengths.tolist()


def infer_reads_arrays(raws, model, threshold=0.5, min_run=15, extension_left=11, extension_right=16,
                       window_size=35, return_scores=False):
    """``infer_reads`` with the result left in CSR form: ``(intervals int64 [n, 2], interval_offsets int64 [R + 1],
    lengths int64 [R][, scores list])`` - what the sharded job gathers (no per-read Python objects)."""
    if window_size != model.window:
        raise ValueError("window_size must equal the model's window (%d)" % model.window)
    arrays = [_as_int16(r) for r in raws]
    for a in arrays:
        if a.size == 0:
            raise IndexError("list index out of range")        # infer.py:184 on an empty read
    lengths = np.array([a.size for a in arrays], np.int64)
    offsets = np.zeros(len(arrays) + 1, np.int64)
    np.cumsum(lengths, out=offsets[1:])
    params = (float(threshold), int(min_run), int(extension_left), int(extension_right))
    results = _run_on_model(model, [(arrays[lo:hi], params, return_scores)
                                    for lo, hi in _cut_groups(offsets, _FIRST_GROUP_SAMPLES, _GROUP_SAMPLES)])
    intervals, ioff = np.zeros((0, 2), np.int64), np.zeros(len(arrays) + 1, np.int64)
    if results:
        intervals = np.concatenate([iv for _, iv, _, _ in results])
        np.cumsum(np.concatenate([np.diff(ioff_g) for _, _, ioff_g, _ in results]), out=ioff[1:])
    if return_scores:
        scores = [s[int(off[r]):int(off[r + 1])] for off, _, _, s in results for r in range(len(off) - 1)]
        return intervals, ioff, lengths, scores
    return intervals, ioff, lengths


_GROUP_SAMPLES = 10_400_000             # one engine pass (2368 tiles of 128 windows) per group
_FIRST_GROUP_SAMPLES = 2_600_000        # a quarter pass: the device starts after ~0.5 ms of staging instead of ~2 ms
_DEPTH = 2                              # groups in flight of infer_reads_arrays and evaluate_reads


def _cut_groups(offsets, first, later):
    """``(lo, hi)`` ranges of consecutive whole reads, in order, of the batch with CSR ``offsets``: the first group
    holds at most ``first`` samples, every later one at most ``later``, unless a single read is longer."""
    groups, lo, want = [], 0, first
    while lo < len(offsets) - 1:
        hi = max(int(np.searchsorted(offsets, offsets[lo] + want, side="right")) - 1, lo + 1)
        groups.append((lo, hi))
        lo, want = hi, later
    return groups


def evaluate_reads(raws, labels, model, thresholds, window_size=35):
    """Confusion counts of labelled raw reads at every threshold: int64 ``[T, 4]`` rows of (tp, fp, tn, fn), in the
    order of ``thresholds`` (1..4096 of them, unsorted / repeated allowed).

    ``labels[i]`` holds one label per sample of ``raws[i]`` (0 / 1; other small integers count as
    ``metrics.confusion_matrix`` counts them).  The reads take the production path - median / MAD normalisation,
    windowing, network - with the probabilities left on the device, and every real sample is counted at every
    threshold on the device (``cf_sweep_thresholds``; padding never enters: the probabilities are already unpadded).
    Row i equals ``metrics.confusion_matrix`` of the labels against ``scores >= thresholds[i]`` for the scores
    ``infer_reads(..., return_scores=True)`` gives; reads with MAD = 0 have NaN scores, predicted 0 everywhere.
    Batches are processed in groups of about one engine pass; no probability travels to the host."""
    arrays, labs = _labelled_reads(raws, labels, model, window_size)
    th = np.ascontiguousarray(np.asarray(thresholds, dtype=np.float64).reshape(-1))
    counts = np.zeros((th.size, 4), np.int64)
    # no positions: checks the thresholds on the host, before any device work, and leaves the counts at zero
    _cabi.check(_cabi.load_library().cf_sweep_thresholds(0, None, 0, None, 0, th.ctypes.data, min(th.size, 2 ** 31 - 1),
                                                         counts.ctypes.data_as(_cabi.c_i64_p), None))
    if not arrays:
        return counts
    offsets = np.zeros(len(arrays) + 1, np.int64)
    np.cumsum([a.size for a in arrays], out=offsets[1:])
    params = (0.5, 15, 11, 16)                                 # only the probabilities are used
    for part in _run_on_model(model, [(arrays[lo:hi], params, False, labs[lo:hi], th)
                                      for lo, hi in _cut_groups(offsets, _GROUP_SAMPLES, _GROUP_SAMPLES)]):
        counts += part
    return counts


def evaluate_reads_curve(raws, labels, model, window_size=35, points=True):
    """The exact curve of labelled raw reads at every distinct score: ``metrics.score_curve`` of the scores
    ``infer_reads(..., return_scores=True)`` gives and the labels (0 / 1 only, one per sample), as a
    ``metrics.ScoreCurve``; reads with MAD = 0 have NaN scores, never positive.

    The reads take ``evaluate_reads``' production path, in groups of about one engine pass; each group's network
    writes its probabilities straight into one device tensor for the whole read set, at the group's offset, and its
    labels go to one uint8 tensor beside it.  One ``cf_curve_create`` then sorts and counts both.  No probability
    travels to the host.  Device memory: 5 B per sample for the probabilities and labels, 8.5 B per sample of sort
    scratch during the count, and 12 B per row of the curve while it is read."""
    from . import metrics
    arrays, labs = _labelled_reads(raws, labels, model, window_size)
    for r, y in enumerate(labs):
        if y.size and int(y.max()) > 1:
            raise ValueError("score curve: read %d has a label other than 0 / 1" % r)
    offsets = np.zeros(len(arrays) + 1, np.int64)
    np.cumsum([a.size for a in arrays], out=offsets[1:])
    total = int(offsets[-1])
    if total == 0:
        return metrics.score_curve(np.zeros(0, np.float32), np.zeros(0, np.uint8), points=points)
    torch = _torch()
    with torch.cuda.device(model.device):
        probs = torch.empty(total, dtype=torch.float32, device="cuda:%d" % model.device)
        labs_dev = torch.empty(total, dtype=torch.uint8, device="cuda:%d" % model.device)
    params = (0.5, 15, 11, 16)                                 # only the probabilities are used
    _run_on_model(model, [(arrays[lo:hi], params, False, labs[lo:hi], None, (probs, labs_dev, int(offsets[lo])))
                          for lo, hi in _cut_groups(offsets, _GROUP_SAMPLES, _GROUP_SAMPLES)])
    return metrics.score_curve(probs, labs_dev, points=points)


def _labelled_reads(raws, labels, model, window_size):
    """The int16 reads and their uint8 labels (one per sample) of ``evaluate_reads`` and ``evaluate_reads_curve``."""
    if window_size != model.window:
        raise ValueError("window_size must equal the model's window (%d)" % model.window)
    arrays = [_as_int16(r) for r in raws]
    labels = list(labels)
    if len(labels) != len(arrays):
        raise ValueError("one label array per read is needed (%d reads, %d label arrays)" % (len(arrays), len(labels)))
    labs = []
    for r, (a, y) in enumerate(zip(arrays, labels)):
        if a.size == 0:
            raise IndexError("list index out of range")        # infer.py:184 on an empty read
        y = np.asarray(y).reshape(-1)
        if y.size != a.size:
            raise ValueError("read %d has %d samples and %d labels" % (r, a.size, y.size))
        y8 = y.astype(np.uint8)
        if not np.array_equal(y8, y):
            raise ValueError("labels must be small non-negative integers")
        labs.append(y8)
    return arrays, labs


_STREAM_DEPTH = 2                       # groups in flight in infer_stream
_STREAM_GROUP_SAMPLES = 2_600_000       # samples per group of infer_stream: a quarter pass (profiles/r3_stream.txt)


def infer_stream(reads, model, threshold=0.5, min_run=15, extension_left=11, extension_right=16, window_size=35,
                 return_scores=False, group_samples=None, max_wait_s=None, depth=_STREAM_DEPTH):
    """Streaming ``infer_reads``: yields ``(intervals, len_read)`` - plus the float32 scores with ``return_scores`` -
    for every read of the iterable ``reads``, in input order, with the results ``infer_reads`` gives for the whole list.

    Reads are pulled lazily and grouped: consecutive reads until the group holds ``group_samples`` samples (default:
    a quarter of an engine pass), or fewer when the input ends or when ``max_wait_s`` seconds have passed since the group's first
    read was taken (checked as each read arrives).  Up to ``depth`` groups run at once, each on its own execution
    context of the model (``cf_exec``), CUDA stream, pinned staging and device buffers, so that small groups overlap
    on the device instead of running one after another.  At most ``depth + 1`` groups of reads are pulled and not
    yet yielded.

    A read that ``infer_reads`` would reject (empty: ``IndexError``; not integer DAC values: ``ValueError``), or an
    exception raised by ``reads`` itself, ends the stream the way the reference's one-file-at-a-time loop meets it:
    every earlier read's result is yielded first, then the exception is raised.  The stream owns all of its buffers
    and contexts and releases them when it is exhausted, closed or collected; streams on one model are independent
    of each other and of ``infer_reads``."""
    if window_size != model.window:
        raise ValueError("window_size must equal the model's window (%d)" % model.window)
    depth = int(depth)
    if depth < 1:
        raise ValueError("depth must be at least 1")
    group_samples = _STREAM_GROUP_SAMPLES if group_samples is None else int(group_samples)
    if group_samples < 1:
        raise ValueError("group_samples must be at least 1")
    params = (float(threshold), int(min_run), int(extension_left), int(extension_right))
    return _stream(iter(reads), model, params, bool(return_scores), group_samples, max_wait_s, depth)


class _Slot(object):
    """Runs one group of reads at a time: a CUDA stream, an event, pinned / device buffers that grow to the largest
    group the slot has run, and the execution context the group runs on - a context of its own (``cf_exec_create``)
    or the model's default context.  Slots on the default context still have a stream each, so that a retired
    group's copies back do not queue behind the next group's kernels; the library orders calls on one context
    across streams."""

    def __init__(self, torch, lib, model, own_context):
        self.torch, self.lib, self.dev = torch, lib, int(model.device)
        self.ex = None
        if own_context:
            ex = ctypes.c_void_p()
            _cabi.check(lib.cf_exec_create(model.handle, ctypes.byref(ex)))
            self.ex = ex
        # cf_exec_infer_reads is cf_infer_reads on a context: the two calls differ only in their first argument
        self.target = self.ex if own_context else model.handle
        self.infer = lib.cf_exec_infer_reads if own_context else lib.cf_infer_reads
        with torch.cuda.device(self.dev):
            self.stream = torch.cuda.Stream()
            self.event = torch.cuda.Event()
        self.buf = {}
        self.group = None

    def _ensure(self, name, n, dtype, pinned=False):
        t = self.buf.get(name)
        if t is None or t.numel() < n:
            n = max(n + n // 4, 1024)
            self.buf[name] = None
            t = self.torch.empty(n, dtype=dtype, pin_memory=pinned) if pinned else \
                self.torch.empty(n, dtype=dtype, device="cuda:%d" % self.dev)
            self.buf[name] = t
        return t

    def submit(self, arrays, params, return_scores, labels=None, thresholds=None, dest=None):
        """Stage, copy and enqueue one group on this slot's stream (returns without waiting for the device).  With
        ``labels`` (one uint8 array per read) the group is counted at ``thresholds`` instead of returning intervals,
        or, with ``dest = (probs, labels, offset)``, its probabilities and labels go to those device tensors at
        ``offset`` and nothing comes back."""
        torch = self.torch
        threshold, min_run, ext_left, ext_right = params
        n = len(arrays)
        offsets = np.zeros(n + 1, np.int64)
        np.cumsum([a.size for a in arrays], out=offsets[1:])
        total = int(offsets[-1])
        cap = 0 if labels is not None else int(self.lib.cf_max_intervals(total, n, min_run))
        with torch.cuda.device(self.dev), torch.cuda.stream(self.stream):
            stage = self._ensure("stage", total, torch.int16, pinned=True)
            raw = self._ensure("raw", total, torch.int16)
            # the intervals [cap, 2], then the n + 1 interval offsets: one copy brings both back
            m = 2 * cap + n + 1
            out = self._ensure("out", m, torch.int64)
            if dest is not None:
                probs, lab_dev = dest[0][dest[2]:dest[2] + total], dest[1][dest[2]:dest[2] + total]
            elif return_scores or labels is not None:
                probs = self._ensure("probs", total, torch.float32)
                lab_dev = self._ensure("lab", total, torch.uint8) if labels is not None else None
            else:
                probs = None
            _concat_into(stage.numpy()[:total], arrays, offsets)
            raw[:total].copy_(stage[:total], non_blocking=True)
            if labels is not None:
                lab_pin = self._ensure("lab_pin", total, torch.uint8, pinned=True)
                np.concatenate(labels, out=lab_pin.numpy()[:total])
                lab_dev[:total].copy_(lab_pin[:total], non_blocking=True)
            _cabi.check(self.infer(
                self.target, raw.data_ptr(), _offsets_ptr(offsets), n, probs.data_ptr() if probs is not None else None,
                out.data_ptr(), out.data_ptr() + 16 * cap, cap, threshold, min_run, ext_left, ext_right,
                self.stream.cuda_stream))
            self._ensure("out_pin", m, torch.int64, pinned=True)[:m].copy_(out[:m], non_blocking=True)
            if return_scores:
                probs_pin = self._ensure("probs_pin", total, torch.float32, pinned=True)
                probs_pin[:total].copy_(probs[:total], non_blocking=True)
            self.event.record(self.stream)
        self.group = (offsets, cap, return_scores, thresholds if labels is not None else None, dest is not None)

    def done(self):
        return self.event.query()

    def results(self):
        """Wait for the group and return ``(offsets, intervals, interval_offsets, scores or None)`` of its reads - or,
        for a group submitted with labels, its int64 ``[T, 4]`` confusion counts (None with ``dest``).  The slot is
        then free."""
        offsets, cap, return_scores, thresholds, to_dest = self.group
        self.group = None
        n, total = len(offsets) - 1, int(offsets[-1])
        if to_dest:
            self.event.synchronize()
            return None
        if thresholds is not None:
            counts = np.zeros((thresholds.size, 4), np.int64)
            # queued behind the group on the slot's stream; synchronises
            _cabi.check(self.lib.cf_sweep_thresholds(
                self.dev, self.buf["probs"].data_ptr(), 0, self.buf["lab"].data_ptr(), total, thresholds.ctypes.data,
                thresholds.size, counts.ctypes.data_as(_cabi.c_i64_p), self.stream.cuda_stream))
            return counts
        self.event.synchronize()
        out = self.buf["out_pin"].numpy()
        ioff = out[2 * cap:2 * cap + n + 1].copy()
        found = int(ioff[-1])
        if found > cap:
            raise _cabi.CatfishError("interval capacity exceeded (%d > %d)" % (found, cap))
        intervals = out[:2 * found].reshape(found, 2).copy()
        scores = self.buf["probs_pin"].numpy()[:total].copy() if return_scores else None
        return offsets, intervals, ioff, scores

    def close(self):
        self.stream.synchronize()               # copies enqueued after the context's own work
        if self.ex is not None:
            self.lib.cf_exec_destroy(self.ex)
            self.ex = None
        self.buf.clear()


def _in_order(groups, depth, take_slot):
    """Runs every group of the iterable ``groups`` (each the arguments of ``_Slot.submit``) and yields the groups'
    ``results`` in input order.  Up to ``depth`` groups are in flight, on slots from ``take_slot()`` that are reused
    once retired: while the device works on one group, the host stages the next.  A finished group goes out as soon
    as it is found; a ``None`` in ``groups`` submits nothing and only gives that chance.  Groups still in flight when
    the caller stops early are waited for, so that their slots can be reused or freed."""
    idle, inflight = [], collections.deque()

    def retire():
        s = inflight.popleft()
        out = s.results()
        idle.append(s)
        return out

    try:
        for group in groups:
            while inflight and inflight[0].done():
                yield retire()
            if group is None:
                continue
            if len(inflight) == depth:                       # bounded read-ahead: the oldest group goes out first
                yield retire()
            s = idle.pop() if idle else take_slot()
            inflight.append(s)                               # first: a failed submit may have enqueued copies
            s.submit(*group)
        while inflight:
            yield retire()
    finally:
        for s in inflight:
            s.stream.synchronize()


def _run_on_model(model, groups):
    """The list of ``_in_order`` results of ``groups`` on default-context slots of the model's pool, ``_DEPTH`` in
    flight.  The call takes the slots it needs from the pool (new ones when it is short) and puts them back when it
    ends, so that concurrent calls never share a buffer and the next call finds its buffers warm."""
    torch, lib = _torch(), _cabi.load_library()
    taken = []

    def take_slot():
        with model._slot_lock:
            s = model._slots.pop() if model._slots else None
        taken.append(s if s is not None else _Slot(torch, lib, model, own_context=False))
        return taken[-1]

    try:
        return list(_in_order(groups, _DEPTH, take_slot))
    finally:
        with model._slot_lock:
            model._slots.extend(taken)


def _stream(it, model, params, return_scores, group_samples, max_wait_s, depth):
    torch, lib = _torch(), _cabi.load_library()
    slots, error = [], []

    def take_slot():
        slots.append(_Slot(torch, lib, model, own_context=True))
        return slots[-1]

    def groups():
        group, n_samples, t_first = [], 0, 0.0
        while True:
            yield None                                         # finished groups go out as soon as they are found
            try:
                a = _as_int16(next(it))
                if a.size == 0:
                    raise IndexError("list index out of range")  # infer.py:184 on an empty read
            except StopIteration:
                break
            except Exception as e:                             # earlier reads' results first, then this
                error.append(e)
                break
            if not group:
                t_first = time.monotonic()
            group.append(a)
            n_samples += a.size
            if n_samples >= group_samples or (max_wait_s is not None and time.monotonic() - t_first >= max_wait_s):
                yield group, params, return_scores
                group, n_samples = [], 0
        if group:
            yield group, params, return_scores

    try:
        for offsets, intervals, ioff, scores in _in_order(groups(), depth, take_slot):
            bounds, lengths = ioff.tolist(), np.diff(offsets).tolist()
            for r in range(len(lengths)):
                hps = IntervalList(intervals[bounds[r]:bounds[r + 1]])
                yield (hps, lengths[r]) if scores is None else (hps, lengths[r], scores[offsets[r]:offsets[r + 1]])
    finally:
        for s in slots:
            s.close()
    if error:
        raise error[0]


def infer_concatenated(raw, offsets, model, threshold=0.5, min_run=15, extension_left=11,
                       extension_right=16, return_scores=False):
    """The C-ABI call of ``infer_reads`` on an already concatenated int16 signal.

    Returns ``(intervals int64 [n,2], interval_offsets int64 [R+1][, scores float32])``."""
    torch = _torch()
    lib = _cabi.load_library()
    raw = np.ascontiguousarray(raw, dtype=np.int16)
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    n_reads = len(offsets) - 1
    total = int(offsets[-1] - offsets[0]) if n_reads > 0 else 0
    cap = int(lib.cf_max_intervals(total, n_reads, min_run))
    intervals = np.empty((cap, 2), np.int64)
    ioff = np.zeros(n_reads + 1, np.int64)
    scores = np.empty(total, np.float32) if return_scores else None
    found = ctypes.c_int64(0)
    with torch.cuda.device(model.device):
        stream = torch.cuda.current_stream()
        _cabi.check(lib.cf_infer_reads_host(
            model.handle, raw.ctypes.data, _offsets_ptr(offsets), n_reads,
            scores.ctypes.data if scores is not None else None,
            intervals.ctypes.data, ioff.ctypes.data, cap, float(threshold), int(min_run),
            int(extension_left), int(extension_right), ctypes.byref(found), stream.cuda_stream))
    intervals = intervals[:found.value]
    if return_scores:
        return intervals, ioff, scores
    return intervals, ioff


# ------------------------------------------------------------------------------ raw signal
def _trimmed_raw(fast5_file):
    """infer.py:87-90: drop the samples before ``first_sample_template``."""
    first_sample = fast5_file["Analyses/Segmentation_000/Summary/segmentation"].attrs["first_sample_template"]
    read_name = fast5_file["Raw/Reads/"].visit(str)
    raw_signal = fast5_file["Raw/Reads/" + read_name + "/Signal"][()]
    return raw_signal[first_sample:]


def process_signal(fast5_file, normalization="median"):
    """infer.py:77-93: trimmed, normalised raw signal (float64) of an open FAST5."""
    return normalize_raw_signal(_trimmed_raw(fast5_file), normalization)


def _as_int16(raw):
    a = np.asarray(raw)
    if a.dtype == np.int16:
        return np.ascontiguousarray(a.reshape(-1))
    if a.dtype.kind in "iu" or (a.dtype.kind == "f" and np.all(a == np.rint(a))):
        if a.size and (a.min() < -32768 or a.max() > 32767):
            raise ValueError("raw signal outside the int16 DAC range")
        return np.ascontiguousarray(a.reshape(-1).astype(np.int16))
    raise ValueError("raw signal must hold integer DAC values (int16)")


def normalize_raw_signal(raw, norm_method):
    """infer.py:96-105: (raw - median) / median(|raw - median|), float64, bit-exact."""
    if norm_method != 'median':
        raise ValueError('norm_method not recognized')
    torch = _torch()
    a = _as_int16(raw)
    if a.size == 0:
        return np.zeros(0, np.float64)            # numpy: nan statistics, empty result
    dev = _device_index()
    offsets = np.array([0, a.size], np.int64)
    with torch.cuda.device(dev):
        rd = torch.from_numpy(a).to("cuda:%d" % dev)
        out = torch.empty(a.size, dtype=torch.float64, device=rd.device)
        _cabi.check(_cabi.load_library().cf_normalize_reads(
            dev, rd.data_ptr(), _offsets_ptr(offsets), 1, None, out.data_ptr(),
            torch.cuda.current_stream().cuda_stream))
        return out.cpu().numpy()


def read_stats(raws, device=None):
    """(shift, scale) = (median, MAD) of every read, float64 [R, 2]."""
    torch = _torch()
    arrays = [_as_int16(r) for r in raws]
    offsets = np.zeros(len(arrays) + 1, np.int64)
    if arrays:
        offsets[1:] = np.cumsum([a.size for a in arrays])
    raw = np.concatenate(arrays) if arrays else np.zeros(0, np.int16)
    dev = _device_index(device)
    with torch.cuda.device(dev):
        rd = torch.from_numpy(raw).to("cuda:%d" % dev)
        st = torch.empty((len(arrays), 2), dtype=torch.float64, device=rd.device)
        _cabi.check(_cabi.load_library().cf_normalize_reads(
            dev, rd.data_ptr(), _offsets_ptr(offsets), len(arrays), st.data_ptr(), None,
            torch.cuda.current_stream().cuda_stream))
        return st.cpu().numpy()


def reshape_input(data, window, n_inputs):
    """infer.py:108-124 (a reshape; no arithmetic)."""
    try:
        data = np.reshape(data, (-1, window, n_inputs))
    except ValueError:
        print(len(data))
        print(len(data[0]))
    return data


# ------------------------------------------------------------------------------ classified output
def class_from_threshold(predicted_scores, threshold=0.5):
    """infer.py:128-138: list of 0/1 labels."""
    torch = _torch()
    s = np.ascontiguousarray(np.asarray(predicted_scores, dtype=np.float64).reshape(-1))
    if s.size == 0:
        return []
    dev = _device_index()
    with torch.cuda.device(dev):
        sd = torch.from_numpy(s).to("cuda:%d" % dev)
        out = torch.empty(s.size, dtype=torch.int64, device=sd.device)
        _cabi.check(_cabi.load_library().cf_class_from_threshold(
            dev, sd.data_ptr(), s.size, float(threshold), out.data_ptr(),
            torch.cuda.current_stream().cuda_stream))
        return out.cpu().numpy().tolist()


def hp_in_pred(predictions, extension_left=11, extension_right=16, label=1):
    """infer.py:141-162: [[start - ext_left, start + len + ext_right], ...] of every run of ``label``."""
    torch = _torch()
    p = np.ascontiguousarray(np.asarray(predictions, dtype=np.int64).reshape(-1))
    if p.size == 0:
        raise IndexError("list index out of range")            # predictions[0], infer.py:151
    dev = _device_index()
    cap = p.size // 2 + 1
    with torch.cuda.device(dev):
        pd = torch.from_numpy(p).to("cuda:%d" % dev)
        out = torch.empty((cap, 2), dtype=torch.int64, device=pd.device)
        n_out = torch.zeros(1, dtype=torch.int64, device=pd.device)
        _cabi.check(_cabi.load_library().cf_hp_in_pred(
            dev, pd.data_ptr(), p.size, int(extension_left), int(extension_right), int(label),
            out.data_ptr(), cap, n_out.data_ptr(), torch.cuda.current_stream().cuda_stream))
        n = int(n_out.item())
        return out[:n].cpu().numpy().tolist()


def correct_short(predictions, threshold=15):
    """infer.py:174-198: runs of a non-zero label shorter than ``threshold`` become 0."""
    torch = _torch()
    p = np.ascontiguousarray(np.asarray(predictions, dtype=np.int64).reshape(-1))
    if p.size == 0:
        raise IndexError("list index out of range")            # predictions[0], infer.py:184
    dev = _device_index()
    with torch.cuda.device(dev):
        pd = torch.from_numpy(p).to("cuda:%d" % dev)
        out = torch.empty_like(pd)
        _cabi.check(_cabi.load_library().cf_correct_short(
            dev, pd.data_ptr(), p.size, int(threshold), out.data_ptr(),
            torch.cuda.current_stream().cuda_stream))
        return out.cpu().numpy()
