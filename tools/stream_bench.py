"""Streaming inference (infer.infer_stream) against one batched infer_reads call on the same reads.

    python tools/stream_bench.py [--reps 3] [--out FILE]

Two workloads of seeded synthetic reads (catfish_b200.synth): A = 4 000 reads of 10 000 samples (BASELINE
configs[0]'s read length), B = 512 reads of U{50 000..200 000} samples (the bench batch).  On each, with the shipped
ResNetRNN: infer_reads on the whole list (the batched yardstick), infer_stream at its default settings and at depth
1 / 2 / 3 x two group sizes, each as host wall clock from the first read handed over to the last result in hand,
closed by a device synchronise.  Both sides do the same work inside the clock: infer_reads returns its per-read
lists, the stream's results are collected into a list; every stream run's output is checked equal to infer_reads'
after the clock stops.  Every configuration is warmed up once, then the configurations run in alternation,
`--reps` rounds, and the median is reported.

A stream creates its execution contexts and they allocate their workspaces on their first group, whereas
infer_reads runs on the model's warm default context.  Two lines split that cost out: "default, warm contexts" runs
the same infer_stream code on contexts kept from the previous run (the measurement substitutes them for the ones
the stream would create), and "context set-up" times cf_exec_create + cf_exec_reserve for one default-size group +
cf_exec_destroy of one context.  Then: the per-read loop infer_class_from_raw on the first 200 reads of A (us per
call), and the time from the start of a stream to its first yielded result, with and without max_wait_s = 0.  The
card's name and power limit are read in the same run and printed first."""
import ctypes
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        return out or "nvidia-smi gave no output"
    except (OSError, subprocess.TimeoutExpired):
        return "nvidia-smi unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from catfish_b200 import _cabi, infer, neural_network, synth
    if not torch.cuda.is_available():
        sys.exit("stream_bench: no CUDA device")
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: %s" % card())
    model = neural_network.load_network("ResNetRNN", None, 30000)
    emit("model: shipped ResNetRNN, engine %s, operand format %s; default group_samples %d, depth %d"
         % (model.resolved_engine, model.operand_format, infer._STREAM_GROUP_SAMPLES, infer._STREAM_DEPTH))
    workloads = [
        ("A: 4000 x 10 000 samples", synth.synth_reads([10_000] * 4000, base_seed=0)),
        ("B: 512 x U{50k..200k} samples", synth.synth_reads(synth.ragged_lengths(512, 50_000, 200_000, seed=1), base_seed=1)),
    ]
    groups = (infer._GROUP_SAMPLES // 4, infer._GROUP_SAMPLES)
    make_slot = infer._Slot
    lib = _cabi.load_library()
    for name, reads in workloads:
        samples = sum(r.size for r in reads)
        want_hps, want_len = infer.infer_reads(reads, model)

        def batched():
            infer.infer_reads(reads, model)
            torch.cuda.synchronize()

        outputs = []                                                # stream outputs, checked outside the clock

        def streamed(**kw):
            def run():
                outputs.append(list(infer.infer_stream(iter(reads), model, **kw)))
                torch.cuda.synchronize()
            return run

        kept = []                                                   # contexts of the warm-context runs

        def warm_streamed():
            pool = []

            def slot(*a, **kw):
                if pool:
                    return pool.pop()
                s = make_slot(*a, **kw)
                s.destroy, s.close = s.close, (lambda: None)         # kept alive across runs
                kept.append(s)
                return s

            def run():
                pool[:] = kept
                infer._Slot = slot
                try:
                    outputs.append(list(infer.infer_stream(iter(reads), model)))
                    torch.cuda.synchronize()
                finally:
                    infer._Slot = make_slot
            return run

        configs = [("infer_reads (whole list)", batched), ("infer_stream default", streamed()),
                   ("infer_stream default, warm contexts", warm_streamed())]
        for depth in (1, 2, 3):
            for g in groups:
                configs.append(("infer_stream depth %d, group %.1fM" % (depth, g / 1e6), streamed(depth=depth, group_samples=g)))
        times = {label: [] for label, _ in configs}
        for label, fn in configs:
            fn()                                                    # warm-up: workspaces, pinned staging
        for _ in range(args.reps):
            for label, fn in configs:
                t0 = time.perf_counter()
                fn()
                times[label].append(time.perf_counter() - t0)
        for got in outputs:
            assert len(got) == len(reads)
            for (h, n), wh, wn in zip(got, want_hps, want_len):
                assert n == wn and np.array_equal(h.array, wh.array), "stream output differs from infer_reads"
        for s in kept:
            s.destroy()
        del outputs[:], kept[:]
        emit("")
        emit("workload %s: %d reads, %.3g samples; median of %d alternating runs" % (name, len(reads), samples, args.reps))
        base = float(np.median(times[configs[0][0]]))
        for label, _ in configs:
            t = float(np.median(times[label]))
            emit("  %-38s %8.2f ms  %7.1f M samples/s  %.3f x infer_reads   (runs: %s ms)"
                 % (label, 1e3 * t, samples / t / 1e6, base / t, ", ".join("%.1f" % (1e3 * x) for x in times[label])))
        setup = []
        for _ in range(args.reps + 1):
            ex = ctypes.c_void_p()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _cabi.check(lib.cf_exec_create(model.handle, ctypes.byref(ex)))
            _cabi.check(lib.cf_exec_reserve(ex, infer._STREAM_GROUP_SAMPLES + max(r.size for r in reads), 2048))
            lib.cf_exec_destroy(ex)
            setup.append(time.perf_counter() - t0)
        emit("  context set-up (create + reserve one default group + destroy): %.2f ms (median of %d after one warm-up)"
             % (1e3 * float(np.median(setup[1:])), args.reps))
        for kw, what in (({}, "default settings"), ({"max_wait_s": 0}, "max_wait_s = 0")):
            firsts = []
            for _ in range(args.reps + 1):
                t0 = time.perf_counter()
                stream = infer.infer_stream(iter(reads), model, **kw)
                first = next(stream)
                firsts.append(time.perf_counter() - t0)
                stream.close()
                assert first[1] == want_len[0] and np.array_equal(first[0].array, want_hps[0].array)
            emit("  first result, %-22s %8.2f ms (median of %d after one warm-up)" % (what, 1e3 * float(np.median(firsts[1:])), args.reps))
        if name.startswith("A"):
            per = []
            for r in reads[:200]:
                t0 = time.perf_counter()
                infer.infer_class_from_raw(r, model)
                per.append(time.perf_counter() - t0)
            t = float(np.median(per[10:]))
            emit("  infer_class_from_raw loop, first 200 reads: median %.0f us per call (%.2f M samples/s)"
                 % (1e6 * t, reads[0].size / t / 1e6))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
