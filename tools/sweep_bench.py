"""Threshold sweeps (K11) on the GPU: the kernel alone, and evaluate_reads against infer_reads with scores.

    python tools/sweep_bench.py [--reps 5] [--out FILE]

1. K11 (`cf_sweep_thresholds`) over 6.4e7 device-resident positions (float32 probabilities: 87 % drawn near 0, 13 %
   near 1, as the shipped model's scores on synthetic reads; uint8 labels) at T = 1, 101 and 4096 thresholds.  Per T:
   the kernels' device time from torch.profiler (count kernel + counts scan, summed over `--reps` calls), the whole
   call between CUDA events (threshold upload, histogram reset, both kernels, count copy), and the count kernel's
   bandwidth at 5 B per position as a fraction of the HBM peak bench.py quotes (MEASURED_PEAKS.json, else its
   fallback).  The 320 MB input exceeds the 126 MB L2, so every call reads it from HBM.
2. On the bench batch (512 reads of U{50 000..200 000} samples, bench.py's first batch), with the shipped ResNetRNN:
   `infer.evaluate_reads` at 101 thresholds against `infer.infer_reads(..., return_scores=True)` followed by nothing
   (the host would still have to count), host wall clock to the result in hand, alternating, median of `--reps`.
   evaluate_reads' counts are checked against numpy counting of infer_reads' scores after the clock stops.
The card's name and power limit are read in the same run and printed first."""
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    from catfish_b200 import _cabi, infer, metrics, neural_network, synth
    if not torch.cuda.is_available():
        sys.exit("sweep_bench: no CUDA device")
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: %s" % card())
    peaks = bench.load_peaks()
    emit("HBM peak used for fractions: %.0f GB/s (%s)" % (peaks["hbm"], peaks["source"]))
    lib = _cabi.load_library()
    dev = torch.cuda.current_device()
    stream = torch.cuda.current_stream()

    # ---------------------------------------------------------------- 1. the kernel
    n = 64_000_000
    rng = np.random.default_rng(0)
    high = rng.random(n) < 0.13
    p = np.where(high, 1.0 - rng.beta(0.5, 8.0, n), rng.beta(0.5, 8.0, n)).astype(np.float32)
    y = (rng.random(n) < np.where(high, 0.9, 0.05)).astype(np.uint8)
    pd, yd = torch.from_numpy(p).cuda(), torch.from_numpy(y).cuda()
    emit("")
    emit("K11 over %.3g positions (%.0f MB read per call); %d calls per T after one warm-up" % (n, 5 * n / 1e6, args.reps))
    for T in (1, 101, 4096):
        th = np.ascontiguousarray(np.linspace(0.0, 1.0, T) if T > 1 else [0.5], dtype=np.float64)
        counts = np.zeros((T, 4), np.int64)

        def call():
            _cabi.check(lib.cf_sweep_thresholds(dev, pd.data_ptr(), 0, yd.data_ptr(), n, th.ctypes.data, T,
                                                counts.ctypes.data_as(_cabi.c_i64_p), stream.cuda_stream))

        call()
        if T == 101:
            assert np.array_equal(counts[[0, 50, 100]], np.array(
                [metrics.confusion_matrix(y, (p.astype(np.float64) >= t).astype(np.int64)) for t in th[[0, 50, 100]]]))
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.reps)]
        for r in range(args.reps):
            ev[2 * r].record()
            call()
            ev[2 * r + 1].record()
        torch.cuda.synchronize()
        call_ms = float(np.median([ev[2 * r].elapsed_time(ev[2 * r + 1]) for r in range(args.reps)]))
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.reps):
                call()
            torch.cuda.synchronize()
        k = {"count": 0.0, "scan": 0.0}
        for e in prof.key_averages():
            if "k11_count_kernel" in e.key:
                k["count"] += e.device_time_total / 1e3
            elif "k11_counts_kernel" in e.key:
                k["scan"] += e.device_time_total / 1e3
        count_ms, scan_ms = k["count"] / args.reps, k["scan"] / args.reps
        gbs = 5 * n / (count_ms * 1e-3) / 1e9 if count_ms else float("nan")
        emit("  T = %4d: count kernel %.3f ms (%.0f GB/s = %.2f of HBM peak), counts scan %.3f ms, whole call %.3f ms"
             % (T, count_ms, gbs, gbs / peaks["hbm"], scan_ms, call_ms))
    del pd, yd

    # ---------------------------------------------------------------- 2. read level
    model = neural_network.load_network("ResNetRNN", None, 30000)
    lengths = synth.ragged_lengths(512, bench.LEN_LO, bench.LEN_HI, seed=1000)
    reads = synth.synth_reads(lengths, base_seed=1000 * 1_000_003)
    lrng = np.random.default_rng(5)
    labels = [(lrng.random(r.size) < 0.13).astype(np.uint8) for r in reads]
    samples = int(lengths.sum())
    th = np.linspace(0.0, 1.0, 101)
    out = {}

    def with_scores():
        out["scores"] = infer.infer_reads(reads, model, return_scores=True)[2]
        torch.cuda.synchronize()

    def evaluated():
        out["counts"] = infer.evaluate_reads(reads, labels, model, th)

    configs = [("infer_reads(return_scores=True)", with_scores), ("evaluate_reads, 101 thresholds", evaluated)]
    times = {name: [] for name, _ in configs}
    for _, fn in configs:
        fn()
    for _ in range(args.reps):
        for name, fn in configs:
            t0 = time.perf_counter()
            fn()
            times[name].append(time.perf_counter() - t0)
    s = np.concatenate(out["scores"]).astype(np.float64)
    yl = np.concatenate(labels)
    sel = [0, 25, 50, 75, 100]
    want = np.array([metrics.confusion_matrix(yl, (s >= th[i]).astype(np.int64)) for i in sel])
    assert np.array_equal(out["counts"][sel], want), "evaluate_reads differs from counting infer_reads' scores"
    emit("")
    emit("bench batch: %d reads, %.4g samples; shipped ResNetRNN, engine %s; median of %d alternating runs"
         % (len(reads), samples, model.resolved_engine, args.reps))
    base = float(np.median(times[configs[0][0]]))
    for name, _ in configs:
        t = float(np.median(times[name]))
        emit("  %-34s %8.2f ms  %7.1f M samples/s  %.3f x the time of infer_reads with scores   (runs: %s ms)"
             % (name, 1e3 * t, samples / t / 1e6, t / base, ", ".join("%.1f" % (1e3 * x) for x in times[name])))
    emit("  probabilities copied to the host: %.0f MB by infer_reads with scores, 0 by evaluate_reads"
         % (4 * samples / 1e6))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
