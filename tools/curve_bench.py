"""Exact score curves (K13) on the GPU: the sort + count alone, evaluate_reads_curve against evaluate_reads, and the
host route they replace.

    python tools/curve_bench.py [--reps 5] [--out FILE]

1. `metrics.score_curve(..., points=False)` over 6.4e7 device-resident positions (float32 probabilities: 87 % drawn
   near 0, 13 % near 1, as the shipped model's scores on synthetic reads - the data of tools/sweep_bench.py; uint8
   labels).  The kernels' device time from torch.profiler (per kernel, summed over `--reps` calls), the whole call
   between CUDA events, and the bytes the passes move (pack: 5 B read + 4 B written per position; each of the four
   scatter passes 4 B read + 4 B written; the run count and emit each read the 4 B keys) against the HBM figure
   bench.py quotes (MEASURED_PEAKS.json, else its fallback).  The 320 MB input exceeds the 126 MB L2.
2. The host route on the same data: the probabilities and labels copied to the host, then the numpy oracle of
   tests/curve_oracle.py (stable argsort, run ends, cumulative counts, areas); one run, timed by the host clock.
3. On the bench batch (512 reads of U{50 000..200 000} samples, bench.py's first batch), with the shipped ResNetRNN:
   `infer.evaluate_reads_curve(points=False)` against `infer.evaluate_reads` at 101 thresholds, host wall clock to the
   result in hand, alternating, median of `--reps`.
The card's name and power limit are read in the same run and printed first."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile
    import bench
    import curve_oracle
    from sweep_bench import card
    from catfish_b200 import infer, metrics, neural_network, synth
    if not torch.cuda.is_available():
        sys.exit("curve_bench: no CUDA device")
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)

    emit("card: %s" % card())
    peaks = bench.load_peaks()
    emit("HBM peak used for fractions: %.0f GB/s (%s)" % (peaks["hbm"], peaks["source"]))

    # ---------------------------------------------------------------- 1. the device call
    n = 64_000_000
    rng = np.random.default_rng(0)
    high = rng.random(n) < 0.13
    p = np.where(high, 1.0 - rng.beta(0.5, 8.0, n), rng.beta(0.5, 8.0, n)).astype(np.float32)
    y = (rng.random(n) < np.where(high, 0.9, 0.05)).astype(np.uint8)
    pd, yd = torch.from_numpy(p).cuda(), torch.from_numpy(y).cuda()
    first = metrics.score_curve(pd, yd, points=False)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.reps)]
    for r in range(args.reps):
        ev[2 * r].record()
        c = metrics.score_curve(pd, yd, points=False)
        ev[2 * r + 1].record()
        assert (c.roc_auc, c.average_precision) == (first.roc_auc, first.average_precision)
    torch.cuda.synchronize()
    call_ms = float(np.median([ev[2 * r].elapsed_time(ev[2 * r + 1]) for r in range(args.reps)]))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            metrics.score_curve(pd, yd, points=False)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if "k13_" in e.key:
            name = e.key.split("(")[0].replace("void ", "").replace("cf::", "")
            per[name] = per.get(name, 0.0) + e.device_time_total / 1e3 / args.reps
    kernel_ms = sum(per.values())
    moved = n * (5 + 4) + 4 * n * 8 + 2 * n * 4
    emit("")
    emit("score_curve(points=False) over %.3g positions; median of %d calls after one warm-up" % (n, args.reps))
    for name, ms in sorted(per.items(), key=lambda kv: -kv[1]):
        emit("  %-40s %.3f ms" % (name, ms))
    emit("  all K13 kernels %.3f ms: %.2f GB moved, %.0f GB/s = %.2f of the HBM peak; whole call %.3f ms"
         % (kernel_ms, moved / 1e9, moved / (kernel_ms * 1e-3) / 1e9, moved / (kernel_ms * 1e-3) / 1e9 / peaks["hbm"],
            call_ms))
    emit("  roc_auc %.12f, average_precision %.12f" % (first.roc_auc, first.average_precision))

    # ---------------------------------------------------------------- 2. the host route
    t0 = time.perf_counter()
    ph, yh = pd.cpu().numpy(), yd.cpu().numpy()
    t1 = time.perf_counter()
    _, counts, auc, ap_ = curve_oracle.curve(ph, yh)
    t2 = time.perf_counter()
    assert abs(auc - first.roc_auc) <= 1e-12 * auc and abs(ap_ - first.average_precision) <= 1e-12 * ap_
    host_ms = 1e3 * (t2 - t0)
    emit("  host route: D2H copy %.1f ms + numpy oracle %.1f ms = %.1f ms, %.0f x the device call (%d rows)"
         % (1e3 * (t1 - t0), 1e3 * (t2 - t1), host_ms, host_ms / call_ms, counts.shape[0]))
    del pd, yd

    # ---------------------------------------------------------------- 3. read level
    model = neural_network.load_network("ResNetRNN", None, 30000)
    lengths = synth.ragged_lengths(512, bench.LEN_LO, bench.LEN_HI, seed=1000)
    reads = synth.synth_reads(lengths, base_seed=1000 * 1_000_003)
    lrng = np.random.default_rng(5)
    labels = [(lrng.random(r.size) < 0.13).astype(np.uint8) for r in reads]
    samples = int(lengths.sum())
    th = np.linspace(0.0, 1.0, 101)
    out = {}

    def swept():
        out["counts"] = infer.evaluate_reads(reads, labels, model, th)

    def curved():
        out["curve"] = infer.evaluate_reads_curve(reads, labels, model, points=False)

    configs = [("evaluate_reads, 101 thresholds", swept), ("evaluate_reads_curve(points=False)", curved)]
    times = {name: [] for name, _ in configs}
    for _, fn in configs:
        fn()
    for _ in range(args.reps):
        for name, fn in configs:
            t0 = time.perf_counter()
            fn()
            times[name].append(time.perf_counter() - t0)
    emit("")
    emit("bench batch: %d reads, %.4g samples; shipped ResNetRNN, engine %s; median of %d alternating runs"
         % (len(reads), samples, model.resolved_engine, args.reps))
    base = float(np.median(times[configs[0][0]]))
    for name, _ in configs:
        t = float(np.median(times[name]))
        emit("  %-36s %8.2f ms  %7.1f M samples/s  %.3f x the time of evaluate_reads   (runs: %s ms)"
             % (name, 1e3 * t, samples / t / 1e6, t / base, ", ".join("%.1f" % (1e3 * x) for x in times[name])))
    emit("  roc_auc %.6f, average_precision %.6f" % (out["curve"].roc_auc, out["curve"].average_precision))
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
