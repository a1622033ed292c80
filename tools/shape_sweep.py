"""Tensor-core engine vs the fp32 CUDA-core engine on the network shapes the tensor-core engine admits besides
the shipped one (narrower networks, conv stacks of three or more blocks), with the shipped shape as a control.

    python tools/shape_sweep.py [--reads 256] [--reps 3] [--out FILE]

Per shape: one seeded model (non-trivial batch-norm statistics) and one seeded ragged batch of int16 reads resident
on the device (U{60k..180k} samples, about 3.1e7 at 256 reads; with the activations of every layer that is far
beyond L2).  cf_infer_reads is timed with the engine AUTO resolves to and with engine="simt", in the same process,
alternating after one warm-up call of each, each call closed by a device synchronise.  One line per shape:
samples/s of each engine and their ratio, max |dp| between the two engines over the whole batch (probabilities
from one further call of each), and ms per call of the k2_conv_stack kernel class (live CUDA events, separate
call).  The card's name and power limit are read in the same run and printed first."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SHAPES = [  # (label, network type, hyper-parameters)
    ("shipped ResNetRNN C32 H64 x3, 2 blocks", "ResNetRNN", dict(layer_size_res=32, n_layers_res=2, layer_size=64, n_layers=3)),
    ("RNN H8 x2", "RNN", dict(layer_size=8, n_layers=2)),
    ("RNN H16 x3", "RNN", dict(layer_size=16, n_layers=3)),
    ("RNN H32 x2", "RNN", dict(layer_size=32, n_layers=2)),
    ("RNN H48 x3", "RNN", dict(layer_size=48, n_layers=3)),
    ("ResNetRNN C16 H32 x2, 2 blocks", "ResNetRNN", dict(layer_size_res=16, n_layers_res=2, layer_size=32, n_layers=2)),
    ("ResNetRNN C32 H16 x2, 1 block", "ResNetRNN", dict(layer_size_res=32, n_layers_res=1, layer_size=16, n_layers=2)),
    ("ResNetRNN C8 H64 x2, 3 blocks", "ResNetRNN", dict(layer_size_res=8, n_layers_res=3, layer_size=64, n_layers=2)),
    ("ResNetRNN C32 H64 x3, 3 blocks", "ResNetRNN", dict(layer_size_res=32, n_layers_res=3, layer_size=64, n_layers=3)),
    ("ResNetRNN C32 H64 x3, 5 blocks", "ResNetRNN", dict(layer_size_res=32, n_layers_res=5, layer_size=64, n_layers=3)),
    ("ResNetRNN C32 H64 x3, 11 blocks", "ResNetRNN", dict(layer_size_res=32, n_layers_res=11, layer_size=64, n_layers=3)),
    ("ResNet C16, 1 block", "ResNet", dict(layer_size_res=16, n_layers_res=1)),
    ("ResNet C24, 2 blocks", "ResNet", dict(layer_size_res=24, n_layers_res=2)),
    ("ResNet C32, 3 blocks", "ResNet", dict(layer_size_res=32, n_layers_res=3)),
    ("ResNet C32, 4 blocks", "ResNet", dict(layer_size_res=32, n_layers_res=4)),
]


def bn_weights(kind, seed, **hpm):
    from catfish_b200 import weights
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


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=30).stdout.strip()
        return out or "nvidia-smi gave no output"
    except (OSError, subprocess.TimeoutExpired):
        return "nvidia-smi unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from catfish_b200 import _cabi, neural_network, synth, weights
    if not torch.cuda.is_available():
        sys.exit("shape_sweep: no CUDA device")
    lib = _cabi.load_library()
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream

    lengths = synth.ragged_lengths(args.reads, 60_000, 180_000, seed=2026)
    raw, off = synth.concat_reads(synth.synth_reads(lengths, base_seed=2027))
    n = int(off[-1])
    raw_dev = torch.from_numpy(raw).to("cuda")
    cap = int(lib.cf_max_intervals(n, args.reads, 15))
    iv_dev = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    ioff_dev = torch.empty(args.reads + 1, dtype=torch.int64, device="cuda")
    probs = [torch.empty(n, dtype=torch.float32, device="cuda") for _ in range(2)]

    lines = ["card: %s (torch: %s)" % (card(), torch.cuda.get_device_name(0)),
             "batch: %d reads, %d samples, device-resident int16; %d timed calls per engine, alternating" % (args.reads, n, args.reps),
             "%-38s %-8s %12s %12s %8s %10s %10s %10s" % ("shape", "engine", "tc samp/s", "simt samp/s", "ratio", "max|dp|",
                                                         "k2 tc ms", "k2 simt ms")]
    print("\n".join(lines), flush=True)

    def call(m, p=None):
        _cabi.check(lib.cf_infer_reads(m.handle, raw_dev.data_ptr(), off.ctypes.data_as(_cabi.c_i64_p), args.reads,
                                       p.data_ptr() if p is not None else None, iv_dev.data_ptr(), ioff_dev.data_ptr(),
                                       cap, 0.5, 15, 11, 16, sp))

    for i, (label, kind, hpm) in enumerate(SHAPES):
        w = bn_weights(kind, 500 + i, **hpm)
        full = dict(weights.SHIPPED_HPARAMS)
        full.update(hpm)
        models = []
        for engine in ("auto", "simt"):
            m = neural_network.build_model(kind, engine=engine, **full)
            m.set_weights(w)
            _cabi.check(lib.cf_model_reserve(m.handle, n, args.reads))
            models.append(m)
        secs = [[], []]
        for k, m in enumerate(models):                  # warm-up
            call(m)
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for k, m in enumerate(models):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                call(m)
                torch.cuda.synchronize()
                secs[k].append(time.perf_counter() - t0)
        k2 = []
        for k, m in enumerate(models):
            _cabi.profile_enable(m.handle, True)
            call(m, probs[k])
            torch.cuda.synchronize()
            k2.append(_cabi.profile_read(m.handle).get("k2_conv_stack", (0.0, 0))[0])
            _cabi.profile_enable(m.handle, False)
        dp = float((probs[0] - probs[1]).abs().max().item())
        rate = [n / float(np.median(s)) for s in secs]
        line = "%-38s %-8s %12.4g %12.4g %8.1f %10.2e %10.3f %10.3f" % (label, models[0].resolved_engine, rate[0], rate[1],
                                                                       rate[0] / rate[1], dp, k2[0], k2[1])
        print(line, flush=True)
        lines.append(line)
        for m in models:
            m.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
