"""Training step time on the GPU (K12, cf_trainer_step), its per-kernel split, and the torch-CPU fp32 autograd step.

    python tools/train_bench.py [--out profiles/r5_train.txt] [--steps 50]

For each network (shipped ResNetRNN, RNN H = 64 x 3, RNN H = 256 x 5) and batch (256, 4096 windows): the step time
from CUDA events around --steps consecutive steps after warm-up (no host synchronisation inside the timed loop), and
positions / s = batch * 35 / step time.  A separate run under torch.profiler gives each kernel's share of the step's
GPU time.  The CPU line is oracle/train.py's op sequence in torch-CPU float32 (forward, autograd backward and the
RMSProp update) on all host cores - a restatement of the step, not TensorFlow.  The card's name and power limit are
read in the same run.
"""
import argparse
import collections
import ctypes
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

CONFIGS = [
    ("shipped ResNetRNN", "ResNetRNN", dict(layer_size=64, n_layers=3, layer_size_res=32, n_layers_res=2)),
    ("RNN H=64 x 3", "RNN", dict(layer_size=64, n_layers=3)),
    ("RNN H=256 x 5", "RNN", dict(layer_size=256, n_layers=5)),
]
BATCHES = [256, 4096]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make(kind, hpm):
    from catfish_b200 import neural_network, weights
    hp = dict(weights.SHIPPED_HPARAMS)
    hp.update(layer_size=64, n_layers=1, layer_size_res=32, n_layers_res=1)
    hp.update(hpm)
    m = neural_network.build_model(kind, engine="simt", **hp)
    m.initialize_network(seed=1)
    return m


def batch(n, seed=0):
    rng = np.random.default_rng(seed)
    return (rng.normal(0, 1, size=(n, 35, 1)).astype(np.float32),
            (rng.random(n * 35) < 0.4).astype(np.uint8))


def gpu_step_ms(m, n, steps, warmup):
    import torch
    from catfish_b200 import _cabi
    lib = _cabi.load_library()
    x, y = batch(n)
    m.train_network(x, y)                  # creates the trainer, sizes its workspace
    tr = m._trainer
    xd = torch.from_numpy(x.reshape(n, 35)).cuda()
    yd = torch.from_numpy(y).cuda()
    st = torch.cuda.current_stream()

    def step(i):
        _cabi.check(lib.cf_trainer_step(tr, xd.data_ptr(), yd.data_ptr(), n, 1e-3, 0.8, 0, i, None, None,
                                        st.cuda_stream))
    for i in range(warmup):
        step(i)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for i in range(steps):
        step(warmup + i)
    b.record(st)
    b.synchronize()
    return a.elapsed_time(b) / steps, step


def kernel_split(step, steps=5):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            step(10_000 + i)
        torch.cuda.synchronize()
    acc = collections.Counter()
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            name = e.key.split("(")[0].replace("void ", "").replace("cf::", "")
            acc[name] += t
    total = sum(acc.values())
    return [(k, v / total) for k, v in acc.most_common(8)], total / steps / 1e3


def cpu_step_ms(kind, hpm, n, reps=2):
    import torch
    from catfish_b200 import weights
    from oracle import train
    w = weights.random_init(kind, seed=1, **hpm)
    x, y = batch(n)
    g = train.TrainGraph(w, dtype=np.float32)
    ms = {k: torch.ones_like(v) for k, v in g.w.items() if v.requires_grad}
    mom = {k: torch.zeros_like(v) for k, v in ms.items()}
    times = []
    for r in range(reps + 1):
        masks = train.dropout_masks(w, 0, r, n, 0.8)
        t0 = time.perf_counter()
        loss = train.loss_of_logits(g.logits(x, 0.8, masks), y)
        loss.backward()
        with torch.no_grad():
            for k in ms:
                gr = g.w[k].grad
                ms[k] += (gr * gr - ms[k]) * 0.1
                mom[k] = 1e-3 * gr / torch.sqrt(ms[k] + 1e-10)
                g.w[k] -= mom[k]
                g.w[k].grad = None
        times.append(time.perf_counter() - t0)
    return 1e3 * min(times[1:])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_train.txt"))
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    import torch
    lines = ["card: %s (name, power limit, max SM clock)" % card(),
             "torch %s, %d host threads" % (torch.__version__, torch.get_num_threads()), ""]
    lines.append("%-18s %6s %12s %14s %s" % ("network", "batch", "step ms", "positions/s", "kernel split (torch.profiler)"))
    for label, kind, hpm in CONFIGS:
        for n in BATCHES:
            m = make(kind, hpm)
            ms, step = gpu_step_ms(m, n, args.steps, args.warmup)
            split, prof_ms = kernel_split(step)
            lines.append("%-18s %6d %12.3f %14.3e  %s" % (label, n, ms, n * 35 / (ms * 1e-3),
                                                           ", ".join("%s %.0f%%" % (k, 100 * f) for k, f in split)))
            lines.append("%-18s %6s %12s %14s  GPU kernel time per step under the profiler: %.3f ms"
                         % ("", "", "", "", prof_ms))
            m.close()
            print(lines[-2], flush=True)
    if not args.no_cpu:
        lines += ["", "torch-CPU fp32 autograd step (oracle/train.py op sequence, forward + backward + RMSProp), "
                      "batch 256, best of 2:"]
        for label, kind, hpm in CONFIGS:
            ms = cpu_step_ms(kind, hpm, 256)
            lines.append("%-18s %6d %12.1f %14.3e" % (label, 256, ms, 256 * 35 / (ms * 1e-3)))
            print(lines[-1], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
