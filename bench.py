#!/usr/bin/env python3
"""Throughput benchmark of the catfish inference hot path (contract in the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--legs main,probs,python,job,configs,cpu,check]
                    [--dump-outputs DIR]

Workload of the headline line (BASELINE.json configs[3], the configuration the metric is quoted on):
ResNetRNN with the shipped checkpoint over synthetic raw-signal reads of ragged length
U{50 000 .. 200 000} samples, sharded by read.  One "step" is one pass of the whole hot path
(median/MAD normalisation, windowing, conv stack, GRU stack, dense+sigmoid, threshold /
short-run removal / interval emission) over one batch of --reads-per-step reads per GPU; the
100 000-read job of configs[3] is a sequence of such batches.  Every rank works on its own
batch (weak scaling), there is no collective on the data path.

* value : samples/s with the int16 signal already resident in HBM (cf_infer_reads)
* e2e   : samples/s through the host-buffer C-ABI call (cf_infer_reads_host): pinned host
          signal -> device, compute, intervals -> host, inside the timed region
* roofline : the dominant kernel class, timed with CUDA events on the launching stream
          during the timed steps
* cpu_baseline : the oracle's torch-fp32 restatement of the TF graph + the reference's
          post-processing, on all host cores, BASELINE.md section 3 (200 x 10k reads, median of 3)

Further legs, extra keys on the same JSON line:
* e2e_probs  : the same host call with the per-position probabilities returned (what RNN.infer returns,
               rnn_class.py:213-219): + 4 B/sample device->host inside the timed region
* e2e_python : what a user of the Python package calls - infer.infer_reads(list of numpy int16 reads):
               ragged concat into pinned staging, the host call, per-read interval lists (host wall clock)
* job        : the reference's loop over one list of files (catfish/catfish:55-56) as ONE sharded job:
               a fixed seeded list of reads, LPT partition by read, every rank infers its shard, rank 0
               gathers all per-read results - all inside the timed region (strong scaling over --gpus)
* configs    : BASELINE.json configs[0], [1] (RNN-only), [2] (ResNet-only), [4] (1M-sample reads), each with
               samples/s, its dominant kernel class and that kernel's roofline fraction (N = 1 only)
* parity_check : two reads of the timed batch against the CPU oracle, outside the timed region

--impl reference times the CPU restatement (TensorFlow itself is not installable offline; see DESIGN.md)
on bounded samples of the same workload.

--dump-outputs DIR writes what the last timed step of `value` returned to its caller (rank 0's batch, which the
seeds make the same from run to run and for every --gpus) as float64 .npy files, so that two builds can be
compared output for output; see dump_outputs.
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree, which may be read-only

METRIC = "raw_signal_samples_per_sec_resnetrnn_infer"
UNIT = "samples/s"
LEN_LO, LEN_HI = 50_000, 200_000
JOB_READS = 16384
JOB_POOL = 4096
JOB_SEED = 20_000
DUMP_BYTES = 64 << 20

# algorithmic work per real sample (SURVEY.md section 8d / BASELINE.md section 4)
BYTES_PER_SAMPLE = {"k1_stats": 2.0, "k6_intervals": 4.0, "k1_window_table": 0.0}


def flops_per_sample(kind, fused=True):
    """Algorithmic FLOPs per real sample by kernel class for the three network types (shipped sizes)."""
    if kind == "ResNet":
        return {"k2_conv_stack": 20608.0, "k5_head": 64.0}
    if kind == "RNN":
        xproj = 2.0 * 2 * (1 * 192 + 2 * 128 * 192)
        rec = 147456.0
    else:
        xproj, rec = 221184.0, 147456.0
    d = {"k5_head": 256.0}
    if kind != "RNN":
        d["k2_conv_stack"] = 20608.0
    if fused:
        d["k4_gru_recurrence"] = xproj + rec
    else:
        d["k3_gru_input_proj"], d["k4_gru_recurrence"] = xproj, rec
    return d


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads-per-step", type=int, default=512)
    ap.add_argument("--engine", default="auto", choices=["auto", "tcgen05", "simt"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--legs", default=None,
                    help="comma list of main,probs,python,job,configs,cpu,check (default: all at N=1; main,job at N>1)")
    ap.add_argument("--job-reads", type=int, default=JOB_READS)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result of the last timed step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tensor_burst=p["bf16_tflops"], tensor_sustained=p["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source="fallback")


class ClockSampler(object):
    """Samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for ts, r in self.rows if t0 <= ts <= t1] or [r for _, r in self.rows]
        for r in rows:
            parts = [p.strip() for p in r.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        # "under load": samples taken while a kernel was running (power above half of the maximum seen);
        # samples that fall into the host-side gap between steps show the idle clock
        if power:
            thr = 0.5 * max(power)
            loaded = [c for c, p in zip(sm, power) if p >= thr] or sm
        else:
            loaded = sm
        return {"sm_mhz": float(np.median(loaded)) if loaded else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_under_load": len(loaded),
                "power_w_max": max(power) if power else None}


def make_batch(n_reads, seed):
    from catfish_b200 import synth
    lengths = synth.ragged_lengths(n_reads, LEN_LO, LEN_HI, seed=seed)
    reads = synth.synth_reads(lengths, base_seed=seed * 1_000_003)
    return synth.concat_reads(reads)


def dump_outputs(out_dir, iv, ioff):
    """Write one cf_infer_reads result (intervals int64 [n, 2], CSR offsets int64 [reads + 1]) as float64, which
    holds these integers exactly: intervals.npy [n, 2], interval_offsets.npy [reads + 1] and read_ids.npy [reads],
    the batch index of each read written.  A result above DUMP_BYTES is cut to a fixed seeded sample of whole reads."""
    counts = np.diff(ioff)
    order = np.random.default_rng(0).permutation(len(counts))
    fits = np.cumsum(16 * counts[order] + 16) <= DUMP_BYTES - 4096           # 16 B per interval, 16 B per read
    reads = np.sort(order[:int(np.count_nonzero(fits))])
    rows = np.concatenate([np.arange(ioff[r], ioff[r + 1]) for r in reads] + [np.zeros(0, np.int64)])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "intervals.npy"), iv[rows].reshape(-1, 2).astype(np.float64))
    np.save(os.path.join(out_dir, "interval_offsets.npy"),
            np.concatenate([[0], np.cumsum(counts[reads])]).astype(np.float64))
    np.save(os.path.join(out_dir, "read_ids.npy"), reads.astype(np.float64))


def workload_config(reads_per_step, engine):
    return {"workload": "ResNetRNN infer, shipped checkpoint ckpnt-30000, synthetic raw-signal reads of ragged length "
                        "U{50k..200k} samples (BASELINE configs[3]), sharded by read",
            "reads_per_step_per_gpu": reads_per_step, "engine": engine, "window": 35,
            "l2": "inputs larger than L2 (signal + intermediates of a step exceed 126 MB); two alternating batches"}


# ------------------------------------------------------------------------------------ CPU arm
def cpu_run(weights, raw, offsets):
    """One pass of the reference path restated on the CPU over the given reads; returns seconds."""
    import torch
    from oracle import postprocess, tf_graph
    if torch.get_num_threads() < (os.cpu_count() or 1):
        torch.set_num_threads(os.cpu_count() or 1)      # torchrun exports OMP_NUM_THREADS=1: use all host cores
    graph = tf_graph.TorchGraph(weights)
    t0 = time.perf_counter()
    n_int = 0
    for r in range(len(offsets) - 1):
        hps, _, _ = postprocess.infer_read(raw[offsets[r]:offsets[r + 1]], graph.infer)
        n_int += len(hps)
    return time.perf_counter() - t0, n_int, torch.get_num_threads()


def run_reference(args):
    """--impl reference: the CPU restatement of the reference path (oracle port), all host threads.

    Same metric / unit / config as the GPU arm; a step is a bounded sample (4 reads of the 512-read step's
    length distribution) so that the whole run ends within minutes; samples/s is size-normalised."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from catfish_b200 import weights as W
    w = W.load_shipped()
    n_reads = 4                                   # bounded sample of the configs[3] length distribution
    batches = [make_batch(n_reads, 9000 + i) for i in range(2)]
    cpu_run(w, batches[0][0][:35 * 200], np.array([0, 35 * 200]))         # page in torch
    for i in range(args.warmup):
        cpu_run(w, *batches[i % 2])
    total_s, total_samples, threads = 0.0, 0, 1
    for i in range(args.steps):
        raw, off = batches[i % 2]
        s, _, threads = cpu_run(w, raw, off)
        total_s += s
        total_samples += int(off[-1])
    value = total_samples / total_s
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total_s / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.reads_per_step, args.engine),
        "reads_per_sec": n_reads * args.steps / total_s,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "each step = %d reads of the step's U{50k..200k} length distribution (a bounded "
                                   "sample of the %d-read step; samples/s is size-normalised); TF-graph CPU "
                                   "restatement, torch fp32 + the reference's post-processing; TensorFlow is not "
                                   "installable offline" % (n_reads, args.reads_per_step)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "host_cores": os.cpu_count(),
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_leg():
    """BASELINE.md section 3: 200 synthetic reads x 10 000 samples, end to end, median of 3 runs after 1 warm-up."""
    from catfish_b200 import synth, weights as W
    reads = synth.synth_reads([10000] * 200, base_seed=77)
    raw, off = synth.concat_reads(reads)
    w = W.load_shipped()
    cpu_run(w, raw[:7000], np.array([0, 7000]))
    cpu_run(w, raw, off)                                     # warm-up run
    runs = []
    threads = 1
    for _ in range(3):
        secs, _, threads = cpu_run(w, raw, off)
        runs.append(secs)
    secs = float(np.median(runs))
    return {"value": len(raw) / secs, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": "BASELINE configs[0]: 200 synthetic reads x 10 000 samples end to end, TF-graph CPU restatement "
                      "(torch fp32) + reference post-processing, median of 3 runs after 1 warm-up (%.1f s each; "
                      "--impl reference times the long-read distribution instead)" % secs,
            "runs_s": runs, "host_cores": os.cpu_count()}


# ------------------------------------------------------------------------------------ roofline helpers
def kernel_table(prof, ms_total, samples, flops, peaks):
    out = {}
    for k, (ms, cnt) in prof.items():
        ent = {"ms": ms, "launches": cnt, "share": ms / ms_total if ms_total else None}
        if ms > 0 and k in flops:
            ent["tflops"] = flops[k] * samples / (ms * 1e-3) / 1e12
            ent["frac_of_tensor_peak"] = ent["tflops"] / peaks["tensor_sustained"]
        elif ms > 0 and BYTES_PER_SAMPLE.get(k):
            ent["gbs"] = BYTES_PER_SAMPLE[k] * samples / (ms * 1e-3) / 1e9
            ent["frac_of_hbm_peak"] = ent["gbs"] / peaks["hbm"]
        out[k] = ent
    return out


def dominant_roofline(prof, ms_total, samples, flops, peaks):
    name, (dom_ms, dom_launches) = max(prof.items(), key=lambda kv: kv[1][0])
    per_launch_s = dom_ms * 1e-3 / max(1, dom_launches)
    units_per_launch = samples / max(1, dom_launches)
    if name in flops:
        achieved = flops[name] * units_per_launch / per_launch_s / 1e12
        roof = {"bound": "tensor", "achieved": achieved, "peak": peaks["tensor_sustained"], "unit": "TFLOP/s",
                "frac": achieved / peaks["tensor_sustained"], "traffic": None}
    else:
        achieved = BYTES_PER_SAMPLE.get(name, 0.0) * units_per_launch / per_launch_s / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm"], "unit": "GB/s",
                "frac": achieved / peaks["hbm"], "traffic": None}
    roof.update({"kernel": name, "launches": dom_launches, "avg_launch_ms": dom_ms / max(1, dom_launches),
                 "share_of_step": dom_ms / ms_total if ms_total else None,
                 "peak_source": peaks["source"] + " (sustained)",
                 "algorithmic_per_sample": flops.get(name, BYTES_PER_SAMPLE.get(name))})
    return roof


def source_fingerprint():
    """sha1 over the sources of the kernels the committed ncu traffic figures belong to (the tensor-core engine and
    every header of csrc/): ties `profiles/r2_traffic.json` to the kernels being timed."""
    h = hashlib.sha1()
    csrc = os.path.join(ROOT, "catfish_b200", "csrc")
    for name in sorted(os.listdir(csrc)):
        if name != "tc_engine.cu" and not name.endswith((".cuh", ".h")):
            continue
        with open(os.path.join(csrc, name), "rb") as f:
            h.update(name.encode())
            h.update(f.read())
    return h.hexdigest()


def attach_traffic(roof):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed
    `ncu --set full` capture - only if that capture was taken from the kernel sources being timed."""
    tpath = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(tpath):
        return
    with open(tpath) as f:
        tj = json.load(f)
    roof["traffic_commit"] = tj.get("commit")
    if tj.get("source_sha1") != source_fingerprint():
        roof["traffic_stale"] = "profiles/r2_traffic.json was captured from other kernel sources (%s); not reported" \
            % tj.get("commit")
        return
    if roof["kernel"] in tj:
        roof["traffic"] = tj[roof["kernel"]]["dram_bytes_per_launch"]
        roof["traffic_source"] = "profiles/r2_traffic.json (%s)" % tj.get("source", "ncu --set full")


# ------------------------------------------------------------------------------------ GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from catfish_b200 import _cabi, infer, neural_network, sharding, synth, weights as W

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        # not launched under torchrun: relaunch ourselves one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    legs = set((args.legs or ("main,probs,python,job,configs,cpu,check" if world == 1 else "main,job,check")).split(","))
    if args.no_cpu_baseline:
        legs.discard("cpu")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _cabi.load_library()
    model = neural_network.load_network("ResNetRNN", None, 30000, device=local_rank, engine=args.engine)
    engine = model.resolved_engine
    handle = model.handle
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    peaks = load_peaks()

    # two alternating batches per rank, staged in pinned host memory and resident on the device
    batches = []
    for b in range(2):
        raw, off = make_batch(args.reads_per_step, 1000 * (rank + 1) + b)
        raw_pin = torch.from_numpy(raw).pin_memory()
        batches.append(dict(raw_pin=raw_pin, raw_dev=raw_pin.to("cuda", non_blocking=True), off=off,
                            n=int(off[-1])))
    n_reads = args.reads_per_step
    cap = max(int(lib.cf_max_intervals(b["n"], n_reads, 15)) for b in batches)
    iv_dev = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
    ioff_dev = torch.empty(n_reads + 1, dtype=torch.int64, device="cuda")
    iv_host = torch.empty((cap, 2), dtype=torch.int64).pin_memory()
    ioff_host = torch.empty(n_reads + 1, dtype=torch.int64).pin_memory()
    found = ctypes.c_int64(0)
    _cabi.check(lib.cf_model_reserve(handle, max(b["n"] for b in batches), n_reads))

    def step_device(i):
        b = batches[i % 2]
        _cabi.check(lib.cf_infer_reads(handle, b["raw_dev"].data_ptr(), b["off"].ctypes.data_as(_cabi.c_i64_p), n_reads,
                                       None, iv_dev.data_ptr(), ioff_dev.data_ptr(), cap, 0.5, 15, 11, 16, sp))

    def step_host(i, probs=None):
        b = batches[i % 2]
        _cabi.check(lib.cf_infer_reads_host(handle, b["raw_pin"].data_ptr(), b["off"].ctypes.data_as(_cabi.c_i64_p),
                                            n_reads, probs.data_ptr() if probs is not None else None,
                                            iv_host.data_ptr(), ioff_host.data_ptr(), cap, 0.5, 15, 11,
                                            16, ctypes.byref(found), sp))
        return int(found.value)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return float(x)

    def timed(step_fn, steps):
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record(stream)
        for i in range(steps):
            step_fn(i)
        ev1.record(stream)
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1))

    for i in range(max(3, args.warmup)):
        step_device(i)
    torch.cuda.synchronize()

    # ---- timed region 1: device-resident inputs, per-kernel-class events on
    _cabi.profile_enable(handle, True)
    launches0 = _cabi.launch_count()
    # address the GPU by UUID: nvidia-smi's index order need not be CUDA's (visible-device remapping)
    try:
        gpu_id = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        gpu_id = local_rank
    sampler = ClockSampler(gpu_id)
    t0 = time.time()
    ms_dev = timed(step_device, args.steps)
    t1 = time.time()
    clocks = sampler.stop(t0, t1)
    launches = _cabi.launch_count() - launches0
    prof = _cabi.profile_read(handle)
    _cabi.profile_enable(handle, False)
    if args.dump_outputs and rank == 0:
        # the last timed step ran batch (steps - 1) % 2; its result is still in iv_dev / ioff_dev
        ioff_last = ioff_dev.cpu().numpy()
        dump_outputs(args.dump_outputs, iv_dev[:int(ioff_last[-1])].cpu().numpy(), ioff_last)

    # ---- timed region 2: host buffers through the public C-ABI call
    for i in range(2):
        step_host(i)
    n_intervals = step_host(0)
    ms_e2e = timed(step_host, args.steps)
    step_host(0)                                     # leave batch 0's result in iv_host / ioff_host (parity check)
    e2e_iv = iv_host[:int(found.value)].numpy().copy()
    e2e_ioff = ioff_host.numpy().copy()

    samples_rank = sum(batches[i % 2]["n"] for i in range(args.steps))
    h2d = int(np.mean([2 * batches[i % 2]["n"] + 16 * (n_reads + 1) for i in range(args.steps)]))
    d2h = int(16 * n_intervals + 8 * (n_reads + 1))
    if world > 1:
        t = torch.tensor([samples_rank, launches], dtype=torch.float64, device="cuda")
        dist.all_reduce(t)
        samples_all, launches_all = float(t[0].item()), int(t[1].item())
    else:
        samples_all, launches_all = float(samples_rank), int(launches)
    value = samples_all / (ms_dev * 1e-3)
    e2e = samples_all / (ms_e2e * 1e-3)
    extra = {}

    # ---- e2e_probs: the host call with the probabilities returned as well
    if "probs" in legs:
        probs_pin = torch.empty(max(b["n"] for b in batches), dtype=torch.float32).pin_memory()
        step_host(0, probs_pin)
        ms_p = timed(lambda i: step_host(i, probs_pin), args.steps)
        extra["e2e_probs"] = {"value": samples_all / (ms_p * 1e-3), "unit": UNIT, "ms_per_step": ms_p / args.steps,
                              "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h + 4 * int(samples_rank / args.steps),
                              "note": "cf_infer_reads_host with probs_host (pinned): per-position probabilities + "
                                      "intervals returned"}
        del probs_pin

    # ---- e2e_python: the package's public Python call on a list of numpy reads (host wall clock)
    if "python" in legs:
        lists = []
        for b in batches:
            r, o = b["raw_pin"].numpy(), b["off"]
            lists.append([np.array(r[o[k]:o[k + 1]]) for k in range(n_reads)])      # separate pageable arrays
        for i in range(2):
            infer.infer_reads(lists[i % 2], model)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.steps):
            hps_py, lens_py = infer.infer_reads(lists[i % 2], model)
        torch.cuda.synchronize()
        ms_py = max_over_ranks((time.perf_counter() - t0) * 1e3)
        extra["e2e_python"] = {"value": samples_all / (ms_py * 1e-3), "unit": UNIT, "ms_per_step": ms_py / args.steps,
                               "ratio_to_e2e": (samples_all / (ms_py * 1e-3)) / e2e,
                               "note": "infer.infer_reads(list of %d numpy int16 arrays): ragged concat into pinned "
                                       "staging + cf_infer_reads_host + per-read IntervalList views; host wall clock"
                                       % n_reads}
        del lists

    # ---- job: one fixed list of reads, LPT shards, host-side gather on rank 0 inside the timed region
    if "job" in legs:
        extra["job"] = job_leg(args, model, rank, world, barrier, max_over_ranks)

    # ---- parity check of the timed binary against the CPU oracle (outside every timed region)
    if "check" in legs and rank == 0:
        extra["parity_check"] = parity_leg(model, batches[0], e2e_iv, e2e_ioff)

    if rank == 0:
        fused = prof.get("k3_gru_input_proj", (0.0, 0))[0] == 0.0
        flops = flops_per_sample("ResNetRNN", fused)
        roof = dominant_roofline(prof, ms_dev, samples_rank, flops, peaks)
        if fused and roof["kernel"] == "k4_gru_recurrence":
            roof["note"] = "fused GRU layer: input projection + recurrence"
        attach_traffic(roof)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": ms_dev / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": {"f16e5": "f16+e5m2 (fp16 product + e5m2 correction product, fp32 accumulate)",
                      "bf16x3": "bf16x3 (split bf16 operands, fp32 accumulate)"}.get(model.operand_format, "f32"),
            "data": "synthetic", "config": workload_config(n_reads, engine),
            "reads_per_sec": world * n_reads * args.steps / (ms_dev * 1e-3),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_all, "clocks": clocks, "roofline": roof,
            "kernels": kernel_table(prof, ms_dev, samples_rank, flops, peaks),
            "intervals_per_step": n_intervals,
        }
        line.update(extra)
    # ---- the other BASELINE configs (N = 1): throughput + dominant kernel + roofline fraction each
    if "configs" in legs and world == 1:
        del batches, iv_dev, iv_host
        torch.cuda.empty_cache()
        line["configs"] = configs_leg(args, model, peaks)
    if "cpu" in legs and world == 1:
        line["cpu_baseline"] = cpu_baseline_leg()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def job_leg(args, model, rank, world, barrier, max_over_ranks):
    """catfish/catfish:55-56 as one sharded job (strong scaling): fixed seeded reads, LPT partition by read,
    every rank infers its shard in batches, rank 0 gathers the per-read results - all inside the timed region."""
    import torch
    from catfish_b200 import infer, sharding, synth
    n = args.job_reads
    # read i is entry i % JOB_POOL of a pool of distinct seeded reads (generating 1e10 distinct synthetic samples
    # on the host would take minutes); lengths and contents repeat with period JOB_POOL, results are per read
    pool_len = synth.ragged_lengths(min(n, JOB_POOL), LEN_LO, LEN_HI, seed=JOB_SEED)
    lengths = pool_len[np.arange(n) % len(pool_len)]
    mine = sharding.shard_for_rank(lengths, rank, world)
    local = {}
    for i in mine:
        k = int(i) % len(pool_len)
        if k not in local:
            local[k] = synth.synth_read(int(pool_len[k]), JOB_SEED * 7 + k)       # only what this rank's shard needs

    class Reads(object):
        def __len__(self):
            return n

        def __getitem__(self, i):
            return local[int(i) % len(pool_len)]

    reads = Reads()
    # warm-up: staging buffers, workspace, and the communicator paths the gather uses (first NCCL all_gather /
    # gather calls set up their channels, which takes longer than the whole job)
    wh, wl = infer.infer_reads([reads[int(i)] for i in mine[:args.reads_per_step]], model)
    sharding.gather_intervals(mine[:len(wh)], wh, wl, n, rank, world)
    if world > 1:
        # staging of the result gather sized for the job (intervals per sample of the warm-up batch, 30 % margin),
        # as a long-running service would have it after its first job
        per_sample = sum(len(h) for h in wh) / max(1, sum(wl))
        sharding.reserve_gather(len(mine), int(1.3 * per_sample * float(lengths[mine].sum())) + 1024, rank, world)
    barrier()
    t0 = time.perf_counter()
    res = sharding.infer_reads_sharded(reads, model, rank, world, batch_reads=args.reads_per_step, lengths=lengths)
    torch.cuda.synchronize()
    secs = max_over_ranks(time.perf_counter() - t0)
    breakdown = {k: max_over_ranks(float(v)) for k, v in sorted(sharding.last_timing.items())}     # max over ranks
    loads = [int(lengths[p].sum()) for p in sharding.partition_reads(lengths, world)]
    out = {"reads": n, "samples": int(lengths.sum()), "seconds": secs, "reads_per_sec": n / secs,
           "samples_per_sec": float(lengths.sum()) / secs, "scaling": "strong", "n_gpus": world,
           "rank_load_max_over_min": max(loads) / max(1, min(loads)),
           "distinct_reads": int(min(n, JOB_POOL)), "breakdown_max_over_ranks": breakdown,
           "note": "LPT shards by read, infer.infer_reads_arrays per batch of %d reads, gather_csr on rank 0, all "
                   "inside the timed region (host wall clock, max over ranks); result_sha1 is over the merged "
                   "per-read (length, intervals) in read order and must not depend on n_gpus" % args.reads_per_step}
    if rank == 0:
        hps, lens = res
        h = hashlib.sha1()
        h.update(np.asarray(lens, np.int64).tobytes())
        for iv in hps:
            h.update(np.ascontiguousarray(iv.array).tobytes())
            h.update(b"|")
        out["result_sha1"] = h.hexdigest()
        out["intervals"] = int(sum(len(iv) for iv in hps))
    return out


def parity_leg(model, batch, e2e_iv, e2e_ioff):
    """Two reads of the timed batch: the timed call's intervals == a separate small call's (batch invariance), and
    that call's probabilities / intervals against the CPU oracle (contract: 1e-3, flips only inside the band)."""
    from catfish_b200 import infer
    from oracle import postprocess, tf_graph
    off = batch["off"]
    picks = [int(i) for i in np.argsort(np.diff(off))[:2]]           # the two shortest reads
    raw = batch["raw_pin"].numpy()
    reads = [np.array(raw[off[i]:off[i + 1]]) for i in picks]
    hps, lens, scores = infer.infer_reads(reads, model, return_scores=True)
    graph = tf_graph.TorchGraph(model.get_weights())
    worst, flips_outside, same_as_batch, same_as_oracle = 0.0, 0, True, True
    for i, r, h, s in zip(picks, reads, hps, scores):
        want_h, _, want_s = postprocess.infer_read(r, graph.infer)
        worst = max(worst, float(np.abs(s - want_s).max()))
        flip = (s.astype(np.float64) >= 0.5) != (want_s >= 0.5)
        flips_outside += int(np.count_nonzero(flip & (np.abs(want_s - 0.5) > 1e-3)))
        same_as_oracle &= bool(h == want_h) or bool(flip.any())
        same_as_batch &= bool(np.array_equal(h.array, e2e_iv[e2e_ioff[i]:e2e_ioff[i + 1]]))
    return {"reads": len(reads), "samples": int(sum(lens)), "max_abs_dp_vs_cpu_oracle": worst,
            "label_flips_outside_1e-3_band": flips_outside, "intervals_equal_oracle_or_flip_in_band": same_as_oracle,
            "intervals_equal_timed_batch": same_as_batch, "ok": worst < 1e-3 and flips_outside == 0 and same_as_batch
            and same_as_oracle}


def configs_leg(args, resnetrnn, peaks):
    """BASELINE.json configs[0], [1], [2], [4] on one GPU: samples/s, dominant kernel class, roofline fraction."""
    import torch
    from catfish_b200 import _cabi, neural_network, synth, weights as W
    lib = _cabi.load_library()
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    steps = args.steps
    out = {}

    def measure(model, kind, step_fn, samples_per_step, reads_per_step, describe, flops_of=None):
        handle = model.handle
        for i in range(3):
            step_fn(i)
        torch.cuda.synchronize()
        _cabi.profile_enable(handle, True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for i in range(steps):
            step_fn(i)
        ev1.record(stream)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        prof = _cabi.profile_read(handle)
        _cabi.profile_enable(handle, False)
        fused = prof.get("k3_gru_input_proj", (0.0, 0))[0] == 0.0
        flops = flops_of(fused) if flops_of else flops_per_sample(kind, fused)
        total = samples_per_step * steps
        roof = dominant_roofline(prof, ms, total, flops, peaks)
        ent = {"workload": describe, "samples_per_sec": total / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps,
               "engine": model.resolved_engine, "operand_format": model.operand_format,
               "dominant_kernel": roof["kernel"], "dominant_share": roof["share_of_step"], "roofline_frac": roof["frac"],
               "roofline_bound": roof["bound"], "roofline_achieved": roof["achieved"], "roofline_unit": roof["unit"],
               "kernels": {k: {"ms_per_step": v["ms"] / steps, "launches_per_step": v["launches"] / steps,
                               **({"frac_of_tensor_peak": v["frac_of_tensor_peak"]} if "frac_of_tensor_peak" in v else {}),
                               **({"frac_of_hbm_peak": v["frac_of_hbm_peak"]} if "frac_of_hbm_peak" in v else {})}
                           for k, v in kernel_table(prof, ms, total, flops, peaks).items() if v["ms"] > 0}}
        if reads_per_step:
            ent["reads_per_sec"] = reads_per_step * steps / (ms * 1e-3)
        return ent

    def reads_step(model, raw_dev, off, n_reads):
        n = int(off[-1])
        cap = int(lib.cf_max_intervals(n, n_reads, 15))
        iv = torch.empty((cap, 2), dtype=torch.int64, device="cuda")
        ioff = torch.empty(n_reads + 1, dtype=torch.int64, device="cuda")
        _cabi.check(lib.cf_model_reserve(model.handle, n, n_reads))

        def fn(i):
            _cabi.check(lib.cf_infer_reads(model.handle, raw_dev.data_ptr(), off.ctypes.data_as(_cabi.c_i64_p), n_reads,
                                           None, iv.data_ptr(), ioff.data_ptr(), cap, 0.5, 15, 11, 16, sp))
        return fn, (iv, ioff)

    # configs[0]: ResNetRNN, 200 reads x 10 000 samples
    raw, off = synth.concat_reads(synth.synth_reads([10000] * 200, base_seed=77))
    raw_dev = torch.from_numpy(raw).cuda()
    fn, keep = reads_step(resnetrnn, raw_dev, off, 200)
    out["c0_resnetrnn_200x10k"] = measure(resnetrnn, "ResNetRNN", fn, int(off[-1]), 200,
                                          "configs[0]: ResNetRNN, shipped checkpoint, 200 synthetic reads x 10 000 "
                                          "samples per step (the CPU-runnable case; cpu_baseline times the same reads)")
    # configs[4]: 1M-sample reads: one read (latency) and a batch of 64 (throughput)
    big = synth.synth_reads([1_000_000] * 8, base_seed=4100)
    raw1, off1 = synth.concat_reads(big[:1])
    raw1_dev = torch.from_numpy(raw1).cuda()
    fn, keep = reads_step(resnetrnn, raw1_dev, off1, 1)
    out["c4_single_1M_read"] = measure(resnetrnn, "ResNetRNN", fn, 1_000_000, 1,
                                       "configs[4]: one 1M-sample read per step, raw int16 (device) -> intervals: "
                                       "ms_per_step is the single-read latency")
    raw64, off64 = synth.concat_reads([big[i % 8] for i in range(64)])
    raw64_dev = torch.from_numpy(raw64).cuda()
    fn, keep = reads_step(resnetrnn, raw64_dev, off64, 64)
    out["c4_batch_64x1M"] = measure(resnetrnn, "ResNetRNN", fn, int(off64[-1]), 64,
                                    "configs[4]: 64 reads x 1M samples per step")
    del raw64_dev, raw1_dev, raw_dev, keep
    # configs[1]: RNN-only (neural_network.py:17-18), random-init H = 64 x 3 layers, 4 000 reads x 20 000 samples
    hp = dict(W.SHIPPED_HPARAMS)
    rnn = neural_network.build_model("RNN", engine=args.engine, **hp)
    rnn.set_weights(W.random_init("RNN", seed=11, layer_size=64, n_layers=3))
    rawr, offr = synth.concat_reads(synth.synth_reads([20000] * 4000, base_seed=5100))
    rawr_dev = torch.from_numpy(rawr).cuda()
    fn, keep = reads_step(rnn, rawr_dev, offr, 4000)
    out["c1_rnn_only_4000x20k"] = measure(rnn, "RNN", fn, int(offr[-1]), 4000,
                                          "configs[1]: RNN-only (layer_size 64 x 3 layers, seeded random-init), 4 000 "
                                          "synthetic reads x 20 000 samples per step")
    del rawr_dev, keep, rnn
    torch.cuda.empty_cache()
    # configs[1], stress variant of SURVEY 8d (networks/train_validate.py:330): RNN-only H = 256 x 5 layers.  Its 384 KB
    # of recurrent weights per direction do not fit one SM, so it runs on the fp32 CUDA-core engine (DESIGN.md
    # section 9); the fraction is still quoted against the bf16 tensor peak.
    hp256 = dict(hp, layer_size=256, n_layers=5)
    rnn256 = neural_network.build_model("RNN", engine=args.engine, **hp256)
    rnn256.set_weights(W.random_init("RNN", seed=13, layer_size=256, n_layers=5))
    raws, offs = synth.concat_reads(synth.synth_reads([20000] * 32, base_seed=5200))
    raws_dev = torch.from_numpy(raws).cuda()
    fn, keep = reads_step(rnn256, raws_dev, offs, 32)

    def flops256(fused):
        xproj = 2.0 * 2 * 1 * 768 + 4 * (2.0 * 2 * 512 * 768)
        rec = 5 * (2.0 * 2 * 256 * 768)
        d = {"k5_head": 1024.0}
        if fused:
            d["k4_gru_recurrence"] = xproj + rec
        else:
            d["k3_gru_input_proj"], d["k4_gru_recurrence"] = xproj, rec
        return d
    out["c1_rnn_only_h256x5_stress"] = measure(rnn256, "RNN", fn, int(offs[-1]), 32,
                                               "configs[1] stress variant: RNN-only layer_size 256 x 5 layers (10.2 MFLOP "
                                               "per sample), seeded random-init, 32 synthetic reads x 20 000 samples per step",
                                               flops_of=flops256)
    del raws_dev, keep, rnn256
    torch.cuda.empty_cache()
    # configs[2]: ResNet-only (resnet_class.py:23), random-init, 1 048 576 windows per call through cf_infer_windows
    res = neural_network.build_model("ResNet", engine=args.engine, **hp)
    res.set_weights(W.random_init("ResNet", seed=12, layer_size_res=32, n_layers_res=2))
    n_win = 1 << 20
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    x = torch.randn((n_win, 35), generator=g, device="cuda", dtype=torch.float32) * 1.5
    p = torch.empty(n_win * 35, dtype=torch.float32, device="cuda")

    def fn_win(i):
        _cabi.check(lib.cf_infer_windows(res.handle, x.data_ptr(), n_win, p.data_ptr(), sp))
    out["c2_resnet_only_1Mwindows"] = measure(res, "ResNet", fn_win, n_win * 35, 0,
                                              "configs[2]: ResNet-only (32 channels x 2 blocks, seeded random-init), "
                                              "1 048 576 windows (3.67e7 samples) per cf_infer_windows call, "
                                              "probabilities written to HBM")
    return out


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
