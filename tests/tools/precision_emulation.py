#!/usr/bin/env python3
"""Emulate tensor-core operand formats on the CPU graph: max |dp| against the fp64 graph.

    python tests/tools/precision_emulation.py [n_reads] [read_len]

Every 32 -> 32 convolution and every GRU matmul of the oracle graph (oracle/tf_graph.py) is replaced by
a product of ROUNDED operands accumulated in fp64 (the tensor core accumulates in fp32; that
difference is below the effects studied here).  The Cin = 1 convolutions, the head and all
elementwise math stay exact, as in the CUDA engine.  Schemes:
  bf16x3     a_hi w_hi + a_lo w_hi + a_hi w_lo, bf16 pieces              (the shipped scheme, 3 passes)
  bf16x1     one bf16 pass                          fp16x1   one fp16 pass
  fp16x2     (a_hi + a_lo) w_hi, fp16 pieces                               (2 passes)
  fp16+e5m2  a_hi w_hi in fp16 + [a_lo 2^s | a_hi 2^-s] [w_hi 2^-s ; w_lo 2^s] in e5m2, the a_hi 2^-s byte
             truncated (it is the top byte of the fp16 value, never stored in HBM)
             (1 fp16 pass + 1 fp8 pass with doubled K = 2 pass-equivalents; DESIGN.md section 4)
  fp16+e5m2 faults, each a correction term lost:  "-lo" drops a_lo w_hi, "-hi" drops a_hi w_lo, "-both" drops both
engine_mm(kind) picks the format per matmul the way the tensor-core engine does.
Test infrastructure only (imports oracle/).
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))
from catfish_b200 import synth, weights  # noqa: E402
from oracle import postprocess, tf_graph  # noqa: E402


def rnd(x, dt):
    return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(dt).to(torch.float32).numpy().astype(np.float64)


def trunc_e5(x):
    """Top byte of fp16(x): the e5m2 of x truncated toward zero to two mantissa bits."""
    h = torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(torch.float16)
    return (h.view(torch.int16) & -256).view(torch.float16).to(torch.float32).numpy().astype(np.float64)


def make_mm(scheme, s_corr=6):
    bf, hf, e5 = torch.bfloat16, torch.float16, torch.float8_e5m2

    def split(x, dt):
        hi = rnd(x, dt)
        return hi, rnd(x - hi, dt)

    def mm(a, w):
        a = np.asarray(a, np.float64)
        w = np.asarray(w, np.float64)
        if scheme == "exact":
            return a @ w
        if scheme == "bf16x1":
            return rnd(a, bf) @ rnd(w, bf)
        if scheme == "fp16x1":
            return rnd(a, hf) @ rnd(w, hf)
        if scheme == "bf16x3":
            ah, al = split(a, bf)
            wh, wl = split(w, bf)
            return ah @ wh + al @ wh + ah @ wl
        if scheme == "fp16x2":
            ah, al = split(a, hf)
            return (ah + al) @ rnd(w, hf)
        if scheme.startswith("fp16+e5m2"):
            fault = scheme[len("fp16+e5m2"):]
            if fault not in ("", "-lo", "-hi", "-both"):
                raise ValueError(scheme)
            wh = rnd(w, hf)
            ah = 2.0 ** s_corr * rnd(rnd(a, hf) / 2.0 ** s_corr, hf)      # main plane = fp16(fp16(a) 2^-s)
            al, wl = a - ah, w - wh
            k = 2.0 ** s_corr
            out = ah @ wh
            if fault not in ("-lo", "-both"):
                out = out + rnd(al * k, e5) @ rnd(wh / k, e5)
            if fault not in ("-hi", "-both"):
                # the a_hi 2^-s byte is the top byte of the fp16 main value (truncated e5m2), as the kernels build it
                out = out + trunc_e5(ah / k) @ rnd(wl * k, e5)
            return out
        raise ValueError(scheme)
    return mm


def engine_mm(kind, f16e5="fp16+e5m2"):
    """Matmul in the operand format the tensor-core engine uses for each product of the H = 64 networks, with
    `f16e5` (a fp16+e5m2 scheme, possibly a fault) where the engine runs f16e5.  ResNetRNN: the convolutions
    (K = 32) and GRU layer 0 (K = 32 + 64) are bf16x3, the 128-wide layers (K = 128 + 64) f16e5.  RNN: every layer is
    f16e5, except that layer 0's scalar input row (K = 1 + 64) is an exact rank-1 update."""
    if kind not in ("ResNetRNN", "RNN"):
        raise ValueError(kind)
    bf3, f16 = make_mm("bf16x3"), make_mm(f16e5)

    def mm(a, w):
        k = np.shape(a)[1]
        if kind == "RNN" and k == 1 + 64:
            a, w = np.asarray(a, np.float64), np.asarray(w, np.float64)
            return a[:, :1] @ w[:1] + f16(a[:, 1:], w[1:])
        return f16(a, w) if kind == "RNN" or k == 128 + 64 else bf3(a, w)
    return mm


def synthetic_windows(n_windows, read_len=7000, seed=300):
    """The first n_windows windows [n, 35, 1] of normalised synthetic reads (seeds seed, seed + 1, ...)."""
    xs, n = [], 0
    while n < n_windows:
        raw = synth.synth_read(read_len, seed + len(xs))
        xs.append(postprocess.pad_and_window(postprocess.normalize_raw_signal(raw))[0])
        n += xs[-1].shape[0]
    return np.concatenate(xs, 0)[:n_windows]


def tile_rms(p, ref, tile=128):
    """RMS of p - ref over each tile of `tile` windows (35 positions each); the last tile counts only the windows
    it has.  A fault confined to some tiles (one chain of the fused GRU kernel) shows in those tiles undiluted."""
    d = np.asarray(p, np.float64) - np.asarray(ref, np.float64)
    per = tile * tf_graph.WINDOW
    return np.array([np.sqrt(np.mean(d[i:i + per] ** 2)) for i in range(0, d.size, per)])


def forward(w, x, mm):
    """oracle/tf_graph.forward_np with pluggable matmuls (same op order)."""
    f8 = np.float64
    kind, n_res, n_rnn = tf_graph.describe(w)
    y = np.asarray(x, np.float32).astype(f8).reshape(-1, 35, 1)

    def conv(i, inp):
        k = w["conv1d%s/kernel" % tf_graph._suffix(i)].astype(f8)
        b = w["conv1d%s/bias" % tf_graph._suffix(i)].astype(f8)
        ksz, cin, cout = k.shape
        pad = (ksz - 1) // 2
        xp = np.pad(inp, ((0, 0), (pad, pad), (0, 0)))
        out = np.zeros(inp.shape[:2] + (cout,), f8)
        for tap in range(ksz):
            sl = xp[:, tap:tap + inp.shape[1], :].reshape(-1, cin)
            out += ((sl @ k[tap]) if cin == 1 else mm(sl, k[tap])).reshape(out.shape)
        return tf_graph._batch_norm_np(out + b, w, i)

    for b_ in range(n_res):
        i = 4 * b_
        sc = conv(i, y)
        o = np.maximum(conv(i + 1, y), 0)
        o = np.maximum(conv(i + 2, o), 0)
        o = np.maximum(conv(i + 3, o), 0)
        y = np.maximum(o + sc, 0)
    for l in range(n_rnn):
        outs = []
        for d, rev in (("fw", False), ("bw", True)):
            p = tf_graph._gru_prefix(l, d)
            wg, bg = w[p + "/gates/kernel"].astype(f8), w[p + "/gates/bias"].astype(f8)
            wc, bc = w[p + "/candidate/kernel"].astype(f8), w[p + "/candidate/bias"].astype(f8)
            hs = wc.shape[1]
            h = np.zeros((y.shape[0], hs), f8)
            out = np.zeros((y.shape[0], 35, hs), f8)
            for s in (range(34, -1, -1) if rev else range(35)):
                xs = y[:, s]
                g = tf_graph._sigmoid_np(mm(np.concatenate([xs, h], 1), wg) + bg)
                r, u = g[:, :hs], g[:, hs:]
                c = np.tanh(mm(np.concatenate([xs, r * h], 1), wc) + bc)
                h = u * h + (1 - u) * c
                out[:, s] = h
            outs.append(out)
        y = np.concatenate(outs, 2)
    z = y.reshape(-1, y.shape[2]) @ w["final_fully_connected/kernel"].astype(f8) + w["final_fully_connected/bias"].astype(f8)
    return tf_graph._sigmoid_np(z.reshape(-1))


if __name__ == "__main__":
    n_reads = int(sys.argv[1]) if len(sys.argv) > 1 else 12
    read_len = int(sys.argv[2]) if len(sys.argv) > 2 else 7000
    w = weights.load_shipped()
    xs = []
    for raw in synth.synth_reads([read_len] * n_reads, base_seed=300):
        xs.append(postprocess.pad_and_window(postprocess.normalize_raw_signal(raw))[0])
    x = np.concatenate(xs, 0)
    ref = forward(w, x, make_mm("exact"))
    print("positions", ref.size)
    for scheme, kw in (("bf16x3", {}), ("bf16x1", {}), ("fp16x1", {}), ("fp16x2", {}), ("fp16+e5m2", {"s_corr": 6}),
                       ("fp16+e5m2", {"s_corr": 8})):
        p = forward(w, x, make_mm(scheme, **kw))
        d = np.abs(p - ref)
        flips = int(np.count_nonzero(((p >= 0.5) != (ref >= 0.5)) & (np.abs(ref - 0.5) > 1e-3)))
        print("%-10s %-14s max|dp| %.2e  p99.9 %.2e  flips outside band %d" % (scheme, kw or "", d.max(), np.quantile(d, 0.999), flips))
