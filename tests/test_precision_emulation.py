"""CPU: the operand-format emulation behind DESIGN.md section 4 keeps its ordering on a small sample
(single 16-bit passes miss the contract's margin, the split formats do not), and the f16e5 budget statistic of
tests/test_gpu_operand_formats.py tells a lost correction term from the correct scheme, as the bf16x3 budget of
tests/test_gpu_precision_budgets.py tells one convolution tap without a correction pass."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))


@pytest.fixture(autouse=True)
def _one_torch_thread():
    # the emulation rounds many small arrays through torch dtype casts, ~30x slower on several intra-op threads
    import torch
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(n)


def test_format_ordering(shipped_weights):
    import precision_emulation as pe
    from catfish_b200 import synth
    from oracle import postprocess
    raw = synth.synth_reads([2100], base_seed=300)[0]
    x = postprocess.pad_and_window(postprocess.normalize_raw_signal(raw))[0]
    ref = pe.forward(shipped_weights, x, pe.make_mm("exact"))
    err = {s: float(np.abs(pe.forward(shipped_weights, x, pe.make_mm(s)) - ref).max())
           for s in ("bf16x3", "fp16+e5m2", "fp16x1", "bf16x1")}
    assert err["bf16x3"] < 1e-4 and err["fp16+e5m2"] < 2e-4
    assert err["fp16+e5m2"] < err["fp16x1"] < err["bf16x1"]
    assert err["bf16x1"] > 1e-3                      # a single bf16 pass breaks the 1e-3 contract


def test_f16e5_fault_budget(shipped_weights):
    """The shipped network in the engine's formats (bf16x3 convolutions and layer 0, f16e5 layers 1 and 2), two
    tiles of synthetic-read windows: the worst-tile RMS of p - p64 is at least 3x larger when a correction term is
    lost, while even the loss of the whole correction stays inside the 1e-3 contract that the other forward tests
    check - so only a budget on the f16e5 error itself can catch it."""
    import precision_emulation as pe
    from oracle import tf_graph
    x = pe.synthetic_windows(2 * 128)
    ref = tf_graph.forward_np(shipped_weights, x, np.float64)
    worst, max_dp = {}, {}
    for fault in ("", "-lo", "-hi", "-both"):
        p = pe.forward(shipped_weights, x, pe.engine_mm("ResNetRNN", "fp16+e5m2" + fault))
        worst[fault] = float(pe.tile_rms(p, ref).max())
        max_dp[fault] = float(np.abs(p - ref).max())
    for fault in ("-lo", "-hi", "-both"):
        assert worst[fault] >= 3 * worst[""], (fault, worst)
    assert max_dp["-both"] < 1e-3, max_dp


def test_bf16x3_one_tap_fault_budget(shipped_weights):
    """The shipped network in the engine's formats, two tiles of synthetic-read windows, with one tap of the first
    32 -> 32 convolution losing a bf16x3 correction pass: max |p - p64| stays inside the 1e-3 contract, while the
    worst-tile RMS is at least 3x that of the correct scheme - the budget of tests/test_gpu_precision_budgets.py
    sees such a fault, the contract tolerance does not."""
    import precision_emulation as pe
    from oracle import tf_graph
    x = pe.synthetic_windows(2 * 128)
    ref = tf_graph.forward_np(shipped_weights, x, np.float64)
    worst, max_dp = {}, {}
    for fault in ("", "-lo", "-hi"):
        bf3 = pe.confine(pe.make_mm("bf16x3" + fault), pe.make_mm("bf16x3"), {1})    # the middle tap
        p = pe.forward(shipped_weights, x, pe.engine_mm("ResNetRNN", bf16x3=bf3))
        worst[fault] = float(pe.tile_rms(p, ref).max())
        max_dp[fault] = float(np.abs(p - ref).max())
    for fault in ("-lo", "-hi"):
        assert worst[fault] >= 3 * worst[""], (fault, worst)
        assert max_dp[fault] < 1e-3, (fault, max_dp)
