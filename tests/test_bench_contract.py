"""bench.py: the reference arm runs without a GPU and prints one JSON line with the contract's keys (CPU);
--dump-outputs writes what the last timed step returned (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = [l for l in out.stdout.splitlines() if l.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["vs_baseline"] is None
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step(tmp_path):
    """The timed steps alternate two seeded batches, so --steps 1 and --steps 2 end on different batches; each dump
    equals a separate call on that batch, in float64."""
    import bench
    from catfish_b200 import infer, neural_network
    model = neural_network.load_network("ResNetRNN", None, 30000)
    n_reads = 16
    for steps in (1, 2):
        d = tmp_path / str(steps)
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--legs", "main", "--reads-per-step",
                              str(n_reads), "--steps", str(steps), "--warmup", "0", "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])["steps"] == steps
        got = {n: np.load(d / (n + ".npy")) for n in ("intervals", "interval_offsets", "read_ids")}
        assert all(v.dtype == np.float64 for v in got.values())
        raw, off = bench.make_batch(n_reads, 1000 + (steps - 1) % 2)
        iv, ioff = infer.infer_concatenated(raw, off, model)
        np.testing.assert_array_equal(got["read_ids"], np.arange(n_reads))
        np.testing.assert_array_equal(got["interval_offsets"], ioff)
        np.testing.assert_array_equal(got["intervals"], iv)
