"""GPU: the fp16 + e5m2 ("f16e5") GRU layers held to their own error budget against float64.

f16e5 (DESIGN.md section 4) is one fp16 MMA plus one e5m2 correction MMA per K = 16 chunk.  Losing a correction
term moves the probabilities by a few 1e-4 at most, well inside the 1e-3 contract the other forward tests check
(tests/test_precision_emulation.py pins that blind spot), so this file bounds the error the format itself
leaves: the RMS of p - p64 over each tile of 128 windows, worst tile.  Window g of cf_infer_windows lies in tile
g // 128, the unit of the fused GRU kernel, whose CTAs run two chains of tiles: a fault on one chain or one ring
stage shows in that chain's tiles.  Each bound B keeps the correct build at most B / 1.5 and every mutant of
tests/tools/f16e5_mutants.patch (and -DCF_EXP=2 of profiles/r2_k4g_sensitivity.patch) at least 1.5 B; the
measured values are in DESIGN.md section 4.
"""
import os
import sys

import numpy as np
import pytest

from catfish_b200 import neural_network, weights
from oracle import tf_graph

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
import precision_emulation as pe  # noqa: E402

pytestmark = pytest.mark.gpu

# worst-tile RMS of p - p64; B200: correct 5.1e-6 / 6.9e-7, the least separated mutant 1.5e-5 / 3.5e-6
SHIPPED_BOUND = 9e-6         # shipped ResNetRNN
RNN_BOUND = 1.5e-6           # RNN-only, H = 64 x 3 layers
# tc_create runs f16e5 only while max |w| * kCandScale * kCorrScale < 60000 (the fp16 weight plane holds S w)
F16E5_WMAX = 60000.0 / (2.8853900817779268 * 64.0)
EDGE_KERNEL = "stack_bidirectional_rnn/cell_1/bidirectional_rnn/fw/gru_cell/candidate/kernel"


def _model(kind, w, **hpm):
    full = dict(weights.SHIPPED_HPARAMS)
    full.update(hpm)
    m = neural_network.build_model(kind, engine="auto", **full)
    m.set_weights(w)
    return m


def _tiles(n_windows):
    return -(-n_windows // 128)


def _check_budget(m, w, x, bound):
    """f16e5 on the tensor-core engine, finite probabilities, worst-tile RMS of p - p64 within `bound`."""
    assert m.operand_format == "f16e5", "the model runs %s, not f16e5" % m.operand_format
    p = m.infer(x)
    assert np.isfinite(p).all()
    tile = pe.tile_rms(p, tf_graph.forward_np(w, x, np.float64))
    worst = int(np.argmax(tile))
    assert tile[worst] <= bound, ("worst per-tile RMS of p - p64 is %.3e in tile %d of %d, bound %.1e"
                                  % (tile[worst], worst, tile.size, bound))


def test_shipped_resnetrnn_budget(shipped_weights):
    # 299 tiles, the last with 56 windows: on 148 SMs the 148 CTAs (74 per direction, a stride of 148 tiles) run two
    # or three tiles on each chain, and chain 1 of the CTAs that hold tiles 296..298 ends before their chain 0
    x = pe.synthetic_windows(298 * 128 + 56)
    assert _tiles(x.shape[0]) % 2 == 1 and x.shape[0] % 128
    _check_budget(_model("ResNetRNN", shipped_weights), shipped_weights, x, SHIPPED_BOUND)


def test_rnn_only_budget():
    # every layer f16e5 (layer 0's scalar input row is an exact rank-1 update); 151 tiles, the last with 40 windows
    hpm = dict(layer_size=64, n_layers=3)
    w = weights.random_init("RNN", seed=11, **hpm)
    x = np.random.default_rng(11).normal(0, 1.5, size=(150 * 128 + 40, 35, 1)).astype(np.float32)
    _check_budget(_model("RNN", w, **hpm), w, x, RNN_BOUND)


@pytest.mark.parametrize("frac", [0.99, 1.01])
def test_format_choice_at_fp16_weight_range(frac, shipped_weights):
    """One candidate weight of a 128-wide layer at 0.99 / 1.01 of the largest |w| f16e5 accepts: its fp16 plane
    value S w kCandScale is then within 1 % of 60000, near the top of fp16's range, in the x part (row 0) and in
    the state part (row 128 + 2)."""
    w = dict(shipped_weights)
    k = w[EDGE_KERNEL].copy()
    k[0, 5] = frac * F16E5_WMAX
    k[130, 9] = -frac * F16E5_WMAX
    w[EDGE_KERNEL] = k
    m = _model("ResNetRNN", w)
    if frac > 1:
        assert m.operand_format == "bf16x3"
        return
    _check_budget(m, w, pe.synthetic_windows(9 * 128 + 48), SHIPPED_BOUND)
