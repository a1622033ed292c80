"""GPU: unit test of the fp16 + e5m2-correction MMA pair (operand packing, UMMA descriptors, mixed MMA kinds
on one TMEM accumulator) against a float64 matmul and a bit-level model of the scheme."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _f16e5_emulated(a, w, s=64.0):
    """Bit-level model of the fp16 + e5m2-correction product (tc_ptx.cuh, tests/tools/precision_emulation.py)."""
    import torch

    def rnd(x, dt):
        return torch.from_numpy(np.ascontiguousarray(x, np.float32)).to(dt).to(torch.float32).numpy().astype(np.float64)
    wh = rnd(w, torch.float16)
    ah = s * rnd(rnd(a, torch.float16) / s, torch.float16)     # the main plane stores fp16(fp16(a) / S)
    al, wl = a.astype(np.float64) - ah, w.astype(np.float64) - wh
    e5 = torch.float8_e5m2
    # the a_h / S byte is the TOP BYTE of fp16(a_h / S): e5m2 of the same value truncated to two mantissa bits
    top = (torch.from_numpy(np.ascontiguousarray(ah / s, np.float32)).to(torch.float16).view(torch.int16) & -256)
    ah_s = top.view(torch.float16).to(torch.float32).numpy().astype(np.float64)
    return ah @ wh + rnd(al * s, e5) @ rnd(wh / s, e5) + ah_s @ rnd(wl * s, e5)


@pytest.mark.parametrize("mode", [0, 1], ids=["ss", "ts"])
@pytest.mark.parametrize("k,n", [(16, 32), (32, 64), (64, 128)])
def test_f16e5_mma_pair(mode, k, n):
    """fp16 MMA + e5m2 correction MMA on one accumulator: operand byte orders, kind::f8f6f4 descriptors."""
    import torch
    from catfish_b200 import _cabi
    lib = _cabi.load_library()
    rng = np.random.default_rng(100 * k + n + mode)
    a = (rng.normal(0, 1, size=(128, k)) * rng.choice([1.0, 20.0], size=(128, 1))).astype(np.float32)
    a[:8] *= 1e-3                      # tiny rows: the corrections leave e5m2's normal range (checked loosely)
    w = rng.normal(0, 0.3, size=(k, n)).astype(np.float32)
    ad = torch.from_numpy(a).cuda()
    out = torch.full((128, n), float("nan"), dtype=torch.float32, device="cuda")
    _cabi.check(lib.cf_selftest_f16e5(0, ad.data_ptr(), k, n, w.ctypes.data, mode, out.data_ptr(),
                                      torch.cuda.current_stream().cuda_stream))
    got = out.cpu().numpy().astype(np.float64)
    exact = a.astype(np.float64) @ w.astype(np.float64)
    scale = np.abs(a).astype(np.float64) @ np.abs(w).astype(np.float64) + 1e-30
    assert np.isfinite(got).all()
    # the scheme's own accuracy: ~2^-14 of sum |a||w| (3e-5 after the sqrt(K) averaging)
    assert (np.abs(got - exact) / scale)[8:].max() < 6e-5
    assert (np.abs(got - exact) / scale)[:8].max() < 5e-4         # fp16 alone: 2^-11
    # and the device reproduces the bit-level model up to fp32 accumulation
    assert (np.abs(got - _f16e5_emulated(a, w)) / scale)[8:].max() < 2e-6
