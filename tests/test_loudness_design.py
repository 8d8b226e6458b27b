"""K-weighting coefficients of the loudness meters (pvgpu_kweighting_design; needs no GPU): ITU-R BS.1770-4's tables at 48 kHz,
and a Python restatement of libebur128's analog-prototype formulas at other rates."""
import math

import numpy as np
import pytest

# ITU-R BS.1770-4, Annex 1, Tables 1 and 2 (48 kHz): shelf b0, b1, b2, a1, a2; high-pass a1, a2 (its b is 1, -2, 1)
BS1770_48K = [1.53512485958697, -2.69169618940638, 1.19839281085285, -1.69065929318241, 0.73248077421585,
              -1.99004745483398, 0.99007225036621]


def kw_coeffs(sr):
    """The formulas pvgpu_kweighting_design restates, in plain Python (float64, the same order of operations)."""
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = math.tan(math.pi * f0 / sr)
    Vh = math.pow(10.0, G / 20.0)
    Vb = math.pow(Vh, 0.4996667741545416)
    a0 = 1.0 + K / Q + K * K
    shelf = [(Vh + Vb * K / Q + K * K) / a0, 2.0 * (K * K - Vh) / a0, (Vh - Vb * K / Q + K * K) / a0,
             2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = math.tan(math.pi * f0 / sr)
    a0 = 1.0 + K / Q + K * K
    return np.array(shelf + [2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0])


def test_kweighting_48k_is_bs1770_4(pvlib):
    import audiomod_b200 as A
    got = A.kweighting_design(48000)
    assert got.dtype == np.float64 and got.shape == (7,)
    assert np.max(np.abs(got - np.array(BS1770_48K))) < 1e-12, got


@pytest.mark.parametrize("sr", [8000, 16000, 22050, 32000, 44100, 48000, 88200, 96000, 192000])
def test_kweighting_other_rates_restate_the_formulas(pvlib, sr):
    import audiomod_b200 as A
    assert np.max(np.abs(A.kweighting_design(sr) - kw_coeffs(sr))) < 1e-12


def test_kweighting_rejects_bad_rates(pvlib):
    import audiomod_b200 as A
    from audiomod_b200 import _lib
    for sr in (0, -1, -48000):
        with pytest.raises(A.PvgpuError) as e:
            A.kweighting_design(sr)
        assert e.value.code == _lib.EINVAL
    assert pvlib.pvgpu_kweighting_design(48000, None) == _lib.EINVAL
