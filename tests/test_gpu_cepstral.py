"""The optional cepstral-envelope modes (PVGPU_GENDER_CEPSTRAL = 8, PVGPU_FORMANT_CEPSTRAL = 9; audiomod_b200/csrc/pv_cepstral.cu)
against the reference built with its commented-out formantShiftSlice calls switched on (oracle/_ref/pvref_drv_cep, see
oracle/Makefile; phasevocoderprocess.cc:824-840, 925-999).  Same bars as the parity modes: counts exact, >= 90 dB, <= 1e-4.

That checker is built from the reference's sources, which the repository does not carry, and the repository has no restatement
of the cepstral routine.  Without it the outputs are held to the same bars against tests/golden/cepstral_outputs.npz: this
project's own outputs, not the reference's, stored as each stream's length and its samples at cases.golden_cols
(tests/golden/make_gpu_golden.py, which checks them against the patched reference first wherever it is present).  They keep
the output from drifting beyond these bars on a checkout without the reference."""
import os

import numpy as np
import pytest

from cases import make_input
from test_gpu_parity import assert_parity, assert_parity_golden

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cepstral_outputs.npz")


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


CEPSTRAL_CASES = [               # mode, semitones, channels, FFT size, sample rate
    (8, 4.0, 1, 2048, 44100),     # male -> female: envelope warp 0.85
    (8, -4.0, 1, 2048, 44100),    # female -> male: 1.17
    (8, 7.0, 2, 1024, 44100),
    (8, -3.0, 2, 4096, 48000),
    (9, 4.0, 1, 2048, 44100),     # formant "preservation": identity warp (whiten and re-colour with the same envelope)
    (9, -5.0, 2, 512, 22050),
    (8, 5.0, 1, 8192, 44100),
]


def cepstral_inputs(ch, sr):
    return [make_input("x", sr, ch, 1.0 - 0.35 * i, 2500 + i) for i in range(2)]


def cepstral_key(mode, semitones, ch, fft, sr):
    return f"mode{mode}_{semitones:+g}st_{ch}ch_fft{fft}_{sr}"


@pytest.mark.parametrize("mode,semitones,ch,fft,sr", CEPSTRAL_CASES)
def test_cepstral_modes_match_patched_reference(A, oracle, mode, semitones, ch, fft, sr):
    xs = cepstral_inputs(ch, sr)
    if oracle.have_ref_cepstral():
        ref = [oracle.run_ref(x, sr, semitones=semitones, mode=mode - 7, fftsize=fft, cepstral=True) for x in xs]

        def check(y, i, what):
            assert_parity(y, ref[i], what)
    else:
        gold, key = np.load(GOLD), cepstral_key(mode, semitones, ch, fft, sr)

        def check(y, i, what):
            assert_parity_golden(y, gold, f"{key}__{i}", what)
    for fused in (False, True):
        b = A.PhaseVocoderBatch(len(xs), xs[0].shape[1], sr, ch, 1.0, semitones, mode, 1, fft)
        b.set_fused(fused)
        ys = b.run(xs)
        kt = b.stats()
        b.close()
        assert kt["kernel_launches"] > 0
        for i, y in enumerate(ys):
            check(y, i, f"cepstral mode {mode} {semitones:+g} st fft {fft} fused={fused} [{i}]")
    # the streaming instance
    from test_gpu_parity import _cli_protocol
    pv = A.phasevocoder(sr, ch, 1.0, semitones, mode, 1, fft)
    y = _cli_protocol(pv, xs[1], sr, mode)
    pv.close()
    check(y, 1, f"cepstral mode {mode} stream")


def test_cepstral_gender_differs_from_bin_warp(A):
    """Mode 8 is not mode 1: the envelope warp changes the timbre differently from the nearest-bin warp."""
    sr = 44100
    x = make_input("x", sr, 1, 0.5, 2600)
    outs = []
    for mode in (1, 8):
        b = A.PhaseVocoderBatch(1, x.shape[1], sr, 1, 1.0, 4.0, mode, 1, 2048)
        outs.append(b.run([x])[0])
        b.close()
    assert outs[0].shape == outs[1].shape and np.max(np.abs(outs[0] - outs[1])) > 1e-2


def test_cepstral_modes_need_a_tiled_fft_size(A):
    from audiomod_b200 import _lib
    with pytest.raises(A.PvgpuError) as e:
        A.PhaseVocoderBatch(1, 1000, 44100, 1, 1.0, 4.0, 8, 1, 256)
    assert e.value.code == _lib.EINVAL
