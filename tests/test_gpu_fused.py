"""The fused resynthesis kernel (k_synth_ola: inverse FFT + window + overlap-add in shared memory + normalisation + Speex
resampler, audiomod_b200/csrc/pv_fused.cu) against the split kernels it replaces and against the oracle.

The fused kernel adds the windowed frames into its shared-memory accumulator in slice order, i.e. with the reference's own
sequence of float additions (phasevocoderprocess.cc:1057-1064), so it must agree with the split path BIT FOR BIT in every
mode; extreme stretch ratios (dozens of overlapping frames), which the split kernels' tables refuse, are checked against the
oracle."""
import numpy as np
import pytest

from cases import CASES, ctor_args, make_input
from test_gpu_parity import assert_parity

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


def _run(A, xs, sr, ch, kw, fused, fpc=0):
    tr, st, mode, core, fft = ctor_args(kw)
    b = A.PhaseVocoderBatch(len(xs), max(x.shape[1] for x in xs), sr, ch, tr, st, mode, core, fft, kw.get("hopsize", 0))
    b.set_fused(fused)          # True / False; None = automatic
    if fpc:
        b.tune(frames_per_chunk=fpc)
    ys = b.run(xs)
    kt = b.stats()
    b.close()
    return ys, kt


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_fused_equals_split_bitwise(A, case):
    name, kw, sr, ch, secs, seed = case
    xs = [make_input(name, sr, ch, secs * f, seed + 3 * i) for i, f in enumerate((1.0, 0.37, 1.21))]
    yf, _ = _run(A, xs, sr, ch, kw, True)
    ys, _ = _run(A, xs, sr, ch, kw, False)
    for i, (a, b) in enumerate(zip(yf, ys)):
        assert a.shape == b.shape
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)), f"{name}[{i}]: fused and split kernels differ"


@pytest.mark.parametrize("fpc", [4, 8, 16, 32, 128])
def test_fused_chunking_is_invisible(A, fpc):
    """State carried between launches (accumulator tail, resampler history) and between rounds inside a launch."""
    sr = 44100
    xs = [make_input("x", sr, 2, 0.8 - 0.3 * i, 2100 + i) for i in range(3)]
    kw = dict(semitones=7.0, mode=0, coremode=1, fftsize=2048)
    want, _ = _run(A, xs, sr, 2, kw, True, 64)
    got, _ = _run(A, xs, sr, 2, kw, True, fpc)
    for a, b in zip(got, want):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("kw,sr,ch", [
    (dict(timeratio=0.1, mode=5, coremode=1, fftsize=2048), 44100, 1),     # outHop = N/60: ~60 frames overlap every sample
    (dict(timeratio=0.25, mode=5, coremode=1, fftsize=1024), 44100, 2),
    (dict(timeratio=4.0, mode=5, coremode=1, fftsize=2048), 44100, 1),
    (dict(timeratio=3.0, semitones=5.0, mode=0, coremode=1, fftsize=4096), 48000, 1),
    (dict(semitones=24.0, mode=0, coremode=1, fftsize=2048), 44100, 2),    # two octaves up: filt_len 256, oversample 4
    (dict(semitones=-24.0, mode=0, coremode=1, fftsize=2048), 44100, 1),   # two octaves down
    (dict(semitones=19.0, mode=2, coremode=1, fftsize=2048), 44100, 1),    # formant warp factor > 2: the Nyquist bin as a source (ADVICE r01)
    (dict(semitones=14.0, mode=1, coremode=1, fftsize=1024), 44100, 2),    # gender, 0.85 * scale > 1.9
])
def test_extreme_ratios_match_oracle(A, oracle, kw, sr, ch):
    xs = [make_input("x", sr, ch, 1.0 - 0.4 * i, 2200 + i) for i in range(2)]
    ref = [oracle.run_offline(x, sr, **kw) for x in xs]
    ys, _ = _run(A, xs, sr, ch, kw, True)
    for i, (y, r) in enumerate(zip(ys, ref)):
        assert_parity(y, r, f"{kw}[{i}]")
    # the streaming instance takes the same kernels with one CTA per channel row
    from test_gpu_parity import _cli_protocol
    tr, st, mode, core, fft = ctor_args(kw)
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft)
    y = _cli_protocol(pv, xs[1], sr, mode)
    pv.close()
    assert_parity(y, ref[1], f"{kw} stream")


def test_many_rows_grid_and_int16(A, oracle):
    """More rows than a CUDA grid's y dimension allows (the fused kernel puts rows on grid.x), int16 PCM rows."""
    from audiomod_b200.synth import synth_int16
    sr, S = 22050, 70000
    base = [synth_int16(2300 + i, sr, 0.06, 1) for i in range(5)]
    xs = [base[i % 5] for i in range(S)]
    b = A.PhaseVocoderBatch(S, xs[0].shape[1], sr, 1, 1.0, 3.0, 0, 1, 512)
    ys = b.run(xs, fmt=A.S16)
    b.close()
    for i in (0, 1, 2, 3, 4, 65535, 65536, S - 1):
        assert np.array_equal(ys[i], ys[i % 5])
    xf = (base[2].astype(np.float64) / 32768.0).astype(np.float32)
    r = oracle.run_offline(xf, sr, semitones=3.0, fftsize=512)
    want = np.clip(r * np.float32(32768.0), -32768.0, 32767.0).astype(np.int32)
    assert np.abs(ys[2].astype(np.int32) - want).max() <= 1


def test_many_channels_take_the_polar_core(A, oracle):
    """Six channels at FFT 4096: the Cartesian lock kernels would need more than the 200 KB shared-memory opt-in (ADVICE r01), so
    the serial polar core takes over -- same results, no launch failure."""
    sr, ch = 44100, 6
    x = make_input("x", sr, ch, 0.4, 2900)
    kw = dict(semitones=3.0, mode=0, coremode=1, fftsize=4096)
    (y,), _ = _run(A, [x], sr, ch, kw, None)
    assert_parity(y, oracle.run_offline(x, sr, **kw), "6 channels, FFT 4096")
