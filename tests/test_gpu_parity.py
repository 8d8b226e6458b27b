"""GPU parity tests (run with -m gpu on a B200).  Everything goes through the C ABI (libpvgpu.so via ctypes); the CPU
oracle and the golden vectors of the unmodified reference are only the checkers.

Bars (BASELINE.json north_star): frame/hop indexing and sample counts exact; audio max-abs error <= 1e-4 of full scale
and >= 90 dB SNR per channel.  Integer/bit work (the analysis FFT, magnitude, atan2f, princarg, robotic mode) is held
to bit-exactness.
"""
import ctypes as C
import os

import numpy as np
import pytest

from cases import CASES, ctor_args, golden_cols, make_input

pytestmark = pytest.mark.gpu

MAX_ABS = 1e-4
MIN_SNR_DB = 90.0
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pv_golden.npz")
_fp = C.POINTER(C.c_float)


def _p(a):
    return a.ctypes.data_as(_fp)


def assert_parity(y, ref, what=""):
    assert y.shape == ref.shape, f"{what}: sample count {y.shape} != reference {ref.shape}"
    for c in range(ref.shape[0]):
        err = y[c].astype(np.float64) - ref[c].astype(np.float64)
        mx = float(np.max(np.abs(err))) if err.size else 0.0
        e = float(np.sum(err ** 2))
        pw = float(np.sum(ref[c].astype(np.float64) ** 2))
        snr = 10 * np.log10(pw / e) if e > 0 and pw > 0 else float("inf")
        assert mx <= MAX_ABS, f"{what} ch{c}: max-abs {mx:.3e}"
        assert snr >= MIN_SNR_DB, f"{what} ch{c}: SNR {snr:.1f} dB"


def assert_parity_golden(y, gold, key, what=""):
    """assert_parity against an output stored as its length (key__n) and its samples at cases.golden_cols (key)."""
    n = int(gold[key + "__n"])
    assert y.shape[1] == n, f"{what}: sample count {y.shape[1]} != stored {n}"
    assert_parity(y[:, golden_cols(n)], gold[key], what)


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


# ---------------------------------------------------------------------------------------------------------------
# stage-level, bit-exact
# ---------------------------------------------------------------------------------------------------------------
def test_device_atan2f_bit_exact(A, pvlib, oracle):
    rng = np.random.default_rng(7)
    n = 1 << 21
    y = rng.standard_normal(n).astype(np.float32) * np.float32(10.0) ** rng.integers(-6, 3, n).astype(np.float32)
    x = rng.standard_normal(n).astype(np.float32) * np.float32(10.0) ** rng.integers(-6, 3, n).astype(np.float32)
    sp = np.array([0.0, -0.0, 1.0, -1.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 3.4e38, 0.4375, 0.6875, 1.1875, 2.4375], np.float32)
    yy, xx = np.meshgrid(sp, sp)
    y = np.concatenate([y, yy.ravel()]).astype(np.float32)
    x = np.concatenate([x, xx.ravel()]).astype(np.float32)
    out = np.zeros_like(y)
    assert pvlib.pvgpu_test_atan2f(0, y.size, _p(y), _p(x), _p(out)) == 0
    ref = oracle.host_atan2f(y, x)
    same = (out.view(np.uint32) == ref.view(np.uint32)) | (np.isnan(out) & np.isnan(ref))
    assert same.all(), f"{(~same).sum()} mismatches"


def test_device_princarg_bit_exact(A, pvlib, oracle):
    rng = np.random.default_rng(8)
    a = np.concatenate([rng.uniform(-40, 40, 200000), np.pi * np.arange(-9, 10), np.float32(np.pi) * np.arange(-9, 10),
                        rng.standard_normal(1000) * 1e-6, [0.0, -0.0, 700.25, -1234.5]]).astype(np.float64)
    out = np.zeros_like(a)
    dp = C.POINTER(C.c_double)
    assert pvlib.pvgpu_test_princarg(0, a.size, a.ctypes.data_as(dp), out.ctypes.data_as(dp)) == 0
    ref = np.array([oracle.lib().pvo_princarg(float(v)) for v in a])
    assert np.array_equal(out.view(np.uint64), ref.view(np.uint64))


@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 8192])
def test_forward_polar_bit_exact(A, pvlib, oracle, n):
    """Hann + fftshift + KissFFT-order real FFT + sqrtf/atan2f: every bin bit-identical (SURVEY 7-1)."""
    from audiomod_b200.synth import synth
    rng = np.random.default_rng(n)
    nf = 12
    frames = np.stack([synth(n + i, 44100, n / 44100.0 + 0.01, 1)[0, :n] for i in range(nf - 3)]
                      + [rng.standard_normal(n).astype(np.float32) * 0.3, np.zeros(n, np.float32),
                         np.full(n, 0.25, np.float32)]).astype(np.float32)
    frames = np.ascontiguousarray(frames)
    h = n // 2 + 1
    mag, ph = np.zeros((nf, h), np.float32), np.zeros((nf, h), np.float32)
    assert pvlib.pvgpu_test_forward_polar(0, n, nf, _p(frames), _p(mag), _p(ph)) == 0
    for i in range(nf):
        rm, rp, _ = oracle.forward_polar(frames[i])
        assert np.array_equal(mag[i].view(np.uint32), rm.view(np.uint32)), f"magnitude differs, frame {i}"
        assert np.array_equal(ph[i].view(np.uint32), rp.view(np.uint32)), f"phase differs, frame {i}"


@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 8192])
def test_inverse_polar_close(A, pvlib, oracle, n):
    rng = np.random.default_rng(n + 1)
    nf, h = 6, n // 2 + 1
    mag = (np.abs(rng.standard_normal((nf, h))) * 50).astype(np.float32)
    ph = rng.uniform(-np.pi, np.pi, (nf, h)).astype(np.float32)
    out = np.zeros((nf, n), np.float32)
    assert pvlib.pvgpu_test_inverse_polar(0, n, nf, _p(mag), _p(ph), _p(out)) == 0
    for i in range(nf):
        ref = oracle.inverse_polar(mag[i] * np.float32(1.0 / n), ph[i], n)  # the device stage includes the 1/N scale
        assert np.max(np.abs(out[i] - ref)) <= 2e-6 * max(1.0, float(np.max(np.abs(ref))))


# ---------------------------------------------------------------------------------------------------------------
# whole path: batch entry point
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_batch_matches_reference_golden(A, gold, case):
    """Golden vectors of the unmodified reference; three ragged copies exercise per-stream lengths."""
    name, kw, sr, ch, secs, seed = case
    x = make_input(name, sr, ch, secs, seed)
    tr, st, mode, core, fft = ctor_args(kw)
    b = A.PhaseVocoderBatch(1, x.shape[1], sr, ch, tr, st, mode, core, fft)
    (y,) = b.run([x])
    assert b.stats()["kernel_launches"] > 0
    b.close()
    assert_parity(y, gold[name + "__out"], name)
    if mode == A.ROBOTIC:
        assert np.array_equal(y.view(np.uint32), gold[name + "__out"].view(np.uint32))


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_batch_ragged_matches_oracle(A, oracle, case):
    name, kw, sr, ch, secs, seed = case
    tr, st, mode, core, fft = ctor_args(kw)
    xs = [make_input(name, sr, ch, secs * f, seed + 11 * i) for i, f in enumerate((1.3, 0.31, 0.9, 0.05))]
    ref = [oracle.run_offline(x, sr, **kw) for x in xs]
    b = A.PhaseVocoderBatch(len(xs), max(x.shape[1] for x in xs), sr, ch, tr, st, mode, core, fft)
    b.tune(frames_per_chunk=7)   # odd chunking: state must carry across chunk boundaries
    ys = b.run(xs)
    b.close()
    for i, (y, r) in enumerate(zip(ys, ref)):
        assert_parity(y, r, f"{name}[{i}]")


@pytest.mark.parametrize("kw,sr,ch", [
    (dict(semitones=5.0, mode=0, coremode=1, fftsize=256), 22050, 2),       # sizes outside 512..8192 take the generic kernels
    (dict(timeratio=1.25, mode=5, coremode=1, fftsize=16384), 48000, 1),
    (dict(semitones=-3.0, mode=2, fftsize=1000), 44100, 1),                 # rounded up to 1024 like the reference
    (dict(semitones=2.0, mode=0, coremode=1, fftsize=2048, hopsize=300), 44100, 2),   # explicit analysis hop
    (dict(timeratio=0.5, mode=5, coremode=0, fftsize=1024, hopsize=128), 44100, 1),
    (dict(semitones=24.0, mode=0, coremode=1, fftsize=1024), 44100, 1),     # two octaves up: oversample 4 table
    (dict(semitones=-12.0, mode=0, coremode=1, fftsize=2048), 44100, 1),    # octave down: up-sampling resampler
    (dict(semitones=3.0, mode=0, coremode=1, fftsize=8192), 44100, 2),      # phase-locked core at 8 bins per thread (up to 3 peaks each)
    (dict(semitones=-2.0, mode=0, coremode=1, fftsize=512), 22050, 1),      # smallest templated size: two warps per stream
    (dict(semitones=5.0, mode=2, coremode=1, fftsize=4096), 48000, 2),      # formant warp on the Cartesian pipeline, 512 threads
    (dict(semitones=-5.0, mode=1, coremode=1, fftsize=1024), 44100, 2),     # gender change, expanding direction
])
def test_unusual_sizes_and_hops(A, oracle, kw, sr, ch):
    xs = [make_input("x", sr, ch, 0.7 - 0.2 * i, 800 + i) for i in range(2)]
    ref = [oracle.run_offline(x, sr, **kw) for x in xs]
    tr, st, mode, core, fft = ctor_args(kw)
    b = A.PhaseVocoderBatch(2, xs[0].shape[1], sr, ch, tr, st, mode, core, fft, kw.get("hopsize", 0))
    ys = b.run(xs)
    b.close()
    for i, (y, r) in enumerate(zip(ys, ref)):
        assert_parity(y, r, f"{kw}[{i}]")
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft, kw.get("hopsize", 0))
    y = _cli_protocol(pv, xs[1], sr, mode)
    pv.close()
    assert_parity(y, ref[1], f"{kw} stream")


def test_empty_and_tiny_streams(A, oracle):
    sr = 44100
    xs = [np.zeros((1, 0), np.float32), make_input("x", sr, 1, 0.001, 1), make_input("x", sr, 1, 0.05, 2), make_input("x", sr, 1, 0.3, 3)]
    ref = [oracle.run_offline(x, sr, semitones=7.0) for x in xs]
    b = A.PhaseVocoderBatch(len(xs), max(x.shape[1] for x in xs), sr, 1, 1.0, 7.0)
    ys = b.run(xs)
    b.close()
    for i, (y, r) in enumerate(zip(ys, ref)):
        assert_parity(y, r, f"tiny[{i}]")


@pytest.mark.parametrize("kw,sr,ch", [
    (dict(semitones=7.0, mode=0, coremode=1, fftsize=2048), 44100, 1),
    (dict(semitones=4.0, mode=0, coremode=1, fftsize=2048), 44100, 2),
    (dict(timeratio=1.5, mode=5, coremode=1, fftsize=1024), 48000, 2),
    (dict(semitones=-3.0, mode=0, coremode=0, fftsize=2048), 44100, 2),
])
def test_silence_gaps_match_oracle(A, oracle, kw, sr, ch):
    """Digital silence makes frames without any spectral peak: the phase-locked core falls back to the classic per-bin
    propagation (phasevocoderprocess.cc:617-636) and later links peaks to a state left by it.  Streams that start with
    silence, contain gaps (in one channel only, too) and end in silence must still match the oracle; the chunk size is
    odd so that the transitions also cross launch boundaries."""
    n = int(0.9 * sr)
    xs = []
    for i in range(4):
        x = make_input("x", sr, ch, 0.9, 900 + i)[:, :n].copy()
        a, b = int((0.15 + 0.1 * i) * sr), int((0.35 + 0.12 * i) * sr)
        if i == 0:
            x[:, :a] = 0.0                    # leading silence: the pass-through first frame is all zeros
        elif i == 1:
            x[:, a:b] = 0.0                   # a gap in every channel
        elif i == 2:
            x[ch - 1, a:b] = 0.0              # a gap in the last channel only (peak lists are shared by the channels)
            x[:, int(0.7 * sr):] = 0.0        # and a silent tail
        else:
            x[:, a:a + 3000] = 0.0            # a gap of about one window: only a few peak-free frames
            x[0, b:b + 2048] = 0.0
        xs.append(x)
    ref = [oracle.run_offline(x, sr, **kw) for x in xs]
    tr, st, mode, core, fft = ctor_args(kw)
    b = A.PhaseVocoderBatch(len(xs), n, sr, ch, tr, st, mode, core, fft)
    b.tune(frames_per_chunk=5)
    ys = b.run(xs)
    b.close()
    for i, (y, r) in enumerate(zip(ys, ref)):
        assert_parity(y, r, f"silence {kw}[{i}]")
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft)
    y = _cli_protocol(pv, xs[1], sr, mode)
    pv.close()
    assert_parity(y, ref[1], f"silence {kw} stream")


@pytest.mark.parametrize("kw", [
    dict(semitones=4.0, mode=0, coremode=1, fftsize=1024),
    dict(timeratio=1.3, mode=5, coremode=1, fftsize=2048),
    dict(semitones=-2.0, mode=2, coremode=1, fftsize=2048),
])
def test_three_channels(A, oracle, kw):
    """More than two channels: the peak lists are still shared by all channels of a stream in processing order
    (phasevocoderimpl.h:237-238); the kernels' run-time channel-count variants must follow it."""
    sr, ch = 44100, 3
    xs = [make_input("x", sr, ch, 0.5 - 0.1 * i, 700 + i) for i in range(2)]
    xs[1][1, 4000:9000] = 0.0   # a silent stretch in the middle channel only
    ref = [oracle.run_offline(x, sr, **kw) for x in xs]
    tr, st, mode, core, fft = ctor_args(kw)
    b = A.PhaseVocoderBatch(2, xs[0].shape[1], sr, ch, tr, st, mode, core, fft)
    b.tune(frames_per_chunk=9)
    ys = b.run(xs)
    b.close()
    for i, (y, r) in enumerate(zip(ys, ref)):
        assert_parity(y, r, f"3ch {kw}[{i}]")
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft)
    y = _cli_protocol(pv, xs[0], sr, mode)
    pv.close()
    assert_parity(y, ref[0], f"3ch {kw} stream")


def test_batch_invariance_bitwise(A):
    """A stream's result does not depend on what else is in the batch nor on chunk / group tuning."""
    sr = 44100
    xs = [make_input("x", sr, 2, 0.4, 40 + i) for i in range(6)]
    outs = []
    for fpc, rpg, order in ((64, 0, range(6)), (5, 4, reversed(range(6))), (1, 2, range(6))):
        order = list(order)
        b = A.PhaseVocoderBatch(6, xs[0].shape[1], sr, 2, 1.0, 4.0)
        b.tune(fpc, rpg)
        ys = b.run([xs[i] for i in order])
        b.close()
        outs.append({i: ys[j] for j, i in enumerate(order)})
    for i in range(6):
        assert np.array_equal(outs[0][i], outs[1][i]) and np.array_equal(outs[0][i], outs[2][i])


def test_stereo_identical_channels_quirk(A, oracle):
    """The reference shares the peak lists between the channels of a stream, so with L == R channel 0 equals the mono
    result bit for bit while channel 1 does not (SURVEY 7-2).  The GPU path must reproduce exactly that."""
    sr = 44100
    m = make_input("x", sr, 1, 0.5, 77)
    st = np.concatenate([m, m], axis=0)
    bm = A.PhaseVocoderBatch(1, m.shape[1], sr, 1, 1.0, 4.0)
    (ym,) = bm.run([m])
    bm.close()
    bs = A.PhaseVocoderBatch(1, m.shape[1], sr, 2, 1.0, 4.0)
    (ys,) = bs.run([st])
    bs.close()
    assert np.array_equal(ys[0], ym[0])
    rs = oracle.run_offline(st, sr, semitones=4.0)
    assert_parity(ys, rs, "L==R")
    assert not np.array_equal(rs[0], rs[1])


def test_time_sliced_host_pipeline(A, oracle):
    """Equal-length streams in one contiguous 2-D host array take the time-sliced pipeline (column-block copies overlapping
    the frame chunks); it must give bit-identical samples to the row-group pipeline and match the oracle."""
    sr, S, ch = 44100, 6, 2
    xs = [make_input("x", sr, ch, 0.6, 700 + i) for i in range(S)]
    n = xs[0].shape[1]
    X = np.ascontiguousarray(np.concatenate(xs, axis=0))          # [S*ch, n], evenly spaced rows
    res = {}
    for name, kw in (("time", dict(frames_per_chunk=16)), ("rows", dict(frames_per_chunk=16, rows_per_group=4))):
        b = A.PhaseVocoderBatch(S, n, sr, ch, 1.0, 7.0)
        b.tune(**kw)
        n_out = b.plan(n)
        Y = np.full((S * ch, int(n_out[0]) + 5), 9.0, np.float32)  # padded pitch: bytes past n_out must stay untouched
        b.run_host_rows([X[r] for r in range(S * ch)], [Y[r] for r in range(S * ch)])
        st = b.stats()
        b.close()
        assert np.all(Y[:, int(n_out[0]):] == 9.0)
        assert st["h2d_bytes"] == X.size * 4 and st["d2h_bytes"] == S * ch * int(n_out[0]) * 4
        res[name] = Y[:, :int(n_out[0])].copy()
    assert np.array_equal(res["time"], res["rows"])
    for i in range(S):
        assert_parity(res["time"][i * ch:(i + 1) * ch], oracle.run_offline(xs[i], sr, semitones=7.0), f"ts[{i}]")


def test_int16_pcm_rows(A, oracle):
    """int16 PCM in and out (the reference CLI's WAV format): device-side conversions follow main/wavfile.cc:733-752 and
    :1294-1306,1508-1526 (x * 32768, clamp, truncate toward zero).  A 1e-7 float difference can flip the truncation by 1 LSB."""
    from audiomod_b200.synth import synth_int16
    sr = 44100
    for ch, kw in ((1, dict(semitones=7.0)), (2, dict(timeratio=1.5, mode=5, fftsize=4096))):
        pcm = [synth_int16(900 + i, sr, 0.5 - 0.1 * i, ch) for i in range(3)]
        b = A.PhaseVocoderBatch(3, pcm[0].shape[1], sr, ch, kw.get("timeratio", 1.0), kw.get("semitones", 0.0), kw.get("mode", 0), 1,
                                kw.get("fftsize", 2048))
        ys = b.run(pcm, fmt=A.S16)
        b.close()
        for x, y in zip(pcm, ys):
            xf = (x.astype(np.float64) * (1.0 / 32768.0)).astype(np.float32)
            r = oracle.run_offline(xf, sr, **kw)
            want = np.clip(r * np.float32(32768.0), -32768.0, 32767.0).astype(np.int32)   # astype truncates toward zero
            assert y.dtype == np.int16 and y.shape == want.shape
            d = np.abs(y.astype(np.int32) - want)
            assert d.max() <= 1 and (d == 0).mean() > 0.995


def test_device_resident_entry_point(A, oracle):
    """pvgpu_batch_run_device with caller-owned device buffers (torch tensors) on torch's current stream."""
    torch = pytest.importorskip("torch")
    sr, S = 44100, 5
    xs = [make_input("x", sr, 1, 0.3, 300 + i) for i in range(S)]
    n = xs[0].shape[1]
    b = A.PhaseVocoderBatch(S, n, sr, 1, 1.0, 7.0)
    n_out = b.plan(n)
    stride, ostride = (n + 3) & ~3, (int(n_out.max()) + 3) & ~3
    ref = [oracle.run_offline(x, sr, semitones=7.0) for x in xs]
    host = torch.from_numpy(np.concatenate(xs, axis=0)).pin_memory()
    # (a) the legacy default stream (handle 0, what torch.cuda.current_stream() is by default), (b) an explicit non-blocking
    # stream: in both the fill kernels queued just before the call and the read-back queued just after it must be ordered
    # around the run without any host synchronisation in between (ADVICE r01: the null handle used to mean "own stream")
    for st in (torch.cuda.current_stream(), torch.cuda.Stream()):
        with torch.cuda.stream(st):
            d_in = torch.zeros((S, stride), dtype=torch.float32, device="cuda")
            d_out = torch.full((S, ostride), 7.0, dtype=torch.float32, device="cuda")
            d_in[:, :n].copy_(host, non_blocking=True)
            b.run_device(d_in.data_ptr(), stride, d_out.data_ptr(), ostride, st.cuda_stream)
            y_dev = d_out.clone()           # same stream, after the run
            d_in.zero_()                    # would corrupt the run if it were not ordered after it
        b.synchronize()
        st.synchronize()
        y = y_dev.cpu().numpy()
        for i in range(S):
            assert_parity(y[i:i + 1, :int(n_out[i])], ref[i], f"dev[{i}]")
    b.close()


# ---------------------------------------------------------------------------------------------------------------
# streaming instance: the modbase / modbase_offline calls
# ---------------------------------------------------------------------------------------------------------------
def _cli_protocol(pv, x, sr, mode, block=0):
    B = block or max(480, sr // 100)
    n, ch = x.shape[1], x.shape[0]
    chunks, produced = [], 0
    for i in range(0, n, B):
        pv.processInData(x[:, i:i + B])
        y = pv.getOutData(pv.getOutSamples())
        chunks.append(y.copy())
        produced += y.shape[1]
    if mode != 5:
        z = np.zeros((ch, B), np.float32)
        while produced < n:
            pv.processInData(z)
            y = pv.getOutData(pv.getOutSamples())
            if n - produced <= y.shape[1]:
                y = y[:, :n - produced]
            chunks.append(y.copy())
            produced += y.shape[1]
    return np.concatenate(chunks, axis=1)


@pytest.mark.parametrize("case", [c for c in CASES if c[0] in ("cfg1_shift_p4_stereo", "cfg2_stretch_1p5_4096", "cfg3_gender_m4",
                                                               "cfg5_whisper_1024", "cfg5_chord_4096", "core0_shift_p3_stereo",
                                                               "constant_1024", "core2_octave_up")],
                         ids=lambda c: c[0])
def test_streaming_offline_api_matches_golden(A, gold, case):
    name, kw, sr, ch, secs, seed = case
    x = make_input(name, sr, ch, secs, seed)
    tr, st, mode, core, fft = ctor_args(kw)
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft)
    y = _cli_protocol(pv, x, sr, mode)
    pv.close()
    assert_parity(y, gold[name + "__out"], name)


@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg5_robotic_512"])
def test_streaming_process_block_matches_golden(A, gold, name):
    """In-place processBlock / outputReady loop of the SDK (README usage, main.cc:562-571)."""
    kw, sr, ch, secs, seed = next((c[1], c[2], c[3], c[4], c[5]) for c in CASES if c[0] == name)
    x = make_input(name, sr, ch, secs, seed)
    tr, st, mode, core, fft = ctor_args(kw)
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft)
    B = max(480, sr // 100)
    kept, dropped = [], 0
    for i in range(0, x.shape[1], B):
        blk = np.ascontiguousarray(x[:, i:i + B])
        before = blk.copy()
        pv.processBlock(blk)
        if pv.outputReady():
            kept.append(blk)
        else:
            dropped += 1
            assert np.array_equal(blk, before), "buffer must be untouched when output is not ready"
    pv.close()
    y = np.concatenate(kept, axis=1)
    assert dropped > 0
    assert_parity(y, gold[name + "__rt"], name + " rt")


def test_streaming_odd_block_sizes(A, oracle):
    """Arbitrary call sizes (0, 1, primes, several windows at once) give the oracle's per-call counts and samples."""
    sr = 44100
    x = make_input("x", sr, 2, 0.7, 91)
    pv = A.phasevocoder(sr, 2, 1.0, -3.0, 0, 1, 1024)
    st = oracle.OracleStream(sr, 2, 1.0, -3.0, 0, 1, 1024)
    sizes = [0, 1, 7, 1023, 1, 4099, 0, 480, 2500, 311]
    pos, k = 0, 0
    while pos < x.shape[1]:
        n = min(sizes[k % len(sizes)], x.shape[1] - pos)
        k += 1
        blk = np.ascontiguousarray(x[:, pos:pos + n])
        pv.processInData(blk)
        st.processInData(blk)
        assert pv.getOutSamples() == st.getOutSamples()
        take = pv.getOutSamples() if k % 3 else pv.getOutSamples() // 2   # sometimes leave samples in the ring
        a, b = pv.getOutData(take), st.getOutData(take)
        assert_parity(a, b, f"call {k}")
        pos += n
    pv.close()
    st.close()


def test_unknown_mode_does_nothing(A):
    pv = A.phasevocoder(44100, 1, 1.0, 0.0, 42, 1, 2048)
    pv.processInData(np.zeros((1, 4800), np.float32))
    assert pv.getOutSamples() == 0
    pv.close()


# ---------------------------------------------------------------------------------------------------------------
# full-size workload: size-independent properties (the oracle would take minutes here)
# ---------------------------------------------------------------------------------------------------------------
def test_full_length_streams_properties(A, oracle):
    """BASELINE config 4 shape at reduced stream count: 10 s streams, +7 semitones, FFT 2048.  Output length equals the
    input length for every stream, duplicate streams are bit-identical, and three streams are checked against the
    oracle end to end."""
    sr, secs, S = 44100, 10.0, 24
    base = [make_input("x", sr, 1, secs, 4000 + i) for i in range(3)]
    xs = [base[i % 3] for i in range(S)]
    b = A.PhaseVocoderBatch(S, xs[0].shape[1], sr, 1, 1.0, 7.0)
    ys = b.run(xs)
    st = b.stats()
    b.close()
    assert st["slices"] == A.plan_counts(xs[0].shape[1], sr, 1, 1.0, 7.0)["n_slices"]
    for i in range(S):
        assert ys[i].shape == (1, 441000)
        assert np.array_equal(ys[i], ys[i % 3])
        assert np.isfinite(ys[i]).all()
    for i in range(3):
        assert_parity(ys[i], oracle.run_offline(base[i], sr, semitones=7.0), f"full[{i}]")
