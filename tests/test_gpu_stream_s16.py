"""Streaming instances and live batches fed int16 PCM rows (pvgpu_*_s16; Python phasevocoder(..., fmt=S16)).

Contract: every stream of an int16 instance produces exactly what a float32 instance produces with the same calls when the
float32 instance is fed s / 32768 and its output is quantised by the reference's WAV writer rule, (short)(int)clamp(x * 32768.f,
-32768, 32767).  Checked bit for bit, call by call, against float32 instances of this library: the kernels are the same, only
the load and the store convert."""
import ctypes as C

import numpy as np
import pytest

from cases import CASES, ctor_args

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


def _quant(y):
    """The reference WAV writer's rule in numpy: float32 multiply, clip, truncate toward zero."""
    y = np.asarray(y, dtype=np.float32)
    return np.clip(y * np.float32(32768.0), -32768.0, 32767.0).astype(np.int32).astype(np.int16)


def _pcm(n, sr, ch, seed, S):
    from audiomod_b200.synth import synth_int16
    return np.ascontiguousarray(np.concatenate([synth_int16(seed + 11 * i, sr, n / sr, ch)[:, :n] for i in range(S)], axis=0))


def _f32(x16):
    from audiomod_b200.synth import int16_to_float
    return np.ascontiguousarray(int16_to_float(x16))


SIZES = [480, 480, 1, 0, 2048, 311, 4099, 480]


def _compare_call_by_call(A, sr, ch, args, X16, S, label):
    """Feeds an int16 and a float32 live batch the same calls (odd sizes, partial retrieves); returns (int16 output, samples
    quantised to the int16 limits)."""
    n = X16.shape[1]
    Xf = _f32(X16)
    s16 = A.phasevocoder(sr, ch, *args, streams=S, fmt=A.S16)
    f32 = A.phasevocoder(sr, ch, *args, streams=S)
    pos, k, outs = 0, 0, []
    while pos < n:
        m = min(SIZES[k % len(SIZES)], n - pos)
        k += 1
        s16.processInData(np.ascontiguousarray(X16[:, pos:pos + m]))
        f32.processInData(np.ascontiguousarray(Xf[:, pos:pos + m]))
        avail = f32.getOutSamples()
        assert s16.getOutSamples() == avail, f"{label}: call {k}"
        take = avail if k % 3 else avail // 2                       # sometimes leave samples in the rings
        a, b = s16.getOutData(take), f32.getOutData(take)
        assert a.dtype == np.int16 and a.shape == b.shape == (S * ch, b.shape[1]), f"{label}: call {k}"
        assert np.array_equal(a, _quant(b)), f"{label}: call {k}: int16 output differs from the quantised float32 output"
        outs.append(a)
        pos += m
    s16.close()
    f32.close()
    y = np.concatenate(outs, axis=1)
    assert y.shape[1] > 0
    return y, int(np.count_nonzero((y == 32767) | (y == -32768)))


S16_CASES = ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo", "cfg3_formant_p4", "cfg3_gender_m4", "cfg5_robotic_512", "cfg5_whisper_1024",
             "cfg5_vocoder_2048", "cfg5_chord_4096", "cfg2_stretch_1p5_4096", "core0_shift_p3_stereo", "core2_octave_up", "shift_m5_1024"]
EXTRA = [("formant_cepstral_p4", dict(semitones=4.0, mode=9, fftsize=2048), 44100, 1, 0.5, 6001),   # mode 9: the cepstral envelope kernel
         ("shift_p5_fft256", dict(semitones=5.0, mode=0, coremode=1, fftsize=256), 44100, 1, 0.4, 6002)]  # generic one-CTA-per-frame kernels
ALL = [c for c in CASES if c[0] in S16_CASES] + EXTRA


@pytest.mark.parametrize("case", ALL, ids=[c[0] for c in ALL])
def test_s16_live_batch_equals_quantised_f32(A, case):
    name, kw, sr, ch, secs, seed = case
    S = 5
    n = int(sr * min(secs, 0.5))
    _compare_call_by_call(A, sr, ch, ctor_args(kw), _pcm(n, sr, ch, seed, S), S, name)


def test_s16_store_saturates(A):
    """Output beyond +-1 is clamped to 32767 / -32768, not wrapped.  The synthetic input peaks well below full scale, so this feeds
    it 16x louder (clipped to int16) through the vocoder and the +7 semitone shift, whose outputs then exceed +-1."""
    saturated = 0
    for name in ("cfg5_vocoder_2048", "cfg4_shift_p7_mono"):
        _, kw, sr, ch, secs, seed = next(c for c in CASES if c[0] == name)
        n = int(sr * min(secs, 0.5))
        loud = np.clip(_pcm(n, sr, ch, seed, 3).astype(np.int32) * 16, -32768, 32767).astype(np.int16)
        saturated += _compare_call_by_call(A, sr, ch, ctor_args(kw), loud, 3, name + " at full scale")[1]
    assert saturated > 0, "expected saturated samples"


@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo"])
def test_s16_fused_back_end(A, monkeypatch, name):
    """The fused inverse-FFT + overlap-add + resampler kernel stores int16 through the same rule."""
    monkeypatch.setenv("PVGPU_FUSED", "1")   # read when an instance is created
    name, kw, sr, ch, secs, seed = next(c for c in CASES if c[0] == name)
    n = int(sr * min(secs, 0.5))
    _compare_call_by_call(A, sr, ch, ctor_args(kw), _pcm(n, sr, ch, seed, 5), 5, name + " fused")


def test_s16_fused_selected_automatically(A):
    """timeratio 0.1 overlaps more frames than the split kernels' tables hold: the fused kernel is chosen on its own."""
    kw, sr, ch = dict(timeratio=0.1, mode=5, coremode=1, fftsize=2048), 44100, 1
    _compare_call_by_call(A, sr, ch, ctor_args(kw), _pcm(int(0.4 * sr), sr, ch, 6100, 3), 3, "timeratio 0.1")


def test_s16_process_block_protocol(A):
    """processBlock / outputReady in place on int16 rows, 64 streams: the same ready flags as the float32 instance, buffers untouched
    while not ready, ready blocks equal the quantised float32 blocks."""
    sr, S, B = 44100, 64, 480
    n = B * 60
    X16 = _pcm(n, sr, 1, 7000, S)
    Xf = _f32(X16)
    s16 = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S, fmt=A.S16)
    f32 = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S)
    ready_blocks = 0
    for pos in range(0, n, B):
        b16 = np.ascontiguousarray(X16[:, pos:pos + B])
        before = b16.copy()
        b32 = np.ascontiguousarray(Xf[:, pos:pos + B])
        s16.processBlock(b16)
        f32.processBlock(b32)
        assert s16.outputReady() == f32.outputReady(), f"block at {pos}"
        if s16.outputReady():
            ready_blocks += 1
            assert np.array_equal(b16, _quant(b32)), f"block at {pos}"
        else:
            assert np.array_equal(b16, before), "buffers must be untouched while output is not ready"
    assert ready_blocks > 40
    s16.close()
    f32.close()


def test_s16_large_live_batch_uses_the_copy_pool(A):
    """320 rows start the row-copy pool (16-bit non-temporal packing on several threads, int16 ring FIFO).  Calls of odd size that
    complete no slice leave the pending samples ending on a 2-byte boundary, so the next call's samples are packed behind them at
    that alignment; one call moves more than the pool's threshold of 256 K samples.  Sampled streams equal their own single int16 instances."""
    from audiomod_b200.synth import synth_int16
    sr, S = 44100, 320
    n = 480 * 25 + 4099 + 64
    base = synth_int16(8100, sr, n / sr, 1)[:, :n]
    X = np.ascontiguousarray(np.concatenate([np.roll(base, 37 * i, axis=1) for i in range(S)], axis=0))
    live = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S, fmt=A.S16)
    picks = (0, 1, 77, S - 1)
    singles = [A.phasevocoder(sr, 1, 1.0, 7.0, fmt=A.S16) for _ in picks]
    sizes = [480] * 10 + [1, 3, 0, 5, 4099, 1, 0, 480, 311, 7] + [480] * 12
    pos = 0
    for m in sizes:
        m = min(m, n - pos)
        live.processInData(np.ascontiguousarray(X[:, pos:pos + m]))
        avail = live.getOutSamples()
        Y = live.getOutData(avail)
        assert Y.dtype == np.int16
        for j, i in enumerate(picks):
            singles[j].processInData(np.ascontiguousarray(X[i:i + 1, pos:pos + m]))
            assert singles[j].getOutSamples() == avail
            assert np.array_equal(Y[i:i + 1], singles[j].getOutData(avail)), f"stream {i} at {pos}"
        pos += m
    live.close()
    for pv in singles:
        pv.close()


@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo", "cfg5_whisper_1024", "cfg2_stretch_1p5_4096"])
def test_s16_device_rows_equal_host_rows(A, name):
    """processInDataDevice / getOutDataDevice on int16 device rows whose pointers are only 2-byte aligned (odd element offsets and
    pitches): the same counts and samples as the int16 host-row calls, everything on one CUDA stream."""
    import torch
    _, kw, sr, ch, secs, seed = next(c for c in CASES if c[0] == name)
    args = ctor_args(kw)
    S = 6
    n = int(sr * min(secs, 0.5))
    X = _pcm(n, sr, ch, seed, S)
    R = S * ch
    pitch_in, pitch_out = n + 3, (1 << 16) + 1
    Xp = np.zeros((R, pitch_in), np.int16)
    Xp[:, 1:n + 1] = X
    host = A.phasevocoder(sr, ch, *args, streams=S, fmt=A.S16)
    dev = A.phasevocoder(sr, ch, *args, streams=S, fmt=A.S16)
    stream = torch.cuda.Stream()
    dX = torch.from_numpy(Xp).cuda()
    dY = torch.zeros((R, pitch_out), dtype=torch.int16, device="cuda")
    pos, k, w, got_host = 0, 0, 0, []
    with torch.cuda.stream(stream):
        while pos < n:
            m = min(SIZES[k % len(SIZES)], n - pos)
            k += 1
            host.processInData(np.ascontiguousarray(X[:, pos:pos + m]))
            avail = host.getOutSamples()
            take = avail if k % 3 else avail // 2
            got_host.append(host.getOutData(take))
            dev.processInDataDevice(dX.data_ptr() + 2 * (1 + pos), pitch_in, m, stream.cuda_stream)
            assert dev.getOutSamples() == avail, f"{name}: call {k}"
            c = dev.getOutDataDevice(dY.data_ptr() + 2 * (1 + w), pitch_out, take, stream.cuda_stream)
            assert c == got_host[-1].shape[1]
            w += c
            pos += m
    stream.synchronize()
    want = np.concatenate(got_host, axis=1)
    assert want.shape[1] == w and 0 < w < pitch_out - 1
    assert np.array_equal(dY[:, 1:1 + w].cpu().numpy(), want), f"{name}: int16 device rows differ from int16 host rows"
    host.close()
    dev.close()


def test_s16_device_rows_process_block_protocol(A):
    import torch
    sr, S, B = 44100, 48, 480
    n = B * 50
    X = _pcm(n, sr, 1, 9100, S)
    pitch = n + 1
    Xp = np.zeros((S, pitch), np.int16)
    Xp[:, 1:n + 1] = X
    host = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S, fmt=A.S16)
    dev = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S, fmt=A.S16)
    stream = torch.cuda.Stream()
    d = torch.from_numpy(Xp).cuda()
    ready = []
    with torch.cuda.stream(stream):
        for pos in range(0, n, B):
            dev.processBlockDevice(d.data_ptr() + 2 * (1 + pos), pitch, B, stream.cuda_stream)     # in place, block by block
            ready.append(dev.outputReady())
    stream.synchronize()
    got = d.cpu().numpy()[:, 1:n + 1]
    for i, pos in enumerate(range(0, n, B)):
        blk = np.ascontiguousarray(X[:, pos:pos + B])
        host.processBlock(blk)
        assert host.outputReady() == ready[i]
        assert np.array_equal(got[:, pos:pos + B], blk), f"block {i}"
    assert sum(ready) > 30
    host.close()
    dev.close()


def test_s16_format_lock_and_arguments(A, pvlib):
    import torch
    from audiomod_b200 import _lib
    from audiomod_b200.phasevocoder import _chan_ptrs, _sp
    L = pvlib
    R, n = 2, 480
    x16 = np.zeros((R, n), np.int16)
    x32 = np.zeros((R, n), np.float32)
    ready = C.c_int(0)

    def msg():
        return L.pvgpu_last_error().decode()

    # float32 after int16 (host and device float32 calls; the retrieve calls too)
    pv = A.phasevocoder(44100, 1, 1.0, 7.0, streams=R, fmt=A.S16)
    pv.processInData(x16)
    assert L.pvgpu_process(pv._h, _chan_ptrs(x32), n) == _lib.ESTATE and "pvgpu_process_s16" in msg()
    assert L.pvgpu_process_block(pv._h, _chan_ptrs(x32), n, C.byref(ready)) == _lib.ESTATE
    assert L.pvgpu_retrieve(pv._h, _chan_ptrs(x32), 1) == -_lib.ESTATE and "pvgpu_retrieve_s16" in msg()
    d32 = torch.zeros((R, n), dtype=torch.float32, device="cuda")
    assert L.pvgpu_process_device(pv._h, C.c_void_p(d32.data_ptr()), n, n, None) == _lib.ESTATE
    with pytest.raises(TypeError):
        pv.processInData(x32)                     # the Python mirror rejects other dtypes rather than casting them
    with pytest.raises(TypeError):
        pv.processBlock(x32)
    # host int16 after device int16 (and the other way round)
    d16 = torch.zeros((R, n), dtype=torch.int16, device="cuda")
    assert L.pvgpu_process_device_s16(pv._h, C.c_void_p(d16.data_ptr()), n, n, None) == _lib.ESTATE and "host and device" in msg()
    pv.close()
    pv = A.phasevocoder(44100, 1, 1.0, 7.0, streams=R, fmt=A.S16)
    pv.processInDataDevice(d16.data_ptr(), n, n)
    torch.cuda.synchronize()
    assert L.pvgpu_process_s16(pv._h, _chan_ptrs(x16, _sp), n) == _lib.ESTATE and "pvgpu_process_device_s16" in msg()
    assert L.pvgpu_retrieve_s16(pv._h, _chan_ptrs(x16, _sp), 1) == -_lib.ESTATE and "pvgpu_retrieve_device_s16" in msg()
    assert L.pvgpu_process_block_s16(pv._h, _chan_ptrs(x16, _sp), n, C.byref(ready)) == _lib.ESTATE
    pv.close()
    # int16 after float32
    pv = A.phasevocoder(44100, 1, 1.0, 7.0, streams=R)
    pv.processInData(x32)
    assert L.pvgpu_process_s16(pv._h, _chan_ptrs(x16, _sp), n) == _lib.ESTATE and "float32 and int16" in msg()
    assert L.pvgpu_retrieve_s16(pv._h, _chan_ptrs(x16, _sp), 1) == -_lib.ESTATE and "pvgpu_retrieve" in msg()
    assert L.pvgpu_process_device_s16(pv._h, C.c_void_p(d16.data_ptr()), n, n, None) == _lib.ESTATE
    assert L.pvgpu_retrieve_device_s16(pv._h, C.c_void_p(d16.data_ptr()), n, 1, None) == -_lib.ESTATE
    # the float32 host / device mix keeps its errors and messages
    assert L.pvgpu_process_device(pv._h, C.c_void_p(d32.data_ptr()), n, n, None) == _lib.ESTATE
    assert msg() == "this instance is fed host rows (pvgpu_process); host and device rows cannot be mixed"
    assert L.pvgpu_retrieve_device(pv._h, C.c_void_p(d32.data_ptr()), n, 1, None) == -_lib.ESTATE
    assert msg() == "this instance is fed host rows; use pvgpu_retrieve"
    pv.close()
    pv = A.phasevocoder(44100, 1, 1.0, 7.0, streams=R)
    pv.processInDataDevice(d32.data_ptr(), n, n)
    torch.cuda.synchronize()
    assert L.pvgpu_process(pv._h, _chan_ptrs(x32), n) == _lib.ESTATE
    assert msg() == "this instance is fed device rows (pvgpu_process_device); host and device rows cannot be mixed"
    assert L.pvgpu_retrieve(pv._h, _chan_ptrs(x32), 1) == -_lib.ESTATE
    assert msg() == "this instance is fed device rows; use pvgpu_retrieve_device"
    pv.close()
    # null or negative arguments
    pv = A.phasevocoder(44100, 1, 1.0, 7.0, streams=R, fmt=A.S16)
    p16 = _chan_ptrs(x16, _sp)
    dp = C.c_void_p(d16.data_ptr())
    assert L.pvgpu_process_s16(None, p16, n) == _lib.EINVAL
    assert L.pvgpu_process_s16(pv._h, None, n) == _lib.EINVAL
    assert L.pvgpu_process_s16(pv._h, p16, -1) == _lib.EINVAL
    assert L.pvgpu_retrieve_s16(None, p16, 1) == -_lib.EINVAL
    assert L.pvgpu_retrieve_s16(pv._h, None, 1) == -_lib.EINVAL
    assert L.pvgpu_retrieve_s16(pv._h, p16, -1) == -_lib.EINVAL
    assert L.pvgpu_process_block_s16(None, p16, n, C.byref(ready)) == _lib.EINVAL
    assert L.pvgpu_process_block_s16(pv._h, p16, n, None) == _lib.EINVAL
    assert L.pvgpu_process_block_s16(pv._h, p16, -1, C.byref(ready)) == _lib.EINVAL
    assert L.pvgpu_process_device_s16(None, dp, n, n, None) == _lib.EINVAL
    assert L.pvgpu_process_device_s16(pv._h, None, n, n, None) == _lib.EINVAL
    assert L.pvgpu_process_device_s16(pv._h, dp, n, -1, None) == _lib.EINVAL
    assert L.pvgpu_process_device_s16(pv._h, dp, n - 1, n, None) == _lib.EINVAL     # pitch shorter than a row
    assert L.pvgpu_retrieve_device_s16(None, dp, n, 1, None) == -_lib.EINVAL
    assert L.pvgpu_retrieve_device_s16(pv._h, None, n, 1, None) == -_lib.EINVAL
    assert L.pvgpu_retrieve_device_s16(pv._h, dp, n, -1, None) == -_lib.EINVAL
    assert L.pvgpu_process_block_device_s16(None, dp, n, n, None, C.byref(ready)) == _lib.EINVAL
    assert L.pvgpu_process_block_device_s16(pv._h, dp, n, n, None, None) == _lib.EINVAL
    assert L.pvgpu_process_block_device_s16(pv._h, dp, n, -1, None, C.byref(ready)) == _lib.EINVAL
    pv.close()
    with pytest.raises(ValueError):
        A.phasevocoder(44100, 1, 1.0, 7.0, fmt=2)
