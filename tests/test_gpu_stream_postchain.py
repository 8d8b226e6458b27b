"""Post-chain of FFT-free effects on streaming instances and live batches (pvgpu_set_postchain; phasevocoder.set_postchain).

The anchor is the batch's post-chain, which tests/test_gpu_postchain.py pins to the reference's effect objects (or to their
stored outputs).  pvgpu_test_postchain runs that same conversion and kernel once over given rows from fresh state; the first test
ties it to the batch bit for bit.  Every other check is bit-identity with paths this library already has: a chained instance
gives exactly the hook applied to the output of the same instance without a chain; int16 instances give exactly the quantised
output of float32 instances with the same chain; device rows give exactly the host rows."""
import ctypes as C

import numpy as np
import pytest

from cases import CASES, ctor_args, make_input
from test_gpu_live_batch import LIVE
from test_gpu_parity import _cli_protocol, assert_parity
from test_gpu_postchain import CHAIN_IDS, CHAINS, EQ_PARAMS, chain_inputs
from test_gpu_stream_s16 import _f32, _pcm, _quant

pytestmark = pytest.mark.gpu

SIZES = [480, 480, 1, 0, 2048, 311, 4099, 480]
COMP_LIM = [("compressor", -20.0, 4.0, 3.0, 5.0, 50.0), ("limiter", -6.0, 2.0, 1.0, 80.0)]


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def all_chains(A):
    """(id, chain): the batch tests' chains, the equalizer object with its defaults and with every band set, biquad sections."""
    sections = [("biquad", t, 500.0 + 400.0 * t, 0.8, 3.0) for t in (3, 6, 7, 8)] + [("gain", 0.9)]
    return (list(zip(CHAIN_IDS, CHAINS)) + [("eq-default", A.equalizer_chain()), ("eq-all-bands", A.equalizer_chain(EQ_PARAMS)),
                                             ("sections", sections)])


CHAIN_NAMES = CHAIN_IDS + ["eq-default", "eq-all-bands", "sections"]


def voice_chain(A):
    """The usual chain of a voice path after the shift: equalizer, compressor, limiter."""
    return A.equalizer_chain(EQ_PARAMS) + COMP_LIM


def hook(pvlib, sr, chain, y):
    """pvgpu_test_postchain: the chain over the rows of y (float32 [rows, n]) from fresh state."""
    from audiomod_b200 import _lib
    from audiomod_b200.phasevocoder import _fx_array
    z = np.array(y, dtype=np.float32, order="C", copy=True)
    if z.shape[1] == 0:
        return z
    arr, n = _fx_array(chain)
    _lib.check(pvlib.pvgpu_test_postchain(0, int(sr), arr, n, z.shape[0], z.shape[1], z.ctypes.data_as(C.POINTER(C.c_float))))
    return z


def _case(name):
    return next(c for c in CASES if c[0] == name)


def _live_inputs(name, S):
    _, kw, sr, ch, secs, seed = _case(name)
    n = int(sr * min(secs, 0.5))
    xs = [make_input(name, sr, ch, n / sr, seed + 11 * i)[:, :n] for i in range(S)]
    return kw, sr, ch, np.ascontiguousarray(np.concatenate(xs, axis=0))


def _feed(pvs, X, sizes=SIZES):
    """The same calls to every instance (odd sizes, sometimes leaving samples in the ring): equal counts call by call; returns
    every instance's retrieved output, concatenated."""
    n = X.shape[1]
    pos, k, outs = 0, 0, [[] for _ in pvs]
    while pos < n:
        m = min(sizes[k % len(sizes)], n - pos)
        k += 1
        for pv in pvs:
            pv.processInData(np.ascontiguousarray(X[:, pos:pos + m]))
        avail = pvs[0].getOutSamples()
        take = avail if k % 3 else avail // 2
        for i, pv in enumerate(pvs):
            assert pv.getOutSamples() == avail, f"call {k}: instance {i}"
            outs[i].append(pv.getOutData(take))
        pos += m
    return [np.concatenate(o, axis=1) for o in outs]


# ---- 1. the hook is the batch's post-chain ----
@pytest.mark.parametrize("ci", range(len(CHAIN_NAMES)), ids=CHAIN_NAMES)
def test_hook_equals_batch_postchain(A, pvlib, ci):
    """Batch with a chain == pvgpu_test_postchain applied to the same batch's plain output, bitwise: split and fused back ends,
    frames_per_chunk 8 and 64 (the effect state crosses chunk boundaries)."""
    _, chain = all_chains(A)[ci]
    sr, ch, st = 44100, 2, -3.0
    xs = chain_inputs(sr, ch)
    for fused in (False, True):
        for fpc in (8, 64):
            ys = {}
            for with_chain in (False, True):
                b = A.PhaseVocoderBatch(len(xs), max(x.shape[1] for x in xs), sr, ch, 1.0, st)
                b.set_fused(fused)
                b.tune(frames_per_chunk=fpc)
                if with_chain:
                    b.set_postchain(chain)
                ys[with_chain] = b.run(xs)
                b.close()
            for i, (plain, chained) in enumerate(zip(ys[False], ys[True])):
                assert np.array_equal(_bits(chained), _bits(hook(pvlib, sr, chain, plain))), f"fused={fused} fpc={fpc} [{i}]"


# ---- 2. a chained live batch equals the hook applied to the plain live batch ----
def _stream_equals_hook(A, pvlib, name, chain, S=5):
    kw, sr, ch, X = _live_inputs(name, S)
    args = ctor_args(kw)
    chained = A.phasevocoder(sr, ch, *args, streams=S)
    plain = A.phasevocoder(sr, ch, *args, streams=S)
    chained.set_postchain(chain)
    y, p = _feed([chained, plain], X)
    chained.close()
    plain.close()
    assert y.shape == p.shape == (S * ch, y.shape[1]) and y.shape[1] > 0
    assert np.array_equal(_bits(y), _bits(hook(pvlib, sr, chain, p))), f"{name}: chained output differs from the hook on the plain output"
    return y


@pytest.mark.parametrize("name", LIVE)
def test_stream_equals_hook(A, pvlib, name):
    _stream_equals_hook(A, pvlib, name, voice_chain(A))


@pytest.mark.parametrize("ci", range(len(CHAIN_NAMES)), ids=CHAIN_NAMES)
def test_stream_equals_hook_every_chain(A, pvlib, ci):
    _stream_equals_hook(A, pvlib, "cfg1_shift_p4_stereo", all_chains(A)[ci][1])


@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo"])
def test_stream_equals_hook_fused_back_end(A, pvlib, monkeypatch, name):
    monkeypatch.setenv("PVGPU_FUSED", "1")   # read when an instance is created
    _stream_equals_hook(A, pvlib, name, voice_chain(A))


# ---- 3. a chained single instance through the CLI protocol equals the chained batch ----
@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo", "cfg2_stretch_1p5_4096"])
def test_stream_equals_batch(A, name):
    """The streaming result is tied to the batch's post-chain, which the batch tests pin to the reference's effect objects."""
    _, kw, sr, ch, secs, seed = _case(name)
    x = make_input(name, sr, ch, secs, seed)
    tr, st, mode, core, fft = ctor_args(kw)
    chain = voice_chain(A)
    pv = A.phasevocoder(sr, ch, tr, st, mode, core, fft)
    pv.set_postchain(chain)
    y = _cli_protocol(pv, x, sr, mode)
    pv.close()
    b = A.PhaseVocoderBatch(1, x.shape[1], sr, ch, tr, st, mode, core, fft)
    b.set_postchain(chain)
    ref = b.run([x])[0]
    b.close()
    assert_parity(y, ref, name)


# ---- 4. int16 rows ----
def _s16_call_by_call(A, name, chain, X16, S, ch):
    _, kw, sr, _, _, _ = _case(name)
    args = ctor_args(kw)
    s16 = A.phasevocoder(sr, ch, *args, streams=S, fmt=A.S16)
    f32 = A.phasevocoder(sr, ch, *args, streams=S)
    s16.set_postchain(chain)
    f32.set_postchain(chain)
    Xf = _f32(X16)
    n = X16.shape[1]
    pos, k, outs = 0, 0, []
    while pos < n:
        m = min(SIZES[k % len(SIZES)], n - pos)
        k += 1
        s16.processInData(np.ascontiguousarray(X16[:, pos:pos + m]))
        f32.processInData(np.ascontiguousarray(Xf[:, pos:pos + m]))
        avail = f32.getOutSamples()
        assert s16.getOutSamples() == avail, f"{name}: call {k}"
        take = avail if k % 3 else avail // 2
        a, b = s16.getOutData(take), f32.getOutData(take)
        assert a.dtype == np.int16 and np.array_equal(a, _quant(b)), f"{name}: call {k}: int16 differs from the quantised float32 output"
        outs.append(a)
        pos += m
    s16.close()
    f32.close()
    y = np.concatenate(outs, axis=1)
    assert y.shape[1] > 0
    return y


@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo", "cfg5_whisper_1024", "cfg2_stretch_1p5_4096"])
def test_s16_equals_quantised_f32(A, name):
    _, kw, sr, ch, secs, seed = _case(name)
    S = 5
    _s16_call_by_call(A, name, voice_chain(A), _pcm(int(sr * min(secs, 0.5)), sr, ch, seed, S), S, ch)


def test_s16_gain_saturates(A):
    """A gain > 1 drives the chain's output to +-1, which quantises to 32767 / -32768."""
    name = "cfg4_shift_p7_mono"
    _, kw, sr, ch, secs, seed = _case(name)
    loud = np.clip(_pcm(int(sr * 0.5), sr, ch, seed, 3).astype(np.int32) * 8, -32768, 32767).astype(np.int16)
    y = _s16_call_by_call(A, name, [("gain", 4.0)], loud, 3, ch)
    assert np.count_nonzero(y == 32767) > 0 and np.count_nonzero(y == -32768) > 0


# ---- 5. device rows ----
@pytest.mark.parametrize("s16", [False, True], ids=["f32", "s16"])
@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo"])
def test_device_rows_equal_host_rows(A, name, s16):
    """Chained device rows (everything on one CUDA stream, no call waiting) == chained host rows, bitwise; int16 rows at pointers
    that are only 2-byte aligned."""
    import torch
    _, kw, sr, ch, secs, seed = _case(name)
    args = ctor_args(kw)
    S = 6
    n = int(sr * min(secs, 0.5))
    R = S * ch
    if s16:
        X = _pcm(n, sr, ch, seed, S)
        fmt, esz, off = A.S16, 2, 1
    else:
        X = np.ascontiguousarray(np.concatenate([make_input(name, sr, ch, n / sr, seed + 5 * i)[:, :n] for i in range(S)], axis=0))
        fmt, esz, off = A.F32, 4, 0
    pitch_in, pitch_out = n + 3, (1 << 16) + 1
    Xp = np.zeros((R, pitch_in), X.dtype)
    Xp[:, off:off + n] = X
    chain = voice_chain(A)
    host = A.phasevocoder(sr, ch, *args, streams=S, fmt=fmt)
    dev = A.phasevocoder(sr, ch, *args, streams=S, fmt=fmt)
    host.set_postchain(chain)
    dev.set_postchain(chain)
    stream = torch.cuda.Stream()
    dX = torch.from_numpy(Xp).cuda()
    dY = torch.zeros((R, pitch_out), dtype=torch.int16 if s16 else torch.float32, device="cuda")
    pos, k, w, got = 0, 0, 0, []
    with torch.cuda.stream(stream):
        while pos < n:
            m = min(SIZES[k % len(SIZES)], n - pos)
            k += 1
            host.processInData(np.ascontiguousarray(X[:, pos:pos + m]))
            avail = host.getOutSamples()
            take = avail if k % 3 else avail // 2
            got.append(host.getOutData(take))
            dev.processInDataDevice(dX.data_ptr() + esz * (off + pos), pitch_in, m, stream.cuda_stream)
            assert dev.getOutSamples() == avail, f"{name}: call {k}"
            c = dev.getOutDataDevice(dY.data_ptr() + esz * (off + w), pitch_out, take, stream.cuda_stream)
            assert c == got[-1].shape[1]
            w += c
            pos += m
    stream.synchronize()
    want = np.concatenate(got, axis=1)
    assert want.shape[1] == w > 0
    have = dY[:, off:off + w].cpu().numpy()
    assert np.array_equal(have, want) if s16 else np.array_equal(_bits(have), _bits(want)), f"{name}: device rows differ from host rows"
    host.close()
    dev.close()


@pytest.mark.parametrize("s16", [False, True], ids=["f32", "s16"])
def test_device_rows_process_block_protocol(A, s16):
    import torch
    sr, S, B = 44100, 48, 480
    n = B * 50
    X = _pcm(n, sr, 1, 9100, S) if s16 else np.ascontiguousarray(
        np.concatenate([make_input("x", sr, 1, n / sr, 9100 + i)[:, :n] for i in range(S)], axis=0))
    fmt, esz = (A.S16, 2) if s16 else (A.F32, 4)
    pitch = n + 1
    Xp = np.zeros((S, pitch), X.dtype)
    Xp[:, 1:n + 1] = X
    chain = voice_chain(A)
    host = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S, fmt=fmt)
    dev = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S, fmt=fmt)
    host.set_postchain(chain)
    dev.set_postchain(chain)
    stream = torch.cuda.Stream()
    d = torch.from_numpy(Xp).cuda()
    ready = []
    with torch.cuda.stream(stream):
        for pos in range(0, n, B):
            dev.processBlockDevice(d.data_ptr() + esz * (1 + pos), pitch, B, stream.cuda_stream)
            ready.append(dev.outputReady())
    stream.synchronize()
    got = d.cpu().numpy()[:, 1:n + 1]
    for i, pos in enumerate(range(0, n, B)):
        blk = np.ascontiguousarray(X[:, pos:pos + B])
        host.processBlock(blk)
        assert host.outputReady() == ready[i]
        assert np.array_equal(got[:, pos:pos + B].view(np.uint16 if s16 else np.uint32), blk.view(np.uint16 if s16 else np.uint32)), f"block {i}"
    assert sum(ready) > 30
    host.close()
    dev.close()


# ---- 6. processBlock ----
def test_process_block_protocol(A, pvlib):
    """64 streams in place: the plain instance's ready flags, buffers untouched while not ready, ready blocks (concatenated) equal
    to the hook on the plain instance's ready blocks."""
    sr, S, B = 44100, 64, 480
    n = B * 60
    X = np.ascontiguousarray(np.concatenate([make_input("x", sr, 1, n / sr, 7000 + i)[:, :n] for i in range(S)], axis=0))
    chain = voice_chain(A)
    chained = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S)
    plain = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S)
    chained.set_postchain(chain)
    got, want = [], []
    for pos in range(0, n, B):
        a = np.ascontiguousarray(X[:, pos:pos + B])
        before = a.copy()
        p = a.copy()
        chained.processBlock(a)
        plain.processBlock(p)
        assert chained.outputReady() == plain.outputReady(), f"block at {pos}"
        if chained.outputReady():
            got.append(a)
            want.append(p)
        else:
            assert np.array_equal(_bits(a), _bits(before)), "buffers must be untouched while output is not ready"
    assert len(got) > 40
    y, p = np.concatenate(got, axis=1), np.concatenate(want, axis=1)
    assert np.array_equal(_bits(y), _bits(hook(pvlib, sr, chain, p)))
    chained.close()
    plain.close()


# ---- 7. set, change and clear mid-stream ----
@pytest.mark.parametrize("s16", [False, True], ids=["f32", "s16"])
def test_set_change_clear_mid_stream(A, pvlib, s16):
    """A chain takes effect at the next call from fresh state; samples already in the ring come out as they were produced; a
    cleared chain gives the plain output again, bit for bit."""
    name = "cfg1_shift_p4_stereo"
    _, kw, sr, ch, secs, seed = _case(name)
    args = ctor_args(kw)
    S = 3
    n = int(sr * 0.6)
    X16 = _pcm(n, sr, ch, seed, S)
    Xf = _f32(X16)
    C1, C2 = voice_chain(A), [("limiter", -3.0, 0.0, 0.5, 20.0), ("gain", 0.8)]
    events = {15: C1, 18: C2, 21: []}    # call index -> chain set before it (the calls before them leave samples in the ring)
    fmt = A.S16 if s16 else A.F32
    pv = A.phasevocoder(sr, ch, *args, streams=S, fmt=fmt)
    ref = A.phasevocoder(sr, ch, *args, streams=S)          # float32, never chained
    feed = X16 if s16 else Xf
    pos, k, outs, plain, done, ring, rings = 0, 0, [], [], 0, 0, []
    bounds = []                                             # (first output position the chain applies to, chain)
    while pos < n:
        if k in events:
            pv.set_postchain(events[k])
            bounds.append((done + ring, events[k]))
            rings.append(ring)
        m = min(SIZES[k % len(SIZES)], n - pos)
        k += 1
        pv.processInData(np.ascontiguousarray(feed[:, pos:pos + m]))
        ref.processInData(np.ascontiguousarray(Xf[:, pos:pos + m]))
        avail = ref.getOutSamples()
        assert pv.getOutSamples() == avail
        take = avail if k % 3 else avail // 2
        outs.append(pv.getOutData(take))
        plain.append(ref.getOutData(take))
        done += take
        ring = avail - take
        pos += m
    pv.close()
    ref.close()
    y, p = np.concatenate(outs, axis=1), np.concatenate(plain, axis=1)
    assert len(bounds) == 3 and all(b0 < b1 for (b0, _), (b1, _) in zip(bounds, bounds[1:])) and bounds[-1][0] < y.shape[1]
    assert all(r > 0 for r in rings), "every set should find samples waiting in the ring"
    want = p.copy()
    for i, (b0, chain) in enumerate(bounds):
        b1 = bounds[i + 1][0] if i + 1 < len(bounds) else p.shape[1]
        if chain:
            want[:, b0:b1] = hook(pvlib, sr, chain, p[:, b0:b1])
    if s16:
        assert np.array_equal(y, _quant(want))
    else:
        assert np.array_equal(_bits(y), _bits(want))
        assert np.array_equal(_bits(y[:, bounds[-1][0]:]), _bits(p[:, bounds[-1][0]:])), "after a clear the output is the plain output"


# ---- 8. many rows: more than one CTA of the chain, the row-copy pool ----
def test_large_live_batch_uses_the_copy_pool(A):
    sr, ch, S = 44100, 1, 320
    n = 480 * 25 + 4099
    base = make_input("x", sr, ch, n / sr, 8100)[:, :n]
    X = np.ascontiguousarray(np.repeat(base, S, axis=0) * (1.0 + 0.01 * np.arange(S, dtype=np.float32))[:, None])
    chain = voice_chain(A)
    live = A.phasevocoder(sr, ch, 1.0, 7.0, streams=S)
    live.set_postchain(chain)
    picks = (0, 1, 77, 200, S - 1)
    singles = [A.phasevocoder(sr, ch, 1.0, 7.0) for _ in picks]
    for pv in singles:
        pv.set_postchain(chain)
    sizes = [480] * 10 + [4099, 1, 0, 480, 311] + [480] * 12
    pos = 0
    for m in sizes:
        m = min(m, n - pos)
        live.processInData(np.ascontiguousarray(X[:, pos:pos + m]))
        avail = live.getOutSamples()
        Y = live.getOutData(avail)
        for j, i in enumerate(picks):
            singles[j].processInData(np.ascontiguousarray(X[i:i + 1, pos:pos + m]))
            assert singles[j].getOutSamples() == avail
            assert np.array_equal(_bits(Y[i:i + 1]), _bits(singles[j].getOutData(avail))), f"stream {i} at {pos}"
        pos += m
    live.close()
    for pv in singles:
        pv.close()


# ---- 9. arguments ----
def test_arguments(A, pvlib):
    from audiomod_b200 import _lib
    from audiomod_b200.phasevocoder import _fx_array
    L = pvlib

    def msg():
        return L.pvgpu_last_error().decode()

    pv = A.phasevocoder(44100, 1, 1.0, 7.0, streams=2)
    b = A.PhaseVocoderBatch(1, 4800, 44100, 1, 1.0, 7.0)
    good, n_good = _fx_array(COMP_LIM)
    many = (_lib.Fx * 13)()
    for i in range(13):
        many[i].kind = _lib.FX_GAIN
        many[i].p[0] = 1.0
    unknown = (_lib.Fx * 1)()
    unknown[0].kind = 9
    ratio0, _ = _fx_array([("compressor", -10.0, 0.0, 6.0, 10.0, 100.0)])
    ratio_neg, _ = _fx_array([("compressor", -10.0, -2.0, 6.0, 10.0, 100.0)])
    bad = [(good, -1), (many, 13), (None, 1), (unknown, 1), (ratio0, 1), (ratio_neg, 1)]
    for arr, cnt in bad:
        assert L.pvgpu_batch_set_postchain(b._h, arr, cnt) == _lib.EINVAL
        want = msg()
        assert L.pvgpu_set_postchain(pv._h, arr, cnt) == _lib.EINVAL
        assert msg() == want, "the batch's messages"
    assert L.pvgpu_set_postchain(None, good, n_good) == _lib.EINVAL
    assert L.pvgpu_set_postchain(pv._h, many, 12) == _lib.OK        # twelve effects are allowed
    assert L.pvgpu_set_postchain(pv._h, None, 0) == _lib.OK         # clearing needs no array
    with pytest.raises(A.PvgpuError):
        pv.set_postchain([("compressor", -10.0, 0.0, 6.0, 10.0, 100.0)])
    pv.close()
    b.close()
    # an instance whose mode does nothing: setting a chain succeeds and changes nothing
    pv = A.phasevocoder(44100, 1, 1.0, 0.0, 42, 1, 2048)
    pv.set_postchain(COMP_LIM)
    pv.processInData(np.zeros((1, 4800), np.float32))
    assert pv.getOutSamples() == 0
    pv.close()
