"""Loudness meters on streaming instances and live batches (pvgpu_set_meters / pvgpu_get_meters / pvgpu_get_meters_device;
phasevocoder.set_meters / meters / metersDevice).

The meters are specified by ITU-R BS.1770-4 and EBU Tech 3341 (momentary and short-term loudness, ungated, every channel weighted
1.0) plus the sample peak.  Anchors: the EBU Tech 3341 sine cases through pvgpu_test_loudness (the meter kernels over given rows
from fresh state), and a float64 restatement in numpy / scipy (K-weighting with lfilter, sub-block energies, windows) that the hook
and every live instance must meet within 1e-4 LU, with exact peaks and sample counts.  Device rows are compared with host rows
bit for bit, and outputs with meters on with outputs with meters off."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.signal import lfilter

from cases import ctor_args, make_input
from test_gpu_stream_postchain import SIZES, _bits, _case, voice_chain
from test_gpu_stream_postchain_params import user_chain
from test_gpu_stream_s16 import _f32, _pcm
from test_loudness_design import kw_coeffs

pytestmark = pytest.mark.gpu

_fp = C.POINTER(C.c_float)


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


# ---- the restatement ----
def _L(sr):
    return (sr + 5) // 10


def energies(x, sr):
    """Sub-block energies [rows, completed sub-blocks] of the K-weighted rows of x (float64 restatement)."""
    c = kw_coeffs(sr)
    y = lfilter([c[0], c[1], c[2]], [1.0, c[3], c[4]], np.asarray(x, np.float64), axis=1)
    z = lfilter([1.0, -2.0, 1.0], [1.0, c[5], c[6]], y, axis=1)
    L = _L(sr)
    nb = z.shape[1] // L
    return (z[:, :nb * L] ** 2).reshape(z.shape[0], nb, L).sum(axis=2)


def loudness(E, nb, W, L, ch):
    """Loudness per stream over the last W of the first nb sub-blocks of E (silence before the first)."""
    win = np.zeros((E.shape[0], W))
    k = min(W, nb)
    if k:
        win[:, W - k:] = E[:, nb - k:nb]
    tot = win.sum(axis=1).reshape(-1, ch).sum(axis=1)
    with np.errstate(divide="ignore"):
        return -0.691 + 10.0 * np.log10(tot / (W * L))


def ref_meters(E, measured, sr, ch):
    L = _L(sr)
    nb = measured // L
    return loudness(E, nb, 4, L, ch), loudness(E, nb, 30, L, ch)


def assert_lu(got, want, what):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isneginf(got), np.isneginf(want)), (what, got, want)
    fin = np.isfinite(want)
    assert np.all(np.isfinite(got[fin])), (what, got)
    if fin.any():
        assert np.max(np.abs(got[fin] - want[fin])) <= 1e-4, (what, np.max(np.abs(got[fin] - want[fin])))


def hook(pvlib, sr, ch, S, x, call):
    """pvgpu_test_loudness: (momentary [S], short-term [S], peak [S * ch]) of float32 rows x [S * ch, n] fed in pieces of call."""
    from audiomod_b200 import _lib
    x = np.ascontiguousarray(x, dtype=np.float32)
    m, s, p = np.empty(S, np.float32), np.empty(S, np.float32), np.empty(S * ch, np.float32)
    _lib.check(pvlib.pvgpu_test_loudness(0, int(sr), ch, S, x.shape[1], int(call), x.ctypes.data_as(_fp), m.ctypes.data_as(_fp),
                                         s.ctypes.data_as(_fp), p.ctypes.data_as(_fp)))
    return m, s, p


def sine(sr, secs, dbfs, ch, f=1000.0):
    t = np.arange(int(sr * secs)) / sr
    return np.tile((10.0 ** (dbfs / 20.0) * np.sin(2 * np.pi * f * t)).astype(np.float32), (ch, 1))


# ---- 1. standard anchors through the hook ----
@pytest.mark.parametrize("sr", [48000, 44100])
def test_ebu_tech3341_cases_1_and_2(pvlib, sr):
    """Cases 1 and 2 of EBU Tech 3341: a stereo 1 kHz sine at -23 and -33 dBFS reads -23.0 and -33.0 LUFS, momentary and short-term
    (after more than 3 s); a mono sine reads 10 log10(2) = 3.01 dB lower than the stereo one."""
    x = np.concatenate([sine(sr, 4.0, -23.0, 2), sine(sr, 4.0, -33.0, 2)])
    m, s, p = hook(pvlib, sr, 2, 2, x, 480)
    assert np.all(np.abs(m - [-23.0, -33.0]) <= 0.1) and np.all(np.abs(s - [-23.0, -33.0]) <= 0.1), (m, s)
    assert np.array_equal(p, np.max(np.abs(x[:, (x.shape[1] - 1) // 480 * 480:]), axis=1))
    mm, ms, _ = hook(pvlib, sr, 1, 2, x[::2], 480)
    assert np.all(np.abs((m - mm) - 10 * math.log10(2)) <= 1e-4) and np.all(np.abs((s - ms) - 10 * math.log10(2)) <= 1e-4), (m - mm, s - ms)


# ---- 2. the hook against the restatement ----
def _signals(sr, ch, S, secs, seed):
    """S streams of ch rows: noise bursts and tones at levels 20 dB apart, one silent stream, one that starts silent."""
    rng = np.random.default_rng(seed)
    n = int(sr * secs)
    x = np.zeros((S * ch, n), np.float32)
    t = np.arange(n) / sr
    for j in range(S):
        if j == 1:
            continue   # silence: -inf
        g = 10.0 ** (-(6 + 10 * j) / 20)
        env = 0.5 + 0.5 * np.sin(2 * np.pi * (0.3 + 0.1 * j) * t)
        for c in range(ch):
            v = g * env * (0.6 * rng.standard_normal(n) + np.sin(2 * np.pi * (200 + 350 * c + 90 * j) * t))
            if j == 2:
                v[:int(1.3 * sr)] = 0.0
            x[j * ch + c] = np.clip(v, -1, 1)
    return x


@pytest.mark.parametrize("sr", [16000, 44100, 48000])
def test_hook_equals_restatement(pvlib, sr):
    """4.3 s (more than the 30 sub-blocks of the short-term ring) of 4 stereo streams: M and S within 1e-4 LU of the float64
    restatement, peaks exact; pieces of the whole signal, of 480 and of 37 samples give bit-identical M and S."""
    ch, S = 2, 4
    x = _signals(sr, ch, S, 4.3, sr)
    n = x.shape[1]
    E = energies(x, sr)
    wm, ws = ref_meters(E, n, sr, ch)
    res = {}
    for call in (n, 480, 37):
        m, s, p = hook(pvlib, sr, ch, S, x, call)
        assert_lu(m, wm, f"momentary, pieces of {call}")
        assert_lu(s, ws, f"short-term, pieces of {call}")
        last = x[:, (n - 1) // call * call:]
        assert np.array_equal(p, np.max(np.abs(last), axis=1)), f"peak, pieces of {call}"
        res[call] = (m, s)
    for call in (480, 37):
        assert np.array_equal(_bits(res[call][0]), _bits(res[n][0])) and np.array_equal(_bits(res[call][1]), _bits(res[n][1])), call
    # between sub-block boundaries the values stay those of the last completed sub-block
    cut = 7 * _L(sr) + 123
    m, s, _ = hook(pvlib, sr, ch, S, x[:, :cut], 480)
    m2, s2, _ = hook(pvlib, sr, ch, S, x[:, :7 * _L(sr)], 480)
    assert np.array_equal(_bits(m), _bits(m2)) and np.array_equal(_bits(s), _bits(s2))
    m, s, p = hook(pvlib, sr, ch, S, x[:, :_L(sr) - 1], 480)
    assert np.all(np.isneginf(m)) and np.all(np.isneginf(s))


# ---- 3. live batches ----
def _drive(pv, X, sizes=SIZES, block=False, meters=True):
    """Feeds X in calls of the given sizes (host rows), draining all output after every call.  Returns (the produced output,
    concatenated; per call: meters() after the call (None with meters=False), output samples that call produced).  block=True:
    processBlock of each size instead; the ready blocks and finally what is left in the ring are the output, and a call's
    production is read off the meters' sample count."""
    n = X.shape[1]
    pos, k, outs, log, was = 0, 0, [], [], 0
    while pos < n:
        m = min(sizes[k % len(sizes)], n - pos)
        k += 1
        a = np.ascontiguousarray(X[:, pos:pos + m])
        if block:
            pv.processBlock(a)
            if pv.outputReady():
                outs.append(a)
            mt = dict(pv.meters()) if meters else {"measured": was}
            mt["ready"] = pv.outputReady()
            log.append((mt, mt["measured"] - was))
            was = mt["measured"]
        else:
            pv.processInData(a)
            made = pv.getOutSamples()
            outs.append(pv.getOutData(made))
            log.append((pv.meters() if meters else None, made))
        pos += m
    if block:
        outs.append(pv.getOutData(pv.getOutSamples()))   # what is left in the ring
    return np.concatenate(outs, axis=1), log


def _check_log(y, log, sr, ch, S, scale=1.0, start=0):
    """Every call's meters against the restatement over the output produced since the meters were enabled (y[:, start:])."""
    z = np.asarray(y[:, start:], np.float64) * scale
    E = energies(z, sr)
    done = 0
    peak = np.zeros(S * ch, np.float32)
    for i, (mt, made) in enumerate(log):
        if made:
            peak = np.max(np.abs(z[:, done:done + made]), axis=1).astype(np.float32)
        done += made
        assert mt["measured"] == done, (i, mt["measured"], done)
        wm, ws = ref_meters(E, done, sr, ch)
        assert_lu(mt["momentary"], wm, f"call {i}: momentary")
        assert_lu(mt["short_term"], ws, f"call {i}: short-term")
        assert np.array_equal(mt["peak"].reshape(-1), peak), f"call {i}: peak"
    assert done == z.shape[1]


LIVE_CASES = ["cfg4_shift_p7_mono", "cfg1_shift_p4_stereo", "cfg3_formant_p4", "cfg5_robotic_512"]


def _live_x(name, S, secs):
    _, kw, sr, ch, _, seed = _case(name)
    n = int(sr * secs)
    x = np.concatenate([make_input(name, sr, ch, secs, seed + 11 * i)[:, :n] * (0.9 ** i) for i in range(S)], axis=0)
    return kw, sr, ch, np.ascontiguousarray(x, dtype=np.float32)


@pytest.mark.parametrize("name", LIVE_CASES)
def test_live_batch_host_f32(A, name):
    """3 streams, 3.5 s, odd call sizes: after every call M and S equal the restatement over everything the instance produced,
    peak = max |that call's output| (of the last call that produced any), measured = samples produced."""
    kw, sr, ch, X = _live_x(name, 3, 3.5)
    pv = A.phasevocoder(sr, ch, *ctor_args(kw), streams=3)
    pv.set_meters()
    y, log = _drive(pv, X)
    pv.close()
    assert y.shape[1] > 30 * _L(sr)
    _check_log(y, log, sr, ch, 3)


# ---- 4. row kinds ----
def test_live_batch_host_s16(A):
    """int16 host rows are measured as delivered: s / 32768."""
    _, kw, sr, ch, _, seed = _case("cfg1_shift_p4_stereo")
    n = int(sr * 3.3)
    X16 = _pcm(n, sr, ch, seed, 3)
    pv = A.phasevocoder(sr, ch, *ctor_args(kw), streams=3, fmt=A.S16)
    pv.set_meters()
    y, log = _drive(pv, X16)
    pv.close()
    assert y.dtype == np.int16
    _check_log(y, log, sr, ch, 3, scale=1.0 / 32768)


def _device_snapshots(A, pv, X, sizes=SIZES):
    """The calls of _drive on device rows, all on one CUDA stream without waiting: metersDevice into a device buffer after every
    call.  Returns ([calls, 2S + R] float32, measured per call)."""
    import torch
    s16 = X.dtype == np.int16
    esz = 2 if s16 else 4
    R, n = X.shape
    dX = torch.from_numpy(np.ascontiguousarray(X)).cuda()
    dY = torch.zeros((R, 2 * n + 64), dtype=torch.int16 if s16 else torch.float32, device="cuda")
    calls = 0
    pos = 0
    while pos < n:
        pos += min(sizes[calls % len(sizes)], n - pos)
        calls += 1
    S = pv.streams_
    snap = torch.full((calls, 2 * S + R), float("nan"), dtype=torch.float32, device="cuda")
    stream = torch.cuda.Stream()
    torch.cuda.synchronize()
    pos, k, w, measured = 0, 0, 0, []
    with torch.cuda.stream(stream):
        while pos < n:
            m = min(sizes[k % len(sizes)], n - pos)
            pv.processInDataDevice(dX.data_ptr() + esz * pos, n, m, stream.cuda_stream)
            w += pv.getOutDataDevice(dY.data_ptr() + esz * w, dY.shape[1], pv.getOutSamples(), stream.cuda_stream)
            measured.append(pv.metersDevice(snap[k].data_ptr(), stream.cuda_stream))
            k += 1
            pos += m
    stream.synchronize()
    return snap.cpu().numpy(), measured


@pytest.mark.parametrize("s16", [False, True], ids=["f32", "s16"])
def test_device_rows_equal_host_rows(A, s16):
    """Device rows, read through pvgpu_get_meters_device after every call, equal host rows of the same kind bit for bit; with a
    per-stream chain, so that the rows differ."""
    _, kw, sr, ch, _, seed = _case("cfg1_shift_p4_stereo")
    S, n = 3, int(sr * 3.2)
    X16 = _pcm(n, sr, ch, seed, S)
    X = X16 if s16 else _f32(X16)
    pvs = []
    for _ in range(2):
        pv = A.phasevocoder(sr, ch, *ctor_args(kw), streams=S, fmt=A.S16 if s16 else A.F32)
        pv.set_postchain(voice_chain(A))
        for j in range(S):
            pv.set_stream_postchain(j, user_chain(A, j))
        pv.set_meters()
        pvs.append(pv)
    _, log = _drive(pvs[0], X)
    snap, measured = _device_snapshots(A, pvs[1], X)
    for pv in pvs:
        pv.close()
    assert len(log) == len(snap)
    for i, (mt, _) in enumerate(log):
        host = np.concatenate([mt["momentary"], mt["short_term"], mt["peak"].reshape(-1)])
        assert np.array_equal(_bits(host), _bits(snap[i])), f"call {i}"
        assert measured[i] == mt["measured"], f"call {i}"
    assert np.isfinite(snap[-1]).all()


# ---- 5. with the post-chain ----
@pytest.mark.parametrize("s16", [False, True], ids=["f32", "s16"])
def test_meters_measure_the_chained_output(A, s16):
    """With the voice chain and per-stream parameters the meters measure what the instance delivers: the chained samples."""
    _, kw, sr, ch, _, seed = _case("cfg4_shift_p7_mono")
    S, n = 4, int(sr * 3.3)
    X16 = _pcm(n, sr, ch, seed, S)
    pv = A.phasevocoder(sr, ch, *ctor_args(kw), streams=S, fmt=A.S16 if s16 else A.F32)
    pv.set_postchain(voice_chain(A))
    for j in range(S):
        pv.set_stream_postchain(j, user_chain(A, j))
    pv.set_meters()
    y, log = _drive(pv, X16 if s16 else _f32(X16))
    pv.close()
    _check_log(y, log, sr, ch, S, scale=1.0 / 32768 if s16 else 1.0)


# ---- 6. meters change nothing ----
@pytest.mark.parametrize("rows", ["host_f32", "host_s16", "device_f32"])
def test_meters_change_nothing(A, rows):
    """330 streams of 3 channels (streams straddle warps): outputs and counts with meters on equal those with meters off, call by
    call, bit for bit; the final meters equal the restatement."""
    sr, ch, S = 44100, 3, 330
    n = int(sr * 0.9)
    from audiomod_b200.synth import synth
    X = np.ascontiguousarray(np.concatenate([synth(9000 + j, sr, 0.9, ch)[:, :n] * (0.97 ** (j % 40)) for j in range(S)]), np.float32)
    s16 = rows == "host_s16"
    if s16:
        X = np.clip(X * 32768.0, -32768, 32767).astype(np.int16)
    on, off = [A.phasevocoder(sr, ch, 1.0, 5.0, streams=S, fmt=A.S16 if s16 else A.F32) for _ in range(2)]
    on.set_meters()
    if rows == "device_f32":
        import torch
        dX = torch.from_numpy(X).cuda()
        outs = []
        for pv in (on, off):
            dY = torch.zeros((S * ch, 2 * n), dtype=torch.float32, device="cuda")
            pos, k, w, counts = 0, 0, 0, []
            while pos < n:
                m = min(SIZES[k % len(SIZES)], n - pos)
                k += 1
                pv.processInDataDevice(dX.data_ptr() + 4 * pos, n, m)
                counts.append(pv.getOutSamples())
                w += pv.getOutDataDevice(dY.data_ptr() + 4 * w, 2 * n, counts[-1])
                pos += m
            torch.cuda.synchronize()
            outs.append((dY[:, :w].cpu().numpy(), counts))
        assert outs[0][1] == outs[1][1]
        assert np.array_equal(_bits(outs[0][0]), _bits(outs[1][0]))
        y = outs[0][0]
        d = torch.zeros(2 * S + S * ch, dtype=torch.float32, device="cuda")
        measured = on.metersDevice(d.data_ptr())
        torch.cuda.synchronize()
        d = d.cpu().numpy()
        final = dict(momentary=d[:S], short_term=d[S:2 * S], measured=measured)
    else:
        pos, k, got = 0, 0, []
        while pos < n:
            m = min(SIZES[k % len(SIZES)], n - pos)
            k += 1
            a = np.ascontiguousarray(X[:, pos:pos + m])
            on.processInData(a)
            off.processInData(a)
            assert on.getOutSamples() == off.getOutSamples(), f"call {k}"
            take = max(0, on.getOutSamples() - k % 2)   # sometimes one sample stays in the ring
            ya, yb = on.getOutData(take), off.getOutData(take)
            assert np.array_equal(ya, yb) if s16 else np.array_equal(_bits(ya), _bits(yb)), f"call {k}"
            got.append(ya)
            pos += m
        final = on.meters()
        # the ring still holds what the last calls left in it: measured counts it, the retrieved output does not
        rest = on.getOutData(on.getOutSamples())
        assert np.array_equal(rest, off.getOutData(off.getOutSamples()))
        y = np.concatenate(got + [rest], axis=1)
    on.close()
    off.close()
    assert final["measured"] == y.shape[1] > 8 * _L(sr)
    wm, ws = ref_meters(energies(np.asarray(y, np.float64) / (32768.0 if s16 else 1.0), sr), y.shape[1], sr, ch)
    assert_lu(final["momentary"], wm, "momentary")
    assert_lu(final["short_term"], ws, "short-term")


# ---- 7. lifecycle ----
def test_enable_midstream_reenable_disable(A, pvlib):
    """Enabled mid-stream the sub-blocks count from that point; enabling again resets the state; disabled, the getters return
    PVGPU_ESTATE; the output equals that of an instance that never had meters."""
    from audiomod_b200 import _lib
    kw, sr, ch, X = _live_x("cfg1_shift_p4_stereo", 2, 4.0)
    cuts = [0, 40 * 480 + 17, 200 * 480 + 5, 260 * 480, X.shape[1]]
    ref = A.phasevocoder(sr, ch, *ctor_args(kw), streams=2)
    want = np.concatenate([_drive(ref, X[:, a:b], meters=False)[0] for a, b in zip(cuts, cuts[1:])], axis=1)
    ref.close()
    pv = A.phasevocoder(sr, ch, *ctor_args(kw), streams=2)
    seg = lambda i, **k: _drive(pv, X[:, cuts[i]:cuts[i + 1]], **k)
    y0, _ = seg(0, meters=False)
    pv.set_meters()
    fresh = pv.meters()
    assert fresh["measured"] == 0 and np.all(np.isneginf(fresh["momentary"])) and np.all(np.isneginf(fresh["short_term"]))
    assert np.all(fresh["peak"] == 0) and fresh["peak"].shape == (2, ch)
    y1, log1 = seg(1)
    _check_log(y1, log1, sr, ch, 2)
    pv.set_meters(True)   # again: fresh state
    assert pv.meters()["measured"] == 0 and np.all(np.isneginf(pv.meters()["short_term"]))
    y2, log2 = seg(2)
    _check_log(y2, log2, sr, ch, 2)
    pv.set_meters(False)
    with pytest.raises(A.PvgpuError) as e:
        pv.meters()
    assert e.value.code == _lib.ESTATE
    y3, _ = seg(3, meters=False)
    pv.close()
    assert np.array_equal(_bits(np.concatenate([y0, y1, y2, y3], axis=1)), _bits(want))


def test_unknown_mode(A):
    """An instance whose mode does nothing: set_meters succeeds and nothing is ever measured."""
    pv = A.phasevocoder(44100, 2, 1.0, 0.0, mode=42, streams=3)
    pv.set_meters()
    for _ in range(5):
        pv.processInData(np.zeros((6, 480), np.float32))
    mt = pv.meters()
    assert mt["measured"] == 0 and np.all(np.isneginf(mt["momentary"])) and np.all(mt["peak"] == 0)
    pv.close()


def test_process_block_protocol(A):
    """processBlock: the meters advance with every call that produces output, also while *ready = 0 (the output waits in the
    ring); the delivered blocks equal those of an instance without meters."""
    sr, S, sizes = 44100, 16, [480, 480, 2400, 311]
    n = 480 * 320
    X = np.ascontiguousarray(np.concatenate([make_input("x", sr, 1, n / sr, 7100 + i)[:, :n] for i in range(S)], axis=0))
    ref = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S)
    want, ref_log = _drive(ref, X, sizes=sizes, block=True, meters=False)
    ref.close()
    pv = A.phasevocoder(sr, 1, 1.0, 7.0, streams=S)
    pv.set_meters()
    y, log = _drive(pv, X, sizes=sizes, block=True)
    pv.close()
    assert [mt["ready"] for mt, _ in log] == [mt["ready"] for mt, _ in ref_log]
    assert np.array_equal(_bits(y), _bits(want))
    assert any(not mt["ready"] and made > 0 for mt, made in log), "no call produced output while not ready"
    assert sum(mt["ready"] for mt, _ in log) > len(log) // 2
    _check_log(y, log, sr, 1, S)


# ---- 8. errors ----
def test_errors(A, pvlib):
    from audiomod_b200 import _lib
    import torch
    L = pvlib
    pv = A.phasevocoder(44100, 1, 1.0, 4.0, streams=2)
    with pytest.raises(A.PvgpuError) as e:   # before enabling
        pv.meters()
    assert e.value.code == _lib.ESTATE
    d = torch.zeros(8, dtype=torch.float32, device="cuda")
    assert L.pvgpu_get_meters_device(pv._h, C.c_void_p(d.data_ptr()), None, None) == _lib.ESTATE
    assert L.pvgpu_set_meters(None, 1) == _lib.EINVAL
    assert L.pvgpu_set_meters(pv._h, 2) == _lib.EINVAL
    pv.set_meters()
    assert L.pvgpu_get_meters(None, None, None, None, None) == _lib.EINVAL
    assert L.pvgpu_get_meters_device(None, C.c_void_p(d.data_ptr()), None, None) == _lib.EINVAL
    assert L.pvgpu_get_meters_device(pv._h, None, None, None) == _lib.EINVAL
    assert L.pvgpu_get_meters(pv._h, None, None, None, None) == _lib.OK   # every output is optional
    pv.processInData(np.zeros((2, 4800), np.float32))
    assert L.pvgpu_get_meters_device(pv._h, C.c_void_p(d.data_ptr()), None, None) == _lib.ESTATE
    assert L.pvgpu_last_error().decode().endswith("use pvgpu_get_meters")
    pv.close()
    dv = A.phasevocoder(44100, 1, 1.0, 4.0, streams=2)
    dv.set_meters()
    x = torch.zeros((2, 4800), dtype=torch.float32, device="cuda")
    dv.processInDataDevice(x.data_ptr(), 4800, 4800)
    assert dv.metersDevice(d.data_ptr()) == dv.getOutSamples()
    with pytest.raises(A.PvgpuError) as e:
        dv.meters()
    assert e.value.code == _lib.ESTATE and "pvgpu_get_meters_device" in str(e.value)
    torch.cuda.synchronize()
    dv.close()
    m = np.zeros(4, np.float32)
    for bad in [(0, 48000, 0, 1, 10, 1), (0, 48000, 1, 0, 10, 1), (0, 48000, 1, 1, -1, 1), (0, 48000, 1, 1, 10, 0), (0, 0, 1, 1, 10, 1)]:
        assert L.pvgpu_test_loudness(*bad, m.ctypes.data_as(_fp), m.ctypes.data_as(_fp), m.ctypes.data_as(_fp), m.ctypes.data_as(_fp)) == _lib.EINVAL, bad
