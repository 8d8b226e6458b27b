"""Per-stream post-chain parameters on streaming instances and live batches (pvgpu_set_stream_postchain;
phasevocoder.set_stream_postchain).

Anchors, as in test_gpu_stream_postchain.py: pvgpu_test_postchain (the batch's conversion and kernel from fresh state, tied
there to the batch bit for bit) applied to the output of the same instance without a chain; int16 instances against the
quantised float32 result; device rows against host rows.  A parameter change in the middle of a stream has no such anchor, so
it is checked against an independent restatement of the effects in numpy: gain and biquad sections exactly (float32 scalar
arithmetic in the kernel's order, no FMA), compressor and limiter as a float64 restatement of pv_post.cu's expressions at the
parity bars.  Every other comparison is bit for bit."""
import math

import numpy as np
import pytest

from cases import ctor_args, make_input
from test_gpu_parity import assert_parity
from test_gpu_postchain import EQ_PARAMS
from test_gpu_stream_postchain import SIZES, _bits, _case, _live_inputs, hook, voice_chain
from test_gpu_stream_s16 import _f32, _pcm, _quant

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


def user_eq(A, j):
    """Stream j's equalizer preset: the bands of EQ_PARAMS (the same sections), its own gains."""
    eq = list(EQ_PARAMS)
    for b in range(8):
        eq[4 * b + 3] += ((j * 7 + 3 * b) % 11 - 5) * 0.5
    return A.equalizer_chain(eq)


def user_chain(A, j):
    """Stream j's preset of voice_chain: the same kinds in the same order, its own EQ gains, compressor threshold, ratio, make-up,
    attack and release, limiter ceiling, make-up, attack and release."""
    comp = ("compressor", -14.0 - (j % 9) * 1.5, 2.0 + (j % 4), 1.0 + 0.5 * (j % 6), 2.0 + (j % 5), 30.0 + 15.0 * (j % 4))
    lim = ("limiter", -1.0 - 0.75 * (j % 7), 1.0 + 0.5 * (j % 3), 0.5 + 0.25 * (j % 4), 40.0 + 10.0 * (j % 5))
    return user_eq(A, j) + [comp, lim]


def _rows(y, j, ch):
    return y[j * ch:(j + 1) * ch]


def _run(pvs, feeds, events=None, sizes=SIZES):
    """The same calls to every host-row instance (pvs[i] fed feeds[i]; odd sizes, every third call leaving half of the output in
    the ring).  events: {call index: f(produced, ring)} run before that call; produced = output samples per row produced so far,
    ring = how many of them wait in the ring.  Returns every instance's retrieved output, concatenated."""
    n = feeds[0].shape[1]
    pos, k, outs, done, ring = 0, 0, [[] for _ in pvs], 0, 0
    while pos < n:
        if events and k in events:
            events[k](done + ring, ring)
        m = min(sizes[k % len(sizes)], n - pos)
        k += 1
        for pv, X in zip(pvs, feeds):
            pv.processInData(np.ascontiguousarray(X[:, pos:pos + m]))
        avail = pvs[0].getOutSamples()
        take = avail if k % 3 else avail // 2
        for i, pv in enumerate(pvs):
            assert pv.getOutSamples() == avail, f"call {k}: instance {i}"
            outs[i].append(pv.getOutData(take))
        done += take
        ring = avail - take
        pos += m
    return [np.concatenate(o, axis=1) for o in outs]


def _run_device(A, pv, X, events=None, sizes=SIZES):
    """The calls of _run on device rows, all on one CUDA stream, the host never waiting between calls (events run between
    enqueued calls).  int16 rows start at 2-byte-aligned pointers.  Returns the retrieved output."""
    import torch
    s16 = X.dtype == np.int16
    esz, off = (2, 1) if s16 else (4, 0)
    R, n = X.shape
    pitch_in, pitch_out = n + 3, 2 * n + 1
    Xp = np.zeros((R, pitch_in), X.dtype)
    Xp[:, off:off + n] = X
    stream = torch.cuda.Stream()
    dX = torch.from_numpy(Xp).cuda()
    dY = torch.zeros((R, pitch_out), dtype=torch.int16 if s16 else torch.float32, device="cuda")
    torch.cuda.synchronize()
    pos, k, w, done, ring = 0, 0, 0, 0, 0
    with torch.cuda.stream(stream):
        while pos < n:
            if events and k in events:
                events[k](done + ring, ring)
            m = min(sizes[k % len(sizes)], n - pos)
            k += 1
            pv.processInDataDevice(dX.data_ptr() + esz * (off + pos), pitch_in, m, stream.cuda_stream)
            avail = pv.getOutSamples()
            take = avail if k % 3 else avail // 2
            c = pv.getOutDataDevice(dY.data_ptr() + esz * (off + w), pitch_out, take, stream.cuda_stream)
            assert c == take
            w += c
            done += take
            ring = avail - take
            pos += m
    stream.synchronize()
    return dY[:, off:off + w].cpu().numpy()


def _per_stream(pv, chains):
    for j, c in enumerate(chains):
        pv.set_stream_postchain(j, c)


def _same(a, b):
    return np.array_equal(a, b) if a.dtype == np.int16 else np.array_equal(_bits(a), _bits(b))


# ---- 1. distinct parameters from the start ----
ROWS = ["host_f32", "host_s16", "device_f32", "device_s16"]


def _distinct_from_start(A, pvlib, name, S, rows):
    _, kw, sr, ch, secs, seed = _case(name)
    args = ctor_args(kw)
    n = int(sr * min(secs, 0.5))
    X16 = _pcm(n, sr, ch, seed, S)
    Xf = _f32(X16)
    chains = [user_chain(A, j) for j in range(S)]
    plain = A.phasevocoder(sr, ch, *args, streams=S)
    chained = A.phasevocoder(sr, ch, *args, streams=S)
    chained.set_postchain(voice_chain(A))
    _per_stream(chained, chains)
    y, p = _run([chained, plain], [Xf, Xf])
    plain.close()
    chained.close()
    assert y.shape == p.shape and y.shape[1] > 0
    for j in range(S):
        assert np.array_equal(_bits(_rows(y, j, ch)), _bits(hook(pvlib, sr, chains[j], _rows(p, j, ch)))), f"{name}: stream {j}"
    if rows == "host_f32":
        return
    s16 = rows.endswith("s16")
    pv = A.phasevocoder(sr, ch, *args, streams=S, fmt=A.S16 if s16 else A.F32)
    pv.set_postchain(voice_chain(A))
    _per_stream(pv, chains)
    X = X16 if s16 else Xf
    got = _run([pv], [X])[0] if rows == "host_s16" else _run_device(A, pv, X)
    pv.close()
    want = _quant(y) if s16 else y
    assert got.shape == want.shape and _same(got, want), f"{name}: {rows} rows differ from the float32 host rows"


@pytest.mark.parametrize("rows", ROWS)
@pytest.mark.parametrize("name,S", [("cfg4_shift_p7_mono", 64), ("cfg1_shift_p4_stereo", 40)])
def test_distinct_parameters_from_the_start(A, pvlib, name, S, rows):
    """Every stream of a live batch with its own parameters == the hook with that stream's chain on the plain live batch; 40
    stereo streams are 80 rows, three one-warp CTAs of which the last is half full."""
    _distinct_from_start(A, pvlib, name, S, rows)


def test_distinct_parameters_many_ctas(A, pvlib):
    """330 mono streams: eleven CTAs of the chain, the last one a partial warp of 10 rows."""
    _distinct_from_start(A, pvlib, "cfg4_shift_p7_mono", 330, "host_f32")


# ---- 2. identity ----
def test_own_parameters_change_nothing(A):
    """Every stream given the instance's own parameters (before the first call, and again mid-stream) == never calling the
    setter, bitwise.  No stream differs from the chain, so the uniform kernel runs here; the per-row kernel on identical
    parameters is test_per_row_kernel_equals_uniform_kernel."""
    name = "cfg1_shift_p4_stereo"
    kw, sr, ch, X = _live_inputs(name, 6)
    args = ctor_args(kw)
    chain = voice_chain(A)
    ref = A.phasevocoder(sr, ch, *args, streams=6)
    pv = A.phasevocoder(sr, ch, *args, streams=6)
    ref.set_postchain(chain)
    pv.set_postchain(chain)
    _per_stream(pv, [chain] * 6)
    y, r = _run([pv, ref], [X, X], events={9: lambda *_: _per_stream(pv, [chain] * 6), 14: lambda *_: pv.set_stream_postchain(2, chain)})
    pv.close()
    ref.close()
    assert _same(y, r)


def test_per_row_kernel_equals_uniform_kernel(A, monkeypatch):
    """The per-row kernel (forced with PVGPU_POST_PER_ROW=1, read when an instance is created) on identical parameters == the uniform kernel,
    bitwise, float32 and int16."""
    name = "cfg1_shift_p4_stereo"
    _, kw, sr, ch, secs, seed = _case(name)
    args = ctor_args(kw)
    S = 5
    X16 = _pcm(int(sr * 0.5), sr, ch, seed, S)
    for fmt, X in ((A.F32, _f32(X16)), (A.S16, X16)):
        outs = []
        for per_row in ("0", "1"):
            monkeypatch.setenv("PVGPU_POST_PER_ROW", per_row)
            pv = A.phasevocoder(sr, ch, *args, streams=S, fmt=fmt)
            pv.set_postchain(voice_chain(A))
            outs.append(_run([pv], [X])[0])
            pv.close()
        assert outs[0].shape[1] > 0 and _same(outs[0], outs[1]), f"fmt {fmt}"


def test_same_parameters_again_mid_stream_change_nothing(A):
    """Stream j given its current (own) parameters again mid-stream changes nothing."""
    name = "cfg4_shift_p7_mono"
    S = 8
    kw, sr, ch, X = _live_inputs(name, S)
    args = ctor_args(kw)
    chains = [user_chain(A, j) for j in range(S)]
    pvs = [A.phasevocoder(sr, ch, *args, streams=S) for _ in range(2)]
    for pv in pvs:
        pv.set_postchain(voice_chain(A))
        _per_stream(pv, chains)
    y, r = _run(pvs, [X, X], events={11: lambda *_: pvs[0].set_stream_postchain(3, chains[3])})
    for pv in pvs:
        pv.close()
    assert _same(y, r)


# ---- 3. a mid-stream update keeps the state and touches no other stream ----
def _fx_coef(A, sr, fx):
    """(kind, float32 coefficients, delay) as make_postchain converts them; its own restatement except for biquad_design."""
    f32 = np.float32
    if fx[0] == "gain":
        return "gain", [f32(fx[1])], 0
    if fx[0] == "compressor":
        thr, ratio, mk, ta, tr = (f32(v) for v in fx[1:])
        return "compressor", [thr, ratio, mk, f32(math.exp(-1 / (0.001 * sr * float(ta)))), f32(math.exp(-1 / (0.001 * sr * float(tr))))], 0
    if fx[0] == "limiter":
        thr, mk, ta, tr = (float(f32(v)) for v in fx[1:])
        return "limiter", [f32(10.0 ** (mk / 20.0)), f32(10.0 ** ((thr - 0.01) / 20.0)), f32(math.exp(-1.0 / (sr * 0.001 * ta))),
                           f32(math.exp(-1.0 / (sr * 0.001 * tr)))], int(sr * 0.001 * 6.0) + 1
    return "biquad", [f32(c) for c in A.biquad_design(int(fx[1]), sr, fx[2], fx[3], fx[4])], 0


def restate(A, sr, chain, new_chain, b, x):
    """One row x through `chain`, switching to new_chain's coefficients at sample b with every effect's state kept."""
    f32 = np.float32
    co, co2 = [_fx_coef(A, sr, f) for f in chain], [_fx_coef(A, sr, f) for f in new_chain]
    assert [c[0] for c in co] == [c[0] for c in co2] and [c[2] for c in co] == [c[2] for c in co2]
    st = []
    for kind, _, delay in co:
        if kind == "biquad":
            st.append([f32(0)] * 4)
        elif kind == "compressor":
            st.append([0.0])
        elif kind == "limiter":
            st.append([10.0 ** (-120.0 / 20.0), 1.0, [0.0] * delay, 0])
        else:
            st.append(None)
    y = np.empty(len(x), np.float32)
    for i in range(len(x)):
        cur = co if i < b else co2
        v = f32(x[i])
        for (kind, p, delay), s in zip(cur, st):
            if kind == "gain":                    # float32, exact
                v = min(max(f32(v * p[0]), f32(-1)), f32(1))
            elif kind == "biquad":                # float32 in the kernel's order, exact
                acc = f32(p[0] * v)
                acc = f32(acc + f32(p[1] * s[0]))
                acc = f32(acc + f32(p[2] * s[1]))
                acc = f32(acc - f32(p[4] * s[2]))
                acc = f32(acc - f32(p[5] * s[3]))
                out = f32(acc / p[3])
                s[1], s[3], s[0], s[2] = s[0], s[2], v, out
                v = out
            elif kind == "compressor":            # float64
                thr, ratio, mk, aa, ar = (float(c) for c in p)
                xv = float(v)
                ax = abs(xv)
                dbx = -120.0 if ax < 1e-6 else 20.0 * math.log10(ax)
                dby = thr + (dbx - thr) / ratio if dbx >= thr else dbx
                dbl = dbx - dby
                alpha = aa if dbl > s[0] else ar
                s[0] = alpha * s[0] + (1.0 - alpha) * dbl
                v = xv * 10.0 ** ((mk - s[0]) / 20.0)
            else:                                 # limiter, float64
                mk, thr, aa, ar = (float(c) for c in p)
                xv = float(v) * mk
                xa = max(abs(xv), 1e-6)
                alpha = aa if xa > s[0] else ar
                s[0] = alpha * s[0] + (1.0 - alpha) * xa
                gain = min(1.0, thr / s[0])
                alpha = aa if gain < s[1] else ar
                s[1] = alpha * s[1] + (1.0 - alpha) * gain
                out = s[2][s[3]] * s[1]
                s[2][s[3]] = xv
                s[3] = (s[3] + 1) % delay
                v = min(max(out, -1.0), 1.0)
        y[i] = v
    return y


LIMITER = [("limiter", -6.0, 2.0, 1.0, 80.0)]
UPDATES = {   # chain, stream j's update, exact
    "eq_gain": (lambda A: A.equalizer_chain(EQ_PARAMS) + [("gain", 0.8)], lambda A: user_eq(A, 4) + [("gain", 1.3)], True),
    "voice": (voice_chain, lambda A: user_chain(A, 5), False),
    "limiter_ceiling": (lambda A: LIMITER, lambda A: [("limiter", -14.0, 2.0, 1.0, 80.0)], False),
}


@pytest.mark.parametrize("what", list(UPDATES))
def test_mid_stream_update_keeps_state_and_isolation(A, what):
    """Stream j updated before call k: every other stream and stream j's samples produced before the call (those waiting in the
    ring included) are bit-identical to a run without the update; stream j equals the restatement with the switch at the first
    sample produced by call k.  The limiter case changes the ceiling while the 6 ms delay line is full."""
    name = "cfg1_shift_p4_stereo"
    _, kw, sr, ch, secs, seed = _case(name)
    args = ctor_args(kw)
    S, j, k = 3, 1, 12
    n = int(sr * 0.4)
    X = np.ascontiguousarray(np.concatenate([make_input(name, sr, ch, n / sr, seed + 11 * i)[:, :n] for i in range(S)], axis=0))
    make_chain, make_update, exact = UPDATES[what]
    chain, upd = make_chain(A), make_update(A)
    pv, same, plain = (A.phasevocoder(sr, ch, *args, streams=S) for _ in range(3))
    pv.set_postchain(chain)
    same.set_postchain(chain)
    at = {}

    def update(produced, ring):
        at["b"], at["ring"] = produced, ring
        pv.set_stream_postchain(j, upd)

    y, r, p = _run([pv, same, plain], [X, X, X], events={k: update})
    for o in (pv, same, plain):
        o.close()
    b = at["b"]
    assert at["ring"] > 0 and b > 300 and b < y.shape[1] - 1000, "the update should find a full delay line and samples in the ring"
    for i in range(S):
        if i != j:
            assert _same(_rows(y, i, ch), _rows(r, i, ch)), f"stream {i} changed"
    assert _same(_rows(y, j, ch)[:, :b], _rows(r, j, ch)[:, :b]), "samples produced before the update changed"
    assert not _same(_rows(y, j, ch)[:, b:], _rows(r, j, ch)[:, b:])
    want = np.stack([restate(A, sr, chain, upd, b, row) for row in _rows(p, j, ch)])
    got = _rows(y, j, ch)
    if exact:
        assert _same(got, want)
    else:
        assert_parity(got, want, what)


# ---- 4. coalescing and ordering ----
def test_updates_coalesce(A):
    """Several updates of one stream between two calls == the last one alone."""
    name = "cfg4_shift_p7_mono"
    S = 4
    kw, sr, ch, X = _live_inputs(name, S)
    args = ctor_args(kw)
    pvs = [A.phasevocoder(sr, ch, *args, streams=S) for _ in range(2)]
    for pv in pvs:
        pv.set_postchain(voice_chain(A))

    def update(*_):
        for c in (user_chain(A, 7), user_chain(A, 8), voice_chain(A), user_chain(A, 9)):
            pvs[0].set_stream_postchain(2, c)
        pvs[1].set_stream_postchain(2, user_chain(A, 9))

    y, r = _run(pvs, [X, X], events={10: update})
    for pv in pvs:
        pv.close()
    assert _same(y, r)


@pytest.mark.parametrize("s16", [False, True], ids=["f32", "s16"])
def test_device_row_updates_equal_host_row_updates(A, s16):
    """Updates between device-row calls on one caller stream, the host never waiting == the same sequence on host rows."""
    name = "cfg1_shift_p4_stereo"
    _, kw, sr, ch, secs, seed = _case(name)
    args = ctor_args(kw)
    S = 6
    X16 = _pcm(int(sr * 0.5), sr, ch, seed, S)
    X = X16 if s16 else _f32(X16)
    fmt = A.S16 if s16 else A.F32
    outs = []
    for dev in (False, True):
        pv = A.phasevocoder(sr, ch, *args, streams=S, fmt=fmt)
        pv.set_postchain(voice_chain(A))
        events = {0: lambda *_: pv.set_stream_postchain(1, user_chain(A, 1)),
                  8: lambda *_: _per_stream(pv, [user_chain(A, 10 + i) for i in range(S)]),
                  9: lambda *_: pv.set_stream_postchain(4, voice_chain(A)),
                  13: lambda *_: (pv.set_stream_postchain(0, user_chain(A, 3)), pv.set_stream_postchain(0, user_chain(A, 2)))}
        outs.append(_run_device(A, pv, X, events) if dev else _run([pv], [X], events)[0])
        pv.close()
    assert outs[0].shape == outs[1].shape and outs[0].shape[1] > 0 and _same(outs[0], outs[1])


def test_set_postchain_discards_per_stream_parameters(A, pvlib):
    """pvgpu_set_postchain after per-stream updates == a fresh instance with that chain (before the first call); mid-stream, the
    output from the set on == the hook with the new chain on the plain output."""
    name = "cfg1_shift_p4_stereo"
    S = 4
    kw, sr, ch, X = _live_inputs(name, S)
    args = ctor_args(kw)
    C2 = [("compressor", -18.0, 3.0, 2.0, 4.0, 40.0), ("limiter", -2.0, 1.0, 1.0, 60.0)]
    fresh, pv, mid, plain = (A.phasevocoder(sr, ch, *args, streams=S) for _ in range(4))
    fresh.set_postchain(voice_chain(A))
    pv.set_postchain(voice_chain(A))
    _per_stream(pv, [user_chain(A, j) for j in range(S)])
    pv.set_postchain(voice_chain(A))
    mid.set_postchain(C2)
    _per_stream(mid, [[("compressor", -10.0 - j, 2.0, 1.0, 3.0, 30.0), ("limiter", -4.0, 1.0, 1.0, 50.0)] for j in range(S)])
    at = {}

    def reset(produced, ring):
        at["b"] = produced
        mid.set_postchain(C2)

    y, f, m, p = _run([pv, fresh, mid, plain], [X] * 4, events={12: reset})
    for o in (pv, fresh, mid, plain):
        o.close()
    assert _same(y, f)
    b = at["b"]
    assert 0 < b < m.shape[1]
    assert _same(m[:, b:], hook(pvlib, sr, C2, p[:, b:]))


# ---- 5. errors ----
def test_arguments(A, pvlib):
    from audiomod_b200 import _lib
    from audiomod_b200.phasevocoder import _fx_array
    L = pvlib
    name = "cfg4_shift_p7_mono"
    S = 2
    kw, sr, ch, X = _live_inputs(name, S)
    args = ctor_args(kw)
    chain = voice_chain(A)
    pv, ref = (A.phasevocoder(sr, ch, *args, streams=S) for _ in range(2))
    for o in (pv, ref):
        o.set_postchain(chain)
        _per_stream(o, [user_chain(A, 0), user_chain(A, 1)])
    good, n = _fx_array(user_chain(A, 6))
    short, n_short = _fx_array(chain[:-1])
    swapped, _ = _fx_array(chain[:-2] + [chain[-1], chain[-2]])
    ratio0, _ = _fx_array(chain[:-2] + [("compressor", -10.0, 0.0, 6.0, 10.0, 100.0), chain[-1]])
    bad = [(-1, good, n, "stream -1 outside [0, 2)"), (2, good, n, "stream 2 outside [0, 2)"),
           (0, short, n_short, f"chain of {n_short} effects; this instance's chain has {n}"),
           (0, swapped, n, f"effect {n - 2} is a limiter; this instance's effect {n - 2} is a compressor"),
           (0, None, n, "null chain"), (1, ratio0, n, "compressor ratio must be positive")]

    def errors(*_):
        for stream, arr, cnt, msg in bad:
            assert L.pvgpu_set_stream_postchain(pv._h, stream, arr, cnt) == _lib.EINVAL, msg
            assert L.pvgpu_last_error().decode() == msg

    y, r = _run([pv, ref], [X, X], events={0: errors, 9: errors})
    assert _same(y, r), "a refused update changed the output"
    pv.close()
    ref.close()
    with pytest.raises(A.PvgpuError):
        pv = A.phasevocoder(sr, ch, *args, streams=S)
        try:
            pv.set_stream_postchain(0, chain)                   # no chain on the instance
        finally:
            assert L.pvgpu_last_error().decode() == "this instance has no post-chain (pvgpu_set_postchain first)"
            pv.close()
    # a single instance is a live batch of one
    one = A.phasevocoder(sr, ch, *args)
    one.set_postchain(chain)
    one.set_stream_postchain(0, user_chain(A, 3))
    with pytest.raises(A.PvgpuError):
        one.set_stream_postchain(1, user_chain(A, 3))
    one.close()
    # an instance whose mode does nothing: the call succeeds and changes nothing
    pv = A.phasevocoder(44100, 1, 1.0, 0.0, 42, 1, 2048)
    pv.set_postchain(chain)
    pv.set_stream_postchain(0, user_chain(A, 2))
    pv.processInData(np.zeros((1, 4800), np.float32))
    assert pv.getOutSamples() == 0
    pv.close()
