"""Stage tests of the analysis kernels and the phase core against the reference restatement (run with -m gpu on a B200).

Analysis (k_analyse_t, k_analyse): every bin bit-identical to oracle.forward_polar of the frame built here, polar and Cartesian,
float32 and int16 rows, aligned / misaligned / partial gathers, in_base offsets and a frame index past 2^32 samples.
Phase core (k_lock_peaks + k_lock_chain on Cartesian spectra; k_phase_lock_t, k_phase_core, k_int_ratio on polar spectra) on the
constructed inputs of test_stage_inputs.py against oracle.phase_core_frames: frame kinds, peak counts, the region of every bin and
every observed rotation bit-identical; rotated bins within 1e-6 |X| (the rotation's sincosf); polar output phases bit-identical.
A failure names the row, frame, bin and decision that differ.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from test_stage_inputs import GENERATORS, hop_of, phase_inc, stream

pytestmark = pytest.mark.gpu

_fp = C.POINTER(C.c_float)
_ip = C.POINTER(C.c_int)
# sqrtf of a subnormal square resolves magnitudes to about sqrt(2^-149) (3.7e-23): the reference's magnitude of a bin scaled to
# 1e-23 can be 0 while the rotated (re, im) keeps it
FLOOR = 2.0 * np.sqrt(2.0 ** -149)
REL = 1e-6
NF = 70   # > 2 * 32 + 1: two full runs of k_lock_peaks plus a part run


def _p(a):
    return a.ctypes.data_as(_fp)


def _i(a):
    return a.ctypes.data_as(_ip)


@pytest.fixture(scope="module")
def L(pvlib):
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return pvlib


def _cfg(n, hop=0, channels=1, coremode=1, mode=0):
    from audiomod_b200 import _lib
    return _lib.Config(sample_rate=44100, channels=channels, time_ratio=1.0, pitch_semitones=0.0, mode=mode, coremode=coremode,
                       fftsize=n, hopsize=hop, device=0)


def _err(L):
    return L.pvgpu_last_error().decode()


# ---------------------------------------------------------------------------------------------------------------------------
# analysis
# ---------------------------------------------------------------------------------------------------------------------------
def _analyse(L, n, hop, spec, fmt, x, in_base, n_in, k0, nf):
    rows, stride = x.shape
    h = n // 2 + 1
    a, b = np.zeros((rows, nf, h), np.float32), np.zeros((rows, nf, h), np.float32)
    n_in = np.ascontiguousarray(n_in, np.int64)
    cfg = _cfg(n, hop)
    rc = L.pvgpu_test_analyse(C.byref(cfg), spec, fmt, rows, x.ctypes.data_as(C.c_void_p), stride, in_base,
                              n_in.ctypes.data_as(C.POINTER(C.c_int64)), k0, nf, _p(a), _p(b))
    assert rc == 0, _err(L)
    return a, b


def _check_analysis(oracle, n, hop, spec, fmt, x, in_base, n_in, k0, nf, a, b):
    rows, stride = x.shape
    xf = x.astype(np.float32) * np.float32(1.0 / 32768.0) if fmt == 1 else x
    for r in range(rows):
        for f in range(nf):
            s = (k0 + f) * hop
            fr = np.zeros(n, np.float32)
            m = max(0, min(n, int(n_in[r]) - s))   # samples of the frame that exist
            if m:
                fr[:m] = xf[r, s - in_base:s - in_base + m]
            rm, rp, ri = oracle.forward_polar(fr)
            ea, eb = (ri[:, 0], ri[:, 1]) if spec else (rm, rp)
            for got, want, what in ((a[r, f], ea, "re" if spec else "mag"), (b[r, f], eb, "im" if spec else "phase")):
                bad = np.flatnonzero(got.view(np.uint32) != want.view(np.uint32))
                assert bad.size == 0, (f"N={n} hop={hop} spec={spec} fmt={fmt}: row {r} frame {k0 + f} ({m} samples) {what} differs "
                                       f"at {bad.size} bins, first bin {bad[0]}: {got[bad[0]]!r} != {want[bad[0]]!r}")


def _rows(rng, fmt, rows, stride):
    if fmt == 1:
        x = rng.integers(-32768, 32768, (rows, stride)).astype(np.int16)
        x[:, :4] = [-32768, 32767, -1, 1]
        return x
    return (rng.standard_normal((rows, stride)) * 0.3).astype(np.float32)


@pytest.mark.parametrize("spec,fmt", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192, 16384])
def test_analyse_bit_exact(L, oracle, n, spec, fmt):
    if spec and n in (256, 16384):
        pytest.skip("Cartesian spectra exist for 512..8192 only (argument test below)")
    rng = np.random.default_rng(n + 10 * spec + fmt)
    for hop in (n // 4, n // 4 + 1):   # even and odd hops: frame starts of both parities
        nf, rows = 12, 4
        k0, in_base = 3, 3 * hop - 7   # the rows start 7 samples before the first frame
        stride = (k0 + nf - 1) * hop + n - in_base + 5
        stride |= 1   # odd row pitch: rows of both alignments
        x = _rows(rng, fmt, rows, stride)
        end = in_base + stride
        n_in = [end,                              # every frame whole
                (k0 + 5) * hop + n,               # frame k0+5 ends exactly at n_in, later ones inside it, then past it
                (k0 + 4) * hop + n // 2 + 1,      # ends inside frame k0+4 on an odd count (a sample pair half in)
                (k0 + 2) * hop]                   # frames from k0+2 on wholly past the end
        a, b = _analyse(L, n, hop, spec, fmt, x, in_base, n_in, k0, nf)
        _check_analysis(oracle, n, hop, spec, fmt, x, in_base, n_in, k0, nf, a, b)


@pytest.mark.parametrize("spec,fmt", [(0, 0), (1, 1)])
def test_analyse_past_2_32_samples(L, oracle, spec, fmt):
    n, hop, nf = 2048, 509, 6
    k0 = (1 << 32) // hop + 5
    assert k0 * hop > 1 << 32
    in_base = k0 * hop - 3
    stride = (nf - 1) * hop + n + 3
    x = _rows(np.random.default_rng(5), fmt, 3, stride)
    n_in = [in_base + stride, k0 * hop + 2 * hop + n - 1, in_base + 3 + 3 * hop + 100]
    a, b = _analyse(L, n, hop, spec, fmt, x, in_base, n_in, k0, nf)
    _check_analysis(oracle, n, hop, spec, fmt, x, in_base, n_in, k0, nf, a, b)


def test_analyse_argument_errors(L):
    x = np.zeros((2, 4096), np.float32)
    n_in = np.full(2, 4096, np.int64)
    a = np.zeros((2, 2, 1025), np.float32)

    def call(cfg, spec=0, fmt=0, rows=2, stride=4096, in_base=0, k0=0, nf=2):
        return L.pvgpu_test_analyse(C.byref(cfg), spec, fmt, rows, x.ctypes.data_as(C.c_void_p), stride, in_base,
                                    n_in.ctypes.data_as(C.POINTER(C.c_int64)), k0, nf, _p(a), _p(a))
    assert call(_cfg(2048, 512)) == 0
    assert call(_cfg(2048, 0)) == 1                       # no explicit hop
    assert call(_cfg(256, 64), spec=1) == 1               # Cartesian spectra only for 512..8192
    assert call(_cfg(16384, 64), spec=1) == 1
    assert call(_cfg(2048, 512), spec=2) == 1
    assert call(_cfg(2048, 512), fmt=2) == 1
    assert call(_cfg(2048, 512), nf=0) == 1
    assert call(_cfg(2048, 512), stride=2000) == 1        # reads past the rows
    assert call(_cfg(2048, 512), in_base=1) == 1          # reads before the rows
    assert call(_cfg(2048, 512), in_base=1, k0=4) == 0


# ---------------------------------------------------------------------------------------------------------------------------
# phase core
# ---------------------------------------------------------------------------------------------------------------------------
KINDS = list(GENERATORS)


@functools.lru_cache(maxsize=2)
def _inputs(n, ch, kinds, nf, coremode):
    """One stream per kind (re_im [S][ch][nf][H][2]), phase increments, polar spectra and the reference's core per stream."""
    from oracle import pv_oracle as O
    x = np.stack([stream(k, n, ch, nf) for k in kinds])
    inc = phase_inc(n, nf)
    mag, ph = O.polar(x)
    refs = [O.phase_core_frames(mag[s], ph[s], inc, hop_of(n), coremode) for s in range(len(kinds))]
    return x, inc, mag, ph, refs


def _core(L, n, ch, spec, kinds, fpl, coremode=1, synth=False, nf=NF):
    """The streams of _inputs through pvgpu_test_phase_core, fpl frames per launch; returns (_inputs(...), outputs)."""
    h, half, maxpk = n // 2 + 1, n // 2, n // 6 + 2
    S = len(kinds)
    inp = _inputs(n, ch, tuple(kinds), nf, coremode)
    x, inc, mag, ph, _ = inp
    a, b = (x[..., 0], x[..., 1]) if spec else (mag, ph)
    rows = S * ch
    o = dict(kind=np.zeros((rows, nf), np.int32), npeaks=np.zeros((rows, nf), np.int32), region=np.zeros((rows, nf, half), np.int32),
             csn=np.zeros((rows, nf, maxpk, 2), np.float32), rot=np.zeros((rows, nf, maxpk), np.float32),
             out_a=np.zeros((rows, nf, h), np.float32), out_b=np.zeros((rows, nf, h), np.float32),
             frames=np.zeros((rows, nf, n), np.float32) if synth else None)
    cfg = _cfg(n, hop_of(n), ch, coremode)
    a2, b2 = np.ascontiguousarray(a.reshape(rows, nf, h)), np.ascontiguousarray(b.reshape(rows, nf, h))
    rc = L.pvgpu_test_phase_core(C.byref(cfg), spec, S, nf, fpl, _i(inc), _p(a2), _p(b2), _i(o["kind"]), _i(o["npeaks"]),
                                 _i(o["region"]), _p(o["csn"]), _p(o["rot"]), _p(o["out_a"]), _p(o["out_b"]),
                                 _p(o["frames"]) if synth else None)
    assert rc == 0, _err(L)
    return inp, o


def _where(kinds, ch, r, f):
    return f"stream {r // ch} ({kinds[r // ch]}) channel {r % ch} frame {f}"


def _check_cartesian(oracle, n, ch, kinds, inp, o, what):
    half = n // 2
    x, _, mags, _, refs = inp
    worst = 0.0
    for s, kind in enumerate(kinds):
        mag, ref = mags[s], refs[s]
        for c in range(ch):
            r = s * ch + c
            for f in range(x.shape[2]):
                at = f"{what}: {_where(kinds, ch, r, f)}"
                kd, npk = o["kind"][r, f], o["npeaks"][r, f]
                assert kd == ref["branch"][c, f], f"{at}: frame kind {kd} != reference {ref['branch'][c, f]}"
                assert npk == ref["npeak"][c, f], f"{at}: {npk} peaks != reference {ref['npeak'][c, f]}"
                want = mag[c, f].astype(np.float64) * np.exp(1j * ref["out_phase"][c, f].astype(np.float64))
                xi = x[s, c, f, :, 0].astype(np.float64) + 1j * x[s, c, f, :, 1]
                if kd == 2:
                    b1, b2 = ref["bin1"][c, f, :npk], ref["bin2"][c, f, :npk]
                    rg = np.repeat(np.arange(npk), b2 - b1)
                    bad = np.flatnonzero(o["region"][r, f] != rg)
                    assert bad.size == 0, (f"{at}: bin {bad[0]} in region {o['region'][r, f, bad[0]]}, reference {rg[bad[0]]} "
                                           f"(peaks {ref['peaks'][c, f, max(0, rg[bad[0]] - 1):rg[bad[0]] + 2]})")
                    rot = o["rot"][r, f, :npk]
                    seen = ~np.isnan(rot)
                    if seen.any():
                        rr = ref["rot"][c, f, :npk]
                        bad = np.flatnonzero(seen & (rot.view(np.uint32) != rr.view(np.uint32)))
                        assert bad.size == 0, f"{at}: rotation of peak {bad[0]} (bin {ref['peaks'][c, f, bad[0]]}) {rot[bad[0]]!r} != {rr[bad[0]]!r}"
                    cs = o["csn"][r, f, :npk].astype(np.float64)
                    got = xi[:half] * (cs[rg, 0] + 1j * cs[rg, 1])
                elif kd == 1:
                    got = o["out_a"][r, f, :half].astype(np.float64) + 1j * o["out_b"][r, f, :half]
                else:
                    got = xi[:half]
                dev = np.abs(got - want[:half])
                lim = REL * np.abs(want[:half]) + FLOOR
                bad = np.flatnonzero(dev > lim)
                assert bad.size == 0, f"{at}: kind {kd} bin {bad[0]} off by {dev[bad[0]]:.3e} (|X| {abs(want[bad[0]]):.3e})"
                nz = np.abs(want[:half]) > FLOOR / REL   # bins where the relative bar binds
                if nz.any():
                    worst = max(worst, float(np.max(dev[:half][nz] / np.abs(want[:half][nz]))))
                # the Nyquist bin passes through every core
                assert o["out_a"][r, f, half] == x[s, c, f, half, 0] and o["out_b"][r, f, half] == x[s, c, f, half, 1], at
            if o["frames"] is not None:
                for f in range(x.shape[2]):
                    want = oracle.inverse_polar(mag[c, f] * np.float32(1.0 / n), ref["out_phase"][c, f], n)
                    got = o["frames"][s * ch + c, f]
                    assert np.max(np.abs(got - want)) <= 2e-6 * max(1.0, float(np.max(np.abs(want)))), f"{what}: synthesis {_where(kinds, ch, s * ch + c, f)}"
    return worst


@pytest.mark.parametrize("fpl", [1, 5, 32, 33, NF])
@pytest.mark.parametrize("ch", [1, 2, 3])
@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 8192])
def test_lock_core_cartesian(L, oracle, n, ch, fpl):
    """k_lock_peaks<N, kC> + k_lock_chain<kC> (kC = 1, 2 and the run-time variant for 3 channels) on every constructed input:
    decisions and observed rotations bit-identical, rotated bins within 1e-6 |X|."""
    if ch == 3 and n == 8192:
        pytest.skip("3 channels at 8192 take the polar core (shared memory); see test_phase_core_argument_errors")
    synth = fpl in (1, NF)
    inp, o = _core(L, n, ch, 1, KINDS, fpl, synth=synth)
    what = f"N={n} C={ch} frames/launch={fpl}"
    worst = _check_cartesian(oracle, n, ch, KINDS, inp, o, what)
    if fpl == 1:   # every locked frame's rotation was observed
        locked = int((o["kind"] == 2).sum())
        assert locked > 0 and int((~np.isnan(o["rot"][..., 0]) & (o["kind"] == 2)).sum()) == locked
    print(f"{what}: largest |rotated - reference| / |X| = {worst:.2e}")


def _check_polar(ch, kinds, inp, o, what):
    _, _, mags, _, refs = inp
    for s, kind in enumerate(kinds):
        mag, ref = mags[s], refs[s]
        for c in range(ch):
            r = s * ch + c
            got, want = o["out_b"][r], ref["out_phase"][c]
            bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
            if bad.size:
                f, i = bad[0]
                raise AssertionError(f"{what}: {_where(kinds, ch, r, f)} (reference branch {ref['branch'][c, f]}, {ref['npeak'][c, f]} peaks): "
                                     f"{len(bad)} phases differ, first bin {i}: {got[f, i]!r} != {want[f, i]!r}")
            assert np.array_equal(o["out_a"][r].view(np.uint32), mag[c].view(np.uint32)), what


@pytest.mark.parametrize("fpl", [5, NF])
@pytest.mark.parametrize("ch", [1, 3])
@pytest.mark.parametrize("n", [512, 1024, 2048, 4096, 8192])
def test_phase_lock_t_polar(L, oracle, n, ch, fpl):
    """k_phase_lock_t (coremode 1 on polar spectra at the templated sizes): output phases bit-identical."""
    inp, o = _core(L, n, ch, 0, KINDS, fpl)
    assert (o["kind"] == -1).all()
    _check_polar(ch, KINDS, inp, o, f"k_phase_lock_t N={n} C={ch} frames/launch={fpl}")


@pytest.mark.parametrize("n,ch,coremode", [(256, 2, 1), (16384, 1, 1), (256, 2, 0), (16384, 1, 0), (2048, 2, 0), (2048, 2, 2), (256, 1, 2)])
def test_phase_core_polar(L, oracle, n, ch, coremode):
    """k_phase_core<true> / <false> at the generic sizes, coremode 0 at a templated size, and k_int_ratio (coremode 2)."""
    for fpl in (7, 40):
        inp, o = _core(L, n, ch, 0, KINDS, fpl, coremode=coremode, nf=40)
        _check_polar(ch, KINDS, inp, o, f"coremode {coremode} N={n} C={ch} frames/launch={fpl}")


def test_phase_core_argument_errors(L):
    h, nf = 1025, 4
    a = np.zeros((2, nf, h), np.float32)
    inc = np.full(nf, 512, np.int32)
    big = np.zeros((3, nf, 4097), np.float32)

    def call(cfg, spec=1, streams=1, nf_=nf, fpl=2, src=a, out=a):
        return L.pvgpu_test_phase_core(C.byref(cfg), spec, streams, nf_, fpl, _i(inc), _p(src), _p(src), None, None, None, None, None,
                                       _p(out), _p(out), None)
    assert call(_cfg(2048, 512, 2)) == 0
    assert call(_cfg(2048, 512, 2), spec=0) == 0
    assert call(_cfg(2048, 512, 2, coremode=0)) == 1            # spec 1 is the phase-locked core only
    assert call(_cfg(2048, 512, 2, coremode=2)) == 1
    assert call(_cfg(2048, 512, 2, mode=6)) == 1                # robotic: no phase core
    assert call(_cfg(2048, 512, 2, mode=-1), spec=0) == 1       # constant
    assert call(_cfg(8192, 2048, 3), src=big, out=big) == 1     # 3 channels at 8192: polar core only
    assert call(_cfg(8192, 2048, 3), spec=0, src=big, out=big) == 0
    assert call(_cfg(2048, 512, 2), spec=2) == 1
    assert call(_cfg(2048, 512, 2), streams=0) == 1
    assert call(_cfg(2048, 512, 2), nf_=0) == 1
    assert call(_cfg(2048, 512, 2), fpl=0) == 1
    assert L.pvgpu_test_phase_core(C.byref(_cfg(2048, 512, 2)), 1, 1, nf, 2, _i(inc), _p(a), _p(a), None, None, None, None, None,
                                   None, _p(a), None) == 1
