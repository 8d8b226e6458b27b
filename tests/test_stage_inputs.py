"""Constructed spectra for the stage tests of the phase core (tests/test_gpu_stage_core.py), and CPU checks that each generator
really produces the case it aims at: the reference's phase core (oracle.phase_core_frames) is run on every generator's output and
its peaks, branches and regions are asserted.  Without these checks a generator could quietly stop covering anything.

Every generator returns Cartesian spectra re_im [channels][frames][N/2+1][2] float32 of one stream.  The GPU tests feed them to
the phase-locked core on Cartesian spectra as they are, and to the polar cores and the reference through oracle.polar, so both
sides start from the same bins.
"""
import numpy as np
import pytest

from audiomod_b200.synth import synth

SIZES = (512, 1024, 2048, 4096, 8192)


def hop_of(n):
    return n // 4


def _rand_phase(rng, shape):
    return rng.uniform(-np.pi, np.pi, shape)


def _pack(mag, ph):
    return np.stack([mag * np.cos(ph), mag * np.sin(ph)], axis=-1).astype(np.float32)


def _flat(mag, rng):
    """Peaks of mag with random phases over a flat background of bins (0.05, 0): equal magnitudes, so no peaks of its own."""
    ph = np.where(mag == 0.05, 0.0, _rand_phase(rng, mag.shape))
    return _pack(mag, ph)


def _low(rng, n, nf, h, scale=0.1):
    """Background bins: small random magnitudes (every bin is within two bins of a constructed high bin, or may be a peak)."""
    return _pack(rng.uniform(0.0, scale, (nf, h)), _rand_phase(rng, (nf, h)))


# ---- generators: one stream's frames, [ch][nf][H][2] -------------------------------------------------------------------------
def natural(n, ch, nf, seed):
    """oracle.forward_polar spectra of synth() audio at the configuration's hop."""
    from oracle import pv_oracle as O
    hop = hop_of(n)
    x = synth(seed, 44100, (n + (nf - 1) * hop) / 44100.0 + 0.01, ch)
    return np.stack([np.stack([O.forward_polar(x[c, k * hop:k * hop + n])[2] for k in range(nf)]) for c in range(ch)])


def noise(n, ch, nf, seed):
    """White-noise spectra: about half / 5 peaks per frame (more than 2 x 128 at N >= 4096)."""
    rng = np.random.default_rng(seed)
    return rng.standard_normal((ch, nf, n // 2 + 1, 2)).astype(np.float32)


def max_density(n, ch, nf, seed):
    """A peak every third bin from bin 2 up to half - 3: (half - 5) // 3 + 1 peaks per frame."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = np.empty((ch, nf, h, 2), np.float32)
    for c in range(ch):
        mag = rng.uniform(0.0, 1.0, (nf, h))
        pk = np.arange(2, half - 2, 3)
        mag[:, pk] = rng.uniform(2.0, 3.0, (nf, pk.size))
        out[c] = _pack(mag, _rand_phase(rng, (nf, h)))
    return out


def ulp_ties(n, ch, nf, seed):
    """Candidate bins whose squared magnitude exceeds their largest neighbour's by 1..40 ulp: the rounded square roots are equal
    for some (not a peak) and differ for others (a peak); the small ones are the exact-sqrt path of lock_is_peak."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = np.empty((ch, nf, h, 2), np.float32)
    cand = np.arange(3, half - 4, 6)
    for c in range(ch):
        for f in range(nf):
            fr = _low(rng, n, 1, h, 0.05)[0]
            v = rng.uniform(0.5, 2.0, cand.size).astype(np.float32)
            q = v * v
            k = rng.integers(1, 41, cand.size)
            k[: min(cand.size, 8)] = np.arange(1, min(cand.size, 8) + 1)   # the smallest steps in every frame
            t = np.sqrt(k * np.spacing(q)).astype(np.float32)
            sr = np.where(rng.random(cand.size) < 0.5, -1, 1).astype(np.float32)
            si = np.where(rng.random(cand.size) < 0.5, -1, 1).astype(np.float32)
            fr[cand + 1, 0], fr[cand + 1, 1] = v * sr, 0.0          # the largest neighbour: q = fl(v^2)
            fr[cand, 0], fr[cand, 1] = v * sr, t * si               # the candidate: fl(fl(v^2) + fl(t^2))
            out[c, f] = fr
    return out


def plateaus(n, ch, nf, seed):
    """Exactly equal neighbours (plateaus of two and three bins, no peak), between true peaks."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = np.empty((ch, nf, h, 2), np.float32)
    for c in range(ch):
        fr = _low(rng, n, nf, h, 0.05)
        for b in range(4, half - 8, 16):
            v = rng.uniform(1.0, 2.0, (nf, 1)).astype(np.float32)
            fr[:, b:b + 2] = np.stack([v, np.zeros_like(v)], -1)                    # two equal bins
            fr[:, b + 5:b + 8] = np.stack([np.zeros_like(v), v], -1)                # three equal bins (im only: same q)
            fr[:, b + 11] = np.concatenate([v * 1.5, v * 0.5], -1)                  # a true peak
        out[c] = fr
    return out


def tiny(n, ch, nf, seed):
    """Bins scaled to 1e-19 .. 1e-23: squared magnitudes that are subnormal, zero, and always below the 1e-30 guard."""
    rng = np.random.default_rng(seed)
    h = n // 2 + 1
    scale = 10.0 ** -rng.uniform(19, 23.5, (ch, nf, 1, 1))
    return (rng.standard_normal((ch, nf, h, 2)) * scale).astype(np.float32)


def edges(n, ch, nf, seed):
    """Even frames: peaks at bins 2 and half - 3.  Odd frames: dominant bins 0, 1, half - 2, half - 1 and a large Nyquist bin,
    which are never peaks.  Interior peaks in both."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = np.empty((ch, nf, h, 2), np.float32)
    for c in range(ch):
        mag = rng.uniform(0.0, 0.1, (nf, h))
        mag[:, 8:half - 8:7] = rng.uniform(1.0, 2.0, (nf, len(range(8, half - 8, 7))))
        mag[0::2, [2, half - 3]] = 5.0
        mag[1::2, [0, 1, half - 2, half - 1, half]] = 1e3
        out[c] = _pack(mag, _rand_phase(rng, (nf, h)))
    return out


def links(n, ch, nf, seed):
    """Alternating frames: previous peaks at c - d and c + d (d = 2..6, equal distance: the link keeps the lower one) and at
    c - d, c + d + 1, then current peaks at c.  Peak sums of both parities set the region starts."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = np.empty((ch, nf, h, 2), np.float32)
    centres = np.arange(10, half - 10, 16)
    d = 2 + (np.arange(centres.size) % 5)
    odd = (np.arange(centres.size) // 5) % 2
    for c in range(ch):
        mag = np.full((nf, h), 0.05)   # a flat background has no peaks of its own
        for f in range(nf):
            if f % 2 == 0:
                mag[f, centres - d] = 2.0
                mag[f, centres + d + odd] = 2.0
            else:
                mag[f, centres] = 2.0
        out[c] = _flat(mag, rng)
    return out


def regions(n, ch, nf, seed):
    """Random peak spacings of 3..9 bins: consecutive peaks whose bin sum is odd (round half away from zero) and even."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = np.empty((ch, nf, h, 2), np.float32)
    for c in range(ch):
        mag = np.full((nf, h), 0.05)
        for f in range(nf):
            pk = np.cumsum(rng.integers(3, 10, half // 3)) + 2
            pk = pk[pk <= half - 3]
            mag[f, pk] = rng.uniform(1.0, 2.0, pk.size)
        out[c] = _flat(mag, rng)
    return out


def sequences(n, ch, nf, seed):
    """Frame sequences: silence (classic frames), a single-peak frame (one region covers everything), peaks after a silent
    frame (classic: no previous peaks), channel 0 silent while channel 1 is not (the peak list is shared), and channels with
    different peak sets (links to bins that were not peaks of the channel's own previous frame).  Frame 0 has peaks in every
    channel, so channel 1 of frame 0 is locked against a zero previous phase."""
    rng = np.random.default_rng(seed)
    half, h = n // 2, n // 2 + 1
    out = noise(n, ch, nf, seed + 1)
    pattern = ["noise", "silence", "silence", "noise", "noise", "single", "single", "noise", "ch0_silent", "ch0_silent", "noise",
               "single", "silence", "single"]
    for f in range(1, nf):
        kind = pattern[f % len(pattern)]
        if kind == "silence":
            out[:, f] = 0.0
        elif kind == "single":
            mag = np.full((ch, h), 0.05)
            mag[:, rng.integers(2, half - 2)] = 3.0
            out[:, f] = _flat(mag, rng)
        elif kind == "ch0_silent":
            out[0, f] = 0.0
    return out


GENERATORS = dict(natural=natural, noise=noise, max_density=max_density, ulp_ties=ulp_ties, plateaus=plateaus, tiny=tiny,
                  edges=edges, links=links, regions=regions, sequences=sequences)


def stream(kind, n, ch, nf, seed=0):
    return GENERATORS[kind](n, ch, nf, 1000 * seed + 17 * n + 3 * ch + list(GENERATORS).index(kind))


def phase_inc(n, nf, seed=0):
    """phaseIncrement of each frame: around 1.5 hops, varying as the divergence correction makes it vary."""
    rng = np.random.default_rng(seed + n)
    return (hop_of(n) * 3 // 2 + rng.integers(-3, 4, nf)).astype(np.int32)


def reference(oracle, re_im, n, inc, coremode=1):
    mag, ph = oracle.polar(re_im)
    return mag, ph, oracle.phase_core_frames(mag, ph, inc, hop_of(n), coremode)


# ---- coverage checks -------------------------------------------------------------------------------------------------------
NF = 12


def _ref(oracle, kind, n, ch=1, nf=NF):
    x = stream(kind, n, ch, nf)
    return x, reference(oracle, x, n, phase_inc(n, nf))


def _peaks(r, c, f):
    return r["peaks"][c, f, :r["npeak"][c, f]]


@pytest.mark.parametrize("n", SIZES)
def test_natural_frames_lock(oracle, n):
    _, (_, _, r) = _ref(oracle, "natural", n, 2)
    assert (r["branch"][:, 1:] == 2).all() and r["npeak"].min() > 0


@pytest.mark.parametrize("n", SIZES)
def test_noise_fills_the_third_record_path(oracle, n):
    _, (_, _, r) = _ref(oracle, "noise", n)
    half = n // 2
    assert abs(r["npeak"].mean() / (half / 5) - 1) < 0.1
    if n >= 4096:   # k_lock_chain: a thread's third record (r >= tid + 2 * 128)
        assert r["npeak"].min() > 2 * 128


@pytest.mark.parametrize("n", SIZES)
def test_max_density(oracle, n):
    _, (_, _, r) = _ref(oracle, "max_density", n)
    half = n // 2
    assert (r["npeak"] == (half - 5) // 3 + 1).all()
    pk = _peaks(r, 0, 1)
    e = 8 if n == 8192 else 4   # bins per thread of k_lock_peaks
    per_thread = np.bincount(pk // e)
    assert per_thread.max() == (3 if e == 8 else 2)


@pytest.mark.parametrize("n", SIZES)
def test_ulp_ties_take_both_outcomes(oracle, n):
    x, (mag, _, r) = _ref(oracle, "ulp_ties", n)
    half = n // 2
    cand = np.arange(3, half - 4, 6)
    q = x[..., 0] * x[..., 0] + x[..., 1] * x[..., 1]   # float32, as the kernel squares
    peak_yes = peak_no = 0
    for f in range(NF):
        pk = set(_peaks(r, 0, f).tolist())
        for b in cand:
            qb, qn = q[0, f, b], q[0, f, b + 1]
            assert qb > qn
            unsure = not (qb > np.float32(qn * np.float32(1.00000048)) and qb > 1e-30)
            if unsure:
                is_pk = b in pk
                assert is_pk == (mag[0, f, b] > mag[0, f, b + 1])
                peak_yes += is_pk
                peak_no += not is_pk
    assert peak_yes > 0 and peak_no > 0, (peak_yes, peak_no)


@pytest.mark.parametrize("n", SIZES)
def test_plateaus_are_not_peaks(oracle, n):
    _, (_, _, r) = _ref(oracle, "plateaus", n)
    half = n // 2
    flat = np.concatenate([np.arange(b, b + 2) for b in range(4, half - 8, 16)] + [np.arange(b + 5, b + 8) for b in range(4, half - 8, 16)])
    true = np.arange(15, half - 8, 16)
    for f in range(NF):
        pk = _peaks(r, 0, f)
        assert not np.isin(flat, pk).any()
        assert np.isin(true, pk).all()


@pytest.mark.parametrize("n", SIZES)
def test_tiny_bins_are_subnormal_zero_and_below_the_guard(oracle, n):
    x, (_, _, r) = _ref(oracle, "tiny", n, nf=24)
    q = x[..., 0] * x[..., 0] + x[..., 1] * x[..., 1]
    assert (q < 1e-30).all()
    assert ((q > 0) & (q < np.finfo(np.float32).tiny)).any() and (q == 0).any()
    assert (r["npeak"] > 0).any() and (r["branch"][0, 1:] == 2).any()
    # peaks decided between subnormal squares
    f, c = np.argwhere(r["npeak"][0] > 0)[0][0], 0
    assert (q[c, f, _peaks(r, c, f)] < np.finfo(np.float32).tiny).any()


@pytest.mark.parametrize("n", SIZES)
def test_edge_bins(oracle, n):
    _, (_, _, r) = _ref(oracle, "edges", n)
    half = n // 2
    for f in range(NF):
        pk = _peaks(r, 0, f)
        if f % 2 == 0:
            assert pk[0] == 2 and pk[-1] == half - 3
        else:
            assert pk[0] > 2 and pk[-1] < half - 3 and len(pk) > 0


@pytest.mark.parametrize("n", SIZES)
def test_links_half_way(oracle, n):
    _, (_, _, r) = _ref(oracle, "links", n)
    half = n // 2
    centres = np.arange(10, half - 10, 16)
    d = 2 + (np.arange(centres.size) % 5)
    odd = (np.arange(centres.size) // 5) % 2
    for f in range(1, NF):
        assert r["branch"][0, f] == 2
        pk = _peaks(r, 0, f)
        if f % 2:
            assert np.array_equal(pk, centres)
        else:
            assert np.array_equal(pk, np.sort(np.concatenate([centres - d, centres + d + odd])))
    assert (odd == 0).any() and (odd == 1).any()   # exact ties and near ties


@pytest.mark.parametrize("n", SIZES)
def test_region_starts_of_both_parities(oracle, n):
    _, (_, _, r) = _ref(oracle, "regions", n)
    odd = even = 0
    for f in range(1, NF):
        assert r["branch"][0, f] == 2
        pk = _peaks(r, 0, f)
        s = pk[:-1] + pk[1:]
        odd += (s % 2 == 1).sum()
        even += (s % 2 == 0).sum()
        assert np.array_equal(r["bin1"][0, f, 1:len(pk)], (s + 1) // 2)   # round((a + b) * 0.5), half away from zero
    assert odd > 0 and even > 0


@pytest.mark.parametrize("n", SIZES)
def test_sequences(oracle, n):
    ch, nf = 2, 28
    x, (_, _, r) = _ref(oracle, "sequences", n, ch, nf)
    half = n // 2
    br, npk = r["branch"], r["npeak"]
    assert br[0, 0] == 0 and br[1, 0] == 2                                  # channel 1 of frame 0: locked, prev_phase 0
    assert ((br == 1) & (npk == 0)).any()                                     # silence: classic
    assert ((br == 1) & (npk > 0)).any()                                      # peaks after silence: classic (nprev == 0)
    single = np.argwhere((br == 2) & (npk == 1))
    assert len(single) > 0
    for c, f in single:
        assert r["bin1"][c, f, 0] == 0 and r["bin2"][c, f, 0] == half
    ch0_silent = [f for f in range(nf) if not x[0, f].any() and x[1, f].any()]
    assert ch0_silent and all(br[1, f] == 1 and npk[1, f] > 0 for f in ch0_silent)   # shared peak list: channel 0 had none
    # links to a bin that was not a peak of the channel's own previous frame (the other channel's peaks are the previous list)
    miss = 0
    for f in range(1, nf):
        for c in range(ch):
            if br[c, f] != 2:
                continue
            prev_list = _peaks(r, ch - 1, f - 1) if c == 0 else _peaks(r, c - 1, f)
            own_prev = set(_peaks(r, c, f - 1).tolist())
            miss += sum(p not in own_prev for p in prev_list)
    assert miss > 0
