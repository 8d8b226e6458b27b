"""The oracle (oracle/pv_oracle.c) is pinned bit-exactly against golden vectors taken from the unmodified reference
(tests/golden/make_golden.py) and, where oracle/_ref has been built, against the reference itself run live.

oracle/_ref is built from the reference's sources, which the repository does not carry.  Without it the live cases compare the
oracle's output with the SHA-256 digests in tests/golden/oracle_live_sha256.json (tests/golden/make_oracle_digests.py): the
oracle's own output, bit for bit, when the digests were taken.  They keep the oracle from drifting on these inputs; its tie to
the reference rests on the stored reference outputs of the golden tests above."""
import hashlib
import json
import os

import numpy as np
import pytest

from cases import CASES, make_input

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "pv_golden.npz")
DIGESTS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_live_sha256.json")
LIVE_CASES = CASES[::4]
SILENCE_CASES = [
    (dict(semitones=7.0, mode=0, coremode=1, fftsize=2048), 44100, 1),
    (dict(semitones=4.0, mode=0, coremode=1, fftsize=2048), 44100, 2),
    (dict(timeratio=1.5, mode=5, coremode=0, fftsize=1024), 48000, 2),
]


def live_input(case):
    name, kw, sr, ch, secs, seed = case
    return make_input(name, sr, ch, secs * 1.7, seed + 77)


def silence_input(sr, ch):
    x = make_input("x", sr, ch, 0.8, 321)
    x[:, :int(0.1 * sr)] = 0.0
    x[:, int(0.3 * sr):int(0.45 * sr)] = 0.0
    x[ch - 1, int(0.55 * sr):int(0.65 * sr)] = 0.0
    return x


def digest(y):
    return {"shape": list(y.shape), "sha256": hashlib.sha256(np.ascontiguousarray(y, np.float32).tobytes()).hexdigest()}


def assert_matches_live_reference(oracle, key, x, sr, kw):
    a = oracle.run_offline(x, sr, **kw)
    if oracle.have_ref():
        b = oracle.run_ref(x, sr, **kw)
        assert a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))
    else:
        with open(DIGESTS) as f:
            assert digest(a) == json.load(f)[key], "oracle output differs from the stored digest"


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_matches_reference_golden(oracle, gold, case):
    name, kw, sr, ch, secs, seed = case
    pcm = gold[name + "__in"]
    x = (pcm.astype(np.float64) * (1.0 / 32768.0)).astype(np.float32)
    assert np.array_equal(x, make_input(name, sr, ch, secs, seed)), "synthetic input generator drifted from the fixture"
    y = oracle.run_offline(x, sr, **kw)
    ref = gold[name + "__out"]
    assert y.shape == ref.shape
    assert np.array_equal(y.view(np.uint32), ref.view(np.uint32)), "oracle is not bit-exact with the reference"


@pytest.mark.parametrize("name", ["cfg4_shift_p7_mono", "cfg5_robotic_512"])
def test_oracle_realtime_protocol_golden(oracle, gold, name):
    """processBlock / outputReady loop (main.cc:562-571): blocks are kept only when outputReady()."""
    kw, sr, ch, secs, seed = next((c[1], c[2], c[3], c[4], c[5]) for c in CASES if c[0] == name)
    x = make_input(name, sr, ch, secs, seed)
    st = oracle.OracleStream(sr, ch, kw.get("timeratio", 1.0), kw.get("semitones", 0.0), kw.get("mode", 0), kw.get("coremode", 1),
                             kw.get("fftsize", 2048))
    B = max(480, sr // 100)
    kept = []
    for i in range(0, x.shape[1], B):
        blk = np.ascontiguousarray(x[:, i:i + B])
        if st.processBlock(blk):
            kept.append(blk)
    y = np.concatenate(kept, axis=1) if kept else np.zeros((ch, 0), np.float32)
    ref = gold[name + "__rt"]
    assert y.shape == ref.shape and np.array_equal(y.view(np.uint32), ref.view(np.uint32))


@pytest.mark.parametrize("case", LIVE_CASES, ids=[c[0] for c in LIVE_CASES])
def test_oracle_matches_live_reference(oracle, case):
    assert_matches_live_reference(oracle, case[0], live_input(case), case[2], case[1])


@pytest.mark.parametrize("kw,sr,ch", SILENCE_CASES)
def test_oracle_silence_matches_live_reference(oracle, kw, sr, ch):
    """Frames without spectral peaks (digital silence) take the classic-propagation branch of the phase-locked core
    (phasevocoderprocess.cc:617-636); pin the oracle's restatement of it against the reference itself."""
    assert_matches_live_reference(oracle, f"silence{SILENCE_CASES.index((kw, sr, ch))}", silence_input(sr, ch), sr, kw)


def test_block_size_independence(oracle):
    """Output does not depend on the block size as long as the ring never overflows (SURVEY 8c)."""
    from audiomod_b200.synth import synth
    x = synth(9, 44100, 0.5, 1)
    a = oracle.run_offline(x, 44100, semitones=7.0, block=480)
    b = oracle.run_offline(x, 44100, semitones=7.0, block=4410)
    assert np.array_equal(a, b)
