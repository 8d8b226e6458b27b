"""Post-chain of FFT-free effects on the batch's output rows (pvgpu_batch_set_postchain; audiomod_b200/csrc/pv_post.cu) against
the unmodified reference's gain / compressor / limiter objects (oracle/_ref/fxref_drv) applied to the unmodified reference's
phase-vocoder output -- the chain an SDK user builds from those objects (README.md:78-94).

Those reference binaries are built from the reference's sources, which the repository does not carry, and the repository has no
restatement of the effect objects.  Without them the outputs are held to the same bars against
tests/golden/postchain_outputs.npz: this project's own outputs, not the reference's, stored as each stream's length and its
samples at cases.golden_cols (tests/golden/make_gpu_golden.py, which checks them against the reference objects first wherever
they are present).  They keep the output from drifting beyond these bars on a checkout without the reference."""
import os

import numpy as np
import pytest

from cases import make_input
from test_gpu_parity import assert_parity, assert_parity_golden

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "postchain_outputs.npz")

CHAINS = [
    [("gain", 1.7)],
    [("compressor", -10.0, 6.0, 6.0, 10.0, 100.0)],
    [("limiter", -10.0, 6.0, 0.0, 100.0)],
    [("gain", 0.6), ("compressor", -20.0, 4.0, 3.0, 5.0, 50.0), ("limiter", -6.0, 2.0, 1.0, 80.0)],
    [("limiter", -3.0, 0.0, 0.5, 20.0), ("limiter", -12.0, 9.0, 0.0, 200.0)],
]
CHAIN_IDS = ["gain", "compressor", "limiter", "all-three", "two-limiters"]
CHAIN_SHAPES = [(1, 7.0, 64), (2, -3.0, 8)]     # channels, semitones, frames per chunk
TS_CHAIN = [("compressor", -15.0, 3.0, 4.0, 10.0, 100.0), ("limiter", -8.0, 3.0, 0.0, 100.0)]


@pytest.fixture(scope="module")
def A(pvlib):
    import audiomod_b200
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    return audiomod_b200


def _checker(oracle, key, reference):
    """check(y, i, what): the i-th output against `reference(i)` (the reference objects) where they were built, else against
    the stored output key__i."""
    if oracle.have_ref() and oracle.have_ref_fx():
        return lambda y, i, what: assert_parity(y, reference(i), what)
    gold = np.load(GOLD)
    return lambda y, i, what: assert_parity_golden(y, gold, f"{key}__{i}", what)


def chain_inputs(sr, ch):
    return [make_input("x", sr, ch, 0.9 - 0.25 * i, 2700 + i) for i in range(3)]


def ts_inputs(sr):
    return [make_input("x", sr, 1, 0.6, 2800 + i) for i in range(5)]


def eq_inputs(sr, ch):
    return [make_input("x", sr, ch, 0.8 - 0.3 * i, 3100 + i) for i in range(2)]


@pytest.mark.parametrize("chain", CHAINS, ids=CHAIN_IDS)
@pytest.mark.parametrize("ch,st,fpc", CHAIN_SHAPES)
def test_postchain_matches_reference_objects(A, oracle, chain, ch, st, fpc):
    sr = 44100
    xs = chain_inputs(sr, ch)
    check = _checker(oracle, f"{CHAIN_IDS[CHAINS.index(chain)]}_{ch}ch_{st:+g}st_fpc{fpc}",
                     lambda i: oracle.run_ref_fx(oracle.run_ref(xs[i], sr, semitones=st), sr, chain))
    outs = {}
    for fused in (False, True):
        b = A.PhaseVocoderBatch(len(xs), xs[0].shape[1], sr, ch, 1.0, st)
        b.set_fused(fused)
        b.tune(frames_per_chunk=fpc)          # the effect state crosses chunk boundaries
        b.set_postchain(chain)
        ys = b.run(xs)
        b.close()
        for i, y in enumerate(ys):
            check(y, i, f"{[c[0] for c in chain]} fused={fused} [{i}]")
        outs[fused] = ys
    for a, c in zip(outs[False], outs[True]):
        assert np.array_equal(a, c)


def test_postchain_time_sliced_host_rows_and_clear(A, oracle):
    """Equal-length streams in one 2-D host array take the time-sliced pipeline: the chain runs on every chunk's columns before
    their D2H copy.  Clearing the chain gives the plain output again."""
    sr, S = 44100, 5
    xs = ts_inputs(sr)
    X = np.ascontiguousarray(np.concatenate(xs, axis=0))
    chain = TS_CHAIN
    check = _checker(oracle, "time_sliced", lambda i: oracle.run_ref_fx(oracle.run_ref(xs[i], sr, semitones=7.0), sr, chain))
    b = A.PhaseVocoderBatch(S, X.shape[1], sr, 1, 1.0, 7.0)
    b.tune(frames_per_chunk=16)
    n_out = int(b.plan(X.shape[1])[0])
    Y = np.zeros((S, n_out), np.float32)
    b.set_postchain(chain)
    b.run_host_rows([X[r] for r in range(S)], [Y[r] for r in range(S)])
    for i in range(S):
        check(Y[i:i + 1], i, f"ts[{i}]")
    b.set_postchain([])
    b.run_host_rows([X[r] for r in range(S)], [Y[r] for r in range(S)])
    # without a chain the output is the phase vocoder's alone, which the oracle restates bit-exactly (test_oracle_vs_ref.py)
    plain = oracle.run_ref(xs[2], sr, semitones=7.0) if oracle.have_ref() else oracle.run_offline(xs[2], sr, semitones=7.0)
    assert_parity(Y[2:3], plain, "cleared")
    from audiomod_b200 import _lib
    q = np.zeros((S, n_out), np.int16)
    b.set_postchain(chain)
    with pytest.raises(A.PvgpuError) as e:
        b.run_host_rows([X[r].astype(np.int16) for r in range(S)], [q[r] for r in range(S)], A.S16)
    assert e.value.code == _lib.EINVAL
    b.close()


EQ_PARAMS = [1, 120, 0.7, 1.0,  1, 300, 0.5, -3.0,  1, 900, 1.2, 4.0,  0, 2000, 0.3, 1.5,
             1, 3100, 2.0, -5.0,  1, 4500, 0.9, 2.5,  1, 7000, 0.6, 3.0,  1, 12000, 0.8, 1.0]
EQ_SPECS = ["default", "all-bands", "sections"]


def eq_chains(A, spec):
    """(the post-chain, the same chain as the reference objects' driver spells it) of one equalizer case."""
    if spec == "default":
        return A.equalizer_chain(), [("equalizer",)]
    if spec == "all-bands":
        return A.equalizer_chain(EQ_PARAMS), [tuple(["equalizer"] + EQ_PARAMS)]
    chain = [("biquad", t, 500.0 + 400.0 * t, 0.8, 3.0) for t in (3, 6, 7, 8)] + [("gain", 0.9)]
    return chain, chain


@pytest.mark.parametrize("spec", EQ_SPECS)
def test_equalizer_and_biquads_match_reference_objects(A, oracle, spec):
    """The 8-band equalizer object (src/equalizer/equalizer.cc) and single biquad sections of every type
    (src/common/filters/biquadfilter.cc), expanded into the post-chain, against the reference's own objects."""
    sr, ch = 44100, 2
    chain, ref_chain = eq_chains(A, spec)
    if spec == "default":
        assert [c[1] for c in chain] == [0]                       # only the 200 Hz high-pass is on by default
    elif spec == "all-bands":
        assert [c[1] for c in chain] == [0, 1, 2, 2, 2, 4, 5]
    xs = eq_inputs(sr, ch)
    check = _checker(oracle, f"eq_{spec}", lambda i: oracle.run_ref_fx(oracle.run_ref(xs[i], sr, semitones=4.0), sr, ref_chain))
    b = A.PhaseVocoderBatch(len(xs), xs[0].shape[1], sr, ch, 1.0, 4.0)
    b.tune(frames_per_chunk=16)
    b.set_postchain(chain)
    ys = b.run(xs)
    b.close()
    for i, y in enumerate(ys):
        check(y, i, f"{spec}[{i}]")
