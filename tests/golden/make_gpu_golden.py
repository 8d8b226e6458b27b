"""Generate tests/golden/{cepstral,postchain}_outputs.npz: the outputs that test_gpu_cepstral.py and test_gpu_postchain.py
check against when the reference binaries they compare with (oracle/_ref/pvref_drv_cep, fxref_drv: built from the reference's
sources, which the repository does not carry) are absent.  The repository has no restatement of the reference's cepstral
routine or effect objects, so these are this project's own outputs, from the path a batch takes by default: they are not the
reference's.  They hold later changes to the bars of those tests around the output they were taken from.  Where the reference
binaries are present, every output is first held to those bars against the reference and nothing is stored if one fails.
Needs a CUDA device:  python tests/golden/make_gpu_golden.py [out_dir]

Each output is stored as its length (key__n) and its samples at cases.golden_cols (key).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import audiomod_b200 as A  # noqa: E402
from cases import golden_cols  # noqa: E402
import test_gpu_cepstral as TC  # noqa: E402
import test_gpu_postchain as TP  # noqa: E402
from oracle import pv_oracle as O  # noqa: E402
from test_gpu_parity import assert_parity  # noqa: E402


def put(data, key, y, reference=None):
    """Store y under key; reference(): the reference binaries' output for it, checked where they are present."""
    if reference is not None:
        assert_parity(y, reference(), key)
    n = y.shape[1]
    data[key + "__n"] = np.int64(n)
    data[key] = np.ascontiguousarray(y[:, golden_cols(n)])


def batch(xs, sr, ch, st, chain=None, fpc=0, mode=0, fft=2048):
    b = A.PhaseVocoderBatch(len(xs), xs[0].shape[1], sr, ch, 1.0, st, mode, 1, fft)
    if fpc:
        b.tune(frames_per_chunk=fpc)
    if chain:
        b.set_postchain(chain)
    ys = b.run(xs)
    b.close()
    return ys


def cepstral():
    data = {}
    for mode, st, ch, fft, sr in TC.CEPSTRAL_CASES:
        xs = TC.cepstral_inputs(ch, sr)
        for i, y in enumerate(batch(xs, sr, ch, st, mode=mode, fft=fft)):
            ref = None
            if O.have_ref_cepstral():
                ref = lambda x=xs[i]: O.run_ref(x, sr, semitones=st, mode=mode - 7, fftsize=fft, cepstral=True)  # noqa: E731
            put(data, f"{TC.cepstral_key(mode, st, ch, fft, sr)}__{i}", y, ref)
    return data


def fx_reference(x, sr, st, chain):
    if not (O.have_ref() and O.have_ref_fx()):
        return None
    return lambda: O.run_ref_fx(O.run_ref(x, sr, semitones=st), sr, chain)


def postchain():
    data, sr = {}, 44100
    for chain, cid in zip(TP.CHAINS, TP.CHAIN_IDS):
        for ch, st, fpc in TP.CHAIN_SHAPES:
            xs = TP.chain_inputs(sr, ch)
            for i, y in enumerate(batch(xs, sr, ch, st, chain, fpc)):
                put(data, f"{cid}_{ch}ch_{st:+g}st_fpc{fpc}__{i}", y, fx_reference(xs[i], sr, st, chain))
    xs = TP.ts_inputs(sr)
    X = np.ascontiguousarray(np.concatenate(xs, axis=0))
    b = A.PhaseVocoderBatch(len(xs), X.shape[1], sr, 1, 1.0, 7.0)
    b.tune(frames_per_chunk=16)
    Y = np.zeros((len(xs), int(b.plan(X.shape[1])[0])), np.float32)
    b.set_postchain(TP.TS_CHAIN)
    b.run_host_rows([X[r] for r in range(len(xs))], [Y[r] for r in range(len(xs))])
    b.close()
    for i in range(len(xs)):
        put(data, f"time_sliced__{i}", Y[i:i + 1], fx_reference(xs[i], sr, 7.0, TP.TS_CHAIN))
    for spec in TP.EQ_SPECS:
        chain, ref_chain = TP.eq_chains(A, spec)
        xs = TP.eq_inputs(sr, 2)
        for i, y in enumerate(batch(xs, sr, 2, 4.0, chain, 16)):
            put(data, f"eq_{spec}__{i}", y, fx_reference(xs[i], sr, 4.0, ref_chain))
    return data


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else HERE
    os.makedirs(out, exist_ok=True)
    print("checking against oracle/_ref" if O.have_ref() else "oracle/_ref is absent: storing this project's outputs unchecked")
    for name, make in (("cepstral", cepstral), ("postchain", postchain)):
        path = os.path.join(out, f"{name}_outputs.npz")
        np.savez_compressed(path, **make())
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
