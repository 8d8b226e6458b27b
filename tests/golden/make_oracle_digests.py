"""Generate tests/golden/oracle_live_sha256.json: SHA-256 digests of the oracle's output on the inputs of the live-reference
cases of tests/test_oracle_vs_ref.py, which check against them where oracle/_ref is absent.

The digests are the oracle's output.  Where oracle/_ref is present, each output is first checked to be bit-identical to the
reference's, so regenerating there stores the reference's output.  The committed file was written without oracle/_ref: it pins
the oracle against drift on these inputs, and the oracle's tie to the reference rests on the stored reference outputs
(tests/golden/pv_golden.npz).   python tests/golden/make_oracle_digests.py
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import pv_oracle as O  # noqa: E402
import test_oracle_vs_ref as T  # noqa: E402


def output(x, sr, kw):
    y = O.run_offline(x, sr, **kw)
    if O.have_ref():
        r = O.run_ref(x, sr, **kw)
        assert y.shape == r.shape and np.array_equal(y.view(np.uint32), r.view(np.uint32)), "the oracle differs from the reference"
    return T.digest(y)


def main():
    print("checking against oracle/_ref" if O.have_ref() else "oracle/_ref is absent: digests of the oracle alone")
    out = {c[0]: output(T.live_input(c), c[2], c[1]) for c in T.LIVE_CASES}
    for i, (kw, sr, ch) in enumerate(T.SILENCE_CASES):
        out[f"silence{i}"] = output(T.silence_input(sr, ch), sr, kw)
    with open(os.path.join(HERE, "oracle_live_sha256.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
