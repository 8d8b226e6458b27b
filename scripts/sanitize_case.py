"""Small cases for compute-sanitizer (one tool per run):
    compute-sanitizer --tool memcheck  python scripts/sanitize_case.py
    compute-sanitizer --tool racecheck python scripts/sanitize_case.py
cfg1 (stereo +4 st) and cfg4 (mono +7 st) batches through the split kernels and the fused kernel, a formant case, a robotic
case (no resampler: the fused kernel stores straight from the accumulator) and one streaming instance.  Prints one line per case; the sanitizer's own summary follows."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import audiomod_b200 as A
from audiomod_b200.synth import synth

secs = float(sys.argv[1]) if len(sys.argv) > 1 else 0.25
ref = {}
for name, ch, st, mode, fft in (("cfg1", 2, 4.0, 0, 2048), ("cfg4", 1, 7.0, 0, 2048), ("formant", 1, 4.0, 2, 2048), ("robotic", 2, 0.0, 6, 1024)):
    xs = [synth(100 + i, 44100, secs * (1.0 - 0.3 * i), ch) for i in range(3)]
    for variant, fused in (("split", False), ("fused", True)):
        b = A.PhaseVocoderBatch(len(xs), xs[0].shape[1], 44100, ch, 1.0, st, mode, 1, fft)
        b.set_fused(fused)
        b.tune(frames_per_chunk=16)
        ys = b.run(xs)
        b.close()
        if variant == "split":
            ref[name] = ys
        same = all(np.array_equal(a, c) for a, c in zip(ys, ref[name]))
        print(f"{name} {variant}: {len(ys)} streams, bit-identical to split: {same}", flush=True)
x = synth(7, 44100, secs, 2)
pv = A.phasevocoder(44100, 2, 1.0, 4.0, 0, 1, 2048)
n = 0
for i in range(0, x.shape[1], 480):
    pv.processInData(x[:, i:i + 480])
    n += pv.getOutData(pv.getOutSamples()).shape[1]
pv.close()
print("streaming instance:", n, "samples", flush=True)
