"""Parity cases shared by the golden generator, the oracle tests and the GPU tests.

Each case: name, constructor keywords (the reference's arguments), sample rate, channels, seconds, seed.
They cover BASELINE.json's five configurations (shortened so the CPU oracle finishes in well under a second each) plus
the edge cases the survey calls out (L == R stereo, coremodes 0 and 2, constant mode, octave shift = direct resampler
table, down-shift, FFT sizes 512..8192).
"""
CASES = [
    ("cfg1_shift_p4_stereo", dict(semitones=4.0, mode=0, coremode=1, fftsize=2048), 44100, 2, 0.6, 1001),
    ("cfg2_stretch_1p5_4096", dict(timeratio=1.5, mode=5, coremode=1, fftsize=4096), 48000, 2, 0.6, 1002),
    ("cfg3_formant_p4", dict(semitones=4.0, mode=2, fftsize=2048), 44100, 1, 0.5, 1003),
    ("cfg3_formant_m4", dict(semitones=-4.0, mode=2, fftsize=2048), 44100, 1, 0.5, 1003),
    ("cfg3_gender_p4", dict(semitones=4.0, mode=1, fftsize=2048), 44100, 1, 0.5, 1004),
    ("cfg3_gender_m4", dict(semitones=-4.0, mode=1, fftsize=2048), 44100, 1, 0.5, 1004),
    ("cfg3_gender_0", dict(semitones=0.0, mode=1, fftsize=2048), 44100, 1, 0.5, 1004),
    ("cfg4_shift_p7_mono", dict(semitones=7.0, mode=0, coremode=1, fftsize=2048), 44100, 1, 0.6, 4000),
    ("cfg5_robotic_512", dict(mode=6, fftsize=512), 44100, 2, 0.3, 5000),
    ("cfg5_robotic_8192", dict(mode=6, fftsize=8192), 44100, 2, 0.6, 5000),
    ("cfg5_whisper_1024", dict(mode=7, fftsize=1024), 44100, 2, 0.3, 5001),
    ("cfg5_whisper_4096", dict(mode=7, fftsize=4096), 44100, 2, 0.4, 5001),
    ("cfg5_vocoder_2048", dict(mode=3, fftsize=2048), 44100, 2, 0.4, 5002),
    ("cfg5_vocoder_512", dict(mode=3, fftsize=512), 44100, 2, 0.3, 5002),
    ("cfg5_chord_4096", dict(mode=4, fftsize=4096), 44100, 2, 0.4, 5003),
    ("cfg5_chord_8192", dict(mode=4, fftsize=8192), 44100, 2, 0.6, 5003),
    ("core0_shift_p3_stereo", dict(semitones=3.0, mode=0, coremode=0, fftsize=2048), 44100, 2, 0.5, 5004),
    ("core2_octave_up", dict(semitones=12.0, mode=0, coremode=2, fftsize=2048), 44100, 1, 0.5, 5005),
    ("shift_m5_1024", dict(semitones=-5.0, mode=0, coremode=1, fftsize=1024), 22050, 1, 0.5, 5006),
    ("stretch_0p7_1024", dict(timeratio=0.7, mode=5, coremode=1, fftsize=1024), 44100, 1, 0.5, 5007),
    ("stretch_2p0_intratio", dict(timeratio=2.0, mode=5, coremode=1, fftsize=1024), 44100, 2, 0.4, 5008),
    ("constant_1024", dict(mode=-1, fftsize=1024), 44100, 1, 0.3, 5009),
    ("stereo_identical_lr", dict(semitones=4.0, mode=0, coremode=1, fftsize=2048), 44100, 2, 0.5, 5010),
]


def make_input(name, sr, ch, secs, seed):
    from audiomod_b200.synth import synth
    x = synth(seed, sr, secs, ch)
    if name == "stereo_identical_lr":
        x[1] = x[0]
    return x


GOLDEN_EDGE, GOLDEN_INNER = 128, 512


def golden_cols(n):
    """The fixed sample positions (of an output n samples long) at which tests/golden/make_gpu_golden.py stores outputs: the
    first and last GOLDEN_EDGE samples (start-up and flush) and GOLDEN_INNER seeded positions in between.  Whole outputs
    would make the stored vectors too large to keep in the repository."""
    import numpy as np
    edge = min(GOLDEN_EDGE, n)
    inner = np.arange(edge, max(edge, n - edge))
    pick = np.random.default_rng(n).choice(inner, min(inner.size, GOLDEN_INNER), replace=False)
    return np.unique(np.concatenate([np.arange(edge), np.arange(max(0, n - edge), n), pick]))


def ctor_args(kw):
    """(timeratio, semitones, mode, coremode, fftsize) in the reference constructor's order."""
    return (kw.get("timeratio", 1.0), kw.get("semitones", 0.0), kw.get("mode", 0), kw.get("coremode", 1), kw.get("fftsize", 2048))
