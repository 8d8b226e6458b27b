"""The reference's own, unmodified CLI linked against libpvgpu.so (oracle/_ref/audiomod-exe-gpu, built by
`make -C oracle gpu-exe`) next to the reference's CPU CLI on the same 16-bit WAV files."""
import os
import subprocess
import wave

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "audiomod-exe")
GPU = os.path.join(ROOT, "oracle", "_ref", "audiomod-exe-gpu")


def _write_wav(path, pcm, sr):
    with wave.open(path, "wb") as w:
        w.setnchannels(pcm.shape[0])
        w.setsampwidth(2)
        w.setframerate(sr)
        w.writeframes(np.ascontiguousarray(pcm.T).tobytes())


def _read_wav(path):
    with wave.open(path, "rb") as w:
        a = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16)
        return a.reshape(-1, w.getnchannels()).T


@pytest.mark.parametrize("args,ch", [(["normal_pitchshift", "4", "1", "2048"], 2), (["time_stretch", "1.5", "1", "4096"], 2),
                                     (["formant_pitchshift", "4", "1", "2048"], 1), (["robotic"], 2)])
def test_reference_cli_on_gpu_library(tmp_path, args, ch):
    if not (os.path.exists(REF) and os.path.exists(GPU)):
        pytest.skip("oracle/_ref/audiomod-exe or audiomod-exe-gpu is absent: make -C oracle ref REF=<reference sources> builds them")
    from audiomod_b200.synth import synth_int16
    sr = 48000 if args[0] == "time_stretch" else 44100
    pcm = synth_int16(1001, sr, 1.5, ch)
    src = str(tmp_path / "in.wav")
    _write_wav(src, pcm, sr)
    outs = []
    for exe, tag in ((REF, "cpu"), (GPU, "gpu")):
        dst = str(tmp_path / f"out_{tag}.wav")
        r = subprocess.run([exe, args[0], src, dst] + args[1:], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and os.path.exists(dst), r.stdout[-500:] + r.stderr[-500:]
        outs.append(_read_wav(dst))
    a, b = outs
    assert a.shape == b.shape
    diff = np.abs(a.astype(np.int32) - b.astype(np.int32))
    assert diff.max() <= 1, f"max diff {diff.max()} LSB"          # float error 1e-7 can flip the int16 truncation by 1 LSB
    assert (diff == 0).mean() > 0.995
