"""File -> file batch front end (pvgpu_run_wav_files) against the reference's own CLI on the same WAV files.

64 files in one call -- 8/16/24/32-bit PCM, mono and stereo, two sample rates, ragged lengths, one with an extra chunk
before the data -- each compared with what `oracle/_ref/audiomod-exe normal_pitchshift in.wav out.wav 4 1 2048` (the
unmodified reference CLI: main/main.cc + main/wavfile.cc) writes: identical header, identical sample count, samples within
1 LSB of the 16-bit output and >= 99.5 % of them identical (a 1e-7 float difference can flip the writer's truncation).

That CLI is built from the reference's sources, which the repository does not carry.  Without it the same bars hold against
reference_cli_file(): the CLI restated, its library by the oracle (pinned bit-exactly to the reference by
test_oracle_vs_ref.py) and its WAV reader and writer by the rules of main/wavfile.cc.
"""
import os
import struct
import subprocess
import wave

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref", "audiomod-exe")


def _write(path, pcm16, sr, bits, extra_chunk=False):
    """pcm16: int16 [ch, n]; written at `bits` per sample (the 16-bit value scaled into the wider / narrower format)."""
    ch, n = pcm16.shape
    x = pcm16.astype(np.int64)
    if bits == 8:
        raw = ((x >> 8) + 128).astype(np.uint8).T.tobytes()
    elif bits == 16:
        raw = pcm16.T.astype("<i2").tobytes()
    elif bits == 24:
        v = (x << 8).T.reshape(-1)
        raw = b"".join(int(s).to_bytes(3, "little", signed=True) for s in v)
    else:
        raw = (x << 16).T.astype("<i4").tobytes()
    fmt = struct.pack("<4sIHHIIHH", b"fmt ", 16, 1, ch, sr, sr * ch * bits // 8, ch * bits // 8, bits)
    extra = struct.pack("<4sI", b"LIST", 12) + b"INFOISFT" + struct.pack("<I", 0) if extra_chunk else b""
    data = struct.pack("<4sI", b"data", len(raw)) + raw
    body = b"WAVE" + fmt + extra + data
    with open(path, "wb") as f:
        f.write(struct.pack("<4sI", b"RIFF", len(body)) + body)


def _read16(path):
    with wave.open(path, "rb") as w:
        a = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2")
        return a.reshape(-1, w.getnchannels()).T, w.getframerate()


def reference_cli_file(oracle, pcm16, sr, bits):
    """The bytes `audiomod-exe normal_pitchshift in.wav out.wav 4 1 2048` writes for the file _write(pcm16, sr, bits) makes:
    samples decoded as value / 2^(bits-1), 8 bit as u8 / 128 - 1, in double (wavfile.cc:672-812); the library run with the
    CLI's block protocol (oracle.run_offline); 16-bit output (main.cc:136) saturated and truncated toward zero,
    (short)(int)clamp(y * 32768.f) (wavfile.cc:1294-1306, 1508-1526), behind a RIFF + fmt(16) + fact(4) + data header
    (wavfile.cc:1135-1182)."""
    ch = pcm16.shape[0]
    if bits == 8:
        x = ((pcm16.astype(np.int64) >> 8) + 128) * (1.0 / 128.0) - 1.0
    else:                       # 16, 24 and 32 bit hold the 16-bit value shifted up: value / 2^(bits-1) == pcm16 / 32768
        x = pcm16 * (1.0 / 32768.0)
    y = oracle.run_offline(x.astype(np.float32), sr, semitones=4.0, mode=0, coremode=1, fftsize=2048)
    q = np.clip(y * np.float32(32768.0), np.float32(-32768.0), np.float32(32767.0)).astype(np.int32).astype("<i2")
    data = np.ascontiguousarray(q.T).tobytes()
    frames = q.shape[1]
    header = struct.pack("<4sI4s4sIHHIIHH4sII4sI", b"RIFF", len(data) + 48, b"WAVE", b"fmt ", 16, 1, ch, sr, 2 * ch * sr, 2 * ch,
                         16, b"fact", 4, frames, b"data", len(data))
    return header + data


def test_wav_batch_matches_reference_cli(tmp_path, pvlib, oracle):
    if pvlib.pvgpu_device_count() < 1:
        pytest.fail("no CUDA device: GPU tests must run on the B200 box")
    import audiomod_b200 as A
    from audiomod_b200.synth import synth_int16
    pairs, meta, pcms = [], [], []
    for i in range(64):
        ch = 1 + (i % 2)
        sr = 48000 if i % 8 == 5 else 44100
        bits = (16, 16, 16, 24, 16, 16, 8, 32)[i % 8]
        secs = 0.25 + 0.05 * (i % 9)
        pcm = synth_int16(3000 + i, sr, secs, ch)
        src, dst = str(tmp_path / f"in{i}.wav"), str(tmp_path / f"gpu{i}.wav")
        _write(src, pcm, sr, bits, extra_chunk=(i == 7))
        pairs.append((src, dst))
        meta.append((ch, sr, bits, pcm.shape[1]))
        pcms.append(pcm)
    res = A.run_wav_files(pairs, 1.0, 4.0, A.NORMAL_SHIFT, A.PHASE_LOCKED, 2048)
    for i, (r, (ch, sr, bits, n)) in enumerate(zip(res, meta)):
        assert r["status"] == 0, (i, r["message"])
        assert (r["channels"], r["sample_rate"], r["bits"], r["frames_in"], r["frames_out"]) == (ch, sr, bits, n, n)
    worst, exact, total = 0, 0, 0
    for i, (src, dst) in enumerate(pairs):
        ref = str(tmp_path / f"ref{i}.wav")
        if os.path.exists(REF):
            p = subprocess.run([REF, "normal_pitchshift", src, ref, "4", "1", "2048"], capture_output=True, text=True, timeout=120)
            assert p.returncode == 0 and os.path.exists(ref), p.stderr[-400:]
        else:
            ch, sr, bits, _ = meta[i]
            with open(ref, "wb") as f:
                f.write(reference_cli_file(oracle, pcms[i], sr, bits))
        a, b = open(dst, "rb").read(), open(ref, "rb").read()
        assert len(a) == len(b), f"file {i}: {len(a)} bytes vs the reference CLI's {len(b)}"
        assert a[:56] == b[:56], f"file {i}: header differs"
        ya, _ = _read16(dst)
        yb, _ = _read16(ref)
        d = np.abs(ya.astype(np.int32) - yb.astype(np.int32))
        worst = max(worst, int(d.max()))
        exact += int((d == 0).sum())
        total += d.size
    assert worst <= 1, f"{worst} LSB"
    assert exact / total >= 0.995


def test_wav_batch_reports_bad_files(tmp_path, pvlib):
    import audiomod_b200 as A
    from audiomod_b200.synth import synth_int16
    good, bad, missing = str(tmp_path / "good.wav"), str(tmp_path / "bad.wav"), str(tmp_path / "missing.wav")
    _write(good, synth_int16(1, 44100, 0.2, 1), 44100, 16)
    open(bad, "wb").write(b"RIFF\x10\x00\x00\x00WAVXjunkjunkjunk")
    res = A.run_wav_files([(good, str(tmp_path / "o1.wav")), (bad, str(tmp_path / "o2.wav")), (missing, str(tmp_path / "o3.wav"))], 1.0, 7.0)
    assert res[0]["status"] == 0 and os.path.exists(tmp_path / "o1.wav")
    assert res[1]["status"] != 0 and "RIFF" in res[1]["message"]
    assert res[2]["status"] != 0 and not os.path.exists(tmp_path / "o3.wav")
