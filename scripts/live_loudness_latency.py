"""Live batch per-call latency with the loudness meters (pvgpu_set_meters), cfg4: mono 44.1 kHz, +7 semitones, FFT 2048,
480-sample blocks, S = 1024 and 4096 streams.

Variants, alternating in one process: meters off and on, each without a post-chain and with the voice chain (four equalizer
sections, compressor, limiter).  With meters on, every call is followed by the getter a server would call (pvgpu_get_meters into
preallocated arrays on host rows, pvgpu_get_meters_device on device rows), inside the timed window.
Passes: int16 host rows through processBlock and float32 device rows through processBlockDevice with a synchronise after each
call (p50 / p99 / max wall time per call); the meter kernels' device time per launch (torch.profiler, a process of its own, with
k_postchain beside them for scale); the card's name, power limit and maximum SM clock (nvidia-smi) in the same run.
Prints one JSON object per measurement.  Usage on a GPU box: python scripts/live_loudness_latency.py [--out FILE]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import audiomod_b200 as A  # noqa: E402
from audiomod_b200 import _lib  # noqa: E402
from audiomod_b200.synth import int16_to_float, synth_int16  # noqa: E402

SR, B, SHIFT, FFT = 44100, 480, 7.0, 2048
SIZES = (1024, 4096)
ROUNDS = 3          # the variants alternate this many times per size
SECS = 2.0          # audio per instance and round: 183 calls of 480 samples
WARM = 20           # calls per instance not timed (first launches, ring and arena growth)
# voice EQ: 100 Hz high-pass, -2 dB at 300 Hz (mud), +3 dB at 3 kHz (presence), 8 kHz low-pass; {use, cutoff, Q, gain} x 8
VOICE_EQ = [1, 100, 0.7, 0.0,  0, 400, 0.3, -1.5,  1, 300, 1.0, -2.0,  0, 2000, 0.3, 1.5,
            1, 3000, 1.0, 3.0,  0, 4000, 0.3, 1.5,  0, 5000, 0.3, -1.5,  1, 8000, 0.7, 0.0]
COMP_LIM = [("compressor", -20.0, 4.0, 3.0, 5.0, 50.0), ("limiter", -3.0, 0.0, 1.0, 80.0)]
VOICE = A.equalizer_chain(VOICE_EQ) + COMP_LIM
VARIANTS = [(meters, chain) for chain in ("none", "voice") for meters in (False, True)]
_fp = C.POINTER(C.c_float)


def name(v):
    return f"meters_{'on' if v[0] else 'off'}/chain_{v[1]}"


def make(S, fmt, v):
    pv = A.phasevocoder(SR, 1, 1.0, SHIFT, A.NORMAL_SHIFT, A.PHASE_LOCKED, FFT, streams=S, fmt=fmt)
    if v[1] == "voice":
        pv.set_postchain(VOICE)
    if v[0]:
        pv.set_meters()
    return pv


def host_calls(S, x, v):
    pv = make(S, A.S16, v)
    L = _lib.lib()
    m, s, p, n = np.empty(S, np.float32), np.empty(S, np.float32), np.empty(S, np.float32), C.c_int64()
    args = (pv._h, m.ctypes.data_as(_fp), s.ctypes.data_as(_fp), p.ctypes.data_as(_fp), C.byref(n))
    times = []
    for i in range(0, x.shape[1] - B + 1, B):
        blk = np.ascontiguousarray(x[:, i:i + B])
        t0 = time.perf_counter()
        pv.processBlock(blk)
        if v[0]:
            _lib.check(L.pvgpu_get_meters(*args))
        times.append(time.perf_counter() - t0)
    pv.close()
    return times[WARM:]


def device_calls(S, d, v, prof=None):
    """Per-call wall time of float32 device rows, the caller's stream synchronised after each call."""
    import torch
    pv = make(S, A.F32, v)
    dm = torch.empty(3 * S, dtype=torch.float32, device="cuda")
    st = torch.cuda.Stream()
    n = d.shape[1]
    times = []
    with torch.cuda.stream(st):
        for i in range(n // B):
            if i == WARM and prof is not None:
                prof.start()
            t0 = time.perf_counter()
            pv.processBlockDevice(d.data_ptr() + 4 * i * B, n, B, st.cuda_stream)
            if v[0]:
                pv.metersDevice(dm.data_ptr(), st.cuda_stream)
            st.synchronize()
            times.append(time.perf_counter() - t0)
        if prof is not None:
            prof.stop()
    pv.close()
    return times[WARM:]


def profile_child():
    """The kernel-time pass, in a process of its own: tracing slows the host, and the timed passes run without it."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for S in SIZES:
        d = torch.from_numpy(inputs(S)[A.F32]).cuda()
        for v in VARIANTS:
            if not v[0]:
                continue
            prof = profile(activities=[ProfilerActivity.CUDA])
            device_calls(S, d, v, prof)
            for e in prof.key_averages():
                if "k_meter" in e.key or ("k_postchain" in e.key and "reset" not in e.key):
                    t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                    print(json.dumps({"pass": "kernel_device_time (torch.profiler, device rows)", "streams": S, "variant": name(v),
                                      "kernel": e.key[:90], "launches": e.count, "us_per_launch": round(t / max(e.count, 1), 2)}), flush=True)


def inputs(S):
    x16 = np.ascontiguousarray(np.tile(synth_int16(2, SR, SECS, 1), (S, 1)))
    return {A.F32: np.ascontiguousarray(int16_to_float(x16)), A.S16: x16}


def stats(t):
    t = np.array(t) * 1e3
    return {"calls": int(t.size), "p50_ms": round(float(np.median(t)), 4), "p99_ms": round(float(np.percentile(t, 99)), 4),
            "max_ms": round(float(t.max()), 4)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--profile-child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.profile_child:
        profile_child()
        return
    import torch
    lines = []

    def emit(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    emit({"gpu": smi.stdout.strip().splitlines()[1:2] or smi.stdout.strip(), "nvidia_smi_rc": smi.returncode,
          "config": f"cfg4 mono {SR} Hz, +{SHIFT} st, FFT {FFT}, {B}-sample blocks ({1e3 * B / SR:.2f} ms of audio)",
          "chain": VOICE, "variants": [name(v) for v in VARIANTS]})
    for S in SIZES:
        xs = inputs(S)
        d = torch.from_numpy(xs[A.F32]).cuda()
        host = {v: [] for v in VARIANTS}
        dev = {v: [] for v in VARIANTS}
        for _ in range(ROUNDS):
            for v in VARIANTS:
                host[v] += host_calls(S, xs[A.S16], v)
                dev[v] += device_calls(S, d, v)
        for v in VARIANTS:
            emit({"pass": "host_rows_processBlock", "rows_fmt": "s16", "streams": S, "variant": name(v), **stats(host[v]),
                  "realtime_streams_per_gpu_at_p99": int(S * (B / SR) * 1e3 / stats(host[v])["p99_ms"])})
        for v in VARIANTS:
            emit({"pass": "device_rows_processBlockDevice_synchronised", "rows_fmt": "f32", "streams": S, "variant": name(v), **stats(dev[v])})
        del xs, d
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--profile-child"], capture_output=True, text=True)
    if child.returncode != 0:
        raise SystemExit(f"profiler pass failed ({child.returncode}):\n{child.stderr[-4000:]}")
    for line in child.stdout.splitlines():
        if line.startswith("{"):
            emit(json.loads(line))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
