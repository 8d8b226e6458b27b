"""Live batch per-call latency with per-stream post-chain parameters (pvgpu_set_stream_postchain), cfg4: mono 44.1 kHz,
+7 semitones, FFT 2048, 480-sample blocks, S = 1024 and 4096 streams, the voice chain (four equalizer sections, compressor,
limiter).

Variants, alternating in one process:
  * one_chain          -- (a) one chain for every stream (pvgpu_set_postchain);
  * same_per_stream    -- (b) the same parameters set per stream (no stream differs from the chain: the uniform kernel runs);
  * same_per_row_kernel -- (b) with PVGPU_POST_PER_ROW=1: the per-row kernel on identical parameters, against (a);
  * distinct           -- (c) distinct parameters per stream (the per-row kernel);
  * distinct_updates   -- (d) (c) plus 64 stream updates before every call (uploaded by the call).
Passes: int16 host rows through processBlock and float32 device rows through processBlockDevice with a synchronise after each
call (p50 / p99 / max wall time per call); the post-chain kernel's device time per launch (torch.profiler, a process of its
own); the setter's host time per update; the card's name, power limit and maximum SM clock (nvidia-smi) in the same run.
Prints one JSON object per measurement.  Usage on a GPU box: python scripts/live_postchain_streams_latency.py [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import audiomod_b200 as A  # noqa: E402
from audiomod_b200 import _lib  # noqa: E402
from audiomod_b200.phasevocoder import _fx_array  # noqa: E402
from audiomod_b200.synth import int16_to_float, synth_int16  # noqa: E402

SR, B, SHIFT, FFT = 44100, 480, 7.0, 2048
SIZES = (1024, 4096)
ROUNDS = 3          # the variants alternate this many times per size
SECS = 2.0          # audio per instance and round: 183 calls of 480 samples
WARM = 20           # calls per instance not timed (first launches, ring and arena growth)
UPDATES = 64        # stream updates before every call of distinct_updates
# voice EQ: 100 Hz high-pass, -2 dB at 300 Hz (mud), +3 dB at 3 kHz (presence), 8 kHz low-pass; {use, cutoff, Q, gain} x 8
VOICE_EQ = [1, 100, 0.7, 0.0,  0, 400, 0.3, -1.5,  1, 300, 1.0, -2.0,  0, 2000, 0.3, 1.5,
            1, 3000, 1.0, 3.0,  0, 4000, 0.3, 1.5,  0, 5000, 0.3, -1.5,  1, 8000, 0.7, 0.0]
COMP_LIM = [("compressor", -20.0, 4.0, 3.0, 5.0, 50.0), ("limiter", -3.0, 0.0, 1.0, 80.0)]
VOICE = A.equalizer_chain(VOICE_EQ) + COMP_LIM
VARIANTS = ["one_chain", "same_per_stream", "same_per_row_kernel", "distinct", "distinct_updates"]


def preset(j):
    """User j's voice preset: the voice chain's kinds, its own EQ gains, compressor and limiter settings (32 distinct presets)."""
    eq = list(VOICE_EQ)
    for b in range(8):
        eq[4 * b + 3] += ((j * 5 + 3 * b) % 9 - 4) * 0.5
    comp = ("compressor", -24.0 + (j % 8), 3.0 + (j % 3), 2.0 + 0.5 * (j % 4), 4.0 + (j % 5), 40.0 + 10.0 * (j % 4))
    lim = ("limiter", -3.0 - 0.5 * (j % 4), 0.5 * (j % 3), 1.0, 60.0 + 10.0 * (j % 3))
    return A.equalizer_chain(eq) + [comp, lim]


PRESETS = [_fx_array(preset(j)) for j in range(32)]
VOICE_ARR = _fx_array(VOICE)


def make(S, fmt, variant):
    os.environ["PVGPU_POST_PER_ROW"] = "1" if variant == "same_per_row_kernel" else "0"   # read when the instance is created
    pv = A.phasevocoder(SR, 1, 1.0, SHIFT, A.NORMAL_SHIFT, A.PHASE_LOCKED, FFT, streams=S, fmt=fmt)
    pv.set_postchain(VOICE)
    L = _lib.lib()
    if variant == "same_per_stream":
        for j in range(S):
            _lib.check(L.pvgpu_set_stream_postchain(pv._h, j, *VOICE_ARR))
    elif variant.startswith("distinct"):
        for j in range(S):
            _lib.check(L.pvgpu_set_stream_postchain(pv._h, j, *PRESETS[j % len(PRESETS)]))
    return pv


class Updater:
    """distinct_updates: UPDATES streams (a rotating window) get another preset before every call; host time per update kept."""
    def __init__(self, pv, S):
        self.pv, self.S, self.i, self.t = pv, S, 0, []

    def __call__(self):
        L = _lib.lib()
        t0 = time.perf_counter()
        for u in range(UPDATES):
            j = (self.i * UPDATES + u) % self.S
            _lib.check(L.pvgpu_set_stream_postchain(self.pv._h, j, *PRESETS[(j + self.i + 1) % len(PRESETS)]))
        self.t.append((time.perf_counter() - t0) / UPDATES)
        self.i += 1


def host_calls(S, x, variant, set_us):
    pv = make(S, A.S16, variant)
    upd = Updater(pv, S) if variant == "distinct_updates" else None
    times = []
    for i in range(0, x.shape[1] - B + 1, B):
        blk = np.ascontiguousarray(x[:, i:i + B])
        if upd:
            upd()
        t0 = time.perf_counter()
        pv.processBlock(blk)
        times.append(time.perf_counter() - t0)
    pv.close()
    if upd:
        set_us += upd.t[WARM:]
    return times[WARM:]


def device_calls(S, d, variant, prof=None):
    """Per-call wall time of float32 device rows, the caller's stream synchronised after each call."""
    import torch
    pv = make(S, A.F32, variant)
    upd = Updater(pv, S) if variant == "distinct_updates" else None
    st = torch.cuda.Stream()
    n = d.shape[1]
    times = []
    with torch.cuda.stream(st):
        for i in range(n // B):
            if i == WARM and prof is not None:
                prof.start()
            if upd:
                upd()
            t0 = time.perf_counter()
            pv.processBlockDevice(d.data_ptr() + 4 * i * B, n, B, st.cuda_stream)
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
            prof = profile(activities=[ProfilerActivity.CUDA])
            device_calls(S, d, v, prof)
            for e in prof.key_averages():
                if "k_postchain" in e.key and "reset" not in e.key:
                    t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
                    print(json.dumps({"pass": "kernel_device_time (torch.profiler, device rows)", "streams": S, "variant": v,
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
          "chain": VOICE, "updates_per_call": UPDATES})
    for S in SIZES:
        xs = inputs(S)
        d = torch.from_numpy(xs[A.F32]).cuda()
        host = {v: [] for v in VARIANTS}
        dev = {v: [] for v in VARIANTS}
        set_us = []
        for _ in range(ROUNDS):
            for v in VARIANTS:
                host[v] += host_calls(S, xs[A.S16], v, set_us)
                dev[v] += device_calls(S, d, v)
        for v in VARIANTS:
            emit({"pass": "host_rows_processBlock", "rows_fmt": "s16", "streams": S, "variant": v, **stats(host[v]),
                  "realtime_streams_per_gpu_at_p99": int(S * (B / SR) * 1e3 / stats(host[v])["p99_ms"])})
        for v in VARIANTS:
            emit({"pass": "device_rows_processBlockDevice_synchronised", "rows_fmt": "f32", "streams": S, "variant": v, **stats(dev[v])})
        emit({"pass": "pvgpu_set_stream_postchain host time (ctypes call included)", "streams": S, "updates": len(set_us) * UPDATES,
              "p50_us": round(1e6 * float(np.median(set_us)), 2), "p99_us": round(1e6 * float(np.percentile(set_us, 99)), 2)})
        del xs, d
    os.environ.pop("PVGPU_POST_PER_ROW", None)
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
