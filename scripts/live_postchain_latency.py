"""Live batch per-call latency with a post-chain of effects (pvgpu_set_postchain) against the same live batch without one, cfg4:
mono 44.1 kHz, +7 semitones, FFT 2048, 480-sample blocks, S = 1024 and 4096 streams.

Variants, alternating in one process:
  * none                     -- no chain;
  * comp_lim                 -- [compressor, limiter];
  * voice                    -- equalizer_chain(VOICE_EQ) + compressor + limiter (the usual chain of a voice path).
Passes: host rows through processBlock, float32 and int16 (p50 / p99 / max wall time per call, what the chain adds at p50 and
p99, real-time streams per GPU at p99); float32 device rows through processBlockDevice, sustained time per call; the post-chain
kernel's own device time per launch (torch.profiler); the card's name, power limit and maximum SM clock (nvidia-smi) in the
same run.  Prints one JSON object per measurement.  Usage on a GPU box: python scripts/live_postchain_latency.py [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import audiomod_b200 as A  # noqa: E402
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
CHAINS = {"none": [], "comp_lim": COMP_LIM, "voice": A.equalizer_chain(VOICE_EQ) + COMP_LIM}
VARIANTS = ("none", "comp_lim", "voice")


def inputs(S):
    x16 = np.ascontiguousarray(np.tile(synth_int16(2, SR, SECS, 1), (S, 1)))
    return {A.F32: np.ascontiguousarray(int16_to_float(x16)), A.S16: x16}


def make(S, fmt, variant):
    pv = A.phasevocoder(SR, 1, 1.0, SHIFT, A.NORMAL_SHIFT, A.PHASE_LOCKED, FFT, streams=S, fmt=fmt)
    pv.set_postchain(CHAINS[variant])
    return pv


def host_calls(S, fmt, x, variant):
    pv = make(S, fmt, variant)
    times = []
    for i in range(0, x.shape[1] - B + 1, B):
        blk = np.ascontiguousarray(x[:, i:i + B])
        t0 = time.perf_counter()
        pv.processBlock(blk)
        times.append(time.perf_counter() - t0)
    pv.close()
    return times[WARM:]


def device_calls(S, x, variant, prof=None):
    import torch
    d = torch.from_numpy(x).cuda()
    pv = make(S, A.F32, variant)
    st = torch.cuda.Stream()
    n = x.shape[1]
    calls = n // B
    with torch.cuda.stream(st):
        for i in range(WARM):
            pv.processBlockDevice(d.data_ptr() + 4 * i * B, n, B, st.cuda_stream)
        st.synchronize()
        t0 = time.perf_counter()
        if prof is not None:
            prof.start()
        for i in range(WARM, calls):
            pv.processBlockDevice(d.data_ptr() + 4 * i * B, n, B, st.cuda_stream)
        st.synchronize()
        total = time.perf_counter() - t0
        if prof is not None:
            prof.stop()
    pv.close()
    return 1e3 * total / (calls - WARM)


def chain_kernel_us(S, x, variant):
    """Device time per launch of the post-chain kernel (k_postchain) over the timed device-row calls, from CUPTI via torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    prof = profile(activities=[ProfilerActivity.CUDA])
    device_calls(S, x, variant, prof)
    total, count = 0.0, 0
    for e in prof.key_averages():
        if "k_postchain<" in e.key and "reset" not in e.key:
            total += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
            count += e.count
    return total / max(count, 1), count


def profile_child():
    """The kernel-time pass, in a process of its own: tracing slows the host, and the timed passes above run without it."""
    for S in SIZES:
        x = inputs(S)[A.F32]
        for v in VARIANTS:
            if v == "none":
                continue
            us, count = chain_kernel_us(S, x, v)
            print(json.dumps({"pass": "k_postchain_device_time (torch.profiler, device rows)", "streams": S, "variant": v,
                              "ctas": (S + 31) // 32, "launches": count, "us_per_launch": round(us, 2)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--profile-child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.profile_child:
        profile_child()
        return
    lines = []

    def emit(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    emit({"gpu": smi.stdout.strip().splitlines()[1:2] or smi.stdout.strip(), "nvidia_smi_rc": smi.returncode,
          "config": f"cfg4 mono {SR} Hz, +{SHIFT} st, FFT {FFT}, {B}-sample blocks ({1e3 * B / SR:.2f} ms of audio)",
          "chains": {k: v for k, v in CHAINS.items()}})
    for S in SIZES:
        xs = inputs(S)
        for fmt, fname in ((A.F32, "f32"), (A.S16, "s16")):
            host = {v: [] for v in VARIANTS}
            for _ in range(ROUNDS):
                for v in VARIANTS:
                    host[v] += host_calls(S, fmt, xs[fmt], v)
            base = np.array(host["none"]) * 1e3
            for v in VARIANTS:
                t = np.array(host[v]) * 1e3
                p50, p99 = float(np.median(t)), float(np.percentile(t, 99))
                rec = {"pass": "host_rows_processBlock", "rows_fmt": fname, "streams": S, "variant": v, "calls": int(t.size),
                       "p50_ms": round(p50, 4), "p99_ms": round(p99, 4), "max_ms": round(float(t.max()), 4),
                       "realtime_streams_per_gpu_at_p99": int(S * (B / SR) * 1e3 / p99)}
                if v != "none":
                    rec["chain_adds_p50_ms"] = round(p50 - float(np.median(base)), 4)
                    rec["chain_adds_p99_ms"] = round(p99 - float(np.percentile(base, 99)), 4)
                emit(rec)
        dev = {v: [] for v in VARIANTS}
        for _ in range(ROUNDS):
            for v in VARIANTS:
                dev[v].append(device_calls(S, xs[A.F32], v))
        base = float(np.median(dev["none"]))
        for v in VARIANTS:
            per = float(np.median(dev[v]))
            rec = {"pass": "device_rows_processBlockDevice", "rows_fmt": "f32", "streams": S, "variant": v,
                   "rounds_ms_per_call": [round(u, 4) for u in dev[v]], "ms_per_call": round(per, 4),
                   "realtime_streams_per_gpu": int(S * (B / SR) * 1e3 / per)}
            if v != "none":
                rec["chain_adds_ms"] = round(per - base, 4)
            emit(rec)
        del xs
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
