"""Live batch per-call latency, float32 rows against int16 rows (pvgpu_process_block vs pvgpu_process_block_s16 and their
device-row twins), cfg4: mono 44.1 kHz, +7 semitones, FFT 2048, 480-sample blocks, S = 1024 and 4096 streams.

One run measures, with float32 and int16 instances alternating in the same process:
  * host rows through processBlock: p50 / p99 / max wall time per call and the real-time streams one GPU keeps up with
    (S x block duration / p99);
  * host rows with PVGPU_STREAM_TRACE=1, in a child process of its own (tracing slows the host): the library's pack / copy /
    kernel breakdown per call;
  * device rows through processBlockDevice: sustained time per call;
  * the card's name, power limit and maximum SM clock (nvidia-smi), taken in the same run.
Prints one JSON object per measurement.  Usage on a GPU box: python scripts/live_s16_latency.py [--out FILE]"""
import argparse
import json
import os
import re
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402

import audiomod_b200 as A  # noqa: E402
from audiomod_b200.synth import int16_to_float, synth_int16  # noqa: E402

SR, B, SHIFT, FFT = 44100, 480, 7.0, 2048
SIZES = (1024, 4096)
ROUNDS = 3          # f32 / s16 alternate this many times per size
SECS = 2.0          # audio per instance and round: 183 calls of 480 samples
WARM = 20           # calls per instance not timed (first launches, ring and arena growth)


def inputs(S):
    x16 = np.ascontiguousarray(np.tile(synth_int16(2, SR, SECS, 1), (S, 1)))
    return {A.F32: np.ascontiguousarray(int16_to_float(x16)), A.S16: x16}


def host_calls(S, fmt, x):
    pv = A.phasevocoder(SR, 1, 1.0, SHIFT, A.NORMAL_SHIFT, A.PHASE_LOCKED, FFT, streams=S, fmt=fmt)
    times = []
    for i in range(0, x.shape[1] - B + 1, B):
        blk = np.ascontiguousarray(x[:, i:i + B])
        t0 = time.perf_counter()
        pv.processBlock(blk)
        times.append(time.perf_counter() - t0)
    pv.close()
    return times[WARM:]


def device_calls(S, fmt, x):
    import torch
    d = torch.from_numpy(x).cuda()
    esz = x.dtype.itemsize
    pv = A.phasevocoder(SR, 1, 1.0, SHIFT, A.NORMAL_SHIFT, A.PHASE_LOCKED, FFT, streams=S, fmt=fmt)
    st = torch.cuda.Stream()
    n = x.shape[1]
    calls = n // B
    with torch.cuda.stream(st):
        for i in range(WARM):
            pv.processBlockDevice(d.data_ptr() + esz * i * B, n, B, st.cuda_stream)
        st.synchronize()
        t0 = time.perf_counter()
        for i in range(WARM, calls):
            pv.processBlockDevice(d.data_ptr() + esz * i * B, n, B, st.cuda_stream)
        st.synchronize()
        total = time.perf_counter() - t0
    pv.close()
    return 1e3 * total / (calls - WARM)


NAMES = {A.F32: "f32", A.S16: "s16"}


def trace_child():
    """PVGPU_STREAM_TRACE=1 is read once per process: this pass runs in a child and marks which instance each report belongs to."""
    for S in SIZES:
        xs = inputs(S)
        for fmt in (A.F32, A.S16):
            sys.stderr.write(f"@@ {NAMES[fmt]} {S}\n")
            sys.stderr.flush()
            host_calls(S, fmt, xs[fmt])


def parse_trace(text):
    """Last full report of every instance: host phases and device phases, microseconds per call."""
    out, cur = [], None
    num = r"([0-9.]+)"
    for line in text.splitlines():
        if line.startswith("@@ "):
            _, f, s = line.split()
            cur = {"rows_fmt": f, "streams": int(s)}
            out.append(cur)
            continue
        m = re.search(rf"pack {num} us, enqueue {num}, device wait {num}, trim {num} \| device: uploads {num}, kernels {num}, "
                      rf"output copy {num}, window compaction {num}", line)
        if m and cur is not None:
            keys = ("host_pack_us", "host_enqueue_us", "host_device_wait_us", "host_trim_us", "dev_uploads_us", "dev_kernels_us",
                    "dev_output_copy_us", "dev_window_compaction_us")
            cur.update({k: float(v) for k, v in zip(keys, m.groups())})
        m = re.search(rf"until the packed block is ready {num} us, input copy \+ placement {num}", line)
        if m and cur is not None:
            cur["dev_until_packed_us"], cur["dev_input_copy_placement_us"] = float(m.group(1)), float(m.group(2))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--trace-child", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.trace_child:
        trace_child()
        return
    lines = []

    def emit(obj):
        s = json.dumps(obj)
        print(s, flush=True)
        lines.append(s)

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    emit({"gpu": smi.stdout.strip().splitlines()[1:2] or smi.stdout.strip(), "nvidia_smi_rc": smi.returncode,
          "config": f"cfg4 mono {SR} Hz, +{SHIFT} st, FFT {FFT}, {B}-sample blocks ({1e3 * B / SR:.2f} ms of audio)"})
    for S in SIZES:
        xs = inputs(S)
        host = {A.F32: [], A.S16: []}
        for _ in range(ROUNDS):
            for fmt in (A.F32, A.S16):
                host[fmt] += host_calls(S, fmt, xs[fmt])
        for fmt in (A.F32, A.S16):
            t = np.array(host[fmt]) * 1e3
            p99 = float(np.percentile(t, 99))
            emit({"pass": "host_rows_processBlock", "rows_fmt": NAMES[fmt], "streams": S, "calls": int(t.size),
                  "p50_ms": round(float(np.median(t)), 4), "p99_ms": round(p99, 4), "max_ms": round(float(t.max()), 4),
                  "realtime_streams_per_gpu_at_p99": int(S * (B / SR) * 1e3 / p99),
                  "bytes_per_call_both_directions": 2 * S * B * xs[fmt].dtype.itemsize})
        dev = {A.F32: [], A.S16: []}
        for _ in range(ROUNDS):
            for fmt in (A.F32, A.S16):
                dev[fmt].append(device_calls(S, fmt, xs[fmt]))
        for fmt in (A.F32, A.S16):
            per = float(np.median(dev[fmt]))
            emit({"pass": "device_rows_processBlockDevice", "rows_fmt": NAMES[fmt], "streams": S, "rounds_ms_per_call": [round(v, 4) for v in dev[fmt]],
                  "ms_per_call": round(per, 4), "realtime_streams_per_gpu": int(S * (B / SR) * 1e3 / per)})
        del xs
    env = dict(os.environ, PVGPU_STREAM_TRACE="1")
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--trace-child"], env=env, capture_output=True, text=True)
    if child.returncode != 0:
        raise SystemExit(f"trace pass failed ({child.returncode}):\n{child.stderr[-4000:]}")
    for rec in parse_trace(child.stderr):
        emit(dict({"pass": "host_rows_trace (PVGPU_STREAM_TRACE=1, last 50 calls)"}, **rec))
    if a.out:
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
