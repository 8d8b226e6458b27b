#!/usr/bin/env python
"""Benchmark of the batched phase-vocoder hot path (BASELINE.json metric: audio-seconds per wall-second,
2048-point pitch shift, batched streams).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--streams S] [--secs T] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference      # the reference's own CPU path on the host cores

Workload (config 4 of BASELINE.json): S = 4096 synthetic mono 44.1 kHz streams of 10 s PER GPU, +7 semitones,
coremode 1 (phase locked), FFT 2048.  A step is one pass of the whole path over that batch.  `value` is measured with
the inputs resident in HBM (7.2 GB of float32 PCM per GPU, far larger than L2); `e2e` goes through the host-buffer
entry point (pinned host memory -> H2D -> kernels -> D2H) every step -- int16 PCM rows (the reference CLI's own WAV
format) lead, float32 rows are reported beside them.  Streams are independent, so multi-GPU is one process per GPU with
its own batch and no collective on the data path; the default line is weak scaling (4096 streams per GPU) and at N > 1
carries the strong-scaling figure (4096 streams in total, BASELINE.json configs[3] read literally) beside it.
After the timed regions a few rows of the batch that was actually timed are compared with the unmodified reference
(oracle/_ref/pvref_drv on the same samples): `parity` in the JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SR, SEMITONES, FFT, COREMODE, MODE = 44100, 7.0, 2048, 1, 0
CHANNELS, TIMERATIO = 1, 1.0
# The judged line is cfg4 (the default).  The other BASELINE.json configurations can be timed with --workload for the
# notes in profiles/; they are parity-test cases, not bench lines.
WORKLOADS = {   # name: (sr, channels, timeratio, semitones, mode, coremode, fftsize, default streams)
    "cfg4": (44100, 1, 1.0, 7.0, 0, 1, 2048, 4096),
    "cfg1": (44100, 2, 1.0, 4.0, 0, 1, 2048, 2048),
    "cfg2": (48000, 2, 1.5, 0.0, 5, 1, 4096, 1024),
    "cfg3-formant": (44100, 1, 1.0, 4.0, 2, 1, 2048, 4096),
    "cfg3-gender": (44100, 1, 1.0, -4.0, 1, 1, 2048, 4096),
    "cfg5-robotic-2048": (44100, 2, 1.0, 0.0, 6, 1, 2048, 1024),
    "cfg5-whisper-2048": (44100, 2, 1.0, 0.0, 7, 1, 2048, 1024),
    "cfg5-vocoder-2048": (44100, 2, 1.0, 0.0, 3, 1, 2048, 1024),
    "cfg5-robotic-512": (44100, 2, 1.0, 0.0, 6, 1, 512, 1024),
    "cfg5-robotic-8192": (44100, 2, 1.0, 0.0, 6, 1, 8192, 1024),
    # not BASELINE configurations: the optional cepstral gender mode, and FFT sizes outside 512..8192 (generic one-CTA-per-frame kernels)
    "cepstral-gender": (44100, 1, 1.0, 4.0, 8, 1, 2048, 4096),
    "generic-256": (44100, 1, 1.0, 7.0, 0, 1, 256, 1024),
    "generic-16384": (48000, 1, 1.25, 0.0, 5, 1, 16384, 256),
}
METRIC = "audio-sec/sec, 2048-pt PV pitch-shift, batched streams"
UNIT = "audio-s/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (default: the workload's)")
    ap.add_argument("--workload", default="cfg4", choices=sorted(WORKLOADS))
    ap.add_argument("--secs", type=float, default=10.0)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames-per-chunk", type=int, default=0)
    ap.add_argument("--rows-per-group", type=int, default=0)
    ap.add_argument("--contexts", type=int, default=0)
    ap.add_argument("--cpu-streams-per-core", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg at N > 1")
    ap.add_argument("--no-latency", action="store_true", help="skip the streaming per-call latency leg")
    ap.add_argument("--parity-rows", type=int, default=4)
    ap.add_argument("--host-alloc", default="numa", choices=["numa", "numa-huge", "torch"],
                    help="pinned host buffers of the e2e legs: pvgpu_host_alloc on the GPU's NUMA node (default), the same on explicit 2 MB pages, or torch pin_memory")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (rank 0; a fixed sample of rows, see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    global SR, CHANNELS, TIMERATIO, SEMITONES, MODE, COREMODE, FFT
    SR, CHANNELS, TIMERATIO, SEMITONES, MODE, COREMODE, FFT, default_streams = WORKLOADS[args.workload]
    if args.streams <= 0:
        args.streams = default_streams
    return args


def workload_config(args, n_gpus):
    return {"workload": f"{args.workload}: {args.streams} synthetic {'mono' if CHANNELS == 1 else 'stereo'} {SR / 1000:g} kHz {args.secs:g} s streams per GPU, "
                        f"time ratio {TIMERATIO:g}, {SEMITONES:+g} semitones, mode {MODE}, coremode {COREMODE}, FFT {FFT}"
                        + (" (BASELINE.json configs[3])" if args.workload == "cfg4" else ""),
            "streams_per_gpu": args.streams, "stream_seconds": args.secs, "sample_rate": SR, "semitones": SEMITONES, "fftsize": FFT,
            "coremode": COREMODE, "channels": CHANNELS, "time_ratio": TIMERATIO, "mode": MODE, "n_gpus": n_gpus, "sharding": "streams split across GPUs, no collective",
            "l2": "inputs (7.2 GB/GPU at the default size) exceed the 126 MB L2; no explicit flush"}


# ---------------------------------------------------------------------------------------------------------------
# CPU side: the unmodified reference (oracle/_ref/pvref_drv, one OS process per stream because the reference keeps
# process-global state) or, if it was not built, the C restatement.  Only used for cpu_baseline / --impl reference.
# ---------------------------------------------------------------------------------------------------------------
def cpu_run(n_streams: int, secs: float, cores: int):
    """Process n_streams synthetic streams on `cores` host cores; returns (audio-s/s, kind, seconds)."""
    from audiomod_b200.synth import synth
    from oracle import pv_oracle as O
    xs = [synth(4000 + i, SR, secs, CHANNELS) for i in range(n_streams)]
    if O.have_ref():
        kind = "reference"
        with tempfile.TemporaryDirectory(prefix="pvbench_") as d:
            for i, x in enumerate(xs):
                x.tofile(os.path.join(d, f"i{i}.f32"))
            cmds = [[O.REF_DRV, str(SR), str(CHANNELS), repr(TIMERATIO), repr(SEMITONES), str(MODE), str(COREMODE), str(FFT),
                     os.path.join(d, f"i{i}.f32"), os.path.join(d, f"o{i}.f32")] for i in range(n_streams)]
            t0 = time.perf_counter()
            running, nxt = [], 0
            while nxt < len(cmds) or running:
                while nxt < len(cmds) and len(running) < cores:
                    running.append(subprocess.Popen(cmds[nxt]))
                    nxt += 1
                p = running.pop(0)
                if p.wait() != 0:
                    raise RuntimeError("reference driver failed")
            dt = time.perf_counter() - t0
    else:
        kind = "port"
        import multiprocessing as mp
        O.lib()
        t0 = time.perf_counter()
        with mp.get_context("fork").Pool(cores) as pool:
            pool.map(_port_one, xs)
        dt = time.perf_counter() - t0
    return n_streams * secs / dt, kind, dt


def _port_one(x):
    from oracle import pv_oracle as O
    return O.run_offline(x, SR, timeratio=TIMERATIO, semitones=SEMITONES, mode=MODE, coremode=COREMODE, fftsize=FFT).shape[1]


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n = max(cores, cores * args.cpu_streams_per_core)
    for _ in range(min(args.warmup, 1)):
        cpu_run(cores, min(args.secs, 2.0), cores)
    vals, times, kind = [], [], "port"
    for _ in range(args.steps):
        v, kind, dt = cpu_run(n, args.secs, cores)
        vals.append(v)
        times.append(dt)
    value = float(np.mean(vals))
    sample = f"{n} of the workload's streams ({args.secs:g} s each) per step, one OS process per stream on {cores} cores"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, args.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU during the timed region (NVML; nvidia-smi as a fallback)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.sm, self.max_sm, self.reasons, self.stop_flag = index, [], [], set(), threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        self.sm.append(float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)))
        self.max_sm.append(float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM)))
        r = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(n, "nvmlDeviceGetCurrentClocksEventReasons") \
            else n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40)):
            if r & bit:
                self.reasons.add(name)

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        c = [v.strip() for v in out.split(",")]
        self.sm.append(float(c[0]))
        self.max_sm.append(float(c[1]))
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[2:]):
            if v.lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self.stop_flag.is_set():
            try:
                self._sample_nvml() if self.nvml else self._sample_smi()
            except Exception:
                pass
            self.stop_flag.wait(0.02 if self.nvml else 0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.max_sm) if self.max_sm else None,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def make_inputs(torch, dev, streams, n, seed):
    """Seeded synthetic PCM generated on the GPU (same recipe family as audiomod_b200/synth.py): 8 harmonics with
    vibrato and tremolo plus noise, quantised to int16 and presented as int16/32768 like the reference WAV reader."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    out = torch.empty((streams, n), dtype=torch.float32, device=dev)
    t = torch.arange(n, dtype=torch.float64, device=dev) / SR
    step = 64
    for s0 in range(0, streams, step):
        m = min(step, streams - s0)
        u = torch.rand((m, 1), generator=g, device=dev, dtype=torch.float64) * 12 - 6
        f0 = 110.0 * 2.0 ** (u / 12.0)
        vph = torch.rand((m, 1), generator=g, device=dev, dtype=torch.float64) * 2 * np.pi
        tph = torch.rand((m, 1), generator=g, device=dev, dtype=torch.float64) * 2 * np.pi
        cyc = f0 * (t[None, :] - 0.01 / (2 * np.pi * 0.7) * torch.cos(2 * np.pi * 0.7 * t[None, :] + vph))
        cyc = (cyc - torch.floor(cyc)).to(torch.float32) * (2 * np.pi)
        x = torch.zeros((m, n), dtype=torch.float32, device=dev)
        for k in range(8):
            ph0 = torch.rand((m, 1), generator=g, device=dev, dtype=torch.float32) * (2 * np.pi)
            x += (0.25 / (k + 1)) * torch.sin((k + 1) * cyc + ph0)
        trem = (0.8 + 0.2 * torch.sin(2 * np.pi * 1.3 * t[None, :] + tph)).to(torch.float32)
        x = x * trem + 0.01 * torch.randn((m, n), generator=g, device=dev, dtype=torch.float32)
        q = torch.round(torch.clamp(x, -1.0, 1.0) * 32767.0)
        out[s0:s0 + m] = (q.to(torch.float64) * (1.0 / 32768.0)).to(torch.float32)
        del cyc, x, trem, q
    return out


def reference_rows(rows_f32):
    """The unmodified reference (one fresh process per stream) on the given [channels, n] float32 streams; falls back to the
    C restatement (pinned bit-exactly to it by tests/test_oracle_vs_ref.py) when oracle/_ref was not shipped."""
    from oracle import pv_oracle as O
    if MODE in (8, 9):   # the optional cepstral modes: checked against the reference built with formantShiftSlice switched on
        if not O.have_ref_cepstral():
            raise SystemExit("the cepstral workloads need oracle/_ref/pvref_drv_cep as their checker (use --no-parity)")
        return [O.run_ref(x, SR, timeratio=TIMERATIO, semitones=SEMITONES, mode=MODE - 7, coremode=COREMODE, fftsize=FFT, cepstral=True)
                for x in rows_f32], "reference"
    if O.have_ref():
        return [O.run_ref(x, SR, timeratio=TIMERATIO, semitones=SEMITONES, mode=MODE, coremode=COREMODE, fftsize=FFT) for x in rows_f32], "reference"
    return [O.run_offline(x, SR, timeratio=TIMERATIO, semitones=SEMITONES, mode=MODE, coremode=COREMODE, fftsize=FFT) for x in rows_f32], "port"


def parity_f32(got, refs):
    """got / refs: lists of [channels, n] arrays.  counts, worst SNR and max-abs over all channels."""
    ok, snr_min, mx = True, float("inf"), 0.0
    for y, r in zip(got, refs):
        if y.shape != r.shape:
            ok = False
            m = min(y.shape[1], r.shape[1])
            y, r = y[:, :m], r[:, :m]
        for c in range(r.shape[0]):
            e = y[c].astype(np.float64) - r[c].astype(np.float64)
            pw, pe = float(np.sum(r[c].astype(np.float64) ** 2)), float(np.sum(e ** 2))
            mx = max(mx, float(np.max(np.abs(e))) if e.size else 0.0)
            if pe > 0 and pw > 0:
                snr_min = min(snr_min, 10 * np.log10(pw / pe))
    return {"rows": sum(r.shape[0] for r in refs), "counts_equal": ok, "min_snr_db": None if np.isinf(snr_min) else snr_min, "max_abs": mx}


def parity_s16(got, refs):
    """int16 rows against the reference's float output through its own WAV writer rule (x * 32768, clamp, truncate)."""
    ok, lsb, exact, total, snr_min = True, 0, 0, 0, float("inf")
    for y, r in zip(got, refs):
        want = np.clip(r * np.float32(32768.0), -32768.0, 32767.0).astype(np.int32)
        if y.shape != want.shape:
            ok = False
            m = min(y.shape[1], want.shape[1])
            y, want = y[:, :m], want[:, :m]
        d = y.astype(np.int32) - want
        lsb = max(lsb, int(np.max(np.abs(d))) if d.size else 0)
        exact += int(np.sum(d == 0))
        total += d.size
        for c in range(want.shape[0]):
            pw, pe = float(np.sum(want[c].astype(np.float64) ** 2)), float(np.sum(d[c].astype(np.float64) ** 2))
            if pe > 0 and pw > 0:
                snr_min = min(snr_min, 10 * np.log10(pw / pe))
    return {"rows": sum(r.shape[0] for r in refs), "counts_equal": ok, "max_lsb": lsb, "exact_frac": exact / max(total, 1),
            "max_abs": lsb / 32768.0, "min_snr_db": None if np.isinf(snr_min) else snr_min}


def stream_latency():
    """Per-call wall time of the streaming drop-in API (processBlock on the CLI's 480-sample blocks, host buffers, one
    instance = one audiomod::phasevocoder object): p50 / p99 in ms for three configurations."""
    import audiomod_b200 as A
    from audiomod_b200.synth import synth
    out = {}
    for name, ch, st, mode in (("cfg4_mono_p7", 1, 7.0, 0), ("cfg1_stereo_p4", 2, 4.0, 0), ("robotic_stereo", 2, 0.0, 6)):
        x = synth(1, 44100, 3.0, ch)
        B = 480
        pv = A.phasevocoder(44100, ch, 1.0, st, mode, 1, 2048)
        times = []
        for i in range(0, x.shape[1] - B, B):
            blk = np.ascontiguousarray(x[:, i:i + B])
            t0 = time.perf_counter()
            pv.processBlock(blk)
            times.append(time.perf_counter() - t0)
        pv.close()
        t = np.array(times[20:]) * 1e3
        out[name] = {"p50": float(np.percentile(t, 50)), "p99": float(np.percentile(t, 99)), "max": float(t.max()), "calls": int(t.size)}
    out["block_samples"] = 480
    out["block_ms_of_audio"] = 1e3 * 480 / 44100
    # live batch (pvgpu_create_multi): S cfg4 streams in lock-step through one instance, the same 480-sample blocks; a call serves
    # all of them.  real_time_streams = how many such streams one GPU keeps up with at this block size (S x block duration / p99).
    live = {}
    for S in (64, 1024, 4096):
        x = np.ascontiguousarray(np.tile(synth(2, 44100, 1.5, 1), (S, 1)))
        x *= (1.0 + 0.001 * np.arange(S, dtype=np.float32))[:, None]          # distinct rows
        pv = A.phasevocoder(44100, 1, 1.0, 7.0, 0, 1, 2048, streams=S)
        times = []
        for i in range(0, x.shape[1] - B, B):
            blk = np.ascontiguousarray(x[:, i:i + B])
            t0 = time.perf_counter()
            pv.processBlock(blk)
            times.append(time.perf_counter() - t0)
        pv.close()
        t = np.array(times[20:]) * 1e3
        p50, p99 = float(np.percentile(t, 50)), float(np.percentile(t, 99))
        live[str(S)] = {"p50": p50, "p99": p99, "max": float(t.max()), "calls": int(t.size), "real_time_streams": int(S * out["block_ms_of_audio"] / p99),
                        "audio_s_per_s": S * out["block_ms_of_audio"] / p50}
    out["live_batch_cfg4"] = live
    # the same live batch fed device rows (pvgpu_process_block_device): nothing crosses PCIe and no call waits for the device, so
    # the figure is the sustained time per call over the whole run (one synchronisation at the end) and the host time to enqueue one
    import torch
    devrows = {}
    for S in (1024, 4096):
        x = np.ascontiguousarray(np.tile(synth(2, 44100, 1.5, 1), (S, 1)))
        x *= (1.0 + 0.001 * np.arange(S, dtype=np.float32))[:, None]
        d = torch.from_numpy(x).cuda()
        pv = A.phasevocoder(44100, 1, 1.0, 7.0, 0, 1, 2048, streams=S)
        st = torch.cuda.Stream()
        n = x.shape[1]
        calls = (n - B) // B
        with torch.cuda.stream(st):
            for i in range(20):                                   # warm-up: allocations, ring growth
                pv.processBlockDevice(d.data_ptr() + 4 * i * B, n, B, st.cuda_stream)
            st.synchronize()
            enq = []
            t0 = time.perf_counter()
            for i in range(20, calls):
                t1 = time.perf_counter()
                pv.processBlockDevice(d.data_ptr() + 4 * i * B, n, B, st.cuda_stream)
                enq.append(time.perf_counter() - t1)
            st.synchronize()
            total = time.perf_counter() - t0
        pv.close()
        per_call = 1e3 * total / max(calls - 20, 1)
        devrows[str(S)] = {"ms_per_call_sustained": per_call, "host_enqueue_ms_p50": float(np.percentile(np.array(enq) * 1e3, 50)), "calls": calls - 20,
                           "real_time_streams": int(S * out["block_ms_of_audio"] / per_call), "audio_s_per_s": S * out["block_ms_of_audio"] / per_call}
    out["live_batch_device_rows_cfg4"] = devrows
    return out


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
        return
    import torch
    import torch.distributed as dist
    import audiomod_b200 as A

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the phase vocoder has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from audiomod_b200 import _lib
    _lib.lib().pvgpu_bind_thread_to_device(local)    # host thread (and its first-touch pages) on the GPU's NUMA node

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(x, op):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t.item())

    def max_over_ranks(x):
        return reduce(x, dist.ReduceOp.MAX) if world > 1 else x

    n = int(round(SR * args.secs))
    stream = torch.cuda.Stream()      # explicit stream: the batch forks from / joins into the caller's stream, events bracket it

    def make_batch(n_streams):
        S = n_streams * CHANNELS
        stride = (n + 3) & ~3
        d_in = torch.zeros((S, stride), dtype=torch.float32, device=dev)
        d_in[:, :n] = make_inputs(torch, dev, S, n, 1234 + rank)
        batch = A.PhaseVocoderBatch(n_streams, n, SR, CHANNELS, TIMERATIO, SEMITONES, MODE, COREMODE, FFT, device=local)
        if args.frames_per_chunk or args.rows_per_group or args.contexts:
            batch.tune(args.frames_per_chunk, args.rows_per_group, args.contexts)
        n_out = batch.plan(n)
        out_stride = (int(n_out.max()) + 3) & ~3
        d_out = torch.zeros((S, out_stride), dtype=torch.float32, device=dev)
        torch.cuda.synchronize()
        return batch, d_in, d_out, stride, out_stride, n_out

    def time_device(batch, d_in, d_out, stride, out_stride, steps, warmup):
        """K steps on `stream`, inputs resident in HBM, CUDA events on the launching stream, max over ranks (ms per step)."""
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                batch.run_device(d_in.data_ptr(), stride, d_out.data_ptr(), out_stride, stream.cuda_stream)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                batch.run_device(d_in.data_ptr(), stride, d_out.data_ptr(), out_stride, stream.cuda_stream)
            e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps

    host_bufs = []

    def host_array(dtype, shape):
        """page-locked host rows for the e2e legs"""
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if args.host_alloc == "torch":
            t = torch.empty(shape, dtype=torch.int16 if np.dtype(dtype) == np.int16 else torch.float32, pin_memory=True)
            host_bufs.append(t)
            return t.numpy()
        hb = A.HostBuffer(nbytes, local, True, args.host_alloc == "numa-huge")
        host_bufs.append(hb)
        return hb.array(dtype, shape)

    def time_host(batch, X, Y, fmt, steps):
        """K steps through the host-buffer entry point; every step copies its inputs H2D and its results D2H.  Timed with
        CUDA events on the device clock around the (synchronous) calls, max over ranks."""
        S = X.shape[0]
        in_rows = [X[r].ctypes.data for r in range(S)]
        out_rows = [Y[r].ctypes.data for r in range(S)]
        batch.run_host_rows(in_rows, out_rows, fmt)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            batch.run_host_rows(in_rows, out_rows, fmt)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)) / steps, batch.stats()

    n_streams = args.streams
    S = n_streams * CHANNELS
    batch, d_in, d_out, stride, out_stride, n_out = make_batch(n_streams)
    info = batch.info()

    # ---- device-resident throughput (the bench contract's `value`) ----
    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            batch.run_device(d_in.data_ptr(), stride, d_out.data_ptr(), out_stride, stream.cuda_stream)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ms_step = time_device(batch, d_in, d_out, stride, out_stride, args.steps, 0)
    stats = batch.stats()
    clocks = sampler.summary()
    audio_sec_per_step = world * n_streams * args.secs
    value = audio_sec_per_step / (ms_step / 1e3)
    n_out_min = int(n_out.min())
    checksum = float(d_out[:, :n_out_min].double().abs().mean().item())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, torch, d_out, n_out, n_streams)

    # rows of THIS batch checked against the reference after the timed regions (first / last / spread in between)
    pr = sorted(set(int(round(i * (n_streams - 1) / max(args.parity_rows - 1, 1))) for i in range(min(args.parity_rows, n_streams))))
    parity = None
    refs = None
    if not args.no_parity:
        xin = [d_in[s * CHANNELS:(s + 1) * CHANNELS, :n].cpu().numpy() for s in pr]
        refs, checker = reference_rows(xin)
        got = [d_out[s * CHANNELS:(s + 1) * CHANNELS, :int(n_out[s])].cpu().numpy() for s in pr]
        parity = {"checker": checker + (": oracle/_ref/pvref_drv, one fresh process per stream" if checker == "reference" else ": oracle/pv_oracle.c"),
                  "streams_checked": pr, "bar": "counts equal, >= 90 dB SNR, max-abs <= 1e-4 per channel",
                  "device_resident_f32": parity_f32(got, refs)}

    # per-kernel CUDA-event times: the same steps once more with one group in flight at a time, so that a kernel's
    # events bracket only that kernel (with the stages overlapped kernels of neighbouring chunks share the SMs)
    batch.tune(contexts=1)
    with torch.cuda.stream(stream):
        batch.run_device(d_in.data_ptr(), stride, d_out.data_ptr(), out_stride, stream.cuda_stream)
    torch.cuda.synchronize()
    batch.profile(True)
    pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        pe0.record(stream)
        for _ in range(args.steps):
            batch.run_device(d_in.data_ptr(), stride, d_out.data_ptr(), out_stride, stream.cuda_stream)
        pe1.record(stream)
    torch.cuda.synchronize()
    ms_serial_step = pe0.elapsed_time(pe1) / args.steps
    ktimes = batch.kernel_times()
    batch.profile(False)
    batch.tune(contexts=args.contexts or 3)

    roofline = make_roofline(args, info, stats, ktimes, ms_step, ms_serial_step, S, n, n_out, clocks)

    # ---- end to end through the host-buffer entry point ----
    e2e = None
    if not args.no_e2e:
        # int16 PCM rows: the reference CLI's own I/O format (16-bit WAV in, 16-bit WAV out, main/main.cc:136)
        q_in, q_out = host_array(np.int16, (S, stride)), host_array(np.int16, (S, out_stride))
        q_in[:] = torch.round(d_in * 32768.0).clamp_(-32768, 32767).to(torch.int16).cpu().numpy()
        dt_ms, st = time_host(batch, q_in, q_out, A.S16, args.steps)
        e2e = {"value": audio_sec_per_step / (dt_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": st["h2d_bytes"] * world,
               "d2h_bytes_per_step": st["d2h_bytes"] * world, "ms_per_step": dt_ms,
               "format": "int16 PCM rows in, int16 PCM rows out (the reference CLI's WAV sample format), page-locked host memory",
               "host_alloc": args.host_alloc, "result_checksum": float(np.abs(q_out[:, :n_out_min].astype(np.float64)).mean() / 32768.0)}
        if parity is not None:
            parity["e2e_s16"] = parity_s16([q_out[s * CHANNELS:(s + 1) * CHANNELS, :int(n_out[s])].copy() for s in pr], refs)
        del q_in, q_out
        for hb in host_bufs:
            if hasattr(hb, "close"):
                hb.close()
        host_bufs.clear()
        # float32 rows beside it (twice the bytes per sample)
        h_in, h_out = host_array(np.float32, (S, stride)), host_array(np.float32, (S, out_stride))
        h_in[:] = d_in.cpu().numpy()
        dt_ms, st = time_host(batch, h_in, h_out, A.F32, args.steps)
        e2e["f32"] = {"value": audio_sec_per_step / (dt_ms / 1e3), "unit": UNIT, "h2d_bytes_per_step": st["h2d_bytes"] * world,
                      "d2h_bytes_per_step": st["d2h_bytes"] * world, "ms_per_step": dt_ms,
                      "format": "float32 rows in, float32 rows out, page-locked host memory",
                      "result_checksum": float(np.abs(h_out[:, :n_out_min].astype(np.float64)).mean())}
        if parity is not None:
            parity["e2e_f32"] = parity_f32([h_out[s * CHANNELS:(s + 1) * CHANNELS, :int(n_out[s])].copy() for s in pr], refs)
        del h_in, h_out
        for hb in host_bufs:
            if hasattr(hb, "close"):
                hb.close()
        host_bufs.clear()
    if parity is not None and world > 1:     # every rank checked its own rows: fold to the worst
        for leg in [k for k in parity if isinstance(parity[k], dict)]:
            d = parity[leg]
            d["counts_equal"] = bool(reduce(1.0 if d["counts_equal"] else 0.0, dist.ReduceOp.MIN) > 0.5)
            d["max_abs"] = reduce(d["max_abs"], dist.ReduceOp.MAX)
            d["min_snr_db"] = reduce(d["min_snr_db"] if d["min_snr_db"] is not None else 1e9, dist.ReduceOp.MIN)
            d["rows"] = int(reduce(float(d["rows"]), dist.ReduceOp.SUM))
        parity["ranks"] = world

    # ---- strong scaling: the literal configs[3], 4096 streams IN TOTAL sharded over the N GPUs ----
    strong = None
    if world > 1 and not args.no_strong:
        batch.close()
        del d_in, d_out
        torch.cuda.empty_cache()
        per = [len(range(*_block(args.streams, world, r))) for r in range(world)]
        b2, i2, o2, st2, ost2, no2 = make_batch(per[rank])
        ms2 = time_device(b2, i2, o2, st2, ost2, args.steps, args.warmup)
        strong = {"scaling": "strong", "total_streams": args.streams, "streams_per_gpu": per, "ms_per_step": ms2,
                  "value": args.streams * args.secs / (ms2 / 1e3), "unit": UNIT}
        if not args.no_e2e:
            S2 = per[rank] * CHANNELS
            q_in, q_out = host_array(np.int16, (S2, st2)), host_array(np.int16, (S2, ost2))
            q_in[:] = torch.round(i2 * 32768.0).clamp_(-32768, 32767).to(torch.int16).cpu().numpy()
            dt_ms, _ = time_host(b2, q_in, q_out, A.S16, args.steps)
            strong["e2e"] = {"value": args.streams * args.secs / (dt_ms / 1e3), "unit": UNIT, "ms_per_step": dt_ms, "format": "int16 PCM rows"}
            del q_in, q_out
        b2.close()
    else:
        batch.close()

    latency = None
    cpu = None
    if rank == 0 and world == 1:
        if not args.no_latency:
            latency = stream_latency()
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            ncpu = max(cores, cores * args.cpu_streams_per_core)
            v, kind, dt = cpu_run(ncpu, args.secs, cores)
            cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                   "sample": f"{ncpu} streams of the same workload ({args.secs:g} s each, float32 sample files through oracle/_ref/pvref_drv = the "
                             f"unmodified reference library driven with audiomod-exe's block protocol; no WAV parsing), one OS process per stream, {dt:.1f} s wall"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": workload_config(args, world), "clocks": clocks, "e2e": e2e,
                "gpu_launches": stats["kernel_launches"] * args.steps, "roofline": roofline, "cpu_baseline": cpu,
                "parity": parity, "strong_scaling": strong, "stream_latency_ms": latency, "result_checksum": checksum,
                "value_definition": "inputs resident in HBM when the timed region starts (bench contract); e2e.value is the SURVEY 8(d) metric "
                                    "with H2D + kernels + D2H inside the timed region"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS, DUMP_BYTES = 16, 48 << 20


def dump_outputs(out_dir, torch, d_out, n_out, n_streams):
    """Write what the last timed step left in d_out, so that two builds can be compared output for output (the inputs are
    seeded: the same arguments give the same inputs).  Every stream's output length and, per channel, the float64 sum and sum
    of squares over all its samples; and the samples themselves of a fixed, seeded choice of streams -- at most DUMP_ROWS, as
    many as fit in DUMP_BYTES, cut to that size if one stream alone is larger.  Samples past a stream's length are zero."""
    os.makedirs(out_dir, exist_ok=True)
    n_out = np.asarray(n_out, dtype=np.int64)
    width = int(n_out.max())
    lengths = torch.as_tensor(np.repeat(n_out, CHANNELS), device=d_out.device)
    col = torch.arange(width, device=d_out.device)
    sums, sumsq = [], []
    for r0 in range(0, d_out.shape[0], 64):
        blk = d_out[r0:r0 + 64, :width].double()
        blk *= col[None, :] < lengths[r0:r0 + 64, None]
        sums.append(blk.sum(1))
        sumsq.append((blk * blk).sum(1))
        del blk
    k = max(1, min(DUMP_ROWS, n_streams, DUMP_BYTES // (4 * CHANNELS * width)))
    cols = min(width, DUMP_BYTES // (4 * CHANNELS * k))
    pick = np.sort(np.random.default_rng(0).choice(n_streams, k, replace=False))
    rows = torch.as_tensor((pick[:, None] * CHANNELS + np.arange(CHANNELS)[None, :]).reshape(-1), device=d_out.device)
    sample = d_out[:, :cols].index_select(0, rows).cpu().numpy().reshape(k, CHANNELS, cols)
    for i, s in enumerate(pick):
        sample[i, :, n_out[s]:] = 0.0
    out = {"output_rows": sample, "output_row_streams": pick.astype(np.float64),
           "output_lengths": n_out.astype(np.float64),
           "output_row_sums": torch.cat(sums).cpu().numpy().reshape(n_streams, CHANNELS),
           "output_row_sumsq": torch.cat(sumsq).cpu().numpy().reshape(n_streams, CHANNELS)}
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _block(n, world, rank):
    base, extra = divmod(n, world)
    start = rank * base + min(rank, extra)
    return start, start + base + (1 if rank < extra else 0)


def make_roofline(args, info, stats, ktimes, ms_step, ms_serial_step, S, n, n_out, clocks):
    """Roofline numbers of the step (DESIGN.md section 5).  `frac` is the HBM fraction of the dominant kernel on the staged-
    traffic model; the binding resource of this path is not DRAM but instruction issue / the L1 data pipe, so the line also
    carries issue_frac (warp instructions per frame from the committed ncu capture) and fp32_frac (SURVEY 8(d)(ii))."""
    N, hop, H, half = info["fftsize"], info["hop"], info["bins"], info["fftsize"] // 2
    slices = stats["slices"]
    shift = hop * info["hs_ratio"]
    P = half / 5.0     # peaks per frame of a noise-like spectrum (strict +-2 local maxima), measured on the synthetic workload
    per_frame = {"analyse": 4 * (hop + 2 * H), "phase_core": 4 * (2 * H + half), "synthesise": 4 * (2 * H + N),
                 "ola_resample": 4 * (N + shift / info["pitch_scale"]), "fixed_phase": 4 * H,
                 "lock_peaks": 4 * 2 * H * (1 + 1.0 / 32) + 16 * P + 2 * half + 8, "lock_chain": 16 * P + 8 + 8 * P,
                 # fused inverse FFT + overlap-add + resampler: spectrum, bin->region map, rotations in; PCM out; OLA tail per chunk
                 "synth_ola": 4 * 2 * H + 2 * half + 8 * P + 8 + 4 * shift / info["pitch_scale"] + 2 * 4 * N / 64.0}
    if ktimes.get("lock_chain", (0, 0))[1] > 0 and ktimes.get("synthesise", (0, 0))[1] > 0:
        per_frame["synthesise"] = 4 * (2 * H + N) + 2 * half + 8 * P + 8
    live = [k for k in per_frame if ktimes.get(k, (0, 0))[1] > 0]
    dom = max(live, key=lambda k: ktimes[k][0])
    dom_ms, dom_launches = ktimes[dom]
    bytes_total = per_frame[dom] * slices * S * args.steps
    achieved = bytes_total / (dom_ms / 1e3) / 1e9
    peak, peak_src = 6650.0, "fallback"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak, peak_src = float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        pass
    prof = {}
    try:   # per-kernel counters of the committed ncu --set full capture (scripts/profile_digest.py)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            prof = json.load(f)
    except Exception:
        pass
    traffic = prof.get(dom, {}).get("dram_bytes_per_frame")
    traffic = traffic * slices * S * args.steps / max(dom_launches, 1) if traffic is not None else None
    kernel_ms_sum = sum(v[0] for v in ktimes.values())
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    frames_per_step = slices * S
    instr = {k: prof.get(k, {}).get("warp_instr_per_frame") for k in live}
    issue_frac = None
    if all(v is not None for v in instr.values()) and instr:
        issue_frac = sum(instr.values()) * frames_per_step / (148 * 4 * sm_mhz * 1e6) / (ms_step / 1e3)
    in_samples_per_s = S * n / (ms_step / 1e3)
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6
    return {"bound": prof.get(dom, {}).get("limiter", "issue slots / L1 data pipe (not DRAM): see issue_frac"), "kernel": dom,
            "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "peak_source": peak_src, "bytes_per_launch": bytes_total / max(dom_launches, 1),
            "avg_launch_ms": dom_ms / max(dom_launches, 1),
            "kernel_share_of_step": dom_ms / max(kernel_ms_sum, 1e-9),
            "kernel_ms_per_step": {k: v[0] / args.steps for k, v in ktimes.items() if v[1]},
            "serialised_ms_per_step": ms_serial_step,
            "staged_bytes_per_frame": {k: per_frame[k] for k in live},
            "step_hbm_frac_staged": sum(per_frame[k] for k in live) * frames_per_step / (ms_step / 1e3) / 1e9 / peak,
            "compulsory_io_frac": (4.0 * (n + float(n_out.max())) * S) / (ms_step / 1e3) / 1e9 / peak,
            "issue_frac": issue_frac, "warp_instr_per_frame": instr,
            "issue_frac_definition": "sum over kernels of warp instructions per frame (committed ncu capture, profiles/traffic.json) x frames per step / "
                                     "(148 SMs x 4 schedulers x sm_mhz) / step time",
            "fp32_frac": 2200.0 * in_samples_per_s / fp32_peak,
            "fp32_frac_definition": "2.2 kflop per input sample (SURVEY 8(d)) x input samples/s / (148 x 128 lanes x 2 x sm_mhz)"}


if __name__ == "__main__":
    main()
