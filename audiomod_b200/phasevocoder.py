"""Host-side mirror of the reference's phase-vocoder interface over the C ABI.

`phasevocoder` mirrors audiomod::phasevocoder (include/dafx/phasevocoder.h:54-80 of the reference:
same constructor arguments, processInData / getOutSamples / getOutData of modbase_offline and
processBlock / outputReady of modbase, include/dafx/modbase.h:43-114).  `PhaseVocoderBatch` is the
throughput entry point: many independent streams, each processed exactly like one fresh
`audiomod-exe` run (main/main.cc:149,471-509).  All arithmetic happens in libpvgpu.so on the GPU.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import Config, Info, check

# mode / coremode constants, include/dafx/phasevocoder.h:22-36
CONSTANT, NORMAL_SHIFT, GENDER_CHANGE, FORMANT_PRESERVE = -1, 0, 1, 2
VOCODER_ROSENBERG, VOCODER_CHORD, NORMAL_STRETCH, ROBOTIC, WHISPER = 3, 4, 5, 6, 7
# extensions (include/pvgpu.h): the reference's commented-out cepstral envelope routine instead of the nearest-bin warp
GENDER_CEPSTRAL, FORMANT_CEPSTRAL = 8, 9
NORMAL_PV, PHASE_LOCKED, INT_RATIO = 0, 1, 2

_fp = C.POINTER(C.c_float)
_sp = C.POINTER(C.c_int16)


def _cfg(sampleRate, numChannels, timeratio, pitchshift, mode, coremode, fftsize, hopsize, device) -> Config:
    return Config(int(sampleRate), int(numChannels), float(timeratio), float(pitchshift), int(mode), int(coremode),
                  int(fftsize), int(hopsize), int(device))


def _info_dict(info: Info) -> dict:
    return {k: getattr(info, k) for k, _ in Info._fields_}


def describe(sampleRate, numChannels, timeratio, pitchshift, mode=NORMAL_SHIFT, coremode=PHASE_LOCKED, fftsize=2048,
             hopsize=0) -> dict:
    """Sizes the reference derives in Impl::calculateSizes (needs no GPU)."""
    info = Info()
    check(_lib.lib().pvgpu_describe(C.byref(_cfg(sampleRate, numChannels, timeratio, pitchshift, mode, coremode, fftsize,
                                                  hopsize, 0)), C.byref(info)))
    return _info_dict(info)


def plan_counts(n_in, sampleRate, numChannels, timeratio, pitchshift, mode=NORMAL_SHIFT, coremode=PHASE_LOCKED, fftsize=2048,
                hopsize=0, block=0) -> dict:
    """Host-only dry run of one stream through the CLI block protocol: output length, slices, dropped slices."""
    v = [C.c_int64() for _ in range(3)]
    check(_lib.lib().pvgpu_plan_counts(C.byref(_cfg(sampleRate, numChannels, timeratio, pitchshift, mode, coremode, fftsize,
                                                     hopsize, 0)), int(n_in), int(block), *[C.byref(x) for x in v]))
    return dict(n_out=v[0].value, n_slices=v[1].value, n_dropped=v[2].value)


def _chan_ptrs(a: np.ndarray, elem=_fp):
    """float** (int16_t** with elem=_sp) for the rows of a 2-D array (vectorised: a live batch has thousands of rows per call)."""
    ptrs = (np.uintp(a.ctypes.data) + np.arange(a.shape[0], dtype=np.uintp) * np.uintp(a.strides[0])).astype(np.uintp)
    return ptrs.ctypes.data_as(C.POINTER(elem))   # keeps a reference to `ptrs`


def _fx_array(chain):
    """(pvgpu_fx array, count) of a chain spelled as (kind name, constructor arguments...) tuples."""
    kinds = {"gain": _lib.FX_GAIN, "compressor": _lib.FX_COMPRESSOR, "limiter": _lib.FX_LIMITER, "biquad": _lib.FX_BIQUAD}
    arr = (_lib.Fx * max(len(chain), 1))()
    for i, fx in enumerate(chain):
        arr[i].kind = kinds[fx[0]]
        for j, v in enumerate(fx[1:]):
            arr[i].p[j] = float(v)
    return arr, len(chain)


class phasevocoder:
    """One stream.  Buffers are planar float32 arrays of shape [numChannels, n].

    streams > 1 makes it a live batch (pvgpu_create_multi): `streams` objects of one configuration advancing in lock-step,
    buffers [streams * numChannels, n] with row = stream * numChannels + channel; every call serves all of them with one set
    of kernel launches, and every stream gets the samples its own object would.

    fmt=S16 makes every buffer int16 PCM (the pvgpu_*_s16 calls): processInData / processBlock take int16 arrays (other dtypes
    are rejected, not cast), getOutData returns int16, and the *Device methods take int16 device rows with pointer offsets and
    pitches in int16 elements.  The samples are those of a float32 object fed s / 32768 whose output is quantised the way the
    reference's WAV writer does."""

    def __init__(self, sampleRate, numChannels, timeratio, pitchshift, mode=NORMAL_SHIFT, coremode=PHASE_LOCKED,
                 fftsize=2048, hopsize=0, device=0, streams=1, fmt=_lib.F32):
        self._h = C.c_void_p()
        if fmt not in (_lib.F32, _lib.S16):
            raise ValueError(f"fmt must be F32 or S16, not {fmt!r}")
        self.fmt = fmt
        s16 = fmt == _lib.S16
        L = _lib.lib()
        self._dtype, self._elem = (np.int16, _sp) if s16 else (np.float32, _fp)
        self._process, self._retrieve, self._block = ((L.pvgpu_process_s16, L.pvgpu_retrieve_s16, L.pvgpu_process_block_s16) if s16
                                                      else (L.pvgpu_process, L.pvgpu_retrieve, L.pvgpu_process_block))
        self._process_dev, self._retrieve_dev, self._block_dev = (
            (L.pvgpu_process_device_s16, L.pvgpu_retrieve_device_s16, L.pvgpu_process_block_device_s16) if s16
            else (L.pvgpu_process_device, L.pvgpu_retrieve_device, L.pvgpu_process_block_device))
        self.streams_ = int(streams)
        self.num_channels_ = int(numChannels) * self.streams_    # rows of every buffer
        self._ready = False
        cfg = _cfg(sampleRate, numChannels, timeratio, pitchshift, mode, coremode, fftsize, hopsize, device)
        if self.streams_ == 1:
            check(_lib.lib().pvgpu_create(C.byref(cfg), C.byref(self._h)))
        else:
            check(_lib.lib().pvgpu_create_multi(C.byref(cfg), self.streams_, C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pvgpu_destroy(self._h)
            self._h = None

    __del__ = close

    def setParams(self, params):  # empty in the reference (phasevocoder.h:62-72)
        pass

    def getParams(self, params):
        pass

    def _check_dtype(self, a) -> None:
        if self.fmt == _lib.S16 and np.asarray(a).dtype != np.int16:
            raise TypeError(f"this instance takes int16 rows, not {np.asarray(a).dtype}")

    def processInData(self, inData: np.ndarray, num_in_samples: int | None = None) -> None:
        self._check_dtype(inData)
        x = np.ascontiguousarray(inData, dtype=self._dtype)
        n = x.shape[1] if num_in_samples is None else int(num_in_samples)
        check(self._process(self._h, _chan_ptrs(x, self._elem), n))

    def getOutSamples(self) -> int:
        return _lib.lib().pvgpu_available(self._h)

    def getOutData(self, num_out_samples: int) -> np.ndarray:
        out = np.zeros((self.num_channels_, max(int(num_out_samples), 1)), dtype=self._dtype)
        k = self._retrieve(self._h, _chan_ptrs(out, self._elem), int(num_out_samples))
        if k < 0:
            check(-k)
        self._ready = True
        return out[:, :k]

    def processBlock(self, bufferData: np.ndarray, num_samples: int | None = None) -> None:
        """In place on a C-contiguous float32 (fmt=S16: int16) [numChannels, n] array."""
        self._check_dtype(bufferData)
        assert bufferData.dtype == self._dtype and bufferData.flags.c_contiguous
        n = bufferData.shape[1] if num_samples is None else int(num_samples)
        ready = C.c_int(0)
        check(self._block(self._h, _chan_ptrs(bufferData, self._elem), n, C.byref(ready)))
        self._ready = bool(ready.value)

    # ---- device rows: float32 (fmt=S16: int16) device memory, row r at ptr + r * pitch elements; enqueued on cuda_stream, no
    # call waits ----
    def processInDataDevice(self, d_ptr: int, pitch: int, n: int, cuda_stream: int = 0) -> None:
        check(self._process_dev(self._h, C.c_void_p(d_ptr), int(pitch), int(n), C.c_void_p(cuda_stream)))

    def getOutDataDevice(self, d_ptr: int, pitch: int, n: int, cuda_stream: int = 0) -> int:
        k = self._retrieve_dev(self._h, C.c_void_p(d_ptr), int(pitch), int(n), C.c_void_p(cuda_stream))
        if k < 0:
            check(-k)
        return k

    def processBlockDevice(self, d_ptr: int, pitch: int, n: int, cuda_stream: int = 0) -> None:
        ready = C.c_int(0)
        check(self._block_dev(self._h, C.c_void_p(d_ptr), int(pitch), int(n), C.c_void_p(cuda_stream), C.byref(ready)))
        self._ready = bool(ready.value)

    def outputReady(self) -> bool:
        return self._ready

    def info(self) -> dict:
        info = Info()
        check(_lib.lib().pvgpu_stream_info(self._h, C.byref(info)))
        return _info_dict(info)

    def set_postchain(self, chain):
        """FFT-free effects on everything this instance outputs, in order (pvgpu_set_postchain): the chains of
        PhaseVocoderBatch.set_postchain, spelled the same way.  Every output sample goes through the chain once before it
        enters the output ring, with each effect's state carried per row from call to call -- what the reference's effect objects
        compute when fed everything getOutData returns.  A live batch applies the chain to every stream; fmt=S16 instances
        quantise the chained float samples.  A new chain starts from fresh effect state at the next call; samples already
        waiting in the ring keep their values.  An empty list clears the chain."""
        arr, n = _fx_array(chain)
        check(_lib.lib().pvgpu_set_postchain(self._h, arr, n))

    def set_stream_postchain(self, stream, chain):
        """Parameters of one stream's chain (pvgpu_set_stream_postchain), spelled as in set_postchain: the same number and kinds of
        effects as the instance's chain, other arguments.  Output produced by later calls uses them; the stream's effect state
        carries over and other streams are untouched.  No device work: safe between real-time calls."""
        arr, n = _fx_array(chain)
        check(_lib.lib().pvgpu_set_stream_postchain(self._h, int(stream), arr, n))

    def set_meters(self, enable=True):
        """Loudness meters on everything this instance outputs, after the post-chain (pvgpu_set_meters): BS.1770-4 momentary
        (400 ms) and short-term (3 s) loudness per stream, ungated, and the sample peak per row.  True starts from fresh state
        (also when already on); False stops them.  Waits for the device: not for the real-time thread."""
        check(_lib.lib().pvgpu_set_meters(self._h, int(bool(enable))))

    def meters(self) -> dict:
        """Host rows: {"momentary": float32 [streams], "short_term": float32 [streams], "peak": float32 [streams, channels],
        "measured": samples per row measured}, as of the last call (pvgpu_get_meters: no device work)."""
        S, ch = self.streams_, self.num_channels_ // self.streams_
        m, s, p = np.empty(S, np.float32), np.empty(S, np.float32), np.empty((S, ch), np.float32)
        n = C.c_int64()
        check(_lib.lib().pvgpu_get_meters(self._h, m.ctypes.data_as(_fp), s.ctypes.data_as(_fp), p.ctypes.data_as(_fp), C.byref(n)))
        return {"momentary": m, "short_term": s, "peak": p, "measured": n.value}

    def metersDevice(self, d_ptr: int, cuda_stream: int = 0) -> int:
        """Device rows: enqueue the copy of [momentary S][short-term S][peak S * channels] float32 to d_ptr on cuda_stream
        (pvgpu_get_meters_device, no wait); returns the samples per row measured."""
        n = C.c_int64()
        check(_lib.lib().pvgpu_get_meters_device(self._h, C.c_void_p(d_ptr), C.c_void_p(cuda_stream), C.byref(n)))
        return n.value


class PhaseVocoderBatch:
    """n_streams independent streams with one configuration (rows are channel-planar)."""

    def __init__(self, n_streams, max_in_samples, sampleRate, numChannels, timeratio, pitchshift, mode=NORMAL_SHIFT,
                 coremode=PHASE_LOCKED, fftsize=2048, hopsize=0, device=0):
        self._h = C.c_void_p()
        self.n_streams, self.channels = int(n_streams), int(numChannels)
        self.n_in = self.n_out = None
        check(_lib.lib().pvgpu_batch_create(C.byref(_cfg(sampleRate, numChannels, timeratio, pitchshift, mode, coremode,
                                                          fftsize, hopsize, device)), self.n_streams, int(max_in_samples),
                                            C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pvgpu_batch_destroy(self._h)
            self._h = None

    __del__ = close

    def info(self) -> dict:
        info = Info()
        check(_lib.lib().pvgpu_batch_info(self._h, C.byref(info)))
        return _info_dict(info)

    def tune(self, frames_per_chunk=0, rows_per_group=0, contexts=0):
        check(_lib.lib().pvgpu_batch_tune(self._h, int(frames_per_chunk), int(rows_per_group), int(contexts)))

    def plan(self, n_in, block: int = 0) -> np.ndarray:
        n_in = np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, dtype=np.int64), (self.n_streams,)))
        n_out = np.zeros(self.n_streams, dtype=np.int64)
        p = C.POINTER(C.c_int64)
        check(_lib.lib().pvgpu_batch_plan(self._h, n_in.ctypes.data_as(p), int(block), n_out.ctypes.data_as(p)))
        self.n_in, self.n_out = n_in, n_out
        return n_out

    def run_device(self, d_in_ptr: int, in_stride: int, d_out_ptr: int, out_stride: int, cuda_stream: int = 0, fmt=_lib.F32):
        """Enqueue one run on the caller's CUDA stream (0 = the legacy default stream); never blocks the host."""
        check(_lib.lib().pvgpu_batch_run_device(self._h, C.c_void_p(d_in_ptr), int(in_stride), C.c_void_p(d_out_ptr),
                                                int(out_stride), fmt, C.c_void_p(cuda_stream)))

    def synchronize(self):
        """Wait for the last run_device."""
        check(_lib.lib().pvgpu_batch_synchronize(self._h))

    def run_host_rows(self, in_rows, out_rows, fmt=_lib.F32):
        """in_rows / out_rows: lists of numpy arrays (or raw addresses), one per channel row."""
        n = self.n_streams * self.channels
        ip, op = (C.c_void_p * n)(), (C.c_void_p * n)()
        for r in range(n):
            ip[r] = in_rows[r] if isinstance(in_rows[r], int) else in_rows[r].ctypes.data
            op[r] = out_rows[r] if isinstance(out_rows[r], int) else out_rows[r].ctypes.data
        check(_lib.lib().pvgpu_batch_run_host(self._h, ip, op, fmt))

    def run(self, streams, fmt=_lib.F32):
        """streams: list of arrays [channels, n_i], float32 (fmt F32) or int16 PCM (fmt S16; converted on the device the
        way the reference's WAV reader / writer does).  Plans for these lengths and returns the outputs in the same format."""
        dt = np.int16 if fmt == _lib.S16 else np.float32
        xs = [np.ascontiguousarray(x, dtype=dt) for x in streams]
        assert len(xs) == self.n_streams and all(x.shape[0] == self.channels for x in xs)
        n_out = self.plan([x.shape[1] for x in xs])
        outs = [np.zeros((self.channels, int(n_out[s])), dtype=dt) for s in range(self.n_streams)]
        in_rows = [xs[s][c] for s in range(self.n_streams) for c in range(self.channels)]
        out_rows = [outs[s][c] for s in range(self.n_streams) for c in range(self.channels)]
        self.run_host_rows(in_rows, out_rows, fmt)
        return outs

    def set_postchain(self, chain):
        """FFT-free effects applied to the float32 output rows, in order (pvgpu_batch_set_postchain; phasevocoder.set_postchain
        takes the same chains for streaming instances): a list of
        ("gain", g), ("compressor", dBThreshold, ratio, dBMakeUpGain, attackMs, releaseMs), ("limiter", dBThreshold, dBMakeUpGain,
        attackMs, releaseMs), ("biquad", type, cutoffFreq, q, dBGain) -- the reference objects' constructor arguments;
        equalizer_chain() expands the equalizer object into biquad entries.  An empty list clears the chain."""
        arr, n = _fx_array(chain)
        check(_lib.lib().pvgpu_batch_set_postchain(self._h, arr, n))

    def set_fused(self, enable=True):
        """True: the fused inverse-FFT + overlap-add + resampler kernel; False: the split kernels; None: automatic (split unless the
        stretch ratio exceeds their table limits).  Bit-identical results in every case."""
        check(_lib.lib().pvgpu_batch_set_fused(self._h, -1 if enable is None else int(bool(enable))))

    KERNEL_KINDS = ("analyse", "phase_core", "synthesise", "ola_resample", "synth_ola", "fixed_phase", "lock_peaks", "lock_chain")

    def profile(self, enable=True):
        check(_lib.lib().pvgpu_batch_profile(self._h, int(bool(enable))))

    def kernel_times(self) -> dict:
        """{kernel kind: (total ms, launches)} since profile(True); synchronises the device."""
        ms = (C.c_double * 8)()
        cnt = (C.c_int64 * 8)()
        check(_lib.lib().pvgpu_batch_kernel_times(self._h, ms, cnt))
        return {k: (ms[i], cnt[i]) for i, k in enumerate(self.KERNEL_KINDS)}

    def stats(self) -> dict:
        v = [C.c_int64() for _ in range(4)]
        check(_lib.lib().pvgpu_batch_stats(self._h, *[C.byref(x) for x in v]))
        return dict(kernel_launches=v[0].value, slices=v[1].value, h2d_bytes=v[2].value, d2h_bytes=v[3].value)


class PhaseVocoderMultiBatch:
    """The same batch sharded across several GPUs of one box inside the library (pvgpu_mbatch_*): one host thread and one
    pvgpu_batch per device, streams partitioned by index, results written straight into the caller's rows."""

    def __init__(self, n_streams, max_in_samples, sampleRate, numChannels, timeratio, pitchshift, mode=NORMAL_SHIFT,
                 coremode=PHASE_LOCKED, fftsize=2048, hopsize=0, devices=None):
        self._h = C.c_void_p()
        self.n_streams, self.channels = int(n_streams), int(numChannels)
        devs = list(devices) if devices is not None else []
        arr = (C.c_int * max(len(devs), 1))(*devs)
        check(_lib.lib().pvgpu_mbatch_create(C.byref(_cfg(sampleRate, numChannels, timeratio, pitchshift, mode, coremode, fftsize,
                                                           hopsize, 0)), self.n_streams, int(max_in_samples),
                                             arr if devs else None, len(devs), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().pvgpu_mbatch_destroy(self._h)
            self._h = None

    __del__ = close

    def plan(self, n_in, block: int = 0) -> np.ndarray:
        n_in = np.ascontiguousarray(np.broadcast_to(np.asarray(n_in, dtype=np.int64), (self.n_streams,)))
        n_out = np.zeros(self.n_streams, dtype=np.int64)
        p = C.POINTER(C.c_int64)
        check(_lib.lib().pvgpu_mbatch_plan(self._h, n_in.ctypes.data_as(p), int(block), n_out.ctypes.data_as(p)))
        self.n_out = n_out
        return n_out

    def owner(self) -> np.ndarray:
        o = np.zeros(self.n_streams, dtype=np.int32)
        check(_lib.lib().pvgpu_mbatch_owner(self._h, o.ctypes.data_as(C.POINTER(C.c_int))))
        return o

    def run_host_rows(self, in_rows, out_rows, fmt=_lib.F32):
        n = self.n_streams * self.channels
        ip, op = (C.c_void_p * n)(), (C.c_void_p * n)()
        for r in range(n):
            ip[r] = in_rows[r] if isinstance(in_rows[r], int) else in_rows[r].ctypes.data
            op[r] = out_rows[r] if isinstance(out_rows[r], int) else out_rows[r].ctypes.data
        check(_lib.lib().pvgpu_mbatch_run_host(self._h, ip, op, fmt))

    def run(self, streams, fmt=_lib.F32):
        dt = np.int16 if fmt == _lib.S16 else np.float32
        xs = [np.ascontiguousarray(x, dtype=dt) for x in streams]
        assert len(xs) == self.n_streams and all(x.shape[0] == self.channels for x in xs)
        n_out = self.plan([x.shape[1] for x in xs])
        outs = [np.zeros((self.channels, int(n_out[s])), dtype=dt) for s in range(self.n_streams)]
        self.run_host_rows([xs[s][c] for s in range(self.n_streams) for c in range(self.channels)],
                           [outs[s][c] for s in range(self.n_streams) for c in range(self.channels)], fmt)
        return outs

    def stats(self) -> dict:
        v = [C.c_int64() for _ in range(3)]
        used = C.c_int()
        check(_lib.lib().pvgpu_mbatch_stats(self._h, *[C.byref(x) for x in v], C.byref(used)))
        return dict(kernel_launches=v[0].value, h2d_bytes=v[1].value, d2h_bytes=v[2].value, devices_used=used.value)


def shard_streams(n_in, n_dev: int) -> np.ndarray:
    """The library's stream -> device partition (needs no GPU): owner index in [0, n_dev) for every stream."""
    n_in = np.ascontiguousarray(np.asarray(n_in, dtype=np.int64))
    owner = np.zeros(n_in.size, dtype=np.int32)
    check(_lib.lib().pvgpu_shard_streams(n_in.ctypes.data_as(C.POINTER(C.c_int64)), int(n_in.size), int(n_dev),
                                         owner.ctypes.data_as(C.POINTER(C.c_int))))
    return owner


class HostBuffer:
    """Page-locked host memory on the NUMA node of a GPU (pvgpu_host_alloc); .array(dtype, shape) views it with numpy."""

    def __init__(self, nbytes: int, device: int = 0, numa_local: bool = True, hugepages: bool = False):
        self.ptr = C.c_void_p()
        self.nbytes = int(nbytes)
        flags = (_lib.HOST_NUMA_LOCAL if numa_local else 0) | (_lib.HOST_HUGEPAGES if hugepages else 0)
        check(_lib.lib().pvgpu_host_alloc(C.byref(self.ptr), self.nbytes, int(device), flags))

    def array(self, dtype, shape) -> np.ndarray:
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        assert n <= self.nbytes
        buf = (C.c_char * n).from_address(self.ptr.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def info(self) -> dict:
        node, huge, nb = C.c_int(), C.c_int(), C.c_size_t()
        check(_lib.lib().pvgpu_host_info(self.ptr, C.byref(node), C.byref(huge), C.byref(nb)))
        return dict(numa_node=node.value, hugepages=bool(huge.value), bytes=nb.value)

    def close(self):
        if getattr(self, "ptr", None) and self.ptr.value:
            _lib.lib().pvgpu_host_free(self.ptr)
            self.ptr = C.c_void_p()

    __del__ = close


def run_wav_files(pairs, timeratio=1.0, pitchshift=0.0, mode=NORMAL_SHIFT, coremode=PHASE_LOCKED, fftsize=2048, hopsize=0, devices=None):
    """File -> file batch: every (in.wav, out.wav) pair is processed like `audiomod-exe <effect> in.wav out.wav ...`
    (pvgpu_run_wav_files).  Returns one dict per file (status, message, sample_rate, channels, bits, frames_in, frames_out)."""
    n = len(pairs)
    jobs = (_lib.WavJob * max(n, 1))()
    keep = []
    for i, (a, b) in enumerate(pairs):
        keep.append((str(a).encode(), str(b).encode()))
        jobs[i].in_path, jobs[i].out_path = keep[-1]
    devs = list(devices) if devices is not None else []
    arr = (C.c_int * max(len(devs), 1))(*devs)
    rc = _lib.lib().pvgpu_run_wav_files(C.byref(_cfg(0, 0, timeratio, pitchshift, mode, coremode, fftsize, hopsize, 0)), jobs, n,
                                        arr if devs else None, len(devs))
    out = [dict(status=jobs[i].status, message=jobs[i].message.decode(errors="replace"), sample_rate=jobs[i].sample_rate,
                channels=jobs[i].channels, bits=jobs[i].bits, frames_in=jobs[i].frames_in, frames_out=jobs[i].frames_out) for i in range(n)]
    if rc != _lib.OK and all(j["status"] == _lib.OK for j in out):
        check(rc)
    return out


def equalizer_chain(paramlist=None):
    """The reference's equalizer object (eight biquad sections, paramlist = [use, cutoff, Q, gain] x 8, None = its defaults)
    as a list of ("biquad", type, cutoff, q, gain) entries for PhaseVocoderBatch.set_postchain and phasevocoder.set_postchain."""
    arr = (_lib.Fx * 8)()
    n = C.c_int()
    pl = None
    if paramlist is not None:
        pl = (C.c_float * 32)(*[float(v) for v in paramlist])
    check(_lib.lib().pvgpu_equalizer_chain(pl, arr, C.byref(n)))
    return [("biquad", int(arr[i].p[0]), arr[i].p[1], arr[i].p[2], arr[i].p[3]) for i in range(n.value)]


def biquad_design(type, sample_rate, cutoff, q, db_gain):
    c = (C.c_float * 6)()
    check(_lib.lib().pvgpu_biquad_design(int(type), int(sample_rate), float(cutoff), float(q), float(db_gain), c))
    return [c[i] for i in range(6)]


def kweighting_design(sample_rate) -> np.ndarray:
    """The meters' K-weighting at this sample rate (pvgpu_kweighting_design, needs no GPU): float64 [shelf b0, b1, b2, a1, a2,
    high-pass a1, a2]; the high-pass has b = (1, -2, 1), both sections a0 = 1."""
    c = np.zeros(7, np.float64)
    check(_lib.lib().pvgpu_kweighting_design(int(sample_rate), c.ctypes.data_as(C.POINTER(C.c_double))))
    return c
