"""ctypes binding of libpvgpu.so (include/pvgpu.h).  The library is the product; there is no Python
or CPU fallback: if it is missing or no CUDA device is usable, calls raise."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpvgpu.so")

OK, EINVAL, ECUDA, ENOMEM, ESTATE = 0, 1, 2, 3, 4
F32, S16 = 0, 1
HOST_NUMA_LOCAL, HOST_HUGEPAGES = 1, 2


class PvgpuError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"pvgpu error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("sample_rate", C.c_int), ("channels", C.c_int), ("time_ratio", C.c_float), ("pitch_semitones", C.c_float),
                ("mode", C.c_int), ("coremode", C.c_int), ("fftsize", C.c_int), ("hopsize", C.c_int), ("device", C.c_int)]


class Info(C.Structure):
    _fields_ = [("fftsize", C.c_int), ("hop", C.c_int), ("bins", C.c_int), ("pitch_scale", C.c_float), ("hs_ratio", C.c_float),
                ("resampler_active", C.c_int), ("resampler_filt_len", C.c_int), ("resampler_num", C.c_uint32),
                ("resampler_den", C.c_uint32), ("outbuf_capacity", C.c_int64)]


class Fx(C.Structure):
    _fields_ = [("kind", C.c_int), ("p", C.c_float * 6)]


FX_GAIN, FX_COMPRESSOR, FX_LIMITER, FX_BIQUAD = 1, 2, 3, 4


class WavJob(C.Structure):
    _fields_ = [("in_path", C.c_char_p), ("out_path", C.c_char_p), ("status", C.c_int), ("sample_rate", C.c_int), ("channels", C.c_int),
                ("bits", C.c_int), ("frames_in", C.c_int64), ("frames_out", C.c_int64), ("message", C.c_char * 160)]


_fp = C.POINTER(C.c_float)
_fpp = C.POINTER(_fp)
_sp = C.POINTER(C.c_int16)
_spp = C.POINTER(_sp)
_vpp = C.POINTER(C.c_void_p)
_i64p = C.POINTER(C.c_int64)

# every symbol include/pvgpu.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "pvgpu_last_error": (C.c_char_p, []),
    "pvgpu_version": (C.c_int, []),
    "pvgpu_device_count": (C.c_int, []),
    "pvgpu_describe": (C.c_int, [C.POINTER(Config), C.POINTER(Info)]),
    "pvgpu_plan_counts": (C.c_int, [C.POINTER(Config), C.c_int64, C.c_int, _i64p, _i64p, _i64p]),
    "pvgpu_create": (C.c_int, [C.POINTER(Config), _vpp]),
    "pvgpu_create_multi": (C.c_int, [C.POINTER(Config), C.c_int, _vpp]),
    "pvgpu_stream_count": (C.c_int, [C.c_void_p]),
    "pvgpu_process_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pvgpu_retrieve_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pvgpu_process_block_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "pvgpu_process_s16": (C.c_int, [C.c_void_p, _spp, C.c_int]),
    "pvgpu_retrieve_s16": (C.c_int, [C.c_void_p, _spp, C.c_int]),
    "pvgpu_process_block_s16": (C.c_int, [C.c_void_p, _spp, C.c_int, C.POINTER(C.c_int)]),
    "pvgpu_process_device_s16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pvgpu_retrieve_device_s16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pvgpu_process_block_device_s16": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "pvgpu_destroy": (None, [C.c_void_p]),
    "pvgpu_process": (C.c_int, [C.c_void_p, _fpp, C.c_int]),
    "pvgpu_available": (C.c_int, [C.c_void_p]),
    "pvgpu_retrieve": (C.c_int, [C.c_void_p, _fpp, C.c_int]),
    "pvgpu_process_block": (C.c_int, [C.c_void_p, _fpp, C.c_int, C.POINTER(C.c_int)]),
    "pvgpu_stream_info": (C.c_int, [C.c_void_p, C.POINTER(Info)]),
    "pvgpu_set_postchain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "pvgpu_set_stream_postchain": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "pvgpu_set_meters": (C.c_int, [C.c_void_p, C.c_int]),
    "pvgpu_get_meters": (C.c_int, [C.c_void_p, _fp, _fp, _fp, _i64p]),
    "pvgpu_get_meters_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, _i64p]),
    "pvgpu_kweighting_design": (C.c_int, [C.c_int, C.POINTER(C.c_double)]),
    "pvgpu_batch_create": (C.c_int, [C.POINTER(Config), C.c_int, C.c_int64, _vpp]),
    "pvgpu_batch_destroy": (None, [C.c_void_p]),
    "pvgpu_batch_plan": (C.c_int, [C.c_void_p, _i64p, C.c_int, _i64p]),
    "pvgpu_batch_run_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pvgpu_batch_synchronize": (C.c_int, [C.c_void_p]),
    "pvgpu_batch_run_host": (C.c_int, [C.c_void_p, _vpp, _vpp, C.c_int]),
    "pvgpu_batch_stats": (C.c_int, [C.c_void_p, _i64p, _i64p, _i64p, _i64p]),
    "pvgpu_batch_info": (C.c_int, [C.c_void_p, C.POINTER(Info)]),
    "pvgpu_batch_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "pvgpu_batch_kernel_times": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), _i64p]),
    "pvgpu_batch_tune": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "pvgpu_batch_set_fused": (C.c_int, [C.c_void_p, C.c_int]),
    "pvgpu_batch_set_postchain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "pvgpu_equalizer_chain": (C.c_int, [_fp, C.c_void_p, C.POINTER(C.c_int)]),
    "pvgpu_biquad_design": (C.c_int, [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, _fp]),
    "pvgpu_run_wav_files": (C.c_int, [C.POINTER(Config), C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_int]),
    "pvgpu_mbatch_create": (C.c_int, [C.POINTER(Config), C.c_int, C.c_int64, C.POINTER(C.c_int), C.c_int, _vpp]),
    "pvgpu_mbatch_destroy": (None, [C.c_void_p]),
    "pvgpu_mbatch_plan": (C.c_int, [C.c_void_p, _i64p, C.c_int, _i64p]),
    "pvgpu_mbatch_run_host": (C.c_int, [C.c_void_p, _vpp, _vpp, C.c_int]),
    "pvgpu_mbatch_stats": (C.c_int, [C.c_void_p, _i64p, _i64p, _i64p, C.POINTER(C.c_int)]),
    "pvgpu_mbatch_owner": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "pvgpu_shard_streams": (C.c_int, [_i64p, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "pvgpu_host_alloc": (C.c_int, [_vpp, C.c_size_t, C.c_int, C.c_int]),
    "pvgpu_host_free": (C.c_int, [C.c_void_p]),
    "pvgpu_host_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "pvgpu_device_numa_node": (C.c_int, [C.c_int]),
    "pvgpu_bind_thread_to_device": (C.c_int, [C.c_int]),
    "pvgpu_test_forward_polar": (C.c_int, [C.c_int, C.c_int, C.c_int, _fp, _fp, _fp]),
    "pvgpu_test_inverse_polar": (C.c_int, [C.c_int, C.c_int, C.c_int, _fp, _fp, _fp]),
    "pvgpu_test_atan2f": (C.c_int, [C.c_int, C.c_int64, _fp, _fp, _fp]),
    "pvgpu_test_princarg": (C.c_int, [C.c_int, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "pvgpu_test_postchain": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int64, _fp]),
    "pvgpu_test_loudness": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _fp, _fp, _fp, _fp]),
    "pvgpu_test_host_structs": (C.c_int, []),
}

_lib = None


def lib() -> C.CDLL:
    """Load libpvgpu.so; raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PvgpuError(ECUDA, f"{LIB_PATH} is missing: build it with `make -C audiomod_b200/csrc` "
                                    "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != OK:
        raise PvgpuError(rc, lib().pvgpu_last_error().decode(errors="replace"))
