"""ctypes wrapper around oracle/libpv_oracle.so and the compiled reference (oracle/_ref).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; never from audiomod_b200/ (the product).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libpv_oracle.so")
REF_DIR = os.path.join(HERE, "_ref")
REF_DRV = os.path.join(REF_DIR, "pvref_drv")
REF_EXE = os.path.join(REF_DIR, "audiomod-exe")
REF_FX = os.path.join(REF_DIR, "fxref_drv")             # the reference's gain / compressor / limiter objects over a float32 file
REF_DRV_CEP = os.path.join(REF_DIR, "pvref_drv_cep")   # the reference with its commented-out cepstral routine switched on

# mode constants of the reference (include/dafx/phasevocoder.h:22-30)
CONSTANT, NORMAL_SHIFT, GENDER_CHANGE, FORMANT_PRESERVE = -1, 0, 1, 2
VOCODER_ROSENBERG, VOCODER_CHORD, NORMAL_STRETCH, ROBOTIC, WHISPER = 3, 4, 5, 6, 7

_lib = None
_fp = C.POINTER(C.c_float)
_fpp = C.POINTER(_fp)


def build(force: bool = False) -> None:
    """Compile the C restatement (and oracle/_ref when /root/reference is present)."""
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(os.path.join(HERE, "pv_oracle.c")):
        subprocess.check_call(["make", "-s", "-C", HERE, "oracle"])
    if os.path.exists("/root/reference/CMakeLists.txt") and (force or not os.path.exists(REF_DRV)):
        subprocess.check_call(["make", "-s", "-j8", "-C", HERE, "ref"])


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        L.pvo_create.restype = C.c_void_p
        L.pvo_create.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int]
        L.pvo_destroy.argtypes = [C.c_void_p]
        L.pvo_process.argtypes = [C.c_void_p, _fpp, C.c_int]
        L.pvo_available.argtypes = [C.c_void_p]
        L.pvo_retrieve.argtypes = [C.c_void_p, _fpp, C.c_int]
        L.pvo_process_block.argtypes = [C.c_void_p, _fpp, C.c_int]
        L.pvo_fftsize.argtypes = [C.c_void_p]
        L.pvo_hop.argtypes = [C.c_void_p]
        L.pvo_pitch_scale.argtypes = [C.c_void_p]
        L.pvo_pitch_scale.restype = C.c_float
        L.pvo_slices.argtypes = [C.c_void_p]
        L.pvo_slices.restype = C.c_long
        L.pvo_dropped.argtypes = [C.c_void_p]
        L.pvo_dropped.restype = C.c_long
        L.pvo_run_offline.restype = C.c_long
        L.pvo_run_offline.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_int, C.c_int,
                                      _fp, C.c_long, _fp, C.c_long, C.c_int, C.POINTER(C.c_long)]
        L.pvo_forward_polar.argtypes = [C.c_int, _fp, _fp, _fp, _fp]
        L.pvo_inverse_polar.argtypes = [C.c_int, _fp, _fp, _fp]
        L.pvo_polar.argtypes = [C.c_long, _fp, _fp, _fp]
        _ip = C.POINTER(C.c_int)
        L.pvo_phase_core_frames.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _ip, _fp, _fp, C.c_int,
                                            _ip, _ip, _ip, _fp, _ip, _ip, _fp]
        L.pvo_host_atan2f.restype = C.c_float
        L.pvo_host_atan2f.argtypes = [C.c_float, C.c_float]
        L.pvo_host_atan2f_vec.argtypes = [_fp, _fp, _fp, C.c_long]
        L.pvo_princarg.restype = C.c_double
        L.pvo_princarg.argtypes = [C.c_double]
        L.pvo_hann.restype = C.c_float
        L.pvo_hann.argtypes = [C.c_int, _fp]
        L.pvo_rand_sequence.argtypes = [C.POINTER(C.c_int), C.c_int]
        L.pvo_host_rand.restype = C.c_int
        L.pvo_resampler_params.argtypes = [C.c_float, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                           C.POINTER(C.c_uint32), C.POINTER(C.c_int), _fp, C.c_int]
        _lib = L
    return _lib


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(_fp)


def _chan_ptrs(a: np.ndarray):
    arr = (_fp * a.shape[0])()
    for c in range(a.shape[0]):
        arr[c] = a[c].ctypes.data_as(_fp)
    return arr


def run_offline(x: np.ndarray, sr: int, timeratio: float = 1.0, semitones: float = 0.0, mode: int = NORMAL_SHIFT,
                coremode: int = 1, fftsize: int = 2048, hopsize: int = 0, block: int = 0, return_slices: bool = False):
    """Whole-stream run of the restatement with the reference CLI's block protocol.
    x: float32 [ch, n].  Returns float32 [ch, n_out]."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    ch, n = x.shape
    cap = int(n * max(1.0, timeratio) * 1.05) + 16 * 8192
    out = np.zeros((ch, cap), dtype=np.float32)
    slices = C.c_long(0)
    k = lib().pvo_run_offline(sr, ch, timeratio, semitones, mode, coremode, fftsize, hopsize,
                              _ptr(x), n, _ptr(out), cap, block, C.byref(slices))
    y = np.ascontiguousarray(out[:, :k])
    return (y, slices.value) if return_slices else y


class OracleStream:
    """Streaming handle on the restatement: the reference's modbase / modbase_offline calls."""

    def __init__(self, sr, ch, timeratio, semitones, mode=NORMAL_SHIFT, coremode=1, fftsize=2048, hopsize=0):
        self.ch = ch
        self.h = lib().pvo_create(sr, ch, timeratio, semitones, mode, coremode, fftsize, hopsize)

    def close(self):
        if self.h:
            lib().pvo_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def processInData(self, x: np.ndarray) -> None:
        x = np.ascontiguousarray(x, dtype=np.float32)
        lib().pvo_process(self.h, _chan_ptrs(x), x.shape[1])

    def getOutSamples(self) -> int:
        return lib().pvo_available(self.h)

    def getOutData(self, n: int) -> np.ndarray:
        out = np.zeros((self.ch, max(n, 1)), dtype=np.float32)
        k = lib().pvo_retrieve(self.h, _chan_ptrs(out), n)
        return out[:, :k]

    def processBlock(self, x: np.ndarray) -> bool:
        """In place on x ([ch, n] float32, C-contiguous); returns outputReady()."""
        assert x.dtype == np.float32 and x.flags.c_contiguous
        return lib().pvo_process_block(self.h, _chan_ptrs(x), x.shape[1]) == 0

    @property
    def hop(self):
        return lib().pvo_hop(self.h)

    @property
    def slices(self):
        return lib().pvo_slices(self.h)


def forward_polar(frame: np.ndarray):
    """Hann * frame -> fftshift -> KissFFT-order real FFT -> (mag, phase, re_im[H,2])."""
    frame = np.ascontiguousarray(frame, dtype=np.float32)
    n = frame.shape[0]
    h = n // 2 + 1
    mag = np.zeros(h, np.float32)
    ph = np.zeros(h, np.float32)
    ri = np.zeros((h, 2), np.float32)
    lib().pvo_forward_polar(n, _ptr(frame), _ptr(mag), _ptr(ph), _ptr(ri))
    return mag, ph, ri


def inverse_polar(mag: np.ndarray, phase: np.ndarray, n: int) -> np.ndarray:
    mag = np.ascontiguousarray(mag, dtype=np.float32)
    phase = np.ascontiguousarray(phase, dtype=np.float32)
    out = np.zeros(n, np.float32)
    lib().pvo_inverse_polar(n, _ptr(mag), _ptr(phase), _ptr(out))
    return out


def polar(re_im: np.ndarray):
    """(re, im) pairs [..., 2] -> (sqrtf(re*re + im*im), atan2f(im, re)) rounded as the reference's forwardPolar."""
    ri = np.ascontiguousarray(re_im, dtype=np.float32)
    mag = np.empty(ri.shape[:-1], np.float32)
    ph = np.empty(ri.shape[:-1], np.float32)
    lib().pvo_polar(mag.size, _ptr(ri), _ptr(mag), _ptr(ph))
    return mag, ph


def phase_core_frames(mag: np.ndarray, phase: np.ndarray, phase_inc, hop: int, coremode: int = 1) -> dict:
    """The reference's phase core (modify_locked / modify_simple / modify_intratio) over the polar frames of one stream,
    mag / phase [ch][n][N/2+1], from fresh-process state, in the reference's channel order.  Returns per (channel, frame):
    branch (0 pass-through, 1 classic, 2 locked, 3 int ratio), npeak, peaks / rot / bin1 / bin2 [ch][n][maxpk] (the first
    npeak entries are valid; rot and bins on locked frames) and out_phase [ch][n][N/2+1]."""
    mag = np.ascontiguousarray(mag, dtype=np.float32)
    phase = np.ascontiguousarray(phase, dtype=np.float32)
    ch, n, h = mag.shape
    N = 2 * (h - 1)
    maxpk = N // 6 + 2
    inc = np.ascontiguousarray(np.broadcast_to(np.asarray(phase_inc, np.int32), (n,)))
    ip = C.POINTER(C.c_int)
    r = dict(branch=np.zeros((ch, n), np.int32), npeak=np.zeros((ch, n), np.int32), peaks=np.zeros((ch, n, maxpk), np.int32),
             rot=np.full((ch, n, maxpk), np.nan, np.float32), bin1=np.zeros((ch, n, maxpk), np.int32),
             bin2=np.zeros((ch, n, maxpk), np.int32), out_phase=np.zeros((ch, n, h), np.float32))
    lib().pvo_phase_core_frames(N, hop, ch, coremode, n, inc.ctypes.data_as(ip), _ptr(mag), _ptr(phase), maxpk,
                                r["branch"].ctypes.data_as(ip), r["npeak"].ctypes.data_as(ip), r["peaks"].ctypes.data_as(ip),
                                _ptr(r["rot"]), r["bin1"].ctypes.data_as(ip), r["bin2"].ctypes.data_as(ip), _ptr(r["out_phase"]))
    return r


def host_atan2f(y: np.ndarray, x: np.ndarray) -> np.ndarray:
    y = np.ascontiguousarray(y, dtype=np.float32)
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.empty_like(y)
    lib().pvo_host_atan2f_vec(_ptr(y), _ptr(x), _ptr(out), y.size)
    return out


def hann(n: int):
    w = np.zeros(n, np.float32)
    area = lib().pvo_hann(n, _ptr(w))
    return w, area


def resampler_params(pitch_scale: float):
    num, den, fl, ov = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
    direct = C.c_int()
    tab = np.zeros(1 << 16, np.float32)
    n = lib().pvo_resampler_params(pitch_scale, C.byref(num), C.byref(den), C.byref(fl), C.byref(ov), C.byref(direct),
                                   _ptr(tab), tab.size)
    return dict(num=num.value, den=den.value, filt_len=fl.value, oversample=ov.value, direct=direct.value, table=tab[:n].copy())


# ---- the compiled, unmodified reference (oracle/_ref) ----
def have_ref() -> bool:
    return os.path.exists(REF_DRV) and os.access(REF_DRV, os.X_OK)


def have_ref_cepstral() -> bool:
    return os.path.exists(REF_DRV_CEP) and os.access(REF_DRV_CEP, os.X_OK)


def run_ref(x: np.ndarray, sr: int, timeratio: float = 1.0, semitones: float = 0.0, mode: int = NORMAL_SHIFT,
            coremode: int = 1, fftsize: int = 2048, block: int = 0, protocol: str = "offline", cepstral: bool = False) -> np.ndarray:
    """Run the unmodified reference library in its own OS process (fresh statics).  cepstral=True: the variant whose gender /
    formant modes (1 / 2) call formantShiftSlice (oracle/Makefile, pvref_drv_cep)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    ch = x.shape[0]
    with tempfile.TemporaryDirectory(prefix="pvref_") as d:
        fi, fo = os.path.join(d, "i.f32"), os.path.join(d, "o.f32")
        x.tofile(fi)
        subprocess.check_call([REF_DRV_CEP if cepstral else REF_DRV, str(sr), str(ch), repr(float(timeratio)), repr(float(semitones)), str(mode),
                               str(coremode), str(fftsize), fi, fo, str(block), protocol])
        y = np.fromfile(fo, dtype=np.float32)
    return y.reshape(ch, -1)


def have_ref_fx() -> bool:
    return os.path.exists(REF_FX) and os.access(REF_FX, os.X_OK)


def run_ref_fx(x: np.ndarray, sr: int, chain) -> np.ndarray:
    """chain: list of ("gain", g) / ("compressor", thr, ratio, makeup, att, rel) / ("limiter", thr, makeup, att, rel) /
    ("biquad", type, cutoff, q, gain) / ("equalizer",) (defaults) / ("equalizer", p0 .. p31), applied in order by the unmodified
    reference's objects (blocks of 480 samples, in place)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    ch = x.shape[0]
    args = []
    for fx in chain:
        if fx[0] == "equalizer" and len(fx) == 1:
            args += ["equalizer", "default"]
        else:
            args += [fx[0]] + [repr(float(v)) for v in fx[1:]]
    with tempfile.TemporaryDirectory(prefix="fxref_") as d:
        fi, fo = os.path.join(d, "i.f32"), os.path.join(d, "o.f32")
        x.tofile(fi)
        subprocess.check_call([REF_FX, str(sr), str(ch), fi, fo] + args)
        y = np.fromfile(fo, dtype=np.float32)
    return y.reshape(ch, -1)
