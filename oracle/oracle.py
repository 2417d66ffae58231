"""ctypes front-end of the CPU oracle (oracle/mmw_oracle.c) and of the reference's
own CPU functions (oracle/_ref/libref_cpu.so, built from /root/reference by
oracle/Makefile where that tree exists).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs — never by the product package.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "_build", "libmmw_oracle.so")
REF_SO = os.path.join(HERE, "_ref", "libref_cpu.so")
REF_BIN = os.path.join(HERE, "_ref", "ref_acceleration")

DET_DTYPE = np.dtype(
    [
        ("frame", "<u4"),
        ("range_bin", "<u2"),
        ("doppler_bin", "<u2"),
        ("power", "<f4"),
        ("noise", "<f4"),
        ("angle_bin", "<i2"),
        ("flags", "<u2"),
        ("angle_rad", "<f4"),
    ]
)
assert DET_DTYPE.itemsize == 24


class CfarParams(C.Structure):
    _fields_ = [
        ("guard_r", C.c_int),
        ("guard_d", C.c_int),
        ("train_r", C.c_int),
        ("train_d", C.c_int),
        ("alpha", C.c_double),
    ]


def build(force: bool = False) -> None:
    """Compile the oracle (and oracle/_ref when /root/reference is present)."""
    if force or not os.path.exists(ORACLE_SO) or (
        os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(HERE, "mmw_oracle.c"))
    ):
        subprocess.run(["make", "-C", HERE, "oracle"], check=True, capture_output=True)
    if os.path.exists("/root/reference/cudaBenchMarking.cpp"):
        subprocess.run(["make", "-C", HERE, "ref"], check=True, capture_output=True)


_vp = C.c_void_p


def _ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(ORACLE_SO):
            build()
        L = C.CDLL(ORACLE_SO)
        L.orc_next_pow2.restype = C.c_int
        L.orc_next_pow2.argtypes = [C.c_int]
        L.orc_fft.argtypes = [C.c_int, _vp]
        L.orc_reshape.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_find_abs_max.restype = C.c_int
        L.orc_find_abs_max.argtypes = [_vp, C.c_int]
        L.orc_distance_from_raw.restype = C.c_double
        L.orc_distance_from_raw.argtypes = [C.c_int, C.c_int, C.c_int]
        L.orc_legacy_frame.restype = C.c_double
        L.orc_legacy_frame.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp]
        L.orc_hann_periodic.argtypes = [C.c_int, _vp]
        L.orc_range_fft.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp]
        L.orc_doppler_fft.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp, _vp]
        L.orc_power.argtypes = [_vp, C.c_int, C.c_int, C.c_int, _vp]
        L.orc_cfar.argtypes = [_vp, C.c_int, C.c_int, C.POINTER(CfarParams), _vp, _vp]
        L.orc_angle_argmax.restype = C.c_int
        L.orc_angle_argmax.argtypes = [_vp, C.c_int, C.c_int, C.POINTER(C.c_double)]
        L.orc_angle_fft_size.restype = C.c_int
        L.orc_angle_fft_size.argtypes = [C.c_int]
        L.orc_angle_rad.restype = C.c_double
        L.orc_angle_rad.argtypes = [C.c_int, C.c_int, C.c_double]
        L.orc_is_group_peak.restype = C.c_int
        L.orc_is_group_peak.argtypes = [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_process_frames.restype = C.c_long
        L.orc_process_frames.argtypes = [
            _vp, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, C.POINTER(CfarParams), C.c_double,
            _vp, C.c_long, C.POINTER(C.c_long), _vp, _vp, _vp, _vp, _vp, C.c_int,
        ]
        L.orc_process_frames_base.restype = C.c_long
        L.orc_process_frames_base.argtypes = [_vp] + L.orc_process_frames.argtypes
        L.orc_process_frames_ratio.restype = C.c_long
        L.orc_process_frames_ratio.argtypes = L.orc_process_frames_base.argtypes + [_vp]
        _lib = L
    return _lib


def next_pow2(n: int) -> int:
    return lib().orc_next_pow2(int(n))


def hann_periodic(n: int) -> np.ndarray:
    w = np.empty(n, np.float32)
    lib().orc_hann_periodic(n, _ptr(w))
    return w


def fft(x: np.ndarray) -> np.ndarray:
    y = np.ascontiguousarray(x, np.complex128).copy()
    lib().orc_fft(y.size, _ptr(y))
    return y


def reshape(shorts: np.ndarray, S: int, C_: int, A: int) -> np.ndarray:
    shorts = np.ascontiguousarray(shorts, np.int16)
    out = np.zeros(S * C_ * A, np.complex128)
    lib().orc_reshape(_ptr(shorts), _ptr(out), shorts.size, S, C_, A)
    return out


def legacy_frame(frame: np.ndarray, base_rx0: np.ndarray, S=100, C_=128, A=4, want_spectrum=False):
    """Returns (maxDis, raw_index[, spectrum]) — reference cpuTiming() loop body."""
    frame = np.ascontiguousarray(frame, np.int16)
    base = np.ascontiguousarray(base_rx0, np.complex128)
    n_ext = next_pow2(S * C_)
    spec = np.empty(n_ext, np.complex128) if want_spectrum else None
    raw = C.c_int(0)
    d = lib().orc_legacy_frame(_ptr(frame), _ptr(base), frame.size, S, C_, A, _ptr(spec), C.addressof(raw))
    return (d, raw.value, spec) if want_spectrum else (d, raw.value)


def range_fft(adc: np.ndarray, S: int, C_: int, A: int, win_r: np.ndarray) -> np.ndarray:
    adc = np.ascontiguousarray(adc, np.int16)
    Sp = next_pow2(S)
    rs = np.empty((A, Sp, C_), np.complex128)
    lib().orc_range_fft(_ptr(adc), S, C_, A, _ptr(np.ascontiguousarray(win_r, np.float32)), _ptr(rs))
    return rs


def doppler_fft(rs: np.ndarray, win_d: np.ndarray) -> np.ndarray:
    A, Sp, C_ = rs.shape
    Cp = next_pow2(C_)
    dc = np.empty((A, Sp, Cp), np.complex128)
    lib().orc_doppler_fft(_ptr(np.ascontiguousarray(rs)), Sp, C_, A, _ptr(np.ascontiguousarray(win_d, np.float32)), _ptr(dc))
    return dc


def power(dc: np.ndarray) -> np.ndarray:
    A, Sp, Cp = dc.shape
    P = np.empty((Sp, Cp), np.float64)
    lib().orc_power(_ptr(np.ascontiguousarray(dc)), Sp, Cp, A, _ptr(P))
    return P


def cfar(P: np.ndarray, guard=(2, 2), train=(8, 4), alpha=15.0):
    P = np.ascontiguousarray(P, np.float64)
    Sp, Cp = P.shape
    prm = CfarParams(guard[0], guard[1], train[0], train[1], float(alpha))
    mask = np.empty((Sp, Cp), np.uint8)
    noise = np.empty((Sp, Cp), np.float64)
    lib().orc_cfar(_ptr(P), Sp, Cp, C.byref(prm), _ptr(mask), _ptr(noise))
    return mask, noise


def angle_argmax(x: np.ndarray, n_theta: int):
    x = np.ascontiguousarray(x, np.complex128)
    ratio = C.c_double(0)
    k = lib().orc_angle_argmax(_ptr(x), x.size, n_theta, C.byref(ratio))
    return k, ratio.value


def angle_fft_size(A: int) -> int:
    return lib().orc_angle_fft_size(A)


def process_frames(adc, n_frames, S, C_, A, win_r, win_d, guard=(2, 2), train=(8, 4), alpha=15.0,
                   lambda_over_d=2.0, det_cap_per_frame=4096, want=(), n_threads=1, base=None):
    """Whole chain.  `want` may name 'rs', 'dc', 'P', 'mask', 'noise' to get the intermediates, and 'ratio' for the
    per-detection ratio 2nd-largest / largest angle-bin power (out['ratio'], aligned with out['dets']).
    base: one frame (int16, capture format) subtracted from every frame before the range window, or None."""
    adc = np.ascontiguousarray(adc, np.int16)
    base = None if base is None else np.ascontiguousarray(base, np.int16).reshape(-1)
    Sp, Cp = next_pow2(S), next_pow2(C_)
    prm = CfarParams(guard[0], guard[1], train[0], train[1], float(alpha))
    dets = np.zeros(det_cap_per_frame * max(n_frames, 1), DET_DTYPE)
    out = {}
    if "rs" in want:
        out["rs"] = np.empty((n_frames, A, Sp, C_), np.complex128)
    if "dc" in want:
        out["dc"] = np.empty((n_frames, A, Sp, Cp), np.complex128)
    if "P" in want:
        out["P"] = np.empty((n_frames, Sp, Cp), np.float64)
    if "mask" in want:
        out["mask"] = np.empty((n_frames, Sp, Cp), np.uint8)
    if "noise" in want:
        out["noise"] = np.empty((n_frames, Sp, Cp), np.float64)
    total = C.c_long(0)
    ratio = np.zeros(dets.size, np.float64) if "ratio" in want else None
    n = lib().orc_process_frames_ratio(
        _ptr(adc), _ptr(base), n_frames, S, C_, A,
        _ptr(np.ascontiguousarray(win_r, np.float32)), _ptr(np.ascontiguousarray(win_d, np.float32)),
        C.byref(prm), float(lambda_over_d), _ptr(dets), dets.size, C.byref(total),
        _ptr(out.get("rs")), _ptr(out.get("dc")), _ptr(out.get("P")), _ptr(out.get("mask")), _ptr(out.get("noise")),
        int(n_threads), _ptr(ratio),
    )
    if ratio is not None:
        out["ratio"] = ratio[:n].copy()
    out["dets"] = dets[:n].copy()
    out["n_total"] = total.value
    return out


# --------------------------------------------------------------------------
# the reference's own CPU functions (only where oracle/_ref was built)
# --------------------------------------------------------------------------
_ref = None


def have_ref() -> bool:
    return os.path.exists(REF_SO)


def ref():
    global _ref
    if _ref is None:
        L = C.CDLL(REF_SO)
        L.ref_next_pow2.restype = C.c_int
        L.ref_next_pow2.argtypes = [C.c_int]
        L.ref_reverse_bits.restype = C.c_int
        L.ref_reverse_bits.argtypes = [C.c_int, C.c_int]
        L.ref_butterfly_fft.argtypes = [C.c_int, _vp]
        L.ref_reshape.argtypes = [_vp, _vp, C.c_int]
        L.ref_find_abs_max.restype = C.c_int
        L.ref_find_abs_max.argtypes = [_vp, C.c_int]
        L.ref_cpu_frame.restype = C.c_double
        L.ref_cpu_frame.argtypes = [_vp, _vp, C.c_int, _vp, _vp]
        L.ref_cpu_time_frames.restype = C.c_double
        L.ref_cpu_time_frames.argtypes = [_vp, C.c_int, _vp, C.c_int, C.POINTER(C.c_double)]
        _ref = L
    return _ref


def ref_fft(x: np.ndarray) -> np.ndarray:
    y = np.ascontiguousarray(x, np.complex128).copy()
    ref().ref_butterfly_fft(y.size, _ptr(y))
    return y


def ref_reshape(shorts: np.ndarray) -> np.ndarray:
    shorts = np.ascontiguousarray(shorts, np.int16)
    out = np.zeros(100 * 128 * 4, np.complex128)
    ref().ref_reshape(_ptr(shorts), _ptr(out), shorts.size)
    return out


def ref_cpu_frame(frame: np.ndarray, base_rx0: np.ndarray, want_spectrum=False):
    frame = np.ascontiguousarray(frame, np.int16)
    base = np.ascontiguousarray(base_rx0, np.complex128)
    spec = np.empty(16384, np.complex128) if want_spectrum else None
    raw = C.c_int(0)
    d = ref().ref_cpu_frame(_ptr(frame), _ptr(base), frame.size, _ptr(spec), C.addressof(raw))
    return (d, raw.value, spec) if want_spectrum else (d, raw.value)


# the comparison of tests/test_oracle_pin.py::test_against_compiled_reference as arrays: computed with the reference's
# functions it is what tests/golden/make_golden.py stores (legacy_reference_direct.npz), with the oracle's what is compared
DIRECT_FFT_SIZES = (2, 16, 4096, 16384)
DIRECT_POW2_ARGS = (1, 2, 3, 100, 12800, 16384, 16385)
DIRECT_BINS = np.sort(np.random.default_rng(11).choice(16384, 2048, replace=False))   # stored sample of 16384-point outputs


def direct_vectors(cap, reshape, cpu_frame, fft, next_pow2, sample=False):
    """cap: legacy capture, frame 0 the base frame.  reshape / cpu_frame / fft / next_pow2: the reference's functions
    (ref_*) or the oracle's.  sample: keep only DIRECT_BINS of the 16384-point spectra and FFT."""
    pick = (lambda a: a[DIRECT_BINS]) if sample else (lambda a: a)
    y = reshape(cap[0])
    out = {"reshape0": y, "pow2": np.array([next_pow2(n) for n in DIRECT_POW2_ARGS])}
    dist, raw = [], []
    for f in range(1, cap.shape[0]):
        d, r, spec = cpu_frame(cap[f], y[:12800], want_spectrum=True)
        dist.append(d)
        raw.append(r)
        out[f"spec{f}"] = pick(spec)
    out["dist"], out["raw"] = np.array(dist), np.array(raw)
    for n in DIRECT_FFT_SIZES:
        X = fft(np.random.default_rng(n).normal(size=n) + 0j)
        out[f"fft{n}"] = pick(X) if n == 16384 else X
    return out


def ref_cpu_time_frames(frames: np.ndarray, base_rx0: np.ndarray):
    """Seconds the reference CPU loop body takes for frames[n][102400] on one thread."""
    frames = np.ascontiguousarray(frames, np.int16)
    base = np.ascontiguousarray(base_rx0, np.complex128)
    chk = C.c_double(0)
    t = ref().ref_cpu_time_frames(_ptr(frames), frames.shape[0], _ptr(base), frames.shape[1], C.byref(chk))
    return t, chk.value
