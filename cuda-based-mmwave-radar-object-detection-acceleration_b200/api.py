"""ctypes binding of libmmw_radar_b200.so — the only compute path of this package.

There is no Python/numpy/torch implementation of any stage here: every call goes through the
C ABI of include/mmw_radar.h / include/mmw_legacy.h into the CUDA kernels, and raises if the
library is missing or a CUDA call fails.  torch is used by callers only for device buffers,
streams and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import build as _build

MMW_OK, MMW_ERR_ARG, MMW_ERR_CUDA, MMW_ERR_STATE, MMW_ERR_OVERFLOW = 0, -1, -2, -3, -4
FLAG_PEAK = 1
RESULT_HEADER_BYTES = 32

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

# every symbol include/mmw_radar.h and include/mmw_legacy.h declare
C_ABI_SYMBOLS = [
    "mmw_default_config", "mmw_create", "mmw_destroy", "mmw_last_error", "mmw_get_info",
    "mmw_set_windows", "mmw_get_windows", "mmw_set_frame_offset", "mmw_stream", "mmw_use_stream",
    "mmw_process_device", "mmw_process_host", "mmw_submit_host", "mmw_wait", "mmw_read_detections", "mmw_read_counts",
    "mmw_device_results", "mmw_device_result_block", "mmw_merge_gathered", "mmw_copy_range_spectrum", "mmw_copy_doppler_cube", "mmw_copy_power_map",
    "mmw_copy_cfar_mask", "mmw_time_device", "mmw_check_guards", "mmw_set_detect_path",
    "mmw_set_graph_mode", "mmw_set_base_frame", "mmw_process_capture_file", "mmw_default_radar_params", "mmw_to_physical",
    "mmw_legacy_process_frame", "mmw_legacy_process_frames", "mmw_legacy_copy_spectrum", "mmw_legacy_shutdown",
    "mmw_legacy_process_device", "mmw_legacy_sync", "mmw_legacy_distance_from_raw", "mmw_legacy_process_file",
    "mmw_legacy_configure",
    "mmw_group_create", "mmw_group_destroy", "mmw_group_size", "mmw_group_context", "mmw_group_set_frame_offset", "mmw_shard_frames",
    "mmw_group_process_host", "mmw_group_process_device", "mmw_group_merged_block", "mmw_group_read_detections",
    "mmw_exchange_create", "mmw_exchange_destroy", "mmw_exchange_handle", "mmw_exchange_connect", "mmw_exchange_put", "mmw_exchange_merge",
    "mmw_exchange_wait",
    "mmw_default_cluster_params", "mmw_set_clustering", "mmw_read_objects", "mmw_read_labels", "mmw_device_objects",
    "mmw_objects_to_physical",
]
# the reference's own entry point (acceleration.h:32), C++ linkage
LEGACY_MANGLED = "_Z14cudaProcessingPsP9Complex_tiPdS2_S2_S2_"


# mmw_object of include/mmw_radar.h (48 bytes); tests/test_cluster_reference.py checks the offsets against the header
OBJ_DTYPE = np.dtype(
    [
        ("frame", "<u4"), ("first_det", "<u4"), ("n_det", "<u4"), ("peak_det", "<u4"),
        ("range_bin", "<f4"), ("doppler_bin", "<f4"), ("angle_rad", "<f4"),
        ("power", "<f4"), ("peak_power", "<f4"), ("peak_noise", "<f4"),
        ("range_min", "<u2"), ("range_max", "<u2"), ("doppler_min", "<i2"), ("doppler_max", "<i2"),
    ]
)
assert OBJ_DTYPE.itemsize == 48
assert [OBJ_DTYPE.fields[n][1] for n in OBJ_DTYPE.names] == [0, 4, 8, 12, 16, 20, 24, 28, 32, 36, 40, 42, 44, 46]
OBJECT_HEADER_BYTES = 32
OBJECTS_CUT, OBJECTS_DETECTIONS_TRUNCATED = 0x1, 0x2       # flag bits of the object header's word 3


class ClusterParams(C.Structure):
    """mmw_cluster_params"""
    _fields_ = [("eps_range", C.c_int), ("eps_doppler", C.c_int), ("eps_angle", C.c_int), ("min_points", C.c_int),
                ("max_objects_per_frame", C.c_int)]


class Config(C.Structure):
    _fields_ = [
        ("n_samples", C.c_int), ("n_chirps", C.c_int), ("n_antennas", C.c_int), ("max_frames", C.c_int),
        ("cfar_guard_r", C.c_int), ("cfar_guard_d", C.c_int), ("cfar_train_r", C.c_int), ("cfar_train_d", C.c_int),
        ("cfar_alpha", C.c_float), ("max_det_per_frame", C.c_int), ("keep_doppler_cube", C.c_int),
        ("lambda_over_d", C.c_float), ("device", C.c_int),
    ]


class Info(C.Structure):
    _fields_ = [
        ("Sp", C.c_int), ("Cp", C.c_int), ("n_theta", C.c_int), ("sm_count", C.c_int),
        ("adc_bytes_per_frame", C.c_longlong), ("algorithmic_bytes_per_frame", C.c_longlong),
        ("workspace_bytes", C.c_longlong), ("kernels_per_batch", C.c_int),
    ]


class RadarParams(C.Structure):
    """mmw_radar_params: the reference's radar constants (cudaBenchMarking.cpp:10-19)."""
    _fields_ = [("f0_hz", C.c_double), ("slope_hz_per_s", C.c_double), ("fs_hz", C.c_double),
                ("chirp_period_s", C.c_double), ("light_speed", C.c_double)]


TARGET_DTYPE = np.dtype([("frame", "<u4"), ("range_m", "<f4"), ("velocity_mps", "<f4"), ("angle_deg", "<f4"),
                         ("snr_db", "<f4"), ("flags", "<u4")])
assert TARGET_DTYPE.itemsize == 24


class RadarError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"mmw error {code}: {msg}")
        self.code = code


_lib = None


def library_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """Loads the shared library (building it with nvcc if it is absent or stale)."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        _build.build()
    if not os.path.exists(_build.LIB):
        raise RuntimeError(f"{_build.LIB} is missing: the CUDA library was not built; there is no fallback path")
    L = C.CDLL(_build.LIB)
    vp, ip = C.c_void_p, C.POINTER(C.c_int)
    L.mmw_last_error.restype = C.c_char_p
    L.mmw_default_config.argtypes = [C.POINTER(Config), C.c_int, C.c_int, C.c_int, C.c_int]
    L.mmw_default_config.restype = None
    L.mmw_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.mmw_destroy.argtypes = [vp]
    L.mmw_destroy.restype = None
    L.mmw_get_info.argtypes = [vp, C.POINTER(Info)]
    L.mmw_set_windows.argtypes = [vp, vp, vp]
    L.mmw_get_windows.argtypes = [vp, vp, vp]
    L.mmw_set_frame_offset.argtypes = [vp, C.c_uint32]
    L.mmw_stream.argtypes = [vp]
    L.mmw_stream.restype = vp
    L.mmw_use_stream.argtypes = [vp, vp]
    L.mmw_process_device.argtypes = [vp, vp, C.c_int]
    L.mmw_process_host.argtypes = [vp, vp, C.c_int, vp, C.c_int, ip]
    L.mmw_submit_host.argtypes = [vp, vp, C.c_int]
    L.mmw_wait.argtypes = [vp, vp, C.c_int, ip]
    L.mmw_read_detections.argtypes = [vp, vp, C.c_int, ip]
    L.mmw_read_counts.argtypes = [vp, vp, C.c_int]
    L.mmw_device_results.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.mmw_device_result_block.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_longlong)]
    L.mmw_merge_gathered.argtypes = [vp, vp, C.c_int, C.c_longlong, vp, C.c_int]
    for name in ("mmw_copy_range_spectrum", "mmw_copy_doppler_cube", "mmw_copy_power_map", "mmw_copy_cfar_mask"):
        getattr(L, name).argtypes = [vp, C.c_int, vp]
    L.mmw_time_device.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.mmw_check_guards.argtypes = [vp, C.POINTER(C.c_longlong)]
    L.mmw_set_detect_path.argtypes = [vp, C.c_int]
    L.mmw_exchange_create.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.mmw_exchange_destroy.argtypes = [vp]
    L.mmw_exchange_destroy.restype = None
    L.mmw_exchange_handle.argtypes = [vp, vp]
    L.mmw_exchange_connect.argtypes = [vp, vp]
    L.mmw_exchange_put.argtypes = [vp]
    L.mmw_exchange_merge.argtypes = [vp, C.POINTER(vp)]
    L.mmw_exchange_wait.argtypes = [vp, vp, C.POINTER(vp)]
    L.mmw_set_graph_mode.argtypes = [vp, C.c_int]
    L.mmw_set_base_frame.argtypes = [vp, vp]
    L.mmw_process_capture_file.argtypes = [vp, C.c_char_p, C.c_longlong, C.c_int, C.c_int, vp, C.c_int, ip, ip]
    L.mmw_default_radar_params.argtypes = [C.POINTER(RadarParams)]
    L.mmw_default_radar_params.restype = None
    L.mmw_to_physical.argtypes = [C.POINTER(RadarParams), C.c_int, C.c_int, vp, C.c_int, vp]
    L.mmw_default_cluster_params.argtypes = [C.POINTER(ClusterParams)]
    L.mmw_default_cluster_params.restype = None
    L.mmw_set_clustering.argtypes = [vp, C.POINTER(ClusterParams)]
    L.mmw_read_objects.argtypes = [vp, vp, C.c_int, ip]
    L.mmw_read_labels.argtypes = [vp, vp, C.c_int, ip]
    L.mmw_device_objects.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    L.mmw_objects_to_physical.argtypes = [C.POINTER(RadarParams), C.c_int, C.c_int, vp, C.c_int, vp]
    L.mmw_legacy_process_device.argtypes = [vp, C.c_int, vp, vp]
    L.mmw_legacy_distance_from_raw.argtypes = [C.c_int]
    L.mmw_legacy_distance_from_raw.restype = C.c_double
    L.mmw_legacy_process_file.argtypes = [C.c_char_p, vp, vp, C.c_int, ip]
    L.mmw_legacy_process_frame.argtypes = [vp, vp, C.c_int, ip]
    L.mmw_legacy_process_frame.restype = C.c_double
    L.mmw_legacy_process_frames.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp]
    L.mmw_legacy_copy_spectrum.argtypes = [vp]
    L.mmw_legacy_shutdown.restype = None
    L.mmw_group_create.argtypes = [C.POINTER(Config), C.POINTER(C.c_int), C.c_int, C.POINTER(vp)]
    L.mmw_group_destroy.argtypes = [vp]
    L.mmw_group_destroy.restype = None
    L.mmw_group_size.argtypes = [vp]
    L.mmw_group_context.argtypes = [vp, C.c_int]
    L.mmw_group_context.restype = vp
    L.mmw_group_set_frame_offset.argtypes = [vp, C.c_uint32]
    L.mmw_shard_frames.argtypes = [C.c_int, C.c_int, C.c_int, ip, ip]
    L.mmw_shard_frames.restype = None
    L.mmw_group_process_host.argtypes = [vp, vp, C.c_int, vp, C.c_int, ip]
    L.mmw_group_process_device.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_int)]
    L.mmw_group_merged_block.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_longlong)]
    L.mmw_group_read_detections.argtypes = [vp, vp, C.c_int, ip]
    L.mmw_legacy_configure.argtypes = [C.c_int, C.c_int]
    cp = getattr(L, LEGACY_MANGLED)
    cp.restype = C.c_double
    cp.argtypes = [vp, vp, C.c_int, vp, vp, vp, vp]
    _lib = L
    return L


def _check(rc: int, allow_overflow: bool = False) -> int:
    if rc == MMW_OK or (allow_overflow and rc == MMW_ERR_OVERFLOW):
        return rc
    raise RadarError(rc, load().mmw_last_error().decode(errors="replace"))


DETECT_AUTO, DETECT_PER_CELL, DETECT_REFFT = 0, 1, 2      # MMW_DETECT_* of include/mmw_radar.h


def last_error() -> str:
    """Text of the last error (or guard-band report) of the calling thread: mmw_last_error()."""
    return load().mmw_last_error().decode(errors="replace")


def _np_ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _dev_ptr(t) -> int:
    """Accepts a torch CUDA tensor or a raw integer device address."""
    if isinstance(t, int):
        return t
    if not t.is_cuda or not t.is_contiguous():
        raise ValueError("expected a contiguous CUDA tensor")
    return t.data_ptr()


def next_pow2(n: int) -> int:
    p = 1
    while p < n:
        p <<= 1
    return p


class RadarContext:
    """One plan + HBM workspace on one GPU (mmw_ctx).  Mirrors what cudaProcessing()
    (acceleration.cu:417-572) allocates per frame, held once for a batch of `max_frames` frames."""

    def __init__(self, n_samples: int, n_chirps: int, n_antennas: int, max_frames: int, *,
                 cfar_guard=(2, 2), cfar_train=(8, 4), cfar_alpha: float = 15.0, max_det_per_frame: int = 1024,
                 keep_doppler_cube: bool = False, lambda_over_d: float = 2.0, device: int = -1):
        self._L = load()
        cfg = Config()
        self._L.mmw_default_config(C.byref(cfg), n_samples, n_chirps, n_antennas, max_frames)
        cfg.cfar_guard_r, cfg.cfar_guard_d = cfar_guard
        cfg.cfar_train_r, cfg.cfar_train_d = cfar_train
        cfg.cfar_alpha = cfar_alpha
        cfg.max_det_per_frame = max_det_per_frame
        cfg.keep_doppler_cube = int(keep_doppler_cube)
        cfg.lambda_over_d = lambda_over_d
        cfg.device = device
        self.cfg = cfg
        self._h = C.c_void_p()
        _check(self._L.mmw_create(C.byref(cfg), C.byref(self._h)))
        info = Info()
        _check(self._L.mmw_get_info(self._h, C.byref(info)))
        self.info = info
        self.S, self.C, self.A = n_samples, n_chirps, n_antennas
        self.Sp, self.Cp, self.n_theta = info.Sp, info.Cp, info.n_theta
        self.max_frames = max_frames
        self.max_det_per_frame = max_det_per_frame
        self.frame_shorts = 2 * n_samples * n_chirps * n_antennas

    # -- lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.mmw_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- configuration
    def set_windows(self, win_range=None, win_doppler=None):
        wr = None if win_range is None else np.ascontiguousarray(win_range, np.float32)
        wd = None if win_doppler is None else np.ascontiguousarray(win_doppler, np.float32)
        if wr is not None and wr.size != self.S:
            raise ValueError("range window must have n_samples entries")
        if wd is not None and wd.size != self.C:
            raise ValueError("doppler window must have n_chirps entries")
        _check(self._L.mmw_set_windows(self._h, None if wr is None else _np_ptr(wr), None if wd is None else _np_ptr(wd)))

    def get_windows(self):
        wr = np.empty(self.S, np.float32)
        wd = np.empty(self.C, np.float32)
        _check(self._L.mmw_get_windows(self._h, _np_ptr(wr), _np_ptr(wd)))
        return wr, wd

    def set_base_frame(self, base_frame=None):
        """Static-clutter removal: one frame in capture format subtracted from every frame (None turns it off)."""
        if base_frame is None:
            _check(self._L.mmw_set_base_frame(self._h, None))
            return
        b = np.ascontiguousarray(base_frame, np.int16).reshape(-1)
        if b.size != self.frame_shorts:
            raise ValueError("base frame must hold one frame (2*S*C*A int16)")
        _check(self._L.mmw_set_base_frame(self._h, _np_ptr(b)))

    def set_graph_mode(self, enable: bool):
        """Replay the launch sequence of a batch as one CUDA graph (for one-frame-per-call streaming)."""
        _check(self._L.mmw_set_graph_mode(self._h, int(bool(enable))))

    def set_detect_path(self, path: int):
        """DETECT_AUTO / DETECT_PER_CELL / DETECT_REFFT: how fused mode gets the antenna snapshots of the detected cells
        (include/mmw_radar.h: mmw_set_detect_path)."""
        _check(self._L.mmw_set_detect_path(self._h, int(path)))
        _check(self._L.mmw_get_info(self._h, C.byref(self.info)))      # kernels_per_batch and workspace_bytes follow the path

    def set_frame_offset(self, first_frame: int):
        _check(self._L.mmw_set_frame_offset(self._h, int(first_frame)))

    def set_clustering(self, **params):
        """Group each frame's detections into objects after every batch (include/mmw_radar.h: mmw_set_clustering).
        Keyword arguments override mmw_default_cluster_params (eps_range, eps_doppler, eps_angle, min_points,
        max_objects_per_frame); no arguments turn clustering off."""
        if not params:
            _check(self._L.mmw_set_clustering(self._h, None))
        else:
            cp = default_cluster_params()
            for k, v in params.items():
                if k not in dict(ClusterParams._fields_):
                    raise TypeError(f"unknown clustering parameter {k!r}")
                setattr(cp, k, int(v))
            _check(self._L.mmw_set_clustering(self._h, C.byref(cp)))
        _check(self._L.mmw_get_info(self._h, C.byref(self.info)))      # kernels_per_batch and workspace_bytes follow

    def read_objects(self, capacity: int | None = None):
        """Objects of the last (clustered) batch. Returns (objects, overflow_flag): overflow when objects were cut, the
        detection list was truncated or capacity was short."""
        cap = capacity if capacity is not None else self.max_frames * self.max_det_per_frame
        objs = np.empty(max(cap, 1), OBJ_DTYPE)
        n = C.c_int(0)
        rc = _check(self._L.mmw_read_objects(self._h, _np_ptr(objs), cap, C.byref(n)), True)
        return objs[: n.value].copy(), rc == MMW_ERR_OVERFLOW

    def read_labels(self, capacity: int | None = None) -> np.ndarray:
        """Object index of every detection of the last batch (aligned with its detection list), -1 for none."""
        cap = capacity if capacity is not None else self.max_frames * self.max_det_per_frame
        labels = np.empty(max(cap, 1), np.int32)
        n = C.c_int(0)
        _check(self._L.mmw_read_labels(self._h, _np_ptr(labels), cap, C.byref(n)))
        return labels[: n.value].copy()

    def device_objects(self):
        """(device address of the object records, device address of the 32-byte object header)."""
        o, h = C.c_void_p(), C.c_void_p()
        _check(self._L.mmw_device_objects(self._h, C.byref(o), C.byref(h)))
        return int(o.value), int(h.value)

    def objects_to_physical(self, objs: np.ndarray, params: RadarParams | None = None) -> np.ndarray:
        return objects_to_physical(objs, self.Sp, self.Cp, params)

    @property
    def stream(self) -> int:
        return int(self._L.mmw_stream(self._h) or 0)

    def use_stream(self, cuda_stream: int | None):
        _check(self._L.mmw_use_stream(self._h, C.c_void_p(cuda_stream or 0)))

    # -- processing
    def process_device(self, adc_dev, n_frames: int):
        """adc_dev: torch int16 CUDA tensor (or device address) of n_frames captures; asynchronous."""
        _check(self._L.mmw_process_device(self._h, C.c_void_p(_dev_ptr(adc_dev)), n_frames))

    def process_host(self, adc_host, n_frames: int, det_capacity: int | None = None, out: np.ndarray | None = None):
        """adc_host: numpy int16 array or a (pinned) CPU torch tensor. Returns (detections, overflow_flag)."""
        if isinstance(adc_host, np.ndarray):
            a = np.ascontiguousarray(adc_host, np.int16)
            ptr, n = a.ctypes.data, a.size
        else:
            ptr, n = adc_host.data_ptr(), adc_host.numel()
        if n < n_frames * self.frame_shorts:
            raise ValueError("capture buffer shorter than n_frames frames")
        cap = det_capacity if det_capacity is not None else n_frames * self.max_det_per_frame
        dets = out if out is not None else np.empty(cap, DET_DTYPE)
        cap = min(cap, dets.size)
        n_det = C.c_int(0)
        rc = _check(self._L.mmw_process_host(self._h, C.c_void_p(ptr), n_frames, _np_ptr(dets), cap, C.byref(n_det)), True)
        return dets[: n_det.value], rc == MMW_ERR_OVERFLOW

    def process_capture_file(self, path: str, first_frame: int = 0, max_frames: int = 0, use_first_as_base: bool = False,
                             det_capacity: int = 1 << 20):
        """Streams a raw capture file (the fhy_direct.bin format) through the chain. Returns (detections, frames done, overflow)."""
        dets = np.empty(det_capacity, DET_DTYPE)
        n_det, n_frames = C.c_int(0), C.c_int(0)
        rc = _check(self._L.mmw_process_capture_file(self._h, os.fsencode(path), first_frame, max_frames, int(use_first_as_base),
                                                     _np_ptr(dets), det_capacity, C.byref(n_det), C.byref(n_frames)), True)
        return dets[: n_det.value].copy(), n_frames.value, rc == MMW_ERR_OVERFLOW

    def to_physical(self, dets: np.ndarray, params: RadarParams | None = None) -> np.ndarray:
        return to_physical(dets, self.Sp, self.Cp, params)

    def submit_host(self, adc_host, n_frames: int):
        """First half of process_host: queue upload + chain + read-back, return at once (keep adc_host alive and pinned)."""
        if isinstance(adc_host, np.ndarray):
            ptr, n = adc_host.ctypes.data, adc_host.size
            if adc_host.dtype != np.int16 or not adc_host.flags["C_CONTIGUOUS"]:
                raise ValueError("submit_host needs a C-contiguous int16 array (it is read after the call returns)")
        else:
            ptr, n = adc_host.data_ptr(), adc_host.numel()
        if n < n_frames * self.frame_shorts:
            raise ValueError("capture buffer shorter than n_frames frames")
        _check(self._L.mmw_submit_host(self._h, C.c_void_p(ptr), n_frames))

    def wait(self, det_capacity: int | None = None, out: np.ndarray | None = None):
        """Second half of process_host: block until the submitted batch is done. Returns (detections, overflow_flag)."""
        cap = det_capacity if det_capacity is not None else self.max_frames * self.max_det_per_frame
        dets = out if out is not None else np.empty(cap, DET_DTYPE)
        cap = min(cap, dets.size)
        n_det = C.c_int(0)
        rc = _check(self._L.mmw_wait(self._h, _np_ptr(dets), cap, C.byref(n_det)), True)
        return dets[: n_det.value], rc == MMW_ERR_OVERFLOW

    def read_detections(self, det_capacity: int | None = None):
        cap = det_capacity if det_capacity is not None else self.max_frames * self.max_det_per_frame
        dets = np.empty(cap, DET_DTYPE)
        n_det = C.c_int(0)
        rc = _check(self._L.mmw_read_detections(self._h, _np_ptr(dets), cap, C.byref(n_det)), True)
        return dets[: n_det.value].copy(), rc == MMW_ERR_OVERFLOW

    def read_counts(self, n_frames: int) -> np.ndarray:
        counts = np.empty(n_frames, np.uint32)
        _check(self._L.mmw_read_counts(self._h, _np_ptr(counts), n_frames))
        return counts

    def device_results(self):
        """(device address of the dense ordered detection list, device address of the 4-word header)."""
        d, h = C.c_void_p(), C.c_void_p()
        _check(self._L.mmw_device_results(self._h, C.byref(d), C.byref(h)))
        return int(d.value), int(h.value)

    def device_result_block(self):
        """(device address, capacity in bytes) of the contiguous [32-byte header | dense records] block."""
        b, n = C.c_void_p(), C.c_longlong(0)
        _check(self._L.mmw_device_result_block(self._h, C.byref(b), C.byref(n)))
        return int(b.value), int(n.value)

    def merge_gathered(self, gathered_dev, n_ranks: int, stride_bytes: int, merged_dev, merged_capacity: int):
        """rank 0: n_ranks gathered result blocks -> one merged block (asynchronous, one kernel)."""
        _check(self._L.mmw_merge_gathered(self._h, C.c_void_p(_dev_ptr(gathered_dev)), n_ranks, stride_bytes,
                                          C.c_void_p(_dev_ptr(merged_dev)), merged_capacity))

    # -- intermediates (canonical layouts)
    def range_spectrum(self, frame: int) -> np.ndarray:
        out = np.empty((self.A, self.Sp, self.C), np.complex64)
        _check(self._L.mmw_copy_range_spectrum(self._h, frame, _np_ptr(out)))
        return out

    def doppler_cube(self, frame: int) -> np.ndarray:
        out = np.empty((self.A, self.Sp, self.Cp), np.complex64)
        _check(self._L.mmw_copy_doppler_cube(self._h, frame, _np_ptr(out)))
        return out

    def power_map(self, frame: int) -> np.ndarray:
        out = np.empty((self.Sp, self.Cp), np.float32)
        _check(self._L.mmw_copy_power_map(self._h, frame, _np_ptr(out)))
        return out

    def cfar_mask(self, frame: int) -> np.ndarray:
        out = np.empty((self.Sp, self.Cp), np.uint8)
        _check(self._L.mmw_copy_cfar_mask(self._h, frame, _np_ptr(out)))
        return out

    # -- timing
    def time_device(self, adc_dev, n_frames: int, iters: int, per_stage: bool = False):
        total = C.c_float(0)
        stages = (C.c_float * 4)()
        _check(self._L.mmw_time_device(self._h, C.c_void_p(_dev_ptr(adc_dev)), n_frames, iters, C.byref(total),
                                       stages if per_stage else None))
        return (total.value, list(stages)) if per_stage else total.value

    def check_guards(self) -> int:
        """Guard bytes overwritten around the context's device buffers since create (needs MMW_GUARD=1 at create): 0 = no
        kernel wrote out of bounds.  include/mmw_radar.h: mmw_check_guards."""
        bad = C.c_longlong(0)
        _check(self._L.mmw_check_guards(self._h, C.byref(bad)))
        return int(bad.value)


class PeerExchange:
    """mmw_exchange_*: the gather of a frame-sharded job's detection lists by copy-engine puts into rank 0's memory
    (include/mmw_radar.h).  `all_gather_bytes(b: bytes) -> list[bytes]` is the launcher's transport for the 64-byte handles."""

    def __init__(self, ctx: "RadarContext", rank: int, n_ranks: int, records_per_rank: int, all_gather_bytes, depth: int = 4):
        """Never raises between the collective calls: a rank whose set-up fails (no peer access, no IPC between the ranks'
        processes, ...) still takes part in the handle all-gather and reports the failure in `self.error` (None = connected),
        so the launcher can agree on a fall-back with a reduction over the ranks instead of hanging in a barrier."""
        self._L = load()
        self.ctx, self.rank, self.n_ranks, self.records_per_rank = ctx, rank, n_ranks, records_per_rank
        self._x, self.error = None, None
        mine = (C.c_ubyte * 64)()
        try:
            if os.environ.get("MMW_EXCHANGE_FAIL_RANK") == str(rank):      # tests: this rank pretends it cannot set up
                raise RadarError(MMW_ERR_STATE, "peer exchange disabled on this rank by MMW_EXCHANGE_FAIL_RANK")
            h = C.c_void_p()
            _check(self._L.mmw_exchange_create(ctx._h, rank, n_ranks, records_per_rank, depth, C.byref(h)))
            self._x = h
            _check(self._L.mmw_exchange_handle(self._x, mine))
        except RadarError as e:
            self.error = e
        everyone = all_gather_bytes(bytes(mine))                           # collective: every rank gets here
        assert len(everyone) == n_ranks and all(len(b) == 64 for b in everyone)
        if self.error is None:
            try:
                blob = (C.c_ubyte * (64 * n_ranks)).from_buffer_copy(b"".join(everyone))
                _check(self._L.mmw_exchange_connect(self._x, blob))
            except RadarError as e:
                self.error = e

    def close(self):
        if getattr(self, "_x", None):
            self._L.mmw_exchange_destroy(self._x)
            self._x = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def put(self):
        if not self.ctx._h.value or not self._x:
            raise RadarError(MMW_ERR_STATE, "PeerExchange.put: the exchange or its context is closed")
        _check(self._L.mmw_exchange_put(self._x))

    def merge(self) -> int:
        p = C.c_void_p()
        _check(self._L.mmw_exchange_merge(self._x, C.byref(p)))
        return p.value

    def wait(self, cuda_stream: int | None = None) -> int:
        p = C.c_void_p()
        _check(self._L.mmw_exchange_wait(self._x, C.c_void_p(cuda_stream or 0), C.byref(p)))
        return p.value


class RadarGroup:
    """A frame-sharded group of GPUs driven by this process (mmw_group_*): one context per device, one NCCL communicator,
    detection lists gathered to the first device.  max_frames is the capacity PER GPU."""

    def __init__(self, n_samples: int, n_chirps: int, n_antennas: int, max_frames: int, devices, **kw):
        self._L = load()
        cfg = Config()
        self._L.mmw_default_config(C.byref(cfg), n_samples, n_chirps, n_antennas, max_frames)
        cfg.cfar_guard_r, cfg.cfar_guard_d = kw.get("cfar_guard", (2, 2))
        cfg.cfar_train_r, cfg.cfar_train_d = kw.get("cfar_train", (8, 4))
        cfg.cfar_alpha = kw.get("cfar_alpha", 15.0)
        cfg.max_det_per_frame = kw.get("max_det_per_frame", 1024)
        cfg.keep_doppler_cube = int(kw.get("keep_doppler_cube", False))
        cfg.lambda_over_d = kw.get("lambda_over_d", 2.0)
        devs = (C.c_int * len(devices))(*devices)
        self._h = C.c_void_p()
        _check(self._L.mmw_group_create(C.byref(cfg), devs, len(devices), C.byref(self._h)))
        self.devices = list(devices)
        self.max_frames, self.max_det_per_frame = max_frames, cfg.max_det_per_frame
        self.frame_shorts = 2 * n_samples * n_chirps * n_antennas

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.mmw_group_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    @property
    def size(self) -> int:
        return self._L.mmw_group_size(self._h)

    def set_frame_offset(self, first_frame: int):
        _check(self._L.mmw_group_set_frame_offset(self._h, int(first_frame)))

    def process_host(self, adc_host, n_frames: int, det_capacity: int | None = None):
        """Host capture -> shards -> chain on every GPU -> NCCL gather to device 0 -> (detections, overflow_flag)."""
        if isinstance(adc_host, np.ndarray):
            a = np.ascontiguousarray(adc_host, np.int16)
            ptr, n = a.ctypes.data, a.size
        else:
            ptr, n = adc_host.data_ptr(), adc_host.numel()
        if n < n_frames * self.frame_shorts:
            raise ValueError("capture buffer shorter than n_frames frames")
        cap = det_capacity if det_capacity is not None else n_frames * self.max_det_per_frame
        dets = np.empty(cap, DET_DTYPE)
        n_det = C.c_int(0)
        rc = _check(self._L.mmw_group_process_host(self._h, C.c_void_p(ptr), n_frames, _np_ptr(dets), cap, C.byref(n_det)), True)
        return dets[: n_det.value], rc == MMW_ERR_OVERFLOW

    def process_device(self, shards, n_frames):
        """shards[i]: torch int16 CUDA tensor on the group's i-th device (or None / an address) holding n_frames[i] frames."""
        ptrs = (C.c_void_p * len(shards))(*[C.c_void_p(_dev_ptr(t) if t is not None else 0) for t in shards])
        cnt = (C.c_int * len(shards))(*[int(v) for v in n_frames])
        _check(self._L.mmw_group_process_device(self._h, ptrs, cnt))

    def read_detections(self, det_capacity: int | None = None):
        cap = det_capacity if det_capacity is not None else self.size * self.max_frames * self.max_det_per_frame
        dets = np.empty(cap, DET_DTYPE)
        n_det = C.c_int(0)
        rc = _check(self._L.mmw_group_read_detections(self._h, _np_ptr(dets), cap, C.byref(n_det)), True)
        return dets[: n_det.value].copy(), rc == MMW_ERR_OVERFLOW

    def merged_block(self):
        b, n = C.c_void_p(), C.c_longlong(0)
        _check(self._L.mmw_group_merged_block(self._h, C.byref(b), C.byref(n)))
        return int(b.value), int(n.value)


def shard_frames(n_frames: int, n_ranks: int, rank: int):
    first, count = C.c_int(0), C.c_int(0)
    load().mmw_shard_frames(n_frames, n_ranks, rank, C.byref(first), C.byref(count))
    return first.value, count.value


def default_radar_params() -> RadarParams:
    rp = RadarParams()
    load().mmw_default_radar_params(C.byref(rp))
    return rp


def to_physical(dets: np.ndarray, Sp: int, Cp: int, params: RadarParams | None = None) -> np.ndarray:
    """Detections -> range [m], radial velocity [m/s], angle [deg], SNR [dB] (mmw_to_physical; host arithmetic)."""
    L = load()
    params = params if params is not None else default_radar_params()
    d = np.ascontiguousarray(dets, DET_DTYPE)
    out = np.empty(d.size, TARGET_DTYPE)
    _check(L.mmw_to_physical(C.byref(params), Sp, Cp, _np_ptr(d), d.size, _np_ptr(out)))
    return out


def default_cluster_params() -> ClusterParams:
    cp = ClusterParams()
    load().mmw_default_cluster_params(C.byref(cp))
    return cp


def objects_to_physical(objs: np.ndarray, Sp: int, Cp: int, params: RadarParams | None = None) -> np.ndarray:
    """Objects -> range [m], radial velocity [m/s], angle [deg] of their mean bins, SNR [dB] of their peak
    (mmw_objects_to_physical; host arithmetic)."""
    L = load()
    params = params if params is not None else default_radar_params()
    o = np.ascontiguousarray(objs, OBJ_DTYPE)
    out = np.empty(o.size, TARGET_DTYPE)
    _check(L.mmw_objects_to_physical(C.byref(params), Sp, Cp, _np_ptr(o), o.size, _np_ptr(out)))
    return out


# ---------------------------------------------------------------------------
# legacy entry point (reference cfg: 100 x 128 x 4)
# ---------------------------------------------------------------------------
def cudaProcessing(frame: np.ndarray, base_frame_rx0: np.ndarray, size: int | None = None, timers: np.ndarray | None = None) -> float:
    """Calls the C++-linkage drop-in symbol exactly as the reference's cudaTiming() does
    (cudaBenchMarking.cpp:377). timers = float64[4] (fft, preProcess, findMax, total), accumulated."""
    L = load()
    frame = np.ascontiguousarray(frame, np.int16)
    base = np.ascontiguousarray(base_frame_rx0, np.complex128)
    if base.size != 12800:
        raise ValueError("base frame must hold 12800 complex values (rx0 of frame 0)")
    t = timers if timers is not None else np.zeros(4, np.float64)
    fn = getattr(L, LEGACY_MANGLED)
    p = t.ctypes.data
    return fn(_np_ptr(frame), _np_ptr(base), frame.size if size is None else size,
              C.c_void_p(p), C.c_void_p(p + 8), C.c_void_p(p + 16), C.c_void_p(p + 24))


def legacy_process_frame(frame: np.ndarray, base_frame_rx0: np.ndarray, size: int | None = None):
    L = load()
    frame = np.ascontiguousarray(frame, np.int16)
    base = np.ascontiguousarray(base_frame_rx0, np.complex128)
    raw = C.c_int(0)
    d = L.mmw_legacy_process_frame(_np_ptr(frame), _np_ptr(base), frame.size if size is None else size, C.byref(raw))
    if d < 0:
        raise RadarError(int(d), L.mmw_last_error().decode(errors="replace"))
    return d, raw.value


def legacy_process_frames(frames: np.ndarray, base_frame_rx0: np.ndarray):
    L = load()
    frames = np.ascontiguousarray(frames, np.int16)
    base = np.ascontiguousarray(base_frame_rx0, np.complex128)
    n = frames.shape[0]
    dist = np.empty(n, np.float64)
    raw = np.empty(n, np.int32)
    _check(L.mmw_legacy_process_frames(_np_ptr(frames), n, _np_ptr(base), frames.shape[1], _np_ptr(dist), _np_ptr(raw)))
    return dist, raw


def legacy_process_device(frames_dev, n_frames: int, base_frame_rx0: np.ndarray, raw_dev):
    """Frames already in HBM -> raw arg-max bins in HBM (asynchronous; legacy_sync() waits)."""
    base = np.ascontiguousarray(base_frame_rx0, np.complex128)
    _check(load().mmw_legacy_process_device(C.c_void_p(_dev_ptr(frames_dev)), n_frames, _np_ptr(base), C.c_void_p(_dev_ptr(raw_dev))))


def legacy_sync():
    _check(load().mmw_legacy_sync())


def legacy_distance_from_raw(raw: int) -> float:
    return load().mmw_legacy_distance_from_raw(int(raw))


def legacy_process_file(path: str, capacity: int = 4096):
    """The reference's cudaTiming() loop in one call: frame 0 is the base frame, every later frame gives a distance."""
    dist = np.empty(capacity, np.float64)
    raw = np.empty(capacity, np.int32)
    n = C.c_int(0)
    _check(load().mmw_legacy_process_file(os.fsencode(path), _np_ptr(dist), _np_ptr(raw), capacity, C.byref(n)))
    k = min(n.value, capacity)
    return dist[:k].copy(), raw[:k].copy(), n.value


def legacy_configure(kernel_variant: int = -1, quiet: int = -1):
    """kernel_variant: 0 pick by batch size, 1 one CTA per frame, 2 the 8-CTA cluster kernel; quiet: silence the per-call line.
    Negative = keep."""
    _check(load().mmw_legacy_configure(int(kernel_variant), int(quiet)))


def legacy_spectrum() -> np.ndarray:
    out = np.empty(16384, np.complex64)
    _check(load().mmw_legacy_copy_spectrum(_np_ptr(out)))
    return out
