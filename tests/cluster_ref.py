"""ctypes front-end of tests/cluster_ref.c, the CPU reference of the clustering stage (include/mmw_radar.h:
mmw_set_clustering).  Test infrastructure only: the C file is compiled on first use into a temporary directory (the
repository tree may be read-only) and removed when the process ends."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

DET_DTYPE = np.dtype([("frame", "<u4"), ("range_bin", "<u2"), ("doppler_bin", "<u2"), ("power", "<f4"), ("noise", "<f4"),
                      ("angle_bin", "<i2"), ("flags", "<u2"), ("angle_rad", "<f4")])
# mmw_object of include/mmw_radar.h (48 bytes)
OBJ_DTYPE = np.dtype(
    [
        ("frame", "<u4"), ("first_det", "<u4"), ("n_det", "<u4"), ("peak_det", "<u4"),
        ("range_bin", "<f4"), ("doppler_bin", "<f4"), ("angle_rad", "<f4"),
        ("power", "<f4"), ("peak_power", "<f4"), ("peak_noise", "<f4"),
        ("range_min", "<u2"), ("range_max", "<u2"), ("doppler_min", "<i2"), ("doppler_max", "<i2"),
    ]
)
assert DET_DTYPE.itemsize == 24 and OBJ_DTYPE.itemsize == 48


class ClusterParams(C.Structure):
    _fields_ = [("eps_range", C.c_int), ("eps_doppler", C.c_int), ("eps_angle", C.c_int), ("min_points", C.c_int),
                ("max_objects_per_frame", C.c_int)]


_lib = None


def lib():
    global _lib
    if _lib is None:
        out = tempfile.mkdtemp(prefix="mmw_cluster_ref_")
        atexit.register(shutil.rmtree, out, True)
        so = os.path.join(out, "libcluster_ref.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else (shutil.which("gcc") or "gcc")
        subprocess.run([cc, "-std=c99", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Werror",
                        "-I", os.path.join(ROOT, "include"), "-o", so, os.path.join(HERE, "cluster_ref.c")],
                       check=True, capture_output=True)
        L = C.CDLL(so)
        vp = C.c_void_p
        L.ref_cluster.restype = C.c_long
        L.ref_cluster.argtypes = [vp, vp, C.c_int, C.c_int, C.POINTER(ClusterParams), vp, C.c_long, vp,
                                  C.POINTER(C.c_long), C.POINTER(C.c_uint32)]
        _lib = L
    return _lib


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def frame_offsets(dets: np.ndarray, n_frames: int, first_frame: int = 0) -> np.ndarray:
    """[n_frames + 1] start of each frame's records in an ordered detection list"""
    f = dets["frame"].astype(np.int64) - first_frame
    return np.searchsorted(f, np.arange(n_frames + 1)).astype(np.uint32)


def cluster(dets: np.ndarray, offsets: np.ndarray, Cp: int, eps_range=2, eps_doppler=2, eps_angle=4, min_points=1,
            max_objects_per_frame=256):
    """ref_cluster: (objects, labels, n_total, flags) of an ordered detection list; offsets has n_frames + 1 entries."""
    d = np.ascontiguousarray(dets, DET_DTYPE)
    off = np.ascontiguousarray(offsets, np.uint32)
    n_frames = off.size - 1
    prm = ClusterParams(eps_range, eps_doppler, eps_angle, min_points, max_objects_per_frame)
    cap = max(1, n_frames * max_objects_per_frame)
    objs = np.zeros(cap, OBJ_DTYPE)
    n_det = int(off[-1]) if off.size else 0
    labels = np.empty(max(1, n_det), np.int32)
    total, flags = C.c_long(0), C.c_uint32(0)
    n = lib().ref_cluster(_ptr(d), _ptr(off), n_frames, Cp, C.byref(prm), _ptr(objs), cap, _ptr(labels),
                          C.byref(total), C.byref(flags))
    return objs[:n].copy(), labels[:n_det].copy(), total.value, flags.value
