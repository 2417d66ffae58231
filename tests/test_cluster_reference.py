"""The clustering definition (tests/cluster_ref.c: ref_cluster) checked without a GPU: its components against scipy's
connected components of the same neighbour graph built independently here, its sums against a Python loop in index order,
the record layout against include/mmw_radar.h, and mmw_objects_to_physical (host arithmetic) against mmw_to_physical."""
import os
import subprocess

import numpy as np
import pytest
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

import cluster_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ref():
    return cluster_ref


def random_list(rng, n_frames, Sp, Cp, n_blobs, blob_r, blob_d, n_theta=64, angle_spread=6, straddle=False, first_frame=0):
    """An ordered detection list of blobs of cells: unique (range, doppler) per frame, sorted by (frame, range, doppler)."""
    from cluster_ref import DET_DTYPE

    recs = []
    for f in range(n_frames):
        cells = {}
        for _ in range(n_blobs):
            r0 = int(rng.integers(0, Sp))
            d0 = (Cp // 2 + int(rng.integers(-4, 4))) % Cp if straddle else int(rng.integers(0, Cp))
            a0 = int(rng.integers(-n_theta // 2, n_theta // 2))
            for _ in range(int(rng.integers(1, 3 * blob_r * blob_d + 2))):
                r = r0 + int(rng.integers(-blob_r, blob_r + 1))
                d = (d0 + int(rng.integers(-blob_d, blob_d + 1))) % Cp
                if 0 <= r < Sp:
                    a = int(np.clip(a0 + rng.integers(-angle_spread, angle_spread + 1), -n_theta // 2, n_theta // 2 - 1))
                    cells[(r, d)] = a
        for (r, d) in sorted(cells):
            recs.append((first_frame + f, r, d, np.float32(rng.uniform(1, 1e4) * (1 + (rng.random() < 0.1) * 1e3)),
                         np.float32(rng.uniform(0.1, 10)), cells[(r, d)], 0,
                         np.float32(np.arcsin(cells[(r, d)] * 2.0 / n_theta))))
    return np.array(recs, DET_DTYPE)


def expected(dets, offsets, Cp, eps_range, eps_doppler, eps_angle, min_points, max_objects_per_frame):
    """(labels, n_total, cut) from scipy's connected components of the neighbour graph"""
    labels = np.full(dets.size, -1, np.int32)
    n_obj, n_total, cut = 0, 0, False
    for f in range(offsets.size - 1):
        s, e = int(offsets[f]), int(offsets[f + 1])
        if e == s:
            continue
        fd = dets[s:e]
        r = fd["range_bin"].astype(np.int64)
        d = fd["doppler_bin"].astype(np.int64)
        d = np.where(d < Cp // 2, d, d - Cp)
        a = fd["angle_bin"].astype(np.int64)
        adj = ((np.abs(r[:, None] - r[None, :]) <= eps_range) & (np.abs(d[:, None] - d[None, :]) <= eps_doppler)
               & (np.abs(a[:, None] - a[None, :]) <= eps_angle))
        _, comp = connected_components(csr_matrix(adj), directed=False)
        first = {}
        for i, c in enumerate(comp):
            first.setdefault(c, i)
        sizes = np.bincount(comp)
        k = 0
        for c, i0 in sorted(first.items(), key=lambda kv: kv[1]):
            if sizes[c] < min_points:
                continue
            n_total += 1
            if k >= max_objects_per_frame:
                cut = True
                continue
            labels[s:e][comp == c] = n_obj
            n_obj += 1
            k += 1
    return labels, n_total, cut


CASES = [
    # (name, frames, Sp, Cp, blobs, blob_r, blob_d, straddle, params)
    ("dense", 5, 64, 64, 12, 3, 3, False, dict()),
    ("eps0", 4, 128, 64, 10, 2, 2, False, dict(eps_range=0, eps_doppler=0, eps_angle=0)),
    ("straddle", 4, 64, 128, 6, 2, 4, True, dict()),
    ("min_points", 5, 128, 128, 20, 2, 2, False, dict(min_points=3)),
    ("cap", 4, 64, 64, 30, 1, 1, False, dict(max_objects_per_frame=5)),
    ("no_angle", 3, 64, 64, 15, 3, 2, False, dict(eps_angle=64)),
    ("wide", 3, 256, 256, 25, 4, 5, False, dict(eps_range=3, eps_doppler=4, eps_angle=2)),
]


@pytest.mark.parametrize("name,F,Sp,Cp,nb,br,bd,straddle,params", CASES, ids=[c[0] for c in CASES])
def test_components_match_scipy(ref, name, F, Sp, Cp, nb, br, bd, straddle, params):
    rng = np.random.default_rng(abs(hash(name)) % 2**32)
    prm = dict(eps_range=2, eps_doppler=2, eps_angle=4, min_points=1, max_objects_per_frame=256)
    prm.update(params)
    dets = random_list(rng, F, Sp, Cp, nb, br, bd, straddle=straddle, first_frame=7)
    off = ref.frame_offsets(dets, F, first_frame=7)
    objs, labels, n_total, flags = ref.cluster(dets, off, Cp, **prm)
    want, want_total, want_cut = expected(dets, off, Cp, **prm)
    assert np.array_equal(labels, want)
    assert n_total == want_total and bool(flags & 1) == want_cut
    assert objs.size == want.max() + 1 if want.size and want.max() >= 0 else objs.size == 0
    for o, ob in enumerate(objs):
        members = np.flatnonzero(labels == o)
        assert ob["first_det"] == members[0] and ob["n_det"] == members.size
        assert ob["frame"] == dets[members[0]]["frame"]
    if name == "straddle":                                # d' has no wrap: blobs across +-Cp/2 are split
        d = dets["doppler_bin"].astype(int)
        d = np.where(d < Cp // 2, d, d - Cp)
        assert (d > Cp // 4).any() and (d < -Cp // 4).any()
        for o in range(objs.size):
            sd = d[labels == o]
            assert not (sd.max() > Cp // 4 and sd.min() < -Cp // 4)
    if name == "cap":
        assert flags & 1 and n_total > objs.size
    if name == "eps0":
        assert (objs["n_det"] == 1).all()


def test_sums_follow_index_order(ref):
    rng = np.random.default_rng(5)
    Cp = 128
    dets = random_list(rng, 3, 128, Cp, 10, 3, 3)
    off = ref.frame_offsets(dets, 3)
    objs, labels, _, _ = ref.cluster(dets, off, Cp)
    assert objs.size > 0 and objs["n_det"].max() > 3
    for o, ob in enumerate(objs):
        sp = sr = sd = sa = 0.0
        peak = None
        rs, ds = [], []
        for i in np.flatnonzero(labels == o):                  # ascending index, fp64 (Python floats)
            p = float(dets[i]["power"])
            d = int(dets[i]["doppler_bin"])
            d = d if d < Cp // 2 else d - Cp
            sp += p
            sr += p * float(dets[i]["range_bin"])
            sd += p * float(d)
            sa += p * float(dets[i]["angle_rad"])
            if peak is None or dets[i]["power"] > dets[peak]["power"]:
                peak = i
            rs.append(int(dets[i]["range_bin"]))
            ds.append(d)
        assert ob["power"] == np.float32(sp)
        assert ob["range_bin"] == np.float32(sr / sp)
        assert ob["doppler_bin"] == np.float32(sd / sp)
        assert ob["angle_rad"] == np.float32(sa / sp)
        assert ob["peak_det"] == peak and ob["peak_power"] == dets[peak]["power"] and ob["peak_noise"] == dets[peak]["noise"]
        assert (ob["range_min"], ob["range_max"], ob["doppler_min"], ob["doppler_max"]) == (min(rs), max(rs), min(ds), max(ds))


def test_equal_power_peak_is_the_lower_index(ref):
    from cluster_ref import DET_DTYPE

    dets = np.array([(0, 5, 3, 7.0, 1.0, 0, 0, 0.0), (0, 5, 4, 9.0, 1.0, 0, 0, 0.0), (0, 6, 3, 9.0, 2.0, 0, 0, 0.0)], DET_DTYPE)
    objs, labels, _, _ = ref.cluster(dets, np.array([0, 3], np.uint32), 64)
    assert objs.size == 1 and objs[0]["peak_det"] == 1 and objs[0]["peak_noise"] == 1.0 and (labels == 0).all()


def test_object_layout_matches_header(pkg, ref, tmp_path):
    src = tmp_path / "off.c"
    names = pkg.api.OBJ_DTYPE.names
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "mmw_radar.h"\nint main(void){printf("%zu'
                   + "".join(" %zu" for _ in names) + '\\n", sizeof(mmw_object)'
                   + "".join(f", offsetof(mmw_object, {n})" for n in names) + ");return 0;}\n")
    exe = tmp_path / "off"
    r = subprocess.run(["/usr/bin/gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True).stdout.split()]
    assert got == [pkg.api.OBJ_DTYPE.itemsize] + [pkg.api.OBJ_DTYPE.fields[n][1] for n in names]
    assert pkg.api.OBJ_DTYPE == ref.OBJ_DTYPE and pkg.api.DET_DTYPE == ref.DET_DTYPE
    assert [f[0] for f in pkg.api.ClusterParams._fields_] == [f[0] for f in ref.ClusterParams._fields_]


def test_default_cluster_params(pkg):
    cp = pkg.api.default_cluster_params()
    assert (cp.eps_range, cp.eps_doppler, cp.eps_angle, cp.min_points, cp.max_objects_per_frame) == (2, 2, 4, 1, 256)


@pytest.mark.parametrize("Sp,Cp", [(256, 128), (512, 256), (64, 1024)])
def test_single_detection_objects_convert_like_detections(pkg, ref, Sp, Cp):
    rng = np.random.default_rng(Sp + Cp)
    dets = random_list(rng, 3, Sp, Cp, 20, 2, 2)
    off = ref.frame_offsets(dets, 3)
    objs, labels, _, _ = ref.cluster(dets, off, Cp, eps_range=0, eps_doppler=0, eps_angle=0, max_objects_per_frame=100000)
    assert (objs["n_det"] == 1).all() and objs.size == dets.size
    t_det = pkg.api.to_physical(dets[objs["first_det"]], Sp, Cp)
    t_obj = pkg.api.objects_to_physical(objs, Sp, Cp)
    for k in ("frame", "range_m", "velocity_mps", "angle_deg", "snr_db"):
        assert t_obj[k].tobytes() == t_det[k].tobytes(), k
    assert (t_obj["flags"] == 0).all()


def test_objects_to_physical_checks_arguments(pkg):
    with pytest.raises(pkg.RadarError) as ei:
        pkg.api.objects_to_physical(np.zeros(1, pkg.api.OBJ_DTYPE), 0, 128)
    assert ei.value.code == pkg.api.MMW_ERR_ARG
    assert pkg.api.objects_to_physical(np.zeros(0, pkg.api.OBJ_DTYPE), 256, 128).size == 0
