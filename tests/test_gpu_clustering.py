"""Clustering on the GPU (include/mmw_radar.h: mmw_set_clustering, csrc/mmw_cluster.cu): objects and labels byte-equal to
the CPU reference (tests/cluster_ref.c: ref_cluster) run on the GPU's own detection list, on every detection path and batch form;
the detection list unchanged; deterministic under contention, per frame, in graph mode and with batches in flight; the caps
flagged.  Every context of this file is created with MMW_GUARD=1 and must leave every guard band untouched."""
import os

import numpy as np
import pytest

import cluster_ref

pytestmark = pytest.mark.gpu

DEFAULT = dict(eps_range=2, eps_doppler=2, eps_angle=4, min_points=1, max_objects_per_frame=256)
PARAM_SETS = [
    dict(),
    dict(min_points=3),
    dict(eps_range=0, eps_doppler=0, eps_angle=0),          # every object a singleton
    dict(eps_angle=256),                                    # >= n_theta: the angle is ignored
]


@pytest.fixture(scope="module")
def ref():
    return cluster_ref


@pytest.fixture(autouse=True)
def guard_env():
    old = os.environ.get("MMW_GUARD")
    os.environ["MMW_GUARD"] = "1"
    yield
    if old is None:
        os.environ.pop("MMW_GUARD", None)
    else:
        os.environ["MMW_GUARD"] = old


def full(params):
    p = dict(DEFAULT)
    p.update(params)
    return p


def object_header(pkg, ctx):
    import torch

    _, h = ctx.device_objects()
    torch.cuda.synchronize()
    return pkg.sharding.device_bytes_view(h, 32, torch.device("cuda", 0)).cpu().numpy().view(np.uint32).copy()


def guards_clean(pkg, ctx):
    bad = ctx.check_guards()
    assert bad == 0, pkg.api.last_error()


def check_against_reference(pkg, ref, ctx, dets, det_overflow, n_frames, first_frame, params):
    """the context's objects, labels and header against ref_cluster on its own detection list"""
    prm = full(params)
    objs, obj_overflow = ctx.read_objects()
    labels = ctx.read_labels()
    hdr = object_header(pkg, ctx)
    off = ref.frame_offsets(dets, n_frames, first_frame)
    w_objs, w_labels, w_total, w_flags = ref.cluster(dets, off, ctx.Cp, **prm)
    assert labels.size == dets.size
    assert labels.tobytes() == w_labels.tobytes(), f"labels differ at {np.flatnonzero(labels != w_labels)[:5]}"
    assert objs.size == w_objs.size
    if objs.tobytes() != w_objs.tobytes():
        diff = [i for i in range(objs.size) if objs[i].tobytes() != w_objs[i].tobytes()]
        raise AssertionError(f"{len(diff)} objects differ, first {diff[0]}: {objs[diff[0]]} vs {w_objs[diff[0]]}")
    assert hdr[0] == w_objs.size and hdr[1] == w_total and hdr[2] == n_frames
    assert (hdr[3] & 1) == (w_flags & 1) and bool(hdr[3] & 2) == bool(det_overflow)
    assert obj_overflow == bool(hdr[3])
    return objs, labels, hdr


# (S, C, A, frames, keep cube, detect path)
CASES = [
    (512, 256, 12, 8, False, 0),
    (256, 128, 4, 64, False, 1),        # MMW_DETECT_PER_CELL
    (256, 128, 4, 64, False, 2),        # MMW_DETECT_REFFT
    (68, 66, 3, 5, False, 0),           # ragged
    (64, 64, 192, 2, False, 0),         # wide array, fused
    (64, 64, 192, 2, True, 0),          # wide array, cube mode
]


@pytest.mark.parametrize("S,C,A,F,keep,path", CASES)
def test_bit_exact_with_the_reference(pkg, ref, S, C, A, F, keep, path):
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=8)
    with pkg.RadarContext(S, C, A, F, keep_doppler_cube=keep, max_det_per_frame=2048) as ctx:
        if path:
            ctx.set_detect_path(path)
        ctx.set_frame_offset(11)
        for params in PARAM_SETS:
            ctx.set_clustering(**full(params))                  # (no arguments would turn it off)
            dets, overflow = ctx.process_host(adc, F)
            assert dets.size > 0
            objs, _, _ = check_against_reference(pkg, ref, ctx, dets, overflow, F, 11, params)
            assert objs.size > 0
            if params.get("eps_range") == 0:
                assert (objs["n_det"] == 1).all()
        guards_clean(pkg, ctx)


def test_a_large_frame(pkg, ref):
    """tens of thousands of detections in one frame (low alpha): the long per-frame walk and big components"""
    S, C, A, F = 512, 256, 4, 2
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=5, n_targets=8)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=65536, cfar_alpha=1.3) as ctx:
        for params in (dict(max_objects_per_frame=65536), dict(min_points=2, eps_angle=2, max_objects_per_frame=4096)):
            ctx.set_clustering(**params)
            dets, overflow = ctx.process_host(adc, F)
            assert dets.size > 10000 * F and not overflow
            objs, _, _ = check_against_reference(pkg, ref, ctx, dets, overflow, F, 0, params)
            assert objs.size > 100
        guards_clean(pkg, ctx)


def test_detections_unchanged(pkg):
    S, C, A, F = 512, 256, 12, 8
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=4, n_targets=8)
    with pkg.RadarContext(S, C, A, F) as plain, pkg.RadarContext(S, C, A, F) as clus:
        k0 = plain.info.kernels_per_batch
        clus.set_clustering()                                           # off, as a context that never enabled it
        assert clus.info.kernels_per_batch == k0
        clus.set_clustering(min_points=2)
        assert clus.info.kernels_per_batch == k0 + 5
        want, wo = plain.process_host(adc, F)
        got, go = clus.process_host(adc, F)
        assert got.tobytes() == want.tobytes() and wo == go
        assert np.array_equal(clus.read_counts(F), plain.read_counts(F))
        clus.set_clustering()
        assert clus.info.kernels_per_batch == k0
        got2, _ = clus.process_host(adc, F)
        assert got2.tobytes() == want.tobytes()
        with pytest.raises(pkg.RadarError) as ei:                        # off: nothing to read
            clus.read_objects()
        assert ei.value.code == pkg.api.MMW_ERR_STATE
        guards_clean(pkg, clus)


def test_argument_checks(pkg):
    with pkg.RadarContext(128, 64, 4, 2, max_det_per_frame=512) as ctx:
        for kw, needle in [(dict(eps_range=17), "eps_range"), (dict(eps_doppler=-1), "eps_doppler"), (dict(eps_angle=-1), "eps_angle"),
                           (dict(min_points=0), "min_points"), (dict(max_objects_per_frame=0), "max_objects_per_frame"),
                           (dict(max_objects_per_frame=513), "max_objects_per_frame")]:
            with pytest.raises(pkg.RadarError) as ei:
                ctx.set_clustering(**kw)
            assert ei.value.code == pkg.api.MMW_ERR_ARG and needle in str(ei.value)
        with pytest.raises(pkg.RadarError) as ei:
            ctx.device_objects()
        assert ei.value.code == pkg.api.MMW_ERR_STATE
        ctx.set_clustering()
        with pytest.raises(pkg.RadarError) as ei:                        # on, but no clustered batch yet
            ctx.set_clustering(eps_range=1)
            ctx.read_labels()
        assert ei.value.code == pkg.api.MMW_ERR_STATE
        guards_clean(pkg, ctx)


def test_repeatable_and_independent_of_other_contexts(pkg):
    import torch

    S, C, A, F = 512, 256, 12, 8
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=6, n_targets=10)
    dev = torch.from_numpy(adc).cuda()
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=2048) as alone:
        alone.set_clustering(min_points=2)
        alone.process_device(dev, F)
        want_o, _ = alone.read_objects()
        want_l = alone.read_labels()
        for _ in range(3):
            alone.process_device(dev, F)
            o, _ = alone.read_objects()
            assert o.tobytes() == want_o.tobytes() and alone.read_labels().tobytes() == want_l.tobytes()
        guards_clean(pkg, alone)
    ctxs = [pkg.RadarContext(S, C, A, F, max_det_per_frame=2048) for _ in range(3)]
    streams = [torch.cuda.Stream() for _ in ctxs]
    try:
        for c, s in zip(ctxs, streams):
            c.use_stream(s.cuda_stream)
            c.set_clustering(min_points=2)
        for rnd in range(5):
            for c in ctxs:
                c.process_device(dev, F)
            for i, c in enumerate(ctxs):
                o, _ = c.read_objects()
                assert o.tobytes() == want_o.tobytes(), f"round {rnd}, context {i}: objects differ"
                assert c.read_labels().tobytes() == want_l.tobytes(), f"round {rnd}, context {i}: labels differ"
        for c in ctxs:
            guards_clean(pkg, c)
    finally:
        for c in ctxs:
            c.close()


def test_a_frame_alone_gives_the_objects_it_gets_in_a_batch(pkg):
    S, C, A, F = 256, 128, 12, 6
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=7, n_targets=8)
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.set_clustering(**DEFAULT)
        dets, _ = ctx.process_host(adc, F)
        objs, _ = ctx.read_objects()
        off = np.searchsorted(dets["frame"], np.arange(F + 1))
        for f in range(F):
            ctx.set_frame_offset(f)
            ctx.process_host(adc[f:f + 1], 1)
            one, _ = ctx.read_objects()
            mine = objs[objs["frame"] == f].copy()
            mine["first_det"] -= np.uint32(off[f])
            mine["peak_det"] -= np.uint32(off[f])
            assert one.tobytes() == mine.tobytes(), f"frame {f}"
        guards_clean(pkg, ctx)


def test_graph_mode_follows_the_frame_offset(pkg):
    S, C, A, F = 256, 128, 12, 4
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=8, n_targets=8)
    with pkg.RadarContext(S, C, A, 1) as eager, pkg.RadarContext(S, C, A, 1) as graphed:
        for c in (eager, graphed):
            c.set_clustering(min_points=2)
        graphed.set_graph_mode(True)
        for k in range(F):
            for c in (eager, graphed):
                c.set_frame_offset(1000 + k)
                c.process_host(adc[k:k + 1], 1)
            want, _ = eager.read_objects()
            got, _ = graphed.read_objects()
            assert want.size > 0 and (got["frame"] == 1000 + k).all()
            assert got.tobytes() == want.tobytes(), f"frame {k}"
            assert graphed.read_labels().tobytes() == eager.read_labels().tobytes()
        guards_clean(pkg, graphed)


def test_submit_and_wait_with_two_batches_in_flight(pkg):
    S, C, A, F = 256, 128, 4, 16
    adc = [np.ascontiguousarray(pkg.synth.cube_batch(F, S, C, A, cfg=9 + i, n_targets=8)) for i in range(2)]
    with pkg.RadarContext(S, C, A, F) as ref, pkg.RadarContext(S, C, A, F) as a, pkg.RadarContext(S, C, A, F) as b:
        for c in (ref, a, b):
            c.set_clustering(eps_angle=8)
        want = []
        for x in adc:
            ref.process_host(x, F)
            want.append(ref.read_objects()[0])
        a.submit_host(adc[0], F)
        b.submit_host(adc[1], F)
        with pytest.raises(pkg.RadarError) as ei:
            a.read_objects()
        assert ei.value.code == pkg.api.MMW_ERR_STATE
        with pytest.raises(pkg.RadarError) as ei:
            a.set_clustering()
        assert ei.value.code == pkg.api.MMW_ERR_STATE
        b.wait()
        a.wait()
        assert a.read_objects()[0].tobytes() == want[0].tobytes()
        assert b.read_objects()[0].tobytes() == want[1].tobytes()
        guards_clean(pkg, a)
        guards_clean(pkg, b)


def test_caps_are_flagged(pkg, ref):
    S, C, A, F = 512, 256, 12, 3
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=8)
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.set_clustering(max_objects_per_frame=2, eps_range=0, eps_doppler=0)
        dets, overflow = ctx.process_host(adc, F)
        objs, labels, hdr = check_against_reference(pkg, ref, ctx, dets, overflow, F, 0, dict(max_objects_per_frame=2, eps_range=0, eps_doppler=0))
        assert hdr[3] & 1 and hdr[1] > hdr[0] and objs.size == 2 * F
        assert (labels == -1).sum() == dets.size - objs["n_det"].sum() > 0
        guards_clean(pkg, ctx)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=8) as ctx:
        ctx.set_clustering(max_objects_per_frame=8)
        dets, overflow = ctx.process_host(adc, F)
        assert overflow
        _, _, hdr = check_against_reference(pkg, ref, ctx, dets, overflow, F, 0, dict(max_objects_per_frame=8))
        assert hdr[3] & 2
        guards_clean(pkg, ctx)
