"""A memcheck of our own: contexts created with MMW_GUARD=1 bracket every device buffer they own with 4 KB guard bands
(include/mmw_radar.h: mmw_check_guards), and after driving every kernel form of the chain — ragged and padded shapes, fused
mode and cube mode, the antenna-split path of small batches, graph mode, static-clutter removal, the wide-array paths
(selective Doppler re-FFT, measure_wide_kernel), detection-capacity overflow, full batches that end exactly
at the buffers' last byte — not one guard byte may have changed.  compute-sanitizer is closed on this pool
(profiles/r2/compute_sanitizer_refused.log); this catches out-of-bounds WRITES of any kernel, to the byte.  The reference's
own kernels would not pass (acceleration.cu:117-150 reads out of bounds, :152-166 leaves element 12 800 unwritten)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# (S, C, A, frames, keep cube, max detections per frame)
CASES = [
    (512, 256, 12, 6, False, 1024),      # cfg3 kernels, several tiles per warp
    (512, 256, 12, 2, True, 1024),       # cube mode
    (256, 128, 4, 40, False, 512),       # cfg2 kernels
    (256, 128, 12, 1, False, 1024),      # one frame: antenna-split Doppler path + power_sum_kernel
    (100, 128, 4, 3, False, 1024),       # the reference's own frame shape: S and C padded (PAD kernels)
    (68, 66, 3, 5, False, 1024),         # ragged: bare multiples of 4 / 2
    (500, 130, 2, 2, True, 1024),        # ragged + cube
    (1024, 64, 2, 2, False, 1024),       # 1024-point range FFT, 64-point Doppler FFT
    (64, 1024, 1, 2, False, 1024),       # 1024-point Doppler FFT
    (64, 64, 192, 2, False, 4096),       # wide array, fused: rows_kernel + doppler_extract_kernel + angle_fft_kernel<256>
    (64, 64, 192, 2, True, 4096),        # wide array with the cube: measure_wide_kernel
    (128, 128, 65, 2, False, 2048),      # odd antenna count, 128-point angle FFT
    (512, 256, 12, 3, False, 8),         # detection capacity overflow (the list is truncated, nothing may spill)
]


@pytest.fixture()
def guard_env():
    old = os.environ.get("MMW_GUARD")
    os.environ["MMW_GUARD"] = "1"
    yield
    if old is None:
        os.environ.pop("MMW_GUARD", None)
    else:
        os.environ["MMW_GUARD"] = old


@pytest.mark.parametrize("S,C,A,F,keep,cap", CASES)
def test_no_kernel_writes_outside_its_buffers(pkg, guard_env, S, C, A, F, keep, cap):
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=6)
    with pkg.RadarContext(S, C, A, F, keep_doppler_cube=keep, max_det_per_frame=cap) as ctx:
        assert ctx.check_guards() == 0                                  # the bands are in place before any kernel ran
        dets, overflow = ctx.process_host(adc, F)                       # full batch: the last frame ends at the buffers' end
        assert len(dets) > 0 and (overflow or cap > 8)
        ctx.process_host(adc[: max(1, F // 2)], max(1, F // 2))          # short batch
        ctx.set_base_frame(adc[0])                                       # static-clutter removal: K1's BASE instantiation
        ctx.process_host(adc, F)
        ctx.set_base_frame(None)
        if not keep:                                                     # the re-FFT detection path on narrow arrays too
            ctx.set_detect_path(pkg.api.DETECT_REFFT)
            ctx.process_host(adc, F)
            ctx.set_detect_path(pkg.api.DETECT_PER_CELL)
            ctx.process_host(adc, F)
            ctx.set_detect_path(pkg.api.DETECT_AUTO)
        ctx.set_graph_mode(True)                                         # latency mode: one frame per call through a CUDA graph
        for f in range(min(F, 3)):
            ctx.process_host(adc[f:f + 1], 1)
        ctx.set_graph_mode(False)
        ctx.power_map(0)                                                 # export kernels
        if keep:
            ctx.doppler_cube(0)
        bad = ctx.check_guards()
    assert bad == 0, pkg.api.last_error()


def test_guard_check_sees_a_stray_write(pkg, guard_env):
    """the checker itself: one byte written past the end of the power map with a plain device memset must be reported"""
    import torch

    S, C, A, F = 128, 64, 4, 2
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=3)
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.process_host(adc, F)
        assert ctx.check_guards() == 0
        dets_ptr, hdr_ptr = ctx.device_results()
        # the header is the first word of the result block, the band before it ends one byte below
        stray = pkg.sharding.device_bytes_view(hdr_ptr - 1, 1, torch.device("cuda", 0))
        stray.fill_(0)
        torch.cuda.synchronize()
        assert ctx.check_guards() == 1
        assert "before its start" in pkg.api.last_error() and "d_result" in pkg.api.last_error()


def test_guard_check_needs_the_switch(pkg):
    os.environ.pop("MMW_GUARD", None)
    with pkg.RadarContext(128, 64, 4, 1) as ctx:
        with pytest.raises(Exception):
            ctx.check_guards()


def test_repeated_runs_under_contention_give_the_same_bytes(pkg):
    """A race check by repetition (racecheck is part of the closed compute-sanitizer): three contexts on three streams run
    the same batch at the same time, twenty rounds, so the persistent FFT kernels, their tile counters and the in-place
    warp-private Doppler passes of different batches share the SMs in ever different interleavings — every round of every
    context must return the bytes of a context running alone, power map included."""
    import torch

    S, C, A, F = 512, 256, 12, 8
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=8)
    dev = torch.from_numpy(adc).cuda()
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=2048) as alone:
        want, _ = alone.process_host(adc, F)
        want = want.copy()
        pmap = alone.power_map(F - 1).copy()
    ctxs = [pkg.RadarContext(S, C, A, F, max_det_per_frame=2048) for _ in range(3)]
    streams = [torch.cuda.Stream() for _ in ctxs]
    try:
        for c, s in zip(ctxs, streams):
            c.use_stream(s.cuda_stream)
        for rnd in range(20):
            for c in ctxs:                                   # queued back to back: the three batches overlap on the device
                c.process_device(dev, F)
            for i, c in enumerate(ctxs):
                got, _ = c.read_detections()
                assert got.tobytes() == want.tobytes(), f"round {rnd}, context {i}: detection list differs"
            if rnd % 5 == 0:
                assert np.array_equal(ctxs[rnd % 3].power_map(F - 1), pmap)
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("kernel", [2, 1])
def test_legacy_kernels_repeat_bit_for_bit(pkg, kernel):
    """the 8-CTA cluster kernel (DSMEM exchange, cluster barriers) and the one-CTA kernel, 200 calls on the same frame: the
    same raw bin and the same spectrum bytes every time"""
    cap = pkg.synth.legacy_capture(2, seed=5)
    base = np.zeros(12800, np.complex128)
    pkg.api.legacy_configure(kernel_variant=kernel, quiet=1)
    try:
        d0, raw0 = pkg.api.legacy_process_frame(cap[1], base)
        spec0 = pkg.api.legacy_spectrum().tobytes()
        for i in range(200):
            d, raw = pkg.api.legacy_process_frame(cap[1], base)
            assert (d, raw) == (d0, raw0)
            if i % 20 == 0:
                assert pkg.api.legacy_spectrum().tobytes() == spec0
    finally:
        pkg.api.legacy_configure(kernel_variant=0)
