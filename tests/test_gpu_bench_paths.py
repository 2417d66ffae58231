"""GPU parity on the EXACT kernel instantiations and batch sizes bench.py times (BASELINE.json configs 2-5): whole
power maps, CFAR masks and detection lists of the CUDA chain, called through the C ABI, against the CPU oracle.

test_gpu_parity.py sweeps shapes at 1-2 frames per batch; at those sizes the launchers pick other kernel forms than the
bench does (the antenna-split Doppler path, run-time-stride twins of the specialised kernels, narrow CFAR strips).
Here the batch sizes are the bench's, so the kernels checked are the kernels timed:

  cfg3  512 x 256 x 12, 64 frames   range<512,..,CT=256>, doppler_fft_warp_kernel<256,..,SPT=512,2> with A = 12 accumulated
                                    in registers over several tiles per warp, cfar_walk<256-bin strips>, measure_kernel
  cfg2  256 x 128 x 4, 1024 frames  range<256, 32-row tiles>, doppler<128,..,SPT=256>, cfar_walk, measure_kernel; two
                                    sampled frames (the oracle is run on those two only)
  cfg5  256 x 128 x 12, 8 frames    the per-sensor cube as a batch, and 1 frame per call through the antenna-split path
                                    + CUDA graph (what the streaming bench runs)
  cfg4  1024 x 512 x 192, 1 frame   range<1024,..,CT=512>, doppler<512,..,SPT=1024, in place, 3 stages>,
                                    measure_wide_kernel / the selective Doppler re-FFT, 256-point angle FFT

Tolerances: tests/chain_check.py, which holds the comparison (check_frames) this file and test_gpu_kernel_forms.py share.
"""
import numpy as np
import pytest

from chain_check import check_frames

pytestmark = pytest.mark.gpu


def _torch_batch(pkg, F, S, C, A, cfg, first_frame=0, n_targets=8):
    import torch

    t = pkg.synth.cube_batch_torch(F, S, C, A, torch.device("cuda", 0), cfg=cfg, first_frame=first_frame, n_targets=n_targets)
    out = t.cpu().numpy()
    del t
    torch.cuda.empty_cache()
    return out


def test_cfg3_bench_batch_fused(pkg, orc):
    """cfg3 at the bench's 64 frames per batch, fused mode: every frame's power map, mask and list against the oracle"""
    S, C, A, F = 512, 256, 12, 64
    adc = _torch_batch(pkg, F, S, C, A, cfg=3)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096) as ctx:
        dets, overflow = ctx.process_host(adc, F)
        assert not overflow
        check_frames(pkg, orc, ctx, dets, adc, list(range(F)), S, C, A, "cfg3 x64 fused", n_threads=16)
        # the device-resident entry point the bench times gives the same bytes
        import torch

        dev = torch.from_numpy(adc).cuda()
        ctx.process_device(dev, F)
        again, _ = ctx.read_detections()
        assert again.tobytes() == dets.tobytes()


def test_cfg3_bench_batch_with_cube(pkg, orc):
    """the same batch with the Doppler cube materialised (CTA-shared Doppler kernel, detections measured from the cube)"""
    S, C, A, F = 512, 256, 12, 16
    adc = _torch_batch(pkg, F, S, C, A, cfg=3)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096, keep_doppler_cube=True) as ctx:
        dets, overflow = ctx.process_host(adc, F)
        assert not overflow
        check_frames(pkg, orc, ctx, dets, adc, [0, 7, 15], S, C, A, "cfg3 x16 cube", n_threads=8)


def test_cfg2_bench_batch_sampled_frames(pkg, orc):
    """cfg2 at the bench's 1024 frames per batch, on the detection path the bench selects for it (MMW_DETECT_REFFT: hit rows
    re-transformed once, angle spectra as FFTs) and on the library's default for narrow arrays (a DFT per detection); the
    oracle checks two sampled frames of each, and the two lists must agree on everything but angle bins at near ties"""
    S, C, A, F = 256, 128, 4, 1024
    adc = _torch_batch(pkg, F, S, C, A, cfg=2)
    lists = {}
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096) as ctx:
        for path, tag in ((pkg.api.DETECT_REFFT, "re-FFT"), (pkg.api.DETECT_PER_CELL, "per-cell")):
            ctx.set_detect_path(path)
            assert int(ctx.info.kernels_per_batch) == (7 if path == pkg.api.DETECT_REFFT else 5)
            dets, overflow = ctx.process_host(adc, F)
            assert not overflow
            check_frames(pkg, orc, ctx, dets, adc, [517, 1023], S, C, A, f"cfg2 x1024 {tag}")
            lists[path] = dets.copy()
    a, b = lists[pkg.api.DETECT_REFFT], lists[pkg.api.DETECT_PER_CELL]
    assert len(a) == len(b)
    for field in ("frame", "range_bin", "doppler_bin", "power", "noise", "flags"):
        assert np.array_equal(a[field], b[field]), field
    differ = int((a["angle_bin"] != b["angle_bin"]).sum())
    print(f"\ncfg2 x1024: {len(a)} detections, angle bins differing between the two detection paths (near ties): {differ}")
    assert differ <= len(a) // 1000 + 2


def test_cfg5_sensor_cube_batch_and_single_calls(pkg, orc):
    """cfg5's 256 x 128 x 12 cube: 8 frames as one batch, and one frame per call (antenna-split Doppler path, CUDA graph,
    advancing frame offsets replaying one graph)"""
    S, C, A, F = 256, 128, 12, 8
    adc = _torch_batch(pkg, F, S, C, A, cfg=5)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096) as ctx:
        dets, overflow = ctx.process_host(adc, F)
        assert not overflow
        check_frames(pkg, orc, ctx, dets, adc, list(range(F)), S, C, A, "cfg5 x8")
    for graph in (False, True):
        with pkg.RadarContext(S, C, A, 1, max_det_per_frame=4096) as ctx:
            ctx.set_graph_mode(graph)
            singles = []
            for f in range(F):
                ctx.set_frame_offset(f)
                singles.append(ctx.process_host(adc[f], 1)[0].copy())
            one = np.concatenate(singles)
            assert one.tobytes() == dets.tobytes(), f"one frame per call (graph={graph}) differs from the batch"
            ctx.set_frame_offset(0)
            d0, _ = ctx.process_host(adc[3], 1)
            check_frames(pkg, orc, ctx, d0, adc[3:4], [0], S, C, A, f"cfg5 single call graph={graph}")


def test_cfg4_full_imaging_frame(pkg, orc):
    """one full 1024 x 512 x 192 frame (403 MB of int16): the cfg4 instantiations of every kernel"""
    S, C, A, F = 1024, 512, 192, 1
    adc = _torch_batch(pkg, F, S, C, A, cfg=4)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=32768) as ctx:
        dets, overflow = ctx.process_host(adc, F)
        assert not overflow
        counts = ctx.read_counts(F)
        assert counts[0] == len(dets) > 0
        check_frames(pkg, orc, ctx, dets, adc, [0], S, C, A, "cfg4 x1", n_threads=1)
