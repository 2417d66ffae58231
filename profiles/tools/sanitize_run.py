"""Small self-checking run sized for compute-sanitizer (memcheck / racecheck / synccheck): the chain on a small cube with both
CFAR kernels (the walk form of the default window, the tiled one of another window), submit/wait, graph mode with advancing frame offsets, the wide-array path (selective Doppler re-FFT + angle
FFT) and the warp-private Doppler kernel, and one legacy frame through both legacy kernels (the 8-CTA DSMEM cluster included).
    [compute-sanitizer --tool memcheck|racecheck|synccheck] python profiles/tools/sanitize_run.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
S, C, A, F = 256, 128, 4, 2
adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=5)
for window in ({}, {"cfar_guard": (1, 3), "cfar_train": (5, 2)}):
    with pkg.RadarContext(S, C, A, F, **window) as ctx:
        dets, _ = ctx.process_host(adc, F)
        ctx.submit_host(adc, F)
        again, _ = ctx.wait()
    assert again.tobytes() == dets.tobytes()
    print("CFAR window", window or "default", len(dets), "detections")
with pkg.RadarContext(512, 64, 12, 1) as ctx:                       # 128-bin strips of a 512-bin map, one frame
    print("512 x 64 x 12:", len(ctx.process_host(pkg.synth.cube_batch(1, 512, 64, 12, cfg=3, n_targets=5), 1)[0]), "detections")
with pkg.RadarContext(256, 256, 2, 4) as ctx:                       # 256-point Doppler FFT, fused: the warp-private kernel (in-place pass 1)
    print("256 x 256 x 2:", len(ctx.process_host(pkg.synth.cube_batch(4, 256, 256, 2, cfg=3, n_targets=5), 4)[0]), "detections")
wide = pkg.synth.cube_batch(2, 64, 64, 40, cfg=3, n_targets=4)      # A >= 32: rows_kernel + doppler_extract_kernel + angle_fft_kernel
with pkg.RadarContext(64, 64, 40, 2) as ctx:
    dw, _ = ctx.process_host(wide, 2)
    print("64 x 64 x 40 (wide path):", len(dw), "detections")
    ctx.set_graph_mode(True)
    for f in range(3):                                              # eager, capture, replay with a patched frame offset
        ctx.set_frame_offset(10 * f)
        g, _ = ctx.process_host(wide, 2)
        assert np.array_equal(g["frame"], dw["frame"] + 10 * f) and np.array_equal(g["angle_bin"], dw["angle_bin"])
cap = pkg.synth.legacy_capture(3, seed=3)
base = np.zeros(12800, np.complex128)
out = []
for var in (2, 1):
    pkg.api.legacy_configure(kernel_variant=var, quiet=1)
    out.append(pkg.api.legacy_process_frame(cap[1], base))
    out.append(pkg.api.legacy_process_frame(cap[2][:51300], base))
assert out[:2] == out[2:], out
print("legacy", out[:2])
