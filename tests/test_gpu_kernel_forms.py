"""Every kernel form the launchers can pick, checked against the fp64 oracle with the strict metric of chain_check.py.

The chain is a set of template instantiations, and the launchers pick one per stage from the shape, the batch size and
the mode: K1's PAD / compile-time-chirp (CT) / static-clutter (BASE) forms, K2's tiled or warp-private kernel with its
PAD and compile-time-Sp (SPT) forms and the antenna-split path of small batches, and the per-cell or re-FFT detection
path.  test_gpu_parity.py sweeps shapes at 1-2 frames per batch and test_gpu_bench_paths.py runs the bench's shapes;
between them many forms that users reach with legal shapes were never compared with a reference.

CASES below names, per case, the forms it is meant to reach; the case runs one batch built from 3 synthetic frames tiled
to F (so the oracle runs only on the frames it checks), records the kernels it launched with torch.profiler, asserts
that the named forms are among them, and compares the first and last frames with orc.process_frames.  A change to a
launcher rule that reroutes a case fails here instead of silently leaving a form unchecked.  Batch sizes: F is past the
antenna-split threshold (n_frames * Sp / 16 * 2 > 148 SMs) wherever the antennas are meant to be accumulated inside K2.
The antenna-split path launches the same K2 instantiation (A is a run-time argument) once per antenna and then
power_sum_kernel, so a multi-antenna case that does not name power_sum_kernel must not launch it: otherwise K2's own
antenna sum went unchecked.  Chirp counts leave the last chirp tile of K1 ragged for that form's tile height (16 / 32
rows; 16 / 8 / 4 with BASE).

test_every_compiled_kernel_is_checked compares the kernels compiled into the library (cuobjdump) with the union of
what CASES launched and EXEMPT, the kernels (by exact name) whose reference check lives in another test: a kernel
form added later needs a case here (or an entry naming its test) before it passes.
"""
import numpy as np
import pytest

from chain_check import WALK_FORMS, cfar_form_name, check_frames, compiled_forms, launched_kernels

pytestmark = pytest.mark.gpu

# (S, C, A, F, mode, detect path, forms the case must launch).  mode: "fused" (power map only), "cube" (Doppler cube
# kept), "base" (cube kept, static-clutter removal: K1's BASE forms).  Forms are written as in the demangled kernel name,
# without the namespace and the parameter list.
CASES = [
    # ---- fused, default detection path (per-cell DFT for A < 32) and the re-FFT path
    (36, 34, 3, 20, "fused", "auto", ["range_fft_kernel<64, 8, 8, 16, 4, true, true, 0, false>",
                                      "doppler_fft_kernel<64, 8, 8, 16, 4, true, 0, 2, false>", "measure_kernel"]),
    (36, 34, 3, 20, "fused", "refft", ["range_fft_kernel<64, 8, 8, 16, 4, true, true, 0, false>",
                                       "doppler_fft_kernel<64, 8, 8, 16, 4, true, 0, 2, false>", "rows_kernel",
                                       "doppler_extract_kernel<64, 8, 8, 8, 4, true>", "angle_fft_kernel<64, 8, 8>"]),
    (200, 130, 4, 6, "fused", "auto", ["range_fft_kernel<256, 16, 16, 32, 8, true, true, 0, false>",
                                       "doppler_fft_warp_kernel<256, 16, 16, 8, true, 0, 2, 2>", "measure_kernel"]),
    (200, 130, 4, 6, "fused", "refft", ["range_fft_kernel<256, 16, 16, 32, 8, true, true, 0, false>",
                                        "doppler_fft_warp_kernel<256, 16, 16, 8, true, 0, 2, 2>",
                                        "doppler_extract_kernel<256, 16, 16, 8, 8, true>"]),
    (256, 256, 4, 5, "fused", "auto", ["range_fft_kernel<256, 16, 16, 32, 8, true, false, 0, false>",
                                       "doppler_fft_warp_kernel<256, 16, 16, 8, false, 0, 2, 2>", "measure_kernel"]),
    (256, 256, 4, 5, "fused", "refft", ["range_fft_kernel<256, 16, 16, 32, 8, true, false, 0, false>",
                                        "doppler_fft_warp_kernel<256, 16, 16, 8, false, 0, 2, 2>",
                                        "doppler_extract_kernel<256, 16, 16, 8, 8, false>"]),
    (300, 300, 2, 3, "fused", "auto", ["range_fft_kernel<512, 16, 32, 16, 8, true, true, 0, false>",
                                       "doppler_fft_kernel<512, 16, 32, 8, 8, true, 0, 3, true>", "measure_kernel"]),
    (300, 300, 2, 3, "fused", "refft", ["range_fft_kernel<512, 16, 32, 16, 8, true, true, 0, false>",
                                        "doppler_fft_kernel<512, 16, 32, 8, 8, true, 0, 3, true>",
                                        "doppler_extract_kernel<512, 16, 32, 8, 8, true>"]),
    (1000, 1000, 2, 2, "fused", "auto", ["range_fft_kernel<1024, 32, 32, 16, 16, false, true, 0, false>",
                                         "doppler_fft_kernel<1024, 32, 32, 8, 8, true, 0, 2, false>", "measure_kernel"]),
    (1000, 1000, 2, 2, "fused", "refft", ["range_fft_kernel<1024, 32, 32, 16, 16, false, true, 0, false>",
                                          "doppler_fft_kernel<1024, 32, 32, 8, 8, true, 0, 2, false>",
                                          "doppler_extract_kernel<1024, 32, 32, 8, 8, true>"]),
    (1024, 1024, 2, 2, "fused", "auto", ["range_fft_kernel<1024, 32, 32, 16, 16, false, false, 0, false>",
                                         "doppler_fft_kernel<1024, 32, 32, 8, 8, false, 0, 2, false>", "measure_kernel"]),
    (1024, 1024, 2, 2, "fused", "refft", ["range_fft_kernel<1024, 32, 32, 16, 16, false, false, 0, false>",
                                          "doppler_fft_kernel<1024, 32, 32, 8, 8, false, 0, 2, false>",
                                          "doppler_extract_kernel<1024, 32, 32, 8, 8, false>"]),
    # the compile-time-shape forms of the bench configurations, at small batches
    (256, 128, 4, 5, "fused", "auto", ["range_fft_kernel<256, 16, 16, 32, 8, true, false, 128, false>",
                                       "doppler_fft_kernel<128, 8, 16, 16, 4, false, 256, 2, false>", "measure_kernel"]),
    (256, 128, 4, 5, "fused", "refft", ["range_fft_kernel<256, 16, 16, 32, 8, true, false, 128, false>",
                                        "doppler_fft_kernel<128, 8, 16, 16, 4, false, 256, 2, false>",
                                        "doppler_extract_kernel<128, 8, 16, 8, 4, false>"]),
    (512, 256, 2, 3, "fused", "auto", ["range_fft_kernel<512, 16, 32, 16, 8, true, false, 256, false>",
                                       "doppler_fft_warp_kernel<256, 16, 16, 8, false, 512, 2, 2>"]),
    (1024, 512, 2, 2, "fused", "auto", ["range_fft_kernel<1024, 32, 32, 16, 16, false, false, 512, false>",
                                        "doppler_fft_kernel<512, 16, 32, 8, 8, false, 1024, 3, true>", "measure_kernel"]),
    (1024, 512, 2, 2, "fused", "refft", ["doppler_fft_kernel<512, 16, 32, 8, 8, false, 1024, 3, true>",
                                         "doppler_extract_kernel<512, 16, 32, 8, 8, false>"]),
    (512, 128, 3, 3, "fused", "auto", ["range_fft_kernel<512, 16, 32, 16, 8, true, false, 0, false>",
                                       "doppler_fft_kernel<128, 8, 16, 16, 4, false, 0, 2, false>"]),
    # antenna-split batches (one single-antenna K2 pass per antenna, then the ordered sum)
    (68, 66, 3, 2, "fused", "refft", ["range_fft_kernel<128, 8, 16, 16, 4, true, true, 0, false>",
                                      "doppler_fft_kernel<128, 8, 16, 16, 4, true, 0, 2, false>", "power_sum_kernel",
                                      "doppler_extract_kernel<128, 8, 16, 8, 4, true>"]),
    # wide arrays (A >= 32: the re-FFT path by default, 128- and 256-point angle FFTs; the wide per-cell kernel)
    (64, 64, 72, 2, "fused", "auto", ["range_fft_kernel<64, 8, 8, 16, 4, true, false, 0, false>", "power_sum_kernel",
                                      "doppler_extract_kernel<64, 8, 8, 8, 4, false>", "angle_fft_kernel<128, 8, 16>"]),
    (64, 64, 72, 2, "fused", "per_cell", ["doppler_fft_kernel<64, 8, 8, 16, 4, false, 0, 2, false>", "power_sum_kernel",
                                          "measure_wide_kernel"]),
    (64, 66, 130, 2, "fused", "auto", ["power_sum_kernel", "doppler_extract_kernel<128, 8, 16, 8, 4, true>",
                                       "angle_fft_kernel<256, 16, 16>"]),
    # ---- cube mode: the CTA-shared Doppler kernel also stores the cube; detections measured from it
    (60, 60, 2, 2, "cube", "auto", ["range_fft_kernel<64, 8, 8, 16, 4, true, true, 0, false>",
                                    "doppler_fft_kernel<64, 8, 8, 16, 4, true, 0, 2, false>", "measure_kernel"]),
    (256, 256, 4, 2, "cube", "auto", ["doppler_fft_kernel<256, 16, 16, 16, 8, false, 0, 2, false>"]),
    (512, 256, 2, 2, "cube", "auto", ["doppler_fft_kernel<256, 16, 16, 16, 8, false, 512, 2, false>"]),
    (256, 512, 2, 2, "cube", "auto", ["range_fft_kernel<256, 16, 16, 32, 8, true, false, 0, false>",
                                      "doppler_fft_kernel<512, 16, 32, 8, 8, false, 0, 3, true>"]),
    (128, 128, 2, 2, "cube", "auto", ["range_fft_kernel<128, 8, 16, 16, 4, true, false, 128, false>",
                                      "doppler_fft_kernel<128, 8, 16, 16, 4, false, 128, 2, false>"]),
    (128, 64, 2, 2, "cube", "auto", ["range_fft_kernel<128, 8, 16, 16, 4, true, false, 0, false>",
                                     "doppler_fft_kernel<64, 8, 8, 16, 4, false, 0, 2, false>"]),
    # ---- static-clutter removal (base frame), cube mode: K1's BASE forms have their own tile heights
    (36, 34, 2, 2, "base", "auto", ["range_fft_kernel<64, 8, 8, 16, 4, true, true, 0, true>"]),
    (64, 64, 2, 2, "base", "auto", ["range_fft_kernel<64, 8, 8, 16, 4, true, false, 0, true>"]),
    (100, 64, 2, 2, "base", "auto", ["range_fft_kernel<128, 8, 16, 16, 4, true, true, 0, true>"]),
    (128, 128, 2, 2, "base", "auto", ["range_fft_kernel<128, 8, 16, 16, 4, true, false, 0, true>"]),
    (200, 130, 2, 2, "base", "auto", ["range_fft_kernel<256, 16, 16, 16, 4, true, true, 0, true>",
                                      "doppler_fft_kernel<256, 16, 16, 16, 8, true, 0, 2, false>"]),
    (256, 64, 2, 2, "base", "auto", ["range_fft_kernel<256, 16, 16, 16, 4, true, false, 0, true>"]),
    (300, 300, 2, 2, "base", "auto", ["range_fft_kernel<512, 16, 32, 8, 4, true, true, 0, true>"]),
    (512, 64, 2, 2, "base", "auto", ["range_fft_kernel<512, 16, 32, 8, 4, true, false, 0, true>"]),
    (1000, 998, 2, 1, "base", "auto", ["range_fft_kernel<1024, 32, 32, 4, 4, false, true, 0, true>"]),
    (1024, 64, 2, 1, "base", "auto", ["range_fft_kernel<1024, 32, 32, 4, 4, false, false, 0, true>"]),
]

# compiled kernels whose reference check lives in another test, by exact name -> that test
EXEMPT = {
    "(anonymous namespace)::legacy_frame_kernel": "test_gpu_parity.py::test_legacy_matches_golden_and_oracle",
    "(anonymous namespace)::legacy_cluster_kernel": "test_gpu_parity.py::test_legacy_matches_golden_and_oracle",
    **{f"cluster_{k}_kernel": "test_gpu_clustering.py::test_bit_exact_with_the_reference"
       for k in ("init", "link", "flatten", "order", "object")},
    "merge_kernel": "test_gpu_properties.py::test_merge_of_gathered_rank_blocks_equals_unsharded",
    # the tiled CFAR kernel and every walk form (WALK_FORMS), each asserted launched there
    **{cfar_form_name(f): "test_gpu_parity.py::test_cfar_kernel_forms_agree_with_oracle" for f in WALK_FORMS},
}


def case_id(c):
    S, C, A, F, mode, path, _ = c
    return f"{S}x{C}x{A}-F{F}-{mode}-{path}"


def _batch(pkg, S, C, A, F, mode):
    """3 synthetic frames tiled to F; with a base frame, the frames carry a static scene and the base is that scene
    (both halved, so that frame - base fits int16 as the capture format requires)"""
    three = pkg.synth.cube_batch(3, S, C, A, cfg=3, n_targets=6)
    base = None
    if mode == "base":
        static = pkg.synth.cube(77, S, C, A, cfg=6, n_targets=2)
        three = (three.astype(np.int32) // 2 + static.astype(np.int32)[None, :] // 2).astype(np.int16)
        base = (static.astype(np.int32) // 2).astype(np.int16)
    return np.ascontiguousarray(three[np.arange(F) % 3]), base


_LAUNCHED = {}            # case id -> library kernels the case launched (filled by _run, read by the coverage test)


def _run(pkg, orc, case, compiled):
    S, C, A, F, mode, path, forms = case
    tag = case_id(case)
    adc, base = _batch(pkg, S, C, A, F, mode)
    frames = sorted({0, F - 1})
    keep = mode != "fused"
    paths = {"auto": pkg.api.DETECT_AUTO, "refft": pkg.api.DETECT_REFFT, "per_cell": pkg.api.DETECT_PER_CELL}
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096, keep_doppler_cube=keep) as ctx:
        ctx.set_detect_path(paths[path])
        if base is not None:
            ctx.set_base_frame(base)
        with launched_kernels() as names:
            dets, overflow = ctx.process_host(adc, F)
            dets = dets.copy()
            ctx.power_map(frames[-1])
            ctx.cfar_mask(frames[-1])
            cubes = {f: ctx.doppler_cube(f) for f in frames} if keep else {}
        ours = names & compiled
        assert ours, f"{tag}: the profiler saw none of the library's kernels (saw {sorted(names)[:5]})"
        _LAUNCHED[tag] = ours
        print(f"\n{tag}: launched {sorted(ours)}")
        missing = [k for k in forms if k not in ours]
        assert not missing, f"{tag}: did not launch {missing}; a launcher rule now routes this case elsewhere"
        if A > 1 and "power_sum_kernel" not in forms:
            assert "power_sum_kernel" not in ours, f"{tag}: took the antenna-split path; K2's antenna sum is not checked"
        assert not overflow
        check_frames(pkg, orc, ctx, dets, adc, frames, S, C, A, tag, n_threads=4, base=base)
        for f, cube in cubes.items():                    # the exported cube is the one the power map was summed from
            P = ctx.power_map(f).astype(np.float64)
            s = (np.abs(cube.astype(np.complex128)) ** 2).sum(0)
            assert np.abs(s - P).max() <= 1e-6 * P.max(), f"{tag} frame {f}: cube and power map disagree"


@pytest.fixture(scope="module")
def compiled(pkg):
    return compiled_forms(pkg)


@pytest.mark.parametrize("case", CASES, ids=case_id)
def test_kernel_form_against_oracle(pkg, orc, compiled, case):
    _run(pkg, orc, case, compiled)


def test_every_compiled_kernel_is_checked(pkg, orc, compiled):
    """compiled kernels == kernels CASES launched | EXEMPT; any other kernel is named"""
    for case in CASES:
        if case_id(case) not in _LAUNCHED:
            _run(pkg, orc, case, compiled)
    launched = set().union(*_LAUNCHED.values())
    exempt = compiled & set(EXEMPT)
    stale = sorted(set(EXEMPT) - compiled)
    assert not stale, f"EXEMPT names kernels the library does not compile: {stale}"
    unchecked = sorted(compiled - launched - exempt)
    print(f"\n{len(compiled)} compiled kernels: {len(launched)} launched by CASES, {len(exempt - launched)} more checked "
          f"elsewhere (EXEMPT)")
    assert not unchecked, f"compiled kernels that no case launches and no other test checks: {unchecked}"


@pytest.mark.parametrize("C", [64, 34, 128, 66, 256, 130, 512, 300, 1024, 1000])
def test_detection_snapshots_hold_every_chirp(pkg, orc, C):
    """The antenna snapshot of a detection (re-FFT path: doppler_extract_kernel<Cp, PAD>; per-cell path: measure_kernel)
    only decides its angle bin, and a clean target's snapshot barely depends on any one chirp: a kernel that dropped or
    mis-weighted one would still pass the scene tests above.  Here the scene is noise (every cell's snapshot a sum of
    independent terms), the Doppler window rectangular (every chirp weighted 1), and CFAR's alpha low, so that thousands
    of cells are detected and their angle bins move with any one chirp: zeroing the last valid chirp of the input changes
    9-47 % of them in the oracle (more at fewer chirps).  Angle bins must equal the oracle's away from ties, on both detection paths, for every Cp and
    with and without chirp padding."""
    S, A, F, alpha = 256, 4, 2, 2.5
    rng = np.random.default_rng(C)
    adc = rng.integers(-2000, 2000, (F, 2 * S * C * A)).astype(np.int16)
    wr, wd = orc.hann_periodic(S), np.ones(C, np.float32)
    ref = orc.process_frames(adc, F, S, C, A, wr, wd, alpha=alpha, want=("P", "noise", "ratio"), n_threads=4)
    thr = alpha * ref["noise"]
    near = np.abs(ref["P"] - thr) <= 1e-5 * thr
    key = lambda d: (d["frame"].astype(np.int64) << 32) | (d["range_bin"].astype(np.int64) << 16) | d["doppler_bin"]
    rk = key(ref["dets"])
    with pkg.RadarContext(S, C, A, F, cfar_alpha=alpha, max_det_per_frame=8192) as ctx:
        ctx.set_windows(None, wd)
        for path, name in ((pkg.api.DETECT_REFFT, "re-FFT"), (pkg.api.DETECT_PER_CELL, "per-cell")):
            ctx.set_detect_path(path)
            dets, overflow = ctx.process_host(adc, F)
            assert not overflow
            gk = key(dets)
            diff = np.setxor1d(gk, rk)
            assert all(near[k >> 32, (k >> 16) & 0xffff, k & 0xffff] for k in diff), f"{name}: hit list differs away from threshold"
            _, gi, ri = np.intersect1d(gk, rk, return_indices=True)
            clear = ref["ratio"][ri] < 1 - 1e-4
            bad = int((dets["angle_bin"][gi] != ref["dets"]["angle_bin"][ri])[clear].sum())
            print(f"\nC={C} {name}: {int(clear.sum())} angle bins compared, {bad} differ")
            assert clear.sum() > 200 and bad == 0, f"{name}: {bad} angle bins differ from the oracle's away from ties"
