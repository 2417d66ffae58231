"""GPU parity: the CUDA chain called through the C ABI against the CPU oracle on the same seeded
inputs.  Tolerances (BASELINE.json north_star): FFT outputs and power maps within 1e-4 of the
map's maximum (fp32 vs the fp64 oracle); CFAR hits bit-exact except cells within 1e-5 (relative)
of their threshold, which are counted and printed; integer/index work bit-exact."""
import numpy as np
import pytest

from chain_check import WALK_FORMS, cfar_form_name, launched_kernels

pytestmark = pytest.mark.gpu

TOL = 1e-4          # relative to the maximum of the array being compared
NEAR = 1e-5         # |P - thr| <= NEAR * thr  -> cell is "at threshold", excluded from the bit-exact claim
# CA-CFAR noise estimate (mean of the training cells) relative to the oracle's: the fp32 window sum only ever adds (~1e-6),
# the rest is the fp32 FFT error of the near-floor cells it averages; measured <= 1.05e-5 on B200 (tests/test_gpu_bench_paths.py)
NOISE_RTOL = 5e-5

# the next three exercise the 256-point angle FFT (A > 64: the cfg4 imaging array), an odd antenna count and the maximum A
SHAPES = [(64, 64, 2), (100, 128, 4), (128, 64, 12), (256, 128, 4), (512, 256, 12), (1024, 64, 2), (64, 1024, 1), (256, 512, 3),
          (64, 64, 192), (128, 128, 65), (64, 64, 256),
          # ragged shapes: S a bare multiple of 4, C a bare multiple of 2, zero-padded to the next power of two on both axes
          (68, 66, 3), (500, 130, 2)]


def relmax(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


@pytest.fixture(scope="module")
def cases(pkg, orc):
    """oracle outputs per shape, computed once"""
    out = {}
    for (S, C, A) in SHAPES:
        F = 2 if S * C * A <= 131072 else 1
        adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=5)
        wr, wd = orc.hann_periodic(S), orc.hann_periodic(C)
        ref = orc.process_frames(adc, F, S, C, A, wr, wd, want=("rs", "dc", "P", "mask", "noise"), n_threads=4)
        out[(S, C, A)] = (F, adc, wr, wd, ref)
    return out


@pytest.mark.parametrize("shape", SHAPES)
def test_range_spectrum(pkg, orc, cases, shape):
    S, C, A = shape
    F, adc, wr, wd, ref = cases[shape]
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.set_windows(None, np.ones(C, np.float32))          # rect Doppler window: plain range FFT
        ctx.process_host(adc, F)
        for f in range(F):
            assert relmax(ctx.range_spectrum(f), ref["rs"][f]) < TOL
        ctx.set_windows(None, None)                            # default Hann: K1 folds w_d[c] into its output
        ctx.process_host(adc, F)
        assert relmax(ctx.range_spectrum(0), ref["rs"][0] * wd.astype(np.float64)) < TOL


@pytest.mark.parametrize("shape", SHAPES)
def test_doppler_cube_and_power_map(pkg, orc, cases, shape):
    S, C, A = shape
    F, adc, wr, wd, ref = cases[shape]
    with pkg.RadarContext(S, C, A, F, keep_doppler_cube=True) as ctx:
        ctx.process_host(adc, F)
        for f in range(F):
            assert relmax(ctx.doppler_cube(f), ref["dc"][f]) < TOL
            assert relmax(ctx.power_map(f), ref["P"][f]) < TOL
    with pkg.RadarContext(S, C, A, F, keep_doppler_cube=False) as ctx:
        ctx.process_host(adc, F)
        assert relmax(ctx.power_map(F - 1), ref["P"][F - 1]) < TOL
        with pytest.raises(pkg.RadarError):
            ctx.doppler_cube(0)


def _near_threshold(ref, alpha):
    thr = alpha * ref["noise"]
    return np.abs(ref["P"] - thr) <= NEAR * thr


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("keep", [False, True])
def test_cfar_and_detections(pkg, orc, cases, shape, keep):
    S, C, A = shape
    F, adc, wr, wd, ref = cases[shape]
    alpha = 15.0
    near = _near_threshold(ref, alpha)
    with pkg.RadarContext(S, C, A, F, keep_doppler_cube=keep) as ctx:
        dets, overflow = ctx.process_host(adc, F)
        assert not overflow
        counts = ctx.read_counts(F)
        for f in range(F):
            m = ctx.cfar_mask(f)
            bad = (m != ref["mask"][f]) & ~near[f]
            assert not bad.any(), f"{bad.sum()} CFAR cells differ away from threshold"
            assert counts[f] == m.sum()
    print(f"\n{shape} keep={keep}: {len(dets)} detections, {int(near.sum())} cells within {NEAR} of threshold (excluded)")
    # ordering and identity of the hit list
    key = lambda d: (int(d["frame"]), int(d["range_bin"]), int(d["doppler_bin"]))
    got, want = [key(d) for d in dets], [key(d) for d in ref["dets"]]
    assert got == sorted(got)
    diff = set(got) ^ set(want)
    assert all(near[k] for k in diff)
    by = {key(d): d for d in ref["dets"]}
    n_theta = orc.angle_fft_size(A)
    assert len(dets) > 0
    for d in dets:
        k = key(d)
        if k not in by:
            continue
        o = by[k]
        assert abs(d["power"] - o["power"]) <= TOL * ref["P"][k[0]].max()
        assert abs(d["noise"] - o["noise"]) <= NOISE_RTOL * o["noise"]
        x = ref["dc"][k[0]][:, k[1], k[2]]
        _, ratio = orc.angle_argmax(x, n_theta)
        if ratio < 1 - 1e-4:                                   # angle arg-max not a near tie
            assert d["angle_bin"] == o["angle_bin"]
            assert abs(d["angle_rad"] - o["angle_rad"]) < 1e-5
        # grouping flag: compare unless a detected neighbour has (almost) the same power
        P = ref["P"][k[0]]
        nb = [P[k[1] + i, (k[2] + j) % P.shape[1]] for i in (-1, 0, 1) for j in (-1, 0, 1)
              if (i or j) and 0 <= k[1] + i < P.shape[0] and ref["mask"][k[0]][k[1] + i, (k[2] + j) % P.shape[1]]]
        if all(abs(v - P[k[1], k[2]]) > 1e-4 * P[k[1], k[2]] for v in nb) and not any(near[k[0]][max(0, k[1] - 1):k[1] + 2].ravel()):
            assert (d["flags"] & 1) == (o["flags"] & 1)


# the last two: the largest windows mmw_create accepts (guard + train = 64 range bins; 31 Doppler bins at Cp = 64, 32 at
# Cp >= 128): the halo covers most of the map, and every row's range window is clamped where the Doppler window wraps
@pytest.mark.parametrize("shape,guard,train,alpha", [((128, 64, 4, 2), (0, 0), (1, 1), 6.0), ((128, 64, 4, 2), (1, 3), (5, 2), 10.0),
                                                     ((128, 64, 4, 2), (4, 1), (12, 7), 12.0), ((128, 64, 4, 2), (2, 2), (8, 4), 4.0),
                                                     ((128, 64, 4, 2), (4, 3), (60, 28), 4.0), ((256, 128, 2, 2), (1, 2), (63, 30), 4.0)],
                         ids=lambda v: "x".join(map(str, v)) if isinstance(v, tuple) else str(v))
def test_cfar_geometries(pkg, orc, shape, guard, train, alpha):
    """non-default guard / training windows take the run-time-bound CFAR path; range edges clamp, Doppler wraps"""
    S, C, A, F = shape
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=11, n_targets=6)
    wr, wd = orc.hann_periodic(S), orc.hann_periodic(C)
    ref = orc.process_frames(adc, F, S, C, A, wr, wd, guard=guard, train=train, alpha=alpha, want=("P", "mask", "noise"))
    thr = alpha * ref["noise"]
    near = np.abs(ref["P"] - thr) <= NEAR * thr
    with pkg.RadarContext(S, C, A, F, cfar_guard=guard, cfar_train=train, cfar_alpha=alpha, max_det_per_frame=8192) as ctx:
        dets, ov = ctx.process_host(adc, F)
        for f in range(F):
            m = ctx.cfar_mask(f)
            assert not ((m != ref["mask"][f]) & ~near[f]).any()
            edge = np.r_[0:train[0] + guard[0] + 1, S - train[0] - guard[0] - 1:S]     # the clamped range rows in particular
            assert not ((m[edge] != ref["mask"][f][edge]) & ~near[f][edge]).any()
    by = {(int(d["frame"]), int(d["range_bin"]), int(d["doppler_bin"])): d for d in ref["dets"]}
    assert len(dets) > 0 and not ov
    for d in dets:
        k = (int(d["frame"]), int(d["range_bin"]), int(d["doppler_bin"]))
        if k in by:
            assert abs(d["noise"] - by[k]["noise"]) <= NOISE_RTOL * by[k]["noise"]


def _walk_form(F, Sp, Cp, sm_count):
    """launch_cfar's rule for the default window: (range bins per strip, Doppler segments of 16 bins per CTA, Sp the kernel
    is specialised for or 0)"""
    cells, want = F * Sp * Cp, 8 * sm_count
    rt = 64
    if Sp % 128 == 0 and cells // (128 * 32) >= want:
        rt = 128
    if Sp % 256 == 0 and cells // (256 * 32) >= want:
        rt = 256
    nchunk = 2
    while nchunk < 8 and Cp % (32 * nchunk) == 0 and cells // (rt * 32 * nchunk) >= want:
        nchunk *= 2
    return rt, nchunk, (Sp if Sp in (256, 512, 1024) else 0)


@pytest.fixture(scope="module")
def sm_count(pkg):
    with pkg.RadarContext(64, 64, 1, 1) as ctx:
        return ctx.info.sm_count


@pytest.mark.parametrize("form", WALK_FORMS, ids=lambda f: "tiled" if f is None else "rt%d-seg%d-spt%d" % f)
def test_cfar_kernel_forms_agree_with_oracle(pkg, orc, sm_count, form):
    """Every form of K3 against the oracle's CFAR on the GPU's own power map: same mask away from threshold cells (the
    clamped range edges included) and the noise estimate of every detection.  The walk kernel's forms are keyed as in
    launch_cfar / run_cfar_walk: strips of 64 / 128 / 256 range bins, Doppler segments of nchunk x 16 bins per CTA, and
    the Sp the kernel is specialised for (0: run-time Sp), reached through the shape and the batch size F for which
    launch_cfar's rule picks it on this GPU (a few synthetic frames tiled to F); the tiled kernel serves every window but
    the default one.  The kernel the batch launched is recorded and must be the one the form names, so a changed launcher
    rule fails here instead of checking another form.  (Sweep records: profiles/experiments/r1_cfar_walk_sweep.log.)"""
    if form is None:
        S, C, F, train = 256, 128, 2, (8, 5)
    else:
        S, C, F = next((S, C, F) for (S, C) in ((256, 128), (64, 256), (128, 256), (512, 256), (1024, 64))
                       for F in range(1, 64 * sm_count) if _walk_form(F, S, C, sm_count) == form)
        train = (8, 4)
    base = pkg.synth.cube_batch(3, S, C, 1, cfg=3, n_targets=6)
    adc = np.ascontiguousarray(base[np.arange(F) % 3])
    import torch

    with pkg.RadarContext(S, C, 1, F, cfar_train=train) as ctx:
        # the device-resident entry point runs the whole batch as one: the host path uploads and processes it in chunks of
        # 48 MB, which would take other forms for the frames of each chunk
        adc_dev = torch.from_numpy(adc).cuda()
        with launched_kernels() as names:
            ctx.process_device(adc_dev, F)
        dets, overflow = ctx.read_detections()
        del adc_dev
        assert not overflow
        cfar = sorted(k for k in names if k.startswith("cfar_"))
        assert cfar == [cfar_form_name(form)], f"{S} x {C}, {F} frames launched {cfar}, not {cfar_form_name(form)}"
        frames = sorted({0, F // 2, F - 1})
        got = {f: (ctx.power_map(f), ctx.cfar_mask(f)) for f in frames}
    for f in frames:
        P, mask = got[f]
        ref_mask, ref_noise = orc.cfar(P, train=train)
        thr = 15.0 * ref_noise
        near = np.abs(P - thr) <= NEAR * thr
        assert not ((mask != ref_mask) & ~near).any(), f"frame {f}: CFAR cells differ away from threshold"
        for edge in (np.r_[0:12], np.r_[S - 12:S]):                      # clamped range rows; all Doppler columns incl. the wrap
            assert not ((mask[edge] != ref_mask[edge]) & ~near[edge]).any(), f"frame {f}: clamped range edge differs"
        d = dets[dets["frame"] == f]
        assert len(d) == int(mask.sum()) > 0
        r, c = d["range_bin"].astype(np.int64), d["doppler_bin"].astype(np.int64)
        assert np.all(np.abs(d["noise"] - ref_noise[r, c]) <= NOISE_RTOL * ref_noise[r, c]), f"frame {f}: noise estimate"


def test_wide_array_paths_agree(pkg, orc):
    """A >= 32 in fused mode: the selective Doppler re-FFT + angle FFT path (default) against the per-detection kernel it
    replaces (mmw_set_detect_path(MMW_DETECT_PER_CELL): direct Doppler DFT + angle DFT per detection) and against cube mode:
    same cells, powers, noise and flags bit for bit; angle bins identical away from ties of the angle spectrum."""
    S, C, A, F = 128, 64, 96, 3
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=13, n_targets=6)
    wr, wd = orc.hann_periodic(S), orc.hann_periodic(C)
    ref = orc.process_frames(adc, F, S, C, A, wr, wd, want=("ratio",), n_threads=3)
    with pkg.RadarContext(S, C, A, F) as ctx:
        new, ov = ctx.process_host(adc, F)
        assert not ov and ctx.info.kernels_per_batch == 7
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.set_detect_path(pkg.api.DETECT_PER_CELL)
        old, _ = ctx.process_host(adc, F)
        assert ctx.info.kernels_per_batch == 5
    with pkg.RadarContext(S, C, A, F, keep_doppler_cube=True) as ctx:
        cube, _ = ctx.process_host(adc, F)
    key = lambda d: (d["frame"].astype(np.int64) << 32) | (d["range_bin"].astype(np.int64) << 16) | d["doppler_bin"]
    rk = key(ref["dets"])
    for other, name in ((old, "per-detection kernel"), (cube, "cube mode")):
        assert len(new) == len(other) > 50, name
        for fld in ("frame", "range_bin", "doppler_bin", "power", "noise", "flags"):
            assert np.array_equal(new[fld], other[fld]), (name, fld)
        _, ni, ri = np.intersect1d(key(new), rk, return_indices=True)
        clear = ref["ratio"][ri] < 1 - 1e-4
        assert np.array_equal(new["angle_bin"][ni][clear], other["angle_bin"][ni][clear]), name
        assert np.array_equal(new["angle_bin"][ni][clear], ref["dets"]["angle_bin"][ri][clear]), name


def test_detection_list_overflow_is_ordered_and_counted(pkg, orc):
    S, C, A, F = 64, 64, 2, 3
    rng = np.random.default_rng(5)
    adc = rng.integers(-3000, 3000, (F, 2 * S * C * A)).astype(np.int16)
    with pkg.RadarContext(S, C, A, F, cfar_alpha=1.5, max_det_per_frame=4096) as ctx:
        full, ov = ctx.process_host(adc, F)
        counts_full = ctx.read_counts(F)
        assert not ov and len(full) == counts_full.sum() and counts_full.min() > 16
    with pkg.RadarContext(S, C, A, F, cfar_alpha=1.5, max_det_per_frame=16) as ctx:
        cut, ov = ctx.process_host(adc, F)
        assert ov and np.array_equal(ctx.read_counts(F), counts_full)        # true totals still reported
        want = np.concatenate([full[full["frame"] == f][:16] for f in range(F)])
        assert cut.tobytes() == want.tobytes()                              # first 16 per frame, in order
        few, ov2 = ctx.process_host(adc, F, det_capacity=5)
        assert ov2 and few.tobytes() == want[:5].tobytes()


def test_full_scale_int16_samples(pkg, orc):
    """sign handling of the IIQQ unpack at the ends of the int16 range (-32768, 32767), alternating per sample"""
    S, C, A, F = 64, 64, 2, 1
    rng = np.random.default_rng(9)
    adc = rng.choice(np.array([-32768, 32767, -1, 0, 1], np.int16), size=(F, 2 * S * C * A))
    adc[0, :16] = [-32768, 32767, 32767, -32768, 32767, -32768, -32768, 32767] * 2
    wr, wd = orc.hann_periodic(S), orc.hann_periodic(C)
    ref = orc.process_frames(adc, F, S, C, A, wr, wd, want=("rs", "P"))
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.process_host(adc, F)
        rs_ref = ref["rs"][0] * wd[None, None, :]
        assert relmax(ctx.range_spectrum(0), rs_ref) < TOL
        assert relmax(ctx.power_map(0), ref["P"][0]) < TOL
        # rectangular windows: the first range bin of a constant full-scale row is exactly S * value
        ctx.set_windows(np.ones(S, np.float32), np.ones(C, np.float32))
        const = np.full((1, 2 * S * C * A), -32768, np.int16)
        ctx.process_host(const, 1)
        r0 = ctx.range_spectrum(0)[:, 0, :]
        assert np.all(r0.real == -32768.0 * S) and np.all(r0.imag == -32768.0 * S)


def test_empty_scene_and_zero_input(pkg):
    S, C, A, F = 128, 64, 4, 2
    with pkg.RadarContext(S, C, A, F) as ctx:
        dets, ov = ctx.process_host(np.zeros((F, 2 * S * C * A), np.int16), F)
        assert len(dets) == 0 and not ov and ctx.read_counts(F).sum() == 0
        assert ctx.power_map(1).max() == 0.0
        with pytest.raises(pkg.RadarError):
            ctx.process_host(np.zeros((F + 1, 2 * S * C * A), np.int16), F + 1)     # beyond max_frames
        with pytest.raises(pkg.RadarError):
            ctx.power_map(F)                                                        # frame outside the batch


def test_user_windows_round_trip(pkg, orc):
    S, C, A = 64, 64, 2
    adc = pkg.synth.cube_batch(1, S, C, A, cfg=8)
    wr = np.hamming(S).astype(np.float32)
    wd = np.blackman(C).astype(np.float32)
    with pkg.RadarContext(S, C, A, 1, keep_doppler_cube=True) as ctx:
        ctx.set_windows(wr, wd)
        g = ctx.get_windows()
        assert np.array_equal(g[0], wr) and np.array_equal(g[1], wd)
        ctx.process_host(adc, 1)
        ref = orc.process_frames(adc, 1, S, C, A, wr, wd, want=("dc", "P"))
        assert relmax(ctx.doppler_cube(0), ref["dc"][0]) < TOL and relmax(ctx.power_map(0), ref["P"][0]) < TOL
        # default windows are the oracle's periodic Hann, bit for bit
        ctx.set_windows(None, None)
        g = ctx.get_windows()
        assert np.array_equal(g[0], orc.hann_periodic(S)) and np.array_equal(g[1], orc.hann_periodic(C))


# ---------------------------------------------------------------- legacy path (reference cfg 100 x 128 x 4)
@pytest.fixture
def legacy_kernel(pkg):
    """forces one form of the legacy frame kernel for the test (mmw_legacy_configure), restores the default afterwards"""
    def pick(name):
        pkg.api.legacy_configure(kernel_variant={"single_cta": 1, "cluster": 2}[name], quiet=1)
    yield pick
    pkg.api.legacy_configure(kernel_variant=0)


@pytest.mark.parametrize("kernel", ["cluster", "single_cta"])
def test_legacy_matches_golden_and_oracle(pkg, orc, golden_dir, kernel, legacy_kernel):
    """both forms of the legacy frame kernel: the 8-CTA cluster (default for single frames) and the single-CTA kernel"""
    legacy_kernel(kernel)
    gold = np.load(f"{golden_dir}/legacy_reference.npz")
    i = 0
    timers = np.zeros(4)
    for sd in gold["cap_seeds"]:
        cap = pkg.synth.legacy_capture(int(gold["cap_frames"]), seed=int(sd), moving=(sd == 2))
        base = orc.reshape(cap[0], 100, 128, 4)[:12800]
        for f in range(1, cap.shape[0]):
            d = pkg.cudaProcessing(cap[f], base, timers=timers)            # the reference's own symbol
            assert d == gold["dist"][i], (d, gold["dist"][i])            # bit-identical double
            spec = pkg.api.legacy_spectrum()
            probes = gold["spec_probes"][i]
            assert np.abs(spec[gold["probe_bins"]] - probes).max() <= TOL * np.abs(probes).max()
            d2, raw = pkg.api.legacy_process_frame(cap[f], base)
            assert raw == gold["raw"][i] and d2 == d
            i += 1
        dist, raw = pkg.api.legacy_process_frames(cap[1:], base)
        n = cap.shape[0] - 1
        assert np.array_equal(dist, gold["dist"][i - n:i]) and np.array_equal(raw, gold["raw"][i - n:i])
    assert timers[3] > 0 and timers[3] >= timers[0] > 0                   # accumulated seconds (+=)


@pytest.mark.parametrize("kernel", ["cluster", "single_cta"])
def test_legacy_full_spectrum_and_edges(pkg, orc, kernel, legacy_kernel):
    legacy_kernel(kernel)
    cap = pkg.synth.legacy_capture(3, seed=21)
    base = orc.reshape(cap[0], 100, 128, 4)[:12800]
    d_ref, raw_ref, spec_ref = orc.legacy_frame(cap[2], base, want_spectrum=True)
    d, raw = pkg.api.legacy_process_frame(cap[2], base)
    assert (d, raw) == (d_ref, raw_ref)
    assert relmax(pkg.api.legacy_spectrum(), spec_ref) < TOL
    # all-zero difference -> arg-max 0 -> 0 m (strict >, cudaBenchMarking.cpp:199)
    assert pkg.api.legacy_process_frame(cap[0], base) == (0.0, 0)
    # the caller may change the base frame between calls (the reference re-uploads it every call)
    base2 = orc.reshape(cap[1], 100, 128, 4)[:12800]
    assert pkg.api.legacy_process_frame(cap[2], base2) == orc.legacy_frame(cap[2], base2)
    assert pkg.api.legacy_process_frame(cap[2], base) == (d_ref, raw_ref)
    # two bins with the same power: the first wins, as in the reference
    k = np.arange(100)
    tone = lambda f0: 1000 * np.exp(2j * np.pi * f0 * k)
    z = np.zeros((128, 4, 100), complex)
    z[:, 0, :] = tone(0.11) + tone(0.23)
    frame = pkg.synth.pack_iiqq(z).reshape(-1)
    zero_base = np.zeros(12800, complex)
    assert pkg.api.legacy_process_frame(frame, zero_base) == orc.legacy_frame(frame, zero_base)


@pytest.mark.parametrize("kernel", ["cluster", "single_cta"])
def test_legacy_many_near_tie_bins(pkg, orc, kernel, legacy_kernel):
    """More near-tie bins than any fixed-size candidate list would hold: 60 equal-amplitude tones whose 12 800-sample
    windows are mutually orthogonal (bins are multiples of 32 = 25 * 16384 / 12800), so the 60 peaks of the 16 384-point
    spectrum agree to ~1e-5 (int16 rounding noise; the top two differ by 2e-7 .. 7e-6) — inside the 1e-4 near-tie window
    of the fp32 pass and at or below its rounding error, far outside fp64 rounding.
    The fp64 re-check must visit all of them in ascending bin order and return the reference's first maximum
    (cudaBenchMarking.cpp:191-206).  Also: a flat spectrum (an impulse at sample 0: every bin exactly 1) -> bin 0."""
    legacy_kernel(kernel)
    k = np.arange(100 * 128)
    zero_base = np.zeros(12800, complex)
    for seed in range(4):
        rng = np.random.default_rng(seed)
        bins = 32 * (2 + rng.permutation(200)[:60])                      # 60 distinct multiples of 32 below 0.4 * 16384
        ph = rng.uniform(0, 2 * np.pi, 60)
        x = sum(1000.0 * np.exp(2j * np.pi * (b / 16384.0) * k + 1j * p) for b, p in zip(bins, ph))
        z = np.zeros((128, 4, 100), complex)
        z[:, 0, :] = x.reshape(128, 100)
        frame = pkg.synth.pack_iiqq(z).reshape(-1)
        d_ref, raw_ref, spec = orc.legacy_frame(frame, zero_base, want_spectrum=True)
        mag = np.abs(spec[:6553]) ** 2
        n_near = int((mag >= mag.max() * (1 - 1e-4)).sum())
        assert n_near > 32, n_near                                       # the case the old 32-entry list gave up on
        assert pkg.api.legacy_process_frame(frame, zero_base) == (d_ref, raw_ref), (seed, n_near)
        assert raw_ref in bins
    z = np.zeros((128, 4, 100), complex)
    z[0, 0, 0] = 1000.0
    frame = pkg.synth.pack_iiqq(z).reshape(-1)
    assert orc.legacy_frame(frame, zero_base) == (0.0, 0)
    assert pkg.api.legacy_process_frame(frame, zero_base) == (0.0, 0)


def test_legacy_upload_paths_and_short_frames(pkg, orc):
    """the host path uploads rx0's rows only: a pinned capture by one strided DMA, a pageable one packed by the CPU; frames
    cut short at any point (inside rx0's row, inside another receiver's, on a row boundary) follow the reference's size rule"""
    import torch

    cap = pkg.synth.legacy_capture(9, seed=6, moving=True)
    base = orc.reshape(cap[0], 100, 128, 4)[:12800]
    want = [orc.legacy_frame(cap[f], base) for f in range(1, 9)]
    d0, r0 = pkg.api.legacy_process_frames(cap[1:], base)
    pinned = torch.from_numpy(cap[1:].copy()).pin_memory()
    d1, r1 = pkg.api.legacy_process_frames(pinned.numpy(), base)
    assert [(float(d), int(r)) for d, r in zip(d0, r0)] == want
    assert np.array_equal(d0, d1) and np.array_equal(r0, r1)
    for size in (102399, 102400 - 600, 64000, 51300, 800 * 17, 800 * 17 + 100, 800 * 17 + 199, 801, 150, 3):
        assert pkg.api.legacy_process_frame(cap[2][:size], base) == orc.legacy_frame(cap[2][:size], base), size


def test_chain_matches_numpy_golden_fixture(pkg, golden_dir):
    """the CUDA chain against tests/golden/chain_numpy.npz — numbers produced by numpy alone (make_chain_golden.py), not by the
    oracle: power map within 1e-4 of its maximum, hit cells exactly away from threshold cells, angle bins away from ties"""
    g = np.load(f"{golden_dir}/chain_numpy.npz")
    for (S, C, A, F, cfg) in [tuple(int(v) for v in row) for row in g["cases"]]:
        tag = f"{S}x{C}x{A}"
        adc = pkg.synth.cube_batch(F, S, C, A, cfg=cfg, n_targets=4)
        with pkg.RadarContext(S, C, A, F) as ctx:
            Sp, Cp = ctx.Sp, ctx.Cp
            dets, overflow = ctx.process_host(adc, F)
            assert not overflow
            for f in range(F):
                P = g[f"P_{tag}_f{f}"]
                assert relmax(ctx.power_map(f), P) < TOL
                mask = np.unpackbits(g[f"mask_{tag}_f{f}"])[: Sp * Cp].reshape(Sp, Cp).astype(bool)
                near = np.unpackbits(g[f"near_{tag}_f{f}"])[: Sp * Cp].reshape(Sp, Cp).astype(bool)
                got = ctx.cfar_mask(f).astype(bool)
                assert np.array_equal(got[~near], mask[~near])
                by = {(int(d["range_bin"]), int(d["doppler_bin"])): d for d in dets[dets["frame"] == f]}
                n_checked = 0
                for (r, d), nz, ab, tie in zip(g[f"hits_{tag}_f{f}"], g[f"noise_at_hits_{tag}_f{f}"], g[f"angle_bin_{tag}_f{f}"],
                                               g[f"angle_tie_{tag}_f{f}"]):
                    if near[r, d]:
                        continue
                    rec = by[(int(r), int(d))]
                    assert abs(rec["noise"] - nz) <= NOISE_RTOL * nz
                    if not tie:
                        assert rec["angle_bin"] == ab
                    n_checked += 1
                assert n_checked > 0


@pytest.mark.parametrize("shape,variants", [((512, 256, 12), ["cube", "split"]), ((256, 128, 4), ["cube", "split"]),
                                            ((500, 130, 2), ["cube", "split"])])
def test_doppler_kernel_forms_give_the_same_bits(pkg, shape, variants):
    """The other forms of K2 run the same arithmetic in the same order as the default one, so the power maps must be equal
    byte for byte: "cube" keeps the Doppler cube (CTA-shared tiles that also store the cube, where fused mode runs the
    warp-private kernel at 256 points), "split" is a one-frame batch (the antenna-split path: one single-antenna K2 pass
    per antenna, then the ordered sum).  The detection list of the split batch equals frame 0's records of the default
    one byte for byte; cube mode measures its snapshots from the cube, so there cells, powers, noise and flags must match.
    Shapes: full length, 128 points, and chirp-padded (130 -> 256 chirps: the PAD instantiations)."""
    S, C, A = shape
    F = 5                                                    # several tiles per warp and a ragged tail
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=3, n_targets=6)
    with pkg.RadarContext(S, C, A, F) as ctx:
        want, _ = ctx.process_host(adc, F)
        want = want.copy()
        pmaps = [ctx.power_map(f).copy() for f in range(F)]
    assert len(want) > 0
    for v in variants:
        with pkg.RadarContext(S, C, A, F, keep_doppler_cube=(v == "cube")) as ctx:
            n = F if v == "cube" else 1
            got, _ = ctx.process_host(adc[:n], n)
            for f in range(n):
                assert np.array_equal(ctx.power_map(f), pmaps[f]), f"{v}: power map of frame {f} differs"
        if v == "split":
            assert got.tobytes() == want[want["frame"] == 0].tobytes(), "split: detection list differs"
        else:
            for fld in ("frame", "range_bin", "doppler_bin", "power", "noise", "flags"):
                assert np.array_equal(got[fld], want[fld]), f"cube: {fld} differs"
