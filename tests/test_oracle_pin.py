"""Pins the CPU oracle: (a) against the golden vectors generated from the reference's own CPU
functions (tests/golden/make_golden.py), (b) directly against those functions where oracle/_ref
exists, else against what make_golden.py stored from them, (c) against numpy fp64 for the stages
the reference lacks (parity unpinned by the reference; the oracle is the spec there)."""
import os

import numpy as np
import pytest


@pytest.fixture(scope="module")
def gold(golden_dir):
    return np.load(f"{golden_dir}/legacy_reference.npz")


def test_kat_ramp16(orc, gold):
    # reference fftTest() input (acceleration.cu:361-365); X[0]=136, X[k] = -8 + 8j cot(pi k/16)
    X = orc.fft(gold["kat_ramp16_in"])
    assert np.array_equal(X, gold["kat_ramp16_out"])
    k = np.arange(1, 16)
    expect = np.concatenate([[136.0], -8 + 8j / np.tan(np.pi * k / 16)])
    assert np.abs(X - expect).max() < 1e-11


def test_fft_matches_reference_bit_for_bit(orc, gold):
    for n in (64, 128, 256, 512, 1024):
        assert np.array_equal(orc.fft(gold[f"fft{n}_in"]), gold[f"fft{n}_out"])
        assert np.abs(orc.fft(gold[f"fft{n}_in"]) - np.fft.fft(gold[f"fft{n}_in"])).max() < 1e-11


def test_reshape_spot_checks(orc, gold):
    s = (np.arange(102400) % 32768).astype(np.int16)
    y = orc.reshape(s, 100, 128, 4)
    assert np.array_equal(y[gold["reshape_idx"]], gold["reshape_val"])
    # values quoted in SURVEY.md §4 (the ones below the int16 wrap of the ramp)
    assert y[0] == 0 + 2j and y[1] == 1 + 3j and y[2] == 4 + 6j and y[100] == 800 + 802j and y[12800] == 200 + 202j


def test_legacy_frames_match_golden(orc, pkg, gold):
    i = 0
    for sd in gold["cap_seeds"]:
        cap = pkg.synth.legacy_capture(int(gold["cap_frames"]), seed=int(sd), moving=(sd == 2))
        base = orc.reshape(cap[0], 100, 128, 4)[:12800]
        for f in range(1, cap.shape[0]):
            d, raw, spec = orc.legacy_frame(cap[f], base, want_spectrum=True)
            assert raw == gold["raw"][i]
            assert d == gold["dist"][i]                       # bit-exact, not 1e-5
            assert np.array_equal(spec[gold["probe_bins"]], gold["spec_probes"][i])
            i += 1
    # the probe quoted in SURVEY.md §8d: tone at 0.123 cycles/sample -> raw 1966, 6.009113 m
    assert gold["raw"][0] == 1966 and abs(gold["dist"][0] - 6.009113) < 1e-6


def test_against_compiled_reference(orc, pkg, golden_dir):
    """reshape, frame results and spectra, FFTs and next_pow2 of the oracle equal the reference's own functions: called
    where oracle/_ref was built, else as stored from them by tests/golden/make_golden.py (legacy_reference_direct.npz,
    the 16384-point outputs at a fixed sample of bins)"""
    cap = pkg.synth.legacy_capture(4, seed=11)
    path = os.path.join(golden_dir, "legacy_reference_direct.npz")
    live = orc.have_ref()
    if live:
        want = orc.direct_vectors(cap, orc.ref_reshape, orc.ref_cpu_frame, orc.ref_fft, orc.ref().ref_next_pow2)
    elif os.path.exists(path):
        want = dict(np.load(path))
    else:
        pytest.skip("needs the reference's own CPU functions (oracle/_ref) or the vectors tests/golden/make_golden.py stores from them")
    got = orc.direct_vectors(cap, lambda s: orc.reshape(s, 100, 128, 4), orc.legacy_frame, orc.fft, orc.next_pow2, sample=not live)
    assert sorted(got) == sorted(want)
    for k in got:
        assert np.array_equal(got[k], want[k]), k


def test_legacy_edge_cases(orc):
    base = np.zeros(12800, np.complex128)
    d, raw = orc.legacy_frame(np.zeros(102400, np.int16), base)
    assert raw == 0 and d == 0.0                              # all-zero spectrum -> index 0 (strict >)
    # two equal peaks: first one wins
    x = np.zeros(16384, np.complex128)
    x[[100, 200]] = 5.0
    assert orc.lib().orc_find_abs_max(x.ctypes.data, 6553) == 100


# after the first three: the ragged shapes test_gpu_kernel_forms.py checks the CUDA chain at against this oracle (S and C
# zero-padded to the next power of two, up to 1000 x 998 -> 1024 x 1024)
@pytest.mark.parametrize("S,C,A", [(64, 64, 2), (100, 128, 4), (128, 64, 12), (36, 34, 3), (60, 60, 2), (68, 66, 3),
                                   (200, 130, 4), (300, 300, 2), (1000, 998, 2), (1000, 1000, 2)])
def test_new_stages_against_numpy(orc, pkg, S, C, A):
    adc = pkg.synth.cube(3, S, C, A, cfg=5, n_targets=4)
    wr, wd = orc.hann_periodic(S), orc.hann_periodic(C)
    assert np.allclose(wr, 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(S) / S), atol=1e-7)
    out = orc.process_frames(adc[None], 1, S, C, A, wr, wd, want=("rs", "dc", "P", "mask", "noise"))
    Sp, Cp = orc.next_pow2(S), orc.next_pow2(C)
    z = pkg.synth.unpack_iiqq(adc.reshape(C, A, 2 * S))
    rs = np.fft.fft(z * wr.astype(np.float64), n=Sp, axis=-1).transpose(1, 2, 0)
    dc = np.fft.fft(rs * wd.astype(np.float64), n=Cp, axis=-1)
    P = (np.abs(dc) ** 2).sum(0)
    assert np.abs(out["rs"][0] - rs).max() <= 1e-12 * np.abs(rs).max()
    assert np.abs(out["dc"][0] - dc).max() <= 1e-12 * np.abs(dc).max()
    assert np.abs(out["P"][0] - P).max() <= 1e-12 * P.max()
    # CFAR, brute force in numpy: every window cell added one by one (a shifted copy of the map per offset); range clamps
    # (rows outside the map are zeros and are not counted), Doppler wraps
    Gr, Gd, Tr, Td, alpha = 2, 2, 8, 4, 15.0
    Wr, Wd = Gr + Tr, Gd + Td

    def box(hr, hd):
        Pz = np.pad(P, ((hr, hr), (0, 0)))
        tot = np.zeros_like(P)
        for i in range(2 * hr + 1):
            for j in range(-hd, hd + 1):
                tot += np.roll(Pz[i:i + Sp], -j, axis=1)
        rows = np.minimum(np.arange(Sp) + hr, Sp - 1) - np.maximum(np.arange(Sp) - hr, 0) + 1
        return tot, rows[:, None] * (2 * hd + 1)

    (wt, wn), (gt, gn) = box(Wr, Wd), box(Gr, Gd)
    noise = (wt - gt) / (wn - gn)
    thr = alpha * noise
    near = np.abs(P - thr) <= 1e-9 * thr
    assert np.allclose(out["noise"][0], noise, rtol=1e-6)
    assert np.array_equal(out["mask"][0][~near], (P > thr)[~near].astype(np.uint8))
    # detections: ordered by (r, d), angle and grouping consistent with their definitions
    dets = out["dets"]
    keys = dets["range_bin"].astype(np.int64) * Cp + dets["doppler_bin"]
    assert np.all(np.diff(keys) > 0) and len(dets) == out["mask"][0].sum() == out["n_total"]
    nth = orc.angle_fft_size(A)
    for d in dets[:: max(1, len(dets) // 16)]:
        x = dc[:, d["range_bin"], d["doppler_bin"]]
        Y = np.abs(np.fft.fft(x, n=nth)) ** 2
        k = int(np.argmax(Y))
        kw = k if k < nth // 2 else k - nth
        top2 = np.sort(Y)[-2:]
        if top2[0] < top2[1] * (1 - 1e-9):
            assert d["angle_bin"] == kw
            assert abs(d["angle_rad"] - np.arcsin(np.clip(2.0 * kw / nth, -1, 1))) < 1e-6
    m = out["mask"][0].astype(bool)
    for d in dets:
        r, dd = int(d["range_bin"]), int(d["doppler_bin"])
        nb = [((r + i), (dd + j) % Cp) for i in (-1, 0, 1) for j in (-1, 0, 1) if (i or j) and 0 <= r + i < Sp]
        nb = [(a, b) for a, b in nb if m[a, b]]
        is_peak = all(P[r, dd] > P[a, b] or (P[r, dd] == P[a, b] and (r, dd) < (a, b)) for a, b in nb)
        assert bool(d["flags"] & 1) == is_peak


def test_multithreaded_oracle_equals_single_thread(orc, pkg):
    S, C, A, F = 64, 64, 4, 5
    adc = pkg.synth.cube_batch(F, S, C, A, cfg=2)
    wr, wd = orc.hann_periodic(S), orc.hann_periodic(C)
    a = orc.process_frames(adc, F, S, C, A, wr, wd, n_threads=1)
    b = orc.process_frames(adc, F, S, C, A, wr, wd, n_threads=4)
    assert a["n_total"] == b["n_total"] and np.array_equal(a["dets"], b["dets"])
    assert np.all(np.diff(a["dets"]["frame"].astype(np.int64)) >= 0)


def test_empty_and_ragged_inputs(orc):
    # noise-free zero cube: nothing detected (P == 0 is never > alpha * 0)
    S, C, A = 64, 64, 2
    adc = np.zeros((1, 2 * S * C * A), np.int16)
    out = orc.process_frames(adc, 1, S, C, A, orc.hann_periodic(S), orc.hann_periodic(C))
    assert out["n_total"] == 0 and len(out["dets"]) == 0
    # capacity smaller than the number of hits: list truncated in order, total still reported
    rng = np.random.default_rng(0)
    adc = rng.integers(-2000, 2000, (1, 2 * S * C * A)).astype(np.int16)
    full = orc.process_frames(adc, 1, S, C, A, orc.hann_periodic(S), orc.hann_periodic(C), alpha=1.5)
    cut = orc.process_frames(adc, 1, S, C, A, orc.hann_periodic(S), orc.hann_periodic(C), alpha=1.5, det_cap_per_frame=7)
    assert full["n_total"] > 7 and cut["n_total"] == full["n_total"] and np.array_equal(cut["dets"], full["dets"][:7])


def _chain_golden_cases(golden_dir):
    g = np.load(f"{golden_dir}/chain_numpy.npz")
    return g, [tuple(int(v) for v in row) for row in g["cases"]]


def test_oracle_matches_numpy_golden_fixture(orc, pkg, golden_dir):
    """tests/golden/chain_numpy.npz (numpy.fft + brute-force sums, generated without oracle code) pins the oracle's
    north-star stages: power map to 1e-12, hit cells exactly away from threshold, angle bins away from ties, peak flags."""
    import hashlib

    g, cases = _chain_golden_cases(golden_dir)
    for (S, C, A, F, cfg) in cases:
        tag = f"{S}x{C}x{A}"
        adc = pkg.synth.cube_batch(F, S, C, A, cfg=cfg, n_targets=4)
        assert hashlib.sha256(adc.tobytes()).digest() == g[f"adc_sha256_{tag}"].tobytes()      # the synthetic input is reproducible
        Sp, Cp = orc.next_pow2(S), orc.next_pow2(C)
        out = orc.process_frames(adc, F, S, C, A, orc.hann_periodic(S), orc.hann_periodic(C), want=("P", "mask", "noise"))
        for f in range(F):
            P = g[f"P_{tag}_f{f}"]
            assert np.abs(out["P"][f] - P).max() <= 1e-12 * P.max()
            mask = np.unpackbits(g[f"mask_{tag}_f{f}"])[: Sp * Cp].reshape(Sp, Cp).astype(bool)
            near = np.unpackbits(g[f"near_{tag}_f{f}"])[: Sp * Cp].reshape(Sp, Cp).astype(bool)
            assert np.array_equal(out["mask"][f].astype(bool)[~near], mask[~near])
            dets = out["dets"][out["dets"]["frame"] == f]
            by = {(int(d["range_bin"]), int(d["doppler_bin"])): d for d in dets}
            for (r, d), nz, ab, tie, pk in zip(g[f"hits_{tag}_f{f}"], g[f"noise_at_hits_{tag}_f{f}"], g[f"angle_bin_{tag}_f{f}"],
                                               g[f"angle_tie_{tag}_f{f}"], g[f"peak_{tag}_f{f}"]):
                if near[r, d]:
                    continue
                rec = by[(int(r), int(d))]
                assert abs(rec["noise"] - nz) <= 1e-6 * nz and bool(rec["flags"] & 1) == bool(pk)
                if not tie:
                    assert rec["angle_bin"] == ab
