"""Shared by the GPU tests that check the CUDA chain against the CPU oracle (test_gpu_bench_paths.py, test_gpu_parity.py,
test_gpu_kernel_forms.py): the strict comparison of a processed batch with the oracle (check_frames), and the names of
the kernels the library compiles and a run launches, so that a test can assert which kernel form it checked.

Tolerances (north_star: fp32 relative error 1e-4 for FFT outputs and power maps; CFAR indices bit-exact except cells
within 1e-5 relative of threshold, which are listed):
  power map   |P - P_ref| <= 2e-6 * max(P_ref) everywhere, AND per-bin relative error <= 1e-5 for every bin above
              1e-3 * max(P_ref) (per-bin relative error is meaningless on near-empty bins: SURVEY.md §7); the measured
              maxima are printed (north_star's bound is 1e-4)
  CFAR mask   bit-exact except cells with |P - alpha * noise| <= 1e-5 * alpha * noise (counted and printed)
  list        keys (frame, range, doppler) in order, identical to the oracle's away from those cells; counts exact
  noise       relative error <= NOISE_RTOL (see below) at every detection
  angle bin   identical unless the oracle's angle spectrum has a second bin within 1e-4 of the maximum
  peak flag   identical unless a detected neighbour's power is within 1e-4 of the cell's, or a threshold cell is adjacent
"""
import contextlib
import os
import re
import subprocess

import numpy as np

ALPHA = 15.0
NEAR = 1e-5
P_ATOL_OF_MAX = 2e-6            # measured on B200: 1.6e-7 .. 3.7e-7 (profiles/r2/parity_maxima_bench_paths.log: test_gpu_bench_paths.py run with -s)
P_RTOL_ABOVE_FLOOR = 1e-5       # measured: 2.4e-7 .. 7.0e-7; north_star allows 1e-4
P_FLOOR_OF_MAX = 1e-3
# The noise estimate is the mean of 248 power-map cells near the noise floor.  Its fp32 sum is add-only (~1e-6), but
# each of those cells carries the fp32 FFT's error, which is relative to the RMS of the whole transform (dominated by
# targets ~1e9 x the floor), not to the cell: ~1e-4 per cell, averaging down over the window.  Measured on B200: 1.4e-6 ..
# 1.05e-5 (the largest on one of the 7 858 detections of the cfg3 batch).
NOISE_RTOL = 3e-5


def check_frames(pkg, orc, ctx, dets, adc, frames, S, C, A, tag, n_threads=8, base=None):
    """compares frames `frames` of the batch just processed on `ctx` (detections `dets`) with the oracle run on those frames;
    `base`: the frame set with ctx.set_base_frame, subtracted by the oracle too"""
    wr, wd = ctx.get_windows()
    sub = np.ascontiguousarray(adc[frames])
    ref = orc.process_frames(sub, len(frames), S, C, A, wr, wd, want=("P", "mask", "noise", "ratio"), n_threads=n_threads,
                             det_cap_per_frame=ctx.max_det_per_frame, base=base)
    stats = dict(p_abs=0.0, p_rel=0.0, near=0, n_det=0, noise_rel=0.0, angle_ties=0, flag_skipped=0)
    for i, f in enumerate(frames):
        Pr, maskr, noiser = ref["P"][i], ref["mask"][i], ref["noise"][i]
        P = ctx.power_map(f).astype(np.float64)
        pmax = Pr.max()
        err = np.abs(P - Pr)
        stats["p_abs"] = max(stats["p_abs"], float(err.max() / pmax))
        assert err.max() <= P_ATOL_OF_MAX * pmax, f"{tag} frame {f}: power map off by {err.max() / pmax:.2e} of its maximum"
        big = Pr >= P_FLOOR_OF_MAX * pmax
        rel = float((err[big] / Pr[big]).max())
        stats["p_rel"] = max(stats["p_rel"], rel)
        assert rel <= P_RTOL_ABOVE_FLOOR, f"{tag} frame {f}: per-bin relative error {rel:.2e} above the floor"
        thr = ALPHA * noiser
        near = np.abs(Pr - thr) <= NEAR * thr
        stats["near"] += int(near.sum())
        m = ctx.cfar_mask(f)
        bad = (m != maskr) & ~near
        assert not bad.any(), f"{tag} frame {f}: {int(bad.sum())} CFAR cells differ away from threshold"
        # detection list of this frame
        got = dets[dets["frame"] == f]
        want = ref["dets"][ref["dets"]["frame"] == i]
        ratio = ref["ratio"][ref["dets"]["frame"] == i]
        assert len(got) == int(m.sum()), f"{tag} frame {f}: list length {len(got)} != mask population {int(m.sum())}"
        gk = got["range_bin"].astype(np.int64) << 16 | got["doppler_bin"]
        wk = want["range_bin"].astype(np.int64) << 16 | want["doppler_bin"]
        assert np.all(np.diff(gk) > 0), f"{tag} frame {f}: list not ordered by (range, doppler)"
        diff = np.setxor1d(gk, wk)
        assert all(near[k >> 16, k & 0xffff] for k in diff), f"{tag} frame {f}: hit list differs away from threshold cells"
        common, gi, wi = np.intersect1d(gk, wk, return_indices=True)
        g, w, rt = got[gi], want[wi], ratio[wi]
        stats["n_det"] += len(common)
        assert len(common) > 0, f"{tag} frame {f}: no detections to compare"
        assert np.abs(g["power"].astype(np.float64) - w["power"]).max() <= P_ATOL_OF_MAX * pmax
        nrel = np.abs(g["noise"].astype(np.float64) - w["noise"]) / w["noise"]
        stats["noise_rel"] = max(stats["noise_rel"], float(nrel.max()))
        assert nrel.max() <= NOISE_RTOL, f"{tag} frame {f}: noise estimate off by {nrel.max():.2e} (relative)"
        clear = rt < 1 - 1e-4
        stats["angle_ties"] += int((~clear).sum())
        assert np.array_equal(g["angle_bin"][clear], w["angle_bin"][clear]), f"{tag} frame {f}: angle bins differ away from ties"
        assert np.abs(g["angle_rad"][clear] - w["angle_rad"][clear]).max(initial=0.0) < 1e-5
        # grouping flag
        Sp, Cp = Pr.shape
        r, d = w["range_bin"].astype(np.int64), w["doppler_bin"].astype(np.int64)
        ok = np.ones(len(w), bool)
        for dr in (-1, 0, 1):
            for dd in (-1, 0, 1):
                rr, dn = r + dr, (d + dd) % Cp
                inside = (rr >= 0) & (rr < Sp)
                rr = rr.clip(0, Sp - 1)
                ok &= ~(inside & near[rr, dn])
                if dr or dd:
                    close = inside & (maskr[rr, dn] != 0) & (np.abs(Pr[rr, dn] - Pr[r, d]) <= 1e-4 * Pr[r, d])
                    ok &= ~close
        stats["flag_skipped"] += int((~ok).sum())
        assert np.array_equal(g["flags"][ok] & 1, w["flags"][ok] & 1), f"{tag} frame {f}: peak flags differ"
    print(f"\n{tag}: frames {list(frames)}: {stats['n_det']} detections compared; power map max error {stats['p_abs']:.2e} of max, "
          f"{stats['p_rel']:.2e} per bin above {P_FLOOR_OF_MAX} of max; noise max rel error {stats['noise_rel']:.2e}; "
          f"{stats['near']} threshold cells excluded, {stats['angle_ties']} angle ties, {stats['flag_skipped']} flags skipped")
    return stats


def kernel_form(name: str) -> str:
    """'void mmw::k<1, true>(mmw::PlanDev, int)' -> 'k<1, true>': the kernel's name with its template arguments.  The
    CUDA demangler writes template arguments with their types ('k<(int)1, (bool)1>', '<unnamed>::'), the C++ one
    without: both come out as the latter."""
    s = " ".join(name.split())
    s = re.sub(r"\((?:int|unsigned int|long)\)(-?\d+)", r"\1", s)
    s = s.replace("(bool)1", "true").replace("(bool)0", "false").replace("<unnamed>", "(anonymous namespace)")
    if s.startswith("void "):
        s = s[5:]
    if s.endswith(")"):                                   # drop the parameter list: the last balanced (...)
        depth = 0
        for i in range(len(s) - 1, -1, -1):
            depth += {")": 1, "(": -1}.get(s[i], 0)
            if depth == 0:
                s = s[:i]
                break
    return s.replace("mmw::", "")


def compiled_forms(pkg) -> set:
    """the kernels in the built library: cuobjdump and cu++filt of the toolkit build.py compiles with"""
    bindir = os.path.dirname(pkg.build._nvcc())
    out = subprocess.run([os.path.join(bindir, "cuobjdump"), "-res-usage", pkg.build.LIB], capture_output=True, text=True,
                         check=True).stdout
    mangled = [ln.split()[1].rstrip(":") for ln in out.splitlines() if ln.strip().startswith("Function ")]
    assert mangled, "cuobjdump lists no kernel in the library"
    names = subprocess.run([os.path.join(bindir, "cu++filt")], input="\n".join(mangled), capture_output=True, text=True,
                           check=True).stdout.split("\n")
    return {kernel_form(n) for n in names if n.strip()}


@contextlib.contextmanager
def launched_kernels():
    """collects the names of the CUDA kernels launched inside the block (torch.profiler sees every kernel of the process)"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    names = set()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], acc_events=True) as prof:
        yield names
        torch.cuda.synchronize()
    names.update(kernel_form(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)


# (strip height, Doppler segments, Sp specialisation) of the CFAR walk kernel, as launch_cfar / run_cfar_walk pick them:
# every cfar_walk_kernel<RT, MINB, SPT> the library compiles, each strip height with each segment length; None is the
# tiled cfar_kernel.  test_gpu_parity.py::test_cfar_kernel_forms_agree_with_oracle checks each of them.
WALK_FORMS = [None, (64, 2, 0), (64, 2, 256), (64, 2, 512), (64, 2, 1024), (64, 4, 0), (64, 8, 0),
              (128, 2, 0), (128, 2, 256), (128, 2, 512), (128, 2, 1024), (128, 4, 0), (128, 8, 0),
              (256, 2, 256), (256, 2, 512), (256, 2, 1024), (256, 4, 256), (256, 4, 512), (256, 4, 1024), (256, 8, 256),
              (256, 8, 512)]
WALK_MINB = {64: 8, 128: 5, 256: 3}            # launch_cfar: run_cfar_walk<RT, MINB>


def cfar_form_name(form) -> str:
    """the kernel a WALK_FORMS entry names (Doppler segments are a run-time argument, not part of it)"""
    if form is None:
        return "cfar_kernel"
    rt, _, spt = form
    return f"cfar_walk_kernel<{rt}, {WALK_MINB[rt]}, {spt}>"
