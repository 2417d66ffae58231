"""Generates tests/golden/legacy_reference.npz and legacy_reference_direct.npz from the REFERENCE's
own CPU functions.

Run where the reference's sources are (oracle/Makefile, REF):  python tests/golden/make_golden.py
It calls the reference code compiled by oracle/Makefile into oracle/_ref/libref_cpu.so
(ReshapeComplex_t, butterfly_fft, FindAbsMax and the cpuTiming() loop body,
cudaBenchMarking.cpp:61-105, :149-206, :273-303) on seeded synthetic captures in the
fhy_direct.bin format and stores the outputs.  A checkout without those sources tests against
these files alone.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
orc = entry.load_oracle()
orc.build()
assert orc.have_ref(), "oracle/_ref/libref_cpu.so missing: /root/reference not present?"

out = {}
# (1) known-answer test: the reference's own fftTest() input, ramp 1..16 (acceleration.cu:361-365)
ramp = np.arange(1, 17).astype(np.complex128)
out["kat_ramp16_in"] = ramp
out["kat_ramp16_out"] = orc.ref_fft(ramp)
# (2) indexing spot checks of ReshapeComplex_t with s[i] = i (SURVEY.md §4)
s = (np.arange(102400) % 32768).astype(np.int16)
y = orc.ref_reshape(s)
idx = np.array([0, 1, 2, 100, 12799, 12800, 25000, 37035, 51199])
out["reshape_idx"] = idx
out["reshape_val"] = y[idx]
# (3) end-to-end: seeded captures through the reference frame loop
seeds = [0, 1, 2]
frames_per_seed = 6
out["cap_seeds"] = np.array(seeds)
out["cap_frames"] = np.array(frames_per_seed)
dist, raw, probes = [], [], []
probe_bins = np.array([0, 1, 163, 164, 1966, 2015, 4096, 6552, 10922, 10923, 16383])
out["probe_bins"] = probe_bins
for sd in seeds:
    cap = pkg.synth.legacy_capture(frames_per_seed, seed=sd, moving=(sd == 2))
    base = orc.ref_reshape(cap[0])[:12800]
    for f in range(1, frames_per_seed):
        d, r, spec = orc.ref_cpu_frame(cap[f], base, want_spectrum=True)
        dist.append(d)
        raw.append(r)
        probes.append(spec[probe_bins])
out["dist"] = np.array(dist)
out["raw"] = np.array(raw, np.int32)
out["spec_probes"] = np.array(probes)
# (4) random-input FFT vectors at the sizes the chain uses
rng = np.random.default_rng(42)
for n in (64, 128, 256, 512, 1024):
    x = rng.normal(size=n) + 1j * rng.normal(size=n)
    out[f"fft{n}_in"] = x
    out[f"fft{n}_out"] = orc.ref_fft(x)
path = os.path.join(ROOT, "tests", "golden", "legacy_reference.npz")
np.savez_compressed(path, **out)
print("wrote", path, os.path.getsize(path), "bytes")
# (5) the direct comparison of tests/test_oracle_pin.py::test_against_compiled_reference, for checkouts without oracle/_ref
direct = orc.direct_vectors(pkg.synth.legacy_capture(4, seed=11), orc.ref_reshape, orc.ref_cpu_frame, orc.ref_fft,
                            orc.ref().ref_next_pow2, sample=True)
path = os.path.join(ROOT, "tests", "golden", "legacy_reference_direct.npz")
np.savez_compressed(path, **direct)
print("wrote", path, os.path.getsize(path), "bytes")
