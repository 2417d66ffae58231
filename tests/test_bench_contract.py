"""bench.py's reference arm runs on the host alone (no GPU): the JSON line the driver parses must carry the contract's
keys for both kinds of baseline — the reference's own CPU code (cfg1, kind "reference" where oracle/_ref was built) and
the oracle port (kind "port") for the stages the reference does not have."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "cpu_baseline", "e2e"}


def _run(args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"] + args, capture_output=True, text=True,
                       timeout=600, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr
    return r.stdout


def test_reference_arm_legacy_workload(orc):
    out = _run(["--workload", "cfg1", "--steps", "1", "--warmup", "0"])
    lines = [l for l in out.splitlines() if l.strip()]
    assert len(lines) == 1                                   # exactly one JSON line on stdout
    d = json.loads(lines[0])
    assert KEYS <= set(d) and d["impl"] == "reference" and d["unit"] == "frames/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == ("reference" if orc.have_ref() else "port") and d["cpu_baseline"]["cores"] == 1
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["higher_is_better"] is True


def test_reference_arm_chain_workload_and_nonzero_ranks_stay_silent():
    d = json.loads(_run(["--workload", "cfg2", "--steps", "1", "--warmup", "0"]).strip())
    assert KEYS <= set(d) and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert "256 samples x 128 chirps x 4 antennas" in d["config"]["workload"]
    # the GPU arm's workload keys under the GPU arm's names (the bounded CPU sample is named separately)
    assert d["config"]["frames_per_gpu_per_step"] == 1024 and d["config"]["sample_frames_per_step"] > 0
    # under torchrun only rank 0 works and prints
    assert _run(["--workload", "cfg2", "--steps", "1", "--warmup", "0"], env={"RANK": "1", "WORLD_SIZE": "2"}).strip() == ""


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout == ""


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_bounded_seeded_sample(tmp_path):
    """past 64 MB the dump keeps one fixed sample of rows, the same rows from every array"""
    import numpy as np

    bench = _bench_module()
    n = 3_000_000
    rows = {"frame": np.arange(n, dtype=np.uint32), "power": np.arange(n, dtype=np.float32) * 0.5, "flags": (np.arange(n) % 3).astype(np.uint16)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), rows)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["flags.npy", "frame.npy", "power.npy", "sample_index.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 1000 * 1000
    a = {f: np.load(tmp_path / "a" / f) for f in files}
    assert a["frame.npy"].dtype == np.float64 and a["power.npy"].dtype == np.float32 and a["flags.npy"].dtype == np.float32
    idx = a["sample_index.npy"].astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    assert np.array_equal(a["frame.npy"], idx) and np.array_equal(a["power.npy"], idx * 0.5) and np.array_equal(a["flags.npy"], idx % 3)
    assert all(np.array_equal(a[f], np.load(tmp_path / "b" / f)) for f in files)


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_batch(pkg, tmp_path):
    """cfg2 at 8 frames, 5 timed steps round-robin over 3 batches in flight: the last step ran lane 1 (frames 8..15), and
    --dump-outputs holds the list the library returns for that batch, field by field"""
    import numpy as np
    import torch

    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg2", "--frames", "8", "--steps", "5",
                        "--warmup", "3", "--inflight", "3", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 5
    S, C, A, F = 256, 128, 4, 8
    adc = pkg.synth.cube_batch_torch(F, S, C, A, torch.device("cuda", 0), cfg=2, first_frame=F)
    with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096) as ctx:
        ctx.set_detect_path(pkg.api.DETECT_REFFT)
        ctx.set_frame_offset(F)
        ctx.process_device(adc, F)
        want, overflow = ctx.read_detections()
    assert len(want) > 0 and not overflow
    assert sorted(os.listdir(out)) == sorted(f"{n}.npy" for n in pkg.DET_DTYPE.names)
    for name in pkg.DET_DTYPE.names:
        got = np.load(out / f"{name}.npy")
        assert got.dtype in (np.float32, np.float64) and np.array_equal(got, want[name]), name


@pytest.mark.gpu
def test_dump_outputs_hold_every_call_of_the_last_cfg5_tick(pkg, tmp_path):
    """cfg5 with 4 sensors: the dump holds the lists of all four one-frame calls of the last tick, in sensor order, each
    equal to the list the library returns for that sensor's frame"""
    import numpy as np
    import torch

    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg5", "--frames", "4", "--steps", "2",
                        "--warmup", "3", "--depth", "2", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    S, C, A = 256, 128, 12
    want = []
    with pkg.RadarContext(S, C, A, 1, max_det_per_frame=4096) as ctx:
        for x in range(4):
            ctx.process_device(pkg.synth.cube_batch_torch(1, S, C, A, torch.device("cuda", 0), cfg=5, first_frame=x), 1)
            want.append(ctx.read_detections()[0])
    assert all(len(d) > 0 for d in want)
    assert np.array_equal(np.load(out / "sensor.npy"), np.repeat(np.arange(4), [len(d) for d in want]))
    whole = np.concatenate(want)
    for name in pkg.DET_DTYPE.names:
        assert np.array_equal(np.load(out / f"{name}.npy"), whole[name]), name
