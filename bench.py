#!/usr/bin/env python
"""bench.py — radar frames/s (ADC cube -> detections) on N B200s, with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg3|cfg2|cfg4|cfg5|cfg1] [--impl ours|reference]
                    [--dump-outputs DIR]

A step = one pass of the whole chain (range FFT -> Doppler FFT + |X|^2 integration -> 2-D CA-CFAR ->
detection records incl. angle FFT + grouping -> dense list) over one batch of synthetic frames per GPU.
  value  frames/s with the batch already resident in HBM (device-timed, max over ranks; for N > 1 the
         timed step includes the NCCL gather of the detection lists to rank 0)
  e2e    frames/s through the host-facing C-ABI call mmw_process_host(): pinned-host capture -> H2D ->
         chain -> D2H of the ordered detection list, every step
  roofline      dominant kernel: algorithmic bytes per launch / CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline  the plain-C oracle (oracle/mmw_oracle.c, kind "port": the reference has no CPU code for
                these stages) timed on the box's host cores on a bounded sample of the same workload
Workloads (BASELINE.json configs):
  cfg3  512 samples x 256 chirps x 12 virtual antennas — the shape north_star's >= 60 % roofline target is quoted on (default)
  cfg2  256 x 128 x 4, batch of 1024 frames (configs[1])
  cfg4  1024 x 512 x 192 imaging cube, 4 frames per GPU per step (configs[3])
  cfg5  64 sensors x (256 x 128 x 12): latency mode — every frame is its own call; p50/p99 per-frame latency (configs[4])
  cfg1  the reference's own path (100 x 128 x 4, rx0, base-frame subtraction, one 16 384-point FFT, arg-max -> metres)
        through the drop-in library; its CPU baseline is the reference's own code (oracle/_ref, kind "reference") (configs[0])
--dump-outputs DIR writes what the last timed step returned, one DIR/<name>.npy per array (the inputs are seeded, so two
builds run with the same arguments can be compared output for output):
  cfg2/cfg3/cfg4  the ordered detection list of the last batch (rank 0's merged list for N > 1), one array per record field
  cfg5            the detection lists of the last tick's one-frame calls, one after another, with a sensor column (rank 0's
                  sensors for N > 1); the device keeps only the last call's list, so the tick is replayed untimed and
                  read call by call, and its last call is checked against the list the timed loop left
  cfg1            raw_bin: the arg-max bin of every frame of the last batch (rank 0's for N > 1)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

METRIC = "radar frames/sec (ADC cube->detections)"
WORKLOADS = {
    # name: kind, S, C, A, frames per GPU per step, BASELINE.json config index
    "cfg3": dict(kind="chain", S=512, C=256, A=12, F=64, idx=2),
    # detect_path=2 (MMW_DETECT_REFFT): 83 k detections per batch — the hit rows are re-transformed once instead of a DFT per
    # detection (list + measure 0.135 -> 0.08 ms; profiles/r2/sweep_k4x_narrow.log); the other shapes keep the library's default
    "cfg2": dict(kind="chain", S=256, C=128, A=4, F=1024, idx=1, detect_path=2),
    "cfg4": dict(kind="chain", S=1024, C=512, A=192, F=4, idx=3),
    "cfg5": dict(kind="stream", S=256, C=128, A=12, F=64, idx=4),
    "cfg1": dict(kind="legacy", S=100, C=128, A=4, F=4096, idx=0),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


class CpuPort:
    """The plain-C oracle (fp64, radix-2 FFTs, frame-parallel with OpenMP) as a CPU baseline: a fixed pool of
    distinct synthetic frames of the workload, processed over and over until the requested amount of work is done."""

    def __init__(self, orc, pkg, S, C, A, cfg_id, cores):
        big = S * C * A > 16 * 1024 * 1024                              # cfg4: 1.6 GB of fp64 scratch per thread
        self.cores = min(cores, 2) if big else cores
        self.orc, self.S, self.C, self.A = orc, S, C, A
        self.pool = pkg.synth.cube_batch(2 if big else max(cores, 8), S, C, A, cfg=cfg_id)
        self.wr, self.wd = orc.hann_periodic(S), orc.hann_periodic(C)
        if not big:
            self.run(1)                                                  # touch code and pages

    def run(self, passes):
        """processes `passes` x pool frames; returns (frames, seconds, detections of the last pass)"""
        n = self.pool.shape[0]
        t0 = time.perf_counter()
        for _ in range(passes):
            out = self.orc.process_frames(self.pool, n, self.S, self.C, self.A, self.wr, self.wd, n_threads=self.cores)
        return passes * n, time.perf_counter() - t0, int(out["n_total"])

    def passes_for(self, seconds):
        n, dt, _ = self.run(1)
        return max(1, int(round(seconds / max(dt, 1e-6))))


class LegacyCpu:
    """cfg1: the reference's own CPU loop body (oracle/_ref/libref_cpu.so, compiled from /root/reference: kind
    "reference"), or the bit-identical oracle restatement where oracle/_ref was not built (kind "port").
    Single-threaded like the reference."""

    def __init__(self, orc, pkg):
        self.orc = orc
        self.cap = pkg.synth.legacy_capture(33, seed=0)
        self.base = orc.reshape(self.cap[0], 100, 128, 4)[:12800]
        self.kind = "reference" if orc.have_ref() else "port"

    def run(self, passes):
        t = 0.0
        for _ in range(passes):
            if self.kind == "reference":
                dt, _ = self.orc.ref_cpu_time_frames(self.cap[1:], self.base)
            else:
                t0 = time.perf_counter()
                for f in range(1, self.cap.shape[0]):
                    self.orc.legacy_frame(self.cap[f], self.base)
                dt = time.perf_counter() - t0
            t += dt
        return passes * (self.cap.shape[0] - 1), t

    def passes_for(self, seconds):
        n, dt = self.run(1)
        return max(1, int(round(seconds / max(dt, 1e-6))))


def workload_text(name):
    w = WORKLOADS[name]
    if w["kind"] == "legacy":
        return (f"cfg1: reference path, 100 samples x 128 chirps x 4 rx per frame, rx0 - base frame, 16384-pt FFT, arg-max -> metres "
                f"(BASELINE.json configs[{w['idx']}])")
    return f"{name}: {w['S']} samples x {w['C']} chirps x {w['A']} antennas"


def chain_workload_text(name):
    """config.workload of the batched chain: the same string on both arms"""
    w = WORKLOADS[name]
    n_theta = 64 if w["A"] <= 64 else 1 << (w["A"] - 1).bit_length()
    return (f"{workload_text(name)}, 2-D CA-CFAR (guard 2x2, train 8x4, alpha 15), {n_theta}-pt angle FFT "
            f"(BASELINE.json configs[{w['idx']}])")


DUMP_BYTES = 64 * 1000 * 1000


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in the narrowest of float32 / float64 that holds it exactly (float32
    for 16-bit integers and 4-byte floats, float64 otherwise).  All arrays are rows of one table (one entry per detection
    or frame); past DUMP_BYTES in all, the same fixed, seeded sample of rows is kept from each and its row numbers go to
    sample_index.npy."""
    arrays = {k: a.astype(np.float64 if a.dtype.itemsize > 4 or (a.dtype.kind != "f" and a.dtype.itemsize > 2) else np.float32)
              for k, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    keep = (DUMP_BYTES - 1024 * (len(arrays) + 1)) // (sum(a.itemsize for a in arrays.values()) + 8)     # 1 KB per .npy header
    if n > keep:
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["sample_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def detection_fields(dets):
    return {name: dets[name] for name in dets.dtype.names}


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores.  cfg1: the reference's own
    code (oracle/_ref).  Other workloads: the reference has no CPU (or GPU) code for the range/Doppler/CFAR/angle chain
    (SURVEY.md §0), so per north_star the plain-C oracle port stands in (kind "port"), frame-parallel on all host cores."""
    if rank != 0:
        return
    pkg, orc = entry.load_package(), entry.load_oracle()
    orc.build()
    w = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    if w["kind"] == "legacy":
        port = LegacyCpu(orc, pkg)
        passes, kind, used = port.passes_for(1.0), port.kind, 1
        run = lambda: port.run(passes)[:2]                                  # noqa: E731
        what = "the reference's own cpuTiming() loop body compiled from /root/reference" if kind == "reference" else "oracle restatement of the reference CPU loop"
    else:
        port = CpuPort(orc, pkg, w["S"], w["C"], w["A"], w["idx"] + 1, cores)
        passes, kind, used = port.passes_for(1.0), "port", port.cores
        run = lambda: port.run(passes)[:2]                                  # noqa: E731
        what = "plain-C fp64 oracle (the reference has no CPU code for these stages)"
    times, per_step = [], 0
    for i in range(args.warmup + args.steps):
        per_step, dt = run()
        if i >= args.warmup:
            times.append(dt)
    T = float(np.sum(times))
    value = per_step * len(times) / T
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * T / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        # the GPU arm's workload keys under the GPU arm's names; a step here is a bounded sample of that workload
        "config": {"workload": workload_text(args.workload) if w["kind"] == "legacy" else chain_workload_text(args.workload),
                   "frames_per_gpu_per_step": args.frames or w["F"], "sample_frames_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": used, "kind": kind,
                         "sample": f"{per_step} frames per step x {len(times)} steps, {what}, {used} thread(s)"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class Env:
    """torch / distributed / stdout plumbing shared by the three workload kinds"""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
        # keep stdout for the one JSON line: libraries (NCCL's version banner) write to fd 1 during init
        sys.stdout.flush()
        self.real_stdout = os.dup(1)
        os.dup2(2, 1)
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.numa = self.bind_to_gpu_numa_node()
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", rank=self.rank, world_size=self.world, device_id=self.dev)
        self.pkg = entry.load_package()

    def bind_to_gpu_numa_node(self):
        """Multi-rank runs: pin this process (and, by first touch, its pinned host buffers) to the CPUs of the NUMA node
        its GPU hangs off, so that the H2D copies of the end-to-end path do not cross sockets.  Returns the node or None."""
        if self.world == 1:
            return None
        try:
            pr = self.torch.cuda.get_device_properties(self.local_rank)
            bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
            if node < 0:
                return None
            cpus = set()
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
            cpus &= os.sched_getaffinity(0)
            if not cpus:
                return None
            os.sched_setaffinity(0, cpus)
            return node
        except (OSError, ValueError, AttributeError):
            return None

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def all_ranks(self, x: float):
        if self.world == 1:
            return [x]
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        out = self.torch.empty(self.world, device=self.dev, dtype=self.torch.float64)
        self.dist.all_gather_into_tensor(out, t)
        return [float(v) for v in out.cpu()]

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def emit(self, line):
        sys.stdout.flush()
        os.dup2(self.real_stdout, 1)
        print(json.dumps(line), flush=True)

    def finish(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` at the workload's bench batch size, read from the
    newest committed `ncu --set full` capture of that workload (profiles/ncu_rN_stages_<workload>_raw.csv, written by
    profiles/ncu_stage_table.py).  Returns (bytes, file name) or (None, None) when no capture names that kernel."""
    import csv
    import glob
    import re

    best = None
    for path in glob.glob(os.path.join(ROOT, "profiles", f"ncu_r*_stages_{workload}_raw.csv")):
        m = re.search(r"ncu_r(\d+)_stages_", os.path.basename(path))
        if m and (best is None or int(m.group(1)) > best[0]):
            best = (int(m.group(1)), path)
    if best is None:
        return None, None
    rows = list(csv.reader(open(best[1])))
    hdr, units = rows[0], rows[1]
    ix = {h: i for i, h in enumerate(hdr)}
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    want = kernel.split("+")[0]
    for r in rows[2:]:
        if want in r[ix["Kernel Name"]]:
            tot = sum(float(r[ix[k]]) * scale[units[ix[k]]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
            return int(tot), os.path.relpath(best[1], ROOT)
    return None, None


STAGE_NAMES = ["range_fft_kernel", "doppler_fft_kernel", "cfar_kernel", "list_kernel+measure_kernel"]
# per-frame detection capacity the bench gives each workload (the dense imaging scene of cfg4 yields ~10 k hits per frame)
MAX_DET = {"cfg2": 4096, "cfg3": 4096, "cfg4": 32768}


def measure_chain(env, name, F, K, W, D, keep_cube=False, e2e_steps=None, share_input=False, keep_outputs=False):
    """One chain workload (cfg2 / cfg3 / cfg4) on every rank: K timed steps with D batches in flight (device-resident input,
    CUDA events, max over ranks; for N > 1 each step ends with the exchange of the detection lists), per-stage times of one
    lane alone, and the end-to-end figure through the host entry points.  Collective: every rank must call it.
    keep_outputs: res["last_dets"] is the detection list of the last timed step (rank 0's merged list for N > 1)."""
    torch, pkg, dev, rank, world = env.torch, env.pkg, env.dev, env.rank, env.world
    w = WORKLOADS[name]
    S, C, A, cfg_idx = w["S"], w["C"], w["A"], w["idx"]
    max_det = MAX_DET[name]
    side = torch.cuda.Stream(device=dev) if world > 1 else None
    host_split = [0.0, 0.0]                                # host seconds inside process_device / inside the exchange's run()
    shared = {}

    class Lane:
        def __init__(self, i):
            self.ctx = pkg.RadarContext(S, C, A, F, keep_doppler_cube=keep_cube, max_det_per_frame=max_det, device=env.local_rank)
            if w.get("detect_path"):
                self.ctx.set_detect_path(w["detect_path"])
            first_frame = (i * world + rank) * F              # weak scaling: every rank owns F frames of each global batch
            self.ctx.set_frame_offset(first_frame)
            if share_input and "adc" in shared:
                self.adc = shared["adc"]                      # side measurements: the lanes read one batch (still larger than L2)
            else:
                self.adc = shared["adc"] = pkg.synth.cube_batch_torch(F, S, C, A, dev, cfg=cfg_idx + 1, first_frame=first_frame)
            self.stream = torch.cuda.Stream(device=dev)
            self.ctx.use_stream(self.stream.cuda_stream)
            self.gather = None

        def step(self):
            with torch.cuda.stream(self.stream):
                t0 = time.perf_counter()
                self.ctx.process_device(self.adc, F)
                t1 = time.perf_counter()
                if self.gather is not None:
                    self.gather.run()
                host_split[0] += t1 - t0
                host_split[1] += time.perf_counter() - t1

        def flush(self):
            if self.gather is not None:
                with torch.cuda.stream(self.stream):
                    self.gather.flush()

    lanes = [Lane(i) for i in range(D)]
    ctx, adc = lanes[0].ctx, lanes[0].adc
    torch.cuda.synchronize()
    dense_ptr, header_ptr = ctx.device_results()
    header_view = pkg.sharding.device_bytes_view(header_ptr, 16, dev)

    # one batch per lane before anything is sized or timed: the detection counts of this scene size the exchange
    for ln in lanes:
        ln.step()
    torch.cuda.synchronize()
    hdr0 = header_view.view(torch.int32).cpu().numpy()
    local_written = int(hdr0[0])
    # exchange step (N > 1 only): NCCL gather of a fixed-size prefix of each rank's result block to rank 0 + one merge kernel,
    # on a side stream behind a snapshot of the block so that it overlaps the next step's kernels (sharding.DetectionGather).
    # The prefix is sized from the warm-up batch (largest count over the ranks + 50 % head-room, whole KB of records):
    # a rank that outgrows it is truncated and flagged (overflow below), never silently.
    gather_records = 0
    if world > 1:
        most = int(max(env.all_ranks(float(local_written))))
        gather_records = min(F * max_det, ((most * 3 // 2 + 1024) // 1024) * 1024)
        for ln in lanes:
            if env.exchange == "peer":
                try:
                    ln.gather = pkg.sharding.PeerDetectionGather(ln.ctx, dev, gather_records)
                except pkg.sharding.PeerExchangeUnavailable as e:   # raised on every rank at once: fall back together
                    if rank == 0:
                        print(f"bench.py: peer exchange unavailable ({e}); using the NCCL gather", file=sys.stderr)
                    env.exchange = "nccl"
            if env.exchange != "peer":
                ln.gather = pkg.sharding.DetectionGather(ln.ctx, dev, gather_records, side=side)
    gather = lanes[0].gather

    for k in range(max(W, D)):
        lanes[k % D].step()
    for ln in lanes:
        ln.flush()
    env.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lanes[0].stream)
    for ln in lanes[1:]:
        ln.stream.wait_event(e0)
    host_split[0] = host_split[1] = 0.0
    t_host = time.perf_counter()
    for k in range(K):
        lanes[k % D].step()
    for ln in lanes:
        ln.flush()                                          # the last steps' gather + merge are inside the timed region
    t_host = (time.perf_counter() - t_host) * 1e3          # host time to ISSUE the K steps (no sync): device-bound if well below ms
    for ln in lanes[1:]:
        ev = torch.cuda.Event()
        ev.record(ln.stream)
        lanes[0].stream.wait_event(ev)
    e1.record(lanes[0].stream)
    env.sync_all()
    ms = e0.elapsed_time(e1)
    ms_by_rank = env.all_ranks(ms)
    host_ms_by_rank = env.all_ranks(t_host)
    ms = max(ms_by_rank)
    last_dets = None
    if keep_outputs:                                        # before the contexts run anything else
        last = lanes[(K - 1) % D]
        if world == 1:
            last_dets = last.ctx.read_detections()[0]
        elif rank == 0:
            last_dets = last.gather.read(pkg.DET_DTYPE)[0]
    frame_counts = ctx.read_counts(F)                       # true per-frame hit counts of this rank's last batch
    hdr = header_view.view(torch.int32).cpu().numpy()
    # the re-FFT detection path (wide arrays in fused mode, or detect_path=2) re-transforms every (frame, range bin) that has
    # hits (doppler_extract_kernel): those rows of the range spectrum are read once more, A * C * 8 bytes each
    hit_rows = 0
    if not keep_cube and int(ctx.info.kernels_per_batch) == 7:
        last = pkg.sharding.records_from_bytes(pkg.sharding.device_bytes_view(dense_ptr, 24 * int(hdr[0]), dev), pkg.DET_DTYPE)
        hit_rows = len(np.unique(last["frame"].astype(np.int64) << 16 | last["range_bin"]))
    local_overflow = int(hdr[3]) or int(frame_counts.max() > max_det)
    if world == 1:
        n_det_step, gather_overflow = int(hdr[0]), 0
    elif rank == 0:
        recs, ghdr = gather.read(pkg.DET_DTYPE)
        n_det_step, gather_overflow = len(recs), int(ghdr[3])
        if os.environ.get("MMW_GATHER_DEBUG", "full") == "full":
            assert np.all(np.diff(recs["frame"].astype(np.int64)) >= 0) and int(ghdr[2]) == world * F     # ordered, all frames accounted for
    else:
        n_det_step, gather_overflow = 0, 0
    overflow = int(max(env.all_ranks(float(local_overflow or gather_overflow))))

    # ---- per-stage device times (events between launches) for the roofline of the dominant kernel ----
    ctx.use_stream(None)
    iters = max(3, min(K, 10))
    total_ms, stage_ms = ctx.time_device(adc, F, iters, per_stage=True)
    stage_ms = [x / iters for x in stage_ms]
    N_adc, N, M = S * C * A, ctx.Sp * ctx.Cp * A, ctx.Sp * ctx.Cp
    stage_bytes = [
        F * (4 * N_adc + 8 * A * ctx.Sp * C),                   # K1: int16 IQ in, range spectrum out
        F * (8 * A * ctx.Sp * C + (8 * N if keep_cube else 0) + 4 * M),   # K2: spectrum in, (cube +) power map out
        F * (4 * M + M // 8),                                   # K3: power map in, bit mask out
        F * (M // 8) + hit_rows * A * C * 8,                    # K4: mask in, hit rows of the range spectrum once more (wide arrays), records out
    ]

    # ---- end to end through the host-facing API: pinned host capture -> H2D -> chain -> D2H list ----
    host = torch.empty((F, ctx.frame_shorts), dtype=torch.int16, pin_memory=True)
    host.copy_(adc)
    torch.cuda.synchronize()
    out = np.empty(F * ctx.max_det_per_frame, pkg.DET_DTYPE)
    e2e_steps = e2e_steps or max(3, min(K, 10))
    # two batches in flight (mmw_submit_host / mmw_wait on two contexts) keep the bus busy while the previous batch's last
    # kernels and read-back finish; with one lane only: the synchronous call
    e2e_ring = [ln.ctx for ln in lanes[:2]]
    for c in e2e_ring:
        c.use_stream(None)

    def e2e_pass(n):
        got = None
        if len(e2e_ring) == 1:
            for _ in range(n):
                got, _ = ctx.process_host(host, F, out=out)
            return got
        for i in range(n + 2):
            c = e2e_ring[i % 2]
            if i >= 2:
                got, _ = c.wait(out=out)
            if i < n:
                c.submit_host(host, F)
        return got

    e2e_pass(2)
    env.sync_all()
    t0 = time.perf_counter()
    dets = e2e_pass(e2e_steps)
    t_e2e = env.max_over_ranks(time.perf_counter() - t0)
    res = dict(
        name=name, F=F, K=K, W=W, D=D, keep_cube=keep_cube, S=S, C=C, A=A, Sp=ctx.Sp, Cp=ctx.Cp,
        fps=world * F * K / (ms * 1e-3), ms=ms, ms_by_rank=ms_by_rank, host_ms_by_rank=host_ms_by_rank,
        host_split=list(host_split), total_ms_one=total_ms / iters, stage_ms=stage_ms, stage_bytes=stage_bytes,
        b_alg=int(ctx.info.algorithmic_bytes_per_frame), kernels_per_batch=int(ctx.info.kernels_per_batch),
        n_det_step=n_det_step, max_det_frame=int(frame_counts.max()), max_det=max_det, overflow=overflow, hit_rows=hit_rows,
        gather_records=gather_records, gather_overflow=gather_overflow,
        exchange=(None if world == 1 else "copy-engine puts into rank 0's memory over NVLink (cudaIpc) + stream wait/write-value flags, one merge kernel on rank 0; "
                  "NCCL for set-up and barriers" if env.exchange == "peer" else "NCCL gather per step + one merge kernel on rank 0"),
        e2e_fps=world * F * e2e_steps / t_e2e, e2e_steps=e2e_steps, e2e_dets=len(dets), e2e_two=len(e2e_ring) > 1,
        h2d_bytes=F * 4 * N_adc, N_adc=N_adc, last_dets=last_dets,
    )
    if world > 1:
        env.sync_all()                                      # no rank unmaps a peer's memory while another may still write to it
    for ln in lanes:
        if ln.gather is not None and hasattr(ln.gather, "close"):
            ln.gather.close()                               # before its context
        ln.ctx.close()
        ln.adc = None
    shared.clear()
    del adc, host, lanes
    torch.cuda.empty_cache()
    if overflow:
        raise SystemExit(f"bench.py: {name}: detection list overflow (most hits in one frame {res['max_det_frame']}, capacity {max_det}; "
                         f"exchange overflow {gather_overflow}): the timed work would be a truncated list — refusing to report it")
    return res


def compact_chain(res, world):
    """the short form of a chain measurement kept under other_workloads of the default line"""
    peak = peaks()[0]
    w = WORKLOADS[res["name"]]
    F, K, ms = res["F"], res["K"], res["ms"]
    return {
        "workload": chain_workload_text(res["name"]), "frames_per_gpu_per_step": F, "steps": K, "batches_in_flight": res["D"],
        "value": res["fps"], "unit": "frames/s", "ms_per_step": ms / K, "ms_per_step_one_in_flight": res["total_ms_one"],
        "stage_ms": dict(zip(STAGE_NAMES, res["stage_ms"])),
        "pipeline_frac_of_measured_hbm_peak": res["b_alg"] * F * K / (ms * 1e-3) / 1e9 / peak,
        "moved_frac_of_measured_hbm_peak": sum(res["stage_bytes"]) * K / (ms * 1e-3) / 1e9 / peak,
        "e2e": {"value": res["e2e_fps"], "unit": "frames/s", "h2d_bytes_per_step": res["h2d_bytes"],
                "d2h_bytes_per_step": 32 + 24 * res["e2e_dets"], "steps": res["e2e_steps"]},
        "detections_per_step": res["n_det_step"], "max_detections_in_one_frame": res["max_det_frame"],
        "max_det_per_frame": res["max_det"], "overflow": res["overflow"], "hit_rows_retransformed": res["hit_rows"] or None,
        "exchange_records_per_rank": res["gather_records"] if world > 1 else None,
        "exchange": res["exchange"],
        "detect_path": {0: "auto", 1: "per-cell", 2: "re-FFT of the hit rows (mmw_set_detect_path)"}[w.get("detect_path", 0)],
        "config_index": w["idx"],
    }


def run_chain(args, env):
    """cfg2 / cfg3 / cfg4: batches through the whole chain"""
    pkg, rank, world = env.pkg, env.rank, env.world
    w = WORKLOADS[args.workload]
    S, C, A, F, cfg_idx = w["S"], w["C"], w["A"], args.frames or w["F"], w["idx"]
    K, W = args.steps, args.warmup
    # `inflight` batches in flight: one context + stream + input batch per lane, steps go round-robin over the lanes, so the
    # tail of one batch's persistent FFT kernels and its latency-bound detection kernels fill with the next batch's work
    # (profiles/experiments: 1 -> 2 in flight is +10 % on cfg3).  Lane 0 is the one the per-stage numbers are taken from.
    D = max(1, args.inflight)
    sampler = ClockSampler(env.local_rank)
    if rank == 0:
        sampler.start()
    res = measure_chain(env, args.workload, F, K, W, D, keep_cube=args.keep_cube, keep_outputs=bool(args.dump_outputs))
    # the other BASELINE.json configs beside the headline shape, on the same box and the same N: configs[1] (cfg2),
    # configs[3] (cfg4, frame-sharded) and configs[4] (cfg5, sensors sharded) — shorter runs, same method
    others = {}
    if args.workload == "cfg3" and not args.no_other:
        for name in ("cfg2", "cfg4"):
            r = measure_chain(env, name, WORKLOADS[name]["F"], 6, 3, 2, share_input=True)
            others[name] = compact_chain(r, world)
        others["cfg5"] = compact_stream(measure_stream(env, "cfg5", WORKLOADS["cfg5"]["F"], 3, 3, depth=4, graph=True), world)
    clocks = sampler.stop() if rank == 0 else None      # sampled every 200 ms from the first timed region to the end of the last

    if rank == 0:
        stage_ms, stage_bytes, ms = res["stage_ms"], res["stage_bytes"], res["ms"]
        dom = int(np.argmax(stage_ms))
        peak, peak_src = peaks()
        achieved = stage_bytes[dom] / (stage_ms[dom] * 1e-3) / 1e9
        b_alg = res["b_alg"]
        traffic, traffic_src = (None, None)
        if F == w["F"] and not args.keep_cube:
            traffic, traffic_src = ncu_traffic(args.workload, STAGE_NAMES[dom])
        gather_bytes = 32 + 24 * res["gather_records"]
        line = {
            "metric": METRIC, "value": res["fps"], "unit": "frames/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": chain_workload_text(args.workload),
                "frames_per_gpu_per_step": F,
                "batches_in_flight": D,
                "ms_per_step_one_in_flight": res["total_ms_one"],
                "sharding": f"frame-sharded x{world}" + ("" if world == 1 else f"; per step a {gather_bytes}-byte result-block prefix per rank (sized from the warm-up batch) goes to rank 0 ({'copy-engine put over NVLink' if env.exchange == 'peer' else 'NCCL gather'}) + merge kernel on a side stream, overlapping the next step (overflow={res['gather_overflow']})"),
                "doppler_cube": "materialised" if args.keep_cube else "fused (not written to HBM)",
                "l2": f"inputs larger than L2: {F * 4 * res['N_adc'] / 1e6:.0f} MB int16 capture + {F * 8 * A * res['Sp'] * C / 1e6:.0f} MB intermediate per step vs 126 MB L2",
                "ms_per_step_by_rank": [m / K for m in res["ms_by_rank"]], "host_issue_ms_per_step_by_rank": [m / K for m in res["host_ms_by_rank"]],
                "host_issue_split_ms_per_step_rank0": {"process_device": res["host_split"][0] / K * 1e3, "exchange": res["host_split"][1] / K * 1e3},
                "rank0_numa_node": env.numa,
                "detections_per_step": res["n_det_step"], "max_detections_in_one_frame": res["max_det_frame"],
                "max_det_per_frame": res["max_det"], "overflow": res["overflow"], "hit_rows_retransformed": res["hit_rows"] or None,
                "detect_path": {0: "auto", 1: "per-cell", 2: "re-FFT of the hit rows (mmw_set_detect_path)"}[w.get("detect_path", 0)],
            },
            "roofline": {
                "bound": "hbm", "kernel": STAGE_NAMES[dom], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "note": "peak is the 1:1 copy figure of MEASURED_PEAKS.json; a bare data mover with this kernel's 1 : 2 read:write mix reaches "
                        "5.75 TB/s with contiguous stores and 5.2 TB/s with 128-byte corner-turned pieces like this kernel's at 512 points "
                        "(profiles/membench_r1.txt)",
                "algorithmic_bytes_per_launch": stage_bytes[dom], "kernel_ms": stage_ms[dom],
                "stage_ms": dict(zip(STAGE_NAMES, stage_ms)),
                "stage_gbs": {n: (b / (t * 1e-3) / 1e9 if t > 0 else None) for n, b, t in zip(STAGE_NAMES, stage_bytes, stage_ms)},
                "pipeline": {"algorithmic_bytes_per_frame": b_alg, "achieved": b_alg * F * K / (ms * 1e-3) / 1e9,
                             "frac": b_alg * F * K / (ms * 1e-3) / 1e9 / peak, "frac_of_8000_nominal": b_alg * F * K / (ms * 1e-3) / 1e9 / 8000.0,
                             "moved_bytes_per_frame": sum(stage_bytes) // F, "moved_frac": sum(stage_bytes) * K / (ms * 1e-3) / 1e9 / peak,
                             "note": "achieved/frac: 28N+8M bytes/frame (SURVEY.md 8d) x frames / step time, per GPU; moved_*: the bytes "
                                     "the kernels of this build actually read and write (fused mode skips the cube)"},
            },
            "e2e": {"value": res["e2e_fps"], "unit": "frames/s", "h2d_bytes_per_step": res["h2d_bytes"],
                    "d2h_bytes_per_step": 32 + 24 * res["e2e_dets"], "steps": res["e2e_steps"],
                    "api": "mmw_submit_host + mmw_wait, two batches in flight (one context each)" if res["e2e_two"] else "mmw_process_host"},
            "gpu_launches": K * (res["kernels_per_batch"] + (1 if world > 1 else 0)),      # + rank 0's merge kernel (NCCL's own kernel is not counted)
            "clocks": clocks,
        }
        if others:
            line["other_workloads"] = others
        if not args.no_cpu_baseline and world == 1:
            orc = entry.load_oracle()
            orc.build()
            cores = os.cpu_count() or 1
            port = CpuPort(orc, pkg, S, C, A, cfg_idx + 1, cores)
            passes = port.passes_for(12.0)                             # about 12 s of wall clock on the host cores
            n, dt, _ = port.run(passes)
            line["cpu_baseline"] = {"value": n / dt, "unit": "frames/s", "cores": port.cores, "kind": "port",
                                    "sample": f"{n} frames ({port.pool.shape[0]} distinct, {passes} passes) of the same workload in {dt:.1f} s; "
                                              f"plain-C fp64 oracle (the reference has no CPU code for these stages), {port.cores} OpenMP threads"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, detection_fields(res["last_dets"]))
        env.emit(line)


def measure_stream(env, name, sensors_total, K, W, depth=4, graph=True, keep_outputs=False):
    """cfg5: 64 sensors x (256 x 128 x 12) at 30 fps — latency mode.  Every frame is its own call (a sensor's frame is
    processed the moment it arrives); sensors are pinned to GPUs (sensor mod N).  A step = one tick = one frame from
    every sensor of this rank.  Collective: every rank must call it.
    keep_outputs: res["last_tick"] holds the detection lists of the last device-resident tick, with a sensor column."""
    torch, pkg, dev, rank, world = env.torch, env.pkg, env.dev, env.rank, env.world
    w = WORKLOADS[name]
    S, C, A, cfg_idx = w["S"], w["C"], w["A"], w["idx"]
    sensors = [x for x in range(sensors_total) if x % world == rank]
    F = len(sensors)
    ctx = pkg.RadarContext(S, C, A, F, max_det_per_frame=4096, device=env.local_rank)
    ctx.set_graph_mode(graph)
    adc = torch.stack([pkg.synth.cube_batch_torch(1, S, C, A, dev, cfg=cfg_idx + 1, first_frame=x)[0] for x in sensors])
    host = torch.empty((F, ctx.frame_shorts), dtype=torch.int16, pin_memory=True)
    host.copy_(adc)
    torch.cuda.synchronize()
    out = np.empty(ctx.max_det_per_frame, pkg.DET_DTYPE)
    frames = [host[i] for i in range(F)]
    dframes = [adc[i] for i in range(F)]
    tick_no = [0]

    def frame_index(i):
        # a running frame index per call, as a live stream has: graph mode patches it into the one captured graph
        return tick_no[0] * sensors_total + sensors[i]

    def tick_host(lat=None):
        n = 0
        for i in range(F):
            t0 = time.perf_counter()
            ctx.set_frame_offset(frame_index(i))
            dets, ov = ctx.process_host(frames[i], 1, out=out)
            if lat is not None:
                lat.append(time.perf_counter() - t0)
            n += len(dets)
            assert not ov
        tick_no[0] += 1
        return n

    # device-resident: one launch sequence (or graph replay) per frame, back to back, no host sync in between
    ctx.set_frame_offset(0)
    for _ in range(W):
        for i in range(F):
            ctx.process_device(dframes[i], 1)
    env.sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st = torch.cuda.ExternalStream(ctx.stream, device=dev)
    e0.record(st)
    for _ in range(K):
        for i in range(F):
            ctx.process_device(dframes[i], 1)
    e1.record(st)
    env.sync_all()
    ms = env.max_over_ranks(e0.elapsed_time(e1))
    last_tick = None
    if keep_outputs:
        # the device holds only the last call's list: the last tick is replayed untimed (same inputs, context and frame
        # offset) and read call by call; its last call must give back the list the timed loop left behind
        timed_last = ctx.read_detections()[0]
        lists = []
        for i in range(F):
            ctx.process_device(dframes[i], 1)
            lists.append(ctx.read_detections()[0])
        assert lists[-1].tobytes() == timed_last.tobytes(), "cfg5: the replayed tick differs from the timed one"
        last_tick = dict(detection_fields(np.concatenate(lists)), sensor=np.repeat(np.array(sensors), [len(d) for d in lists]))

    # host path: every frame H2D -> chain -> D2H, synchronous per frame; wall-clock latency per call
    for _ in range(W):
        tick_host()
    env.sync_all()
    lat = []
    t0 = time.perf_counter()
    n_det = 0
    for _ in range(K):
        n_det = tick_host(lat)
    t_sync = env.max_over_ranks(time.perf_counter() - t0)
    lat_us = np.sort(np.array(lat)) * 1e6
    # the same calls split in two (mmw_submit_host / mmw_wait) over a ring of contexts: `depth` frames in flight, the upload
    # of frame k+1 under the kernels and read-back of frame k
    depth = max(1, depth)
    ring = [pkg.RadarContext(S, C, A, 1, max_det_per_frame=4096, device=env.local_rank) for _ in range(depth)]
    for c in ring:
        c.set_graph_mode(graph)

    def tick_pipelined():
        n = 0
        for i in range(F + depth):
            c = ring[i % depth]
            if i >= depth:
                n += len(c.wait(out=out)[0])
            if i < F:
                c.set_frame_offset(frame_index(i))
                c.submit_host(frames[i], 1)
        tick_no[0] += 1
        return n

    for _ in range(W):
        tick_pipelined()
    env.sync_all()
    t0 = time.perf_counter()
    n_det_pipe = 0
    for _ in range(K):
        n_det_pipe = tick_pipelined()
    t_pipe = env.max_over_ranks(time.perf_counter() - t0)
    for c in ring:
        c.close()
    assert n_det_pipe == n_det, (n_det_pipe, n_det)
    # the same tick as one batch (all sensors' frames together)
    big = np.empty(F * ctx.max_det_per_frame, pkg.DET_DTYPE)
    ctx.set_frame_offset(0)
    for _ in range(2):
        ctx.process_host(host, F, out=big)
    t1 = time.perf_counter()
    for _ in range(max(3, K)):
        ctx.process_host(host, F, out=big)
    tick_batched_ms = (time.perf_counter() - t1) / max(3, K) * 1e3
    res = dict(
        name=name, S=S, C=C, A=A, cfg_idx=cfg_idx, sensors_total=sensors_total, F=F, K=K, W=W, depth=depth, graph=graph,
        fps=sensors_total * K / (ms * 1e-3), ms=ms, n_theta=ctx.n_theta, b_alg=int(ctx.info.algorithmic_bytes_per_frame),
        kernels_per_batch=int(ctx.info.kernels_per_batch), frame_shorts=ctx.frame_shorts,
        lat_p50=float(lat_us[len(lat_us) // 2]), lat_p99=float(lat_us[min(len(lat_us) - 1, int(0.99 * len(lat_us)))]),
        lat_max=float(lat_us[-1]), lat_n=int(len(lat_us)), tick_batched_ms=tick_batched_ms,
        sync_fps=sensors_total * K / t_sync, pipe_fps=sensors_total * K / t_pipe, t_pipe=t_pipe, n_det=n_det, last_tick=last_tick,
    )
    ctx.close()
    del adc, host
    torch.cuda.empty_cache()
    return res


def compact_stream(res, world):
    """the short form of the streaming measurement kept under other_workloads of the default line"""
    return {
        "workload": f"cfg5: {res['sensors_total']} sensors x ({res['S']} x {res['C']} x {res['A']}), one call per frame (latency mode) "
                    f"(BASELINE.json configs[{res['cfg_idx']}])",
        "sensors_per_gpu": res["F"], "sharding": f"sensor mod {world}", "cuda_graph": res["graph"], "steps": res["K"],
        "value": res["fps"], "unit": "frames/s", "required_frames_per_s": 30 * res["sensors_total"],
        "latency_us": {"p50": res["lat_p50"], "p99": res["lat_p99"], "max": res["lat_max"], "samples": res["lat_n"],
                       "what": "wall clock of one mmw_process_host(1 frame) call: pinned host -> H2D -> kernels -> D2H -> return"},
        "e2e": {"value": res["pipe_fps"], "unit": "frames/s", "h2d_bytes_per_step": res["F"] * res["frame_shorts"] * 2,
                "d2h_bytes_per_step": res["F"] * 32 + 24 * res["n_det"], "steps": res["K"],
                "api": f"mmw_submit_host + mmw_wait, 1 frame per call, {res['depth']} frames in flight (one context each)"},
        "realtime_margin_x": (1000.0 / 30.0) / (res["t_pipe"] / res["K"] * 1e3),
        "config_index": res["cfg_idx"],
    }


def run_stream(args, env):
    """cfg5 as its own bench line"""
    pkg, rank, world = env.pkg, env.rank, env.world
    w = WORKLOADS[args.workload]
    S, C, A, cfg_idx = w["S"], w["C"], w["A"], w["idx"]
    sensors_total = args.frames or w["F"]
    K, W = args.steps, args.warmup
    sampler = ClockSampler(env.local_rank)
    if rank == 0:
        sampler.start()
    res = measure_stream(env, args.workload, sensors_total, K, W, depth=args.depth, graph=not args.no_graph,
                         keep_outputs=bool(args.dump_outputs))
    clocks = sampler.stop() if rank == 0 else None
    F, ms = res["F"], res["ms"]
    if rank == 0:
        peak, peak_src = peaks()
        b_alg = res["b_alg"]
        line = {
            "metric": METRIC, "value": res["fps"], "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": f"cfg5: {sensors_total} sensors x ({S} x {C} x {A}), one call per frame (latency mode), 2-D CA-CFAR, "
                            f"{res['n_theta']}-pt angle FFT (BASELINE.json configs[{cfg_idx}])",
                "sensors_per_gpu": F, "sharding": f"sensor mod {world}", "cuda_graph": not args.no_graph,
                "required_frames_per_s": 30 * sensors_total,
                "latency_us": {"p50": res["lat_p50"], "p99": res["lat_p99"], "max": res["lat_max"], "samples": res["lat_n"],
                               "what": "wall clock of one mmw_process_host(1 frame) call: pinned host -> H2D -> kernels -> D2H -> return"},
                "tick_as_one_batch_ms": res["tick_batched_ms"], "realtime_margin_x": (1000.0 / 30.0) / (res["t_pipe"] / K * 1e3),
                "one_call_per_frame_synchronous_frames_per_s": res["sync_fps"],
                "frame_index": "advances with every call (graph mode patches it into the captured graph: no re-capture)",
                "l2": "latency mode: one 1.5 MB frame per call (fits L2 by construction; this workload is launch/PCIe-latency bound, not HBM bound)",
                "detections_last_tick": res["n_det"],
            },
            "roofline": {"bound": "hbm", "kernel": "whole chain (latency-bound)", "achieved": b_alg * sensors_total * K / (ms * 1e-3) / 1e9 / world,
                         "peak": peak, "unit": "GB/s", "frac": b_alg * sensors_total * K / (ms * 1e-3) / 1e9 / world / peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": b_alg,
                         "note": "SURVEY.md 8d: cfg5 is latency-bound; the figure to read is config.latency_us"},
            "e2e": {"value": res["pipe_fps"], "unit": "frames/s", "h2d_bytes_per_step": F * res["frame_shorts"] * 2,
                    "d2h_bytes_per_step": F * 32 + 24 * res["n_det"], "steps": K,
                    "api": f"mmw_submit_host + mmw_wait, 1 frame per call, {res['depth']} frames in flight (one context each)"},
            "gpu_launches": K * F * (res["kernels_per_batch"] + 1), "clocks": clocks,      # +1: power_sum_kernel of the antenna-split Doppler path
        }
        if not args.no_cpu_baseline and world == 1:
            orc = entry.load_oracle()
            orc.build()
            cores = os.cpu_count() or 1
            port = CpuPort(orc, pkg, S, C, A, cfg_idx + 1, cores)
            n, dt, _ = port.run(port.passes_for(12.0))
            line["cpu_baseline"] = {"value": n / dt, "unit": "frames/s", "cores": port.cores, "kind": "port",
                                    "sample": f"{n} frames in {dt:.1f} s, plain-C fp64 oracle, {port.cores} OpenMP threads (frame-parallel)"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, res["last_tick"])
        env.emit(line)


def run_legacy(args, env):
    """cfg1: the reference's own single-frame chain through the drop-in library"""
    torch, pkg, dev, rank, world = env.torch, env.pkg, env.dev, env.rank, env.world
    F = args.frames or WORKLOADS["cfg1"]["F"]
    K, W = args.steps, args.warmup
    orc = entry.load_oracle()
    orc.build()
    distinct = pkg.synth.legacy_capture(65, seed=rank)
    base = orc.reshape(distinct[0], 100, 128, 4)[:12800]
    reps = (F + 63) // 64
    cap = np.tile(distinct[1:], (reps, 1))[:F]                      # F frames = 819 MB at F = 4096: larger than L2
    frames = torch.from_numpy(cap).to(dev)
    raw = torch.empty(F, dtype=torch.int32, device=dev)
    L = pkg.api.load()
    for _ in range(W):
        pkg.api.legacy_process_device(frames, F, base, raw)
    pkg.api.legacy_sync()
    env.sync_all()
    sampler = ClockSampler(env.local_rank)
    if rank == 0:
        sampler.start()
    # device time: the library's own stream; wall clock around sync'd launches (kernel time >> launch latency at F = 4096)
    t0 = time.perf_counter()
    for _ in range(K):
        pkg.api.legacy_process_device(frames, F, base, raw)
    pkg.api.legacy_sync()
    ms = env.max_over_ranks((time.perf_counter() - t0) * 1e3)
    got = raw.cpu().numpy()
    want = np.array([orc.legacy_frame(distinct[1 + f], base)[1] for f in range(8)])
    assert np.array_equal(got[:8], want), "legacy raw bins differ from the reference CPU path"
    fps = world * F * K / (ms * 1e-3)
    # e2e (a): batched host entry point from pinned host memory; (b) the reference's calling pattern: one cudaProcessing per frame
    n_host = min(F, 1024)
    host_pinned = torch.from_numpy(cap[:n_host]).pin_memory()       # the contract's e2e: inputs in pinned host memory
    host = host_pinned.numpy()
    pkg.api.legacy_process_frames(host, base)
    t0 = time.perf_counter()
    e2e_steps = max(3, min(K, 10))
    for _ in range(e2e_steps):
        pkg.api.legacy_process_frames(host, base)
    t_e2e = env.max_over_ranks(time.perf_counter() - t0)
    pkg.api.legacy_configure(quiet=1)
    timers = np.zeros(4)
    pkg.cudaProcessing(distinct[1], base, timers=timers)
    t0 = time.perf_counter()
    n_drop = 256
    for f in range(n_drop):
        pkg.cudaProcessing(distinct[1 + f % 64], base, timers=timers)
    t_drop = time.perf_counter() - t0
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peak, peak_src = peaks()
        alg = 51200                                                   # rx0 of one frame: 128 chirps x 100 samples x 4 B
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms / K,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text("cfg1"), "frames_per_gpu_per_step": F,
                       "l2": f"inputs larger than L2: {F * 204800 / 1e6:.0f} MB of captures per step",
                       "dropin_cudaProcessing_frames_per_s": n_drop / t_drop,
                       "dropin_note": "the reference's own calling pattern: one synchronous cudaProcessing() per 200 KB frame (cudaBenchMarking.cpp:374-378)"},
            "roofline": {"bound": "hbm", "kernel": "legacy_frame_kernel", "achieved": alg * F * K / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg * F * K / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg * F,
                         "note": "one 16 384-point FFT per frame inside one SM's shared memory (batches; single-frame calls run on an 8-CTA cluster): shared-memory/issue bound, not HBM bound (only rx0, 1/4 of the capture, is read)"},
            "e2e": {"value": world * n_host * e2e_steps / t_e2e, "unit": "frames/s", "h2d_bytes_per_step": n_host * 51200,
                    "d2h_bytes_per_step": n_host * 4, "steps": e2e_steps,
                    "api": "mmw_legacy_process_frames (pinned host captures of 204 800 B per frame; one strided DMA uploads rx0's rows, "
                           "the 51 200 B per frame this chain reads)"},
            "gpu_launches": K, "clocks": clocks,
        }
        if not args.no_cpu_baseline and world == 1:
            port = LegacyCpu(orc, pkg)
            n, dt = port.run(port.passes_for(10.0))
            line["cpu_baseline"] = {"value": n / dt, "unit": "frames/s", "cores": 1, "kind": port.kind,
                                    "sample": f"{n} frames in {dt:.1f} s through the reference's cpuTiming() loop body "
                                              f"({'compiled from /root/reference into oracle/_ref' if port.kind == 'reference' else 'oracle restatement'}), single thread like the reference"}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"raw_bin": got})
        env.emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--frames", type=int, default=0, help="frames (cfg5: sensors) per GPU per step (default: workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl"],
                    help="N > 1: how the detection lists reach rank 0: copy-engine puts into rank 0's memory over NVLink + stream memory "
                         "operations (mmw_exchange_*; NCCL carries the set-up only), or an NCCL gather per step")
    ap.add_argument("--no-other", action="store_true", help="cfg3: skip the side measurements of cfg2 / cfg4 / cfg5 (configs[1], [3], [4])")
    ap.add_argument("--inflight", type=int, default=3, help="cfg2/cfg3/cfg4: batches in flight (contexts on their own streams, steps round-robin)")
    ap.add_argument("--depth", type=int, default=4, help="cfg5: one-frame calls in flight on the end-to-end path (ring of contexts, mmw_submit_host / mmw_wait)")
    ap.add_argument("--no-graph", action="store_true", help="cfg5: launch the kernels one by one instead of replaying a CUDA graph")
    ap.add_argument("--keep-cube", action="store_true", help="materialise the Doppler cube in HBM (default: fused)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (the detection list field by field; cfg1: the arg-max bins) "
                                                             "as DIR/<name>.npy, at most 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")))
        return
    env = Env()
    env.exchange = args.exchange
    {"chain": run_chain, "stream": run_stream, "legacy": run_legacy}[WORKLOADS[args.workload]["kind"]](args, env)
    env.finish()


if __name__ == "__main__":
    main()
