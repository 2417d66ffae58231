"""Device cost of the clustering kernels (mmw_set_clustering) on the bench workloads: stage times through mmw_time_device
(CUDA events between launches; stage 4 = detection records + the clustering kernels when on), clustering off and on in
alternation on the same input, several repeats each.  cfg2 / cfg3 / cfg4: one batch of the bench's shape and scene per call;
cfg5: one-frame calls (latency mode).  Default clustering parameters.
--kernels adds, in a separate pass, the device time of each clustering kernel from torch.profiler (CUDA activities).
Run on the GPU box:  python profiles/cluster_cost.py [cfg3 cfg2 cfg4 cfg5] [--repeats R] [--iters I] [--kernels]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
# (S, C, A, frames per call, bench scene index, per-frame detection capacity, detect path) as bench.py runs them
WORKLOADS = {"cfg2": (256, 128, 4, 1024, 2, 4096, 2), "cfg3": (512, 256, 12, 64, 3, 4096, 0),
             "cfg4": (1024, 512, 192, 4, 4, 32768, 0), "cfg5": (256, 128, 12, 1, 5, 1024, 0)}
ON = dict(min_points=1)          # any keyword turns clustering on; the rest stays at mmw_default_cluster_params


def arg(name, default):
    return int(sys.argv[sys.argv.index(name) + 1]) if name in sys.argv else default


def main():
    repeats, iters = arg("--repeats", 5), arg("--iters", 20)
    names = [a for a in sys.argv[1:] if a in WORKLOADS] or ["cfg2", "cfg3", "cfg4", "cfg5"]
    dev = torch.device("cuda", 0)
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    print(f"GPU: {torch.cuda.get_device_name(0)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}", flush=True)
    print(f"method: mmw_time_device per_stage, {iters} batches per sample, {repeats} samples per setting, off/on alternating", flush=True)
    for wl in names:
        S, C, A, F, scene, max_det, path = WORKLOADS[wl]
        adc = pkg.synth.cube_batch_torch(F, S, C, A, dev, cfg=scene)
        with pkg.RadarContext(S, C, A, F, max_det_per_frame=max_det) as ctx:
            if path:
                ctx.set_detect_path(path)
            ctx.set_clustering(**ON)
            dets, _ = ctx.process_host(adc.cpu().numpy(), F)
            objs, _ = ctx.read_objects()
            k_on = ctx.info.kernels_per_batch
            ctx.set_clustering()
            k_off = ctx.info.kernels_per_batch
            samples = {"off": [], "on": []}
            for rep in range(repeats):
                for mode in ("off", "on"):
                    ctx.set_clustering(**(ON if mode == "on" else {}))
                    ctx.time_device(adc, F, 3)                       # warm-up of this setting
                    tot, st = ctx.time_device(adc, F, iters, per_stage=True)
                    samples[mode].append([tot / iters] + [s / iters for s in st])
            off, on = np.array(samples["off"]), np.array(samples["on"])
            d_stage4 = on[:, 4] - off[:, 4]
            print(f"{wl} {S}x{C}x{A} F={F}: {dets.size} detections, {objs.size} objects per call; kernels {k_off} -> {k_on}", flush=True)
            for mode, a in (("off", off), ("on", on)):
                med = np.median(a, axis=0)
                print(f"  clustering {mode:3s}: total {med[0]:.4f} ms (min {a[:, 0].min():.4f} max {a[:, 0].max():.4f}) | "
                      f"range {med[1]:.4f} doppler {med[2]:.4f} cfar {med[3]:.4f} stage4 {med[4]:.4f} "
                      f"(min {a[:, 4].min():.4f} max {a[:, 4].max():.4f})", flush=True)
            detect_only = np.median(off[:, 4])
            cost = np.median(d_stage4)
            print(f"  clustering cost: {cost:.4f} ms per call (stage-4 difference, median of {repeats}; spread "
                  f"{d_stage4.min():.4f}..{d_stage4.max():.4f}) vs detection stage {detect_only:.4f} ms: "
                  f"{'below' if cost < detect_only else 'NOT below'} it ({cost / detect_only:.2f}x)", flush=True)
            if "--kernels" in sys.argv:
                kernel_times(ctx, adc, F, iters)
        del adc
        torch.cuda.empty_cache()


def kernel_times(ctx, adc, F, iters):
    from torch.profiler import ProfilerActivity, profile

    ctx.set_clustering(**ON)
    ctx.time_device(adc, F, 3)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.time_device(adc, F, iters)
        torch.cuda.synchronize()
    rows = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and "kernel" in ev.name:
            name = ev.name.split("(")[0].split("<")[0].replace("void ", "").replace("mmw::", "")
            t = getattr(ev, "device_time", None)
            t = ev.cuda_time if t is None else t
            rows.setdefault(name, []).append(t)
    for name, ts in sorted(rows.items(), key=lambda kv: -sum(kv[1])):
        print(f"    {name:32s} {np.mean(ts):8.2f} us x {len(ts) // iters}", flush=True)


if __name__ == "__main__":
    main()
