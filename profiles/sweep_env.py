"""Stage times of a bench workload under different values of one environment switch read at mmw_create
(MMW_SCHED: how the persistent FFT kernels take their tiles).
    python profiles/sweep_env.py cfg3 MMW_SCHED=0,1,3"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
SHAPES = {"cfg3": (512, 256, 12, 64), "cfg2": (256, 128, 4, 1024), "cfg4": (1024, 512, 192, 4), "cfg5": (256, 128, 12, 64)}
dev = torch.device("cuda", 0)
wls = [a for a in sys.argv[1:] if "=" not in a] or ["cfg3"]
name, vals = [a for a in sys.argv[1:] if "=" in a][0].split("=")
for wl in wls:
    S, C, A, F = SHAPES[wl]
    adc = pkg.synth.cube_batch_torch(F, S, C, A, dev, cfg=3)
    for v in vals.split(","):
        os.environ[name] = v
        with pkg.RadarContext(S, C, A, F, max_det_per_frame=4096) as ctx:
            ctx.time_device(adc, F, 3)
            tot, st = ctx.time_device(adc, F, 20, per_stage=True)
            print(f"{wl} {name}={v}: total {tot / 20:.4f} ms | range {st[0] / 20:.4f} doppler {st[1] / 20:.4f} cfar {st[2] / 20:.4f} detect {st[3] / 20:.4f}", flush=True)
    del adc
