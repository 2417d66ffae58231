"""Does the Doppler kernel run faster when its input (the range spectrum K1 has just written) is still in L2?
Per-stage device times for small batches of the cfg3 shape, where the whole intermediate fits in the 126 MB L2,
against the bench batch (64 frames, 805 MB intermediate).  Run on the GPU box: python profiles/l2_probe.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
S, C, A = 512, 256, 12
dev = torch.device("cuda", 0)
for F in (2, 4, 6, 8, 16, 64):
    adc = pkg.synth.cube_batch_torch(F, S, C, A, dev, cfg=3)
    with pkg.RadarContext(S, C, A, F) as ctx:
        ctx.time_device(adc, F, 3)
        tot, st = ctx.time_device(adc, F, 50, per_stage=True)
        n = 50
        print(f"F={F:3d} rs={F * 12.58:.0f} MB: range {st[0] / n / F * 1e3:.2f} us/frame, doppler {st[1] / n / F * 1e3:.2f} us/frame, "
              f"cfar {st[2] / n * 1e3:.1f} us, detect {st[3] / n * 1e3:.1f} us, batch {tot / n * 1e3:.1f} us", flush=True)
    del adc
