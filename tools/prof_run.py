"""Time a few device-resident launches of the fused optimiser on a named config (CUDA events), and with --cycles
print the mean SM cycles per iteration of each kernel phase.

    python tools/prof_run.py --config 5 --objects 4736 --iters 20 [--threads T] [--layout L] [--cycles]

ODAM_SQ_LIB times another build of the library (tools/ab_run.sh).
"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from odam_b200 import api, synthetic  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--config", type=int, default=2)
ap.add_argument("--objects", type=int, default=None)
ap.add_argument("--iters", type=int, default=None)
ap.add_argument("--views", type=int, default=None)
ap.add_argument("--threads", type=int, default=0)
ap.add_argument("--max-slices", type=int, default=0)
ap.add_argument("--launches", type=int, default=2)
ap.add_argument("--cycles", action="store_true")
ap.add_argument("--cluster", type=int, default=0)
ap.add_argument("--layout", type=int, default=0, help="odam_sq_options.code_layout: 0 auto, 1 straight-line, 2 compact")
a = ap.parse_args()
c = synthetic.CONFIGS[a.config]
scene = synthetic.make_scene(a.objects or c["n_objects"], a.views or c["n_views"], seed=a.config, device="cuda:0")
tracks = api.pack_scene(scene)
dt = api.DeviceTracks(tracks, "cuda:0", api.prior_table() if c["prior"] else None)
iters = a.iters or c["n_iters"]
out = None
ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.launches + 1)]
ev[0].record()
for k in range(a.launches):
    out = api.optimize_device(dt, n_iters=iters, threads=a.threads, max_slices=a.max_slices, out=out, cluster=a.cluster, code_layout=a.layout)
    ev[k + 1].record()
torch.cuda.synchronize()
units = float(tracks.total_views) * iters
for k in range(a.launches):
    ms = ev[k].elapsed_time(ev[k + 1])
    print(f"launch {k}: {ms:.3f} ms  {units / ms / 1e3:.1f} M unit/s  "
          f"{api.algorithmic_flops(tracks.view_off[1:] - tracks.view_off[:-1], iters) / ms / 1e9:.2f} TFLOP/s")
print("flagged", int((out["status"].cpu() & 3 != 0).sum()))
if a.cycles:
    cyc = torch.zeros((tracks.n, 16), dtype=torch.int64, device="cuda:0")
    api.optimize_device(dt, n_iters=iters, threads=a.threads, max_slices=a.max_slices, out=out, cycles=cyc, cluster=a.cluster, code_layout=a.layout)
    torch.cuda.synchronize()
    c = cyc.cpu().numpy().astype(float) / iters
    names = ["F: combine slices", "B fix-up walk (eta)", "D points", "E project", "F: butterfly + barrier", "F: resolve arg + exact re-evaluation", "G: end-of-iteration barrier", "C cdf",
             "B0 eta (powers, ratios, placement)", "F: loss term + gradient", "wait for omega warps", "rebuilds (count)",
             "G: cross-warp sum + cluster exchange", "G: barrier", "G: gradient, Adam, derive (warp 0)", "-"]
    print("mean SM cycles per iteration per object (thread 0's view):")
    tot = np.delete(c, 11, axis=1).sum(1).mean()
    for k in [8, 1, 7, 10, 2, 3, 0, 5, 9, 4, 12, 13, 14, 6]:
        print(f"  {names[k]:40s} {c[:, k].mean():9.0f}  ({c[:, k].mean() / tot:5.1%})")
    print(f"  {'total':40s} {tot:9.0f}     tree rebuilds per object: {c[:, 11].mean() * iters:.1f}")
