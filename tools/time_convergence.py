"""Device time and fit quality of the fused optimiser's early stopping (odam_sq_optimize_converge) and step reduction
on a plateau (odam_sq_optimize_plateau) against the default entry, with CUDA events.

    python tools/time_convergence.py [--configs 2,3,4,5] [--out profiles/plateau_timing.txt]

Per config (synthetic.make_config, its own iteration count and prior) every variant is launched device-resident
(api.optimize_device, launch options fixed from the host copy of view_off):
  default     every object runs all iterations (the default build)
  never       the convergence build with patience 0: it never stops, so this is the cost of the build itself
  stop        patience 20, rel_tol 1e-3
  stop+best   the same, returning each object's lowest-loss iterate (keep_best)
  stop10      patience 10, rel_tol 1e-3: the stop rule at the patience of the step-reduction variants
  p10 f.3 R2  patience 10, rel_tol 1e-3; on a plateau the step shrinks by 0.3, twice, before the object stops
  (+best)     the same with keep_best
  p10 f.5 R3  factor 0.5, three reductions
  p20 f.3 R1  patience 20 (that of `stop`), one reduction by 0.3
Every setting tried is reported.  Every shape is warmed up first.  The variants alternate window by window in one
process; each figure is the median over 7 windows of at least 100 ms.  Per variant the report gives the mean and
largest iterations run, the mean reductions taken, the median over objects of the ratio of the object's lowest loss
to its lowest loss in the default run, and the median centre error (m) and relative dimension error against the
scene's ground truth.  The card's name and power limit are printed in the same run."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from odam_b200 import api, synthetic  # noqa: E402
from tools.time_autograd import card  # noqa: E402
from tools.time_objective import window_ms  # noqa: E402

VARIANTS = {"default": {}, "never": dict(patience=0, rel_tol=1e-3), "stop": dict(patience=20, rel_tol=1e-3),
            "stop+best": dict(patience=20, rel_tol=1e-3, keep_best=True), "stop10": dict(patience=10, rel_tol=1e-3),
            "p10 f.3 R2": dict(patience=10, rel_tol=1e-3, max_reductions=2, lr_factor=0.3),
            "(+best)": dict(patience=10, rel_tol=1e-3, max_reductions=2, lr_factor=0.3, keep_best=True),
            "p10 f.5 R3": dict(patience=10, rel_tol=1e-3, max_reductions=3, lr_factor=0.5),
            "p20 f.3 R1": dict(patience=20, rel_tol=1e-3, max_reductions=1, lr_factor=0.3)}


def errors(params, gt):
    """(median centre error in m, median relative dimension error) of [n, 9] parameters."""
    p = params.astype(np.float64)
    centre = np.linalg.norm(p[:, :3] - gt["centre"], axis=1)
    dims = np.abs(2 * p[:, 4:7] ** 2 - gt["dims"]) / gt["dims"]
    return float(np.median(centre)), float(np.median(dims))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="2,3,4,5")
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_convergence.py needs a CUDA device")
    lines = [card()]
    print(lines[-1], flush=True)
    prior = api.prior_table()
    for idx in (int(c) for c in args.configs.split(",")):
        cfg = synthetic.CONFIGS[idx]
        scene = synthetic.make_config(idx)
        tracks = api.pack_scene(scene)
        dt = api.DeviceTracks(tracks, "cuda:0", prior if cfg["prior"] else None)
        q = api.query_launch(tracks.view_off)
        fixed = dict(threads=q["threads"], max_slices=q["max_slices"], cluster=q["cluster"], code_layout=q["code_layout"])
        n_iters = cfg["n_iters"]
        outs = {}

        def launcher(name):
            def fn():
                outs[name] = api.optimize_device(dt, n_iters=n_iters, out=outs.get(name), **VARIANTS[name], **fixed)
            return fn

        fns = {name: launcher(name) for name in VARIANTS}
        for _ in range(2):
            for fn in fns.values():
                fn()
        torch.cuda.synchronize()
        reps = max(1, int(np.ceil(100.0 / window_ms(fns["default"], 1))))
        times = {name: [] for name in VARIANTS}
        for _ in range(args.windows):
            for name, fn in fns.items():
                times[name].append(window_ms(fn, reps))
        med = {k: float(np.median(v)) for k, v in times.items()}
        lines.append(f"config {idx}: {cfg['name']}, {n_iters} iterations ({tracks.n} objects, {tracks.total_views} views, "
                     f"{q['threads']} threads, cluster {q['cluster']}, layout {q['code_layout']}; {reps} launches per "
                     f"window)")
        lowest = lambda o: np.nanmin(o["loss"].cpu().numpy().astype(np.float64), axis=1)   # every first loss is run
        low0 = lowest(outs["default"])
        for k, v in times.items():
            o = outs[k]
            iters = o["iters"].cpu().numpy() if "iters" in o else np.full(tracks.n, n_iters)
            red = o["reductions"].cpu().numpy().mean() if "reductions" in o else 0.0
            ce, de = errors(o["params"].cpu().numpy(), scene.gt)
            lines[-1] += (f"\n  {k:10s} {med[k]:9.3f} ms/launch (window spread {(max(v) - min(v)) / med[k] * 100:.1f} %)"
                          f"  speed-up {med['default'] / med[k]:.3f}  iterations mean {iters.mean():6.1f} max "
                          f"{iters.max():3d}  reductions mean {red:4.2f}  lowest loss / default's, median "
                          f"{np.nanmedian(lowest(o) / low0):.4f}  median error centre {ce * 1000:.1f} mm, dims "
                          f"{100 * de:.2f} %")
        print(lines[-1], flush=True)
        del dt, outs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
