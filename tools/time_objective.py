"""Device time of the fused optimiser's objective build (odam_sq_optimize_objective: per-side weights and a robust
residual loss) against the default build, with CUDA events.

    python tools/time_objective.py [--configs 2,3,4,5] [--out profiles/objective_timing.txt]

Per config (synthetic.make_config, its own iteration count and prior) every variant is launched device-resident
(api.optimize_device, launch options fixed from the host copy of view_off):
  default     the reference's masked L1 (the default build)
  weights     L1 with random weights in [0.1, 2), a fifth of them 0, read from a CUDA tensor (objective build)
  cauchy      Cauchy (c = 8 px) without weights (objective build)
  objective   Cauchy with the weights
weights and cauchy split the objective build's cost between the weight loads and the loss arithmetic.  Every shape is
warmed up first.  The variants alternate window by window in one process; each figure is the median over 7 windows of
at least 100 ms.  The card's name and power limit are printed in the same run."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from odam_b200 import api, synthetic  # noqa: E402
from tools.time_autograd import card  # noqa: E402


def window_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="2,3,4,5")
    ap.add_argument("--windows", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_objective.py needs a CUDA device")
    lines = [card()]
    print(lines[-1], flush=True)
    prior = api.prior_table()
    for idx in (int(c) for c in args.configs.split(",")):
        cfg = synthetic.CONFIGS[idx]
        tracks = api.pack_scene(synthetic.make_config(idx))
        dt = api.DeviceTracks(tracks, "cuda:0", prior if cfg["prior"] else None)
        rng = np.random.default_rng(idx)
        w = rng.uniform(0.1, 2.0, (tracks.total_views, 4)).astype(np.float32)
        w[rng.uniform(size=w.shape) < 0.2] = 0
        wt = torch.from_numpy(w).cuda()
        q = api.query_launch(tracks.view_off)
        fixed = dict(threads=q["threads"], max_slices=q["max_slices"], cluster=q["cluster"], code_layout=q["code_layout"])
        n_iters = cfg["n_iters"]
        variants = {"default": {}, "weights": dict(side_weight=wt),
                    "cauchy": dict(loss="cauchy", loss_scale=8.0),
                    "objective": dict(side_weight=wt, loss="cauchy", loss_scale=8.0)}
        outs = {}

        def launcher(name):
            def fn():
                outs[name] = api.optimize_device(dt, n_iters=n_iters, out=outs.get(name), **variants[name], **fixed)
            return fn

        fns = {name: launcher(name) for name in variants}
        for _ in range(2):
            for fn in fns.values():
                fn()
        torch.cuda.synchronize()
        reps = max(1, int(np.ceil(100.0 / window_ms(fns["default"], 1))))
        times = {name: [] for name in variants}
        for _ in range(args.windows):
            for name, fn in fns.items():
                times[name].append(window_ms(fn, reps))
        med = {k: float(np.median(v)) for k, v in times.items()}
        lines.append(f"config {idx}: {cfg['name']}, {n_iters} iterations ({tracks.n} objects, {tracks.total_views} views, "
                     f"{q['threads']} threads, cluster {q['cluster']}, layout {q['code_layout']}; {reps} launches per "
                     f"window)")
        for k, v in times.items():
            lines[-1] += (f"\n  {k:9s} {med[k]:9.3f} ms/launch (window spread {(max(v) - min(v)) / med[k] * 100:.1f} %)"
                          f"  ratio {med[k] / med['default']:.4f}")
        print(lines[-1], flush=True)
        del dt, wt, outs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
