"""Device time of the differentiable ops (odam_b200/autograd.py) beside one fused optimiser step, with CUDA events.

    python tools/time_autograd.py [--configs 2,3,5]

Per config (synthetic.make_config: 2 = 50 x 50 views, 3 = 2000 x 30, 5 = 50k x 20; the prior as the config says) it
times, per call:
  points fwd        surface_points(params)                      (sampler + 1000 points per object)
  points fwd+bwd    surface_points, then backward of a fixed upstream gradient
  sides fwd         box_sides(params, view_off, Ms)
  sides fwd+bwd     box_sides, then backward of a fixed upstream gradient of pred (the two kernels alone)
  loss fwd+bwd      box_loss(...).sum().backward()               (box_sides and its VJP + the torch ops of the loss)
  fused 1 step      api.optimize_device(n_iters=1)               (the fused optimiser: sampler, sides, gradient, Adam)
Every shape is warmed up first; each figure is the median over 5 timed windows of at least 100 ms.  The working sets
of configs 2 and 3 fit in L2 and are read from there after the first pass.  The card's name and power limit are printed
in the same run."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from odam_b200 import api, synthetic  # noqa: E402
from odam_b200 import autograd as AG  # noqa: E402


def per_call_ms(fn, min_window_ms=100.0, windows=5):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(3, int(np.ceil(min_window_ms / max(e0.elapsed_time(e1), 1e-3))))
    out = []
    for _ in range(windows):
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / reps)
    return float(np.median(out)), reps


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        lim = r.stdout.strip() or r.stderr.strip()
    except OSError as e:
        lim = f"nvidia-smi unavailable ({e})"
    return f"{name}; power limit, max SM clock: {lim}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="2,3,5")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_autograd.py needs a CUDA device")
    print(card())
    prior_np = api.prior_table()
    for idx in (int(c) for c in args.configs.split(",")):
        cfg = synthetic.CONFIGS[idx]
        tracks = api.pack_scene(synthetic.make_config(idx))
        use_prior = cfg["prior"]
        dt = api.DeviceTracks(tracks, "cuda:0", prior_np if use_prior else None)
        params = dt.init.clone().requires_grad_(True)
        voff, Ms, box, mask = dt.view_off, dt.Ms, dt.box, dt.mask
        kw = dict(prior=dt.prior, cls=dt.cls, s0=dt.init[:, 4:7].clone()) if use_prior else {}
        G = torch.randn((tracks.n, 1000, 3), device="cuda", generator=torch.Generator("cuda").manual_seed(0))
        Gs = torch.randn((tracks.total_views, 4), device="cuda", generator=torch.Generator("cuda").manual_seed(1))

        def points_fwd():
            with torch.no_grad():
                AG.surface_points(params)

        def points_fwd_bwd():
            params.grad = None
            torch.autograd.backward(AG.surface_points(params), G)

        def sides_fwd():
            with torch.no_grad():
                AG.box_sides(params, voff, Ms)

        def sides_fwd_bwd():
            params.grad = None
            torch.autograd.backward(AG.box_sides(params, voff, Ms)[0], Gs)

        def loss_fwd_bwd():
            params.grad = None
            AG.box_loss(params, voff, Ms, box, mask, **kw).sum().backward()

        def fused():
            api.optimize_device(dt, n_iters=1)

        print(f"config {idx}: {cfg['name']} ({tracks.n} objects, {tracks.total_views} views, prior {use_prior})")
        for name, fn in (("points fwd", points_fwd), ("points fwd+bwd", points_fwd_bwd), ("sides fwd", sides_fwd),
                         ("sides fwd+bwd", sides_fwd_bwd), ("loss fwd+bwd", loss_fwd_bwd), ("fused 1 step", fused)):
            ms, reps = per_call_ms(fn)
            print(f"  {name:15s} {ms * 1e3:10.1f} us/call  ({reps} calls per window)")
        del dt, params, G
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
