#!/usr/bin/env python
"""bench.py -- object-iterations/sec of the fused superquadric optimiser on B200 (see DESIGN.md, 'Measurement').

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config 2] [--impl native|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A "step" is ONE pass of the hot path over one batch: every object of the workload optimised for the
config's full iteration count (200) in one persistent kernel launch.  Unit of work = one
(object x view x iteration) with 1000 surface samples (BASELINE.md).

value   device-resident throughput: inputs already in HBM, CUDA events around each step on the launching
        stream (torch's current stream; the library launches on the stream it is given), max over ranks.
e2e     the same metric through the public host-buffer API (odam_b200.api.optimize_host -> C ABI
        odam_sq_optimize_host): pinned staging, H2D of every input, kernel, D2H of parameters + per-iteration
        loss + status, all inside the timed region (wall clock around the synchronous call).
roofline  FP32: algorithmic flops (SURVEY 8d: iters*(37,000*V+30,000) per object) / kernel time, against the
        FFMA peak measured live by the library's micro-benchmark (nominal 148*128*2*1.965 GHz = 74.4 TFLOP/s is
        printed beside it); the HBM figure is reported too, to show the path is nowhere near memory-bound.
cpu_baseline / --impl reference   the reference's optimiser loop (oracle/torch_oracle.py, an op-for-op port
        pinned bit-for-bit to the reference; with oracle/_ref's compiled reference sampler when present) on the
        host cores, on a bounded sample of the same workload.
sfu     roofline.sfu: one MUFU.RCP per point-view (1000 per unit) against 148 SMs x 16 SFU lanes x clock.
e2e_call_site   the reference-facing entry point itself: 82-column tracks -> odam_b200.run_multi_view.optim_process ->
        result dict (staging, H2D, kernel, D2H, oriented boxes on the device, result objects), host buffers throughout.
--dump-outputs DIR   what the last timed step returned (native: params, loss, status of rank 0, plus the all-gathered
        params with several GPUs; reference: params and loss of its sample) as DIR/<name>.npy.  Inputs are seeded, so
        two builds run with the same arguments can be compared output for output.
Multi-GPU: the headline stays weak scaling -- every rank optimises its own scene of the named shape (objects are
independent, no data-path collective) and the final parameters are all-gathered over NCCL inside the timed step -- and
`strong` carries what north_star names: ONE batch (BASELINE configs 3 and 5) sharded by object across the N ranks
(contiguous blocks balanced by views, odam_b200.sharding), each rank's block in one launch, one all-gather of [n, 9].
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

METRIC = "object-iterations/sec (objects x views x iters)"
UNIT = "obj*view*iter/s"
SM_COUNT, NOMINAL_CLOCK_GHZ = 148, 1.965


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "MEASURED_PEAKS.json (of measured)"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "B200_PROFILING.md fallback (of fallback)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe).

    An `nvidia-smi -lms` child needs ~100 ms to deliver its first sample -- longer than a short timed region -- so it is
    launched when the bench starts and its time-stamped samples are cut to the window [begin(), stop()] afterwards.
    (Polling NVML from a thread of this process was tried and rejected: it slowed the 2-GPU step by 14 %.)"""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, period_ms=10):
        self.path = os.path.join(tempfile.gettempdir(), f"odam_clocks_{os.getpid()}.csv")
        self.gpu, self.period, self.proc, self.t0 = gpu_index, period_ms, None, None

    def launch(self):
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", str(self.period)], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def start(self):   # the timed region begins
        import datetime
        self.t0 = datetime.datetime.now()

    def stop(self):
        import datetime
        t1 = datetime.datetime.now()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0,
               "source": f"nvidia-smi -lms {self.period}, samples inside the timed window"}
        if self.proc is None:
            return out
        time.sleep(2.5 * self.period / 1e3)   # let the last sample of the window reach the file
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.f.close()
        rows = []
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                rows.append((datetime.datetime.strptime(c[0], "%Y/%m/%d %H:%M:%S.%f"), float(c[1]), float(c[2]), c[5:9]))
            except ValueError:
                continue
        os.unlink(self.path)
        lo = (self.t0 or t1) - datetime.timedelta(milliseconds=self.period)
        inside = [r for r in rows if lo <= r[0] <= t1 + datetime.timedelta(milliseconds=2 * self.period)]
        if not inside and rows:   # clock skew or a very short window: fall back to the samples nearest to it
            inside, out["source"] = rows[-3:], out["source"] + " (none inside: last samples before the stop)"
        reasons = set()
        for r in inside:
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if inside:
            out.update(sm_mhz=float(np.median([r[1] for r in inside])), sm_max_mhz=inside[-1][2],
                       reasons=sorted(reasons), samples=len(inside))
        return out


def workload(cfg_idx, rank, n_objects=None, device="cpu"):
    from odam_b200 import api, synthetic
    c = synthetic.CONFIGS[cfg_idx]
    n = n_objects or c["n_objects"]
    # rank 0 is exactly the named config (seed = config index, SURVEY 8d); other ranks draw their own scenes
    scene = synthetic.make_scene(n, c["n_views"], seed=cfg_idx + 1000 * rank, device=device)
    tracks = api.pack_scene(scene)
    prior = api.prior_table() if c["prior"] else None
    return c, scene, tracks, prior


# ------------------------------------------------------------------------------------------------------
def cpu_port_worker(job):
    """One object of the reference loop on one core (module-level so that multiprocessing can pickle it).
    Returns (seconds, final parameters [9], loss of every iteration)."""
    import torch
    torch.set_num_threads(job["threads"])
    from oracle import torch_oracle
    t0 = time.perf_counter()
    r = torch_oracle.run(job["translate"], job["angle"], job["dims"], job["Ms"], job["box"], job["mask"], job["prior33"],
                         n_iters=job["iters"], representation="super_quadric", anomaly=True, record=False)
    return time.perf_counter() - t0, r["final"], r["loss"]


def cpu_jobs(scene, tracks, prior, objs, iters, threads):
    V = scene.V
    jobs = []
    for i in objs:
        jobs.append(dict(translate=scene.translate[i], angle=scene.angle[i], dims=scene.dims[i], Ms=scene.P_cws[i],
                         box=tracks.box[i * V:(i + 1) * V], mask=tracks.mask[i * V:(i + 1) * V],
                         prior33=None if prior is None else prior[tracks.cls[i]].reshape(3, 3), iters=iters,
                         threads=threads))
    return jobs


def map_reference_sampler():
    """dlopen oracle/_ref in THIS process too: the workers that use it are short-lived, and the driver records which
    native libraries the bench process itself has mapped."""
    import ctypes
    from oracle import c_oracle
    if c_oracle.have_ref_sampler():
        return ctypes.CDLL(c_oracle.ref_sampler_path())
    return None


def cpu_baseline_config1(budget_s=40.0, threads=None, max_objects=None):
    """SURVEY 8d / BASELINE configs[0]: 1 scene, 10 objects x 20 views, 200 iterations, prior on, as shipped (anomaly
    mode on, sequential objects, torch's default intra-op threads -- or `threads`).  Runs the whole config (about half
    a minute) unless the budget or `max_objects` ends it first; whole objects only."""
    import torch
    from odam_b200 import api, synthetic
    from oracle import c_oracle
    c_oracle.build()
    map_reference_sampler()
    c = synthetic.CONFIGS[1]
    scene = synthetic.make_scene(c["n_objects"], c["n_views"], seed=1)
    tracks = api.pack_scene(scene)
    prior = api.prior_table()
    default_threads = torch.get_num_threads()
    threads = threads or default_threads
    done, t_total = 0, 0.0
    for i in range(scene.n if max_objects is None else min(scene.n, max_objects)):
        t_total += cpu_port_worker(cpu_jobs(scene, tracks, prior, [i], c["n_iters"], threads)[0])[0]
        done += 1
        if t_total > budget_s:
            break
    torch.set_num_threads(default_threads)
    units = done * scene.V * c["n_iters"]
    return {"value": units / t_total, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"config 1 ({c['name']}, {c['n_iters']} iterations, prior on): {done} of {scene.n} objects, all "
                      f"{c['n_iters']} iterations, sequential objects as run_multi_view.py:44-69, torch intra-op "
                      f"threads={threads}, anomaly mode on (as shipped), sampler="
                      f"{'oracle/_ref (reference C++)' if c_oracle.have_ref_sampler() else 'oracle C restatement'}",
            "seconds": t_total}


def cpu_baseline_sequential(scene, tracks, prior, budget_s=15.0):
    """As the reference runs it (run_multi_view.py:44-69): objects one after another in one process, torch's
    default intra-op threads, anomaly mode on as shipped.  Bounded sample: whole objects at a reduced iteration
    count until ~budget_s of CPU work is spent."""
    import torch
    from oracle import c_oracle
    c_oracle.build()
    map_reference_sampler()
    threads = torch.get_num_threads()
    iters, done, t_total = 40, 0, 0.0
    for i in range(min(scene.n, 64)):
        t_total += cpu_port_worker(cpu_jobs(scene, tracks, prior, [i], iters, threads)[0])[0]
        done += 1
        if t_total > budget_s:
            break
    units = done * scene.V * iters
    return {"value": units / t_total, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{done} objects x {scene.V} views x {iters} iterations of the workload, sequential objects, "
                      f"torch intra-op threads={threads}, anomaly mode on (as shipped), sampler="
                      f"{'oracle/_ref (reference C++)' if c_oracle.have_ref_sampler() else 'oracle C restatement'}",
            "seconds": t_total}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on all host cores (one object per
    process, as many processes as cores -- objects are independent), bounded sample per step."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    import multiprocessing as mp
    from oracle import c_oracle
    c_oracle.build()
    map_reference_sampler()
    cfg, scene, tracks, prior = workload(args.config, 0, args.objects)
    cores = len(os.sched_getaffinity(0))
    n_obj = min(scene.n, cores)
    iters = args.ref_iters
    jobs = cpu_jobs(scene, tracks, prior, list(range(n_obj)), iters, 1)
    units = n_obj * scene.V * iters
    times = []
    with mp.get_context("spawn").Pool(min(cores, n_obj)) as pool:
        for k in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            res = pool.map(cpu_port_worker, jobs, chunksize=1)
            dt = time.perf_counter() - t0
            if k >= args.warmup:
                times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"params": np.stack([r[1] for r in res]), "loss": np.stack([r[2] for r in res])})
    ms = 1e3 * float(np.mean(times))
    value = units / (ms / 1e3)
    sample = (f"{n_obj} objects x {scene.V} views x {iters} iterations per step (of {scene.n} x {scene.V} x "
              f"{cfg['n_iters']}), one object per process on {min(cores, n_obj)} processes, torch threads=1 each, "
              f"anomaly mode on (as shipped), sampler="
              f"{'oracle/_ref (reference C++)' if c_oracle.have_ref_sampler() else 'oracle C restatement'}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config {args.config}: {cfg['name']}, {cfg['n_iters']} iterations, "
                                   f"prior={'on' if cfg['prior'] else 'off'}", "objects": scene.n, "views": scene.V,
                       "iters": cfg["n_iters"], "bounded_sample": sample},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": min(cores, n_obj), "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------------------
def time_config(api, torch, dt, n_iters, steps, warmup, flush, dist=None, gath=None, sampler=None):
    """K device-resident steps with CUDA events on torch's current stream (= the launching stream).
    Returns (per-step ms list for the whole step, per-step ms list for the kernel alone)."""
    out = api.optimize_device(dt, n_iters=n_iters)
    for _ in range(max(0, warmup - 1)):
        api.optimize_device(dt, n_iters=n_iters, out=out)
        if dist is not None:
            dist.all_gather_into_tensor(gath, out["params"])
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    if sampler is not None:
        sampler.start()   # clocks are sampled from here on: the timed steps (and the e2e steps that follow)
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    for k in range(steps):
        flush.zero_()  # L2 flush between timed iterations (256 MiB > 126 MB L2), outside the event pair
        ev[k][0].record()
        api.optimize_device(dt, n_iters=n_iters, out=out)
        ev[k][1].record()
        if dist is not None:
            dist.all_gather_into_tensor(gath, out["params"])
        ev[k][2].record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    return [e[0].elapsed_time(e[2]) for e in ev], [e[0].elapsed_time(e[1]) for e in ev], out


def run_native(args):
    import torch
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(dev))
    from odam_b200 import _lib, api
    _lib.check(_lib.load().odam_sq_init(local_rank))
    clocks = ClockSampler(local_rank)
    if rank == 0 and args.clocks != "off":
        clocks.launch()   # running by the time the timed region starts; cut to that window afterwards

    cfg, scene, tracks, prior = workload(args.config, rank, args.objects, device=dev)
    n_iters = cfg["n_iters"]
    views = np.diff(tracks.view_off)
    units_rank = float(views.sum()) * n_iters
    dt = api.DeviceTracks(tracks, dev, prior)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gath = torch.empty((world * tracks.n, 9), dtype=torch.float32, device=dev) if world > 1 else None

    step_ms, kern_ms, out = time_config(api, torch, dt, n_iters, args.steps, args.warmup, flush, dist, gath,
                                        clocks if rank == 0 and args.clocks != "off" else None)
    tot = torch.tensor([sum(step_ms), sum(kern_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
    total_ms, kernel_ms = float(tot[0]), float(tot[1])
    ms_per_step = total_ms / args.steps
    value = world * units_rank / (ms_per_step / 1e3)
    status = out["status"].cpu().numpy()
    # host copies now: the multi-GPU e2e steps below reuse `out` and `gath`
    last_step = None
    if args.dump_outputs and rank == 0:
        last_step = {k: v.cpu().numpy() for k, v in out.items()}
        if world > 1:
            last_step["params_all_ranks"] = gath.cpu().numpy()

    # ---- e2e through the host-buffer API (H2D + kernel + D2H inside the timed region) ----
    e2e_steps = max(3, min(args.steps, 10))
    api.optimize_host(tracks, prior=prior, n_iters=n_iters, device=local_rank)  # warm-up (workspace allocation)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if world == 1:
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            api.optimize_host(tracks, prior=prior, n_iters=n_iters, device=local_rank)
        e2e_path = "odam_b200.api.optimize_host -> odam_sq_optimize_host (pinned staging inside the library)"
    else:
        # N GPUs: the same bytes cross the bus, but the step stays on the stream -- H2D of every input from pinned host
        # memory, one launch, the all-gather of the final parameters on the device, D2H of the gathered parameters and
        # of this rank's loss log into pinned memory, ONE synchronisation per step
        pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        host_in = {k: pin(getattr(tracks, k)) for k in ("init", "cls", "view_off", "Ms", "box", "mask")}
        if prior is not None:
            host_in["prior"] = pin(prior)
        dev_in = {k: torch.empty_like(v, device=dev) for k, v in host_in.items()}
        host_out = {"gath": torch.empty((world * tracks.n, 9), dtype=torch.float32).pin_memory(),
                    "loss": torch.empty((tracks.n, n_iters), dtype=torch.float32).pin_memory(),
                    "status": torch.empty((tracks.n,), dtype=torch.int32).pin_memory()}
        dte = api.DeviceTracks(tracks, dev, prior)

        def e2e_step():
            for k, v in host_in.items():
                dev_in[k].copy_(v, non_blocking=True)
            dte.init, dte.cls, dte.view_off, dte.Ms, dte.box, dte.mask = (dev_in[k] for k in ("init", "cls", "view_off", "Ms", "box", "mask"))
            if prior is not None:
                dte.prior = dev_in["prior"]
            api.optimize_device(dte, n_iters=n_iters, out=out)
            dist.all_gather_into_tensor(gath, out["params"])
            host_out["gath"].copy_(gath, non_blocking=True)
            host_out["loss"].copy_(out["loss"], non_blocking=True)
            host_out["status"].copy_(out["status"], non_blocking=True)
            torch.cuda.synchronize()
        e2e_step()
        dist.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        e2e_path = ("pinned host buffers -> H2D -> odam_b200.api.optimize_device (odam_sq_optimize) -> NCCL all-gather on the "
                    "device -> D2H of gathered parameters + loss log + status, one synchronisation per step")
    e2e_ms = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    clk = clocks.stop() if rank == 0 else None   # sampled across the device-timed AND the e2e timed regions
    SV, n = tracks.total_views, tracks.n
    h2d = n * 36 + n * 4 + (n + 1) * 4 + SV * (48 + 16 + 4) + (288 if prior is not None else 0) + n_iters * 16
    d2h = (world if world > 1 else 1) * n * 36 + n * n_iters * 4 + n * 4
    e2e_value = world * units_rank / (float(e2e_ms[0]) / 1e3)

    # ---- strong scaling: ONE batch sharded by object across the ranks (BASELINE configs 3 and 5) ----
    strong = []
    if not args.no_strong:
        for ci in args.strong:
            strong.append(strong_scaling(api, torch, dist, ci, rank, world, dev, flush))

    # ---- the reference-facing call site (tracks -> optim_process -> result dict), rank 0 ----
    call_site = None
    if rank == 0 and not args.no_call_site:
        call_site = time_call_site(scene, cfg, local_rank)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (only) kernel ----
    peaks, peak_src = measured_peaks()
    fma_peak = api.fma_peak_tflops(local_rank)
    flops = api.algorithmic_flops(views, n_iters)
    kern_s = kernel_ms / args.steps / 1e3
    achieved = flops / kern_s / 1e12
    algo_bytes = float(SV * 68 + n * (36 + 36 + 4 * n_iters + 4))
    roofline = {"bound": "fp32", "achieved": achieved, "peak": fma_peak, "unit": "TFLOP/s", "frac": achieved / fma_peak,
                "traffic": None,
                "peak_source": "FFMA-chain micro-benchmark run by this process (odam_sq_fma_peak); nominal "
                               f"{SM_COUNT}*128*2*{NOMINAL_CLOCK_GHZ} GHz = {SM_COUNT * 128 * 2 * NOMINAL_CLOCK_GHZ / 1e3:.1f} TFLOP/s",
                "frac_of_nominal": achieved / (SM_COUNT * 128 * 2 * NOMINAL_CLOCK_GHZ / 1e3),
                "algorithmic_flops_per_launch": flops, "kernel_ms": kern_s * 1e3,
                "hbm": {"achieved_gbs": algo_bytes / kern_s / 1e9, "peak_gbs": peaks["hbm_gbs"],
                        "frac": algo_bytes / kern_s / 1e9 / peaks["hbm_gbs"], "algorithmic_bytes": algo_bytes,
                        "peak_source": peak_src}}
    sfu_peak = SM_COUNT * 16 * (clk["sm_mhz"] * 1e6 if clk and clk.get("sm_mhz") else NOMINAL_CLOCK_GHZ * 1e9)
    sfu_ops = float(views.sum()) * n_iters * 1000.0 + tracks.n * n_iters * 12000.0   # SURVEY 8d: 1 rcp per point-view, 12 per point
    roofline["sfu"] = {"achieved_tops": sfu_ops / kern_s / 1e12, "peak_tops": sfu_peak / 1e12,
                       "frac": sfu_ops / kern_s / sfu_peak,
                       "note": "algorithmic SFU-class ops of the reference formulation (SURVEY 8d: 1000 per unit + 12000 per "
                               "object-iteration; the kernel evaluates the per-point transcendentals once per grid node instead) "
                               "against 148 SMs x 16 SFU lanes x the SM clock sampled during the run"}
    traffic_file = os.path.join(REPO, "profiles", "traffic.json")
    if os.path.exists(traffic_file):
        with open(traffic_file) as f:
            roofline["traffic"] = json.load(f).get(f"config{args.config}")
        roofline["traffic_source"] = ("profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set "
                                      "full` capture of this config (not re-measured by this run)")

    # ---- other BASELINE configs at 1 GPU (short runs; the headline stays the named config) ----
    sweep = []
    if world == 1 and not args.no_sweep:
        for ci in args.sweep:
            if ci == args.config:
                continue
            c2, _, tr2, pr2 = workload(ci, 0, None, device=dev)
            dt2 = api.DeviceTracks(tr2, dev, pr2)
            est = float(np.diff(tr2.view_off).sum()) * c2["n_iters"] / 6e8          # seconds per step, roughly
            sw_steps = 10 if est < 0.1 else 3                                         # >= 10 timed steps unless a step is long
            s_ms, k_ms, o2 = time_config(api, torch, dt2, c2["n_iters"], sw_steps, 3, flush)
            v2 = np.diff(tr2.view_off)
            ks = sum(k_ms) / len(k_ms) / 1e3
            ach = api.algorithmic_flops(v2, c2["n_iters"]) / ks / 1e12
            sweep.append({"config": ci, "workload": c2["name"], "value": float(v2.sum()) * c2["n_iters"] / ks,
                          "ms_per_step": ks * 1e3, "steps": sw_steps, "fp32_tflops": ach, "roofline_frac": ach / fma_peak,
                          "roofline_frac_of_nominal": ach / (SM_COUNT * 128 * 2 * NOMINAL_CLOCK_GHZ / 1e3),
                          "bad_status": int((o2["status"].cpu().numpy() & 3 != 0).sum())})
            del dt2

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"config {args.config}: {cfg['name']}, {n_iters} iterations, "
                                   f"prior={'on' if cfg['prior'] else 'off'} (per GPU; weak scaling)",
                       "objects_per_gpu": tracks.n, "views": int(views.max()), "iters": n_iters, "samples": 1000,
                       "l2": "256 MiB memset between timed steps (inputs are < L2)",
                       "launch": dict(zip(("threads", "smem_bytes", "ctas_per_sm", "ctas_per_object", "code_layout"), launch_info(api, tracks)))},
            "clocks": clk, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                                   "d2h_bytes_per_step": int(d2h), "ms_per_step": float(e2e_ms[0]), "steps": e2e_steps},
            "gpu_launches": args.steps, "roofline": roofline,
            "objects_flagged": int((status & 3 != 0).sum()), "sweep": sweep, "strong": strong,
            "e2e_call_site": call_site}
    line["e2e"]["path"] = e2e_path
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline_config1(args.cpu_budget * 2.5)
        line["cpu_baseline_headline_config"] = cpu_baseline_sequential(scene, tracks, prior, args.cpu_budget)
        line["cpu_baseline_1thread"] = cpu_baseline_config1(args.cpu_budget, threads=1, max_objects=3)   # SURVEY 8d: 1 thread too
    if last_step is not None:
        dump_outputs(args.dump_outputs, last_step)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def strong_scaling(api, torch, dist, cfg_idx, rank, world, dev, flush):
    """ONE batch of BASELINE config `cfg_idx`, identical on every rank (seed = config index), sharded by object:
    contiguous blocks balanced by views -> this rank's block in one persistent launch -> one NCCL all-gather of the
    final [n, 9] parameters on the same stream.  Timed with CUDA events on that stream, max over ranks; enough steps
    for >= ~150 ms of timed work."""
    from odam_b200 import sharding, synthetic
    c = synthetic.CONFIGS[cfg_idx]
    scene = synthetic.make_scene(c["n_objects"], c["n_views"], seed=cfg_idx, device=dev)
    tracks = api.pack_scene(scene)
    prior = api.prior_table() if c["prior"] else None
    n_iters = c["n_iters"]
    parts = sharding.partition_by_views(tracks.view_off, world)
    lo, hi = parts[rank]
    dt = api.DeviceTracks(tracks.slice(lo, hi), dev, prior)
    counts = [h - l for l, h in parts]
    pad = max(counts)
    out = api.optimize_device(dt, n_iters=n_iters)
    buf = torch.zeros((pad, 9), dtype=torch.float32, device=dev)
    gath = torch.empty((world * pad, 9), dtype=torch.float32, device=dev) if world > 1 else None

    def step():
        api.optimize_device(dt, n_iters=n_iters, out=out)
        if world > 1:
            buf[: hi - lo].copy_(out["params"])
            dist.all_gather_into_tensor(gath, buf)
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    units = float(tracks.total_views) * n_iters
    est_ms = units / (6e8 * world) * 1e3
    steps = int(min(50, max(3, np.ceil(150.0 / est_ms))))
    if world > 1:
        dist.barrier()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)]
    for k in range(steps):
        flush.zero_()
        ev[k][0].record()
        step()
        ev[k][1].record()
    torch.cuda.synchronize()
    tot = torch.tensor([sum(e[0].elapsed_time(e[1]) for e in ev)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        dist.barrier()
    ms = float(tot[0]) / steps
    status = out["status"].cpu().numpy()
    res = {"config": cfg_idx, "workload": f"{c['name']}, {n_iters} iterations, ONE batch sharded by object across {world} GPU(s)",
           "n_gpus": world, "value": units / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "warmup": 3,
           "objects_per_rank": counts, "scaling": "strong", "all_gather_bytes": int(world * pad * 36) if world > 1 else 0,
           "fp32_tflops": api.algorithmic_flops(np.diff(tracks.view_off), n_iters) / (ms / 1e3) / 1e12,
           "bad_status_rank0": int((status & 3 != 0).sum())}
    del dt, out, buf, gath
    return res


def time_call_site(scene, cfg, device):
    """tracks -> odam_b200.run_multi_view.optim_process -> result dict, the call OdamProcess.optim_process makes
    (src/processor.py:352-368): 82-column host tracks in, SuperQuadric objects + oriented boxes out."""
    from odam_b200 import synthetic
    from odam_b200.run_multi_view import optim_process
    seq = synthetic.scene_to_tracks(scene)
    T_wcs, P_cws = list(seq["T_wcs"]), list(seq["P_cws"])
    args = (seq["tracks"], seq["img_names"], T_wcs, P_cws, seq["img_h"], seq["img_w"], seq["K"], "super_quadric",
            bool(cfg["prior"]), cfg["n_iters"], 10)
    out = optim_process(*args, device=device)
    ts = []
    for _ in range(5):
        t0 = time.perf_counter()
        out = optim_process(*args, device=device)
        ts.append(time.perf_counter() - t0)
    ms = 1e3 * float(np.median(ts))
    units = float(scene.n * scene.V * cfg["n_iters"])
    return {"value": units / (ms / 1e3), "unit": UNIT, "ms_per_call": ms, "calls": 5, "objects": scene.n, "views": scene.V,
            "entry": "odam_b200.run_multi_view.optim_process(tracks, img_names, T_wcs, P_cws, h, w, K, 'super_quadric', "
                     "prior, n_iters, n_views): vectorised staging, H2D, one optimiser launch + one oriented-box launch "
                     "behind it in the same C-ABI call, D2H, result objects",
            "returned": sorted(out)}


def launch_info(api, tracks):
    q = api.query_launch(tracks.view_off)
    return q["threads"], q["smem_bytes"], q["ctas_per_sm"], q["cluster"], q["code_layout"]


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries print there too (NCCL's version banner, for one), so fd 1
    is pointed at stderr for the duration of the run and the JSON line is written to the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: each array as path/<name>.npy, floats as float32/float64 and integers (status flags, indices) as
    float64, so that two builds can be compared output for output.  Beyond DUMP_LIMIT_BYTES in all, every array keeps
    the same share of its rows, drawn with a fixed seed, and the kept row indices go to path/<name>_rows.npy."""
    arrays = {k: np.asarray(v) for k, v in arrays.items()}
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float32 if v.dtype.kind == "f" else np.float64)
              for k, v in arrays.items()}
    total = sum(v.nbytes for v in arrays.values())
    # when sampling, the kept row indices (8 bytes a row) count too, and 1 MiB is left for the .npy headers
    scale = (DUMP_LIMIT_BYTES - (1 << 20)) / sum(v.nbytes + 8 * (len(v) if v.ndim else 0) for v in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES and a.ndim and len(a) > 1:
            keep = max(1, int(len(a) * scale))
            rows = np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))
            a = a[rows]
            np.save(os.path.join(path, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(path, f"{name}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json configs index (1-based); 2 = headline")
    ap.add_argument("--objects", type=int, default=None, help="override the object count (debugging)")
    ap.add_argument("--sweep", type=int, nargs="*", default=[3, 4, 5])
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--strong", type=int, nargs="*", default=[3, 5], help="configs for the sharded (strong-scaling) measurement")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--no-call-site", action="store_true")
    ap.add_argument("--clocks", default="smi", choices=["smi", "off"], help="clock sampler (off: diagnostics only)")
    ap.add_argument("--cpu-budget", type=float, default=15.0)
    ap.add_argument("--ref-iters", type=int, default=20)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
    claim_stdout()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
