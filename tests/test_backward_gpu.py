"""GPU tests of the fused kernel's backward pass (phase F) and Adam update (phase G) on their own.

The parity tests compare parameters after Adam steps, and Adam normalises the gradient by its running magnitude, so a
gradient off by a few per cent passes them.  Here every launch also returns the last iteration's gradient, Adam
moments, grids, eta buckets, arg-extreme samples and predicted sides, and:
  - the gradient is held to TAU_KERNEL * scale of a float64 restatement of the same step under the kernel's own
    discrete decisions (oracle/grad64.py; scale = sum of |d term / d p_k| over the live terms and the prior);
  - those decisions are checked for legitimacy: each predicted side is the float64 projection of its arg point and
    the float64 extremum over all valid points, to the get_bbox tolerance;
  - on the reference's recorded states the gradient and moments are compared with the reference's own;
  - Adam is recomputed in float64 from the kernel's own gradient for many schedules;
  - the per-stream cache of Adam bias-correction tables is exercised with interleaved and concurrent schedules.
"""
import time

import numpy as np
import pytest

from golden_cases import EDGE_KINDS, all_cases, edge_object, wide_cases
from launch_checks import EXTRAS, TAU_KERNEL, check_launch, pack
from oracle import grad64 as G64

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntests/test_backward_gpu.py wall time {time.time() - t0:.1f} s")


def _ragged_tracks(api):
    """The batch of test_ragged_tracks_edge_cases: 1, 3, 11, 20, 64, 300 views, a view behind the camera, a track with
    every side masked."""
    from odam_b200 import synthetic
    from odam_b200.api import init_params
    Vs = [1, 3, 11, 20, 64, 300, 20, 20]
    scene = synthetic.make_scene(len(Vs), 300, seed=5)
    objs = []
    for i, V in enumerate(Vs):
        M = scene.P_cws[i][:V].reshape(V, 12).astype(np.float32)
        m = scene.mask[i][:V].copy()
        if i == 6:
            M[0, 8:12] = -M[0, 8:12]
        if i == 7:
            m[:] = 0
        objs.append((init_params(scene.translate[i], scene.angle[i], scene.dims[i]), M, scene.box[i][:V], m, scene.cls[i]))
    return pack(objs)


@pytest.mark.parametrize("n_iters", [1, 5])
def test_gradient_ragged_batch_every_cta_size(api, n_iters):
    """Ragged batch at every CTA size and both code layouts (the compact one exists up to 256 threads)."""
    tracks, prior = _ragged_tracks(api), api.prior_table()
    for threads in (64, 128, 256, 512, 1024):
        for layout in ((1, 2) if threads <= 256 else (1,)):
            check_launch(api, tracks, prior, n_iters, label=f"ragged threads={threads} layout={layout} iters={n_iters}",
                          threads=threads, code_layout=layout)


def test_gradient_view_tiled_clusters(api):
    """1-4 CTAs per object (partial gradients exchanged through DSMEM), views [50, 37, 3, 2, 64]."""
    from odam_b200 import synthetic
    from odam_b200.api import init_params
    Vs = [50, 37, 3, 2, 64]
    sc = synthetic.make_scene(len(Vs), 64, seed=13)
    tracks = pack([(init_params(sc.translate[i], sc.angle[i], sc.dims[i]), sc.P_cws[i][:V].reshape(V, 12),
                     sc.box[i][:V], sc.mask[i][:V], sc.cls[i]) for i, V in enumerate(Vs)])
    for c in (1, 2, 3, 4):
        check_launch(api, tracks, api.prior_table(), 4, label=f"cluster={c}", cluster=c)


def test_gradient_long_tracks(api):
    """1500 and 2500 views (several views per thread), automatic cluster and a single CTA."""
    from odam_b200 import synthetic
    for V in (1500, 2500):
        tracks = api.pack_scene(synthetic.make_scene(2, V, seed=21))
        for cluster in (0, 1):
            check_launch(api, tracks, api.prior_table(), 2, label=f"V={V} cluster={cluster}", cluster=cluster)


@pytest.mark.parametrize("representation", ["cube", "quadric", "super_quadric"])
def test_gradient_edge_objects(api, representation):
    """Extreme exponents (h = +-6), yaws on the axes, a view behind the camera, an all-masked track, a single view;
    with and without the prior; every representation (frozen shapes report a zero shape gradient)."""
    objs = []
    for kind in EDGE_KINDS:
        init, Ms, box, mask, cls = edge_object(kind)
        if representation == "cube":
            init[7:9] = -10000.0
        elif representation == "quadric":
            init[7:9] = 0.0
        objs.append((init, Ms, box, mask, cls))
    tracks = pack(objs)
    for prior in (api.prior_table(), None):
        for n_iters in (1, 3):
            check_launch(api, tracks, prior, n_iters, representation,
                          label=f"edge objects {representation} prior={prior is not None} iters={n_iters}")


def test_gradient_after_200_free_iterations(api):
    """Config 2 (50 objects x 50 views), 200 free-running iterations: shapes have drifted far from the start; the last
    iteration's gradient of every object against float64."""
    from odam_b200 import synthetic
    tracks = api.pack_scene(synthetic.make_config(2))
    check_launch(api, tracks, api.prior_table(), 200, label="config 2, iteration 200")


def test_gradient_and_moments_vs_reference_records(api, golden_runs, golden_wide):
    """Every recorded reference state, one teacher-forced kernel step: on the steps whose discrete decisions agree
    with the reference's, the kernel's gradient and Adam moments against the reference's recorded grad, m and v.
    m = 0.9 m0 + 0.1 g and v = 0.999 v0 + 0.001 g^2 inherit the gradient's bound."""
    tau = 2 * TAU_KERNEL
    ulp = lambda x: np.spacing(np.abs(x).astype(np.float32)).astype(np.float64)
    steps = agree = 0
    worst = np.zeros(9)
    for case in all_cases(golden_runs) + wide_cases(golden_wide):
        P, M, V = case.states_before()
        live = case.mask.astype(bool)
        opt = case.repr == "super_quadric"
        nc = 9 if opt else 7
        for s in range(case.iters):
            tracks = case.tracks(P[s:s + 1])
            o = api.optimize_host(tracks, prior=case.prior_table, n_iters=1, representation=case.repr, m0=M[s:s + 1],
                                  v0=V[s:s + 1], step0=s, s0=case.init[None, 4:7], extras=EXTRAS)
            steps += 1
            arg, pred = o["out_arg"].reshape(case.V, 4), o["out_pred"].reshape(case.V, 4)
            same = (np.array_equal(case.arg[s][live], arg[live]) and np.array_equal(case.eta_idx[s], o["out_eta_idx"][0])
                    and np.array_equal(case.resid_sign[s][live], np.sign(pred - case.box)[live]))
            if not same:
                continue
            agree += 1
            etas, omegas = G64.angles(o["out_grids"][0], o["out_eta_idx"][0])
            g64, sc = G64.grad64(P[s], case.Ms, case.box, case.mask, etas, omegas, arg, np.sign(pred - case.box),
                                 case.prior33, case.init[4:7], opt)
            g, m, v = o["out_grad"][0].astype(np.float64), o["out_m"][0].astype(np.float64), o["out_v"][0].astype(np.float64)
            rg, rm, rv = case.grad[s].astype(np.float64), case.m[s].astype(np.float64), case.v[s].astype(np.float64)
            r = G64.ratio(g[:nc], rg[:nc], sc[:nc])
            label = (getattr(case, "name", case.k), s)
            assert (r <= tau).all(), (label, r)
            bm = 0.1 * tau * sc + 4 * ulp(rm)
            bv = 0.001 * 2 * np.abs(rg) * tau * sc + 4 * ulp(rv)
            assert (np.abs(m - rm)[:nc] <= bm[:nc]).all(), (label, m, rm)
            assert (np.abs(v - rv)[:nc] <= bv[:nc]).all(), (label, v, rv)
            if not opt:   # frozen shapes: the moments pass through
                assert np.array_equal(o["out_m"][0][7:9], M[s][7:9]) and np.array_equal(o["out_v"][0][7:9], V[s][7:9])
            worst[:nc] = np.maximum(worst[:nc], r)
    print(f"reference records: {steps} teacher-forced steps, {agree} with the reference's decisions; worst "
          f"|g - g_ref| / scale " + " ".join(f"{x:.1e}" for x in worst))
    assert agree >= 0.95 * steps


@pytest.mark.parametrize("representation", ["cube", "quadric", "super_quadric"])
def test_adam_step_in_isolation(api, representation):
    """From random Adam state, one step at step0 in {0, 1, 7, 199, 1e4, 1e6}, lr in {0.01, 0.003, 0.05, 0} and
    lr_shape in {0.1, 0.02}: m and v within 4 ulp of the float64 update of the kernel's own gradient (ulp of the
    largest of the value, the old value and the new contribution), the new parameters within 4 ulp of the float64 update
    plus 1 ulp of the parameter.  lr = 0 leaves the parameters bit-identical; frozen shapes come back bit-identical with
    a zero shape gradient and their moments passed through."""
    from odam_b200 import synthetic
    rng = np.random.default_rng(7)
    tracks = api.pack_scene(synthetic.make_scene(6, 12, seed=17), representation)
    n = tracks.n
    m0 = (rng.normal(0, 1, (n, 9)) * 10.0 ** rng.uniform(-4, 1, (n, 9))).astype(np.float32)
    v0 = (10.0 ** rng.uniform(-8, 2, (n, 9))).astype(np.float32)
    s0 = tracks.init[:, 4:7] * np.float32(1.1)
    opt = representation == "super_quadric"
    ulp = lambda x: np.spacing(np.abs(x).astype(np.float32)).astype(np.float64)
    for step0 in (0, 1, 7, 199, 10 ** 4, 10 ** 6):
        for lr in (0.01, 0.003, 0.05, 0.0):
            for lr_shape in (0.1, 0.02):
                o = api.optimize_host(tracks, prior=api.prior_table(), n_iters=1, representation=representation,
                                      lr=lr, lr_shape=lr_shape, m0=m0, v0=v0, step0=step0, s0=s0, extras=EXTRAS)
                label = (representation, step0, lr, lr_shape)
                g = o["out_grad"].astype(np.float64)
                M0, V0, P0 = m0.astype(np.float64), v0.astype(np.float64), tracks.init.astype(np.float64)
                m64 = M0 + 0.1 * (g - M0)
                v64 = 0.999 * V0 + 0.001 * g * g
                m, v = o["out_m"].astype(np.float64), o["out_v"].astype(np.float64)
                step = step0 + 1
                bc1, bc2 = 1 - 0.9 ** step, 1 - 0.999 ** step
                rate = np.where(np.arange(9) < 7, lr, lr_shape)
                upd = -rate / bc1 * m / (np.sqrt(v) / np.sqrt(bc2) + 1e-8)
                k = slice(0, 9 if opt else 7)
                assert (np.abs(m - m64)[:, k] <= 4 * ulp(np.maximum.reduce([np.abs(m64), np.abs(M0), 0.1 * np.abs(g)]))[:, k]).all(), label
                assert (np.abs(v - v64)[:, k] <= 4 * ulp(np.maximum.reduce([v64, V0, 0.001 * g * g]))[:, k]).all(), label
                p = o["params"].astype(np.float64)
                assert (np.abs(p - (P0 + upd))[:, k] <= (4 * ulp(upd) + ulp(P0 + upd))[:, k]).all(), (label, p - P0 - upd)
                if lr == 0:
                    assert np.array_equal(o["params"][:, :7], tracks.init[:, :7]), label
                if not opt:
                    assert np.array_equal(o["params"][:, 7:9], tracks.init[:, 7:9]), label
                    assert (o["out_grad"][:, 7:9] == 0).all(), label
                    assert np.array_equal(o["out_m"][:, 7:9], m0[:, 7:9]) and np.array_equal(o["out_v"][:, 7:9], v0[:, 7:9])


def test_adam_table_cache_schedules(api):
    """Launches with different (lr, lr_shape, step0, n_iters) interleaved A B A C B A through the host entry equal the
    same calls made alone; device-entry launches of different schedules on one stream and then on 20 streams at once
    (more than the 16 cached tables, so entries are recycled while others are in flight) each equal the host-entry
    result of their own schedule after one synchronise."""
    import torch
    from odam_b200 import synthetic
    tracks = api.pack_scene(synthetic.make_scene(8, 16, seed=23))
    prior = api.prior_table()
    sched = {"A": dict(lr=0.01, lr_shape=0.1, n_iters=12), "B": dict(lr=0.05, lr_shape=0.02, n_iters=7),
             "C": dict(lr=0.003, lr_shape=0.1, n_iters=12)}
    steps = {"A": 0, "B": 5, "C": 199}
    host = lambda k: api.optimize_host(tracks, prior=prior, step0=steps[k], **sched[k])
    alone = {k: host(k) for k in sched}
    for k in "ABACBA":
        o = host(k)
        assert np.array_equal(o["params"], alone[k]["params"]) and np.array_equal(o["loss"], alone[k]["loss"]), k
    # the device entry has no step0: its schedules differ in lr, lr_shape and n_iters
    dsched = [dict(lr=0.01 * (1 + j % 5), lr_shape=0.1 / (1 + j % 3), n_iters=5 + j % 7) for j in range(20)]
    ref = [api.optimize_host(tracks, prior=prior, **s) for s in dsched]
    dt = api.DeviceTracks(tracks, "cuda:0", prior)
    torch.cuda.synchronize()
    outs = [api.optimize_device(dt, **dsched[j]) for j in (0, 1, 0, 2, 1, 0)]
    torch.cuda.synchronize()
    for j, d in zip((0, 1, 0, 2, 1, 0), outs):
        assert np.array_equal(d["params"].cpu().numpy(), ref[j]["params"]), j
        assert np.array_equal(d["loss"].cpu().numpy(), ref[j]["loss"]), j
    streams = [torch.cuda.Stream() for _ in dsched]
    outs = []
    for s, kw in zip(streams, dsched):
        with torch.cuda.stream(s):
            outs.append(api.optimize_device(dt, **kw))
    torch.cuda.synchronize()
    for j, d in enumerate(outs):
        assert np.array_equal(d["params"].cpu().numpy(), ref[j]["params"]), j
        assert np.array_equal(d["loss"].cpu().numpy(), ref[j]["loss"]), j
