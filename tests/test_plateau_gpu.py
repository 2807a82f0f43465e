"""GPU tests of the fused optimiser's opt-in step reduction on a plateau (odam_sq_optimize_plateau[_host], api keywords
max_reductions and lr_factor).

The batches are the launch-shape rows of test_launch_shapes_gpu (every production build, staged and unstaged, in both
regimes, clusters of 1 to 4 CTAs), so each of the five plateau builds, which carry the step-size level, runs where the
library selects it.  Without and with an objective (Cauchy, random weights, a cosine schedule), every check is
exact:

1. The float32 restatement of the rule (tests/plateau_rule.py) applied to the run's own loss gives its iters,
   best_iter and reduce_iter: the decisions depend only on the losses the run wrote.
2. Up to an object's first reduction, its loss and parameter history are those of the convergence entry's run, which
   stops there; an object that never reduced matches that run in every output.
3. Replay: sampled objects re-run alone through the entry without the rule (odam_sq_optimize_objective_host), for
   their `iters` iterations under the schedule they actually saw (lr_scale_seen of their reduce_iter), give the same
   loss, parameter history, Adam moments, gradient and status; the parameters are the replay's last iterate, or with
   keep_best its lowest-loss one.  Without an objective the replay runs the default builds, which pins the reduced
   steps to the default arithmetic.
4. The device entry equals the host entry, and the fused oriented boxes are those of the returned parameters.
"""
import numpy as np
import pytest

from plateau_rule import lr_scale_seen, plateau_rule
from test_launch_shapes_gpu import LATENCY, SHAPES
from test_objective_gpu import _objective, _row_tracks

pytestmark = pytest.mark.gpu

ROWS = SHAPES + LATENCY
N_ITERS = 150
RULE = dict(patience=10, rel_tol=1e-3)
PLAT = dict(max_reductions=2, lr_factor=0.3)
R = PLAT["max_reductions"]
HIST = ("out_param_hist", "out_m", "out_v", "out_grad")


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


def _check_rule(run, n):
    """Check 1.  Returns (iters, best_iter, reduce_iter) of the restatement."""
    want = [plateau_rule(run["loss"][i], RULE["patience"], RULE["rel_tol"], R) for i in range(n)]
    iters = np.array([w[0] for w in want])
    best = np.array([w[1] for w in want])
    red = np.array([w[2] for w in want], np.int32).reshape(n, R)
    assert run["reduce_iter"].shape == (n, R) and run["reduce_iter"].dtype == np.int32
    assert np.array_equal(run["iters"], iters)
    assert np.array_equal(run["best_iter"], best)
    assert np.array_equal(run["reduce_iter"], red)
    assert np.array_equal(run["reductions"], (red >= 0).sum(1))
    for i in range(n):
        assert np.isnan(run["loss"][i, iters[i]:]).all() and np.isnan(run["out_param_hist"][i, iters[i]:]).all(), i
    return iters, best, red


def _check_against_convergence(run, conv, n):
    """Check 2."""
    for i in range(n):
        if run["reductions"][i] == 0:
            for key in run:
                if key not in ("reductions", "reduce_iter"):
                    assert np.array_equal(run[key][i], conv[key][i], equal_nan=True), (i, key)
            continue
        j0 = run["reduce_iter"][i, 0]
        assert conv["iters"][i] == j0, i
        assert np.array_equal(run["loss"][i, :j0], conv["loss"][i, :j0]), i
        assert np.array_equal(run["out_param_hist"][i, :j0], conv["out_param_hist"][i, :j0]), i


def _sample(run, rng, k=8):
    """Up to k objects that reduced their step: every one with R reductions that then stopped comes first, the rest
    at random."""
    red, iters = run["reductions"], run["iters"]
    full = np.nonzero((red == R) & (iters < N_ITERS))[0]
    some = np.setdiff1d(np.nonzero(red > 0)[0], full)
    pick = list(rng.permutation(full)[: k // 2]) + list(rng.permutation(some))
    return pick[:k]


@pytest.mark.parametrize("kind", [None, "cauchy"])
@pytest.mark.parametrize("row", ROWS, ids=[r.name for r in ROWS])
def test_rule_and_replay(api, row, kind):
    """Checks 1-3 on one launch-shape row, without and with an objective."""
    tracks, prior = _row_tracks(row), api.prior_table()
    n = tracks.n
    obj = _objective(tracks, kind, N_ITERS)
    kw = dict(prior=prior, n_iters=N_ITERS, extras=HIST, **row.options, **obj, **RULE)
    runs = {kb: api.optimize_host(tracks, **kw, **PLAT, keep_best=kb) for kb in (False, True)}
    run = runs[False]
    iters, best, red = _check_rule(run, n)
    assert (run["reductions"] > 0).any(), (row.name, "no object reduced its step")
    print(f"\n  {row.name} {kind or 'l1'}: reductions {np.bincount(run['reductions'], minlength=R + 1).tolist()}, "
          f"{int((iters < N_ITERS).sum())} of {n} stopped, iterations mean {iters.mean():.1f} max {iters.max()}")
    # keep_best changes the returned parameters only
    for key in run:
        if key != "params":
            assert np.array_equal(runs[True][key], run[key], equal_nan=True), (row.name, key)
    for kb in (False, True):
        _check_against_convergence(runs[kb], api.optimize_host(tracks, **kw, keep_best=kb), n)
    # 3: replays alone, under the schedule each object saw, on the entry without the rule
    q = api.query_launch(tracks.view_off, **row.options)
    fixed = dict(threads=q["threads"], max_slices=q["max_slices"], cluster=q["cluster"])
    base = obj.get("lr_scale")
    for i in _sample(run, np.random.default_rng(5)):
        a, b = int(tracks.view_off[i]), int(tracks.view_off[i + 1])
        k = int(iters[i])
        sched = lr_scale_seen(red[i], PLAT["lr_factor"], k, None if base is None else base[:k])
        o_i = dict(obj, lr_scale=sched)
        if obj:
            o_i.update(side_weight=obj["side_weight"][a:b])
        replay = api.optimize_host(tracks.slice(i, i + 1), prior=prior, n_iters=k, extras=HIST, **fixed, **o_i)
        label = (row.name, int(i), k, red[i].tolist())
        assert np.array_equal(replay["loss"][0], run["loss"][i, :k]), label
        assert np.array_equal(replay["out_param_hist"][0], run["out_param_hist"][i, :k]), label
        for key in ("status", "out_m", "out_v", "out_grad"):
            assert np.array_equal(replay[key][0], run[key][i]), label + (key,)
        assert np.array_equal(runs[False]["params"][i], replay["params"][0]), label
        bi = best[i]
        want = replay["params"][0] if bi < 0 else tracks.init[i] if bi == 0 else replay["out_param_hist"][0, bi - 1]
        assert np.array_equal(runs[True]["params"][i], want), label + ("keep_best",)


@pytest.mark.parametrize("row", [SHAPES[2], SHAPES[4], SHAPES[6], LATENCY[0], LATENCY[1]], ids=lambda r: r.name)
def test_device_entry_and_fused_boxes(api, row):
    """The device entry (with an objective, keep_best and the fused boxes) gives the host entry's bits, and the fused
    oriented boxes equal oriented_boxes_host of the returned parameters."""
    import torch
    tracks, prior = _row_tracks(row), api.prior_table()
    obj = _objective(tracks, "cauchy", N_ITERS)
    kw = dict(n_iters=N_ITERS, keep_best=True, **RULE, **PLAT, **row.options)
    host = api.optimize_host(tracks, prior=prior, extras=("out_corners", "out_box_flag"), **kw, **obj)
    dt = api.DeviceTracks(tracks, "cuda:0", prior)
    corners = torch.zeros((tracks.n, 8, 3), dtype=torch.float64, device="cuda:0")
    dev_obj = dict(obj, side_weight=torch.from_numpy(obj["side_weight"]).cuda())
    dev = api.optimize_device(dt, corners=corners, **kw, **dev_obj)
    torch.cuda.synchronize()
    for k in ("params", "loss", "status", "iters", "best_iter", "reductions", "reduce_iter"):
        assert np.array_equal(dev[k].cpu().numpy(), host[k], equal_nan=True), (row.name, k)
    assert np.array_equal(dev["corners"].cpu().numpy(), host["out_corners"])
    ref, flags = api.oriented_boxes_host(host["params"])
    assert np.array_equal(host["out_corners"], ref)
    assert np.array_equal(host["out_box_flag"], flags)
    assert (host["reductions"] > 0).any()
    # the dict of a call without reductions can be written again with them; the default entry after a plateau run on
    # the same stream gets its own Adam table again
    out = api.optimize_device(dt, n_iters=N_ITERS, **row.options)
    again = api.optimize_device(dt, n_iters=N_ITERS, out=out, **RULE, **PLAT, **row.options)
    torch.cuda.synchronize()
    assert again is out and "reduce_iter" in out
    plain = {k: v.cpu().numpy() for k, v in api.optimize_device(dt, n_iters=N_ITERS, **row.options).items()}
    torch.cuda.synchronize()
    ref = api.optimize_host(tracks, prior=prior, n_iters=N_ITERS, **row.options)
    for k in ("params", "loss", "status"):
        assert np.array_equal(plain[k], ref[k]), (row.name, k)
