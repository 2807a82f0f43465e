"""GPU tests of the fused optimiser's opt-in early stopping (odam_sq_optimize_converge[_host], api keywords patience,
rel_tol and keep_best).

The batches are the launch-shape rows of test_launch_shapes_gpu (every production build, staged and unstaged, in both
regimes, clusters of 1 to 4 CTAs), so each of the five convergence builds runs where the library selects it.  Every
check compares a run with the rule against a full run of the same inputs without it, object by object, exactly:

1. iters and best_iter equal the float32 restatement of the rule (tests/convergence_rule.py) applied to the full
   run's loss; the loss and parameter history of the iterations run are the full run's bits, the rest NaN; the
   parameters are those after the last step run, or with keep_best those at which the lowest loss was evaluated; the
   status flags are the full run's for the objects that ran to the end and a subset of them for the others.  Without
   and with an objective (Cauchy, random weights, a cosine schedule).
2. patience = 0 and keep_best = 0 give every output of the entry without the rule, bit for bit.
3. Sampled stopped objects, replayed alone for their `iters` iterations on the entry without the rule, give the same
   parameters, Adam moments, gradient and status; an object alone gives the bits it has inside the batch.
4. The device entry equals the host entry, and the fused oriented boxes are those of the returned parameters.
"""
import numpy as np
import pytest

from convergence_rule import stop_rule
from launch_checks import object_row
from test_launch_shapes_gpu import LATENCY, SHAPES
from test_objective_gpu import _objective, _row_tracks

pytestmark = pytest.mark.gpu

ROWS = SHAPES + LATENCY
N_ITERS = 150
RULE = dict(patience=10, rel_tol=1e-3)
HIST = ("out_param_hist", "out_m", "out_v", "out_grad")


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


def _check_against_full(tracks, full, run, keep_best):
    """Check 1 for every object of a run with RULE against the full run of the same inputs.  Returns iters."""
    n = tracks.n
    iters = np.array([stop_rule(full["loss"][i], **RULE)[0] for i in range(n)])
    best = np.array([stop_rule(full["loss"][i], **RULE)[1] for i in range(n)])
    assert np.array_equal(run["iters"], iters)
    assert np.array_equal(run["best_iter"], best)
    for i in range(n):
        k = iters[i]
        assert np.array_equal(run["loss"][i, :k], full["loss"][i, :k]), i
        assert np.isnan(run["loss"][i, k:]).all(), i
        assert np.array_equal(run["out_param_hist"][i, :k], full["out_param_hist"][i, :k]), i
        assert np.isnan(run["out_param_hist"][i, k:]).all(), i
        want = full["out_param_hist"][i, k - 1]
        if keep_best and best[i] >= 0:
            want = tracks.init[i] if best[i] == 0 else full["out_param_hist"][i, best[i] - 1]
        assert np.array_equal(run["params"][i], want), (i, k, best[i])
        if k == N_ITERS:
            for key in ("status", "out_m", "out_v", "out_grad"):
                assert np.array_equal(run[key][i], full[key][i]), (i, key)
        else:
            assert run["status"][i] & ~full["status"][i] == 0, (i, run["status"][i], full["status"][i])
    return iters


@pytest.mark.parametrize("kind", [None, "cauchy"])
@pytest.mark.parametrize("row", ROWS, ids=[r.name for r in ROWS])
def test_rule_against_full_run(api, row, kind):
    """Checks 1-3 on one launch-shape row, without and with an objective."""
    tracks, prior = _row_tracks(row), api.prior_table()
    obj = _objective(tracks, kind, N_ITERS)
    kw = dict(prior=prior, n_iters=N_ITERS, extras=HIST, **row.options, **obj)
    full = api.optimize_host(tracks, **kw)
    stopped = None
    for keep_best in (False, True):
        run = api.optimize_host(tracks, **kw, **RULE, keep_best=keep_best)
        iters = _check_against_full(tracks, full, run, keep_best)
        if stopped is None:
            stopped = np.nonzero(iters < N_ITERS)[0]
            assert len(stopped), (row.name, "no object stopped")
            print(f"\n  {row.name} {kind or 'l1'}: {len(stopped)} of {tracks.n} objects stopped, iterations mean "
                  f"{iters.mean():.1f} max {iters.max()}")
            kept = run
    # 2: the rule's build with patience 0 is the entry without it
    never = api.optimize_host(tracks, **kw, patience=0, rel_tol=1e-3)
    assert (never["iters"] == N_ITERS).all()
    assert np.array_equal(never["best_iter"], [stop_rule(x, 0, 0.0)[1] for x in full["loss"]])
    for key in ("params", "loss", "status") + HIST:
        assert np.array_equal(never[key], full[key]), (row.name, key)
    # 3: stopped objects replayed alone for their iterations, and alone with the rule
    q = api.query_launch(tracks.view_off, **row.options)
    fixed = dict(threads=q["threads"], max_slices=q["max_slices"], cluster=q["cluster"])
    rng = np.random.default_rng(3)
    for i in rng.choice(stopped, min(3, len(stopped)), replace=False):
        a, b = int(tracks.view_off[i]), int(tracks.view_off[i + 1])
        alone = tracks.slice(i, i + 1)
        o_i = dict(obj)
        if obj:
            o_i.update(side_weight=obj["side_weight"][a:b])
        k = int(kept["iters"][i])
        replay_kw = dict(o_i, lr_scale=o_i["lr_scale"][:k]) if obj else o_i
        replay = api.optimize_host(alone, prior=prior, n_iters=k, extras=HIST, **fixed, **replay_kw)
        for key in ("params", "status", "out_m", "out_v", "out_grad"):
            assert np.array_equal(replay[key][0], kept[key][i]), (row.name, int(i), key)
        one = api.optimize_host(alone, prior=prior, n_iters=N_ITERS, extras=HIST, **fixed, **o_i, **RULE)
        one = object_row(one, np.array([0, b - a]), 0)
        mine = object_row(kept, tracks.view_off, i)
        for key in mine:
            assert np.array_equal(one[key], mine[key], equal_nan=True), (row.name, int(i), key)


@pytest.mark.parametrize("row", [SHAPES[2], SHAPES[4], SHAPES[6], LATENCY[0], LATENCY[1]], ids=lambda r: r.name)
def test_device_entry_and_fused_boxes(api, row):
    """The device entry (with an objective, keep_best and the fused boxes) gives the host entry's bits, and the fused
    oriented boxes equal oriented_boxes_host of the returned parameters."""
    import torch
    tracks, prior = _row_tracks(row), api.prior_table()
    obj = _objective(tracks, "cauchy", N_ITERS)
    kw = dict(n_iters=N_ITERS, keep_best=True, **RULE, **row.options)
    host = api.optimize_host(tracks, prior=prior, extras=("out_corners", "out_box_flag"), **kw, **obj)
    dt = api.DeviceTracks(tracks, "cuda:0", prior)
    corners = torch.zeros((tracks.n, 8, 3), dtype=torch.float64, device="cuda:0")
    dev_obj = dict(obj, side_weight=torch.from_numpy(obj["side_weight"]).cuda())
    dev = api.optimize_device(dt, corners=corners, **kw, **dev_obj)
    torch.cuda.synchronize()
    for k in ("params", "loss", "status", "iters", "best_iter"):
        assert np.array_equal(dev[k].cpu().numpy(), host[k], equal_nan=True), (row.name, k)
    assert np.array_equal(dev["corners"].cpu().numpy(), host["out_corners"])
    ref, flags = api.oriented_boxes_host(host["params"])
    assert np.array_equal(host["out_corners"], ref)
    assert np.array_equal(host["out_box_flag"], flags)
    assert (host["iters"] < N_ITERS).any()
    # a dict of a call without the rule can be written again with it
    out = api.optimize_device(dt, n_iters=N_ITERS, **row.options)
    again = api.optimize_device(dt, n_iters=N_ITERS, out=out, **RULE, **row.options)
    torch.cuda.synchronize()
    assert again is out and "iters" in out
