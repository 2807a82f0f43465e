"""Checks shared by the GPU tests of the fused optimiser: packing objects into one batch, the last iteration's gradient
of every object of a launch against float64 under the kernel's own decisions, and one object's first iterations
against the C oracle."""
import numpy as np

from golden_cases import TOL_LOSS, TOL_PARAM, rel_loss, rel_param
from oracle import grad64 as G64

# About 10x the reference's own measured error (5.4e-7, tests/test_backward_ref.py) and ~34 eps32: the kernel sums the
# same terms in another order (warp butterfly, warps, cluster ranks).
TAU_KERNEL = 4e-6
EXTRAS = ("out_grad", "out_m", "out_v", "out_grids", "out_eta_idx", "out_arg", "out_pred", "out_param_hist")
DECISIONS = ("out_arg", "out_eta_idx", "out_pred")
PER_VIEW = ("out_arg", "out_pred")   # outputs with one row per view; the others have one row per object
BBOX_RTOL, BBOX_ATOL = 2e-6, 2e-3   # test_get_bbox_csr_many_objects: float64 get_bbox of the kernel's own points


def pack(objs):
    """[(init, Ms, box, mask, cls)] -> PackedTracks."""
    from odam_b200.api import PackedTracks
    off = np.concatenate([[0], np.cumsum([len(o[1]) for o in objs])]).astype(np.int32)
    return PackedTracks(np.stack([o[0] for o in objs]).astype(np.float32), np.array([o[4] for o in objs], np.int32), off,
                        np.concatenate([o[1] for o in objs]).astype(np.float32),
                        np.concatenate([o[2] for o in objs]).astype(np.float32),
                        np.concatenate([o[3] for o in objs]).astype(np.uint8))


def object_row(out, view_off, i):
    """Object i's part of every output of a launch over the objects of view_off."""
    a, b = int(view_off[i]), int(view_off[i + 1])
    return {k: (v[a:b] if k in PER_VIEW else v[i]) for k, v in out.items()}


def check_decisions(state, etas, omegas, Ms, pred, arg, label):
    """pred = float64 projection of the arg point = float64 extremum over every valid point (up to near-ties)."""
    u, w, valid = G64.project(state, etas, omegas, Ms)
    V = len(Ms)
    tol = lambda x: BBOX_ATOL + BBOX_RTOL * np.abs(x)
    for sd in range(4):
        c = u if sd < 2 else w
        big = np.where(valid, c, np.inf if sd % 2 == 0 else -np.inf)
        ext = big.min(1) if sd % 2 == 0 else big.max(1)
        has = arg[:, sd] >= 0
        at = c[np.arange(V), np.maximum(arg[:, sd], 0)]
        assert (np.abs(pred[has, sd] - at[has]) <= tol(at[has])).all(), (label, sd, "pred != projection of arg point")
        assert valid[np.arange(V), np.maximum(arg[:, sd], 0)][has].all(), (label, sd, "arg point not valid")
        assert (np.abs(pred[has, sd] - ext[has]) <= tol(ext[has])).all(), (label, sd, "arg point is not the extremum")
        assert (np.abs(pred[~has, sd]) == 1e6).all(), (label, sd, "no valid point but no sentinel")


def check_launch(api, tracks, prior=None, n_iters=1, representation="super_quadric", label="", quiet=False, **kw):
    """One launch with every diagnostic output; the last iteration's gradient of every object against float64 under
    the kernel's own decisions; prints the worst ratio per component unless quiet.  Returns the launch's outputs and
    that worst ratio [9]."""
    o = api.optimize_host(tracks, prior=prior, n_iters=n_iters, representation=representation, extras=EXTRAS, **kw)
    opt = representation == "super_quadric"
    nc = 9 if opt else 7
    worst = np.zeros(9)
    for i in range(tracks.n):
        a, b = int(tracks.view_off[i]), int(tracks.view_off[i + 1])
        state = tracks.init[i] if n_iters == 1 else o["out_param_hist"][i, -2]
        etas, omegas = G64.angles(o["out_grids"][i], o["out_eta_idx"][i])
        Ms, box, mask = tracks.Ms[a:b], tracks.box[a:b], tracks.mask[a:b]
        pred, arg = o["out_pred"][a:b], o["out_arg"][a:b]
        if b > a:
            check_decisions(state, etas, omegas, Ms, pred, arg, (label, i))
        p33 = None if prior is None else prior[tracks.cls[i]].reshape(3, 3)
        g, sc = G64.grad64(state, Ms, box, mask, etas, omegas, arg, np.sign(pred - box), p33, tracks.init[i][4:7], opt)
        r = G64.ratio(o["out_grad"][i][:nc], g[:nc], sc[:nc])
        assert (r <= TAU_KERNEL).all(), (label, i, b - a, r, o["out_grad"][i], g)
        if not opt:
            assert (o["out_grad"][i][7:9] == 0).all(), (label, i)
        worst[:nc] = np.maximum(worst[:nc], r)
    if not quiet:
        print(f"  {label}: worst |g - g64| / scale " + " ".join(f"{x:.1e}" for x in worst))
    return o, worst


def oracle_first_iterations(coracle, tracks, i, prior, iters, launch, loss0):
    """Object i of `tracks` against the C oracle over its first `iters` iterations.  launch(k) gives the object's
    outputs (object_row) of a k-iteration launch with the DECISIONS extras; loss0 is its first loss in the launch under
    test, which starts from the oracle's own state and must agree.  BASELINE tolerances hold when every discrete
    decision of those iterations (arg-extreme point, residual sign, eta bucket) agrees with the oracle's; a near-tie
    resolved differently by two fp32 implementations moves the parameters by up to lr -- such an object is bounded here
    and returned as (i, worst relative parameter error, worst relative loss error) for the caller to count (DESIGN.md
    section 2), not exempted silently.  Returns None for an object that agrees."""
    a, b = tracks.view_off[i], tracks.view_off[i + 1]
    r = coracle.run(tracks.init[i], tracks.Ms[a:b], tracks.box[a:b], tracks.mask[a:b],
                    None if prior is None else prior[tracks.cls[i]], iters, record_indices=True)
    assert rel_loss(loss0, r["loss"][0]) <= TOL_LOSS, i          # same state: the forward must agree
    # the optional outputs describe the LAST iteration of a launch, so iteration k is read from a k-iteration launch
    # of the same deterministic trajectory
    live = tracks.mask[a:b].astype(bool)
    agree, worst_p, worst_l = True, 0.0, 0.0
    for k in range(1, iters + 1):
        o = launch(k)
        agree &= np.array_equal(o["out_arg"].reshape(-1, 4)[live], r["arg"][k - 1][live])
        agree &= np.array_equal(o["out_eta_idx"], r["eta_idx"][k - 1].astype(np.uint8))
        agree &= np.array_equal(np.sign(o["out_pred"].reshape(-1, 4) - tracks.box[a:b])[live],
                                np.sign(r["pred"][k - 1] - tracks.box[a:b])[live])
        worst_p = max(worst_p, float(rel_param(o["params"], r["params"][k - 1]).max()))
        worst_l = max(worst_l, float(rel_loss(o["loss"], r["loss"][:k]).max()))
    if agree:
        assert worst_p <= TOL_PARAM and worst_l <= TOL_LOSS, (i, worst_p, worst_l)
        return None
    assert worst_p <= 2e-2, (i, worst_p)
    return int(i), worst_p, worst_l
