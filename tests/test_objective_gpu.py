"""GPU tests of the fused optimiser's opt-in objective: per-side weights, robust residual losses and a learning-rate
schedule (odam_sq_optimize_objective[_host], api.optimize_host / optimize_device keywords).

The batches are the launch-shape rows of test_launch_shapes_gpu (every production build, staged and unstaged, in both
regimes), so each of the five objective builds runs where the library selects it.

1. Identity: all-one weights, L1 and an all-ones schedule (the objective build) equal the default build bit for bit.
2. A side of weight 0 is a masked-out side, bit for bit, status included.
3. Every object's last-iteration gradient against the float64 restatement (tests/objective64.py) under the kernel's
   own decisions, for each loss kind with random weights, at 1 and 5 iterations.
4. torch.optim.Adam through autograd.box_loss with the same objective and a non-constant schedule, teacher-forced
   against the fused entry step by step.
5. A zero schedule entry leaves the parameters of that iteration unchanged.
6. Device entry = host entry; an object alone = the same object in a batch; argument errors on tensors.
7. What the feature is for: a config-2 scene with a fifth of every object's boxes replaced by random ones, fitted with
   L1, Cauchy, and weights that drop the corrupted views (printed, not gated).
"""
import numpy as np
import pytest

from golden_cases import EDGE_KINDS, TOL_LOSS, TOL_PARAM, edge_object, rel_loss, rel_param
from launch_checks import EXTRAS, TAU_KERNEL, check_decisions, object_row, pack
from oracle import grad64 as G64
from test_launch_shapes_gpu import LATENCY, SHAPES, _tracks
import objective64 as O64

pytestmark = pytest.mark.gpu

ROWS = SHAPES + LATENCY
SCALE = {"l1": None, "smooth_l1": 4.0, "cauchy": 8.0}   # beta / c in pixels: the synthetic detections carry 3 px noise


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


_cache = {}


def _row_tracks(row):
    """The row's batch: test_launch_shapes_gpu's for the dense rows; the edge objects, or two 1500-view tracks, for the
    latency-regime rows."""
    if row.name not in _cache:
        if row in SHAPES:
            _cache[row.name] = _tracks(row)
        elif row.name == "11 edge objects":
            _cache[row.name] = pack([edge_object(k) for k in EDGE_KINDS])
        else:
            from odam_b200 import api, synthetic
            _cache[row.name] = api.pack_scene(synthetic.make_scene(*row.groups[0], seed=21))
    return _cache[row.name]


def _weights(tracks, seed, zeros=0.2):
    rng = np.random.default_rng(seed)
    w = rng.uniform(0.1, 2.0, (tracks.total_views, 4)).astype(np.float32)
    w[rng.uniform(size=w.shape) < zeros] = 0
    return w


def _objective(tracks, kind, n_iters):
    """The keywords of no objective, or of Cauchy with random weights and a cosine schedule."""
    if kind is None:
        return {}
    sched = (0.5 * (1 + np.cos(np.pi * np.arange(n_iters) / n_iters))).astype(np.float32)
    return dict(side_weight=_weights(tracks, 9), loss="cauchy", loss_scale=8.0, lr_scale=sched)


def _same(a, b, keys, label):
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), (label, k)


@pytest.mark.parametrize("row", ROWS, ids=[r.name for r in ROWS])
def test_identity(api, row):
    """All-one weights, loss="l1" and lr_scale of ones run the objective build and give the default build's bits in
    params, loss, status and every diagnostic output."""
    tracks, prior, n_iters = _row_tracks(row), api.prior_table(), 5
    ref = api.optimize_host(tracks, prior=prior, n_iters=n_iters, extras=EXTRAS, **row.options)
    obj = api.optimize_host(tracks, prior=prior, n_iters=n_iters, extras=EXTRAS, **row.options,
                            side_weight=np.ones((tracks.total_views, 4), np.float32), loss="l1",
                            lr_scale=np.ones(n_iters, np.float32))
    _same(ref, obj, ("params", "loss", "status") + EXTRAS, row.name)


@pytest.mark.parametrize("row", [ROWS[0], ROWS[6], LATENCY[0]], ids=lambda r: r.name)
@pytest.mark.parametrize("loss", ["l1", "cauchy"])
def test_zero_weight_is_masked_out(api, row, loss):
    """Zeroing the weights of a seeded fifth of the sides (and of every side of the objects the default run flags with
    ODAM_SQ_ST_NO_VALID_PT: the behind-camera edge object) equals masking those sides out, bit for bit, status
    included: the flag follows the effective weight, so those objects are flagged in neither run."""
    from odam_b200.api import PackedTracks
    tracks, prior = _row_tracks(row), api.prior_table()
    w = np.ones((tracks.total_views, 4), np.float32)
    w[np.random.default_rng(7).uniform(size=w.shape) < 0.2] = 0
    behind = np.nonzero(api.optimize_host(tracks, prior=prior, n_iters=1, **row.options)["status"] & 4)[0]
    assert len(behind) == 1, behind
    for i in behind:
        w[tracks.view_off[i]:tracks.view_off[i + 1]] = 0
    masked = PackedTracks(tracks.init, tracks.cls, tracks.view_off, tracks.Ms, tracks.box,
                          (tracks.mask * (w != 0)).astype(np.uint8))
    kw = dict(prior=prior, n_iters=5, extras=EXTRAS, loss=loss, loss_scale=SCALE[loss], **row.options)
    a = api.optimize_host(tracks, side_weight=w, **kw)
    # the masked run needs the objective build too (for L1: weights of 1), so both run the same machine code
    b = api.optimize_host(masked, side_weight=np.ones_like(w), **kw)
    _same(a, b, ("params", "loss", "status") + EXTRAS, (row.name, loss))
    assert not any(a["status"][i] for i in behind)


def _check_gradients(api, tracks, prior, n_iters, label, options, **obj):
    o = api.optimize_host(tracks, prior=prior, n_iters=n_iters, extras=EXTRAS, **options, **obj)
    w = obj.get("side_weight")
    worst = np.zeros(9)
    for i in range(tracks.n):
        a, b = int(tracks.view_off[i]), int(tracks.view_off[i + 1])
        state = tracks.init[i] if n_iters == 1 else o["out_param_hist"][i, -2]
        etas, omegas = G64.angles(o["out_grids"][i], o["out_eta_idx"][i])
        Ms, box, mask = tracks.Ms[a:b], tracks.box[a:b], tracks.mask[a:b]
        pred, arg = o["out_pred"][a:b], o["out_arg"][a:b]
        if b > a:
            check_decisions(state, etas, omegas, Ms, pred, arg, (label, i))
        g, sc = O64.grad64(state, Ms, box, mask, etas, omegas, arg, np.sign(pred - box), prior[tracks.cls[i]].reshape(3, 3),
                           tracks.init[i][4:7], True, weight=None if w is None else w[a:b], loss=obj["loss"],
                           loss_scale=obj["loss_scale"], residual=pred - box)
        r = G64.ratio(o["out_grad"][i], g, sc)
        assert (r <= TAU_KERNEL).all(), (label, i, b - a, r, o["out_grad"][i], g)
        worst = np.maximum(worst, r)
    return worst


@pytest.mark.parametrize("row", ROWS, ids=[r.name for r in ROWS])
def test_gradient_against_float64(api, row):
    """For each loss kind with random weights (a fifth of them zero) and a non-constant schedule, at 1 and 5
    iterations: every object's last-iteration gradient within TAU_KERNEL * scale of the float64 restatement, with rho'
    taken at the kernel's own fp32 residual (tests/objective64.py says why)."""
    tracks, prior = _row_tracks(row), api.prior_table()
    out = []
    for k, loss in enumerate(SCALE):
        w = _weights(tracks, k)
        worst = np.zeros(9)
        for n_iters in (1, 5):
            sched = np.linspace(1.0, 0.2, n_iters).astype(np.float32)
            worst = np.maximum(worst, _check_gradients(api, tracks, prior, n_iters, (row.name, loss, n_iters),
                                                       row.options, side_weight=w, loss=loss,
                                                       loss_scale=SCALE[loss], lr_scale=sched))
        out.append(f"{loss} {worst.max():.1e}")
    print(f"\n  {row.name}: worst |g - g64| / scale " + ", ".join(out))


@pytest.mark.parametrize("loss", ["smooth_l1", "cauchy"])
def test_torch_optim_adam_loop_matches_fused_objective(api, loss):
    """20 steps of torch.optim.Adam (the reference's two parameter groups) through box_loss(weight=, loss=,
    loss_scale=) with the prior, the learning rates set every step from a cosine schedule as a torch scheduler sets
    group["lr"].  At every state the fused objective entry is teacher-forced for one step from the optimiser's own m, v
    and step count with lr_scale = [that step's factor]: on the steps whose decisions agree, parameters within
    TOL_PARAM and loss within TOL_LOSS, and decisions agree on at least 80 % of the object-steps."""
    import torch
    from odam_b200 import autograd as AG
    from odam_b200.api import PackedTracks
    from test_autograd_gpu import _config2, _dev
    tr = _config2(api).slice(0, 6)
    prior = api.prior_table()
    d = _dev(tr, prior=prior)
    w = _weights(tr, 11)
    wt = torch.from_numpy(w).cuda()
    lin = d["params"][:, :7].clone().requires_grad_(True)
    shp = d["params"][:, 7:9].clone().requires_grad_(True)
    opt = torch.optim.Adam([{"params": [lin]}, {"params": [shp], "lr": 0.1}], lr=0.01)
    base = [g["lr"] for g in opt.param_groups]
    sched = (0.5 * (1 + np.cos(np.pi * np.arange(20) / 20))).astype(np.float32)
    s0 = tr.init[:, 4:7].copy()
    checked = total = 0
    worst_p = worst_l = 0.0
    for it in range(20):
        for g, b in zip(opt.param_groups, base):
            g["lr"] = b * float(sched[it])
        state = torch.cat([lin, shp], 1).detach().cpu().numpy()
        st = lambda key: (np.zeros((tr.n, 9), np.float32) if not opt.state else
                          torch.cat([opt.state[lin][key], opt.state[shp][key]], 1).cpu().numpy())
        ft = PackedTracks(state, tr.cls, tr.view_off, tr.Ms, tr.box, tr.mask)
        o = api.optimize_host(ft, prior=prior, n_iters=1, m0=st("exp_avg"), v0=st("exp_avg_sq"), step0=it, s0=s0,
                              extras=("out_arg",), side_weight=w, loss=loss, loss_scale=SCALE[loss],
                              lr_scale=sched[it:it + 1])
        opt.zero_grad()
        params = torch.cat([lin, shp], 1)
        L = AG.box_loss(params, d["view_off"], d["Ms"], d["box"], d["mask"], prior=d["prior"], cls=d["cls"], s0=d["s0"],
                        weight=wt, loss=loss, loss_scale=SCALE[loss])
        _, arg = AG.box_sides(params.detach(), d["view_off"], d["Ms"])
        L.sum().backward()
        opt.step()
        after = torch.cat([lin, shp], 1).detach().cpu().numpy()
        L, arg = L.detach().cpu().numpy(), arg.cpu().numpy()
        for i in range(tr.n):
            a, b = int(tr.view_off[i]), int(tr.view_off[i + 1])
            total += 1
            if not np.array_equal(arg[a:b], o["out_arg"][a:b]):
                continue
            checked += 1
            rp = float(rel_param(after[i], o["params"][i]).max())
            rl = float(rel_loss(L[i], o["loss"][i, 0]))
            assert rp <= TOL_PARAM and rl <= TOL_LOSS, (it, i, rp, rl)
            worst_p, worst_l = max(worst_p, rp), max(worst_l, rl)
    print(f"\n  {loss}: torch.optim.Adam loop, {total} object-steps, {checked} with the fused kernel's decisions; worst "
          f"rel err params {worst_p:.1e}, loss {worst_l:.1e}")
    assert checked >= 0.8 * total


def test_zero_schedule_entry_freezes_the_step(api):
    """Where lr_scale[it] == 0 the parameters after iteration it equal those after it - 1 (or the start), bit for bit,
    on the default builds (schedule alone) and the objective build.  A schedule of ones alone is the default run."""
    tracks, prior = _row_tracks(SHAPES[0]), api.prior_table()
    sched = np.array([0, 1, 0, 0, 0.5, 0, 1], np.float32)
    ref = api.optimize_host(tracks, prior=prior, n_iters=len(sched), extras=("out_param_hist",))
    ones = api.optimize_host(tracks, prior=prior, n_iters=len(sched), extras=("out_param_hist",),
                             lr_scale=np.ones_like(sched))
    _same(ref, ones, ("params", "loss", "status", "out_param_hist"), "ones")
    for obj in (dict(), dict(loss="cauchy", loss_scale=8.0, side_weight=_weights(tracks, 3))):
        o = api.optimize_host(tracks, prior=prior, n_iters=len(sched), extras=("out_param_hist",), lr_scale=sched, **obj)
        h = np.concatenate([tracks.init[:, None], o["out_param_hist"]], 1)
        for it in np.nonzero(sched == 0)[0]:
            assert np.array_equal(h[:, it + 1], h[:, it]), (obj.keys(), it)
        for it in np.nonzero(sched != 0)[0]:
            assert not np.array_equal(h[:, it + 1], h[:, it]), (obj.keys(), it)


@pytest.mark.parametrize("row", [SHAPES[2], SHAPES[6], LATENCY[0]], ids=lambda r: r.name)
def test_entries_and_batches(api, row):
    """The device entry with a CUDA weight tensor and the host entry give the same bits; sampled objects run alone
    (the latency-regime builds) give the bits they have inside the batch."""
    import torch
    tracks, prior = _row_tracks(row), api.prior_table()
    w = _weights(tracks, 5)
    kw = dict(loss="cauchy", loss_scale=8.0, lr_scale=np.linspace(1, 0.3, 5).astype(np.float32))
    o = api.optimize_host(tracks, prior=prior, n_iters=5, extras=EXTRAS, side_weight=w, **kw, **row.options)
    dt = api.DeviceTracks(tracks, "cuda:0", prior)
    dev = api.optimize_device(dt, n_iters=5, side_weight=torch.from_numpy(w).cuda(), **kw, **row.options)
    torch.cuda.synchronize()
    for k in ("params", "loss", "status"):
        assert np.array_equal(dev[k].cpu().numpy(), o[k]), (row.name, "device entry", k)
    q = api.query_launch(tracks.view_off, **row.options)
    fixed = dict(threads=q["threads"], max_slices=q["max_slices"], cluster=q["cluster"])
    for i in np.random.default_rng(1).choice(tracks.n, min(4, tracks.n), replace=False):
        a, b = int(tracks.view_off[i]), int(tracks.view_off[i + 1])
        one = api.optimize_host(tracks.slice(i, i + 1), prior=prior, n_iters=5, extras=EXTRAS, side_weight=w[a:b],
                                **kw, **fixed)
        one = object_row(one, np.array([0, b - a]), 0)
        mine = object_row(o, tracks.view_off, i)
        for k in mine:
            assert np.array_equal(one[k], mine[k], equal_nan=True), (row.name, int(i), k)


def test_tensor_argument_errors(api):
    """side_weight of optimize_device and weight of box_loss: wrong shape, dtype or device raise ValueError, as do an
    unknown loss or a robust kind without a scale > 0."""
    import torch
    from odam_b200 import autograd as AG
    from test_autograd_gpu import _dev
    tracks = pack([edge_object("plain"), edge_object("V1")])
    SV = tracks.total_views
    dt = api.DeviceTracks(tracks, "cuda:0")
    good = torch.ones((SV, 4), dtype=torch.float32, device="cuda:0")
    bad = [torch.ones((SV + 1, 4), device="cuda:0"), torch.ones((SV, 4), dtype=torch.float64, device="cuda:0"),
           torch.ones((SV, 4)), torch.ones((4, SV), device="cuda:0").t()]
    for w in bad:
        with pytest.raises(ValueError):
            api.optimize_device(dt, n_iters=2, side_weight=w)
    for kw in (dict(loss="huber", loss_scale=1.0), dict(loss="cauchy"), dict(lr_scale=np.ones(3))):
        with pytest.raises(ValueError):
            api.optimize_device(dt, n_iters=2, side_weight=good, **kw)
    d = _dev(tracks)
    args = (d["params"], d["view_off"], d["Ms"], d["box"], d["mask"])
    for w in bad[:3]:
        with pytest.raises(ValueError):
            AG.box_loss(*args, weight=w)
    for kw in (dict(loss="huber", loss_scale=1.0), dict(loss="cauchy"), dict(loss="smooth_l1", loss_scale=0.0),
               dict(loss="cauchy", loss_scale=float("nan"))):
        with pytest.raises(ValueError):
            AG.box_loss(*args, **kw)
    # the defaults are today's loss, and all-one weights do not change it
    assert torch.equal(AG.box_loss(*args), AG.box_loss(*args, weight=good))


def test_corrupted_boxes_report(api):
    """A seeded config-2 scene with 20 % of every object's views given random boxes, 200 iterations: median centre error
    (m) and median relative dimension error against the scene's ground truth for L1, Cauchy (c = 8 px), and L1 with the
    corrupted views weighted 0.  Printed, not gated."""
    from odam_b200 import synthetic
    from odam_b200.api import PackedTracks
    sc = synthetic.make_config(2)
    tr = api.pack_scene(sc)
    rng = np.random.default_rng(2)
    box = tr.box.copy()
    w = np.ones_like(box)
    for i in range(tr.n):
        a = int(tr.view_off[i])
        bad = a + rng.choice(sc.V, sc.V // 5, replace=False)
        x = np.sort(rng.uniform(20, synthetic.IMG_W - 20, (len(bad), 2)), 1)
        y = np.sort(rng.uniform(20, synthetic.IMG_H - 20, (len(bad), 2)), 1)
        box[bad] = np.stack([x[:, 0], x[:, 1], y[:, 0], y[:, 1]], 1)
        w[bad] = 0
    noisy = PackedTracks(tr.init, tr.cls, tr.view_off, tr.Ms, box, tr.mask)
    prior = api.prior_table()
    runs = {"clean boxes, L1": (tr, {}), "corrupted, L1": (noisy, {}),
            "corrupted, Cauchy c=8": (noisy, dict(loss="cauchy", loss_scale=8.0)),
            "corrupted, smooth L1 beta=4": (noisy, dict(loss="smooth_l1", loss_scale=4.0)),
            "corrupted, corrupted views weighted 0": (noisy, dict(side_weight=w))}
    lines = []
    for name, (t, kw) in runs.items():
        o = api.optimize_host(t, prior=prior, n_iters=200, **kw)
        p = o["params"].astype(np.float64)
        centre = np.linalg.norm(p[:, :3] - sc.gt["centre"], axis=1)
        dims = np.abs(2 * p[:, 4:7] ** 2 - sc.gt["dims"]) / sc.gt["dims"]
        lines.append(f"  {name:40s} median centre error {np.median(centre):.3f} m, median dims error "
                     f"{100 * np.median(dims):.1f} %")
    print("\n  config 2 (50 objects x 50 views), 200 iterations, 20 % of each object's views with random boxes:\n"
          + "\n".join(lines))
