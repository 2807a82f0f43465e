"""GPU tests of the differentiable ops (odam_b200/autograd.py): surface_points, box_sides and box_loss.

- Forward: surface_points equals the library's sampler bit for bit; the box_sides decisions are legitimate (each side is
  the float64 projection of its arg sample and the float64 extremum; the +-1e6 sentinel appears exactly where it wins).
- Against the fused optimiser: the same sides where the arg agrees, and the same gradient and loss as one teacher-forced
  step of the fused kernel.
- Against float64 (oracle/grad64.py) under the ops' own decisions, at TAU_KERNEL * scale.
- Against the reference's recorded states, and a torch.optim.Adam loop teacher-forced against the fused kernel.
- Plumbing: determinism, batch independence, streams, n = 0, gradient accumulation, argument errors.
"""
import numpy as np
import pytest

from golden_cases import EDGE_KINDS, FLOOR, TOL_LOSS, TOL_PARAM, all_cases, edge_object, rel_loss, rel_param, wide_cases
from oracle import grad64 as G64
from surface_vjp64 import surface_vjp64
from test_backward_gpu import EXTRAS, TAU_KERNEL, _check_decisions, _pack, _ragged_tracks

pytestmark = pytest.mark.gpu

TAU = TAU_KERNEL
REPRS = ("cube", "quadric", "super_quadric")


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


@pytest.fixture(scope="module")
def AG():
    from odam_b200 import autograd
    return autograd


def _torch():
    import torch
    return torch


def _dev(tracks, device="cuda:0", prior=None):
    """PackedTracks -> dict of CUDA tensors the ops take (view_off stays on the host: it is checked there)."""
    torch = _torch()
    t = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(device)
    return dict(params=t(tracks.init, np.float32), view_off=torch.from_numpy(np.ascontiguousarray(tracks.view_off, np.int32)),
                Ms=t(tracks.Ms, np.float32), box=t(tracks.box, np.float32), mask=t(tracks.mask, np.uint8),
                cls=t(tracks.cls, np.int32), s0=t(tracks.init[:, 4:7], np.float32),
                prior=None if prior is None else t(prior, np.float32))


def _with_repr(tracks, representation):
    from odam_b200.api import PackedTracks
    init = tracks.init.copy()
    if representation == "cube":
        init[:, 7:9] = -10000.0
    elif representation == "quadric":
        init[:, 7:9] = 0.0
    return PackedTracks(init, tracks.cls, tracks.view_off, tracks.Ms, tracks.box, tracks.mask)


def _edge_tracks(representation="super_quadric"):
    return _with_repr(_pack([edge_object(k) for k in EDGE_KINDS]), representation)


def _long_tracks(api, V):
    from odam_b200 import synthetic
    return api.pack_scene(synthetic.make_scene(2, V, seed=21))


def _config2(api):
    from odam_b200 import synthetic
    return api.pack_scene(synthetic.make_config(2))


def _grads(AG, d, prior=None, G=None):
    """(pred, arg, loss, grad of box_loss.sum()) and, when G is given, the surface VJP of G; numpy."""
    torch = _torch()
    p = d["params"].clone().requires_grad_(True)
    pred, arg = AG.box_sides(p, d["view_off"], d["Ms"])
    kw = {} if prior is None else dict(prior=d["prior"], cls=d["cls"], s0=d["s0"])
    loss = AG.box_loss(p, d["view_off"], d["Ms"], d["box"], d["mask"], **kw)
    loss.sum().backward()
    out = [pred.detach().cpu().numpy(), arg.cpu().numpy(), loss.detach().cpu().numpy(), p.grad.cpu().numpy()]
    if G is not None:
        q = d["params"].clone().requires_grad_(True)
        (AG.surface_points(q) * torch.from_numpy(G).to(q.device)).sum().backward()
        out.append(q.grad.cpu().numpy())
    torch.cuda.synchronize()
    return out


def _ulps(a, b):
    return np.abs(a.astype(np.float64) - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)).astype(np.float32))


# ---------------------------------------------------------------------------------------------------------------- 1


def test_surface_points_forward_bit_identical(api, AG):
    """surface_points equals odam_sq_sample_points_host bit for bit: ragged batch, edge objects, config 2."""
    torch = _torch()
    for label, tr in (("ragged", _ragged_tracks(api)), ("edge", _edge_tracks()), ("config 2", _config2(api))):
        pts = AG.surface_points(torch.from_numpy(tr.init).cuda()).cpu().numpy()
        ref = api.sample_points_host(tr.init)
        assert pts.shape == (tr.n, 1000, 3) and np.array_equal(pts, ref), label
        print(f"  surface_points {label}: {tr.n} objects bit-identical")


def _check_sentinels(state, etas, omegas, Ms, pred, arg, label):
    """The sentinel wins exactly where, in float64, the first minimum (maximum) of valid ? coord : +-1e6 is not a valid
    sample."""
    u, w, valid = G64.project(state, etas, omegas, Ms)
    for sd in range(4):
        c = u if sd < 2 else w
        big = 1e6 if sd % 2 == 0 else -1e6
        cand = np.where(valid, c, big)
        win = cand.argmin(1) if sd % 2 == 0 else cand.argmax(1)
        sentinel = ~valid[np.arange(len(Ms)), win]
        assert np.array_equal(arg[:, sd] < 0, sentinel), (label, sd)
        assert (pred[sentinel, sd] == big).all(), (label, sd)


@pytest.mark.parametrize("batch", ["ragged", "edge", "V1500", "V2500"])
def test_box_sides_decisions(api, AG, batch):
    """Every (view, side): pred is the float64 projection of the arg sample and the float64 extremum over valid samples;
    the +-1e6 sentinel appears exactly where no valid sample beats it."""
    tr = {"ragged": lambda: _ragged_tracks(api), "edge": _edge_tracks, "V1500": lambda: _long_tracks(api, 1500),
          "V2500": lambda: _long_tracks(api, 2500)}[batch]()
    d = _dev(tr)
    pred, arg = (x.cpu().numpy() for x in AG.box_sides(d["params"], d["view_off"], d["Ms"]))
    o = api.optimize_host(tr, n_iters=1, extras=("out_grids", "out_eta_idx"))
    for i in range(tr.n):
        a, b = int(tr.view_off[i]), int(tr.view_off[i + 1])
        etas, omegas = G64.angles(o["out_grids"][i], o["out_eta_idx"][i])
        _check_decisions(tr.init[i], etas, omegas, tr.Ms[a:b], pred[a:b], arg[a:b], (batch, i))
        _check_sentinels(tr.init[i], etas, omegas, tr.Ms[a:b], pred[a:b], arg[a:b], (batch, i))
    print(f"  box_sides {batch}: {tr.total_views} views, {int((arg < 0).sum())} sentinel sides, decisions legitimate")


# ------------------------------------------------------------------------------------------------------------ 2 + 3


def _vs_fused(api, AG, tr, prior, representation, label):
    """One n_iters = 1 fused launch against box_sides / box_loss on the same batch.  Returns counts."""
    tr = _with_repr(tr, representation)
    o = api.optimize_host(tr, prior=prior, n_iters=1, representation=representation, extras=EXTRAS)
    d = _dev(tr, prior=prior)
    pred, arg, loss, g = _grads(AG, d, prior)
    fp, fa = o["out_pred"], o["out_arg"]
    same = arg == fa
    assert np.array_equal(pred[same], fp[same]), label
    beyond = np.where(np.arange(4) % 2 == 0, pred >= 1e6, pred <= -1e6)
    clip = ~same & (fa < 0) & (arg >= 0) & beyond           # the fused kernel's documented +-1e6 clipping
    other = ~same & ~clip
    assert (_ulps(pred[other], fp[other]) <= 2).all(), (label, pred[other], fp[other])
    nc = 9 if representation == "super_quadric" else 7
    worst_f, worst_64 = np.zeros(9), np.zeros(9)
    agree_obj = 0
    for i in range(tr.n):
        a, b = int(tr.view_off[i]), int(tr.view_off[i + 1])
        etas, omegas = G64.angles(o["out_grids"][i], o["out_eta_idx"][i])
        p33 = None if prior is None else prior[tr.cls[i]].reshape(3, 3)
        sign = np.sign(pred[a:b] - tr.box[a:b])
        g64, sc = G64.grad64(tr.init[i], tr.Ms[a:b], tr.box[a:b], tr.mask[a:b], etas, omegas, arg[a:b], sign, p33,
                             tr.init[i][4:7], True)
        r = G64.ratio(g[i], g64, sc)
        assert (r <= TAU).all(), (label, i, "vs float64", r, g[i], g64)
        worst_64 = np.maximum(worst_64, r)
        if not same[a:b].all():
            continue
        agree_obj += 1
        rf = G64.ratio(g[i][:nc], o["out_grad"][i][:nc].astype(np.float64), sc[:nc])
        assert (rf <= 2 * TAU).all(), (label, i, "vs fused", rf, g[i], o["out_grad"][i])
        worst_f[:nc] = np.maximum(worst_f[:nc], rf)
        assert rel_loss(loss[i], o["loss"][i, 0]) <= TOL_LOSS, (label, i, loss[i], o["loss"][i, 0])
    print(f"  {label}: sides {int(same.sum())}/{same.size} with the fused kernel's arg, {int(other.sum())} others within "
          f"2 ulp, {int(clip.sum())} beyond the fused kernel's +-1e6 clip; objects agreeing {agree_obj}/{tr.n}; worst "
          f"|g - g_fused| / scale " + " ".join(f"{x:.1e}" for x in worst_f) + "; worst |g - g64| / scale "
          + " ".join(f"{x:.1e}" for x in worst_64))
    return agree_obj


@pytest.mark.parametrize("representation", REPRS)
def test_box_loss_vs_fused_and_float64(api, AG, representation):
    """Ragged batch, edge objects, 1500 and 2500 views, with and without the prior: sides against the fused kernel's
    out_pred / out_arg, box_loss(...).sum().backward() against its out_grad (2 TAU scale) and out_loss (1e-5) on the
    objects whose decisions agree, and against float64 under the ops' own decisions (TAU scale) everywhere."""
    batches = [("ragged", _ragged_tracks(api)), ("edge", _edge_tracks())]
    if representation == "super_quadric":
        batches += [("V1500", _long_tracks(api, 1500)), ("V2500", _long_tracks(api, 2500))]
    for name, tr in batches:
        for prior in (api.prior_table(), None):
            _vs_fused(api, AG, tr, prior, representation, f"{name} {representation} prior={prior is not None}")


def test_surface_vjp_vs_float64(api, AG):
    """surface_points backward for seeded random upstream gradients within TAU * scale of float64 (surface_vjp64) under
    the kernel's own sample angles: ragged batch, edge objects, config 2."""
    torch = _torch()
    rng = np.random.default_rng(3)
    for label, tr in (("ragged", _ragged_tracks(api)), ("edge", _edge_tracks()), ("config 2", _config2(api))):
        G = rng.normal(size=(tr.n, 1000, 3)).astype(np.float32)
        p = torch.from_numpy(tr.init).cuda().requires_grad_(True)
        (AG.surface_points(p) * torch.from_numpy(G).cuda()).sum().backward()
        g = p.grad.cpu().numpy()
        o = api.optimize_host(tr, n_iters=1, extras=("out_grids", "out_eta_idx"))
        worst = np.zeros(9)
        for i in range(tr.n):
            etas, omegas = G64.angles(o["out_grids"][i], o["out_eta_idx"][i])
            g64, sc = surface_vjp64(tr.init[i], etas, omegas, G[i])
            r = G64.ratio(g[i], g64, sc)
            assert (r <= TAU).all(), (label, i, r)
            worst = np.maximum(worst, r)
        print(f"  surface VJP {label}: worst |g - g64| / scale " + " ".join(f"{x:.1e}" for x in worst))


# ---------------------------------------------------------------------------------------------------------------- 4


def test_box_loss_vs_reference_records(api, AG, golden_runs, golden_wide):
    """Every recorded reference state: box_loss within 1e-5 of the recorded loss; on the states whose decisions (eta
    buckets, arg, residual signs) agree with the reference's, the gradient within 2 TAU scale of the recorded one."""
    torch = _torch()
    tau = 2 * TAU
    steps = agree = fused_agree = 0
    worst, worst_l = np.zeros(9), 0.0
    for case in all_cases(golden_runs) + wide_cases(golden_wide):
        P = case.states_before()[0]
        tr = case.tracks(P)
        prior = case.prior_table
        o = api.optimize_host(tr, prior=prior, n_iters=1, representation=case.repr, s0=np.tile(case.init[4:7], (len(P), 1)),
                              extras=("out_arg", "out_pred", "out_eta_idx", "out_grids"))
        d = _dev(tr, prior=prior)
        d["s0"] = torch.from_numpy(np.tile(case.init[4:7], (len(P), 1)).astype(np.float32)).cuda()
        pred, arg, loss, g = _grads(AG, d, prior)
        live = case.mask.astype(bool)
        nc = 9 if case.repr == "super_quadric" else 7
        V = case.V
        for s in range(case.iters):
            steps += 1
            label = (getattr(case, "name", case.k), s)
            rl = 0.0 if loss[s] == case.loss[s] == 0 else float(rel_loss(loss[s], case.loss[s]))
            assert rl <= TOL_LOSS, (label, loss[s], case.loss[s])
            worst_l = max(worst_l, rl)
            a, p_ = arg[s * V:(s + 1) * V], pred[s * V:(s + 1) * V]
            fa, fp = o["out_arg"][s * V:(s + 1) * V], o["out_pred"][s * V:(s + 1) * V]
            eta_ok = np.array_equal(case.eta_idx[s], o["out_eta_idx"][s])
            fused_agree += (eta_ok and np.array_equal(case.arg[s][live], fa[live])
                            and np.array_equal(case.resid_sign[s][live], np.sign(fp - case.box)[live]))
            if not (eta_ok and np.array_equal(case.arg[s][live], a[live])
                    and np.array_equal(case.resid_sign[s][live], np.sign(p_ - case.box)[live])):
                continue
            agree += 1
            etas, omegas = G64.angles(o["out_grids"][s], o["out_eta_idx"][s])
            _, sc = G64.grad64(P[s], case.Ms, case.box, case.mask, etas, omegas, a, np.sign(p_ - case.box), case.prior33,
                               case.init[4:7], case.repr == "super_quadric")
            r = G64.ratio(g[s][:nc], case.grad[s][:nc].astype(np.float64), sc[:nc])
            assert (r <= tau).all(), (label, r)
            worst[:nc] = np.maximum(worst[:nc], r)
    print(f"  reference records: {steps} states; decisions agree with the reference's on {agree} (ops) and "
          f"{fused_agree} (fused kernel); worst loss rel err {worst_l:.1e}; worst |g - g_ref| / scale "
          + " ".join(f"{x:.1e}" for x in worst))
    assert agree >= 0.95 * steps


# ---------------------------------------------------------------------------------------------------------------- 5


def test_torch_optim_adam_loop_matches_fused(api, AG):
    """20 iterations of torch.optim.Adam with the reference's two parameter groups (lr 0.01 for translation, yaw and
    scales, 0.1 for the shapes; sq_libs.py:373-380) through box_loss with the prior, on a few config-2 objects.  At every
    state the fused kernel is teacher-forced for one step from the optimiser's own m, v and step count: on the steps
    whose decisions agree, parameters within 1e-4 (floor 1e-3) and loss within 1e-5."""
    torch = _torch()
    tr = _config2(api).slice(0, 6)
    prior = api.prior_table()
    d = _dev(tr, prior=prior)
    lin = d["params"][:, :7].clone().requires_grad_(True)
    shp = d["params"][:, 7:9].clone().requires_grad_(True)
    opt = torch.optim.Adam([{"params": [lin]}, {"params": [shp], "lr": 0.1}], lr=0.01)
    s0 = tr.init[:, 4:7].copy()
    checked = total = 0
    worst_p = worst_l = 0.0
    for it in range(20):
        state = torch.cat([lin, shp], 1).detach().cpu().numpy()
        st = lambda key: (np.zeros((tr.n, 9), np.float32) if not opt.state else
                          torch.cat([opt.state[lin][key], opt.state[shp][key]], 1).cpu().numpy())
        from odam_b200.api import PackedTracks
        ft = PackedTracks(state, tr.cls, tr.view_off, tr.Ms, tr.box, tr.mask)
        o = api.optimize_host(ft, prior=prior, n_iters=1, m0=st("exp_avg"), v0=st("exp_avg_sq"), step0=it, s0=s0,
                              extras=("out_arg",))
        opt.zero_grad()
        params = torch.cat([lin, shp], 1)
        loss = AG.box_loss(params, d["view_off"], d["Ms"], d["box"], d["mask"], prior=d["prior"], cls=d["cls"], s0=d["s0"])
        _, arg = AG.box_sides(params.detach(), d["view_off"], d["Ms"])
        loss.sum().backward()
        opt.step()
        after = torch.cat([lin, shp], 1).detach().cpu().numpy()
        loss, arg = loss.detach().cpu().numpy(), arg.cpu().numpy()
        for i in range(tr.n):
            a, b = int(tr.view_off[i]), int(tr.view_off[i + 1])
            total += 1
            if not np.array_equal(arg[a:b], o["out_arg"][a:b]):
                continue
            checked += 1
            rp = float(rel_param(after[i], o["params"][i]).max())
            rl = float(rel_loss(loss[i], o["loss"][i, 0]))
            assert rp <= TOL_PARAM and rl <= TOL_LOSS, (it, i, rp, rl)
            worst_p, worst_l = max(worst_p, rp), max(worst_l, rl)
    print(f"  torch.optim.Adam loop: {total} object-steps, {checked} with the fused kernel's decisions; worst rel err "
          f"params {worst_p:.1e} (floor {FLOOR}), loss {worst_l:.1e}")
    assert checked >= 0.8 * total


# ---------------------------------------------------------------------------------------------------------------- 6


def test_deterministic_and_batch_independent(api, AG):
    """Gradients bit-identical run to run, and for an object alone or inside a 500-object batch; device-resident
    view_off gives the same results as a host copy."""
    torch = _torch()
    from odam_b200 import synthetic
    from odam_b200.api import PackedTracks
    tr = _ragged_tracks(api)
    G = np.random.default_rng(5).normal(size=(tr.n, 1000, 3)).astype(np.float32)
    prior = api.prior_table()
    d = _dev(tr, prior=prior)
    r1, r2 = _grads(AG, d, prior, G), _grads(AG, d, prior, G)
    for x, y in zip(r1, r2):
        assert np.array_equal(x, y)
    d["view_off"] = d["view_off"].cuda()
    for x, y in zip(r1, _grads(AG, d, prior, G)):
        assert np.array_equal(x, y)
    big = api.pack_scene(synthetic.make_scene(500, 20, seed=9))
    at = 123
    for i in (0, 5):   # one view and 300 views
        a, b = int(tr.view_off[i]), int(tr.view_off[i + 1])
        alone = PackedTracks(tr.init[i:i + 1], tr.cls[i:i + 1], np.array([0, b - a], np.int32), tr.Ms[a:b], tr.box[a:b],
                             tr.mask[a:b])
        lo, hi = big.slice(0, at), big.slice(at, 500)
        voff = np.concatenate([lo.view_off, lo.total_views + b - a + hi.view_off]).astype(np.int32)
        batch = PackedTracks(np.concatenate([lo.init, alone.init, hi.init]), np.concatenate([lo.cls, alone.cls, hi.cls]),
                             voff, np.concatenate([lo.Ms, alone.Ms, hi.Ms]), np.concatenate([lo.box, alone.box, hi.box]),
                             np.concatenate([lo.mask, alone.mask, hi.mask]))
        Gb = np.random.default_rng(6).normal(size=(501, 1000, 3)).astype(np.float32)
        Gb[at] = G[i]
        ra = _grads(AG, _dev(alone, prior=prior), prior, G[i:i + 1])
        rb = _grads(AG, _dev(batch, prior=prior), prior, Gb)
        v0 = int(batch.view_off[at])
        assert np.array_equal(ra[0], rb[0][v0:v0 + b - a]) and np.array_equal(ra[1], rb[1][v0:v0 + b - a]), i
        assert np.array_equal(ra[3][0], rb[3][at]), (i, "box_loss gradient")
        assert np.array_equal(ra[4][0], rb[4][at]), (i, "surface gradient")
    print("  gradients bit-identical run to run, with device view_off, and alone vs in a 501-object batch")


def test_streams_empty_accumulation_and_errors(api, AG):
    """A non-default stream gives the default stream's results; n = 0 works; surface_points and box_loss in one loss
    accumulate into one params.grad; Ms gets no gradient; bad arguments raise ValueError."""
    torch = _torch()
    tr = _ragged_tracks(api)
    prior = api.prior_table()
    G = np.random.default_rng(8).normal(size=(tr.n, 1000, 3)).astype(np.float32)
    d = _dev(tr, prior=prior)
    ref = _grads(AG, d, prior, G)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        other = _grads(AG, d, prior, G)
    for x, y in zip(ref, other):
        assert np.array_equal(x, y)
    # n = 0
    p0 = torch.zeros((0, 9), device="cuda", requires_grad=True)
    v0 = torch.zeros(1, dtype=torch.int32)
    M0 = torch.zeros((0, 12), device="cuda")
    assert tuple(AG.surface_points(p0).shape) == (0, 1000, 3)
    pred0, arg0 = AG.box_sides(p0, v0, M0)
    assert tuple(pred0.shape) == (0, 4) and tuple(arg0.shape) == (0, 4)
    l0 = AG.box_loss(p0, v0, M0, torch.zeros((0, 4), device="cuda"), torch.zeros((0, 4), device="cuda"))
    (l0.sum() + AG.surface_points(p0).sum()).backward()
    assert tuple(p0.grad.shape) == (0, 9)
    # one params.grad from both ops; Ms is a constant
    p = d["params"].clone().requires_grad_(True)
    Ms = d["Ms"].clone().requires_grad_(True)
    loss = (AG.surface_points(p) * torch.from_numpy(G).cuda()).sum() + \
        AG.box_loss(p, d["view_off"], Ms, d["box"], d["mask"], prior=d["prior"], cls=d["cls"], s0=d["s0"]).sum()
    loss.backward()
    assert Ms.grad is None
    assert np.array_equal(p.grad.cpu().numpy(), ref[3] + ref[4])
    # errors
    bad = d["view_off"].clone()
    bad[-1] += 1
    with pytest.raises(ValueError):
        AG.box_sides(d["params"], bad, d["Ms"])
    with pytest.raises(ValueError):
        AG.box_sides(d["params"], d["view_off"], d["Ms"][:-1])
    with pytest.raises(ValueError):
        AG.box_sides(d["params"].cpu(), d["view_off"], d["Ms"])
    with pytest.raises(ValueError):
        AG.box_sides(d["params"], d["view_off"], d["Ms"].cpu())
    with pytest.raises(ValueError):
        AG.surface_points(d["params"].double())
    with pytest.raises(ValueError):
        AG.box_loss(d["params"], d["view_off"], d["Ms"], d["box"], d["mask"], prior=d["prior"])
    with pytest.raises(ValueError):
        AG.box_loss(d["params"], d["view_off"], d["Ms"], d["box"].cpu(), d["mask"])
    if torch.cuda.device_count() > 1:
        d1 = _dev(tr, "cuda:1", prior)
        with pytest.raises(ValueError):
            AG.box_sides(d["params"], d["view_off"], d1["Ms"])
        other = _grads(AG, d1, prior, G)
        for x, y in zip(ref, other):
            assert np.array_equal(x, y)
        print("  cuda:1 gives cuda:0's results")
    print("  streams, n = 0, accumulation, Ms.grad is None and argument errors: ok")
