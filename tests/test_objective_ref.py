"""CPU tests of the optimiser's opt-in objective (odam_sq_objective: per-side weights, robust residual losses, a
learning-rate schedule), without a GPU.

- The float64 restatement of its gradient (tests/objective64.py) against central differences of its loss, for each
  loss kind, with random weights that include zeros.
- The three residual losses against torch's smooth_l1_loss and the formulas of include/odam_sq.h.
- Argument validation of odam_sq_optimize_objective[_host] (ODAM_SQ_ERR_ARG before any CUDA call) and of the Python
  keywords of api.optimize_host.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import objective64 as O64
from golden_cases import edge_object
from oracle import c_oracle
from oracle import grad64 as G64

KINDS = ("l1", "smooth_l1", "cauchy")
ERR_ARG = -1
p = C.c_void_p(16)


def _ae32(p9):
    """(a, e) of a parameter row in float32 (a = s^2, e = 0.2 + 1.4 sigmoid(h))."""
    p9 = np.asarray(p9, np.float32)
    sig = (1 / (1 + np.exp(-p9[7:9].astype(np.float64)))).astype(np.float32)
    return p9[4:7] * p9[4:7], sig * np.float32(1.4) + np.float32(0.2)


def _decisions(init, Ms, box):
    """Sample angles of init, the float64 arg-extreme valid sample of every (view, side) and the residual signs."""
    smp = c_oracle.sample(*_ae32(init))
    u, w, valid = G64.project(init, smp["etas"], smp["omegas"], Ms)
    arg = np.full((len(Ms), 4), -1, np.int64)
    for sd in range(4):
        c = u if sd < 2 else w
        big = np.where(valid, c, np.inf if sd % 2 == 0 else -np.inf)
        idx = big.argmin(1) if sd % 2 == 0 else big.argmax(1)
        arg[:, sd] = np.where(valid.any(1), idx, -1)
    uv = O64.arg_uv(init, Ms, smp["etas"], smp["omegas"], arg)
    return smp["etas"], smp["omegas"], arg, np.sign(uv - box)


@pytest.mark.parametrize("loss", KINDS)
def test_grad64_against_central_differences(loss):
    """Edge objects, random weights with a quarter of them zero: the restated gradient equals central differences of
    the float64 loss with the decisions held, within 1e-6 of the conditioning scale.  The same comparison with the
    weights left out of the gradient fails, so the weights are really in it."""
    c_oracle.build()
    rng = np.random.default_rng(KINDS.index(loss))
    worst = 0.0
    for kind in ("plain", "h+6", "h-6", "yaw+pi/2", "behind", "V1"):
        init, Ms, box, mask, _ = edge_object(kind)
        etas, omegas, arg, sign = _decisions(init, Ms, box)
        weight = rng.uniform(0, 2, size=box.shape).astype(np.float32) * (rng.uniform(size=box.shape) > 0.25)
        r = np.abs(O64.arg_uv(init, Ms, etas, omegas, arg) - box)
        scale = float(np.median(r[np.isfinite(r) & (mask != 0)])) if loss != "l1" else None
        g, sc = O64.grad64(init, Ms, box, mask, etas, omegas, arg, sign, weight=weight, loss=loss, loss_scale=scale)
        p0 = np.asarray(init, np.float32).astype(np.float64)
        fd = np.zeros(9)
        for k in range(9):
            h = 1e-6 * max(1.0, abs(p0[k]))
            e = np.zeros(9)
            e[k] = h
            fd[k] = (O64.loss64(p0 + e, Ms, box, mask, etas, omegas, arg, weight, loss, scale) -
                     O64.loss64(p0 - e, Ms, box, mask, etas, omegas, arg, weight, loss, scale)) / (2 * h)
        err = np.abs(g - fd) / np.maximum(sc, 1e-12)
        assert (err <= 1e-6).all(), (kind, loss, err, g, fd)
        worst = max(worst, float(err.max()))
        if (weight[mask != 0] != 1).any() and sc.max() > 0:
            g1, _ = O64.grad64(init, Ms, box, mask, etas, omegas, arg, sign, loss=loss, loss_scale=scale)
            assert (np.abs(g1 - fd) / np.maximum(sc, 1e-12)).max() > 1e-3, (kind, loss)
    print(f"  {loss}: worst |g64 - central difference| / scale {worst:.1e}")


def test_grad64_defaults_are_grad64():
    """With no weight and L1 the extended restatement returns grad64's result bit for bit; all-one weights agree."""
    c_oracle.build()
    init, Ms, box, mask, _ = edge_object("plain")
    etas, omegas, arg, sign = _decisions(init, Ms, box)
    g0, s0 = G64.grad64(init, Ms, box, mask, etas, omegas, arg, sign)
    g1, s1 = O64.grad64(init, Ms, box, mask, etas, omegas, arg, sign)
    assert np.array_equal(g0, g1) and np.array_equal(s0, s1)
    g2, s2 = O64.grad64(init, Ms, box, mask, etas, omegas, arg, sign, weight=np.ones_like(box))
    assert np.array_equal(g0, g2) and np.array_equal(s0, s2)


@pytest.mark.parametrize("scale", [0.5, 3.0, 40.0])
def test_residual_losses(scale):
    """rho and rho' of each kind: smooth_l1 against torch.nn.functional.smooth_l1_loss (value and autograd derivative),
    Cauchy against 0.5 c^2 log1p((r/c)^2) and r / (1 + (r/c)^2) under autograd, L1 against |r|."""
    r = np.concatenate([np.linspace(-100, 100, 401), [0.0, scale, -scale, np.nextafter(scale, 0), 1e6, -1e6]])
    t = torch.tensor(r, dtype=torch.float64, requires_grad=True)
    ref = torch.nn.functional.smooth_l1_loss(t, torch.zeros_like(t), reduction="none", beta=scale)
    d, = torch.autograd.grad(ref.sum(), t)
    v, dv = O64.rho64(r, "smooth_l1", scale)
    np.testing.assert_allclose(v, ref.detach().numpy(), rtol=1e-15, atol=0)
    np.testing.assert_allclose(dv, d.numpy(), rtol=1e-15, atol=0)
    ref = 0.5 * scale ** 2 * torch.log1p((t / scale) ** 2)
    d, = torch.autograd.grad(ref.sum(), t)
    v, dv = O64.rho64(r, "cauchy", scale)
    np.testing.assert_allclose(v, ref.detach().numpy(), rtol=1e-14, atol=0)
    np.testing.assert_allclose(dv, d.numpy(), rtol=1e-14, atol=1e-300)
    v, dv = O64.rho64(r, "l1", scale)
    assert np.array_equal(v, np.abs(r)) and np.array_equal(dv, np.sign(r))


# ---------------------------------------------------------------------------------------------- argument validation


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import _lib, build
    build.build()
    return _lib.load()


def _obj(side_weight=None, loss=0, loss_scale=0.0, lr_scale=None):
    from odam_b200 import _lib
    o = _lib.Objective()
    o.side_weight, o.loss, o.loss_scale, o.lr_scale = side_weight, loss, loss_scale, lr_scale
    return o


def test_objective_entries(lib):
    """Both objective entries reject, before any CUDA call: an unknown loss, a robust kind without a finite scale > 0,
    a negative or non-finite schedule entry, and the cycle counts with the weighted/robust build; the host entry also a
    negative or non-finite weight.  n == 0 stays a no-op, and the checks of odam_sq_optimize still apply."""
    from odam_b200 import _lib
    voff = np.array([0, 2, 5], np.int32)
    host = lambda a: a.ctypes.data_as(C.c_void_p)
    cyc = _lib.Options()
    cyc.out_cycles = p
    for f, last in ((lib.odam_sq_optimize_objective, None), (lib.odam_sq_optimize_objective_host, 0)):
        def call(obj, opt=None, n=2, n_iters=3, init=p):
            return f(init, None, host(voff), p, p, p, None, n, n_iters, 0, 0.01, 0.1, p, p, None,
                     None if obj is None else C.byref(obj), None if opt is None else C.byref(opt), last)
        for loss in (-1, 3):
            assert call(_obj(loss=loss)) == ERR_ARG, loss
        for kind in (1, 2):
            for bad in (0.0, -1.0, float("nan"), float("inf")):
                assert call(_obj(loss=kind, loss_scale=bad)) == ERR_ARG, (kind, bad)
        for bad in (-0.5, float("nan"), float("inf")):
            sched = np.array([1.0, bad, 1.0], np.float32)
            assert call(_obj(lr_scale=host(sched))) == ERR_ARG, bad
        assert call(_obj(side_weight=p), cyc) == ERR_ARG
        assert call(_obj(loss=2, loss_scale=1.0), cyc) == ERR_ARG
        assert call(_obj(loss=9), init=None) == ERR_ARG
        assert call(_obj(loss=2, loss_scale=1.0), n=0) == 0
        assert call(None, n=0) == 0
    f = lib.odam_sq_optimize_objective_host
    for bad in (-1.0, float("nan"), float("inf"), -float("inf")):
        w = np.ones((5, 4), np.float32)
        w[3, 2] = bad
        assert f(p, None, host(voff), p, p, p, None, 2, 1, 0, 0.01, 0.1, p, p, None, C.byref(_obj(side_weight=host(w))),
                 None, 0) == ERR_ARG, bad


def test_python_keywords(lib):
    """api.optimize_host's objective keywords: names, shapes and a missing scale are ValueErrors; values the library
    rejects raise its OdamSqError.  None of these reaches the GPU."""
    from odam_b200 import api, _lib
    from launch_checks import pack
    tr = pack([edge_object("plain"), edge_object("V1")])
    SV = tr.total_views
    bad_value = [dict(loss="huber", loss_scale=1.0), dict(loss="cauchy"), dict(loss="smooth_l1"),
                 dict(side_weight=np.ones((SV + 1, 4))), dict(side_weight=np.ones(SV)), dict(lr_scale=np.ones(2))]
    for kw in bad_value:
        with pytest.raises(ValueError):
            api.optimize_host(tr, n_iters=3, **kw)
    w = np.ones((SV, 4), np.float32)
    w[0, 0] = -1
    rejected = [dict(side_weight=w), dict(loss="cauchy", loss_scale=0.0), dict(loss="smooth_l1", loss_scale=float("nan")),
                dict(lr_scale=[1, float("inf"), 1]), dict(lr_scale=[1, -1, 1])]
    for kw in rejected:
        with pytest.raises(_lib.OdamSqError, match="invalid argument"):
            api.optimize_host(tr, n_iters=3, **kw)
