"""CPU tests of the fused optimiser's opt-in early stopping (odam_sq_convergence), without a GPU.

- The float32 restatement of the rule (tests/convergence_rule.py) on hand-built loss curves with known answers.
- Argument validation of odam_sq_optimize_converge[_host] (ODAM_SQ_ERR_ARG before any CUDA call) and of the Python
  keywords of api.optimize_host and api.optimize_device.
"""
import ctypes as C

import numpy as np
import pytest

from convergence_rule import keep_factor, stop_rule
from golden_cases import edge_object

ERR_ARG = -1
p = C.c_void_p(16)
nan, inf = float("nan"), float("inf")


# ------------------------------------------------------------------------------------------------ the rule itself


def test_constant_curve():
    """No iteration after the first improves: the run stops after patience + 1 iterations, best at 0."""
    for patience in (1, 5, 20):
        assert stop_rule(np.full(100, 3.0), patience, 1e-3) == (patience + 1, 0)
    assert stop_rule(np.full(10, 3.0), 20, 1e-3) == (10, 0)   # patience never runs out


def test_strictly_decreasing_curve():
    """Every step improves by 1 %: with rel_tol below that the run never stops and the best is the last; with rel_tol
    above it no step is significant, but the best still follows the lowest loss."""
    loss = 10.0 * 0.99 ** np.arange(60)
    assert stop_rule(loss, 5, 1e-3) == (60, 59)
    assert stop_rule(loss, 5, 0.0) == (60, 59)
    assert stop_rule(loss, 5, 2e-2) == (6, 5)


def test_ties_keep_the_first_index():
    loss = [5.0, 4.0, 3.0, 3.0, 3.0, 3.0, 3.0]
    assert stop_rule(loss, 0, 0.0) == (7, 2)
    assert stop_rule(loss, 2, 0.0) == (5, 2)   # a tie is no improvement
    assert stop_rule([2.0, 1.0, 3.0, 1.0, 1.0], 0, 0.0) == (5, 1)


def test_rel_tol_zero_counts_every_strict_decrease():
    one_ulp = np.nextafter(np.float32(3.0), np.float32(0))
    assert stop_rule([3.0, 3.0, one_ulp, 3.0, 3.0], 2, 0.0) == (5, 2)
    assert stop_rule([3.0, 3.0, one_ulp, 3.0, 3.0], 2, 1e-3) == (3, 2)


def test_significance_is_an_fp32_product():
    """L < best * keep with keep = (float)(1 - rel_tol) and the product rounded to float32: a loss equal to that
    product is not significant, one ulp below it is."""
    best, rel_tol = np.float32(7.3), 1e-3
    thr = np.float32(best * keep_factor(rel_tol))
    assert keep_factor(rel_tol) == np.float32(1.0 - float(np.float32(rel_tol)))
    below = np.nextafter(thr, np.float32(0))
    assert stop_rule([best, thr, thr, thr], 2, rel_tol) == (3, 1)
    assert stop_rule([best, below, thr, thr], 2, rel_tol) == (4, 1)


def test_nan_and_inf_entries():
    """Non-finite losses are neither improvements nor bests; they count towards the patience like any other
    iteration, and a run whose losses are all non-finite stops with b = -1."""
    assert stop_rule([nan, nan, nan, nan, nan], 2, 0.0) == (3, -1)
    assert stop_rule([inf, -inf, nan, inf], 0, 0.0) == (4, -1)
    assert stop_rule([nan, 4.0, nan, 3.0, nan, nan, nan], 2, 0.0) == (6, 3)
    assert stop_rule([4.0, -inf, 3.0], 0, 0.0) == (3, 2)   # -inf is not a loss below 3


def test_patience_zero_never_stops():
    for loss in (np.full(50, 1.0), [nan] * 50, 10.0 * 0.9 ** np.arange(50)):
        assert stop_rule(loss, 0, 0.5)[0] == 50
    assert stop_rule([3.0, 1.0, 2.0, 2.0], 0, 0.0) == (4, 1)


# ---------------------------------------------------------------------------------------------- argument validation


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import _lib, build
    build.build()
    return _lib.load()


def _conv(patience=0, rel_tol=0.0, keep_best=0, out_iters=None, out_best_iter=None):
    from odam_b200 import _lib
    c = _lib.Convergence()
    c.patience, c.rel_tol, c.keep_best, c.out_iters, c.out_best_iter = patience, rel_tol, keep_best, out_iters, \
        out_best_iter
    return c


def test_converge_entries(lib):
    """Both entries reject, before any CUDA call: patience < 0, a rel_tol that is not finite or outside [0, 1),
    keep_best other than 0 or 1, and conv together with out_pred, out_arg, out_eta_idx, out_grids or out_cycles.  The
    checks of the objective entry still apply, and n == 0 stays a no-op."""
    from odam_b200 import _lib
    voff = np.array([0, 2, 5], np.int32)
    host = lambda a: a.ctypes.data_as(C.c_void_p)
    for f, last in ((lib.odam_sq_optimize_converge, None), (lib.odam_sq_optimize_converge_host, 0)):
        def call(conv, opt=None, obj=None, n=2, init=p):
            return f(init, None, host(voff), p, p, p, None, n, 3, 0, 0.01, 0.1, p, p, None,
                     None if obj is None else C.byref(obj), None if conv is None else C.byref(conv),
                     None if opt is None else C.byref(opt), last)
        for bad in (dict(patience=-1), dict(rel_tol=-1e-3), dict(rel_tol=1.0), dict(rel_tol=1.5), dict(rel_tol=nan),
                    dict(rel_tol=inf), dict(rel_tol=-inf), dict(keep_best=2), dict(keep_best=-1)):
            assert call(_conv(**bad)) == ERR_ARG, bad
            assert call(_conv(**bad), n=0) == ERR_ARG, bad
        for name in ("out_pred", "out_arg", "out_eta_idx", "out_grids", "out_cycles"):
            o = _lib.Options()
            setattr(o, name, p)
            assert call(_conv(patience=20, rel_tol=1e-3), o) == ERR_ARG, name
            assert call(_conv(), o) == ERR_ARG, name   # any conv, even one that never stops
        obj = _lib.Objective()
        obj.loss = 7
        assert call(_conv(patience=20), obj=obj) == ERR_ARG   # the objective's own checks
        assert call(_conv(patience=20), init=None) == ERR_ARG
        assert call(_conv(patience=20, rel_tol=1e-3, keep_best=1), n=0) == 0
        assert call(None, n=0) == 0


def test_python_keywords(lib):
    """api.optimize_host and optimize_device: each bad keyword is a ValueError before the library is called, as is
    early stopping together with an output that describes the last iteration."""
    from odam_b200 import api
    from launch_checks import pack
    tr = pack([edge_object("plain"), edge_object("V1")])
    bad = [dict(patience=-1), dict(patience=1.5), dict(patience=True), dict(patience="3"), dict(rel_tol=-0.1),
           dict(rel_tol=1.0), dict(rel_tol=nan), dict(rel_tol=inf), dict(keep_best=2), dict(keep_best="yes")]
    for kw in bad:
        with pytest.raises(ValueError):
            api.optimize_host(tr, n_iters=3, **kw)
        with pytest.raises(ValueError):
            api.optimize_device(object(), n_iters=3, **kw)   # rejected before the tracks are looked at
    for name in ("out_pred", "out_arg", "out_eta_idx", "out_grids"):
        with pytest.raises(ValueError, match=name):
            api.optimize_host(tr, n_iters=3, patience=20, rel_tol=1e-3, extras=(name,))
        with pytest.raises(ValueError, match=name):
            api.optimize_host(tr, n_iters=3, keep_best=True, extras=("out_m", name))
