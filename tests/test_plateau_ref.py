"""CPU tests of the fused optimiser's opt-in step reduction on a plateau (odam_sq_plateau), without a GPU.

- The float32 restatement of the rule (tests/plateau_rule.py) on hand-built loss curves with known
  answers, and against stop_rule when no reduction is allowed.
- The schedule an object ran under (lr_scale_seen), which the GPU tests replay.
- Argument validation of odam_sq_optimize_plateau[_host] (ODAM_SQ_ERR_ARG before any CUDA call) and of the Python
  keywords max_reductions and lr_factor of api.optimize_host and api.optimize_device.
"""
import ctypes as C

import numpy as np
import pytest

from convergence_rule import stop_rule
from plateau_rule import lr_scale_seen, plateau_rule
from golden_cases import edge_object

ERR_ARG = -1
p = C.c_void_p(16)
nan, inf = float("nan"), float("inf")


# ------------------------------------------------------------------------------------------------ the rule itself


def test_reduction_then_stop():
    """A constant curve: the patience runs out at `patience`, the window restarts there, and after R reductions the
    run stops; the best stays the first loss."""
    assert plateau_rule(np.full(100, 3.0), 5, 1e-3, 1) == (11, 0, [6])
    assert plateau_rule(np.full(100, 3.0), 5, 1e-3, 2) == (16, 0, [6, 11])
    assert plateau_rule(np.full(100, 3.0), 1, 0.0, 3) == (5, 0, [2, 3, 4])
    # R reductions that never all happen: the unused ones are -1
    assert plateau_rule(np.full(12, 3.0), 5, 1e-3, 3) == (12, 0, [6, 11, -1])


def test_window_restarts_after_a_reduction():
    """The window after a reduction counts from the reduction's iteration, and an improvement inside it restarts it
    again; best is not reset by a reduction."""
    loss = [5.0, 4.0, 4.0, 4.0, 3.0, 3.0, 3.0, 3.0, 3.0, 3.0]
    # patience 2: out at k=3 (last=1) -> reduce, last=3; k=4 improves -> last=4; out at k=6 -> reduce, last=6;
    # out at k=8 -> stop
    assert plateau_rule(loss, 2, 0.0, 2) == (9, 4, [4, 7])
    assert plateau_rule(loss, 2, 0.0, 1) == (7, 4, [4])
    # a loss after the reduction that ties the best (not below it) is no improvement
    assert plateau_rule([2.0, 3.0, 3.0, 2.0, 2.0, 2.0], 2, 0.0, 1) == (5, 0, [3])


def test_nan_losses():
    """Non-finite losses are neither improvements nor bests and count towards the patience, before and after a
    reduction."""
    assert plateau_rule([nan] * 10, 2, 0.0, 2) == (7, -1, [3, 5])
    assert plateau_rule([4.0, nan, nan, 3.0, nan, nan, nan, nan], 2, 0.0, 1) == (6, 3, [3])
    assert plateau_rule([4.0, -inf, inf, nan, 3.5, nan, nan], 2, 0.0, 1) == (7, 4, [3])


def test_reduction_at_the_last_iteration():
    """A reduction decided at the last iteration is reported with reduce_iter = n_iters, a level no iteration ran."""
    assert plateau_rule(np.full(6, 3.0), 5, 1e-3, 2) == (6, 0, [6, -1])
    s = lr_scale_seen([6, -1], 0.5, 6)
    assert np.array_equal(s, np.ones(6, np.float32))


def test_no_reduction_is_the_stop_rule():
    rng = np.random.default_rng(0)
    curves = [np.full(40, 3.0), 10.0 * 0.99 ** np.arange(60), [nan, 4.0, nan, 3.0, nan, nan, nan],
              [5.0, 4.0, 3.0, 3.0, 3.0, 3.0, 3.0]]
    curves += [np.minimum.accumulate(rng.uniform(1, 2, 80)) + rng.normal(0, 1e-3, 80) for _ in range(20)]
    for loss in curves:
        for patience, rel_tol in ((1, 0.0), (3, 1e-3), (10, 1e-2), (0, 0.0)):
            iters, b, red = plateau_rule(loss, patience, rel_tol, 0)
            assert (iters, b) == stop_rule(loss, patience, rel_tol)
            assert red == []
    # and reductions only ever lengthen a run, at the same iterations up to the first one
    for loss in curves[4:]:
        i0, b0 = stop_rule(loss, 5, 1e-3)
        i1, b1, red = plateau_rule(loss, 5, 1e-3, 2)
        assert i1 >= i0 and (red[0] == -1 or red[0] == i0)


def test_schedule_seen():
    """lr_scale_seen: f_r = (float)factor^r, times lr_scale in float32, from each reduce_iter on."""
    s = lr_scale_seen([3, 5], 0.3, 7)
    f1, f2 = np.float32(float(np.float32(0.3))), np.float32(float(np.float32(0.3)) ** 2)
    assert np.array_equal(s, np.array([1, 1, 1, f1, f1, f2, f2], np.float32))
    base = np.linspace(1, 0.1, 7).astype(np.float32)
    s = lr_scale_seen([2, -1], 0.5, 7, base)
    assert np.array_equal(s[:2], base[:2]) and np.array_equal(s[2:], base[2:] * np.float32(0.5))
    assert s.dtype == np.float32


# ---------------------------------------------------------------------------------------------- argument validation


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import _lib, build
    build.build()
    return _lib.load()


def _conv(patience=10, rel_tol=1e-3):
    from odam_b200 import _lib
    c = _lib.Convergence()
    c.patience, c.rel_tol = patience, rel_tol
    return c


def _plat(max_reductions=2, factor=0.3):
    from odam_b200 import _lib
    pl = _lib.Plateau()
    pl.max_reductions, pl.factor = max_reductions, factor
    return pl


def test_plateau_entries(lib):
    """Both entries reject, before any CUDA call: plat without conv or with patience 0, max_reductions outside 1 .. 8,
    and a factor that is not finite or outside (0, 1).  The checks of the convergence entry still apply, plat == NULL
    is that entry, and n == 0 stays a no-op."""
    from odam_b200 import _lib
    voff = np.array([0, 2, 5], np.int32)
    host = lambda a: a.ctypes.data_as(C.c_void_p)
    ref = lambda x: None if x is None else C.byref(x)
    for f, last in ((lib.odam_sq_optimize_plateau, None), (lib.odam_sq_optimize_plateau_host, 0)):
        def call(plat, conv="default", opt=None, obj=None, n=2, init=p):
            conv = _conv() if conv == "default" else conv
            return f(init, None, host(voff), p, p, p, None, n, 3, 0, 0.01, 0.1, p, p, None, ref(obj), ref(conv),
                     ref(plat), ref(opt), last)
        bad = [dict(max_reductions=0), dict(max_reductions=-1), dict(max_reductions=9), dict(factor=0.0),
               dict(factor=1.0), dict(factor=1.5), dict(factor=-0.5), dict(factor=nan), dict(factor=inf),
               dict(factor=-inf)]
        for kw in bad:
            assert call(_plat(**kw)) == ERR_ARG, kw
            assert call(_plat(**kw), n=0) == ERR_ARG, kw
        assert call(_plat(), conv=None) == ERR_ARG
        assert call(_plat(), conv=None, n=0) == ERR_ARG
        assert call(_plat(), conv=_conv(patience=0)) == ERR_ARG
        assert call(_plat(), conv=_conv(patience=0), n=0) == ERR_ARG
        # the convergence entry's own checks, with and without plat
        for conv in (_conv(patience=-1), _conv(rel_tol=1.0), _conv(rel_tol=nan)):
            assert call(_plat(), conv=conv) == ERR_ARG
            assert call(None, conv=conv) == ERR_ARG
        for name in ("out_pred", "out_arg", "out_eta_idx", "out_grids", "out_cycles"):
            o = _lib.Options()
            setattr(o, name, p)
            assert call(_plat(), opt=o) == ERR_ARG, name
        obj = _lib.Objective()
        obj.loss = 7
        assert call(_plat(), obj=obj) == ERR_ARG
        assert call(_plat(), init=None) == ERR_ARG
        # valid arguments, nothing to run
        assert call(_plat(1, 1e-6), n=0) == 0
        assert call(_plat(8, np.nextafter(np.float32(1), np.float32(0))), n=0) == 0
        assert call(None, n=0) == 0
        assert call(None, conv=None, n=0) == 0


def test_python_keywords(lib):
    """api.optimize_host and optimize_device: max_reductions > 0 needs patience > 0 and an lr_factor in (0, 1), an
    lr_factor needs max_reductions > 0, and each bad value is a ValueError before the library is called."""
    from odam_b200 import api
    from launch_checks import pack
    tr = pack([edge_object("plain"), edge_object("V1")])
    rule = dict(patience=10, rel_tol=1e-3)
    bad = [dict(max_reductions=2, lr_factor=0.3),                       # no patience
           dict(max_reductions=2, lr_factor=0.3, rel_tol=1e-3, keep_best=True),
           dict(rule, max_reductions=2),                                # no lr_factor
           dict(rule, lr_factor=0.3),                                   # no max_reductions
           dict(lr_factor=0.3),
           dict(rule, max_reductions=9, lr_factor=0.3), dict(rule, max_reductions=-1, lr_factor=0.3),
           dict(rule, max_reductions=1.0, lr_factor=0.3), dict(rule, max_reductions=True, lr_factor=0.3),
           dict(rule, max_reductions=2, lr_factor=0.0), dict(rule, max_reductions=2, lr_factor=1.0),
           dict(rule, max_reductions=2, lr_factor=1 - 1e-9),              # 1.0 in float32
           dict(rule, max_reductions=2, lr_factor=1e-50),                 # 0.0 in float32
           dict(rule, max_reductions=2, lr_factor=-0.3), dict(rule, max_reductions=2, lr_factor=nan),
           dict(rule, max_reductions=2, lr_factor=inf), dict(rule, max_reductions=2, lr_factor="0.3"),
           dict(rule, max_reductions=2, lr_factor=True)]
    for kw in bad:
        with pytest.raises(ValueError):
            api.optimize_host(tr, n_iters=3, **kw)
        with pytest.raises(ValueError):
            api.optimize_device(object(), n_iters=3, **kw)   # rejected before the tracks are looked at
    with pytest.raises(ValueError, match="out_grids"):
        api.optimize_host(tr, n_iters=3, **rule, max_reductions=2, lr_factor=0.3, extras=("out_grids",))
