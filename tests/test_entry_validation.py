"""CPU tests of the C entries' argument validation: NULL pointers, negative sizes and out-of-range arguments give
ODAM_SQ_ERR_ARG, and n == 0 is a no-op, all before any CUDA call, so they run without a GPU.  The dummy pointers are
never dereferenced; host arrays that the entries read (view offsets, classes) are real.  The entries of the
differentiable ops are covered in tests/test_autograd_ref.py."""
import ctypes as C

import numpy as np
import pytest

ERR_ARG = -1
p = C.c_void_p(16)


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import _lib, build
    build.build()
    return _lib.load()


def host(a):
    return a.ctypes.data_as(C.c_void_p)


def nulled(k, count):
    a = [p] * count
    a[k] = None
    return a


def test_sample_points(lib):
    for f, last in ((lib.odam_sq_sample_points, None), (lib.odam_sq_sample_points_host, 0)):
        assert f(None, 1, p, last) == ERR_ARG
        assert f(p, 1, None, last) == ERR_ARG
        assert f(p, -1, p, last) == ERR_ARG
        assert f(p, 0, p, last) == 0


def test_project_boxes(lib):
    for f, last in ((lib.odam_sq_project_boxes, None), (lib.odam_sq_project_boxes_host, 0)):
        for k in range(4):
            a = nulled(k, 4)
            assert f(a[0], a[1], a[2], 1, a[3], last) == ERR_ARG, k
        assert f(p, p, p, -1, p, last) == ERR_ARG
        assert f(p, p, p, 0, p, last) == 0
    # host view offsets index the staged camera matrices: they start at 0 and never decrease
    for bad in ([0, -4], [1, 5], [0, 5, 3]):
        voff = np.array(bad, np.int32)
        assert lib.odam_sq_project_boxes_host(p, host(voff), p, len(bad) - 1, p, 0) == ERR_ARG, bad


def test_oriented_boxes(lib):
    for f, last in ((lib.odam_sq_oriented_boxes, None), (lib.odam_sq_oriented_boxes_host, 0)):
        assert f(None, 1, p, p, p, last) == ERR_ARG
        assert f(p, 1, None, p, p, last) == ERR_ARG
        assert f(p, -1, p, p, p, last) == ERR_ARG
        assert f(p, 0, p, None, None, last) == 0   # flags and points are optional
    f = lib.odam_sq_oriented_boxes_of_points_host
    assert f(None, 1, 8, p, p, 0) == ERR_ARG
    assert f(p, 1, 8, None, p, 0) == ERR_ARG
    assert f(p, -1, 8, p, p, 0) == ERR_ARG
    assert f(p, 1, 0, p, p, 0) == ERR_ARG
    assert f(p, 1, 1025, p, p, 0) == ERR_ARG   # at most 1024 points per set
    assert f(p, 0, 8, p, None, 0) == 0


def test_merge_cost(lib):
    f = lib.odam_sq_merge_cost_host
    assert f(None, p, 2, p, p, p, 0) == ERR_ARG
    assert f(p, p, 2, None, None, None, 0) == ERR_ARG   # no output asked for
    assert f(p, p, -1, p, p, p, 0) == ERR_ARG
    assert f(p, None, 0, p, None, None, 0) == 0


def test_probes(lib):
    assert lib.odam_sq_fma_peak(0, None) == ERR_ARG
    n = C.c_longlong()
    assert lib.odam_sq_selftest(0, 1, 100, None) == ERR_ARG
    assert lib.odam_sq_selftest(0, 1, -1, C.byref(n)) == ERR_ARG
    assert lib.odam_sq_cluster_capacity(0, 2, None) == ERR_ARG
    k = C.c_int()
    for cluster in (1, 5):
        assert lib.odam_sq_cluster_capacity(0, cluster, C.byref(k)) == ERR_ARG


def test_optimize(lib):
    """Both optimiser entries share one validation; the host entry also checks the offsets and classes it stages."""
    voff, cls = np.array([0, 2, 5], np.int32), np.array([1, 7], np.int32)
    for f, last in ((lib.odam_sq_optimize, None), (lib.odam_sq_optimize_host, 0)):
        def call(init=p, cls_=host(cls), voff_=host(voff), prior=None, n=2, n_iters=1, repr_=0, params=p, loss=p):
            return f(init, cls_, voff_, p, p, p, prior, n, n_iters, repr_, 0.01, 0.1, params, loss, None, None, last)
        assert call(init=None) == ERR_ARG
        assert call(voff_=None) == ERR_ARG
        assert call(params=None) == ERR_ARG
        assert call(loss=None) == ERR_ARG
        assert call(n=-1) == ERR_ARG
        assert call(n_iters=-1) == ERR_ARG
        assert call(repr_=3) == ERR_ARG
        assert call(repr_=-1) == ERR_ARG
        assert call(prior=p, cls_=None) == ERR_ARG   # the prior is looked up by class
        assert call(n=0) == 0
        assert call(n_iters=0) == 0
    f = lib.odam_sq_optimize_host
    for bad in ([1, 2, 5], [0, 3, 2]):
        voff_bad = np.array(bad, np.int32)
        assert f(p, None, host(voff_bad), p, p, p, None, 2, 1, 0, 0.01, 0.1, p, p, None, None, 0) == ERR_ARG, bad
    cls_bad = np.array([1, 8], np.int32)   # 8 classes
    assert f(p, host(cls_bad), host(voff), p, p, p, p, 2, 1, 0, 0.01, 0.1, p, p, None, None, 0) == ERR_ARG
