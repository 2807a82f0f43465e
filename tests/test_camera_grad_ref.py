"""CPU tests of the camera gradient of the differentiable box sides (box_sides / box_loss with camera_grad=True) that
need no GPU.

- The float64 restatement of dL/dMs (tests/sides_ms_vjp64.py) against central differences in float64 under the same
  decisions, on edge objects.  This pins the oracle the GPU tests hold the kernel to.
- odam_sq_box_sides_vjp_cameras rejects bad arguments before any CUDA call.
- The Python wrappers with camera_grad=True reject wrong dtypes, shapes, devices and offsets before any launch.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_cases import edge_object
from oracle import grad64 as G64
from oracle import torch_oracle
from sides_ms_vjp64 import sides_ms_vjp64


def _arg64(p9, etas, omegas, Ms):
    """The float64 arg-extreme sample of every (view, side) under the reference's rule, -1 where a sentinel wins."""
    u, w, valid = G64.project(p9, etas, omegas, Ms)
    arg = np.empty((len(Ms), 4), np.int64)
    for s in range(4):
        c = u if s < 2 else w
        cand = np.where(valid, c, 1e6 if s % 2 == 0 else -1e6)
        a = cand.argmin(1) if s % 2 == 0 else cand.argmax(1)
        arg[:, s] = np.where(valid[np.arange(len(Ms)), a], a, -1)
    return arg


def _sides64(pts, Ms, arg, c):
    """Per view: sum over the live sides of c * pred in float64 (pts [1000, 3], Ms [V, 3, 4] float64)."""
    V = Ms.shape[0]
    out = np.zeros(V)
    for s in range(4):
        live = arg[:, s] >= 0
        ph = np.concatenate([pts[np.maximum(arg[:, s], 0)], np.ones((V, 1))], 1)      # [V, 4]
        q = np.einsum("vij,vj->vi", Ms, ph)
        out += np.where(live, c[:, s] * q[:, s >> 1] / (np.abs(q[:, 2]) + G64.LIM), 0.0)
    return out


def test_sides_ms_vjp64_vs_central_differences():
    """On edge objects (plain, h = +-6, a view behind the camera, a single view) and seeded upstream gradients, the
    float64 dL/dMs within 1e-7 * scale of float64 central differences of the sides under the same decisions."""
    rng = np.random.default_rng(13)
    sampler = torch_oracle.default_sampler()
    worst, terms = 0.0, 0
    for kind in ("plain", "h+6", "h-6", "behind", "V1"):
        p9, Ms, _, _, _ = edge_object(kind)
        leaves = [torch.tensor(p9[0:3]), torch.tensor(p9[3]), torch.tensor(p9[4:7]), torch.tensor(p9[7:9])]
        _, etas, omegas = torch_oracle.surface_points(*leaves, sampler)
        etas, omegas = etas.numpy().ravel(), omegas.numpy().ravel()
        arg = _arg64(p9, etas, omegas, Ms)
        c = rng.normal(size=arg.shape).astype(np.float32)
        g, scale = sides_ms_vjp64(p9, etas, omegas, Ms, arg, c)
        with torch.no_grad():
            pts = G64._world(torch.tensor(p9, dtype=G64.F64), torch.tensor(etas, dtype=G64.F64),
                             torch.tensor(omegas, dtype=G64.F64)).numpy()
        M = Ms.astype(np.float64).reshape(-1, 3, 4)
        fd = np.zeros_like(g)
        for k in range(12):
            h = 1e-6 * max(1.0, float(np.abs(M.reshape(-1, 12)[:, k]).max()))
            Mp, Mm = M.copy(), M.copy()
            Mp.reshape(-1, 12)[:, k] += h
            Mm.reshape(-1, 12)[:, k] -= h
            fd[:, k] = (_sides64(pts, Mp, arg, c) - _sides64(pts, Mm, arg, c)) / (2 * h)
        r = G64.ratio(g, fd, scale)
        assert (r <= 1e-7).all(), (kind, r.max())
        assert (g[(arg < 0).all(1)] == 0).all(), kind                   # an all-sentinel view has no gradient
        if kind == "behind":
            assert (arg[0] < 0).all()
        worst = max(worst, float(r.max()))
        terms += int((arg >= 0).sum())
    print(f"sides_ms_vjp64 vs central differences on {terms} live sides: worst |g - fd| / scale {worst:.1e}")


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import _lib, build
    build.build()
    return _lib.load()


def test_c_entry_rejects_bad_arguments(lib):
    """Each required pointer NULL, n < 0 and total_views < 0 give ODAM_SQ_ERR_ARG; out_grad_params = NULL is accepted
    and n == 0 is a no-op, all without a GPU (the dummy pointers are never dereferenced)."""
    p = C.c_void_p(16)
    ERR_ARG = -1
    f = lib.odam_sq_box_sides_vjp_cameras
    for k in (0, 1, 2, 3, 4, 6):   # params, view_off, Ms, arg, grad_pred, out_grad_Ms
        a = [p] * 7
        a[k] = None
        assert f(a[0], a[1], a[2], a[3], a[4], 1, 4, a[5], a[6], None) == ERR_ARG, k
    assert f(p, p, p, p, p, -1, 4, p, p, None) == ERR_ARG
    assert f(p, p, p, p, p, 1, -1, p, p, None) == ERR_ARG
    assert f(p, p, p, p, p, 0, 4, p, p, None) == 0
    assert f(p, p, p, p, p, 0, 4, None, p, None) == 0


def test_wrapper_validation_with_camera_grad():
    """camera_grad=True keeps every ValueError of the default path: wrong dtype, shape or device and inconsistent host
    offsets raise before anything is launched."""
    from odam_b200 import autograd as AG
    p = torch.zeros(2, 9)
    voff = torch.tensor([0, 1, 3], dtype=torch.int32)
    Ms = torch.zeros(3, 12, requires_grad=True)
    box, mask = torch.zeros(3, 4), torch.ones(3, 4, dtype=torch.uint8)
    sides = lambda *a: AG.box_sides(*a, camera_grad=True)
    with pytest.raises(ValueError, match="CUDA"):
        sides(p, voff, Ms)
    with pytest.raises(ValueError, match="CUDA"):
        AG.box_loss(p, voff, Ms.reshape(3, 3, 4), box, mask, camera_grad=True)
    with pytest.raises(ValueError, match="float32"):
        sides(p.double(), voff, Ms)
    with pytest.raises(ValueError, match="Ms"):
        sides(p, voff, Ms.double())
    with pytest.raises(ValueError, match="Ms"):
        sides(p, voff, torch.zeros(3, 11, requires_grad=True))
    with pytest.raises(ValueError, match="int32"):
        sides(p, voff.long(), Ms)
    with pytest.raises(ValueError, match=r"n \+ 1"):
        sides(p, torch.tensor([0, 3], dtype=torch.int32), Ms)
    for bad in ([0, 1, 4], [1, 1, 3], [0, 4, 3]):
        with pytest.raises(ValueError, match="view_off"):
            sides(p, torch.tensor(bad, dtype=torch.int32), Ms)
