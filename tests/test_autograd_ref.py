"""CPU tests of the differentiable ops (odam_b200/autograd.py) that need no GPU.

- The float64 oracle of the surface-points backward pass (tests/surface_vjp64.py) against fp32 torch autograd
  of the bit-identical port of the reference's surface (oracle/torch_oracle.py surface_points) on every recorded golden
  state, within TAU_REF times the per-component conditioning scale.  This pins the oracle the GPU tests hold the
  kernels to, as tests/test_backward_ref.py does for the loss gradient.
- The three C entries of the ops reject bad arguments before any CUDA call.
- The Python wrappers reject wrong dtypes, shapes, devices and offsets before any launch.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_cases import all_cases, wide_cases
from oracle import grad64 as G64
from surface_vjp64 import surface_vjp64
from oracle import torch_oracle

TAU_REF = 1e-6


def test_surface_vjp64_pins_reference_autograd(golden_runs, golden_wide):
    """Every recorded golden state, a seeded upstream gradient per state: fp32 autograd through the reference's surface
    within TAU_REF * scale of the float64 vector-Jacobian product under the same sample angles."""
    rng = np.random.default_rng(11)
    sampler = torch_oracle.default_sampler()
    worst = np.zeros(9)
    states = 0
    for case in all_cases(golden_runs) + wide_cases(golden_wide):
        P = case.states_before()[0]
        for p9 in P:
            leaves = [torch.tensor(p9[0:3], requires_grad=True), torch.tensor(p9[3], requires_grad=True),
                      torch.tensor(p9[4:7], requires_grad=True), torch.tensor(p9[7:9], requires_grad=True)]
            pts, etas, omegas = torch_oracle.surface_points(*leaves, sampler)
            G = rng.normal(size=(1000, 3)).astype(np.float32)
            (pts * torch.from_numpy(G)).sum().backward()
            g32 = np.concatenate([np.atleast_1d(x.grad.numpy()) for x in leaves])
            g64, sc = surface_vjp64(p9, etas.numpy().ravel(), omegas.numpy().ravel(), G)
            r = G64.ratio(g32, g64, sc)
            assert (r <= TAU_REF).all(), (getattr(case, "name", case.k), r)
            worst = np.maximum(worst, r)
            states += 1
    print(f"surface VJP, reference fp32 autograd vs float64 on {states} states: worst |g - g64| / scale "
          + " ".join(f"{x:.1e}" for x in worst))


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import _lib, build
    build.build()
    return _lib.load()


def test_c_entries_reject_bad_arguments(lib):
    """NULL pointers, n < 0 and total_views < 0 give ODAM_SQ_ERR_ARG and n == 0 is a no-op, all without a GPU (the
    dummy pointers are never dereferenced)."""
    p = C.c_void_p(16)
    ERR_ARG = -1
    assert lib.odam_sq_sample_points_vjp(None, p, 1, p, None) == ERR_ARG
    assert lib.odam_sq_sample_points_vjp(p, None, 1, p, None) == ERR_ARG
    assert lib.odam_sq_sample_points_vjp(p, p, 1, None, None) == ERR_ARG
    assert lib.odam_sq_sample_points_vjp(p, p, -1, p, None) == ERR_ARG
    assert lib.odam_sq_sample_points_vjp(p, p, 0, p, None) == 0
    for k in range(5):
        a = [p] * 5
        a[k] = None
        assert lib.odam_sq_box_sides(a[0], a[1], a[2], 1, 4, a[3], a[4], None) == ERR_ARG, k
    assert lib.odam_sq_box_sides(p, p, p, -1, 4, p, p, None) == ERR_ARG
    assert lib.odam_sq_box_sides(p, p, p, 1, -1, p, p, None) == ERR_ARG
    assert lib.odam_sq_box_sides(p, p, p, 0, 4, p, p, None) == 0
    for k in range(6):
        a = [p] * 6
        a[k] = None
        assert lib.odam_sq_box_sides_vjp(a[0], a[1], a[2], a[3], a[4], 1, 4, a[5], None) == ERR_ARG, k
    assert lib.odam_sq_box_sides_vjp(p, p, p, p, p, -1, 4, p, None) == ERR_ARG
    assert lib.odam_sq_box_sides_vjp(p, p, p, p, p, 1, -1, p, None) == ERR_ARG
    assert lib.odam_sq_box_sides_vjp(p, p, p, p, p, 0, 4, p, None) == 0


def test_wrapper_validation_without_gpu():
    """Wrong dtype, shape or device and inconsistent host offsets raise ValueError before anything is launched."""
    from odam_b200 import autograd as AG
    p = torch.zeros(2, 9)
    voff = torch.tensor([0, 1, 3], dtype=torch.int32)
    Ms = torch.zeros(3, 12)
    box, mask = torch.zeros(3, 4), torch.ones(3, 4, dtype=torch.uint8)
    with pytest.raises(ValueError, match="CUDA"):
        AG.surface_points(p)
    with pytest.raises(ValueError, match="float32"):
        AG.surface_points(p.double())
    with pytest.raises(ValueError, match="shape"):
        AG.surface_points(torch.zeros(2, 8))
    with pytest.raises(ValueError, match="CUDA"):
        AG.box_sides(p, voff, Ms)
    with pytest.raises(ValueError, match="CUDA"):
        AG.box_loss(p, voff, Ms.reshape(3, 3, 4), box, mask)
    with pytest.raises(ValueError, match="float32"):
        AG.box_sides(p.double(), voff, Ms)
    with pytest.raises(ValueError, match="Ms"):
        AG.box_sides(p, voff, Ms.double())
    with pytest.raises(ValueError, match="Ms"):
        AG.box_sides(p, voff, torch.zeros(3, 11))
    with pytest.raises(ValueError, match="int32"):
        AG.box_sides(p, voff.long(), Ms)
    with pytest.raises(ValueError, match=r"n \+ 1"):
        AG.box_sides(p, torch.tensor([0, 3], dtype=torch.int32), Ms)
    for bad in ([0, 1, 4], [1, 1, 3], [0, 4, 3]):   # wrong end (Ms has 3 views), wrong start, decreasing
        with pytest.raises(ValueError, match="view_off"):
            AG.box_sides(p, torch.tensor(bad, dtype=torch.int32), Ms)
