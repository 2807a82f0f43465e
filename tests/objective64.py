"""Float64 restatement of the fused optimiser's gradient under the opt-in objective (odam_sq_objective): per-side
weights and the robust residual losses, with the step's discrete decisions held fixed.

Each live (view, side) term is w * rho(uv - target) / V.  Its gradient is w * rho'(r) * d uv / d p / V, so it is
oracle/grad64.py's gradient with w * rho'(r) in place of the L1 sign: the same float64 chain rule, and a conditioning
scale that carries the weight.  r is a decision held fixed like the L1 sign: checks of an fp32 implementation pass its
own residual pred - box (whose value check_decisions verifies separately), because rho' is continuous in r and an fp32
residual differs from the float64 one by a few ulp of the projected coordinate -- up to 1e-5 of rho' for pixel-sized
beta or c, more than the fp32 gradient itself is allowed to be off.  With the defaults (no weight,
L1) this is grad64 itself, arithmetic untouched.
"""
import numpy as np
import torch

from oracle import grad64 as G64

F64 = torch.float64


def rho64(r, loss, scale):
    """(rho(r), rho'(r)) in float64 numpy."""
    r = np.asarray(r, np.float64)
    z = np.abs(r)
    if loss == "l1":
        return z, np.sign(r)
    if loss == "smooth_l1":
        quad = z < scale
        return np.where(quad, 0.5 * r * r / scale, z - 0.5 * scale), np.where(quad, r / scale, np.sign(r))
    if loss == "cauchy":
        t = r / scale
        return 0.5 * scale * scale * np.log1p(t * t), r / (1 + t * t)
    raise ValueError(loss)


def arg_uv(p9, Ms, etas, omegas, arg):
    """Float64 projection [V, 4] of every (view, side)'s arg-extreme sample (NaN where arg < 0)."""
    u, w, _ = G64.project(p9, etas, omegas, Ms)
    V = len(u)
    a = np.asarray(arg).reshape(V, 4)
    out = np.full((V, 4), np.nan)
    for sd in range(4):
        c = u if sd < 2 else w
        has = a[:, sd] >= 0
        out[has, sd] = c[np.arange(V)[has], a[has, sd]]
    return out


def grad64(p9, Ms, box, mask, etas, omegas, arg, sign, prior33=None, s0=None, optimize_shapes=True, weight=None,
           loss="l1", loss_scale=None, residual=None):
    """oracle/grad64.grad64 with the objective's weight [V, 4] (None = 1), loss and loss_scale.  sign: the sign of the
    kernel's pred - box (the L1 decision); the robust kinds take rho' at `residual` [V, 4] (the implementation's own
    pred - box), or at the float64 residual of the arg samples when it is None."""
    V = int(np.asarray(Ms).reshape(-1, 12).shape[0])
    sign = np.asarray(sign, np.float64).reshape(V, 4)
    if loss == "l1":
        coef = sign
    elif residual is not None:
        r = np.asarray(residual, np.float64).reshape(V, 4)
    else:
        r = arg_uv(p9, Ms, etas, omegas, arg) - np.asarray(box, np.float32).astype(np.float64).reshape(V, 4)
    if loss != "l1":
        coef = np.where(np.isfinite(sign) & np.isfinite(r), rho64(np.nan_to_num(r), loss, loss_scale)[1], np.nan)
    if weight is not None:
        coef = coef * np.asarray(weight, np.float32).astype(np.float64).reshape(V, 4)
    return G64.grad64(p9, Ms, box, mask, etas, omegas, arg, coef, prior33, s0, optimize_shapes)


def loss64(p, Ms, box, mask, etas, omegas, arg, weight=None, loss="l1", loss_scale=None):
    """The 2-D term of one object's loss in float64 at parameters p [9] (float64), the samples of each (view, side)
    held at arg: sum over live terms of w * rho(uv - target) / V (no prior).  For central differences."""
    V = int(np.asarray(Ms).reshape(-1, 12).shape[0])
    a = np.asarray(arg).reshape(V, 4)
    w = np.ones((V, 4)) if weight is None else np.asarray(weight, np.float32).astype(np.float64).reshape(V, 4)
    live = (np.asarray(mask).reshape(V, 4) != 0) & (a >= 0) & (w > 0)
    vi, sd = np.nonzero(live)
    if not vi.size:
        return 0.0
    with torch.no_grad():
        P = torch.tensor(np.asarray(p, np.float64), dtype=F64).expand(vi.size, 9)
        idx = a[vi, sd]
        pts = G64._world(P, torch.tensor(np.asarray(etas, np.float32)[idx], dtype=F64),
                         torch.tensor(np.asarray(omegas, np.float32)[idx], dtype=F64))
        M = torch.tensor(np.asarray(Ms, np.float32).reshape(V, 3, 4)[vi], dtype=F64)
        q = torch.einsum("tij,tj->ti", M[:, :, :3], pts) + M[:, :, 3]
        d = torch.abs(q[:, 2]) + G64.LIM
        uv = (torch.where(torch.tensor(sd < 2), q[:, 0], q[:, 1]) / d).numpy()
    r = uv - np.asarray(box, np.float32).astype(np.float64).reshape(V, 4)[vi, sd]
    return float((w[vi, sd] * rho64(r, loss, loss_scale)[0]).sum() / V)
