"""Float64 vector-Jacobian product of the projected box sides with respect to the camera matrices -- the oracle of the
camera gradient of box_sides (camera_grad=True).

TEST INFRASTRUCTURE ONLY.  With the sample angles and the arg sample of every (view, side) held fixed, side s of view v
is pred = q_r / (|q_z| + 1e-6f), q = M_v [X, Y, Z, 1] the projection of its arg sample and r = s >> 1 (sq_libs.py:397-401).
The world points are the float64 surface of oracle/grad64.py (`_world`).
"""
import numpy as np
import torch

from oracle.grad64 import F64, LIM, _world


def sides_ms_vjp64(p9, etas, omegas, Ms, arg, grad_pred):
    """The gradient of sum over the (v, s) with arg >= 0 of grad_pred[v, s] * pred[v, s] with respect to Ms, in float64,
    and its conditioning scale: per entry, the sum over those terms of |d term / d M_v[k]| with every world coordinate
    replaced by the sum of the magnitudes it is formed from (|x cos| + |y sin| + |t_x|, ...), since the fp32 point
    carries a rounding error of that size.

    p9: parameters; etas, omegas [1000]: the sample angles; Ms [V, 12]; arg [V, 4] (< 0: a sentinel won, no term);
    grad_pred [V, 4]: the upstream gradient.  Returns (g [V, 12], scale [V, 12])."""
    Ms = np.asarray(Ms, np.float32).reshape(-1, 12)
    V = Ms.shape[0]
    arg = np.asarray(arg).reshape(V, 4)
    c32 = np.asarray(grad_pred, np.float32).reshape(V, 4)
    g, scale = np.zeros((V, 12)), np.zeros((V, 12))
    vi, sd = np.nonzero(arg >= 0)
    if not vi.size:
        return g, scale
    idx = arg[vi, sd]
    p = torch.tensor(np.asarray(p9, np.float32).reshape(9), dtype=F64)
    eta = torch.tensor(np.asarray(etas, np.float32)[idx], dtype=F64)
    om = torch.tensor(np.asarray(omegas, np.float32)[idx], dtype=F64)
    with torch.no_grad():
        pts = _world(p, eta, om)                                                           # [T, 3]
        local = _world(torch.cat([torch.zeros(4, dtype=F64), p[4:]]), eta, om)             # no yaw, no translation
        cz, sz = torch.cos(p[3]).abs(), torch.sin(p[3]).abs()
        lx, ly = local[:, 0].abs(), local[:, 1].abs()
        mag = torch.stack([lx * cz + ly * sz + p[0].abs(), lx * sz + ly * cz + p[1].abs(), local[:, 2].abs() + p[2].abs(),
                           torch.ones_like(lx)], 1)                                       # [T, 4]
    ph = torch.cat([pts, torch.ones_like(pts[:, :1])], 1)
    M = torch.tensor(Ms[vi].reshape(-1, 3, 4), dtype=F64).requires_grad_(True)             # one copy per term
    q = torch.einsum("tij,tj->ti", M, ph)
    d = torch.abs(q[:, 2]) + LIM
    num = torch.where(torch.tensor(sd < 2), q[:, 0], q[:, 1])
    c = torch.tensor(c32[vi, sd], dtype=F64)
    rows, = torch.autograd.grad((c * num / d).sum(), M)                                    # [T, 3, 4]
    np.add.at(g, vi, rows.reshape(-1, 12).numpy())
    with torch.no_grad():
        sc = torch.zeros_like(rows)
        t = torch.arange(len(vi))
        sc[t, torch.tensor(sd >> 1)] = (c.abs() / d)[:, None] * mag
        sc[:, 2] = (c * num).abs()[:, None] / (d * d)[:, None] * mag
    np.add.at(scale, vi, sc.reshape(-1, 12).numpy())
    return g, scale
