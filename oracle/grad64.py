"""Float64 restatement of one optimiser step's gradient, with the step's discrete decisions held fixed.

TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py.

The loss of sq_libs.py:395-475 is piecewise smooth: once the sample angles (eta bucket and omega index of every
sample), the arg-extreme sample of every (view, side) and the sign of every L1 residual are fixed, it is a smooth
function of the nine parameters.  This module evaluates that function in float64 torch autograd and returns its
gradient together with a per-component conditioning scale, the sum over every live (view, side) term and the prior
of |d term / d p_k|.  An fp32 implementation that sums the same terms in any order is expected within a small
multiple of eps32 * scale of the float64 gradient; a dropped, doubled or mis-weighted term is not.

Restated ops (all in float64, constants as they reach the fp32 code):
  a = s^2, e = sigmoid(h) * 1.4 + 0.2                               sq_libs.py:26-27, 580-582
  zero angles nudged to 1e-6f                                        sampling.py:591-592
  signed powers, the 1e-6f magnitude clamp, rotz, translation        sampling.py:508-509, 600-615; sq_libs.py:556-595
  projection through |z| + 1e-6f, masked L1 mean over ALL V          sq_libs.py:395-430
  prior 20 (s0 - s)^T A (s0 - s)                                     sq_libs.py:463-466
"""
import numpy as np
import torch

from . import c_oracle

F64 = torch.float64
LIM = float(np.float32(1e-6))   # the reference's 1e-6 literal as fp32 tensors hold it


def omega_index():
    """Omega grid index of every sample: int(u[1000 + i] * 201) of the sampler's uniform stream (sampling.cpp:210-212);
    it does not depend on the parameters."""
    u = c_oracle.uniform_stream(2 * c_oracle.N_SAMPLES)
    return (u[c_oracle.N_SAMPLES:] * np.float32(c_oracle.GRID)).astype(np.int64)


def angles(grids, eta_idx, omega_idx=None):
    """Sample angles from the two 201-entry grids ([2, 201]: eta, omega) and the per-sample grid indices."""
    grids = np.asarray(grids, np.float32).reshape(2, -1)
    omega_idx = omega_index() if omega_idx is None else np.asarray(omega_idx, np.int64)
    return grids[0][np.asarray(eta_idx, np.int64)], grids[1][omega_idx]


def _world(p, eta, om):
    """World points of the surface samples (eta, om) for parameter rows p [..., 9] (float64 torch)."""
    lim = torch.tensor(LIM, dtype=F64)
    one = torch.tensor(1.0, dtype=F64)
    a = p[..., 4:7] ** 2
    e = torch.sigmoid(p[..., 7:9]) * 1.4 + 0.2
    eta = torch.where(eta == 0, lim, eta)
    om = torch.where(om == 0, lim, om)
    sp = lambda x, q: torch.sign(x) * torch.abs(x) ** q
    ce, se = sp(torch.cos(eta), e[..., 0]), sp(torch.sin(eta), e[..., 0])
    co, so = sp(torch.cos(om), e[..., 1]), sp(torch.sin(om), e[..., 1])
    clamp = lambda v: torch.where(v > 0, one, -one) * torch.maximum(torch.abs(v), lim)
    x, y, z = clamp(a[..., 0] * ce * co), clamp(a[..., 1] * ce * so), clamp(a[..., 2] * se)
    c, s = torch.cos(p[..., 3]), torch.sin(p[..., 3])
    return torch.stack([x * c - y * s + p[..., 0], x * s + y * c + p[..., 1], z + p[..., 2]], -1)


def project(p9, etas, omegas, Ms):
    """Float64 forward pass over every sample and view: (u [V,N], w [V,N], valid [V,N]) with the reference's
    z > 0.5 validity and |z| + 1e-6 denominator (sq_libs.py:397-401)."""
    with torch.no_grad():
        p = torch.tensor(np.asarray(p9, np.float32), dtype=F64)
        pts = _world(p, torch.tensor(etas, dtype=F64), torch.tensor(omegas, dtype=F64))       # [N,3]
        M = torch.tensor(np.asarray(Ms, np.float32).reshape(-1, 3, 4), dtype=F64)
        q = torch.einsum("vij,nj->vni", M[:, :, :3], pts) + M[:, None, :, 3]                 # [V,N,3]
        d = torch.abs(q[..., 2]) + LIM
        return (q[..., 0] / d).numpy(), (q[..., 1] / d).numpy(), (q[..., 2] > 0.5).numpy()


def grad64(p9, Ms, box, mask, etas, omegas, arg, sign, prior33=None, s0=None, optimize_shapes=True):
    """Gradient of one step's loss in float64 with the step's decisions held fixed.

    p9: the parameters before the step; Ms [V,12], box [V,4], mask [V,4]: the object's views;
    etas, omegas [1000]: the sample angles (before the zero nudge, or after: both give the same);
    arg [V,4]: arg-extreme sample per (view, side), < 0 where a sentinel won; sign [V,4]: sign of pred - box;
    prior33: the 3x3 prior matrix or None; s0 [3]: the prior anchor (default: the scales of p9).
    Returns (g [9], scale [9]); with frozen shapes (optimize_shapes False) both are 0 at [7:9], otherwise scale[7:9]
    also carries the fp32 conditioning of 1 - sigmoid(h).
    """
    p9 = np.asarray(p9, np.float32).reshape(9)
    V = int(np.asarray(Ms).reshape(-1, 12).shape[0])
    arg = np.asarray(arg).reshape(V, 4)
    sign = np.asarray(sign).reshape(V, 4)
    live = (np.asarray(mask).reshape(V, 4) != 0) & (arg >= 0) & (sign != 0) & np.isfinite(sign)
    vi, sd = np.nonzero(live)
    rows = torch.zeros((0, 9), dtype=F64)
    if vi.size:
        P = torch.tensor(p9, dtype=F64).expand(vi.size, 9).clone().requires_grad_(True)   # one copy per term
        idx = arg[vi, sd]
        pts = _world(P, torch.tensor(np.asarray(etas, np.float32)[idx], dtype=F64),
                     torch.tensor(np.asarray(omegas, np.float32)[idx], dtype=F64))
        M = torch.tensor(np.asarray(Ms, np.float32).reshape(V, 3, 4)[vi], dtype=F64)       # [T,3,4]
        q = torch.einsum("tij,tj->ti", M[:, :, :3], pts) + M[:, :, 3]
        d = torch.abs(q[:, 2]) + LIM
        uv = torch.where(torch.tensor(sd < 2), q[:, 0], q[:, 1]) / d
        target = torch.tensor(np.asarray(box, np.float32).reshape(V, 4)[vi, sd], dtype=F64)
        terms = torch.tensor(sign[vi, sd], dtype=F64) * (uv - target) / V
        rows, = torch.autograd.grad(terms.sum(), P)                                           # [T,9]: d term / d p
    g = rows.sum(0).numpy()
    scale = rows.abs().sum(0).numpy()
    if prior33 is not None:
        A = np.asarray(prior33, np.float32).astype(np.float64).reshape(3, 3)
        s = p9[4:7].astype(np.float64)
        dd = (s if s0 is None else np.asarray(s0, np.float32).astype(np.float64)) - s
        gp = -20.0 * (A + A.T) @ dd
        g[4:7] += gp
        scale[4:7] += np.abs(gp)
    if not optimize_shapes:
        g[7:9] = 0
        scale[7:9] = 0
    else:
        # the chain factor sigmoid(h) (1 - sigmoid(h)) is formed in fp32 from a rounded sigmoid: 1 - sigmoid(h) then
        # carries a relative error of eps32 * sigmoid / (1 - sigmoid), 400 eps32 at h = 6
        sig = 1 / (1 + np.exp(-p9[7:9].astype(np.float64)))
        scale[7:9] *= np.maximum(1, sig / (1 - sig))
    return g, scale


def ratio(g32, g64, scale):
    """|g32 - g64| / scale per component; 0 where both sides vanish, inf where only the scale does."""
    err = np.abs(np.asarray(g32, np.float64) - g64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(scale > 0, err / np.where(scale > 0, scale, 1), np.where(err > 0, np.inf, 0.0))
