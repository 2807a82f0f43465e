"""Float64 vector-Jacobian product of the surface samples -- the oracle of the surface_points backward pass.

TEST INFRASTRUCTURE ONLY.  It restates the surface with the same float64 ops as oracle/grad64.py (`_world`): signed
powers, the 1e-6f magnitude clamp, rotz, translation (sampling.py:591-615, sq_libs.py:556-595), with the sample angles
held fixed.
"""
import numpy as np
import torch

from oracle.grad64 import F64, _world


def surface_vjp64(p9, etas, omegas, G):
    """The gradient of sum_i G_i . pts_i with respect to the nine parameters in float64, and its conditioning scale
    sum_i |d(G_i . pts_i)/d p_k|.

    p9: parameters; etas, omegas [1000]: the sample angles; G [1000, 3]: the upstream gradient.  As in grad64,
    scale[7:9] also carries the fp32 conditioning of 1 - sigmoid(h).  Returns (g [9], scale [9])."""
    p9 = np.asarray(p9, np.float32).reshape(9)
    G = torch.tensor(np.asarray(G, np.float64).reshape(-1, 3), dtype=F64)
    N = G.shape[0]
    P = torch.tensor(p9, dtype=F64).expand(N, 9).clone().requires_grad_(True)   # one copy per sample
    pts = _world(P, torch.tensor(np.asarray(etas, np.float32), dtype=F64),
                 torch.tensor(np.asarray(omegas, np.float32), dtype=F64))
    rows, = torch.autograd.grad((G * pts).sum(), P)                                 # [N, 9]
    g = rows.sum(0).numpy()
    scale = rows.abs().sum(0).numpy()
    with np.errstate(over="ignore"):   # h = -10000 (cube): sigmoid 0
        sig = 1 / (1 + np.exp(-p9[7:9].astype(np.float64)))
    scale[7:9] *= np.maximum(1, sig / (1 - sig))
    return g, scale
