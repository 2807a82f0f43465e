"""CPU tests of the optimiser's gradient itself, not only of the Adam step that consumes it.

Adam divides the gradient by its own running magnitude (from a fresh state the first update is exactly lr * sign(g)),
so parameter comparisons are nearly blind to a gradient that is off by a few per cent.  Here the gradient is compared
directly with a float64 restatement of the same step (oracle/grad64.py) that holds the step's discrete decisions
fixed: sample angles, arg-extreme sample per (view, side) and residual signs.  The bound is TAU_REF times the
per-component conditioning scale (sum of |d term / d p_k| over the live terms and the prior), so it holds for any
summation order and fails for a dropped, doubled or mis-weighted term.
"""
import ctypes
import ctypes.util

import numpy as np
import pytest
import torch

from golden_cases import EDGE_KINDS, all_cases, edge_object, wide_cases
from oracle import c_oracle, torch_oracle
from oracle import grad64 as G64

# Worst |g32 - g64| / scale measured over every recorded golden state: 5.4e-7 (reference, yaw component), see the
# printed per-component maxima.  About 8 eps32; a 1 % error in one term of a 20-view object is ~1e-3.
TAU_REF = 1e-6

_libm = ctypes.CDLL(ctypes.util.find_library("m"))
_libm.expf.restype, _libm.expf.argtypes = ctypes.c_float, [ctypes.c_float]


@pytest.fixture(scope="module", autouse=True)
def _built():
    c_oracle.build()


def _ae32(p9):
    """(a, e) as the fp32 C oracle hands them to the sampler (glibc expf, no contraction; sq_oracle.c:274-279)."""
    p9 = np.asarray(p9, np.float32)
    a = p9[4:7] * p9[4:7]
    sig = np.array([np.float32(1) / (np.float32(1) + np.float32(_libm.expf(float(-h)))) for h in p9[7:9]], np.float32)
    return a, sig * np.float32(1.4) + np.float32(0.2)


def _print_worst(label, worst):
    print(f"{label}: worst |g - g64| / scale per component " + " ".join(f"{x:.2e}" for x in worst))


def _oracle_ratios(init9, Ms, box, mask, prior33, n_iters, representation, s0=None, **kw):
    """Runs the fp32 C oracle and returns, per iteration, |grad - g64| / scale under the oracle's own decisions."""
    opt = representation == "super_quadric"
    o = c_oracle.run(init9, Ms, box, mask, prior33, n_iters, opt, s0=s0, record_indices=True, **kw)
    assert o["rc"] == 0
    P = np.vstack([np.asarray(init9, np.float32)[None], o["params"][:-1]])
    nc = 9 if opt else 7
    out = []
    for it in range(n_iters):
        smp = c_oracle.sample(*_ae32(P[it]))
        assert np.array_equal(smp["eta_idx"], o["eta_idx"][it]) and np.array_equal(smp["omega_idx"], o["omega_idx"][it])
        sign = np.sign(o["pred"][it] - box)
        g, sc = G64.grad64(P[it], Ms, box, mask, smp["etas"], smp["omegas"], o["arg"][it], sign, prior33,
                           P[0][4:7] if s0 is None else s0, opt)
        if not opt:
            assert np.array_equal(o["grad"][it][7:9], np.zeros(2, np.float32))
        out.append(G64.ratio(o["grad"][it][:nc], g[:nc], sc[:nc]))
        if len(out[-1]) < 9:
            out[-1] = np.concatenate([out[-1], np.zeros(9 - nc)])
    return out


def test_float64_restatement_pins_reference_gradient(golden_runs, golden_wide):
    """Every recorded golden state (ref_runs.npz and ref_runs_wide.npz): the reference's own fp32 gradient is within
    TAU_REF * scale of the float64 restatement under the reference's decisions, which the bit-identical torch port
    supplies (etas, omegas, arg, pred per step)."""
    nt = torch.get_num_threads()
    torch.set_num_threads(1)   # the recorded bits at V = 300 are those of single-threaded reductions
    worst = np.zeros(9)
    try:
        for case in all_cases(golden_runs) + wide_cases(golden_wide):
            if hasattr(case, "name"):
                tr = torch_oracle.run(case.translate, case.angle, case.dims, case.Ms64, case.box64, case.mask,
                                      case.prior33, case.iters, case.repr, anomaly=False)
            else:
                G = golden_runs
                tr = torch_oracle.run(G["translate"][case.obj], G["angle"][case.obj], G["dims"][case.obj],
                                      G["P_cws"][case.obj][:case.V], G["box"][case.obj][:case.V],
                                      G["mask"][case.obj][:case.V], case.prior33, case.iters, case.repr, anomaly=False)
            assert np.array_equal(tr["grad"], case.grad, equal_nan=True), getattr(case, "name", case.k)
            P = case.states_before()[0]
            nc = 9 if case.repr == "super_quadric" else 7   # the reference records the unapplied shape gradient
            for it in range(case.iters):
                g, sc = G64.grad64(P[it], case.Ms, case.box, case.mask, tr["etas"][it], tr["omegas"][it],
                                   tr["arg"][it], np.sign(tr["pred"][it] - case.box), case.prior33, case.init[4:7],
                                   case.repr == "super_quadric")
                r = G64.ratio(case.grad[it][:nc], g[:nc], sc[:nc])
                assert (r <= TAU_REF).all(), (getattr(case, "name", case.k), it, r)
                worst[:nc] = np.maximum(worst[:nc], r)
    finally:
        torch.set_num_threads(nt)
    _print_worst("reference (torch port) vs float64", worst)


def test_c_oracle_gradient_on_golden_states(golden_runs, golden_wide):
    """The C oracle's analytic backward pass (sq_oracle.c) from every recorded reference state: one step, its gradient
    against the float64 restatement under the oracle's own decisions."""
    worst = np.zeros(9)
    for case in all_cases(golden_runs) + wide_cases(golden_wide):
        P, M, V = case.states_before()
        for s in range(case.iters):
            r, = _oracle_ratios(P[s], case.Ms, case.box, case.mask, case.prior33, 1, case.repr, s0=case.init[4:7],
                                m0=M[s], v0=V[s], step0=s)
            assert (r <= TAU_REF).all(), (getattr(case, "name", case.k), s, r)
            worst = np.maximum(worst, r)
    _print_worst("C oracle on golden states vs float64", worst)


@pytest.mark.parametrize("representation", ["cube", "quadric", "super_quadric"])
@pytest.mark.parametrize("with_prior", [True, False])
def test_c_oracle_gradient_synthetic(representation, with_prior):
    """Seeded synthetic objects at the edges of the backward pass, every representation, with and without the prior:
    5 free-running oracle steps each, every step's gradient against float64."""
    from odam_b200.api import prior_table
    table = prior_table()
    worst = np.zeros(9)
    for kind in EDGE_KINDS:
        if representation != "super_quadric" and kind.startswith("h"):
            continue   # frozen shapes: the exponents stay at their initial values
        init, Ms, box, mask, cls = edge_object(kind)
        if representation == "cube":
            init[7:9] = -10000.0
        elif representation == "quadric":
            init[7:9] = 0.0
        prior = table[cls].reshape(3, 3) if with_prior else None
        for it, r in enumerate(_oracle_ratios(init, Ms, box, mask, prior, 5, representation)):
            assert (r <= TAU_REF).all(), (kind, it, r)
            worst = np.maximum(worst, r)
    _print_worst(f"C oracle, synthetic {representation} prior={with_prior} vs float64", worst)
