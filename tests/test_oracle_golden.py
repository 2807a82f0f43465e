"""CPU tests: the oracles in oracle/ against the committed outputs of the reference itself (tests/golden/)."""
import numpy as np
import pytest

from golden_cases import TOL_LOSS, TOL_PARAM, all_cases, rel_loss, rel_param, wide_cases
from oracle import c_oracle, torch_oracle


@pytest.fixture(scope="module", autouse=True)
def _built():
    c_oracle.build()


def test_uniform_stream_known_answers(sampler_kat):
    """float(mt19937(0)()) * 2^-32 (SURVEY section 4): u0..u3, u1000, u1001 and the bound that keeps int(u*201) < 201."""
    u = c_oracle.uniform_stream()
    assert np.array_equal(u[:8], sampler_kat["uniforms_head"])
    assert np.allclose(u[[0, 1, 2, 3, 1000, 1001]],
                       [0.548813522, 0.592844605, 0.715189338, 0.844265759, 0.310380816, 0.277773678], atol=2e-9)
    assert int(u[1000] * np.float32(201)) == 62 and int(u[1001] * np.float32(201)) == 55
    assert u.max() < 1.0


def test_c_sampler_bit_exact_vs_reference(sampler_kat):
    for k in range(len(sampler_kat["a"])):
        o = c_oracle.sample(sampler_kat["a"][k], sampler_kat["e"][k])
        assert np.array_equal(o["etas"], sampler_kat["etas"][k]), k
        assert np.array_equal(o["omegas"], sampler_kat["omegas"][k]), k


def test_sampler_edge_semantics():
    """cos(float(pi)/2) < 0 makes the last CDF increment negative for small exponents (SURVEY H3); the centre of each
    grid is exactly 0; both grids are strictly decreasing in angle."""
    o = c_oracle.sample(np.array([0.5, 0.4, 0.3], np.float32), np.array([0.2, 0.9], np.float32))
    assert o["cdf"][199] > o["cdf"][200] == 1.0
    for g in (o["eta_grid"], o["omega_grid"]):
        assert (g == 0).sum() == 1 and np.all(np.diff(g) < 0)
    assert len(np.unique(o["omegas"])) <= 201 and o["eta_idx"].max() <= 200


def test_torch_oracle_bit_identical_to_reference(golden_runs):
    """The op-for-op torch port reproduces the reference's trajectories bit for bit (first 12 iterations of every
    case here; all iterations are asserted when the fixtures are generated)."""
    for case in all_cases(golden_runs):
        n = 12
        t = torch_oracle.run(golden_runs["translate"][case.obj], golden_runs["angle"][case.obj],
                             golden_runs["dims"][case.obj], golden_runs["P_cws"][case.obj][:case.V],
                             golden_runs["box"][case.obj][:case.V], golden_runs["mask"][case.obj][:case.V],
                             case.prior33, n, case.repr, anomaly=False)
        assert np.array_equal(t["init"], case.init)
        for x in ("params", "grad", "m", "v", "loss"):
            assert np.array_equal(t[x], getattr(case, x)[:n]), (case.k, x)
        live = case.mask.astype(bool)
        assert np.array_equal(t["arg"][:, live], case.arg[:n][:, live])


def test_c_oracle_teacher_forced_vs_reference(golden_runs):
    """Every 4th recorded reference state -> one C-oracle step -> reference's next state, BASELINE tolerances;
    steps whose discrete decisions differ from the reference's are the only ones allowed outside."""
    viol = steps = 0
    for case in all_cases(golden_runs):
        P, M, V = case.states_before()
        live = case.mask.astype(bool)
        for s in range(0, case.iters, 4):
            o = c_oracle.run(P[s], case.Ms, case.box, case.mask, case.prior33, 1, case.repr == "super_quadric",
                             m0=M[s], v0=V[s], step0=s, s0=case.init[4:7], record_indices=True)
            steps += 1
            assert rel_loss(o["loss"][0], case.loss[s]) <= TOL_LOSS
            ok = rel_param(o["params"][0], case.params[s]).max() <= TOL_PARAM
            same = (np.array_equal(o["arg"][0][live], case.arg[s][live]) and np.array_equal(o["eta_idx"][0], case.eta_idx[s])
                    and np.array_equal(np.sign(o["pred"][0] - case.box)[live], case.resid_sign[s][live]))
            assert ok or not same, (case.k, s)
            viol += not ok
    assert viol <= max(1, steps // 100)


def test_c_oracle_free_running_first_iterations(golden_runs):
    for case in all_cases(golden_runs):
        o = c_oracle.run(case.init, case.Ms, case.box, case.mask, case.prior33, 10, case.repr == "super_quadric")
        assert rel_loss(o["loss"], case.loss[:10]).max() <= TOL_LOSS
        assert rel_param(o["params"], case.params[:10]).max() <= TOL_PARAM


def test_oracle_points_vs_reference(golden_runs):
    for case in all_cases(golden_runs)[:4]:
        pts = c_oracle.points(case.params[-1])
        close = np.isclose(pts, case.final_points, rtol=2e-6, atol=2e-7).all(1)
        assert close.mean() > 0.995


def test_torch_oracle_bit_identical_on_wide_cases(golden_wide):
    """The BASELINE view counts (V = 50, 30, 300) and the loop's edge cases (view behind the camera, fully masked
    views, all-masked track, object straddling z = 0.5): the torch port reproduces the reference bit for bit
    (first 6 iterations here; every iteration was asserted when the fixture was generated)."""
    import torch
    nt = torch.get_num_threads()
    torch.set_num_threads(1)   # as when the fixtures were recorded: at V = 300 torch's reductions split across threads
    try:                       # and the reference's own bits depend on the thread count
        for case in wide_cases(golden_wide):
            n = min(6, case.iters)
            t = torch_oracle.run(case.translate, case.angle, case.dims, case.Ms64, case.box64, case.mask, case.prior33,
                                 n, case.repr, anomaly=False)
            assert np.array_equal(t["init"], case.init), case.name
            for x in ("params", "grad", "m", "v", "loss"):
                assert np.array_equal(t[x], getattr(case, x)[:n], equal_nan=True), (case.name, x)
    finally:
        torch.set_num_threads(nt)


def test_c_oracle_teacher_forced_on_wide_cases(golden_wide):
    """The C restatement pinned at the BASELINE shapes: every 3rd recorded reference state -> one step -> the
    reference's next state within the BASELINE tolerances unless a discrete decision differs."""
    viol = steps = 0
    for case in wide_cases(golden_wide):
        P, M, V = case.states_before()
        live = case.mask.astype(bool)
        for s in range(0, case.iters, 3):
            o = c_oracle.run(P[s], case.Ms, case.box, case.mask, case.prior33, 1, case.repr == "super_quadric",
                             m0=M[s], v0=V[s], step0=s, s0=case.init[4:7], record_indices=True)
            steps += 1
            same = (np.array_equal(o["arg"][0][live], case.arg[s][live]) and np.array_equal(o["eta_idx"][0], case.eta_idx[s])
                    and np.array_equal(np.sign(o["pred"][0] - case.box)[live], case.resid_sign[s][live]))
            okl = rel_loss(o["loss"][0], case.loss[s]) <= TOL_LOSS or (case.loss[s] == 0 and o["loss"][0] == 0)
            okp = rel_param(o["params"][0], case.params[s]).max() <= TOL_PARAM
            assert (okl and okp) or not same, (case.name, s, rel_loss(o["loss"][0], case.loss[s]))
            viol += not (okl and okp)
    assert viol <= max(1, steps // 50), (viol, steps)


def test_reference_sampler_batch_semantics():
    """One reference call with B*M > 1: the generator is seeded once per CALL (sampling.cpp:169) and keeps drawing, so
    primitive p sees uniforms [2000p, 2000p + 2000) -- only primitive 0 equals a B = M = 1 call."""
    from conftest import golden
    S = golden("sampler_batch.npz")
    a, e = S["a"].reshape(-1, 3), S["e"].reshape(-1, 2)
    u = c_oracle.uniform_stream(2000 * len(a))
    for p in range(len(a)):
        o = c_oracle.sample(a[p], e[p])
        up = u[2000 * p: 2000 * p + 2000]
        cdf = o["cdf"]
        # libstdc++ lower_bound over the (possibly non-monotone) CDF, then the omega index int(u * 201)
        idx = np.array([_lower_bound(cdf, x) for x in up[:1000]])
        assert np.array_equal(o["eta_grid"][idx], S["etas"].reshape(-1, 1000)[p]), p
        assert np.array_equal(o["omega_grid"][(up[1000:] * np.float32(201)).astype(np.int32)], S["omegas"].reshape(-1, 1000)[p]), p


def _lower_bound(cdf, val):
    first, n = 0, len(cdf)
    while n > 0:
        half = n >> 1
        if cdf[first + half] < val:
            first, n = first + half + 1, n - half - 1
        else:
            n = half
    return min(first, len(cdf) - 1)
