"""Parity at BASELINE.json's full sizes through size-independent properties: an object's trajectory must not depend
on what else is in the launch (bit-exact against the same object launched in a small batch), the launch is
deterministic, the first iterations of sampled objects match the CPU oracle, nothing is flagged, and the optimisation
does what it is for (the loss falls)."""
import numpy as np
import pytest

from launch_checks import DECISIONS, object_row, oracle_first_iterations

pytestmark = pytest.mark.gpu


def _check(api, coracle, cfg_idx, n_objects=None, n_iters=None, sample=8, oracle_iters=4):
    import torch
    from odam_b200 import synthetic
    c = synthetic.CONFIGS[cfg_idx]
    n_iters = n_iters or c["n_iters"]
    scene = synthetic.make_scene(n_objects or c["n_objects"], c["n_views"], seed=cfg_idx, device="cuda:0")
    tracks = api.pack_scene(scene)
    prior = api.prior_table() if c["prior"] else None
    dt = api.DeviceTracks(tracks, "cuda:0", prior)
    out = api.optimize_device(dt, n_iters=n_iters)
    out2 = api.optimize_device(dt, n_iters=n_iters, out={k: torch.empty_like(v) for k, v in out.items()})
    torch.cuda.synchronize()
    P, L, S = (out[k].cpu().numpy() for k in ("params", "loss", "status"))
    assert np.array_equal(P, out2["params"].cpu().numpy()) and np.array_equal(L, out2["loss"].cpu().numpy())
    assert (S & 3 == 0).all(), f"{int((S & 3 != 0).sum())} objects flagged"
    assert np.isfinite(P).all() and np.isfinite(L).all()
    assert (L[:, -1] < L[:, 0]).mean() > 0.99
    rng = np.random.default_rng(cfg_idx)
    pick = np.sort(rng.choice(tracks.n, size=min(sample, tracks.n), replace=False))
    # the launch configuration (CTA size, slices, cluster) is chosen from the batch statistics; replay the picked objects
    # with the SAME configuration so that only the batch composition differs
    cfg = api.query_launch(tracks.view_off)
    flips = []
    for i in pick:
        # ... except the code layout on every other pick: the two builds of the kernel must agree bit for bit
        layout = cfg["code_layout"] if (i % 2 == 0 or cfg["threads"] > 256) else 3 - cfg["code_layout"]
        alone = tracks.slice(i, i + 1)
        one = api.optimize_host(alone, prior=prior, n_iters=n_iters, threads=cfg["threads"],
                                max_slices=cfg["max_slices"], cluster=cfg["cluster"], code_layout=layout)
        assert np.array_equal(one["params"][0], P[i]) and np.array_equal(one["loss"][0], L[i]), i
        # the kernel's discrete decisions at every one of the first iterations, from the object launched alone
        launch = lambda k: object_row(api.optimize_host(alone, prior=prior, n_iters=k, extras=DECISIONS),
                                      alone.view_off, 0)
        flip = oracle_first_iterations(coracle, tracks, i, prior, oracle_iters, launch, L[i, 0])
        if flip:
            flips.append(flip)
    print(f"config {cfg_idx}: {len(pick)} sampled objects x {oracle_iters} iterations vs the C oracle: "
          f"{len(pick) - len(flips)} agree in every discrete decision and are inside the BASELINE tolerances; "
          f"{len(flips)} with a differently resolved near-tie: {flips}")
    assert len(flips) <= len(pick) // 4, flips
    return L


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


@pytest.fixture(scope="module")
def coracle():
    from oracle import c_oracle
    c_oracle.build()
    return c_oracle


def test_config2_50_objects_50_views(api, coracle):
    _check(api, coracle, 2)


def test_config3_2000_objects_30_views(api, coracle):
    _check(api, coracle, 3)


def test_config4_500_objects_300_views(api, coracle):
    _check(api, coracle, 4, sample=4)


def test_config5_50k_objects_20_views_no_prior(api, coracle):
    _check(api, coracle, 5, sample=6)
