"""Every build of the fused optimiser at a batch shape that selects it.

sq_optimize_kernel ships as five production builds (straight-line 256, 512 and 1024 threads with 64 registers, compact
256, and the 128-register solo 512 of the latency regime), each with a cycle-mark twin, and a launch either stages its
cameras, boxes and masks into shared memory or reads them from global memory.  The builds are different machine code,
so each is checked where the library picks it: SHAPES lists dense batches (more CTAs than SMs) whose statistics select
every build but the solo one, staged and unstaged.  The eleven edge objects of golden_cases replace objects spread
through each batch, so that their semantics run under the dense builds too.

  - test_shapes_select_their_builds (CPU): each row still selects its build, CTA size, cluster, slices and staging,
    and the rows with the latency-regime batches of the existing tests cover every production build, staged and
    unstaged in both regimes.
  - test_launch_shape (GPU), per row at 1 and 5 iterations: every object's last-iteration gradient against float64
    under the kernel's own decisions (launch_checks.check_launch); sampled objects against the C oracle over their
    first iterations; the sampled objects replayed alone (the latency-regime build, and the other code layout up to
    256 threads) bit-identical in every output; the cycle-mark twin and the device entry bit-identical to the host
    entry; only the behind-camera object flagged, and only with ODAM_SQ_ST_NO_VALID_PT.
"""
import time
from collections import namedtuple

import numpy as np
import pytest

from golden_cases import EDGE_KINDS, edge_object
from launch_checks import DECISIONS, EXTRAS, check_launch, object_row, oracle_first_iterations, pack

N_SMS = 148                # query_launch without an initialised device answers for a B200
STAGE_BYTES_PER_VIEW = 68  # 12 + 4 floats and 4 mask bytes of a view in the staging area
EDGE_VIEWS = [1 if k == "V1" else 12 for k in EDGE_KINDS]   # golden_cases.edge_object
BUILDS = {"plain 256", "plain 512", "plain 1024", "compact 256", "solo 512"}

# query_launch's smem_bytes (dynamic + static shared memory) of an unstaged launch whose CTAs hold no more views than
# threads, by CTA size; a staged launch adds STAGE_BYTES_PER_VIEW for each view of the longest track a CTA holds,
# rounded up to 4 views
UNSTAGED_SMEM = {256: 40672, 320: 42848, 512: 49376, 1024: 66784}

# groups: (objects, views) -- the later groups' tracks spread evenly among the first group's; edges: swap the edge
# objects in
Row = namedtuple("Row", "name groups options build threads cluster slices ctas_per_sm smem_bytes staged edges",
                 defaults=(True,))
SHAPES = [
    Row("200x30", ((200, 30),), {}, "plain 512", 512, 1, 8, 2, 51552, True),            # two wide CTAs per SM
    Row("160x20", ((160, 20),), {}, "plain 512", 512, 1, 12, 2, 50736, True),
    Row("300x60", ((300, 60),), {}, "plain 256", 256, 1, 8, 4, 44752, True),
    Row("300x60-compact", ((300, 60),), dict(code_layout=2), "compact 256", 256, 1, 8, 4, 44752, True),
    Row("160x200", ((160, 200),), {}, "plain 256", 256, 2, 8, 4, 47472, True),
    Row("160x250", ((160, 250),), {}, "plain 512", 320, 2, 8, 3, 51552, True),
    Row("300x30", ((300, 30),), {}, "compact 256", 256, 1, 8, 4, 42848, True),
    Row("200x30-1024", ((200, 30),), dict(threads=1024), "plain 1024", 1024, 1, 8, 1, 68960, True),
    # a few long tracks among many short ones: four CTAs' staging areas would not fit an SM's shared memory
    Row("290x20+10x256", ((290, 20), (10, 256)), {}, "compact 256", 256, 1, 8, 4, 40672, False),
    Row("290x20+10x256-plain", ((290, 20), (10, 256)), dict(code_layout=1), "plain 256", 256, 1, 8, 4, 40672, False),
]
# the latency-regime batches of test_backward_gpu and test_parity_gpu (edge objects, 1500-view tracks)
LATENCY = [
    Row("11 edge objects", ((10, 12), (1, 1)), {}, "solo 512", 512, 1, 25, 1, 50192, True, False),
    Row("2x1500", ((2, 1500),), {}, "solo 512", 512, 4, 25, 1, 49376, False, False),
    Row("2x1500-cluster1", ((2, 1500),), dict(cluster=1), "plain 1024", 1024, 1, 25, 1, 82016, False, False),
]


def _group_of(groups):
    """Group index of every object of the batch: the later groups' objects spread evenly among the first group's."""
    n = sum(m for m, _ in groups)
    which = np.zeros(n, int)
    for g, (m, _) in enumerate(groups[1:], 1):
        which[np.round((np.arange(m) + 0.5) * n / m).astype(int)] = g
    assert [int((which == g).sum()) for g in range(len(groups))] == [m for m, _ in groups]
    return which


def _edge_at(n):
    return np.round(np.linspace(0, n - 1, len(EDGE_KINDS))).astype(int)


def view_counts(row):
    if not row.edges:
        return np.concatenate([[V] * m for m, V in row.groups])
    which = _group_of(row.groups)
    assert (which[_edge_at(len(which))] == 0).all()   # edge objects replace objects of the first group
    counts = np.array([row.groups[g][1] for g in which])
    counts[_edge_at(len(counts))] = EDGE_VIEWS
    return counts


def _offsets(counts):
    return np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)


def _staging_bytes(views):
    return STAGE_BYTES_PER_VIEW * (-(-views // 4) * 4)


def expected_launch(row):
    return dict(threads=row.threads, smem_bytes=row.smem_bytes, ctas_per_sm=row.ctas_per_sm, cluster=row.cluster,
                code_layout=2 if row.build.startswith("compact") else 1, max_slices=row.slices)


def build_of(q, n):
    """The build a launch of n objects with query_launch result q runs (pick_build in sq_kernels.cu): the compact
    layout's 256-thread build; up to 512 threads with every CTA alone on its SM, the solo build; else the smallest
    straight-line build that holds the CTA."""
    if q["code_layout"] == 2:
        return "compact 256"
    if n * q["cluster"] <= N_SMS and q["threads"] <= 512:
        return "solo 512"
    return "plain %d" % next(t for t in (256, 512, 1024) if q["threads"] <= t)


def test_shapes_select_their_builds():
    """query_launch on the CPU: every row keeps its CTA size, cluster, code layout, slices, resident CTAs per SM (1 for
    the solo build's 128 registers, 2 for two 512-thread CTAs at 64) and shared memory -- with it the staging decision.
    The rows together cover all five production builds, and staged and unstaged launches in both regimes."""
    from odam_b200 import api
    covered = set()
    for row in SHAPES + LATENCY:
        counts = view_counts(row)
        q = api.query_launch(_offsets(counts), **row.options)
        assert q == expected_launch(row), (row.name, q)
        assert build_of(q, len(counts)) == row.build, row.name
        dense = len(counts) * q["cluster"] > N_SMS
        assert dense == (row in SHAPES), row.name
        longest = -(-int(counts.max()) // q["cluster"])   # views of the longest track a CTA holds
        if longest <= row.threads:
            assert row.smem_bytes == UNSTAGED_SMEM[row.threads] + row.staged * _staging_bytes(longest), row.name
        else:
            assert longest > 256 and not row.staged, row.name   # a CTA with more than 256 views is never staged
        covered.add((row.build, dense, row.staged))
    assert {b for b, _, _ in covered} == BUILDS
    assert {(d, s) for _, d, s in covered} == {(True, True), (True, False), (False, True), (False, False)}
    # the staging edge of the mixed rows: with tracks of 240 views instead of 256, four CTAs' staging areas fit
    q = api.query_launch(_offsets(view_counts(SHAPES[-2]._replace(groups=((290, 20), (10, 240))))))
    assert (q["threads"], q["code_layout"], q["smem_bytes"]) == (256, 2, 56992)
    assert q["smem_bytes"] == UNSTAGED_SMEM[256] + _staging_bytes(240)


@pytest.fixture(scope="module")
def api():
    from odam_b200 import api
    return api


@pytest.fixture(scope="module")
def coracle():
    from oracle import c_oracle
    c_oracle.build()
    return c_oracle


@pytest.fixture(scope="module")
def _wall_time():
    t0 = time.time()
    yield
    print(f"\ntests/test_launch_shapes_gpu.py wall time {time.time() - t0:.1f} s")


_scenes = {}


def _tracks(row):
    """The row's batch: objects of synthetic scenes (one scene per group), the edge objects swapped in."""
    from odam_b200 import synthetic
    from odam_b200.api import init_params
    scenes = []
    for g, (m, V) in enumerate(row.groups):
        if (m, V) not in _scenes:
            _scenes[m, V] = synthetic.make_scene(m, V, seed=40 + V, device="cuda:0")
        scenes.append(_scenes[m, V])
    taken = [0] * len(scenes)
    objs = []
    for g in _group_of(row.groups):
        sc, j = scenes[g], taken[g]
        taken[g] += 1
        objs.append((init_params(sc.translate[j], sc.angle[j], sc.dims[j]), sc.P_cws[j].reshape(-1, 12), sc.box[j],
                     sc.mask[j], sc.cls[j]))
    for kind, p in zip(EDGE_KINDS, _edge_at(len(objs))):
        objs[p] = edge_object(kind)
    tracks = pack(objs)
    assert np.array_equal(np.diff(tracks.view_off), view_counts(row))
    return tracks


@pytest.mark.gpu
@pytest.mark.parametrize("row", SHAPES, ids=[r.name for r in SHAPES])
def test_launch_shape(api, coracle, _wall_time, row):
    import torch
    tracks = _tracks(row)
    prior = api.prior_table()
    q = api.query_launch(tracks.view_off, **row.options)
    assert q == expected_launch(row) and build_of(q, tracks.n) == row.build, (row.name, q)
    fixed = dict(threads=q["threads"], max_slices=q["max_slices"], cluster=q["cluster"])
    edge_at = _edge_at(tracks.n)
    behind = edge_at[EDGE_KINDS.index("behind")]
    rng = np.random.default_rng(SHAPES.index(row))
    pick = np.sort(np.concatenate([rng.choice(np.setdiff1d(np.arange(tracks.n), edge_at), 5, replace=False),
                                   rng.choice(edge_at, 1)]))
    layouts = (1, 2) if q["threads"] <= 256 else (1,)
    dt = api.DeviceTracks(tracks, "cuda:0", prior)
    worst = np.zeros(9)
    replays = 0
    for n_iters in (1, 5):
        label = f"{row.name} iters={n_iters}"
        o, w = check_launch(api, tracks, prior, n_iters, label=label, quiet=True, **row.options)
        worst = np.maximum(worst, w)
        assert not (o["status"] & 3).any(), (label, np.nonzero(o["status"] & 3)[0])
        assert np.array_equal(np.nonzero(o["status"])[0], [behind]) and o["status"][behind] == 4, label
        # an object's trajectory does not depend on its batch: alone it runs the latency-regime build(s)
        for i in pick:
            row_i = object_row(o, tracks.view_off, i)
            alone = tracks.slice(i, i + 1)
            for layout in layouts:
                one = api.optimize_host(alone, prior=prior, n_iters=n_iters, extras=EXTRAS, code_layout=layout, **fixed)
                one = object_row(one, alone.view_off, 0)
                for k in row_i:
                    assert np.array_equal(one[k], row_i[k]), (label, int(i), layout, k)
                replays += 1
        # the device entry (launch options from the host copy of view_off, caller-supplied max_views) with and
        # without the cycle marks
        cyc = torch.zeros((tracks.n, 16), dtype=torch.int64, device="cuda:0")
        plain = api.optimize_device(dt, n_iters=n_iters, **row.options)
        marked = api.optimize_device(dt, n_iters=n_iters, cycles=cyc, **row.options)
        torch.cuda.synchronize()
        for k in ("params", "loss", "status"):
            assert np.array_equal(plain[k].cpu().numpy(), o[k]), (label, "device entry", k)
            assert np.array_equal(marked[k].cpu().numpy(), o[k]), (label, "cycle-mark twin", k)
        c = cyc.cpu().numpy()
        assert (c >= 0).all() and (c.sum(1) > 0).all(), label
    # the first iterations of the sampled objects, read from launches of the whole batch, against the C oracle
    iters = 3
    dec = {k: api.optimize_host(tracks, prior=prior, n_iters=k, extras=DECISIONS, **row.options)
           for k in range(1, iters + 1)}
    flips = []
    for i in pick:
        flip = oracle_first_iterations(coracle, tracks, i, prior, iters,
                                       lambda k: object_row(dec[k], tracks.view_off, i), dec[1]["loss"][i, 0])
        if flip:
            flips.append(flip)
    print(f"\n  {row.name}: {row.build}, {q['threads']} threads, cluster {q['cluster']}, {q['max_slices']} slices, "
          f"{'staged' if row.staged else 'unstaged'}; worst |g - g64| / scale "
          + " ".join(f"{x:.1e}" for x in worst)
          + f"; C oracle: {len(pick) - len(flips)} of {len(pick)} agree, near-tie flips {flips}; {replays} replays "
          f"alone, cycle-mark twin and device entry bit-identical")
    assert len(flips) <= len(pick) // 4, flips
