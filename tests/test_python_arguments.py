"""The Python layer's checked path into the library and its single home for each reference convention.

CPU tests: every host wrapper raises ValueError, before any library call, for an array whose size disagrees with n or
the view offsets (the C entries size their copies from those, not from the arrays), and the vectorised starting row
and line-form helpers agree bit for bit with the per-object forms they replace.  The GPU test covers the tensor
checks of optimize_device and DeviceTracks."""
import os

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REPRS = ("super_quadric", "cube", "quadric")


def _tracks():
    from odam_b200 import api, synthetic
    return api.pack_scene(synthetic.make_scene(3, 5, seed=1))


def _replace(tracks, **kw):
    from odam_b200 import api
    d = dict(init=tracks.init, cls=tracks.cls, view_off=tracks.view_off, Ms=tracks.Ms, box=tracks.box, mask=tracks.mask)
    d.update(kw)
    return api.PackedTracks(**d)


def _row(translate, angle, dims, representation):
    """One object's starting row, written out as the reference builds it (sq_libs.py:353-369)."""
    p = np.empty(9, np.float32)
    p[0:3] = np.asarray(translate, np.float64)
    p[3] = np.float64(angle)
    p[4:7] = np.sqrt(np.asarray(dims, np.float64) / 2)
    p[7:9] = -10000.0 if representation == "cube" else -0.0
    return p


def _lines(box, mask):
    """The reference's line dicts, written out side by side (quadric_helper.py:69-109)."""
    names = ("x_min", "x_max", "y_min", "y_max")
    return [{n: (np.array([1, 0, -float(b[s])]) if n[0] == "x" else np.array([0, 1, -float(b[s])]))
             for s, n in enumerate(names) if m[s]} for b, m in zip(box, mask)]


def _same_lines(a, b):
    return len(a) == len(b) and all(
        x.keys() == y.keys() and all(x[k].dtype == y[k].dtype and x[k].tobytes() == y[k].tobytes() for k in x)
        for x, y in zip(a, b))


def _bad_calls():
    from odam_b200 import api
    f32 = lambda *s: np.ones(s, np.float32)
    voff = np.array([0, 2, 5], np.int32)
    tr = _tracks()
    n, SV = tr.n, tr.total_views
    return {
        "project_boxes: view_off past Ms": lambda: api.project_boxes_host(f32(1, 9), np.array([0, 50], np.int32), f32(1, 12)),
        "project_boxes: view_off shorter than n + 1": lambda: api.project_boxes_host(f32(3, 9), voff[:2], f32(2, 12)),
        "project_boxes: view_off longer than n + 1": lambda: api.project_boxes_host(f32(1, 9), voff, f32(5, 12)),
        "project_boxes: params not rows of 9": lambda: api.project_boxes_host(f32(2, 8), voff, f32(5, 12)),
        "sample_on_batch: fewer epsilons": lambda: api.sample_on_batch(f32(4, 1, 3), f32(1, 1, 2)),
        "sample_on_batch: shapes not triples": lambda: api.sample_on_batch(f32(4, 1, 2), f32(4, 1, 2)),
        "optimize_host: view_off shorter than n + 1": lambda: api.optimize_host(_replace(tr, view_off=tr.view_off[:2])),
        "optimize_host: init rows": lambda: api.optimize_host(_replace(tr, init=tr.init[:2])),
        "optimize_host: Ms rows": lambda: api.optimize_host(_replace(tr, Ms=tr.Ms[:-1])),
        "optimize_host: box rows": lambda: api.optimize_host(_replace(tr, box=tr.box[:-1])),
        "optimize_host: mask rows": lambda: api.optimize_host(_replace(tr, mask=tr.mask[:-1])),
        "optimize_host: prior [9]": lambda: api.optimize_host(tr, prior=f32(9)),
        "optimize_host: m0 rows": lambda: api.optimize_host(tr, m0=f32(n - 1, 9), v0=f32(n, 9), step0=1),
        "optimize_host: s0 columns": lambda: api.optimize_host(tr, s0=f32(n, 2)),
        "oriented_boxes_of_points: last axis 4": lambda: api.oriented_boxes_of_points_host(f32(2, 10, 4)),
        "oriented_boxes_of_points: one set, last axis 2": lambda: api.oriented_boxes_of_points_host(f32(10, 2)),
        "sample_points: params not rows of 9": lambda: api.sample_points_host(f32(10)),
        "oriented_boxes: params not rows of 9": lambda: api.oriented_boxes_host(f32(2, 8)),
        "merge_cost: boxes not [n, 8, 3]": lambda: api.merge_cost_host(np.ones((2, 8, 2))),
        "merge_cost: one class per box": lambda: api.merge_cost_host(np.ones((3, 8, 3)), np.zeros(2, np.int32)),
        "optimize_host: Ms longer than view_off[-1]": lambda: api.optimize_host(_replace(tr, Ms=np.ones((SV + 1, 12)))),
    }


@pytest.mark.parametrize("case", sorted(_bad_calls()))
def test_mismatched_host_arrays_raise_value_error(case):
    with pytest.raises(ValueError, match="must have shape"):
        _bad_calls()[case]()


def test_offsets_that_decrease_stay_the_entrys_error():
    """Start-at-0 and monotone offsets are the C entry's check (ODAM_SQ_ERR_ARG, before any CUDA call)."""
    from odam_b200 import _lib, api
    for bad, rows in (([0, -4], 1), ([1, 5], 5), ([0, 5, 3], 3)):
        with pytest.raises(_lib.OdamSqError, match="invalid argument"):
            api.project_boxes_host(np.ones((len(bad) - 1, 9), np.float32), np.array(bad, np.int32),
                                   np.ones((rows, 12), np.float32))


def test_host_array_keeps_dtype_contiguity_and_none():
    from odam_b200 import _lib
    a = np.arange(24, dtype=np.float64).reshape(4, 6)[:, ::2]           # strided
    b = _lib.host_array("a", a, np.float32, (3, 4))
    assert b.dtype == np.float32 and b.flags.c_contiguous and b.shape == (3, 4)
    assert np.array_equal(b.reshape(-1), a.reshape(-1).astype(np.float32))
    assert _lib.host_array("a", None, np.float32, (3, 4)) is None
    with pytest.raises(ValueError, match=r"a must have shape \[5, 4\], got \[4, 3\]"):
        _lib.host_array("a", a, np.float32, (5, 4))


@pytest.mark.parametrize("representation", REPRS)
def test_init_params_vectorised_matches_rows(representation):
    from odam_b200 import api
    rng = np.random.default_rng(4)
    n = 37
    T, A, D = rng.normal(0, 3, (n, 3)), rng.uniform(-4, 4, n), rng.uniform(0.05, 2, (n, 3))
    want = np.stack([_row(T[i], A[i], D[i], representation) for i in range(n)])
    got = api.init_params(T, A, D, representation)
    assert got.shape == (n, 9) and got.dtype == np.float32 and got.tobytes() == want.tobytes()
    assert api.init_params(T[5], A[5], D[5], representation).tobytes() == want[5].tobytes()
    assert api.init_params(T[:0], A[:0], D[:0], representation).shape == (0, 9)
    with pytest.raises(AssertionError):
        api.init_params(T, A, D, "sphere")


@pytest.mark.parametrize("representation", REPRS)
def test_pack_scene_and_optimizer_rows_match_per_object_rows(representation):
    from odam_b200 import api, synthetic
    from odam_b200.sq_libs import SuperQuadricOptimizer
    scene = synthetic.make_scene(6, 8, seed=9)
    want = np.stack([_row(scene.translate[i], scene.angle[i], scene.dims[i], representation) for i in range(scene.n)])
    assert api.pack_scene(scene, representation).init.tobytes() == want.tobytes()
    for i in range(scene.n):
        opt = SuperQuadricOptimizer(scene.translate[i], scene.angle[i], scene.dims[i], int(scene.cls[i]), representation,
                                    True)
        assert opt.Q_init.params().tobytes() == want[i].tobytes() and opt.Q_init.obj_class == int(scene.cls[i])


def test_track_quadric_params_match_per_track_rows():
    from odam_b200 import processor
    G = np.load(os.path.join(REPO, "tests", "golden", "prepare_tracks.npz"))
    tracks = [G[f"t{t}_track"] for t in range(6)]
    want = np.stack([_row(np.mean(t[:, 9:12], axis=0), np.mean(t[:, 12], axis=0),
                          np.clip(np.mean(t[:, 6:9], axis=0), a_min=0.05, a_max=np.inf), "super_quadric") for t in tracks])
    assert processor.track_quadric_params(tracks).tobytes() == want.tobytes()
    assert processor.track_quadric_params([]).shape == (0, 9)


def test_line_form_round_trips_synthetic_scenes():
    from odam_b200 import api, synthetic
    scene = synthetic.make_scene(4, 12, seed=2)
    for i in range(scene.n):
        lines = scene.gt_lines(i)
        assert _same_lines(lines, _lines(scene.box[i], scene.mask[i]))
        box, mask = api.pack_lines(lines)
        assert mask.tobytes() == scene.mask[i].tobytes()
        assert box.tobytes() == np.where(scene.mask[i] > 0, scene.box[i], 0).astype(np.float32).tobytes()
        back = api.unpack_lines(box, mask)
        assert _same_lines(back, _lines(box, mask))
        assert all(b.tobytes() == m.tobytes() for b, m in zip(api.pack_lines(back), (box, mask)))


def test_line_form_round_trips_call_site_stages():
    from odam_b200 import api
    from odam_b200.run_multi_view import lines_of, stage_object
    G = np.load(os.path.join(REPO, "tests", "golden", "call_site.npz"))
    for t in range(4):
        s = stage_object(G[f"t{t}_track"], G["frame_ids"], 968, 1296)
        lines = lines_of(s)
        assert _same_lines(lines, _lines(s["box"], s["mask"]))
        box, mask = api.pack_lines(lines)
        assert box.tobytes() == s["box"].tobytes() and mask.tobytes() == s["mask"].tobytes()
        assert _same_lines(api.unpack_lines(box, mask), lines)


@pytest.mark.gpu
def test_device_tensor_checks():
    """optimize_device checks a reused out, cycles and corners against n, n_iters and the tracks' device before the
    launch; DeviceTracks shapes the prior as [8, 9]."""
    import torch
    from odam_b200 import api
    tr = _tracks()
    dev = torch.device("cuda:0")
    dt = api.DeviceTracks(tr, dev, api.prior_table())
    out = api.optimize_device(dt, n_iters=5)
    first = {k: v.clone() for k, v in out.items()}
    assert api.optimize_device(dt, n_iters=5, out=out) is out
    torch.cuda.synchronize()
    assert all(torch.equal(first[k], out[k]) for k in first)
    n = tr.n
    bad = {
        "loss for other n_iters": dict(n_iters=6, out=out),
        "status of another dtype": dict(n_iters=5, out=dict(out, status=out["status"].long())),
        "params not contiguous": dict(n_iters=5, out=dict(out, params=torch.empty((9, n), device=dev).t())),
        "params on the host": dict(n_iters=5, out=dict(out, params=out["params"].cpu())),
        "cycles [n, 15]": dict(cycles=torch.zeros((n, 15), dtype=torch.int64, device=dev)),
        "cycles int32": dict(cycles=torch.zeros((n, 16), dtype=torch.int32, device=dev)),
        "corners [n + 1, 8, 3]": dict(corners=torch.zeros((n + 1, 8, 3), dtype=torch.float64, device=dev)),
        "corners float32": dict(corners=torch.zeros((n, 8, 3), dtype=torch.float32, device=dev)),
    }
    for name, kw in bad.items():
        with pytest.raises(ValueError, match="must be a contiguous"):
            api.optimize_device(dt, **kw)
    torch.cuda.synchronize()
    assert all(torch.equal(first[k], out[k]) for k in first), "a rejected call wrote into out"
    with pytest.raises(ValueError, match=r"prior must have shape \[8, 9\]"):
        api.DeviceTracks(tr, dev, api.prior_table()[0])
