"""CPU tests of the drop-in boundary: the C-ABI library loads and exports every symbol include/odam_sq.h declares,
the product package never touches oracle/, and the host-side mirror of the reference interface behaves."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from odam_b200 import build
    build.build()
    from odam_b200 import _lib
    return _lib.load()


def test_header_is_plain_c_and_links(lib, tmp_path):
    """The boundary is a C ABI: the header compiles as strict C99 and a C program links against the library
    (no C++ or torch types in the signatures).  The program only calls the no-GPU housekeeping entries."""
    from odam_b200 import _lib
    src = tmp_path / "abi.c"
    src.write_text('''#include <stdio.h>
#include <string.h>
#include "odam_sq.h"
int main(void) {
    odam_sq_options o;
    memset(&o, 0, sizeof o);
    int32_t voff[3] = {0, 20, 40};
    int threads = 0, layout = 0, slices = 0;
    if (odam_sq_abi_version() != ODAM_SQ_ABI_VERSION) return 1;
    if (odam_sq_query_launch(voff, 2, &o, &threads, NULL, NULL, NULL, &layout, &slices) != 0) return 2;
    if (odam_sq_optimize_host(NULL, NULL, NULL, NULL, NULL, NULL, NULL, 1, 1, 0, 0.01f, 0.1f, NULL, NULL, NULL, NULL, 0) >= 0) return 3;
    printf("%d %d %d %s\\n", threads, layout, slices, odam_sq_error_string(-1));
    return 0;
}
''')
    exe = tmp_path / "abi"
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(REPO, "include"),
                    str(src), "-o", str(exe), "-L", libdir, "-lodam_sq", f"-Wl,-rpath,{libdir}"], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stderr)
    threads, layout, slices = (int(x) for x in r.stdout.split()[:3])
    assert threads % 32 == 0 and layout in (1, 2) and 1 <= slices <= 25


def test_graft_entry_build():
    """The driver's "does it build" check: every native piece compiles for sm_100a and the package imports."""
    sys.path.insert(0, REPO)
    import __graft_entry__
    __graft_entry__.build()


def test_header_symbols_exported(lib):
    hdr = open(os.path.join(REPO, "include", "odam_sq.h")).read()
    declared = set(re.findall(r"\b(odam_sq_[a-z_0-9]+)\s*\(", hdr))
    assert {"odam_sq_optimize", "odam_sq_optimize_host", "odam_sq_sample_points_host",
            "odam_sq_sample_on_batch_host", "odam_sq_project_boxes_host"} <= declared
    for name in declared:
        assert hasattr(lib, name), name
    from odam_b200 import _lib
    assert set(_lib.EXPORTS) == declared
    assert lib.odam_sq_abi_version() == 4
    assert lib.odam_sq_error_string(-1) == b"invalid argument"


def test_options_struct_layout_matches_header():
    """ctypes mirror of odam_sq_options: field order/names as in the header."""
    from odam_b200 import _lib
    hdr = open(os.path.join(REPO, "include", "odam_sq.h")).read()
    body = hdr[hdr.index("typedef struct odam_sq_options {"):hdr.index("} odam_sq_options;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\b\*?\s*([a-z_0-9]+)\s*;", body)
    assert names == [f[0] for f in _lib.Options._fields_]


def test_argument_validation_without_gpu(lib):
    """Bad arguments are rejected before any CUDA call (so this runs on a CPU-only box)."""
    z = ctypes.c_void_p(0)
    assert lib.odam_sq_optimize_host(z, z, z, z, z, z, z, 1, 1, 0, 0.01, 0.1, z, z, z, None, 0) == -1
    assert lib.odam_sq_sample_on_batch_host(z, z, z, z, 1, 1, 1000, 201, 0, 0) == -1
    a = np.zeros(3, np.float32)
    p = a.ctypes.data_as(ctypes.c_void_p)
    assert lib.odam_sq_sample_on_batch_host(p, p, p, p, 1, 1, 999, 201, 0, 0) == -1   # only N=1000 / 201 / seed 0
    th, sm, c, cl, lay = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    voff = np.array([0, 20, 40], np.int32)
    assert lib.odam_sq_query_launch(voff.ctypes.data_as(ctypes.c_void_p), 2, None, ctypes.byref(th), ctypes.byref(sm),
                                    ctypes.byref(c), ctypes.byref(cl), ctypes.byref(lay), None) == 0
    assert th.value % 32 == 0 and 32 <= th.value <= 1024 and sm.value > 0 and c.value >= 1 and cl.value in (1, 2, 3, 4)
    assert lay.value == 1   # two objects never share an SM: the straight-line build
    voff = np.arange(0, 20 * 1001, 20, dtype=np.int32)   # 1000 short tracks: several CTAs per SM, compact build
    assert lib.odam_sq_query_launch(voff.ctypes.data_as(ctypes.c_void_p), 1000, None, ctypes.byref(th), None, None,
                                    None, ctypes.byref(lay), None) == 0
    assert lay.value == 2 and th.value == 256


@pytest.mark.parametrize("n, views, threads, ctas_per_sm", [
    (50, 20, 512, 1),      # latency regime, the solo build: 128 registers per thread
    (4, 3000, 768, 1),     # latency regime, wider than the solo build: the 1024-thread build
    (160, 20, 512, 2),     # dense, two wide CTAs per SM
    (300, 300, 320, 3),    # dense, long tracks
    (1000, 20, 256, 4),    # dense, the compact build
])
def test_query_launch_ctas_per_sm(lib, n, views, threads, ctas_per_sm):
    """The resident CTAs per SM that odam_sq_query_launch reports (bench.py's launch record) follow the register budget
    of the build the optimiser launches."""
    from odam_b200 import api
    q = api.query_launch(np.arange(0, views * (n + 1), views, dtype=np.int32))
    assert (q["threads"], q["ctas_per_sm"]) == (threads, ctas_per_sm)


@pytest.mark.parametrize("n, views", [(50, 20), (160, 20), (300, 300)])
def test_compact_layout_wider_than_its_builds_is_rejected(lib, n, views):
    """The compact layout has builds of up to 256 threads.  Forced onto a batch for which the library picks wider CTAs
    (latency regime, two wide CTAs per SM, long dense tracks), it is an invalid argument, as it is with the wide CTA
    size given -- not a configuration without a kernel."""
    from odam_b200 import _lib, api
    voff = np.arange(0, views * (n + 1), views, dtype=np.int32)
    for threads in (0, 512):
        with pytest.raises(_lib.OdamSqError, match="invalid argument"):
            api.query_launch(voff, threads=threads, code_layout=2)
    q = api.query_launch(voff, threads=256, code_layout=2)
    assert (q["threads"], q["code_layout"]) == (256, 2)


def test_no_gpu_means_loud_failure_not_fallback(lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("has a GPU")
    from odam_b200 import _lib, api, synthetic
    tracks = api.pack_scene(synthetic.make_scene(2, 10, seed=3))
    with pytest.raises(_lib.OdamSqError):
        api.optimize_host(tracks, n_iters=1)


def test_product_never_imports_oracle():
    """Static: no file under odam_b200/ mentions the oracle package; dynamic: importing the product does not load it."""
    for root, _, files in os.walk(os.path.join(REPO, "odam_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+(\.+)?oracle\b", txt, re.M), f
                assert not re.search(r"sq_oracle|c_oracle|torch_oracle|libsq_oracle", txt), f
    code = ("import sys; sys.path.insert(0, %r); import odam_b200.sq_libs, odam_b200.run_multi_view, odam_b200.api; "
            "assert not any(m == 'oracle' or m.startswith('oracle.') for m in sys.modules)" % REPO)
    subprocess.run([sys.executable, "-c", code], check=True)


def test_packing_mirrors_reference_line_dicts():
    from odam_b200 import api, synthetic
    scene = synthetic.make_scene(3, 12, seed=2)
    tr = api.pack_scene(scene)
    for i in range(3):
        box, mask = api.pack_lines(scene.gt_lines(i))
        a, b = tr.view_off[i], tr.view_off[i + 1]
        assert np.array_equal(mask, tr.mask[a:b]) and np.array_equal(box[mask > 0], tr.box[a:b][mask > 0])
    p = api.init_params([1, 2, 3], 0.5, [0.5, 0.72, 0.98], "cube")
    assert np.allclose(p[4:7], np.sqrt(np.array([0.5, 0.72, 0.98]) / 2)) and np.all(p[7:9] == -10000)
    assert np.signbit(api.init_params([0, 0, 0], 0, [1, 1, 1])[7])  # shapes start at -0.0 (sq_libs.py:369)
    sub = tr.slice(1, 3)
    assert sub.n == 2 and sub.view_off[0] == 0 and sub.total_views == tr.view_off[3] - tr.view_off[1]


def test_prior_table_matches_reference_data(golden_runs):
    from odam_b200 import api
    tab = api.prior_table()
    assert tab.shape == (8, 9)
    assert np.array_equal(tab, golden_runs["prior_by_class"].astype(np.float32).reshape(8, 9))


def test_optimizer_constructor_mirrors_reference():
    from odam_b200.sq_libs import SuperQuadricOptimizer
    o = SuperQuadricOptimizer(np.array([0.1, 0.2, 0.3]), 0.4, np.array([0.5, 0.6, 0.7]), 5, "super_quadric", True)
    q = o.Q_init
    assert q.obj_class == 5 and o.use_prior and o.loss_log == []
    assert q.scales.dtype.is_floating_point and q.scales.requires_grad and q.translate.requires_grad
    assert np.allclose(q.scales.detach().numpy(), np.sqrt(np.array([0.5, 0.6, 0.7]) / 2).astype(np.float32))
    assert set(o.scale_prior) == {"03211117", "04379243", "02808440", "02747177", "04256520", "03001627", "02933112",
                                  "02871439"}
    with pytest.raises(AssertionError):
        SuperQuadricOptimizer(np.zeros(3), 0.0, np.ones(3), 0, "sphere", True)
    import pickle
    q2 = pickle.loads(pickle.dumps(q))   # results are pickled per sequence (run_processor.py:85-92)
    assert np.array_equal(q2.params(), q.params())


def test_prepare_tracks_projection_matches_reference():
    """odam_b200.processor against the reference's own _prepare_tracks loop body (tests/golden/prepare_tracks.npz):
    the float64 camera transform / projection / min-max is bit-identical on the reference's points, and the
    mean-pose quadric (dims clipped at 0.05) gives the reference's surface to fp32 rounding."""
    from odam_b200 import processor
    from oracle import c_oracle
    c_oracle.build()
    G = np.load(os.path.join(REPO, "tests", "golden", "prepare_tracks.npz"))
    for t in range(6):
        box = processor.project_points_reference_way(G[f"t{t}_pts"], G["T_wc"], G["K"])
        assert np.array_equal(box, G[f"t{t}_box"]), t
        P = processor.track_quadric_params([G[f"t{t}_track"]])
        pts = c_oracle.points(P[0]).astype(np.float32)
        assert np.abs(pts - G[f"t{t}_pts"]).max() <= 5e-7, t
        assert np.abs(processor.project_points_reference_way(pts, G["T_wc"], G["K"]) - G[f"t{t}_box"]).max() <= 1e-3


def test_loss_log_reads_like_the_references_list():
    """loss_log keeps floats and hands out the reference's [tensor] entries (sq_libs.py:471) when read."""
    import torch
    from odam_b200.sq_libs import LossLog
    log = LossLog()
    assert log == [] and len(log) == 0
    log.extend_values(np.array([1.5, 0.25, 3.0], np.float32))
    log.append([torch.tensor(7.0)])   # the reference's own form still works
    assert len(log) == 4 and isinstance(log, list)
    assert isinstance(log[0], list) and torch.is_tensor(log[0][0]) and log[0][0].dtype == torch.float32
    assert [float(e[0]) for e in log] == [1.5, 0.25, 3.0, 7.0]
    assert [float(e[0]) for e in log[1:3]] == [0.25, 3.0] and float(log[-1][0]) == 7.0
    assert np.array_equal(log.values(), np.array([1.5, 0.25, 3.0, 7.0], np.float32))


def test_call_site_staging_matches_reference():
    """stage_object / get_3d_box / compute_oriented_bbox against outputs of the reference's own helpers."""
    from odam_b200 import api
    from odam_b200.postprocess import compute_oriented_bbox, get_3d_box
    from odam_b200.run_multi_view import stage_object
    from scipy.spatial.transform import Rotation
    G = np.load(os.path.join(REPO, "tests", "golden", "call_site.npz"))
    for t in range(4):
        s = stage_object(G[f"t{t}_track"], G["frame_ids"], 968, 1296)
        assert s["obj_class"] == int(G[f"t{t}_class"])
        assert np.allclose(s["t_wo"], G[f"t{t}_T_wo"][:3, 3]) and np.allclose(s["R"], G[f"t{t}_T_wo"][:3, :3])
        assert np.allclose(s["dims"], G[f"t{t}_dims"])
        assert np.array_equal(np.array(s["valid_frames"]), G[f"t{t}_valid"])
        assert np.array_equal(s["mask"], G[f"t{t}_mask"]) and np.array_equal(s["box"], G[f"t{t}_box"].astype(np.float32))
        from odam_b200.run_multi_view import lines_of
        box, mask = api.pack_lines(lines_of(s))            # and through the reference's dict form
        assert np.array_equal(mask, s["mask"]) and np.array_equal(box, s["box"])
        assert np.isclose(Rotation.from_matrix(s["R"]).as_euler("zxy")[0], float(G[f"t{t}_yaw"]))
        assert np.allclose(get_3d_box(s["dims"], s["R"], s["t_wo"]), G[f"t{t}_bbox_dl"])
    for k in range(6):
        assert np.allclose(compute_oriented_bbox(G[f"obb{k}_pts"]), G[f"obb{k}_box"], atol=1e-9)


def test_batched_staging_matches_reference_call_site():
    """stage_tracks (all tracks at once) against what the reference's own optim_process derived before optimising
    (tests/golden/optim_process.npz): the detector boxes of every track, and -- for the track with too few views, which
    the reference returns un-optimised -- the initial quadric bit for bit."""
    from odam_b200.run_multi_view import boxes_3d, stage_object, stage_tracks
    G = np.load(os.path.join(REPO, "tests", "golden", "optim_process.npz"))
    n = len(G["rows"])
    tracks = [G[f"track{i}"] for i in range(n)]
    st = stage_tracks(tracks, G["img_names"], int(G["img_h"]), int(G["img_w"]))
    assert np.array_equal(st["cls"], G["obj_class"])
    assert np.abs(boxes_3d(st["dims"], st["yaw"], st["t_wo"]) - G["bboxes_dl"]).max() < 1e-12
    short = int(np.argmin(G["rows"]))
    init = np.concatenate([st["t_wo"][short], [st["yaw"][short]], np.sqrt(st["dims"][short] / 2), [-0.0, -0.0]]).astype(np.float32)
    assert np.array_equal(init, G["quadrics"][short])
    for i in range(n):   # one by one == all at once
        s1 = stage_object(tracks[i], G["img_names"], int(G["img_h"]), int(G["img_w"]))
        a, b = st["view_off"][i], st["view_off"][i + 1]
        assert np.array_equal(s1["box"], st["box"][a:b]) and np.array_equal(s1["mask"], st["mask"][a:b])
        assert s1["valid_frames"] == st["frame_idx"][a:b].tolist() and s1["yaw"] == st["yaw"][i]
    # shuffled rows, a duplicated frame (the first row wins, tracking_gt_utils.py:181) and unsorted frame ids
    rng = np.random.default_rng(0)
    t0 = tracks[0]
    dup = np.concatenate([t0, t0[3:4] + np.array([0.0] + [1.0] * 81)[None]])
    perm = rng.permutation(len(G["img_names"]))
    a = stage_tracks([dup], G["img_names"][perm], int(G["img_h"]), int(G["img_w"]))
    b = stage_tracks([t0], G["img_names"], int(G["img_h"]), int(G["img_w"]))
    order = np.argsort(perm[a["frame_idx"]])
    assert np.array_equal(perm[a["frame_idx"]][order], b["frame_idx"]) and np.array_equal(a["box"][order], b["box"])
    assert stage_tracks([], G["img_names"], 968, 1296)["view_off"].tolist() == [0]


def test_native_staging_matches_numpy_mirror_and_numpy_mean():
    """odam_sq_stage_tracks_host (one native pass over the rows of all tracks) against its vectorised numpy mirror on
    random ragged tracks -- frames outside frame_ids, duplicated frames, empty tracks, permuted frame ids, boxes across
    the 20 px border -- and the mean centre against the reference's own expression np.mean(track[:, 9:12], axis=0)
    (tracking_gt_utils.py:155), bit for bit."""
    from odam_b200.run_multi_view import stage_tracks, stage_tracks_numpy
    rng = np.random.default_rng(5)
    for trial in range(60):
        n, F = int(rng.integers(0, 12)), int(rng.integers(1, 40))
        tracks = []
        for i in range(n):
            R = int(rng.integers(0 if i % 7 == 3 else 1, F + 5))
            t = -np.ones((R, 82))
            t[:, 0], t[:, 1] = rng.integers(-2, F + 3, R), rng.integers(0, 8, R)
            x0, y0 = rng.uniform(-30, 1200, R), rng.uniform(-30, 900, R)
            t[:, 2], t[:, 3], t[:, 4], t[:, 5] = x0, y0, x0 + rng.uniform(5, 400, R), y0 + rng.uniform(5, 300, R)
            t[:, 6:9], t[:, 9:12], t[:, 12] = rng.uniform(0.2, 2, (R, 3)), rng.uniform(-3, 3, (R, 3)), rng.uniform(-4, 4, R)
            tracks.append(t)
        fid = rng.permutation(F + 2)[:F]
        a, b = stage_tracks(tracks, fid, 968, 1296), stage_tracks_numpy(tracks, fid, 968, 1296)
        full = np.array([len(t) > 0 for t in tracks], bool)
        assert np.array_equal(a["cls"][full], b["cls"][full])
        for k in ("view_off", "frame_idx", "box", "mask", "n_present"):
            assert np.array_equal(a[k], b[k]), (trial, k)
        for k in ("t_wo", "yaw", "dims"):
            assert np.allclose(a[k], b[k], rtol=0, atol=1e-14), (trial, k)
        for i, t in enumerate(tracks):
            if len(t):
                assert np.array_equal(a["t_wo"][i], np.mean(t[:, 9:12], axis=0))
