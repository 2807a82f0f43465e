"""Array-level Python API over the C ABI (include/odam_sq.h): packed tracks in, optimised parameters out.

Two flavours, both one persistent CUDA launch for all objects:
  optimize_host(...)    numpy arrays on the host; H2D/D2H happen inside the library call
                        (this is what the SuperQuadricOptimizer drop-in uses)
  optimize_device(...)  torch CUDA tensors, enqueued on torch's current stream, no synchronisation
"""
import ctypes as C
import json
import os
from dataclasses import dataclass

import numpy as np

from . import _lib

SIDES = ("x_min", "x_max", "y_min", "y_max")
CLASS_MAPPER = {0: "03211117", 1: "04379243", 2: "02808440", 3: "02747177",
                4: "04256520", 5: "03001627", 6: "02933112", 7: "02871439"}  # reference sq_libs.py:13-22


@dataclass
class PackedTracks:
    """CSR-packed inputs of n objects (layouts: include/odam_sq.h)."""
    init: np.ndarray      # [n,9]  f32
    cls: np.ndarray       # [n]    i32
    view_off: np.ndarray  # [n+1]  i32
    Ms: np.ndarray        # [SV,12] f32
    box: np.ndarray       # [SV,4] f32
    mask: np.ndarray      # [SV,4] u8

    @property
    def n(self):
        return int(self.cls.shape[0])

    @property
    def total_views(self):
        return int(self.view_off[-1])

    def slice(self, lo, hi):
        """Objects [lo, hi) as their own packed problem (used to shard by object across GPUs)."""
        a, b = int(self.view_off[lo]), int(self.view_off[hi])
        return PackedTracks(self.init[lo:hi].copy(), self.cls[lo:hi].copy(),
                            (self.view_off[lo:hi + 1] - a).astype(np.int32), self.Ms[a:b].copy(),
                            self.box[a:b].copy(), self.mask[a:b].copy())


def init_params(translate, angle, dims, representation="super_quadric"):
    """What SuperQuadricOptimizer.__init__ builds (reference sq_libs.py:353-369): [t3, yaw, sqrt(dims/2), h2].
    translate [..., 3], angle [...], dims [..., 3] -> [..., 9] float32 (one object's values give [9])."""
    assert representation in ("cube", "super_quadric", "quadric")
    angle = np.asarray(angle, np.float64)
    p = np.empty(angle.shape + (9,), np.float32)
    p[..., 0:3] = np.asarray(translate, np.float64)
    p[..., 3] = angle
    p[..., 4:7] = np.sqrt(np.asarray(dims, np.float64) / 2)
    p[..., 7:9] = -10000.0 if representation == "cube" else -0.0
    return p


def pack_lines(gt_lines):
    """list[V] of {side: line} -> (box[V,4] f32, mask[V,4] u8); the target is -line[-1] after the
    reference's float32 store (sq_libs.py:438-451)."""
    V = len(gt_lines)
    box = np.zeros((V, 4), np.float32)
    mask = np.zeros((V, 4), np.uint8)
    for v, d in enumerate(gt_lines):
        for s, name in enumerate(SIDES):
            if name in d:
                box[v, s] = -np.float32(d[name][-1])
                mask[v, s] = 1
    return box, mask


def unpack_lines(box, mask):
    """The inverse of pack_lines: (box[V,4], mask[V,4]) -> the reference's list[V] of {side: line}, with the float64
    lines [1, 0, -x] and [0, 1, -y] of quadric_helper.py:69-109 for the sides the mask keeps."""
    return [{name: np.array([1, 0, -float(v)] if name[0] == "x" else [0, 1, -float(v)])
             for name, v, keep in zip(SIDES, b, m) if keep} for b, m in zip(box, mask)]


def pack_scene(scene, representation="super_quadric"):
    """odam_b200.synthetic.Scene -> PackedTracks."""
    n, V = scene.n, scene.V
    init = init_params(scene.translate, scene.angle, scene.dims, representation)
    return PackedTracks(init=init, cls=scene.cls.astype(np.int32),
                        view_off=(np.arange(n + 1) * V).astype(np.int32),
                        Ms=np.ascontiguousarray(scene.P_cws.reshape(n * V, 12), np.float32),
                        box=np.ascontiguousarray(scene.box.reshape(n * V, 4), np.float32),
                        mask=np.ascontiguousarray(scene.mask.reshape(n * V, 4), np.uint8))


_prior_cache = {}


def load_scale_prior(path=None):
    """{synset id: 3x3 float64} -- the reference opens ./src/super_quadric/scale_prior relative to the cwd
    (sq_libs.py:388); the same file is honoured here when present, else the packaged export of it."""
    key = path or "default"
    if key not in _prior_cache:
        cand = path or "./src/super_quadric/scale_prior"
        if os.path.exists(cand):
            import pickle
            with open(cand, "rb") as f:
                _prior_cache[key] = {k: np.asarray(v, np.float64) for k, v in pickle.load(f).items()}
        elif path is not None:
            raise FileNotFoundError(path)
        else:
            with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "scale_prior.json")) as f:
                _prior_cache[key] = {k: np.asarray(v, np.float64) for k, v in json.load(f)["matrices"].items()}
    return _prior_cache[key]


def prior_table(path=None):
    """[8,9] float32, row = class id (float32 cast as at sq_libs.py:390-391)."""
    pr = load_scale_prior(path)
    return np.stack([np.asarray(pr[CLASS_MAPPER[c]], np.float64).astype(np.float32).reshape(9) for c in range(8)])


def query_launch(view_off, threads=0, max_slices=0, cluster=0, code_layout=0):
    """The launch configuration the library would choose for these tracks (odam_sq_query_launch)."""
    L = _lib.load()
    view_off = np.ascontiguousarray(view_off, np.int32)
    o = _lib.Options()
    o.threads, o.max_slices, o.cluster, o.code_layout = int(threads), int(max_slices), int(cluster), int(code_layout)
    th, sm, cps, cl, lay, ms = (C.c_int() for _ in range(6))
    _lib.check(L.odam_sq_query_launch(_lib.ptr(view_off), len(view_off) - 1, C.byref(o), C.byref(th), C.byref(sm),
                                      C.byref(cps), C.byref(cl), C.byref(lay), C.byref(ms)))
    return dict(threads=th.value, smem_bytes=sm.value, ctas_per_sm=cps.value, cluster=cl.value, code_layout=lay.value,
                max_slices=ms.value)


def cluster_capacity(device=0):
    """{cluster size: objects that can get a cluster of that many CTAs with every CTA alone on its SM}
    (odam_sq_cluster_capacity; 2..4)."""
    L = _lib.load()
    out = {}
    for c in (2, 3, 4):
        v = C.c_int(0)
        _lib.check(L.odam_sq_cluster_capacity(int(device), c, C.byref(v)))
        out[c] = v.value
    return out


def check_classes(cls):
    """KeyError for the first class id outside 0..7: with the prior on, the reference's CLASS_MAPPER lookup
    (sq_libs.py:464) fails the same way."""
    cls = np.asarray(cls)
    bad = cls[(cls < 0) | (cls > 7)]
    if bad.size:
        raise KeyError(int(bad[0]))


def check_finite(status, objects=None):
    """RuntimeError naming the objects whose status has ST_NONFINITE (the reference raises from torch anomaly mode at
    the offending step).  objects[i] is the caller's index of row i (default: i)."""
    bad = np.nonzero(status & _lib.ST_NONFINITE)[0]
    if bad.size:
        raise RuntimeError(f"superquadric optimisation produced NaN/Inf for object(s) "
                           f"{(bad if objects is None else np.asarray(objects)[bad]).tolist()} "
                           "(the reference raises from torch anomaly mode, sq_libs.py:456)")


def _track_arrays(tracks):
    """(init, cls, view_off, Ms, box, mask) of PackedTracks as the optimiser entries read them, each checked against
    n and view_off[-1]."""
    n, a = tracks.n, _lib.host_array
    voff = a("view_off", tracks.view_off, np.int32, (n + 1,))
    SV = int(voff[-1])
    return (a("init", tracks.init, np.float32, (n, 9)), a("cls", tracks.cls, np.int32, (n,)), voff,
            a("Ms", tracks.Ms, np.float32, (SV, 12)), a("box", tracks.box, np.float32, (SV, 4)),
            a("mask", tracks.mask, np.uint8, (SV, 4)))


def optimize_host(tracks, prior=None, n_iters=200, representation="super_quadric", lr=0.01, lr_shape=0.1,
                  device=0, threads=0, max_slices=0, m0=None, v0=None, step0=0, s0=None, extras=(), cluster=0,
                  code_layout=0):
    """Run the fused optimiser on packed host arrays.  Returns dict(params[n,9], loss[n,n_iters], status[n], ...extras).

    prior: None (no prior term) or an [8,9] float32 table (see prior_table()).
    extras: names of optional outputs of odam_sq_options (out_m, out_v, out_grad, out_pred, out_arg,
            out_eta_idx, out_grids, out_param_hist; out_corners (+ out_box_flag): the oriented boxes of the optimised
            objects, computed by a second launch fused behind the optimiser inside the same call).
    """
    L = _lib.load()
    init, cls, voff, Ms, box, mask = _track_arrays(tracks)
    n, SV = len(init), int(voff[-1])
    pr = _lib.host_array("prior", prior, np.float32, (8, 9))
    if pr is not None:
        check_classes(cls)
    o = _lib.Options()
    o.threads, o.max_slices, o.step0, o.cluster = int(threads), int(max_slices), int(step0), int(cluster)
    o.code_layout = int(code_layout)
    keep = dict(m0=_lib.host_array("m0", m0, np.float32, (n, 9)), v0=_lib.host_array("v0", v0, np.float32, (n, 9)),
                s0=_lib.host_array("s0", s0, np.float32, (n, 3)))
    shapes = dict(out_m=((n, 9), np.float32), out_v=((n, 9), np.float32), out_grad=((n, 9), np.float32),
                  out_pred=((SV, 4), np.float32), out_arg=((SV, 4), np.int32),
                  out_eta_idx=((n, _lib.N_SAMPLES), np.uint8), out_grids=((n, 2, _lib.GRID), np.float32),
                  out_param_hist=((n, n_iters, 9), np.float32),
                  out_corners=((n, 8, 3), np.float64), out_box_flag=(n, np.int32))
    keep.update((name, np.zeros(*shapes[name])) for name in extras)
    for name, arr in keep.items():
        setattr(o, name, _lib.ptr(arr))
    out = dict(params=np.zeros((n, 9), np.float32), loss=np.zeros((n, n_iters), np.float32),
               status=np.zeros(n, np.int32))
    rc = L.odam_sq_optimize_host(_lib.ptr(init), _lib.ptr(cls), _lib.ptr(voff), _lib.ptr(Ms), _lib.ptr(box),
                                 _lib.ptr(mask), _lib.ptr(pr), n, n_iters, _lib.REPR[representation],
                                 lr, lr_shape, _lib.ptr(out["params"]), _lib.ptr(out["loss"]),
                                 _lib.ptr(out["status"]), C.byref(o), device)
    _lib.check(rc)
    out.update((name, keep[name]) for name in extras)
    return out


def sample_points_host(params, device=0):
    """compute_ellipsoid_points for [n,9] parameter rows -> [n,1000,3] float32 world points."""
    L = _lib.load()
    p = _lib.host_array("params", params, np.float32, (-1, 9))
    out = np.zeros((len(p), _lib.N_SAMPLES, 3), np.float32)
    _lib.check(L.odam_sq_sample_points_host(_lib.ptr(p), len(p), _lib.ptr(out), device))
    return out


def sample_on_batch(shapes, epsilons, n_samples=1000, device=0):
    """Drop-in for learnable_primitives.fast_sampler.fast_sample_on_batch (reference _sampler.pyx:413-441):
    shapes [B,M,3], epsilons [B,M,2] float32 -> (etas, omegas) [B,M,N] float32."""
    L = _lib.load()
    B, M = np.shape(shapes)[:2]
    a = _lib.host_array("shapes", shapes, np.float32, (B, M, 3))
    e = _lib.host_array("epsilons", epsilons, np.float32, (B, M, 2))
    etas = np.zeros((B, M, n_samples), np.float32)
    omegas = np.zeros((B, M, n_samples), np.float32)
    _lib.check(L.odam_sq_sample_on_batch_host(_lib.ptr(a), _lib.ptr(e), _lib.ptr(etas), _lib.ptr(omegas), B, M,
                                              n_samples, _lib.GRID, 0, device))
    return etas, omegas


def project_boxes_host(params, view_off, Ms, device=0):
    """get_bbox for every (object, view): [SV,4] = x_min,x_max,y_min,y_max."""
    L = _lib.load()
    p = _lib.host_array("params", params, np.float32, (-1, 9))
    voff = _lib.host_array("view_off", view_off, np.int32, (len(p) + 1,))
    SV = int(voff[-1])
    M = _lib.host_array("Ms", Ms, np.float32, (SV, 12))
    out = np.zeros((max(SV, 0), 4), np.float32)   # offsets that do not start at 0 or decrease are the entry's ERR_ARG
    _lib.check(L.odam_sq_project_boxes_host(_lib.ptr(p), _lib.ptr(voff), _lib.ptr(M), len(p), _lib.ptr(out), device))
    return out


def oriented_boxes_host(params, device=0, want_points=False):
    """compute_ellipsoid_points + compute_oriented_bbox for [n,9] parameter rows in ONE launch (odam_sq_oriented_boxes_host):
    returns corners [n,8,3] float64 (upper four first), flags [n] int32 and, when asked, the points [n,1000,3] float32."""
    L = _lib.load()
    p = _lib.host_array("params", params, np.float32, (-1, 9))
    n = len(p)
    corners = np.zeros((n, 8, 3), np.float64)
    flags = np.zeros(n, np.int32)
    pts = np.zeros((n, _lib.N_SAMPLES, 3), np.float32) if want_points else None
    _lib.check(L.odam_sq_oriented_boxes_host(_lib.ptr(p), n, _lib.ptr(corners), _lib.ptr(flags), _lib.ptr(pts), device))
    return (corners, flags, pts) if want_points else (corners, flags)


def oriented_boxes_of_points_host(points, device=0):
    """compute_oriented_bbox (reference box_utils.py:319-410) of point sets [n, n_pts, 3] (n_pts <= 1024); one set may
    be given as [n_pts, 3]."""
    L = _lib.load()
    shape = np.shape(points)
    n, n_pts = ((1,) + shape if len(shape) == 2 else shape)[:2]
    pts = _lib.host_array("points", points, np.float32, (n, n_pts, 3))
    corners = np.zeros((n, 8, 3), np.float64)
    flags = np.zeros(n, np.int32)
    _lib.check(L.odam_sq_oriented_boxes_of_points_host(_lib.ptr(pts), n, n_pts, _lib.ptr(corners), _lib.ptr(flags), device))
    return corners, flags


def merge_cost_host(boxes, cls=None, device=0, want_iou=False):
    """The cost matrix of merge_process (reference run_merge.py:90-121): boxes [n,8,3] float64 (bboxes_qc), cls [n] class
    ids or None -> cost [n,n] float64 (1 - IoU3D where the classes allow a merge, else 1; symmetric, zero diagonal).
    want_iou: also the raw (iou3d, iou2d) matrices for i < j."""
    L = _lib.load()
    b = _lib.host_array("boxes", boxes, np.float64, (-1, 8, 3))
    n = len(b)
    c = _lib.host_array("cls", cls, np.int32, (n,))
    cost = np.zeros((n, n), np.float64)
    i3 = np.zeros((n, n), np.float64) if want_iou else None
    i2 = np.zeros((n, n), np.float64) if want_iou else None
    _lib.check(L.odam_sq_merge_cost_host(_lib.ptr(b), _lib.ptr(c), n, _lib.ptr(cost), _lib.ptr(i3), _lib.ptr(i2), device))
    return (cost, i3, i2) if want_iou else cost


class DeviceTracks:
    """PackedTracks resident in HBM as torch tensors (plumbing only: allocation + stream)."""

    def __init__(self, tracks, device, prior=None):
        import torch
        self.torch = torch
        self.device = torch.device(device)
        init, cls, self.view_off_host, Ms, box, mask = _track_arrays(tracks)
        prior = _lib.host_array("prior", prior, np.float32, (8, 9))
        t = lambda a: None if a is None else torch.from_numpy(a).to(self.device)
        self.n, self.total_views = tracks.n, tracks.total_views
        self.init, self.cls, self.view_off, self.Ms = t(init), t(cls), t(self.view_off_host), t(Ms)
        self.box, self.mask, self.prior = t(box), t(mask), t(prior)


def optimize_device(dt, n_iters=200, representation="super_quadric", lr=0.01, lr_shape=0.1, threads=0,
                    max_slices=0, out=None, cycles=None, cluster=0, code_layout=0, corners=None):
    """Enqueue one fused launch on torch's current stream; returns dict of CUDA tensors (no sync).
    out: the dict of a previous call with the same n and n_iters, to be written again.
    cycles: optional int64 CUDA tensor [n, 16], per-phase SM cycles (diagnostics; slot names in tools/prof_run.py).
    corners: optional float64 CUDA tensor [n, 8, 3] -- the oriented boxes of the optimised objects, from a second launch
    enqueued right behind the optimiser (odam_sq_options.out_corners)."""
    torch = dt.torch
    dev = dt.init.device   # the tracks' device, with its index
    shapes = dict(params=(torch.float32, (dt.n, 9)), loss=(torch.float32, (dt.n, n_iters)), status=(torch.int32, (dt.n,)))
    if out is None:
        out = {k: torch.empty(shape, dtype=dtype, device=dev) for k, (dtype, shape) in shapes.items()}
    else:
        for k, (dtype, shape) in shapes.items():
            _lib.check_tensor(f"out[{k!r}]", out[k], dtype, shape, dev)
    if cycles is not None:
        _lib.check_tensor("cycles", cycles, torch.int64, (dt.n, 16), dev)
    if corners is not None:
        _lib.check_tensor("corners", corners, torch.float64, (dt.n, 8, 3), dev)
        out["corners"] = corners
    o = _lib.Options()
    if threads == 0 or cluster == 0 or code_layout == 0:
        # choose on the host from the host copy of view_off (avoids the library's D2H read-back)
        q = query_launch(dt.view_off_host, threads, max_slices, cluster, code_layout)
        threads, cluster, code_layout, max_slices = q["threads"], q["cluster"], q["code_layout"], q["max_slices"]
    o.threads, o.max_slices, o.cluster, o.code_layout = int(threads), int(max_slices), int(cluster), int(code_layout)
    o.max_views = int(np.diff(dt.view_off_host).max()) if dt.n else 0
    p = _lib.tensor_ptr
    o.out_cycles, o.out_corners = p(cycles), p(corners)
    with torch.cuda.device(dev):
        rc = _lib.load().odam_sq_optimize(p(dt.init), p(dt.cls), p(dt.view_off), p(dt.Ms), p(dt.box), p(dt.mask),
                                          p(dt.prior), dt.n, n_iters, _lib.REPR[representation], lr, lr_shape,
                                          p(out["params"]), p(out["loss"]), p(out["status"]), C.byref(o),
                                          _lib.current_stream(dev))
    _lib.check(rc)
    return out


def fma_peak_tflops(device=0):
    """Measured FP32 FMA roofline of the device (library micro-benchmark), TFLOP/s."""
    L = _lib.load()
    v = C.c_double()
    _lib.check(L.odam_sq_fma_peak(device, C.byref(v)))
    return v.value


def algorithmic_flops(view_counts, n_iters):
    """SURVEY.md 8(d): flops(run) = sum_obj iters * (37,000 * V_obj + 30,000) FP32 flop."""
    v = np.asarray(view_counts, np.float64)
    return float((n_iters * (37000.0 * v + 30000.0)).sum())
