"""Batched drop-in for the reference call site ``src/scripts/run_multi_view.py:22-76`` (``optim_process``), which
``OdamProcess.optim_process`` (src/processor.py:352-368) delegates to.

Same signature and return dict; the difference is structural.  The reference loops over objects in Python three
times (``load_pred_object`` per object per frame, one ``SuperQuadricOptimizer.run`` per object at 2.8 s each, one
Qhull call per object); here

  1. staging is ONE native call over the rows of ALL objects (`stage_tracks` -> ``odam_sq_stage_tracks_host``): class,
     mean centre, chordal mean of the per-frame yaws (closed form for rotations about z instead of scipy's
     ``Rotation.mean`` per object), mean dims, and for every usable frame the detected box sides with the 20 px border
     rule -- straight into the packed C-ABI arrays;
  2. every eligible object is optimised by ONE persistent kernel launch (``odam_sq_optimize_host``);
  3. ONE more launch, enqueued behind it inside the same call (``odam_sq_options.out_corners``), samples all final
     surfaces and computes their oriented boxes on the device (convex hull + min-area rectangle,
     csrc/sq_postproc.cuh) -- one synchronisation and one copy back for both.

Staging restates only what the optimiser consumes of ``tracking_gt_utils.load_pred_object`` (:145-211) and skips what
it never reads (plane vectors, depth planes).  Track rows are the 82-float layout of processor.py:98-108.
"""
import numpy as np

from . import _lib, api
from .postprocess import compute_oriented_bbox, get_3d_box, rotz  # noqa: F401  (host mirrors, re-exported)
from .sq_libs import SuperQuadric

EDGE_THRESHOLD = 20  # tracking_gt_utils.py:199


def mean_yaw(yaw):
    """Chordal L2 mean of rotations about z -- what ``averaging_T_wos`` (tracking_gt_utils.py:59-66) gets from scipy's
    ``Rotation.from_matrix(...).mean()`` followed by ``as_euler("zxy")[0]`` (run_multi_view.py:57): for quaternions
    (0, 0, sin t/2, cos t/2) the principal eigenvector of sum(q q^T) has the angle atan2(sum sin t, sum cos t)."""
    yaw = np.asarray(yaw, np.float64)
    return float(np.arctan2(np.sin(yaw).sum(), np.cos(yaw).sum()))


def stage_object(track, frame_ids, img_h, img_w):
    """One track staged on its own (same result as its row of `stage_tracks`); kept for callers that stage object by
    object.  Returns dict(obj_class, t_wo, R, yaw, dims, valid_frames, box [Vvalid,4], mask [Vvalid,4])."""
    st = stage_tracks([track], frame_ids, img_h, img_w)
    a, b = st["view_off"][0], st["view_off"][1]
    return dict(obj_class=int(st["cls"][0]), t_wo=st["t_wo"][0], R=rotz(st["yaw"][0]), yaw=float(st["yaw"][0]),
                dims=st["dims"][0], valid_frames=st["frame_idx"][a:b].tolist(), box=st["box"][a:b], mask=st["mask"][a:b])


def stage_tracks(tracks, frame_ids, img_h, img_w):
    """What run_multi_view.py:31-58 derives for every track, for all tracks in one native call
    (``odam_sq_stage_tracks_host``, csrc/sq_stage.h: one pass over the rows, no CUDA).  Same dict as
    `stage_tracks_numpy`, its vectorised numpy mirror."""
    import ctypes as C
    n = len(tracks)
    L = _lib.load()
    arrs = [np.ascontiguousarray(t, np.float64).reshape(-1, 82) for t in tracks]
    rows_per = np.array([a.shape[0] for a in arrs], np.int64)
    total = int(rows_per.sum())
    fid = np.ascontiguousarray(frame_ids, np.int64).reshape(-1)
    ptrs = (C.c_void_p * max(n, 1))(*[a.ctypes.data for a in arrs])
    cls, t_wo, yaw, dims = np.zeros(n, np.int32), np.zeros((n, 3)), np.zeros(n), np.zeros((n, 3))
    view_off, n_present = np.zeros(n + 1, np.int32), np.zeros(n, np.int64)
    frame_idx, box, mask = np.zeros(total, np.int64), np.zeros((total, 4), np.float32), np.zeros((total, 4), np.uint8)
    _lib.check(L.odam_sq_stage_tracks_host(ptrs, _lib.ptr(rows_per), n, 82, _lib.ptr(fid), len(fid), int(img_h), int(img_w),
                                           _lib.ptr(cls), _lib.ptr(t_wo), _lib.ptr(yaw), _lib.ptr(dims), _lib.ptr(view_off),
                                           _lib.ptr(frame_idx), _lib.ptr(box), _lib.ptr(mask), _lib.ptr(n_present)))
    sv = int(view_off[n])
    return dict(cls=cls, t_wo=t_wo, yaw=yaw, dims=dims, view_off=view_off, frame_idx=frame_idx[:sv], box=box[:sv],
                mask=mask[:sv], n_present=n_present)


def stage_tracks_numpy(tracks, frame_ids, img_h, img_w):
    """The numpy mirror of `stage_tracks` (kept for cross-checking the native entry), vectorised over all rows of all
    tracks.

    Returns dict of arrays: cls [n] (int(median(class column)), tracking_gt_utils.py:153), t_wo [n,3] (mean centre over
    ALL rows, :155), yaw [n] (chordal mean of the yaws of the frames that are in `frame_ids`), dims [n,3] (mean over
    those frames), and CSR-packed per usable frame (a frame of `frame_ids` present in the track whose box keeps at
    least one side after the 20 px border rule): view_off [n+1], frame_idx [SV] (index into frame_ids), box [SV,4] /
    mask [SV,4] in the C-ABI order x_min, x_max, y_min, y_max."""
    n = len(tracks)
    frame_ids = np.asarray(frame_ids)
    rows_per = np.array([len(t) for t in tracks], np.int64)
    if n == 0 or rows_per.sum() == 0:
        z = np.zeros
        return dict(cls=z(n, np.int32), t_wo=z((n, 3)), yaw=z(n), dims=z((n, 3)), view_off=z(n + 1, np.int32),
                    frame_idx=z(0, np.int64), box=z((0, 4), np.float32), mask=z((0, 4), np.uint8), n_present=z(n, np.int64))
    # only the first 13 of the 82 columns are read here: frame, class, box (4), dims (3), centre (3), yaw
    cat = np.concatenate([np.asarray(t, np.float64).reshape(-1, 82)[:, :13] for t in tracks], 0)
    obj = np.repeat(np.arange(n), rows_per)
    starts = np.concatenate([[0], np.cumsum(rows_per)[:-1]])
    # class: int(np.median(column)) per track
    order = np.lexsort((cat[:, 1], obj))
    sc = cat[order, 1]
    lo, hi = starts + (rows_per - 1) // 2, starts + rows_per // 2
    cls = ((sc[np.minimum(lo, len(sc) - 1)] + sc[np.minimum(hi, len(sc) - 1)]) / 2).astype(np.int64).astype(np.int32)
    # centre: np.mean over all rows of the track (sequential float64 accumulation, as numpy's axis-0 reduction)
    nz = rows_per > 0
    t_wo = np.zeros((n, 3))
    t_wo[nz] = np.add.reduceat(cat[:, 9:12], starts[nz], axis=0) / rows_per[nz, None]
    # rows whose frame is one of frame_ids; first row of the track per frame (np.where(...)[0][0]); frames in the
    # order of frame_ids
    fsort = np.argsort(frame_ids, kind="stable")
    fs = frame_ids[fsort]
    rf = cat[:, 0].astype(np.int32)
    pos = np.searchsorted(fs, rf)
    pos_c = np.minimum(pos, len(fs) - 1)
    present = fs[pos_c] == rf if len(fs) else np.zeros(len(rf), bool)
    fidx = fsort[pos_c]
    keep = np.nonzero(present)[0]
    key = obj[keep] * (len(frame_ids) + 1) + fidx[keep]
    _, first = np.unique(key, return_index=True)          # sorted by (object, frame index); first row per frame
    rows = keep[first]
    robj = obj[rows]
    n_present = np.bincount(robj, minlength=n)
    pstart = np.concatenate([[0], np.cumsum(n_present)[:-1]])
    has = n_present > 0
    yaw_r = cat[rows, 12]
    s_sum, c_sum, dims = np.zeros(n), np.zeros(n), np.zeros((n, 3))
    if has.any():
        s_sum[has] = np.add.reduceat(np.sin(yaw_r), pstart[has])
        c_sum[has] = np.add.reduceat(np.cos(yaw_r), pstart[has])
        dims[has] = np.add.reduceat(cat[rows, 6:9], pstart[has], axis=0) / n_present[has, None]
    yaw = np.arctan2(s_sum, c_sum)
    bb = cat[rows, 2:6]                                                  # x_min, y_min, x_max, y_max (pixels)
    box = np.stack([bb[:, 0], bb[:, 2], bb[:, 1], bb[:, 3]], axis=1)     # -> x_min, x_max, y_min, y_max
    hi_lim = np.array([img_w, img_w, img_h, img_h], np.float64) - EDGE_THRESHOLD
    mask = (box > EDGE_THRESHOLD) & (box < hi_lim)                        # quadric_helper.py:87-107
    valid = mask.any(axis=1)                                              # run_multi_view.py:52-55
    n_valid = np.bincount(robj[valid], minlength=n)
    view_off = np.concatenate([[0], np.cumsum(n_valid)]).astype(np.int32)
    return dict(cls=cls, t_wo=t_wo, yaw=yaw, dims=dims, view_off=view_off, frame_idx=fidx[rows][valid],
                box=np.where(mask[valid], box[valid], 0.0).astype(np.float32), mask=mask[valid].astype(np.uint8),
                n_present=n_present)


def lines_of(stage):
    """The reference's list-of-dicts form of a staged object's boxes (for SuperQuadricOptimizer.run)."""
    return api.unpack_lines(stage["box"], stage["mask"])


def boxes_3d(dims, yaw, centre):
    """get_3d_box (box_utils.py:286-308) for n objects at once: [n,8,3]."""
    dims, yaw, centre = np.asarray(dims, np.float64), np.asarray(yaw, np.float64), np.asarray(centre, np.float64)
    sx = np.array([1, 1, -1, -1, 1, 1, -1, -1]) / 2
    sy = np.array([1, -1, -1, 1, 1, -1, -1, 1]) / 2
    sz = np.array([1, 1, 1, 1, -1, -1, -1, -1]) / 2
    x, y, z = dims[:, 0:1] * sx, dims[:, 1:2] * sy, dims[:, 2:3] * sz
    c, s = np.cos(yaw)[:, None], np.sin(yaw)[:, None]
    return np.stack([c * x - s * y + centre[:, 0:1], s * x + c * y + centre[:, 1:2], z + centre[:, 2:3]], -1)


def optim_process(tracks, img_names, T_wcs, P_cws, img_h, img_w, K, representation, prior, n_iters, n_views,
                  device=0, devices=None):
    """reference run_multi_view.py:22-76, all objects in one launch.  T_wcs and K are accepted for signature
    compatibility (the optimiser only needs P_cws = K @ inv(T_wc)[:3, :], processor.py:311).
    devices: optional list of CUDA device indices -- the eligible objects are then sharded by object across them
    (contiguous blocks balanced by views, odam_b200.sharding), one host thread per device."""
    n = len(tracks)
    st = stage_tracks(tracks, img_names, img_h, img_w)
    bboxes_dl = boxes_3d(st["dims"], st["yaw"], st["t_wo"])
    init = api.init_params(st["t_wo"], st["yaw"], st["dims"], representation)
    views = np.diff(st["view_off"])
    run = np.nonzero(views >= n_views)[0]                       # :59-62 eligibility
    params = init.copy()
    bboxes_qc = bboxes_dl.copy()
    if prior:
        api.check_classes(st["cls"])                            # every track's, eligible or not
    if run.size:
        sel = np.nonzero(np.repeat(views >= n_views, views))[0]        # the packed views of the eligible objects
        P32 = np.ascontiguousarray(np.asarray(P_cws, np.float64).reshape(-1, 12)[st["frame_idx"][sel]], np.float32)
        packed = api.PackedTracks(init=init[run], cls=st["cls"][run].astype(np.int32),
                                  view_off=np.concatenate([[0], np.cumsum(views[run])]).astype(np.int32),
                                  Ms=P32, box=st["box"][sel], mask=st["mask"][sel])
        table = api.prior_table() if prior else None
        if devices and len(devices) > 1:
            from .sharding import optimize_on_devices
            out = optimize_on_devices(packed, table, n_iters, representation, devices)
        else:
            out = api.optimize_host(packed, prior=table, n_iters=n_iters, representation=representation, device=device,
                                    extras=("out_corners", "out_box_flag"))   # :66-67 fused behind the optimiser
        api.check_finite(out["status"], run)
        params[run] = out["params"]
        corners = out.get("out_corners")
        if corners is None:   # sharded over several devices: one more launch for all surfaces + oriented boxes
            corners, _flags = api.oriented_boxes_host(out["params"], device=device)   # :66-67
        bboxes_qc[run] = corners
    quadrics = [SuperQuadric.from_params(params[i], int(st["cls"][i])) for i in range(n)]
    return {"tracks": tracks, "bboxes_qc": list(bboxes_qc), "bboxes_dl": list(bboxes_dl), "quadrics": quadrics}


def merge_cost_matrix(data, device=0):
    """The cost matrix of ``merge_process`` (reference src/scripts/run_merge.py:90-121) for the dict `optim_process`
    returns: all n(n-1)/2 pair costs from one launch (``odam_sq_merge_cost_host``).  Feed it to
    ``AgglomerativeClustering(n_clusters=None, distance_threshold=0.95, affinity="precomputed", linkage="average")``
    exactly as the reference does (:81-85,122); the clustering itself stays sklearn."""
    cls = np.array([int(np.median(np.asarray(t)[:, 1])) for t in data["tracks"]], np.int32)
    return api.merge_cost_host(np.stack(data["bboxes_qc"]), cls, device=device)
