"""Synthetic ScanNet-like posed views and 2-D detections for the superquadric optimiser.

ScanNet and the pretrained detector are not available offline, so the benchmark and the
parity tests run on scenes drawn by the recipe of SURVEY.md section 8(d):
image 1296x968 (reference src/datasets/scan_net_track.py:111-112), fx=fy=1170, cx=648, cy=484,
``P_cw = K @ inv(T_wc)[:3, :]`` (src/processor.py:311), sides within 20 px of the image border
dropped (src/super_quadric/quadric_helper.py:87-107), views with no surviving side dropped
(src/scripts/run_multi_view.py:52-55).

One deliberate simplification: the ground-truth 2-D box of a view is the bounding box of the
ground-truth superquadric sampled on a regular 48x96 (eta, omega) lattice, instead of the
reference's ``SuperQuadric.get_bbox`` (1000 sampler points).  It only shapes the synthetic
detections; nothing on the optimisation path depends on it.

All random draws come from ``numpy.random.default_rng(seed)`` so a scene is identical on every
host; the (heavy) lattice projection runs in float64 torch on the device given.
"""
from dataclasses import dataclass

import numpy as np
import torch

from .api import SIDES, unpack_lines  # noqa: F401  (SIDES: the order of the last axis of box and mask)

IMG_W, IMG_H = 1296, 968
K = np.array([[1170.0, 0.0, 648.0], [0.0, 1170.0, 484.0], [0.0, 0.0, 1.0]])
EDGE = 20.0


@dataclass
class Scene:
    """n objects x V views each, in the layout the C-ABI takes (include/odam_sq.h)."""
    translate: np.ndarray   # [n,3] f64  initial centre (averaged detector output)
    angle: np.ndarray       # [n]   f64  initial yaw
    dims: np.ndarray        # [n,3] f64  initial 3-D box dimensions (NOT api.init_params' scales)
    cls: np.ndarray         # [n]   i32  class id 0..7
    P_cws: np.ndarray       # [n,V,3,4] f64 projection matrices
    box: np.ndarray         # [n,V,4] f64 detected sides in SIDES order, pixels
    mask: np.ndarray        # [n,V,4] u8  1 = side kept
    gt: dict                # ground truth (centre, yaw, dims, logits) for diagnostics

    @property
    def n(self):
        return self.translate.shape[0]

    @property
    def V(self):
        return self.P_cws.shape[1]

    def gt_lines(self, i):
        """Object i's detections in the reference's list-of-dicts form (quadric_helper.py:69-109)."""
        return unpack_lines(self.box[i], self.mask[i])


def _lattice(n_eta=48, n_omega=96):
    eta = (np.arange(n_eta) + 0.5) / n_eta * np.pi - np.pi / 2
    om = (np.arange(n_omega) + 0.5) / n_omega * 2 * np.pi - np.pi
    eta, om = np.meshgrid(eta, om, indexing="ij")
    return eta.ravel(), om.ravel()


def _look_at(eye, target):
    """Camera-to-world rotation, camera axes x right / y down / z forward, world +z up."""
    f = target - eye
    f = f / np.linalg.norm(f, axis=-1, keepdims=True)
    up = np.zeros_like(f)
    up[..., 2] = 1.0
    r = np.cross(f, up)
    r = r / np.linalg.norm(r, axis=-1, keepdims=True)
    u = np.cross(r, f)
    return np.stack([r, -u, f], axis=-1)  # columns = camera axes in world


def make_scene(n_objects, n_views, seed, device="cpu", oversample=2.0):
    rng = np.random.default_rng(seed)
    n, V = n_objects, n_views
    Vd = int(np.ceil(V * oversample)) + 4
    cls = rng.integers(0, 8, size=n).astype(np.int32)
    centre = np.concatenate([rng.uniform(-3, 3, (n, 2)), rng.uniform(0.2, 1.0, (n, 1))], 1)
    dims = rng.uniform(0.3, 1.5, (n, 3))
    yaw = rng.uniform(-np.pi, np.pi, n)
    logits = rng.uniform(-2, 2, (n, 2))
    # cameras
    rad = rng.uniform(2, 4, (n, Vd))
    azi = rng.uniform(0, 2 * np.pi, (n, Vd))
    hgt = centre[:, 2:3] + rng.uniform(0.5, 1.5, (n, Vd))
    eye = np.stack([centre[:, 0:1] + rad * np.cos(azi), centre[:, 1:2] + rad * np.sin(azi), hgt], -1)
    tgt = centre[:, None, :] + rng.normal(0, 0.2, (n, Vd, 3))
    R_wc = _look_at(eye, tgt)                                   # [n,Vd,3,3]
    R_cw = np.swapaxes(R_wc, -1, -2)
    t_cw = -np.einsum("nvij,nvj->nvi", R_cw, eye)
    P = K @ np.concatenate([R_cw, t_cw[..., None]], -1)         # [n,Vd,3,4]
    noise = rng.normal(0, 3.0, (n, Vd, 4))
    init_t = centre + rng.normal(0, 0.1, (n, 3))
    init_yaw = yaw + rng.normal(0, 0.2, n)
    init_dims = dims * rng.uniform(0.8, 1.2, (n, 3))

    # ground-truth boxes: project the GT superquadric lattice (float64, chunked over objects)
    eta, om = _lattice()
    dev = torch.device(device)
    eta_t = torch.tensor(eta, device=dev)
    om_t = torch.tensor(om, device=dev)
    sp = lambda c, p: torch.sign(c) * torch.abs(c) ** p
    box = np.empty((n, Vd, 4))
    chunk = max(1, int(2e7 // (Vd * eta.size)))
    for lo in range(0, n, chunk):
        hi = min(n, lo + chunk)
        a = torch.tensor(dims[lo:hi] / 2, device=dev)            # a = s^2 = dims/2
        e = torch.sigmoid(torch.tensor(logits[lo:hi], device=dev)) * 1.4 + 0.2
        ce, se = torch.cos(eta_t)[None], torch.sin(eta_t)[None]
        co, so = torch.cos(om_t)[None], torch.sin(om_t)[None]
        x = a[:, 0:1] * sp(ce, e[:, 0:1]) * sp(co, e[:, 1:2])
        y = a[:, 1:2] * sp(ce, e[:, 0:1]) * sp(so, e[:, 1:2])
        z = a[:, 2:3] * sp(se, e[:, 0:1])
        cz = torch.tensor(np.cos(yaw[lo:hi]), device=dev)[:, None]
        sz = torch.tensor(np.sin(yaw[lo:hi]), device=dev)[:, None]
        c = torch.tensor(centre[lo:hi], device=dev)
        pw = torch.stack([x * cz - y * sz + c[:, 0:1], x * sz + y * cz + c[:, 1:2], z + c[:, 2:3],
                          torch.ones_like(x)], -1)              # [m,L,4]
        q = torch.einsum("nvij,nlj->nvli", torch.tensor(P[lo:hi], device=dev), pw)
        uv = q[..., :2] / q[..., 2:3]
        front = (q[..., 2] > 0.5).all(-1)
        b = torch.stack([uv[..., 0].amin(-1), uv[..., 0].amax(-1), uv[..., 1].amin(-1), uv[..., 1].amax(-1)], -1)
        b[~front] = float("nan")
        box[lo:hi] = b.cpu().numpy()
    box = box + noise
    lim = np.array([IMG_W, IMG_W, IMG_H, IMG_H], np.float64)
    keep = (box > EDGE) & (box < lim - EDGE)                    # NaN compares false
    ok = keep.any(-1)                                           # [n,Vd]
    # first V usable views of each object, original order preserved
    order = np.argsort(~ok, axis=1, kind="stable")[:, :V]
    if not np.take_along_axis(ok, order, 1).all():
        bad = np.where(~np.take_along_axis(ok, order, 1).all(1))[0]
        raise RuntimeError(f"{bad.size} objects have fewer than {V} usable views; raise oversample")
    take = lambda x: np.take_along_axis(x, order.reshape(n, V, *([1] * (x.ndim - 2))), 1)
    box, keep, P = take(box), take(keep), take(P)
    T_wc = np.zeros((n, Vd, 4, 4))
    T_wc[..., :3, :3], T_wc[..., :3, 3], T_wc[..., 3, 3] = R_wc, eye, 1.0
    box_raw = box.copy()
    box = np.where(keep, box, 0.0)
    return Scene(translate=init_t, angle=init_yaw, dims=init_dims, cls=cls, P_cws=P, box=box,
                 mask=keep.astype(np.uint8),
                 gt=dict(centre=centre, yaw=yaw, dims=dims, logits=logits, T_wcs=take(T_wc), box_raw=box_raw))


def scene_to_tracks(scene, rows_per_object=None, seed=0):
    """A Scene as the inputs of the reference's call site ``optim_process`` (run_multi_view.py:22): every object owns
    its own block of frames (object i is seen in frames i*V .. i*V+V-1 of one long sequence), one 82-float track row
    per (object, frame) in the layout of processor.py:98-108 -- [0] frame id, [1] class, [2:6] box x_min,y_min,x_max,
    y_max in pixels, [6:9] dims, [9:12] centre, [12] yaw, [13] score, rest -1.  Per-row detector noise on dims, centre
    and yaw is drawn around the scene's initial values, so the averaged pose the call site derives is close to them.
    rows_per_object[i] < V keeps only the first rows (an object seen in too few frames is not optimised).
    Returns dict(tracks, img_names, T_wcs, P_cws, img_h, img_w, K)."""
    rng = np.random.default_rng(seed)
    n, V = scene.n, scene.V
    tracks = []
    for i in range(n):
        rows = V if rows_per_object is None else int(rows_per_object[i])
        t = -np.ones((rows, 82))
        t[:, 0] = i * V + np.arange(rows)
        t[:, 1] = scene.cls[i]
        b = scene.gt["box_raw"][i, :rows]
        t[:, 2:6] = np.stack([b[:, 0], b[:, 2], b[:, 1], b[:, 3]], 1)
        t[:, 6:9] = scene.dims[i][None] * rng.uniform(0.97, 1.03, (rows, 3))
        t[:, 9:12] = scene.translate[i][None] + rng.normal(0, 0.02, (rows, 3))
        t[:, 12] = scene.angle[i] + rng.normal(0, 0.03, rows)
        t[:, 13] = rng.uniform(0.5, 1.0, rows)
        tracks.append(t)
    return dict(tracks=tracks, img_names=np.arange(n * V), T_wcs=scene.gt["T_wcs"].reshape(n * V, 4, 4),
                P_cws=scene.P_cws.reshape(n * V, 3, 4), img_h=IMG_H, img_w=IMG_W, K=K)


# BASELINE.json configs -> (objects, views, iterations, prior); seed = config index (SURVEY 8d)
CONFIGS = {
    1: dict(n_objects=10, n_views=20, n_iters=200, prior=True, name="1 scene, 10 objects x 20 views"),
    2: dict(n_objects=50, n_views=50, n_iters=200, prior=True, name="single scene, 50 objects x 50 views"),
    3: dict(n_objects=2000, n_views=30, n_iters=200, prior=True, name="100 scenes, 2000 objects x 30 views"),
    4: dict(n_objects=500, n_views=300, n_iters=200, prior=True, name="long tracks, 500 objects x 300 views"),
    5: dict(n_objects=50000, n_views=20, n_iters=200, prior=False, name="stress, 50k objects x 20 views, no prior"),
}


def make_config(idx, device="cpu", n_objects=None):
    c = CONFIGS[idx]
    return make_scene(n_objects or c["n_objects"], c["n_views"], seed=idx, device=device)
