"""Drop-in for the projection loop of ``OdamProcess._prepare_tracks`` (reference src/processor.py:181-207), which the
online tracker runs once per frame over every live track: mean pose and size of the track -> a superquadric with
shape logits 0 -> its 1000 surface points -> their bounding box in the current camera, written into the last four
columns of the track.

The reference builds one ``SuperQuadric`` per track and samples it on the CPU (torch + the C++ sampler, ~1 ms per
track).  Here the surfaces of ALL tracks come from one launch (``odam_sq_sample_points_host``, the bit-exact device
sampler); the camera transform, projection and min/max are the reference's own float64 numpy operations
(``geometry_utils.get_homogeneous`` :7-49, ``projection`` :276-316), applied per track exactly as it does --
including its conventions: no z > 0 test, division by z, dims clipped at 0.05 (processor.py:195).
"""
import numpy as np

from . import api


def track_quadric_params(tracks):
    """[n, 9] C-ABI parameters (api.init_params, shape logits 0) of the mean-pose quadric of every track
    (processor.py:191-196); tracks = list of [rows, 82] arrays, columns 6:9 dims, 9:12 centre, 12 yaw."""
    n = len(tracks)
    t_wo, azi_wo, dimensions = np.zeros((n, 3)), np.zeros(n), np.zeros((n, 3))
    for i, track in enumerate(tracks):   # the reference's own per-track np.mean calls, for its float64 rounding
        track = np.asarray(track)
        azi_wo[i] = np.mean(track[:, 12], axis=0)
        t_wo[i] = np.mean(track[:, 9: 12], axis=0)
        dimensions[i] = np.clip(np.mean(track[:, 6: 9], axis=0), a_min=0.05, a_max=np.inf)
    return api.init_params(t_wo, azi_wo, dimensions)   # float64 -> float32 as SuperQuadric.__init__ does (torch.tensor)


def project_points_reference_way(pts, T_wc, K):
    """[x_min, y_min, x_max, y_max] of float32 points [N, 3] in camera T_wc (processor.py:198-202)."""
    homo = np.concatenate([pts, np.ones_like(pts[:, 2:])], axis=1)          # get_homogeneous
    box_3d_c = (homo @ np.linalg.inv(T_wc).T)[:, :3]
    pix = box_3d_c @ np.asarray(K).T                                          # projection(): pts @ intr_mat.T ...
    pix = pix / pix[:, -1:]                                                   # ... / z (no validity test)
    x_min, y_min, _ = np.min(pix, axis=0)
    x_max, y_max, _ = np.max(pix, axis=0)
    return np.array([x_min, y_min, x_max, y_max])


def prepare_track_boxes(tracks, T_wc, K, device=0):
    """Copy of ``tracks`` with ``track[:, -4:]`` = projected box of the track's quadric in camera ``T_wc``
    (the loop of processor.py:188-205; ``_preprocess_tracks`` -- the matcher's tensor layout -- is not part of this)."""
    tracks = [np.array(t, copy=True) for t in tracks]
    if not tracks:
        return tracks
    pts = api.sample_points_host(track_quadric_params(tracks), device=device)   # [n, 1000, 3] float32, one launch
    for track, p in zip(tracks, pts):
        track[:, -4:] = project_points_reference_way(p, T_wc, K)[None]
    return tracks
