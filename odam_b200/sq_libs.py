"""Drop-in for the hot-path classes of the reference's ``src/super_quadric/sq_libs.py``.

Same names, constructor arguments, attributes and return values as
  SuperQuadricOptimizer  (reference sq_libs.py:351-527)
  SuperQuadric           (reference sq_libs.py:531-595)
so that ``src/scripts/run_multi_view.py:56-67`` and ``src/processor.py:196`` work unchanged when they import
these instead (see INTEGRATION.md).  The arithmetic does not happen here: ``run`` packs its arguments and makes
ONE call into the CUDA library (``odam_sq_optimize_host``, include/odam_sq.h), which runs every iteration of
every object in a single persistent sm_100a kernel.  There is no CPU fallback; without the library or a B200
these classes raise.

Differences a caller can observe (all documented in DESIGN.md):
  * ``Q_init``'s leaf tensors are updated once, after the last iteration (the reference mutates them every step).
  * ``optimizer`` is a light object holding Adam's state (exp_avg, exp_avg_sq, step) so that repeated ``run``
    calls continue the same optimiser trajectory, as they do with the reference's ``torch.optim.Adam``.
  * NaN/Inf in the optimisation raises ``RuntimeError`` after the launch (the reference raises from torch's
    anomaly mode at the offending step).
Use ``optimize_batch`` to optimise many objects in one launch -- that is the fast path.
"""
import numpy as np
import torch

from . import _lib, api

CLASS_MAPPER = dict(api.CLASS_MAPPER)  # reference sq_libs.py:13-22


def squashing(shape, min_=0.2, max_=1.6):  # reference sq_libs.py:26-27
    return torch.sigmoid(shape) * (max_ - min_) + min_


class _Sampler:
    """Stand-in for EqualDistanceSamplerSQ(1000) (reference learnable_primitives/sampling.py:394-399)."""
    n_samples = _lib.N_SAMPLES

    def sample_on_batch(self, shapes, epsilons):
        return api.sample_on_batch(shapes, epsilons, self.n_samples)


class SuperQuadric:
    """Parameter container + forward sampler (reference sq_libs.py:531-595).  Picklable; leaf tensors as there.

    The four leaf tensors (``shapes``, ``translate``, ``angle``, ``scales``: float32, requires_grad) are created the
    first time they are read: the batched call site returns one object per track, and building four tensors for
    each eagerly costs more than the kernel launch that optimised them all.  Until then the parameters live in one
    packed float32[9] row (the C-ABI layout)."""

    _LEAVES = {"translate": slice(0, 3), "angle": 3, "scales": slice(4, 7), "shapes": slice(7, 9)}

    def __init__(self, translate, angle, scales, shapes):
        p = np.empty(9, np.float32)
        p[0:3] = np.asarray(translate, np.float64)
        p[3] = np.float64(angle)
        p[4:7] = np.asarray(scales, np.float64)      # the scales of api.init_params
        p[7:9] = np.asarray(shapes, np.float64)
        self.__dict__["_p"] = p
        self.__dict__["_t"] = {}
        self.sampler = _Sampler()

    @classmethod
    def from_params(cls, p9, obj_class=None):
        """From a packed float32[9] row [t3, yaw, s3, h2] (no tensor is built)."""
        self = cls.__new__(cls)
        self.__dict__["_p"] = np.array(p9, np.float32).reshape(9)
        self.__dict__["_t"] = {}
        self.sampler = _Sampler()
        if obj_class is not None:
            self.obj_class = obj_class
        return self

    # -- the reference's leaf tensors, materialised on demand ---------------------------------------------
    def __getattr__(self, name):
        leaves = type(self)._LEAVES
        if name in leaves and "_t" in self.__dict__:
            t = self.__dict__["_t"]
            if name not in t:
                v = self.__dict__["_p"][leaves[name]]
                t[name] = torch.tensor(np.array(v), dtype=torch.float32, requires_grad=True)
            return t[name]
        raise AttributeError(name)

    def __setattr__(self, name, value):
        if name in type(self)._LEAVES:
            self.__dict__["_t"][name] = value
        else:
            self.__dict__[name] = value

    def __getstate__(self):
        # pickles look like the reference's: the four tensors as plain attributes
        d = {k: v for k, v in self.__dict__.items() if k not in ("_p", "_t")}
        for name in type(self)._LEAVES:
            d[name] = getattr(self, name)
        return d

    def __setstate__(self, d):
        d = dict(d)
        t = {name: d.pop(name) for name in type(self)._LEAVES}
        self.__dict__.update(d)
        self.__dict__["_t"] = t
        self.__dict__["_p"] = np.zeros(9, np.float32)
        self.__dict__["_p"][:] = self.params()

    # -- packed view ------------------------------------------------------------------------------------
    def params(self):
        """[t3, yaw, s3, h2] float32, the C-ABI layout (read from the tensors where they exist: a caller may have
        changed them)."""
        p = self.__dict__["_p"].copy()
        with torch.no_grad():
            for name, t in self.__dict__["_t"].items():
                p[type(self)._LEAVES[name]] = t.detach().numpy().reshape(-1) if t.dim() else float(t)
        return p

    def _set_params(self, p):
        self.__dict__["_p"][:] = p
        with torch.no_grad():
            for name, t in self.__dict__["_t"].items():   # same tensor objects, updated in place (as the reference's step)
                v = p[type(self)._LEAVES[name]]
                t.copy_(torch.from_numpy(np.array(v, np.float32)).reshape(t.shape))

    # -- reference API ----------------------------------------------------------------------------------
    def compute_ellipsoid_points(self, use_numpy):
        """1000 world points of the surface (reference sq_libs.py:577-595), computed on the GPU.
        Returns (points, None); a float32 numpy array when use_numpy else a (non-differentiable) tensor."""
        pts = api.sample_points_host(self.params()[None])[0]
        return (pts if use_numpy else torch.from_numpy(pts)), None

    def get_bbox(self, P_cw, if_vectorize=False, line_form=False):
        """[min_x, min_y, max_x, max_y] of the projected samples (reference sq_libs.py:547-554)."""
        M = np.ascontiguousarray(np.asarray(P_cw, np.float64).reshape(1, 12), np.float32)
        b = api.project_boxes_host(self.params()[None], np.array([0, 1], np.int32), M)[0]
        return np.array([b[0], b[2], b[1], b[3]])

    def rotz(self, angle):
        """z rotation matrix (reference sq_libs.py:556-575)."""
        cosz, sinz = torch.cos(angle), torch.sin(angle)
        zeros = angle.detach() * 0
        ones = zeros.detach() + 1
        return torch.stack([cosz, -sinz, zeros, sinz, cosz, zeros, zeros, zeros, ones], dim=0).reshape(3, 3)


class LossLog(list):
    """``loss_log`` of the reference (sq_libs.py:471): a list with one ``[tensor(total loss)]`` entry per iteration.
    The values arrive from the GPU as one float32 array per run; they are kept as Python floats and wrapped into the
    reference's ``[tensor]`` form when read (creating 10 000 scalar tensors eagerly costs several times the
    optimisation itself).  ``len``, indexing, slicing, iteration, ``append`` and ``extend`` behave like the list's."""

    @staticmethod
    def _wrap(v):
        return v if isinstance(v, list) else [torch.tensor(v, dtype=torch.float32)]

    def extend_values(self, values):
        list.extend(self, (float(v) for v in values))

    def __getitem__(self, i):
        v = list.__getitem__(self, i)
        return [self._wrap(x) for x in v] if isinstance(i, slice) else self._wrap(v)

    def __iter__(self):
        return (self._wrap(v) for v in list.__iter__(self))

    def values(self):
        """float32 array of the losses logged so far (entries appended by hand in the reference's form included)."""
        return np.array([float(v[0]) if isinstance(v, list) else v for v in list.__iter__(self)], np.float32)


class _AdamState:
    """What the drop-in keeps of ``torch.optim.Adam``: moments and step count (packed like the parameters)."""

    def __init__(self, optimize_shapes):
        self.exp_avg = np.zeros(9, np.float32)
        self.exp_avg_sq = np.zeros(9, np.float32)
        self.step = 0
        self.param_groups = [{"lr": 0.01, "betas": (0.9, 0.999), "eps": 1e-8}]
        if optimize_shapes:
            self.param_groups.append({"lr": 0.1, "betas": (0.9, 0.999), "eps": 1e-8})

    def zero_grad(self):
        pass


class SuperQuadricOptimizer:
    """reference sq_libs.py:351-527: same constructor, ``run`` / ``run_with_intermediate``, ``Q_init``, ``loss_log``."""

    def __init__(self, translate, quat, scales, obj_class, representation, prior):
        # `quat` is the yaw angle (reference run_multi_view.py:57); `scales` are box dimensions (sq_libs.py:361)
        self.use_prior = prior
        self.representation = representation
        self.Q_init = SuperQuadric.from_params(api.init_params(translate, quat, scales, representation))
        self.Q_init.obj_class = obj_class
        self.optimizer = _AdamState(representation == "super_quadric")
        # reference sq_libs.py:388-392: ./src/super_quadric/scale_prior relative to the cwd; the packaged export of
        # the same data file is used when that path does not exist
        self.scale_prior = {k: torch.tensor(v).float() for k, v in api.load_scale_prior().items()}
        self.loss_log = LossLog()
        self.device = 0

    # -- packing ----------------------------------------------------------------------------------------
    def _pack(self, gt_lines, Ms):
        Ms = np.ascontiguousarray(np.asarray(Ms, np.float64).reshape(-1, 12), np.float32)  # torch.tensor(Ms).float()
        if isinstance(gt_lines, tuple):   # already packed (box[V,4] float32 pixels, mask[V,4]) by the batched call site
            box, mask = np.ascontiguousarray(gt_lines[0], np.float32), np.ascontiguousarray(gt_lines[1], np.uint8)
        else:
            box, mask = api.pack_lines(gt_lines)
        if len(box) != Ms.shape[0]:
            raise ValueError("one projection matrix per set of lines expected")
        return Ms, box, mask

    def run(self, gt_lines, gt_planes, Ms, n_iters=200):
        """One launch, n_iters Adam steps; returns self.Q_init (same instance, tensors updated in place)."""
        optimize_batch([self], [gt_lines], [Ms], n_iters)
        return self.Q_init

    def run_with_intermediate(self, gt_lines, gt_planes, Ms, n_iters=200):
        """As the reference (sq_libs.py:478-527): also the surface points and oriented box after every step."""
        hist = optimize_batch([self], [gt_lines], [Ms], n_iters, want_history=True)[0]
        # the surfaces and oriented boxes of all n_iters intermediate states from ONE launch
        boxes, _flags, pts = api.oriented_boxes_host(hist, device=self.device, want_points=True)
        steps = [{"bbox_qc": boxes[i], "surface_points": pts[i]} for i in range(n_iters)]
        return self.Q_init, steps


def optimize_batch(optimizers, gt_lines_list, Ms_list, n_iters=200, device=None, want_history=False):
    """Optimise many SuperQuadricOptimizer objects in ONE kernel launch (the batched call site, INTEGRATION.md).

    All optimizers must share representation / use_prior (as they do in run_multi_view.optim_process, where both
    are function arguments) and have taken the same number of Adam steps so far.  Updates every Q_init, loss_log
    and Adam state in place; returns the per-step parameter history [n_iters, 9] per object when asked."""
    if not optimizers:
        return []
    o0 = optimizers[0]
    if any(o.representation != o0.representation or bool(o.use_prior) != bool(o0.use_prior)
           or o.optimizer.step != o0.optimizer.step for o in optimizers):
        raise ValueError("optimize_batch needs a homogeneous batch (representation, prior, step count)")
    Ms, box, mask, off = [], [], [], [0]
    for o, lines, M in zip(optimizers, gt_lines_list, Ms_list):
        m, b, k = o._pack(lines, M)
        Ms.append(m); box.append(b); mask.append(k); off.append(off[-1] + m.shape[0])
    prior = None
    if o0.use_prior:
        prior = np.zeros((8, 9), np.float32)
        for o in optimizers:   # KeyError for an unknown class, as in the reference (sq_libs.py:464)
            c = o.Q_init.obj_class
            prior[c] = o.scale_prior[CLASS_MAPPER[c]].numpy().reshape(9)
    tracks = api.PackedTracks(init=np.stack([o.Q_init.params() for o in optimizers]),
                              cls=np.array([o.Q_init.obj_class if o.use_prior else 0 for o in optimizers], np.int32),
                              view_off=np.array(off, np.int32), Ms=np.concatenate(Ms), box=np.concatenate(box),
                              mask=np.concatenate(mask))
    continuing = o0.optimizer.step > 0
    out = api.optimize_host(
        tracks, prior=prior, n_iters=n_iters, representation=o0.representation,
        lr=o0.optimizer.param_groups[0]["lr"], lr_shape=o0.optimizer.param_groups[-1]["lr"],
        device=o0.device if device is None else device,
        m0=np.stack([o.optimizer.exp_avg for o in optimizers]) if continuing else None,
        v0=np.stack([o.optimizer.exp_avg_sq for o in optimizers]) if continuing else None,
        step0=o0.optimizer.step, extras=("out_m", "out_v") + (("out_param_hist",) if want_history else ()))
    for i, o in enumerate(optimizers):
        o.Q_init._set_params(out["params"][i])
        o.optimizer.exp_avg, o.optimizer.exp_avg_sq = out["out_m"][i].copy(), out["out_v"][i].copy()
        o.optimizer.step += n_iters
        o.loss_log.extend_values(out["loss"][i])   # read back as a list of 1-element [tensor] lists, as :471
    api.check_finite(out["status"])
    return [out["out_param_hist"][i] for i in range(len(optimizers))] if want_history else []
