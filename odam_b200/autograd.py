"""Differentiable ops on CUDA tensors: the optimiser's maths as ordinary PyTorch autograd.

The fused optimiser (api.optimize_device) runs a fixed number of Adam steps on one fixed loss.  These ops expose the
pieces of that loss so that callers can build their own: add loss terms, use another optimiser or a learning-rate
schedule, or backpropagate into parameters produced by other modules.

  surface_points(params)                  -> [n, 1000, 3]   compute_ellipsoid_points (sq_libs.py:577-595)
  box_sides(params, view_off, Ms, camera_grad=False)
                                          -> (pred [SV, 4], arg [SV, 4] int32)
                                             the projected box sides of constraint_2d (sq_libs.py:397-413)
  box_loss(params, view_off, Ms, box, mask, prior=None, cls=None, s0=None, camera_grad=False, weight=None, loss="l1",
           loss_scale=None) -> [n]
                                             the optimiser's per-object loss (sq_libs.py:420-430 + :463-466), or the
                                             weighted robust objective of api.optimize_host(side_weight=, loss=, ...)

params is a float32 CUDA tensor [n, 9]: translation x, y, z | yaw | scales s1, s2, s3 | shape logits h1, h2, the layout of
include/odam_sq.h.  Object i owns the views view_off[i] .. view_off[i+1]-1 of Ms ([SV, 12] or [SV, 3, 4] float32 camera
matrices P_cw on the same device).  view_off is int32 [n+1], on the CPU (then it is checked: starts at 0, monotone, ends at
SV) or on the device (then the kernels clamp each object's views to [0, SV]).

Forward and backward passes are CUDA kernels (csrc/sq_autograd.cuh) enqueued on the current stream of params' device.
Backward passes recompute the surface samples from params; gradients are deterministic, bit for bit, and independent of
the batch an object is evaluated in.  The sampler's discrete choices (which surface angles are sampled) and the
arg-extreme sample of every side are piecewise constant in params and carry no gradient, exactly as in the reference.
Double backward is not supported.

By default Ms is a constant: it is detached and its gradient stays None.  With camera_grad=True box_sides and box_loss
also return dL/dMs, through the caller's reshape of Ms, from the same backward kernel (its second pass, one thread per
view): joint object and camera refinement.  Rows of Ms that no object owns get 0.  Cameras shared by several objects are
gathered per frame, Ms = P[frame_idx] (run_multi_view.stage_tracks returns frame_idx); torch's backward of that gather
sums with atomics and is bit-reproducible only under torch.use_deterministic_algorithms(True).  dL/dMs itself is
deterministic either way.
"""
import math

import torch
from torch.autograd.function import once_differentiable

from . import _lib

N_SAMPLES = _lib.N_SAMPLES
_p, _stream = _lib.tensor_ptr, _lib.current_stream


def _check_params(params):
    if not isinstance(params, torch.Tensor):
        raise ValueError("params must be a torch.Tensor")
    if params.dtype != torch.float32:
        raise ValueError(f"params must be float32, got {params.dtype}")
    if params.dim() != 2 or params.shape[1] != 9:
        raise ValueError(f"params must have shape [n, 9], got {list(params.shape)}")


def _check_cuda(name, t, device):
    if not t.is_cuda:
        raise ValueError(f"{name} must be a CUDA tensor")
    if device is not None and t.device != device:
        raise ValueError(f"{name} is on {t.device}, params on {device}")


def _views(params, view_off, Ms):
    """Validates (params, view_off, Ms) and returns (Ms as [SV, 12], view_off as an int32 tensor on params' device)."""
    _check_params(params)
    if not isinstance(Ms, torch.Tensor) or Ms.dtype != torch.float32:
        raise ValueError("Ms must be a float32 tensor")
    if Ms.dim() == 3 and tuple(Ms.shape[1:]) == (3, 4):
        Ms = Ms.reshape(-1, 12)
    if Ms.dim() != 2 or Ms.shape[1] != 12:
        raise ValueError(f"Ms must have shape [SV, 12] or [SV, 3, 4], got {list(Ms.shape)}")
    if not isinstance(view_off, torch.Tensor) or view_off.dtype != torch.int32:
        raise ValueError("view_off must be an int32 tensor")
    n, SV = params.shape[0], Ms.shape[0]
    if view_off.dim() != 1 or view_off.shape[0] != n + 1:
        raise ValueError(f"view_off must have shape [n + 1] = [{n + 1}], got {list(view_off.shape)}")
    if not view_off.is_cuda:
        v = view_off.tolist()
        if v[0] != 0 or v[-1] != SV or any(b < a for a, b in zip(v, v[1:])):
            raise ValueError(f"view_off must start at 0, never decrease and end at the number of views ({SV})")
    _check_cuda("params", params, None)
    _check_cuda("Ms", Ms, params.device)
    if view_off.is_cuda:
        _check_cuda("view_off", view_off, params.device)
    if SV >= 2 ** 31 // 4:
        raise ValueError("too many views for int32 indexing")
    return Ms.contiguous(), view_off.to(params.device).contiguous()


class _SurfacePoints(torch.autograd.Function):
    @staticmethod
    def forward(ctx, params):
        n = params.shape[0]
        out = torch.empty((n, N_SAMPLES, 3), dtype=torch.float32, device=params.device)
        if n:
            L = _lib.load()
            with torch.cuda.device(params.device):
                _lib.check(L.odam_sq_sample_points(_p(params), n, _p(out), _stream(params.device)))
        ctx.save_for_backward(params)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_xyz):
        params, = ctx.saved_tensors
        n = params.shape[0]
        grad = torch.zeros_like(params)
        if n:
            g = grad_xyz.to(torch.float32).contiguous()
            L = _lib.load()
            with torch.cuda.device(params.device):
                _lib.check(L.odam_sq_sample_points_vjp(_p(params), _p(g), n, _p(grad), _stream(params.device)))
        return grad


class _BoxSides(torch.autograd.Function):
    @staticmethod
    def forward(ctx, params, view_off, Ms):
        n, SV = params.shape[0], Ms.shape[0]
        pred = torch.empty((SV, 4), dtype=torch.float32, device=params.device)
        arg = torch.empty((SV, 4), dtype=torch.int32, device=params.device)
        if n and SV:
            L = _lib.load()
            with torch.cuda.device(params.device):
                _lib.check(L.odam_sq_box_sides(_p(params), _p(view_off), _p(Ms), n, SV, _p(pred), _p(arg),
                                               _stream(params.device)))
        ctx.save_for_backward(params, view_off, Ms, arg)
        ctx.mark_non_differentiable(arg)
        return pred, arg

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_pred, _grad_arg):
        params, view_off, Ms, arg = ctx.saved_tensors
        n, SV = params.shape[0], Ms.shape[0]
        cams = ctx.needs_input_grad[2]   # Ms is attached only with camera_grad=True
        # camera-only refinement (params frozen) passes NULL: the kernel then skips the params pass
        grad = torch.zeros_like(params) if ctx.needs_input_grad[0] or not cams else None
        grad_Ms = torch.zeros((SV, 12), dtype=torch.float32, device=params.device) if cams else None
        if n and SV and grad_pred is not None:
            g = grad_pred.to(torch.float32).contiguous()
            L = _lib.load()
            with torch.cuda.device(params.device):
                if cams:
                    _lib.check(L.odam_sq_box_sides_vjp_cameras(_p(params), _p(view_off), _p(Ms), _p(arg), _p(g), n, SV,
                                                               _p(grad), _p(grad_Ms),
                                                               _stream(params.device)))
                else:
                    _lib.check(L.odam_sq_box_sides_vjp(_p(params), _p(view_off), _p(Ms), _p(arg), _p(g), n, SV,
                                                       _p(grad), _stream(params.device)))
        return grad, None, grad_Ms


def surface_points(params):
    """The 1000 world-space surface samples of every object, [n, 1000, 3] float32, differentiable with respect to params
    (the drop-in's compute_ellipsoid_points returns the same points without a graph)."""
    _check_params(params)
    _check_cuda("params", params, None)
    return _SurfacePoints.apply(params.contiguous())


def box_sides(params, view_off, Ms, camera_grad=False):
    """Projected box sides of every (object, view): pred [SV, 4] (x_min, x_max, y_min, y_max), differentiable with
    respect to params, and arg [SV, 4] int32, the sample that attains each side (-1 where no sample is in front of the
    camera, z > 0.5, and pred holds the reference's +-1e6 sentinel).  Ms gets no gradient unless camera_grad is True;
    then pred is differentiable with respect to Ms too (sides with arg -1 contribute nothing)."""
    Ms12, voff = _views(params, view_off, Ms)
    return _BoxSides.apply(params.contiguous(), voff, Ms12 if camera_grad else Ms12.detach())


def box_loss(params, view_off, Ms, box, mask, prior=None, cls=None, s0=None, camera_grad=False, weight=None, loss="l1",
             loss_scale=None):
    """The optimiser's loss per object, [n] float32: the sum over the four sides of the mean over all V views of the
    object of mask * |pred - box| (NaN terms count 0), plus 20 (s0 - s)^T A (s0 - s) with A = prior[cls] when a prior
    table is given.

    box [SV, 4] float32 detected sides (x_min, x_max, y_min, y_max), mask [SV, 4] (nonzero = side present), prior
    [8, 9] float32 per-class matrices (api.prior_table()), cls [n] class ids 0..7, s0 [n, 3] the anchor scales (the
    reference takes the scales at the start of its run).  The sum of this loss over objects, backpropagated, gives the
    fused optimiser's gradient.  camera_grad=True also backpropagates into Ms (box_sides).

    weight, loss, loss_scale: the objective of api.optimize_host(side_weight=, loss=, loss_scale=) in torch ops, each
    term weight * mask * rho(pred - box) with rho = |r| ("l1", the default), torch's smooth_l1_loss with beta =
    loss_scale ("smooth_l1") or 0.5 c^2 log1p((r / c)^2) with c = loss_scale ("cauchy"); weight [SV, 4] float32 on
    params' device, finite and >= 0 (not checked), or None = 1.  With the defaults this is the reference's loss."""
    pred, _ = box_sides(params, view_off, Ms, camera_grad)
    n, SV, dev = params.shape[0], pred.shape[0], params.device
    for name, t in (("box", box), ("mask", mask)) + ((("weight", weight),) if weight is not None else ()):
        if not isinstance(t, torch.Tensor) or tuple(t.shape) != (SV, 4):
            raise ValueError(f"{name} must be a tensor of shape [SV, 4] = [{SV}, 4]")
        _check_cuda(name, t, dev)
    if box.dtype != torch.float32:
        raise ValueError("box must be float32")
    if weight is not None and weight.dtype != torch.float32:
        raise ValueError("weight must be float32")
    if loss not in _lib.LOSS:
        raise ValueError(f"loss must be one of {', '.join(_lib.LOSS)}, got {loss!r}")
    if loss != "l1" and not (loss_scale is not None and math.isfinite(loss_scale) and loss_scale > 0):
        raise ValueError(f"loss={loss!r} needs a finite loss_scale > 0, got {loss_scale!r}")
    if prior is not None:
        if cls is None or s0 is None:
            raise ValueError("a prior needs cls and s0 (the anchor scales, [n, 3])")
        if not isinstance(prior, torch.Tensor) or prior.dtype != torch.float32 or prior.numel() != 72:
            raise ValueError("prior must be a float32 tensor [8, 9]")
        if not isinstance(cls, torch.Tensor) or tuple(cls.shape) != (n,) or cls.dtype.is_floating_point:
            raise ValueError(f"cls must be an integer tensor of shape [{n}]")
        if not isinstance(s0, torch.Tensor) or tuple(s0.shape) != (n, 3) or s0.dtype != torch.float32:
            raise ValueError(f"s0 must be a float32 tensor of shape [{n}, 3]")
        for name, t in (("prior", prior), ("cls", cls), ("s0", s0)):
            _check_cuda(name, t, dev)
    # clamped into [0, SV] and made monotone without a host round trip: device offsets are not checked on the host
    voff = torch.cummax(view_off.to(dev, torch.int64).clamp(0, SV), 0).values
    if loss == "l1":
        l =torch.abs(pred - box)
    elif loss == "smooth_l1":
        l = torch.nn.functional.smooth_l1_loss(pred, box, reduction="none", beta=loss_scale)
    else:
        t = (pred - box) / loss_scale
        l = 0.5 * loss_scale * loss_scale * torch.log1p(t * t)
    w = mask.to(torch.float32) if weight is None else mask.to(torch.float32) * weight
    l = torch.where(torch.isnan(l), torch.zeros_like(l), l) * w
    per_side = torch.segment_reduce(l, "sum", offsets=voff, axis=0, unsafe=True)          # [n, 4]
    V = (voff[1:] - voff[:-1]).to(torch.float32)
    loss = (per_side / V[:, None]).sum(1)
    if prior is not None:
        A = prior.reshape(8, 3, 3)[cls.long()]
        d = s0 - params[:, 4:7]
        loss = loss + torch.einsum("ni,nij,nj->n", d, A, d) * 20
    return loss
