"""ctypes binding of include/odam_sq.h.  There is NO fallback: if the CUDA library is missing or the
call fails, this raises -- the product path never computes on the CPU."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# ODAM_SQ_LIB selects another build of the same library (A/B timing of source trees: each built with
# `python -m odam_b200.build --force --out odam_b200/lib/ab/libodam_sq_<name>.so`, then tools/ab_run.sh <name>...)
LIB_PATH = os.environ.get("ODAM_SQ_LIB") or os.path.join(HERE, "lib", "libodam_sq.so")

REPR = {"super_quadric": 0, "cube": 1, "quadric": 2}
ST_NONFINITE, ST_SAMPLER, ST_NO_VALID_PT = 1, 2, 4
N_SAMPLES, GRID = 1000, 201


class Options(C.Structure):
    """odam_sq_options (include/odam_sq.h)."""
    _fields_ = [("threads", C.c_int), ("max_slices", C.c_int), ("cluster", C.c_int), ("max_views", C.c_int),
                ("code_layout", C.c_int),
                ("m0", C.c_void_p), ("v0", C.c_void_p), ("step0", C.c_int), ("s0", C.c_void_p),
                ("out_m", C.c_void_p), ("out_v", C.c_void_p), ("out_grad", C.c_void_p), ("out_pred", C.c_void_p),
                ("out_arg", C.c_void_p), ("out_eta_idx", C.c_void_p), ("out_grids", C.c_void_p),
                ("out_param_hist", C.c_void_p), ("out_cycles", C.c_void_p),
                ("out_corners", C.c_void_p), ("out_box_flag", C.c_void_p)]


class OdamSqError(RuntimeError):
    pass


_vp, _ci, _cf = C.c_void_p, C.c_int, C.c_float
_OPT = [_vp] * 7 + [_ci, _ci, _ci, _cf, _cf] + [_vp] * 3 + [C.POINTER(Options)]
# every entry of include/odam_sq.h -> its argtypes
ARGTYPES = {
    "odam_sq_abi_version": [],
    "odam_sq_error_string": [_ci],
    "odam_sq_last_cuda_error": [],
    "odam_sq_init": [_ci],
    "odam_sq_optimize": _OPT + [_vp],
    "odam_sq_optimize_host": _OPT + [_ci],
    "odam_sq_sample_points": [_vp, _ci, _vp, _vp],
    "odam_sq_sample_points_host": [_vp, _ci, _vp, _ci],
    "odam_sq_project_boxes": [_vp, _vp, _vp, _ci, _vp, _vp],
    "odam_sq_project_boxes_host": [_vp, _vp, _vp, _ci, _vp, _ci],
    "odam_sq_query_launch": [_vp, _ci, C.POINTER(Options)] + [C.POINTER(_ci)] * 6,
    "odam_sq_sample_on_batch_host": [_vp] * 4 + [_ci] * 6,
    "odam_sq_fma_peak": [_ci, C.POINTER(C.c_double)],
    "odam_sq_selftest": [_ci, C.c_uint32, C.c_longlong, C.POINTER(C.c_longlong)],
    "odam_sq_oriented_boxes": [_vp, _ci, _vp, _vp, _vp, _vp],
    "odam_sq_oriented_boxes_host": [_vp, _ci, _vp, _vp, _vp, _ci],
    "odam_sq_oriented_boxes_of_points_host": [_vp, _ci, _ci, _vp, _vp, _ci],
    "odam_sq_merge_cost_host": [_vp, _vp, _ci, _vp, _vp, _vp, _ci],
    "odam_sq_cluster_capacity": [_ci, _ci, C.POINTER(_ci)],
    "odam_sq_stage_tracks_host": [_vp, _vp, _ci, _ci, _vp, _ci, _ci, _ci] + [_vp] * 9,
    "odam_sq_sample_points_vjp": [_vp, _vp, _ci, _vp, _vp],
    "odam_sq_box_sides": [_vp, _vp, _vp, _ci, _ci, _vp, _vp, _vp],
    "odam_sq_box_sides_vjp": [_vp, _vp, _vp, _vp, _vp, _ci, _ci, _vp, _vp],
    "odam_sq_box_sides_vjp_cameras": [_vp, _vp, _vp, _vp, _vp, _ci, _ci, _vp, _vp, _vp],
}
EXPORTS = tuple(ARGTYPES)

_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OdamSqError(f"{LIB_PATH} is missing: build it with `python -m odam_b200.build` "
                              "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        missing = [f for f in EXPORTS if not hasattr(L, f)]
        if missing:
            raise OdamSqError(f"{LIB_PATH} does not export {', '.join(missing)}")
        for name, argtypes in ARGTYPES.items():
            getattr(L, name).argtypes = argtypes
        L.odam_sq_error_string.restype = C.c_char_p
        L.odam_sq_last_cuda_error.restype = C.c_char_p
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        L = load()
        msg = L.odam_sq_error_string(rc).decode()
        if rc == -2:
            msg += ": " + L.odam_sq_last_cuda_error().decode()
        raise OdamSqError(f"odam_sq error {rc}: {msg}")


def ptr(a):
    """numpy array -> void* (None passes NULL)."""
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def host_array(name, a, dtype, shape):
    """A caller's array as a C-contiguous numpy array of `dtype` and `shape` (numpy's reshape rules), None for None.
    The C entries size their copies from n and the view offsets, not from the arrays, so an array of another size
    is a ValueError here rather than a read or write past its end."""
    if a is None:
        return None
    a = np.ascontiguousarray(a, dtype)
    try:
        return a.reshape(shape)
    except ValueError:
        raise ValueError(f"{name} must have shape {list(shape)}, got {list(a.shape)}") from None


def check_tensor(name, t, dtype, shape, device):
    """ValueError unless t is a contiguous `dtype` tensor of exactly `shape` on `device`."""
    if tuple(t.shape) != tuple(shape) or t.dtype != dtype or not t.is_contiguous() or t.device != device:
        raise ValueError(f"{name} must be a contiguous {dtype} tensor of shape {list(shape)} on {device}, got "
                         f"{t.dtype} {list(t.shape)} on {t.device} (contiguous: {t.is_contiguous()})")


def tensor_ptr(t):
    """torch tensor -> void* (None passes NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream(device):
    """torch's current stream on `device` as the cudaStream_t the C entries take."""
    import torch
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
