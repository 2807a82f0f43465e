"""ctypes binding of include/odam_sq.h.  There is NO fallback: if the CUDA library is missing or the
call fails, this raises -- the product path never computes on the CPU."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
# ODAM_SQ_LIB selects another build of the same library (A/B timing of kernel variants, tools/ab_build.sh)
LIB_PATH = os.environ.get("ODAM_SQ_LIB") or os.path.join(HERE, "lib", "libodam_sq.so")

REPR = {"super_quadric": 0, "cube": 1, "quadric": 2}
ST_NONFINITE, ST_SAMPLER, ST_NO_VALID_PT = 1, 2, 4
N_SAMPLES, GRID = 1000, 201

EXPORTS = ("odam_sq_abi_version", "odam_sq_error_string", "odam_sq_last_cuda_error", "odam_sq_init",
           "odam_sq_optimize", "odam_sq_optimize_host", "odam_sq_sample_points", "odam_sq_sample_points_host",
           "odam_sq_project_boxes", "odam_sq_project_boxes_host", "odam_sq_query_launch",
           "odam_sq_sample_on_batch_host", "odam_sq_fma_peak", "odam_sq_selftest", "odam_sq_oriented_boxes",
           "odam_sq_oriented_boxes_host", "odam_sq_oriented_boxes_of_points_host", "odam_sq_merge_cost_host",
           "odam_sq_cluster_capacity", "odam_sq_stage_tracks_host", "odam_sq_sample_points_vjp", "odam_sq_box_sides",
           "odam_sq_box_sides_vjp")


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


_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OdamSqError(f"{LIB_PATH} is missing: build it with `python -m odam_b200.build` "
                              "(there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        vp, ci, cf = C.c_void_p, C.c_int, C.c_float
        L.odam_sq_abi_version.restype = ci
        L.odam_sq_error_string.restype = C.c_char_p
        L.odam_sq_error_string.argtypes = [ci]
        L.odam_sq_last_cuda_error.restype = C.c_char_p
        L.odam_sq_init.argtypes = [ci]
        opt_args = [vp] * 7 + [ci, ci, ci, cf, cf] + [vp] * 3 + [C.POINTER(Options)]
        L.odam_sq_optimize.argtypes = opt_args + [vp]
        L.odam_sq_optimize_host.argtypes = opt_args + [ci]
        L.odam_sq_sample_points.argtypes = [vp, ci, vp, vp]
        L.odam_sq_sample_points_host.argtypes = [vp, ci, vp, ci]
        L.odam_sq_project_boxes.argtypes = [vp, vp, vp, ci, vp, vp]
        L.odam_sq_project_boxes_host.argtypes = [vp, vp, vp, ci, vp, ci]
        L.odam_sq_sample_on_batch_host.argtypes = [vp] * 4 + [ci] * 6
        L.odam_sq_oriented_boxes.argtypes = [vp, ci, vp, vp, vp, vp]
        L.odam_sq_oriented_boxes_host.argtypes = [vp, ci, vp, vp, vp, ci]
        L.odam_sq_oriented_boxes_of_points_host.argtypes = [vp, ci, ci, vp, vp, ci]
        L.odam_sq_merge_cost_host.argtypes = [vp, vp, ci, vp, vp, vp, ci]
        L.odam_sq_fma_peak.argtypes = [ci, C.POINTER(C.c_double)]
        L.odam_sq_selftest.argtypes = [ci, C.c_uint32, C.c_longlong, C.POINTER(C.c_longlong)]
        L.odam_sq_query_launch.argtypes = [vp, ci, C.POINTER(Options)] + [C.POINTER(ci)] * 6
        L.odam_sq_cluster_capacity.argtypes = [ci, ci, C.POINTER(ci)]
        L.odam_sq_stage_tracks_host.argtypes = [vp, vp, ci, ci, vp, ci, ci, ci] + [vp] * 9
        L.odam_sq_sample_points_vjp.argtypes = [vp, vp, ci, vp, vp]
        L.odam_sq_box_sides.argtypes = [vp, vp, vp, ci, ci, vp, vp, vp]
        L.odam_sq_box_sides_vjp.argtypes = [vp, vp, vp, vp, vp, ci, ci, vp, vp]
        for f in EXPORTS:
            if getattr(L, f).restype is None:
                pass
            getattr(L, f)
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
