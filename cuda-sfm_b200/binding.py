"""ctypes binding of the C ABI declared in include/sfmb200.h.

This is the Python analogue of the stub a reference maintainer would write
(INTEGRATION.md); it holds no algorithmic code.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path() -> str:
    return os.path.join(HERE, "libsfmb200.so")


class SfmError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"sfmb200 error {code}: {msg}")
        self.code = code


_f = C.POINTER(C.c_float)
_i = C.POINTER(C.c_int32)
_vp = C.c_void_p

# name -> (restype, argtypes); must list every symbol of include/sfmb200.h
SIGNATURES = {
    "sfmb200_last_error": (C.c_char_p, []),
    "sfmb200_version": (C.c_int, []),
    "sfmb200_build_info": (C.c_char_p, []),
    "sfmb200_small_path_debug": (C.c_int, [_vp]),
    "sfmb200_create": (C.c_int, [_f, _f, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]),
    "sfmb200_destroy": (C.c_int, [_vp]),
    "sfmb200_set_option": (C.c_int, [_vp, C.c_int, C.c_int]),
    "sfmb200_set_stream": (C.c_int, [_vp, _vp]),
    "sfmb200_synchronize": (C.c_int, [_vp]),
    "sfmb200_set_points_sift": (C.c_int, [_vp, _vp, C.c_int]),
    "sfmb200_set_points_sift_filtered": (C.c_int, [_vp, _vp, C.c_int, C.c_float, C.c_float, _vp, C.POINTER(C.c_int32)]),
    "sfmb200_set_points_xy": (C.c_int, [_vp, _vp, C.c_int]),
    "sfmb200_set_points_xy_host": (C.c_int, [_vp, _vp, C.c_int]),
    "sfmb200_set_points_normalised": (C.c_int, [_vp, _vp, C.c_int]),
    "sfmb200_set_points_xy_ragged": (C.c_int, [_vp, _vp, _vp]),
    "sfmb200_run_device_ragged": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_uint64, C.c_float]),
    "sfmb200_run_host_ragged": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_uint64, C.c_float, _vp, _vp, _vp, _vp, _vp]),
    "sfmb200_get_point_counts": (C.c_int, [_vp, _vp]),
    "sfmb200_estimate_e": (C.c_int, [_vp, _vp, C.c_int, C.c_uint64, C.c_float]),
    "sfmb200_estimate_e_slice": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_float]),
    "sfmb200_copy_to_vbo_coloured": (C.c_int, [_vp, C.c_int, _vp, _vp, C.c_float, C.c_int, C.c_float, C.c_float]),
    "sfmb200_mg_handle_bytes": (C.c_int, []),
    "sfmb200_mg_init": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "sfmb200_mg_connect": (C.c_int, [_vp, _vp]),
    "sfmb200_estimate_e_mg": (C.c_int, [_vp, _vp, C.c_int, C.c_uint64, C.c_float]),
    "sfmb200_mg_status": (C.c_int, [_vp, _vp]),
    "sfmb200_mg_set_timeout_ms": (C.c_int, [_vp, C.c_int]),
    "sfmb200_mg_close": (C.c_int, [_vp]),
    "sfmb200_chain_views": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "sfmb200_bundle_adjust_global": (C.c_int, [_vp, _vp, _vp, C.c_int, _vp, _vp]),
    "sfmb200_bundle_adjust": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "sfmb200_estimate_e_adaptive": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_float, C.c_float, _vp]),
    "sfmb200_best_buffer": (C.c_int, [_vp, C.POINTER(_vp)]),
    "sfmb200_adopt_best": (C.c_int, [_vp, _vp, C.c_int, C.c_uint64]),
    "sfmb200_find_homography": (C.c_int, [_vp, C.c_int, C.c_uint64, C.c_float, _vp, _vp]),
    "sfmb200_refine_e": (C.c_int, [_vp, C.c_int]),
    "sfmb200_get_refit_iterations": (C.c_int, [_vp, _vp]),
    "sfmb200_pose_candidates": (C.c_int, [_vp]),
    "sfmb200_choose_pose": (C.c_int, [_vp]),
    "sfmb200_triangulate": (C.c_int, [_vp]),
    "sfmb200_run_host": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_uint64, C.c_float, _vp, _vp, _vp, _vp, _vp]),
    "sfmb200_run_device": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_uint64, C.c_float]),
    "sfmb200_copy_to_vbo": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "sfmb200_get_E": (C.c_int, [_vp, _vp]),
    "sfmb200_set_E": (C.c_int, [_vp, _vp]),
    "sfmb200_get_best": (C.c_int, [_vp, _vp, _vp]),
    "sfmb200_get_poses": (C.c_int, [_vp, _vp]),
    "sfmb200_get_pose_index": (C.c_int, [_vp, _vp]),
    "sfmb200_get_points": (C.c_int, [_vp, C.c_int, _vp]),
    "sfmb200_get_points_host": (C.c_int, [_vp, C.c_int, _vp]),
    "sfmb200_get_inlier_counts": (C.c_int, [_vp, C.c_int, _vp]),
    "sfmb200_get_E_candidates": (C.c_int, [_vp, C.c_int, _vp]),
    "sfmb200_get_X": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "sfmb200_get_inlier_mask": (C.c_int, [_vp, C.c_int, _vp]),
    "sfmb200_device_views": (C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_int)]),
    "sfmb200_score_plan": (C.c_int, [_vp, _i]),
    "sfmb200_launch_count": (C.c_int64, [_vp]),
    "sfmb200_stage_times": (C.c_int, [_vp, C.c_int, _vp, C.POINTER(C.c_int)]),
    "sfmb200_fma_probe": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    "sfmb200_host_svd3": (None, [_f, _f, _f, _f]),
    "sfmb200_host_svd3_reference_orientation": (None, [_f, _f, _f, _f]),
    "sfmb200_host_solve_hypothesis": (None, [_f, _f]),
    "sfmb200_host_solve_hypothesis_projector": (None, [_f, _f]),
    "sfmb200_host_null4": (None, [_f, _f]),
    "sfmb200_host_null4_fast": (C.c_int, [_f, _f]),
    "sfmb200_host_dlt_null": (C.c_int, [_f, _f]),
    "sfmb200_host_dlt_null_power4": (None, [_f, _f]),
    "sfmb200_host_inv4": (C.c_int, [_f, _f]),
    "sfmb200_host_sample_indices": (None, [C.c_uint64, C.c_uint64, C.c_int, _i]),
    "sfmb200_host_sample_indices_disjoint": (None, [C.c_uint64, C.c_uint64, C.c_int, _i]),
    # kernels.h facade wrappers (la_wrappers.cu)
    "sfmb200_la_mmul": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "sfmb200_la_mmul_batched": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    "sfmb200_la_mmul_transpose_batched": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp]),
    "sfmb200_la_invert": (C.c_int, [_vp, _vp, C.c_int, C.c_int, _vp]),
    "sfmb200_la_svd_batched": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "sfmb200_la_transpose_batched": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _vp]),
    "sfmb200_la_vecnorm": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_float, C.c_float, _vp]),
    "sfmb200_la_elementwise": (C.c_int, [C.c_int, _vp, _vp, C.c_int, _vp]),
    "sfmb200_la_threshold_count": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_float, _vp]),
    "sfmb200_la_row_extraction": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "sfmb200_la_argmax_first": (C.c_int, [_vp, C.c_int, _i, _vp]),
    "sfmb200_la_copy_point": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp]),
    "sfmb200_la_design_matrix": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int, C.c_int, _vp]),
    "sfmb200_la_normalize_E": (C.c_int, [_vp, C.c_int, _vp]),
    "sfmb200_la_candidate_poses": (C.c_int, [_vp, _vp, _vp, _vp]),
    "sfmb200_la_triangulation_A": (C.c_int, [_vp, _vp, _vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_int, _vp]),
    "sfmb200_la_normalize_pt": (C.c_int, [_vp, _vp, C.c_int, _vp]),
    "sfmb200_la_copy_to_vbo": (C.c_int, [C.c_int, _vp, _vp, C.c_float, _vp]),
}


class Lib:
    """Loaded library with typed functions; every int-returning call is checked."""

    def __init__(self, path: str | None = None):
        path = path or lib_path()
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} is missing: build it with `python cuda-sfm_b200/build.py` "
                "(there is no CPU fallback for the sfmb200 hot path)"
            )
        self.path = path
        self.cdll = C.CDLL(path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(self.cdll, name)
            fn.restype = res
            fn.argtypes = args
            setattr(self, "_" + name, fn)

    def last_error(self) -> str:
        return self._sfmb200_last_error().decode()

    def call(self, name: str, *args):
        rc = getattr(self, "_" + name)(*args)
        if rc != 0:
            raise SfmError(rc, self.last_error())
        return rc

    def raw(self, name: str):
        return getattr(self, "_" + name)


_LIB: Lib | None = None


def load_library(path: str | None = None) -> Lib:
    global _LIB
    if _LIB is None or (path and path != _LIB.path):
        _LIB = Lib(path)
    return _LIB
