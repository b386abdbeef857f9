"""ctypes binding of include/dfusion.h (libdfusion.so).

This is the only way Python reaches the CUDA kernels: plain pointers and sizes, no torch types cross the
boundary.  torch is used by callers for device memory and streams only.  The loader FAILS LOUDLY when the
library is missing -- there is no CPU fallback in the product path.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
# DF_LIB_VARIANT=<tag> loads libdfusion_<tag>.so instead (instrumented / A-B builds made by tools/build_variant.py; measurement only)
_LIB_PATH = _HERE / (f"libdfusion_{os.environ['DF_LIB_VARIANT']}.so" if os.environ.get("DF_LIB_VARIANT") else "libdfusion.so")
_lib = None
MISSING: list[str] = []


class Volume(C.Structure):
    _fields_ = [("data", C.c_void_p), ("dims", C.c_int * 3), ("voxel_size", C.c_float * 3),
                ("trunc_dist", C.c_float), ("max_weight", C.c_int)]


class Aff3f(C.Structure):
    _fields_ = [("R", C.c_float * 9), ("t", C.c_float * 3)]


class Intr(C.Structure):
    _fields_ = [("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float)]


class KinfuParams(C.Structure):
    """df_kinfu_params (include/dfusion.h) == KinFuParams, kinfu.hpp:15-47"""
    _fields_ = [("cols", C.c_int), ("rows", C.c_int), ("intr", Intr),
                ("volume_dims", C.c_int * 3), ("volume_size", C.c_float * 3), ("volume_pose", Aff3f),
                ("bilateral_sigma_depth", C.c_float), ("bilateral_sigma_spatial", C.c_float), ("bilateral_kernel_size", C.c_int),
                ("icp_truncate_depth_dist", C.c_float), ("icp_dist_thres", C.c_float), ("icp_angle_thres", C.c_float),
                ("icp_iter_num", C.c_int * 4),
                ("tsdf_min_camera_movement", C.c_float), ("tsdf_trunc_dist", C.c_float), ("tsdf_max_weight", C.c_int),
                ("raycast_step_factor", C.c_float), ("gradient_delta_factor", C.c_float),
                ("light_pose", C.c_float * 3),
                ("solver_nonlinear_iters", C.c_int), ("solver_linear_iters", C.c_int),
                ("max_nodes", C.c_int), ("node_step", C.c_int), ("cloud_capacity", C.c_int), ("flags", C.c_int),
                ("fusion_weight_scale", C.c_float), ("extend_radius", C.c_float)]


class F2Params(C.Structure):
    """df_f2_params (include/dfusion.h)"""
    _fields_ = [("reg_lambda", C.c_double), ("tukey_c", C.c_double), ("huber_delta", C.c_double), ("lm_mu", C.c_double),
                ("gn_iters", C.c_int), ("reg_k", C.c_int), ("flags", C.c_int), ("lin_iters", C.c_int)]


_vp, _sz, _i, _f = C.c_void_p, C.c_size_t, C.c_int, C.c_float

# name -> (restype, argtypes); must list every symbol declared in include/dfusion.h
PROTOTYPES = {
    "df_error_string": (C.c_char_p, [_i]),
    "df_version": (_i, []),
    "df_clear_volume": (_i, [Volume, _vp]),
    "df_compute_dists": (_i, [_vp, _sz, _i, _i, Intr, _vp, _sz, _vp]),
    "df_integrate": (_i, [Volume, _vp, _sz, _i, _i, Aff3f, Intr, _vp, _vp]),
    "df_volume_activity_bytes": (_sz, [Volume]),
    "df_integrate_workspace_bytes": (_sz, [_i, _i]),
    "df_integrate_launch_count": (_i, [Volume]),
    "df_integrate_last_kernel": (_i, []),
    "df_integrate_selftest": (_i, [_vp, _vp]),
    "df_integrate_tracked": (_i, [Volume, _vp, _sz, _i, _i, Aff3f, Intr, _vp, _vp, _vp, _vp]),
    "df_raycast_points": (_i, [Volume, Aff3f, C.POINTER(C.c_float), Intr, _i, _i, _f, _f, _vp, _sz, _vp, _sz, _vp]),
    "df_raycast_points_tracked": (_i, [Volume, Aff3f, C.POINTER(C.c_float), Intr, _i, _i, _f, _f, _vp, _sz, _vp, _sz, _vp, _vp]),
    "df_raycast_points_stats_tracked": (_i, [Volume, Aff3f, C.POINTER(C.c_float), Intr, _i, _i, _f, _f, _vp, _sz, _vp, _sz, _vp, _vp, _vp, _vp]),
    "df_raycast_touched_bytes": (_sz, [Volume]),
    "df_raycast_points_stats": (_i, [Volume, Aff3f, C.POINTER(C.c_float), Intr, _i, _i, _f, _f, _vp, _sz, _vp, _sz, _vp, _vp, _vp]),
    "df_project_workspace_bytes": (_sz, [_i, _i]),
    "df_project_and_remove": (_i, [_vp, _sz, _i, _i, Intr, _vp, _sz, _i, _i, _vp, _vp]),
    "df_extract_workspace_bytes": (_sz, [Volume]),
    "df_extract_cloud": (_i, [Volume, Aff3f, _vp, _i, _vp, _vp, _vp]),
    "df_extract_cloud_tracked": (_i, [Volume, Aff3f, _vp, _i, _vp, _vp, _vp, _vp]),
    "df_extract_normals": (_i, [Volume, _vp, _i, _vp, Aff3f, C.POINTER(C.c_float), _f, _vp, _vp]),
    "df_extract_mesh_workspace_bytes": (_sz, [Volume]),
    "df_extract_mesh": (_i, [Volume, Aff3f, _vp, _vp, _vp, _i, _vp, _i, _vp, _vp, _vp]),
    "df_bilateral": (_i, [_vp, _sz, _i, _i, _vp, _sz, _i, _f, _f, _vp]),
    "df_truncate_depth": (_i, [_vp, _sz, _i, _i, _f, _vp]),
    "df_pyr_down": (_i, [_vp, _sz, _i, _i, _vp, _sz, _f, _vp]),
    "df_points_normals": (_i, [Intr, _vp, _sz, _i, _i, _vp, _sz, _vp, _sz, _vp]),
    "df_resize_points_normals": (_i, [_vp, _sz, _vp, _sz, _i, _i, _vp, _sz, _vp, _sz, _vp]),
    "df_render_image": (_i, [_vp, _sz, _vp, _sz, _i, _i, C.POINTER(C.c_float), _vp, _sz, _vp]),
    "df_render_tangent_colors": (_i, [_vp, _sz, _i, _i, _vp, _sz, _vp]),
    "df_render_image_depth": (_i, [_vp, _sz, _vp, _sz, _i, _i, Intr, C.POINTER(C.c_float), _vp, _sz, _vp]),
    "df_normals_mask_depth": (_i, [Intr, _vp, _sz, _i, _i, _vp, _sz, _vp]),
    "df_cloud_to_depth": (_i, [_vp, _sz, _i, _i, _vp, _sz, _vp]),
    "df_resize_depth_normals": (_i, [_vp, _sz, _vp, _sz, _i, _i, _vp, _sz, _vp, _sz, _vp]),
    "df_icp_accumulate": (_i, [_vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz, _i, _i, Intr, Aff3f, _f, _f, _vp, _vp]),
    "df_icp_estimate": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i),
                             C.POINTER(_sz), _i, C.POINTER(_i), Intr, _f, _f, _vp, _vp, _vp, _vp]),
    "df_icp_accumulate_depth": (_i, [_vp, _sz, _vp, _sz, _vp, _sz, _vp, _sz, _i, _i, Intr, Aff3f, _f, _f, _vp, _vp]),
    "df_icp_estimate_depth": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_i), C.POINTER(_i),
                                   C.POINTER(_sz), C.POINTER(_sz), _i, C.POINTER(_i), Intr, _f, _f, _vp, _vp, _vp, _vp]),
    "df_knn8": (_i, [_vp, _i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "df_node_grid_bytes": (_sz, [_i]),
    "df_build_node_grid": (_i, [_vp, _i, _vp, _vp]),
    "df_extend_field_workspace_bytes": (_sz, [_i]),
    "df_extend_field": (_i, [_vp, _i, _i, _vp, _vp, _i, _vp, _i, _f, _i, _vp, _vp, _vp]),
    "df_warp": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, Aff3f, _i, _vp, _vp, _vp]),
    "df_integrate_warped_workspace_bytes": (_sz, [_i, _i, _i]),
    "df_integrate_warped_launch_count": (_i, []),
    "df_integrate_warped": (_i, [Volume, _vp, _sz, _i, _i, Aff3f, Aff3f, Intr, _vp, _i, _vp, _f, _vp, _vp, _vp, _vp]),
    "df_solve_workspace_bytes": (_sz, [_i, _i]),
    "df_solve_knn_buffers": (_i, [_vp, _i, _i, C.POINTER(_vp), C.POINTER(_vp)]),
    "df_solve_data_term": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "df_solve_f2_workspace_bytes": (_sz, [_i, _i, _i]),
    "df_solve_f2": (_i, [_vp, _i, _vp, _vp, _vp, _i, _i, C.POINTER(F2Params), _vp, _vp, _vp]),
    "df_kinfu_set_f2_params": (_i, [_vp, C.POINTER(F2Params)]),
    "df_kinfu_default_params": (None, [C.POINTER(KinfuParams), _i]),
    "df_kinfu_create": (_vp, [C.POINTER(KinfuParams)]),
    "df_kinfu_destroy": (None, [_vp]),
    "df_kinfu_reset": (_i, [_vp]),
    "df_kinfu_process_host": (_i, [_vp, _vp, _sz]),
    "df_kinfu_batch_process_host": (_i, [C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_sz), _i, C.POINTER(_i)]),
    "df_kinfu_process_device": (_i, [_vp, _vp, _sz]),
    "df_kinfu_get_stage_ms": (_i, [_vp, C.POINTER(C.c_float), _i]),
    "df_kinfu_dynamicfusion": (_i, [_vp, _vp, _sz, _vp, _sz]),
    "df_kinfu_get_pose": (_i, [_vp, _i, C.POINTER(C.c_float)]),
    "df_kinfu_get_info": (_i, [_vp, C.POINTER(C.c_longlong), _i]),
    "df_kinfu_get_buffer": (_i, [_vp, _i, C.POINTER(_vp), C.POINTER(_sz), C.POINTER(_i), C.POINTER(_i)]),
    "df_kinfu_set_stream": (_i, [_vp, _vp]),
    "df_kinfu_read_buffer": (_i, [_vp, _i, _vp, _sz]),
    "df_kinfu_join": (_i, [_vp]),
    "df_kinfu_set_overrides": (_i, [_vp, _vp, _sz, _vp, _vp, _i]),
    "df_kinfu_state_digest": (_i, [_vp, C.POINTER(C.c_ulonglong)]),
    "df_kinfu_extract_mesh": (_i, [_vp, _i, _vp, _vp, _vp, _i, _vp, _i, C.POINTER(_i)]),
}


def lib_path() -> Path:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load libdfusion.so; raise (never fall back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        raise RuntimeError(
            f"{_LIB_PATH} is missing: build it with `python -m dynamicfusion_b200.build` "
            "(nvcc, sm_100a).  dynamicfusion_b200 has no CPU fallback.")
    lib = C.CDLL(str(_LIB_PATH))
    MISSING.clear()
    for name, (res, args) in PROTOTYPES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:       # header/library mismatch: calling it raises, tests/test_capi.py asserts none
            MISSING.append(name)
            continue
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        raise RuntimeError(f"libdfusion: CUDA error {status}: {load().df_error_string(status).decode()}")


def make_aff(R, t) -> Aff3f:
    a = Aff3f()
    flat = [float(v) for row in R for v in row] if hasattr(R[0], "__len__") else [float(v) for v in R]
    for i in range(9):
        a.R[i] = flat[i]
    for i in range(3):
        a.t[i] = float(t[i])
    return a


def make_intr(fx, fy, cx, cy) -> Intr:
    return Intr(float(fx), float(fy), float(cx), float(cy))


def make_volume(ptr: int, dims, voxel_size, trunc_dist: float, max_weight: int) -> Volume:
    v = Volume()
    v.data = ptr
    for i in range(3):
        v.dims[i] = int(dims[i])
        v.voxel_size[i] = float(voxel_size[i])
    v.trunc_dist = float(trunc_dist)
    v.max_weight = int(max_weight)
    return v


def f9(vals):
    arr = (C.c_float * 9)()
    flat = [float(v) for row in vals for v in row] if hasattr(vals[0], "__len__") else [float(v) for v in vals]
    for i in range(9):
        arr[i] = flat[i]
    return arr
