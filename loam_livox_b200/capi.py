"""ctypes binding of libloamlivox_b200.so (include/loamlivox_b200.h).

The CUDA library is the product: importing this module without the shared object, or creating a context without a
B200-class GPU, fails loudly — there is no CPU or PyTorch fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libloamlivox_b200.so")

LL_FMT_XYZI16, LL_FMT_PCL32, LL_FMT_STRIDED = 0, 1, 2
LL_I_NONE, LL_I_UINT8, LL_I_UINT16, LL_I_FLOAT32 = 0, 2, 4, 7   # sensor_msgs/PointField datatype codes
LL_HOST, LL_DEVICE = 0, 1
LL_OK, LL_ERR_INVALID, LL_ERR_CUDA, LL_ERR_CAPACITY, LL_ERR_NO_BLOCKS, LL_ERR_CAP_BINDS = 0, -1, -2, -3, -4, -5
LL_IPC_HANDLE_BYTES = 64

EXPORTS = [
    "ll_config_default", "ll_ctx_create", "ll_ctx_destroy", "ll_ctx_warmup", "ll_last_error", "ll_ctx_stream", "ll_ctx_sync", "ll_extract", "ll_extract_reset", "ll_piece_bounds",
    "ll_get_features", "ll_extract_point_info", "ll_extract_split_idx", "ll_voxel_downsample", "ll_map_build", "ll_map_release", "ll_map_size",
    "ll_map_build_sharded", "ll_knn", "ll_reg_state_default", "ll_register", "ll_build_blocks", "ll_normal_equations", "ll_solve", "ll_transform",
    "ll_debug_knn_blocks", "ll_scan_to_pose", "ll_comm_local_handle", "ll_comm_connect", "ll_launch_count", "ll_cellmap_create", "ll_cellmap_release", "ll_cellmap_append",
    "ll_cellmap_assemble", "ll_cellmap_reserve", "ll_cellmap_stats", "ll_voxel_downsample_dev", "ll_transform_dev", "ll_last_features_dev", "ll_mapper_config_default", "ll_mapper_create", "ll_mapper_release",
    "ll_mapper_process_scan", "ll_mapper_pose", "ll_map_rebuild", "ll_debug_solver_cycles", "ll_state_snapshot_bytes", "ll_set_point_layout", "ll_format_pose_log", "ll_reg_state_yaml", "ll_cap_uniform", "ll_map_shard_info", "ll_shard_plan", "ll_align_cfg_default", "ll_scene_align", "ll_frame_to_pose", "ll_features_to_pointcloud2",
]


class Config(C.Structure):
    _fields_ = [("corner_curvature", C.c_float), ("surface_curvature", C.c_float), ("minimum_view_angle", C.c_float), ("livox_min_dis", C.c_float),
                ("livox_min_sigma", C.c_float), ("max_fov_deg", C.c_float), ("time_interval_pts", C.c_float), ("max_scan_points", C.c_int), ("max_features", C.c_int)]


class RegState(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("if_motion_deblur", "current_frame_index", "mapping_init_accumulate_frames", "icp_max_iterations", "cere_max_iterations",
                                       "cere_prerun_times", "icp_plane", "icp_line", "maximum_allow_residual_block", "rng_seed")] + \
               [(n, C.c_double) for n in ("para_max_angular_rate", "para_max_speed", "max_final_cost", "minimum_pt_time_stamp", "maximum_pt_time_stamp",
                                          "minimum_icp_R_diff", "minimum_icp_T_diff", "inliner_dis", "inlier_ratio", "maximum_dis_plane_for_match",
                                          "maximum_dis_line_for_match", "huber_a")] + \
               [("q_w_last", C.c_double * 4), ("t_w_last", C.c_double * 3), ("q_w_curr", C.c_double * 4), ("t_w_curr", C.c_double * 3),
                ("para_buffer_incremental", C.c_double * 7)]


class RegResult(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("status", "registered", "num_residual_blocks", "icp_iterations", "corner_used", "surf_used", "total_lm_iterations",
                                       "total_evaluations")] + \
               [("q_w_curr", C.c_double * 4), ("t_w_curr", C.c_double * 3), ("q_w_incre", C.c_double * 4), ("t_w_incre", C.c_double * 3)] + \
               [(n, C.c_double) for n in ("inlier_threshold", "final_cost", "initial_cost", "angular_diff", "t_diff")] + \
               [("gpu_ms_total", C.c_float), ("gpu_ms_knn", C.c_float), ("gpu_ms_knn_all", C.c_float), ("gpu_ms_solve_all", C.c_float),
                ("gpu_ms_select_all", C.c_float), ("gpu_ms_sort", C.c_float)]


class PipelineCfg(C.Structure):
    _fields_ = [("pieces", C.c_int), ("use_piece", C.c_int), ("extractor_leaf_corner", C.c_float), ("extractor_leaf_surf", C.c_float),
                ("mapping_leaf_corner", C.c_float), ("mapping_leaf_surf", C.c_float), ("whole_frame", C.c_int)]


class PointLayout(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("point_step", "offset_x", "offset_y", "offset_z", "offset_intensity", "intensity_datatype")]


class MapperConfig(C.Structure):
    _fields_ = [("line_resolution", C.c_float), ("plane_resolution", C.c_float), ("cell_resolution", C.c_float), ("threshold_cell_revisit", C.c_int),
                ("maximum_search_range_corner", C.c_float), ("maximum_search_range_surface", C.c_float), ("maximum_in_fov_angle", C.c_float),
                ("down_sample_replace", C.c_int), ("max_cells", C.c_int), ("matching_mode", C.c_int), ("maximum_history_size", C.c_int),
                ("reserve_map_points", C.c_int), ("reserve_store_points", C.c_int),
                ("pipeline", PipelineCfg), ("reg", RegState)]


class MapperStats(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n_corner", "n_surf", "map_corner", "map_surf", "cells_in_fov_corner", "cells_in_fov_surf", "appended_corner", "appended_surf")] + \
               [(n, C.c_float) for n in ("ms_front_end", "ms_refresh", "ms_register", "ms_append")]


class ShardInfo(C.Structure):
    _fields_ = [("rank", C.c_int), ("world", C.c_int), ("cell_size", C.c_float), ("halo_corner", C.c_float), ("halo_surf", C.c_float), ("origin", C.c_float * 3),
                ("dims", C.c_int * 3), ("kept_corner", C.c_longlong), ("kept_surf", C.c_longlong), ("total_corner", C.c_longlong), ("total_surf", C.c_longlong)]


class AlignCfg(C.Structure):
    _fields_ = [("line_res", C.c_float), ("plane_res", C.c_float), ("maximum_icp_iteration", C.c_int), ("maximum_residual_block", C.c_int),
                ("accepted_threshold", C.c_float), ("rng_seed", C.c_int), ("t_init", C.c_double * 3)]


class LoamLivoxError(RuntimeError):
    pass


_LIB = None


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    if not os.path.exists(LIB_PATH):
        raise LoamLivoxError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                             "There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, ci, cf, cd = C.c_void_p, C.c_size_t, C.c_int, C.c_float, C.c_double
    L.ll_config_default.argtypes = [C.POINTER(Config)]
    L.ll_ctx_create.argtypes = [C.POINTER(Config), ci, C.POINTER(vp)]
    L.ll_ctx_destroy.argtypes = [vp]
    L.ll_last_error.argtypes = [vp]
    L.ll_last_error.restype = C.c_char_p
    L.ll_ctx_stream.argtypes = [vp]
    L.ll_ctx_stream.restype = vp
    L.ll_ctx_sync.argtypes = [vp]
    L.ll_extract.argtypes = [vp, vp, sz, ci, ci, cd, C.POINTER(ci)]
    L.ll_extract_reset.argtypes = [vp]
    L.ll_piece_bounds.argtypes = [vp, ci, vp, vp]
    L.ll_get_features.argtypes = [vp, cf, cf, vp, C.POINTER(sz), vp, C.POINTER(sz), vp, C.POINTER(sz)]
    L.ll_extract_point_info.argtypes = [vp] + [vp] * 8
    L.ll_extract_split_idx.argtypes = [vp, vp, ci, C.POINTER(ci)]
    L.ll_voxel_downsample.argtypes = [vp, vp, sz, ci, ci, cf, vp, C.POINTER(sz)]
    L.ll_map_build.argtypes = [vp, vp, sz, vp, sz, ci, ci, C.POINTER(vp)]
    L.ll_map_build_sharded.argtypes = [vp, vp, sz, vp, sz, ci, ci, ci, ci, cf, cf, cf, C.POINTER(vp)]
    L.ll_map_shard_info.argtypes = [vp, C.POINTER(ShardInfo), vp, sz]
    L.ll_shard_plan.argtypes = [vp, vp, ci, vp]
    L.ll_align_cfg_default.argtypes = [C.POINTER(AlignCfg)]
    L.ll_scene_align.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, sz, ci, ci, C.POINTER(AlignCfg), C.POINTER(RegResult), C.POINTER(ci)]
    L.ll_map_release.argtypes = [vp]
    L.ll_map_size.argtypes = [vp, ci]
    L.ll_map_size.restype = sz
    L.ll_knn.argtypes = [vp, vp, ci, vp, sz, vp, vp]
    L.ll_reg_state_default.argtypes = [C.POINTER(RegState)]
    L.ll_reg_state_yaml.argtypes = [C.POINTER(RegState), ci]
    L.ll_cap_uniform.argtypes = [ci, ci, ci, ci]
    L.ll_cap_uniform.restype = cf
    L.ll_register.argtypes = [vp, vp, vp, sz, vp, sz, ci, ci, C.POINTER(RegState), C.POINTER(RegResult)]
    L.ll_build_blocks.argtypes = [vp, vp, vp, sz, vp, sz, ci, ci, C.POINTER(RegState), vp, vp, vp, C.POINTER(ci), C.POINTER(ci)]
    L.ll_debug_knn_blocks.argtypes = [vp, vp, vp, sz, vp, sz, ci, ci, C.POINTER(RegState), ci, vp, vp, vp, vp, vp, vp, C.POINTER(ci)]
    L.ll_normal_equations.argtypes = [vp, vp, vp]
    L.ll_solve.argtypes = [vp, ci, vp, C.POINTER(cd), C.POINTER(cd), C.POINTER(ci)]
    L.ll_transform.argtypes = [vp, vp, vp, vp, sz, ci, ci, vp]
    L.ll_scan_to_pose.argtypes = [vp, vp, vp, sz, ci, ci, cd, C.POINTER(PipelineCfg), C.POINTER(RegState), C.POINTER(RegResult), C.POINTER(ci), C.POINTER(ci)]
    L.ll_frame_to_pose.argtypes = [vp, vp, ci, vp, vp, ci, ci, vp, C.POINTER(PipelineCfg), C.POINTER(RegState), C.POINTER(RegResult), C.POINTER(ci), C.POINTER(ci)]
    L.ll_features_to_pointcloud2.argtypes = [vp, ci, vp, sz, C.POINTER(sz)]
    L.ll_comm_local_handle.argtypes = [vp, vp]
    L.ll_comm_connect.argtypes = [vp, ci, ci, vp]
    L.ll_cellmap_create.argtypes = [vp, cf, ci, ci, C.POINTER(vp)]
    L.ll_cellmap_release.argtypes = [vp]
    L.ll_cellmap_append.argtypes = [vp, vp, vp, sz, ci, ci]
    L.ll_cellmap_assemble.argtypes = [vp, vp, vp, vp, cf, cf, cf, ci, vp, sz, C.POINTER(sz), C.POINTER(ci), C.POINTER(vp)]
    L.ll_ctx_warmup.argtypes = [vp]
    L.ll_cellmap_reserve.argtypes = [vp, vp, C.c_size_t, C.c_size_t]
    L.ll_cellmap_stats.argtypes = [vp, vp, C.POINTER(ci), C.POINTER(ci), C.POINTER(ci)]
    L.ll_voxel_downsample_dev.argtypes = [vp, vp, sz, cf, vp, C.POINTER(sz)]
    L.ll_transform_dev.argtypes = [vp, vp, vp, vp, sz, vp]
    L.ll_last_features_dev.argtypes = [vp, C.POINTER(vp), C.POINTER(sz), C.POINTER(vp), C.POINTER(sz)]
    L.ll_debug_solver_cycles.argtypes = [vp, vp]
    L.ll_state_snapshot_bytes.argtypes = []
    L.ll_set_point_layout.argtypes = [vp, C.POINTER(PointLayout)]
    L.ll_format_pose_log.argtypes = [C.POINTER(RegResult), C.c_char_p, sz]
    L.ll_map_rebuild.argtypes = [vp, vp, vp, sz, vp, sz, ci, ci]
    L.ll_mapper_config_default.argtypes = [C.POINTER(MapperConfig)]
    L.ll_mapper_create.argtypes = [vp, C.POINTER(MapperConfig), C.POINTER(vp)]
    L.ll_mapper_release.argtypes = [vp]
    L.ll_mapper_process_scan.argtypes = [vp, vp, sz, ci, ci, cd, C.POINTER(RegResult), C.POINTER(MapperStats)]
    L.ll_mapper_pose.argtypes = [vp, vp, vp, C.POINTER(ci)]
    L.ll_launch_count.argtypes = [vp]
    L.ll_launch_count.restype = C.c_uint64
    _LIB = L
    return L


def default_config(**kw) -> Config:
    c = Config()
    lib().ll_config_default(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def default_reg_state(**kw) -> RegState:
    s = RegState()
    lib().ll_reg_state_default(C.byref(s))
    for k, v in kw.items():
        if isinstance(getattr(s, k), C.Array):
            getattr(s, k)[:] = list(v)
        else:
            setattr(s, k, v)
    return s


def yaml_reg_state(realtime: bool = False, **kw) -> RegState:
    """The shipped YAML values exactly (cap 200 / 150, max_allow_final_cost 2.0)."""
    s = RegState()
    lib().ll_reg_state_yaml(C.byref(s), int(bool(realtime)))
    for k, v in kw.items():
        if isinstance(getattr(s, k), C.Array):
            getattr(s, k)[:] = list(v)
        else:
            setattr(s, k, v)
    return s


def _ptr(a):
    """numpy array -> (void*, keepalive); int -> raw (device) pointer."""
    if isinstance(a, (int, np.integer)):
        return C.c_void_p(int(a))
    return C.c_void_p(a.ctypes.data)


def _pts(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    assert a.ndim == 2 and a.shape[1] in (4, 8), "points must be [n,4] (XYZI16) or [n,8] (pcl::PointXYZI)"
    return a, (LL_FMT_XYZI16 if a.shape[1] == 4 else LL_FMT_PCL32)
