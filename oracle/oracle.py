"""ctypes binding of oracle/liboracle.so — ORACLE, TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this module.
The shipped product path (loam_livox_b200/) never does.  PARITY UNPINNED: see oracle/orc_math.hpp.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")


class RegParams(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("if_motion_deblur", "current_frame_index", "mapping_init_accumulate_frames", "icp_max_iterations",
                                       "cere_max_iterations", "cere_prerun_times", "icp_plane", "icp_line", "maximum_allow_residual_block", "num_threads", "rng_seed", "_pad")] + \
               [(n, C.c_double) for n in ("para_max_angular_rate", "para_max_speed", "max_final_cost", "minimum_pt_time_stamp", "maximum_pt_time_stamp",
                                          "minimum_icp_R_diff", "minimum_icp_T_diff", "inliner_dis", "inlier_ratio", "maximum_dis_plane_for_match",
                                          "maximum_dis_line_for_match", "huber_a")] + \
               [("q_w_last", C.c_double * 4), ("t_w_last", C.c_double * 3), ("q_w_curr", C.c_double * 4), ("t_w_curr", C.c_double * 3),
                ("para_buffer_incremental", C.c_double * 7)]


class RegResult(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("status", "registered", "num_residual_blocks", "icp_iterations", "corner_used", "surf_used", "total_lm_iterations",
                                       "total_cost_evals", "total_jac_evals", "total_line_search_steps")] + \
               [("q_w_curr", C.c_double * 4), ("t_w_curr", C.c_double * 3), ("q_w_incre", C.c_double * 4), ("t_w_incre", C.c_double * 3)] + \
               [(n, C.c_double) for n in ("inlier_threshold", "final_cost", "initial_cost", "angular_diff", "t_diff", "seconds_knn_build", "seconds_total")]


class Trace(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("corner_avail", "surf_avail", "blocks_before_select", "blocks_after_select", "lm_iters1", "lm_iters2")] + \
               [("inlier_threshold", C.c_double), ("x1", C.c_double * 7), ("x2", C.c_double * 7)] + \
               [(n, C.c_double) for n in ("cost1_initial", "cost1_final", "cost2_initial", "cost2_final")]


def default_params(**kw) -> RegParams:
    """Precision-YAML values (/root/reference/config/performance_precision.yaml, launch/rosbag.launch:9-11) with the
    residual-block cap raised so the reference's random drop never triggers (SURVEY.md §8d)."""
    p = RegParams()
    p.if_motion_deblur = 0
    p.current_frame_index = 1000
    p.mapping_init_accumulate_frames = 50
    p.icp_max_iterations = 15
    p.cere_max_iterations = 50
    p.cere_prerun_times = 2
    p.icp_plane = 1
    p.icp_line = 1
    p.maximum_allow_residual_block = 1000000
    p.num_threads = 1
    p.para_max_angular_rate = 20.0
    p.para_max_speed = 0.3
    p.max_final_cost = 1.0e9
    p.minimum_pt_time_stamp = 0.0
    p.maximum_pt_time_stamp = 0.1
    p.minimum_icp_R_diff = 0.01
    p.minimum_icp_T_diff = 0.01
    p.inliner_dis = 0.02
    p.inlier_ratio = 0.80
    p.maximum_dis_plane_for_match = 50.0
    p.maximum_dis_line_for_match = 2.0
    p.huber_a = 0.1
    p.q_w_last[:] = [1, 0, 0, 0]
    p.t_w_last[:] = [0, 0, 0]
    p.q_w_curr[:] = [1, 0, 0, 0]
    p.t_w_curr[:] = [0, 0, 0]
    p.para_buffer_incremental[:] = [0, 0, 0, 1, 0, 0, 0]
    for k, v in kw.items():
        if isinstance(getattr(p, k), C.Array):
            getattr(p, k)[:] = list(v)
        else:
            setattr(p, k, v)
    return p


def build(force: bool = False) -> str:
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".cpp", ".hpp"))]
    # a read-only tree (a built checkout the benchmark runs from) keeps the library it was built with
    if force or not os.path.exists(so) or (os.access(_HERE, os.W_OK) and any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return so


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    so = build()   # rebuilds only when a source is newer than the library
    L = C.CDLL(so)
    L.orc_hw_threads.restype = C.c_int
    L.orc_cap_uniform.argtypes = [C.c_int] * 4
    L.orc_cap_uniform.restype = C.c_float
    L.orc_voxel_grid.argtypes = [f32p, C.c_int, C.c_float, f32p]
    L.orc_voxel_grid.restype = C.c_int
    L.orc_kdtree_build.argtypes = [f32p, C.c_int]
    L.orc_kdtree_build.restype = C.c_void_p
    L.orc_kdtree_free.argtypes = [C.c_void_p]
    L.orc_kdtree_knn.argtypes = [C.c_void_p, f32p, C.c_int, C.c_int, i32p, f32p, i32p, C.c_int]
    L.orc_knn_brute.argtypes = [f32p, C.c_int, f32p, C.c_int, C.c_int, i32p, f32p, i32p]
    L.orc_extractor_create.argtypes = [C.c_float] * 5
    L.orc_extractor_create.restype = C.c_void_p
    L.orc_extractor_free.argtypes = [C.c_void_p]
    L.orc_extractor_extract.argtypes = [C.c_void_p, f32p, C.c_int, C.c_double]
    L.orc_extractor_extract.restype = C.c_int
    L.orc_extractor_point_info.argtypes = [C.c_void_p, i32p, i32p, f32p, f32p, f32p, f32p, f32p, i32p]
    L.orc_extractor_split_idx.argtypes = [C.c_void_p, i32p, C.c_int]
    L.orc_extractor_split_idx.restype = C.c_int
    L.orc_extractor_scans.argtypes = [C.c_void_p, i32p, i32p, C.c_int]
    L.orc_extractor_scans.restype = C.c_int
    L.orc_extractor_piece_bounds.argtypes = [C.c_void_p, C.c_int, f32p, f32p]
    L.orc_extractor_get_features.argtypes = [C.c_void_p, C.c_float, C.c_float, f32p, C.POINTER(C.c_int), f32p, C.POINTER(C.c_int), f32p, C.POINTER(C.c_int)]
    L.orc_extractor_current_time.argtypes = [C.c_void_p]
    L.orc_extractor_current_time.restype = C.c_double
    L.orc_register.argtypes = [f32p, C.c_int, C.c_void_p, f32p, C.c_int, C.c_void_p, f32p, C.c_int, f32p, C.c_int, C.POINTER(RegParams), C.POINTER(RegResult),
                               C.POINTER(Trace), C.c_int, C.POINTER(C.c_int)]
    L.orc_register.restype = C.c_int
    L.orc_transform.argtypes = [f32p, C.c_int, f64p, f64p, f32p]
    L.orc_build_blocks.argtypes = [f32p, C.c_int, C.c_void_p, f32p, C.c_int, C.c_void_p, f32p, C.c_int, f32p, C.c_int, C.POINTER(RegParams), f64p, i32p, C.c_int,
                                   C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.orc_build_blocks.restype = C.c_int
    L.orc_evaluate.argtypes = [f64p, C.c_int, f64p, f64p, C.c_double, C.c_double, f64p, f64p, f64p, f64p, C.c_void_p, C.c_void_p]
    L.orc_solve.argtypes = [f64p, C.c_int, f64p, f64p, C.c_double, C.c_double, C.c_int, f64p, f64p]
    L.orc_inlier_threshold.argtypes = [f64p, C.c_int, C.c_double]
    L.orc_inlier_threshold.restype = C.c_double
    L.orc_plus.argtypes = [f64p, f64p, C.c_double, f64p]
    L.orc_cellmap_create.argtypes = [C.c_float, C.c_int]
    L.orc_cellmap_create.restype = C.c_void_p
    L.orc_cellmap_free.argtypes = [C.c_void_p]
    L.orc_cellmap_append.argtypes = [C.c_void_p, f32p, C.c_int]
    L.orc_cellmap_cells.argtypes = [C.c_void_p]
    L.orc_cellmap_points.argtypes = [C.c_void_p]
    L.orc_cellmap_frame_idx.argtypes = [C.c_void_p]
    L.orc_cellmap_assemble.argtypes = [C.c_void_p, f64p, f64p, C.c_float, C.c_float, C.c_float, C.c_int, f32p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    _LIB = L
    return L


def _c32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def voxel_grid(pts, leaf):
    pts = _c32(pts)
    out = np.empty_like(pts)
    m = lib().orc_voxel_grid(pts, pts.shape[0], leaf, out)
    return out[:m].copy()


class KdTree:
    def __init__(self, pts):
        self.pts = _c32(pts)
        self.h = lib().orc_kdtree_build(self.pts, self.pts.shape[0])

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_kdtree_free(self.h)
            self.h = None

    def knn(self, q, k=5, threads=1):
        q = _c32(q)
        n = q.shape[0]
        idx = np.empty((n, k), np.int32)
        d2 = np.empty((n, k), np.float32)
        found = np.empty(n, np.int32)
        lib().orc_kdtree_knn(self.h, q, n, k, idx, d2, found, threads)
        return idx, d2, found


def knn_brute(map_pts, q, k=5):
    map_pts, q = _c32(map_pts), _c32(q)
    n = q.shape[0]
    idx = np.empty((n, k), np.int32)
    d2 = np.empty((n, k), np.float32)
    found = np.empty(n, np.int32)
    lib().orc_knn_brute(map_pts, map_pts.shape[0], q, n, k, idx, d2, found)
    return idx, d2, found


class Extractor:
    """Livox_laser restatement.  Defaults = the values the ROS node writes into the object
    (/root/reference/config/performance_precision.yaml:14-18, laser_feature_extractor.hpp:152-154,854,859)."""

    def __init__(self, corner_curvature=0.1, surface_curvature=0.005, minimum_view_angle=5.0, min_dis=0.1, min_sigma=7e-4):
        self.h = lib().orc_extractor_create(corner_curvature, surface_curvature, minimum_view_angle, min_dis, min_sigma)
        self.n = 0

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_extractor_free(self.h)
            self.h = None

    def extract(self, raw, stamp):
        raw = _c32(raw)
        self.n = raw.shape[0]
        return lib().orc_extractor_extract(self.h, raw, self.n, float(stamp))

    def point_info(self):
        n = self.n
        o = dict(pt_type=np.empty(n, np.int32), pt_label=np.empty(n, np.int32), curvature=np.empty(n, np.float32), view_angle=np.empty(n, np.float32),
                 depth_sq2=np.empty(n, np.float32), time_stamp=np.empty(n, np.float32), polar_dis_sq2=np.empty(n, np.float32), polar_direction=np.empty(n, np.int32))
        lib().orc_extractor_point_info(self.h, o["pt_type"], o["pt_label"], o["curvature"], o["view_angle"], o["depth_sq2"], o["time_stamp"], o["polar_dis_sq2"], o["polar_direction"])
        return o

    def split_idx(self):
        buf = np.empty(self.n + 1, np.int32)
        m = lib().orc_extractor_split_idx(self.h, buf, buf.shape[0])
        return buf[:m].copy()

    def scans(self):
        a = np.empty(self.n + 1, np.int32)
        b = np.empty(self.n + 1, np.int32)
        m = lib().orc_extractor_scans(self.h, a, b, a.shape[0])
        return a[:m].copy(), b[:m].copy()

    def piece_bounds(self, pieces):
        s = np.empty(pieces, np.float32)
        e = np.empty(pieces, np.float32)
        lib().orc_extractor_piece_bounds(self.h, pieces, s, e)
        return s, e

    def get_features(self, min_blur=0.0, max_blur=1.0):
        n = self.n
        c = np.empty((n, 4), np.float32)
        s = np.empty((n, 4), np.float32)
        f = np.empty((n, 4), np.float32)
        nc, ns, nf = C.c_int(), C.c_int(), C.c_int()
        lib().orc_extractor_get_features(self.h, min_blur, max_blur, c, C.byref(nc), s, C.byref(ns), f, C.byref(nf))
        return c[:nc.value].copy(), s[:ns.value].copy(), f[:nf.value].copy()


def transform(pts, q, t):
    pts = _c32(pts)
    out = np.empty_like(pts)
    lib().orc_transform(pts, pts.shape[0], np.asarray(q, np.float64), np.asarray(t, np.float64), out)
    return out


def register(map_c, tree_c, map_s, tree_s, scan_c, scan_s, params, want_trace=False):
    map_c, map_s, scan_c, scan_s = _c32(map_c), _c32(map_s), _c32(scan_c), _c32(scan_s)
    res = RegResult()
    cap = 64
    tr = (Trace * cap)()
    ntr = C.c_int(0)
    st = lib().orc_register(map_c, map_c.shape[0], tree_c.h, map_s, map_s.shape[0], tree_s.h, scan_c, scan_c.shape[0], scan_s, scan_s.shape[0],
                            C.byref(params), C.byref(res), tr, cap, C.byref(ntr))
    if want_trace:
        return st, res, [tr[i] for i in range(ntr.value)]
    return st, res


def build_blocks(map_c, tree_c, map_s, tree_s, scan_c, scan_s, params):
    map_c, map_s, scan_c, scan_s = _c32(map_c), _c32(map_s), _c32(scan_c), _c32(scan_s)
    cap = scan_c.shape[0] + scan_s.shape[0] + 1
    blocks = np.zeros((cap, 11), np.float64)
    src = np.zeros((cap, 2), np.int32)
    ca, sa = C.c_int(), C.c_int()
    m = lib().orc_build_blocks(map_c, map_c.shape[0], tree_c.h, map_s, map_s.shape[0], tree_s.h, scan_c, scan_c.shape[0], scan_s, scan_s.shape[0],
                               C.byref(params), blocks, src, cap, C.byref(ca), C.byref(sa))
    return blocks[:m].copy(), src[:m].copy(), ca.value, sa.value


def evaluate(blocks, q_last, t_last, x, huber_a=0.1, bound=0.3, want_full=False):
    blocks = np.ascontiguousarray(blocks, np.float64)
    M = blocks.shape[0]
    cost = np.zeros(1)
    g = np.zeros(6)
    jtj = np.zeros(36)
    r = np.zeros(3 * M) if want_full else None
    J = np.zeros(18 * M) if want_full else None
    lib().orc_evaluate(blocks, M, np.asarray(q_last, np.float64), np.asarray(t_last, np.float64), huber_a, bound, np.asarray(x, np.float64), cost, g, jtj,
                       r.ctypes.data if want_full else None, J.ctypes.data if want_full else None)
    if want_full:
        return cost[0], g, jtj.reshape(6, 6), r, J.reshape(3 * M, 6)
    return cost[0], g, jtj.reshape(6, 6)


def solve(blocks, q_last, t_last, x, max_iter, huber_a=0.1, bound=0.3):
    blocks = np.ascontiguousarray(blocks, np.float64)
    x = np.array(x, np.float64)
    summ = np.zeros(9)
    lib().orc_solve(blocks, blocks.shape[0], np.asarray(q_last, np.float64), np.asarray(t_last, np.float64), huber_a, bound, max_iter, x, summ)
    keys = ("initial_cost", "final_cost", "iterations", "successful", "unsuccessful", "line_search_steps", "termination", "cost_evals", "jac_evals")
    return x, dict(zip(keys, summ))


def inlier_threshold(residuals, ratio=0.8):
    residuals = np.ascontiguousarray(residuals, np.float64)
    return lib().orc_inlier_threshold(residuals, residuals.shape[0] // 3, ratio)


def plus(x, delta, bound=0.3):
    out = np.zeros(7)
    lib().orc_plus(np.asarray(x, np.float64), np.asarray(delta, np.float64), bound, out)
    return out


def scene_align(source_line, source_plane, target_line, target_plane, t_init=(0.0, 0.0, 0.0), line_res=0.4, plane_res=0.4, maximum_icp_iteration=10,
                maximum_residual_block=5000, accepted_threshold=0.2, rng_seed=0, threads=1):
    """Scene_alignment::find_tranfrom_of_two_mappings (/root/reference/source/scene_alignment.hpp:269-353; object set-up :233-243) from the point where
    the four feature clouds exist.  One persistent Point_cloud_registration: increment and pose carry over between the three scales."""
    p = default_params(icp_line=0, icp_plane=1, max_final_cost=20000.0, para_max_speed=1000.0, para_max_angular_rate=360 * 57.3, inliner_dis=0.2,
                       current_frame_index=10000000, mapping_init_accumulate_frames=100, icp_max_iterations=maximum_icp_iteration, cere_max_iterations=50,
                       cere_prerun_times=2, maximum_allow_residual_block=maximum_residual_block, rng_seed=rng_seed, num_threads=threads,
                       t_w_curr=list(t_init), para_buffer_incremental=[0, 0, 0, 1] + list(t_init))
    res, runs = None, 0
    for scale in (8, 4, 0):
        lr, pr = max(line_res * scale, line_res), plane_res * scale
        if pr < plane_res:
            pr = plane_res
            p.icp_max_iterations = maximum_icp_iteration * 2
        sl, sp = voxel_grid(source_line, np.float32(lr)), voxel_grid(source_plane, np.float32(pr))
        tl, tp = voxel_grid(target_line, np.float32(lr)), voxel_grid(target_plane, np.float32(pr))
        runs += 1
        if sl.shape[0] == 0 or sp.shape[0] == 0:
            continue
        st, r = register(sl, KdTree(sl), sp, KdTree(sp), tl, tp, p)
        if st < 0:
            raise RuntimeError(f"oracle registration failed ({st})")
        res = r
        p.q_w_curr[:] = list(r.q_w_curr); p.t_w_curr[:] = list(r.t_w_curr)
        p.para_buffer_incremental[:] = [r.q_w_incre[1], r.q_w_incre[2], r.q_w_incre[3], r.q_w_incre[0]] + list(r.t_w_incre)
        if r.registered and r.inlier_threshold > np.float32(accepted_threshold) * 2:
            break
    return res, runs


class CellMap:
    """Points_cloud_map<float> as the matching path uses it (append_cloud, cells-in-radius + FOV + per-cell VoxelGrid)."""

    def __init__(self, resolution=1.0, revisit_threshold=2000):
        self.h = lib().orc_cellmap_create(resolution, revisit_threshold)

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_cellmap_free(self.h)
            self.h = None

    def append_cloud(self, pts):
        pts = _c32(pts)
        lib().orc_cellmap_append(self.h, pts, pts.shape[0])

    def cells(self):
        return lib().orc_cellmap_cells(self.h)

    def points(self):
        return lib().orc_cellmap_points(self.h)

    def frame_idx(self):
        return lib().orc_cellmap_frame_idx(self.h)

    def assemble(self, q, t, search_range=100.0, fov_angle=45.0, leaf=0.4, replace=True):
        cap = max(self.points(), 1)
        out = np.empty((cap, 4), np.float32)
        nt, nf = C.c_int(), C.c_int()
        n = lib().orc_cellmap_assemble(self.h, np.asarray(q, np.float64), np.asarray(t, np.float64), search_range, fov_angle, leaf, int(replace), out, cap, C.byref(nt), C.byref(nf))
        return out[:n].copy(), nf.value


class Mapper:
    """Laser_mapping::process_new_scan + update_buff_for_matching (matching_mode 0: history window; 1: cell map) glued from the oracle pieces above, single-threaded
    (/root/reference/source/laser_mapping.hpp:1316-1521, :460-566, :1266-1297).  The background refresh of the match map is run at the start
    of the next scan with the pose the previous scan ended with, which is what the reference does with maximum_parallel_thread = 1."""

    def __init__(self, params=None, line_resolution=0.1, plane_resolution=0.4, cell_resolution=1.0, revisit_threshold=2000, search_range=100.0,
                 fov_angle=45.0, replace=True, extractor_leaf_corner=0.1, extractor_leaf_surf=0.2, threads=1, matching_mode=0, maximum_history_size=400):
        self.params = params if params is not None else default_params()
        self.line_resolution, self.plane_resolution = line_resolution, plane_resolution
        self.search_range, self.fov_angle, self.replace = search_range, fov_angle, replace
        self.leaf_c, self.leaf_s = extractor_leaf_corner, extractor_leaf_surf
        self.cells_corner, self.cells_surf = CellMap(cell_resolution, revisit_threshold), CellMap(cell_resolution, revisit_threshold)
        self.ex = Extractor()
        self.q = np.array(list(self.params.q_w_curr), np.float64)
        self.t = np.array(list(self.params.t_w_curr), np.float64)
        self.matching_mode, self.maximum_history_size = matching_mode, maximum_history_size
        self.his_corner, self.his_surf = [], []                      # m_laser_cloud_{corner,surface}_history (:1446-1478)
        self.last_his_add_q, self.last_his_add_t = np.array([1.0, 0, 0, 0]), np.zeros(3)   # uninitialised in the reference: defined as identity / 0
        self.frame_index = 0
        self.last_time_stamp = 0.0
        self.dirty = False
        self.map_c = self.map_s = None
        self.tree_c = self.tree_s = None
        self.threads = threads
        self.last = {}

    def process_scan(self, raw, stamp):
        self.ex.extract(raw, stamp)
        c, s, full = self.ex.get_features(0.0, 1.0)
        c = voxel_grid(voxel_grid(c, self.leaf_c), self.line_resolution)       # laser_feature_extractor.hpp:379-380 then laser_mapping.hpp:1367-1370
        s = voxel_grid(voxel_grid(s, self.leaf_s), self.plane_resolution)      # :372-373 then :1371-1373
        # :1336-1350: time-stamp range from the full cloud; init_pointcloud_registration sees the frame index BEFORE the increment
        max_t = max(np.float32(-10000.0), full[:, 3].max()) if full.shape[0] else np.float32(-10000.0)   # find_min_max_intensity (:1243-1253)
        min_ts, max_ts = self.last_time_stamp, float(max_t)
        self.last_time_stamp = float(max_t)
        frame_index_for_reg = self.frame_index
        self.frame_index += 1
        if self.dirty:
            if self.matching_mode == 0:      # :518-531: concatenation of the history window
                z = np.zeros((0, 4), np.float32)
                mc, fc = (np.concatenate(self.his_corner) if self.his_corner else z), 0
                ms, fs = (np.concatenate(self.his_surf) if self.his_surf else z), 0
            else:
                mc, fc = self.cells_corner.assemble(self.q, self.t, self.search_range, self.fov_angle, self.line_resolution, self.replace)
                ms, fs = self.cells_surf.assemble(self.q, self.t, self.search_range, self.fov_angle, self.plane_resolution, self.replace)
            self.map_c, self.map_s = voxel_grid(mc, self.line_resolution), voxel_grid(ms, self.plane_resolution)
            self.tree_c = KdTree(self.map_c) if self.map_c.shape[0] else None
            self.tree_s = KdTree(self.map_s) if self.map_s.shape[0] else None
            self.dirty = False
            self.last.update(cells_in_fov_corner=fc, cells_in_fov_surf=fs)
        status, res = 1, None
        if self.tree_c is not None and self.tree_s is not None:
            p = RegParams.from_buffer_copy(self.params)
            p.current_frame_index = frame_index_for_reg
            p.minimum_pt_time_stamp, p.maximum_pt_time_stamp = min_ts, max_ts
            p.rng_seed = self.params.rng_seed + frame_index_for_reg
            p.num_threads = self.threads
            p.q_w_last[:] = list(self.q); p.q_w_curr[:] = list(self.q)
            p.t_w_last[:] = list(self.t); p.t_w_curr[:] = list(self.t)
            p.para_buffer_incremental[:] = [0, 0, 0, 1, 0, 0, 0]
            status, res = register(self.map_c, self.tree_c, self.map_s, self.tree_s, c, s, p)
        self.last.update(n_corner=c.shape[0], n_surf=s.shape[0], map_corner=0 if self.map_c is None else self.map_c.shape[0],
                         map_surf=0 if self.map_s is None else self.map_s.shape[0], status=status, res=res)
        if status == 0:
            return status, self.q.copy(), self.t.copy()
        q = np.array(list(res.q_w_curr)) if res is not None else self.q
        t = np.array(list(res.t_w_curr)) if res is not None else self.t
        wc = voxel_grid(transform(c, q, t), self.line_resolution) if c.shape[0] else c
        ws = voxel_grid(transform(s, q, t), self.plane_resolution) if s.shape[0] else s
        # :1439-1478: r_diff / t_diff use the pose adopted from the PREVIOUS scan (m_q_w_curr is overwritten only at :1498); steps are 0 (:83-84)
        r_diff = 2.0 * np.arccos(min(1.0, abs(float(np.dot(self.q, self.last_his_add_q))))) * 57.3
        t_diff = float(np.linalg.norm(self.t - self.last_his_add_t))
        if len(self.his_corner) < self.maximum_history_size or t_diff > 0.0 or r_diff > 0.0:
            self.last_his_add_q, self.last_his_add_t = self.q.copy(), self.t.copy()
            self.his_corner.append(wc); self.his_surf.append(ws)
        if len(self.his_corner) > self.maximum_history_size:
            self.his_corner.pop(0)
        if len(self.his_surf) > self.maximum_history_size:
            self.his_surf.pop(0)
        self.cells_corner.append_cloud(wc)
        self.cells_surf.append_cloud(ws)
        self.last.update(appended_corner=wc.shape[0], appended_surf=ws.shape[0])
        self.dirty = True
        self.q, self.t = q.copy(), t.copy()
        return status, self.q.copy(), self.t.copy()
