"""Host-side mirror of the reference's C++ interface for the hot path, over the C-ABI (ctypes).

Names, argument meaning and return conventions follow the reference so the parity tests read like its call sites:

  Livox_laser.extract_laser_features / get_features      /root/reference/source/livox_feature_extractor.hpp:722,219
  voxel_grid_filter (pcl::VoxelGrid::filter)             /root/reference/source/laser_mapping.hpp:1367-1373
  Map (update_buff_for_matching's KdTreeFLANN pair)      /root/reference/source/laser_mapping.hpp:533-559
  Point_cloud_registration.find_out_incremental_transfrom / pointcloudAssociateToMap
                                                         /root/reference/source/point_cloud_registration.hpp:163,673
Everything here is plumbing: the arithmetic runs in the CUDA kernels of libloamlivox_b200.so.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .capi import LoamLivoxError, _pts


class Context:
    """One CUDA stream + device arenas (the reference creates one Point_cloud_registration per worker thread)."""

    def __init__(self, device: int = 0, **cfg):
        self._lib = capi.lib()
        self.cfg = capi.default_config(**cfg)
        h = C.c_void_p()
        st = self._lib.ll_ctx_create(C.byref(self.cfg), device, C.byref(h))
        if st != capi.LL_OK:
            raise LoamLivoxError(f"ll_ctx_create failed ({st}): a CUDA device (sm_100a) is required, there is no CPU fallback")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self._lib.ll_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, st):
        if st != capi.LL_OK:
            raise LoamLivoxError(f"status {st}: {self._lib.ll_last_error(self.h).decode()}")

    def set_point_layout(self, point_step, offset_x=0, offset_y=4, offset_z=8, offset_intensity=12, intensity_datatype=capi.LL_I_FLOAT32):
        """Record layout of LL_FMT_STRIDED inputs (a sensor_msgs/PointCloud2 payload: what pcl::fromROSMsg resolves by field name)."""
        L = capi.PointLayout(point_step, offset_x, offset_y, offset_z, offset_intensity, intensity_datatype)
        self.check(self._lib.ll_set_point_layout(self.h, C.byref(L)))
        self._layout_step = point_step

    def warmup(self):
        """One toy registration now: first-use costs (module loads, first cooperative launch) are paid here instead of in the first real scan."""
        self.check(self._lib.ll_ctx_warmup(self.h))

    def launches(self) -> int:
        return int(self._lib.ll_launch_count(self.h))

    def sync(self):
        self.check(self._lib.ll_ctx_sync(self.h))

    def stream(self) -> int:
        return int(self._lib.ll_ctx_stream(self.h) or 0)


def format_pose_log(result: capi.RegResult) -> str:
    """One accepted scan in the reference's poses.log format (laser_mapping.hpp:1506-1511)."""
    buf = C.create_string_buffer(1024)
    n = capi.lib().ll_format_pose_log(C.byref(result), buf, 1024)
    if n < 0:
        raise LoamLivoxError("ll_format_pose_log failed")
    return buf.value.decode()


class Livox_laser:
    """Mirror of class Livox_laser (livox_feature_extractor.hpp:77)."""

    def __init__(self, ctx: Context):
        self.ctx = ctx
        self.n = 0
        ctx.check(ctx._lib.ll_extract_reset(ctx.h))   # a new Livox_laser object has no cross-scan history

    def extract_laser_features(self, laserCloudIn, time_stamp: float) -> int:
        """Returns laserCloudScans.size() (number of petals handed back; the caller drops the frame if <= 5)."""
        pts, fmt = _pts(laserCloudIn)
        self.n = pts.shape[0]
        ns = C.c_int(0)
        self.ctx.check(self.ctx._lib.ll_extract(self.ctx.h, pts.ctypes.data, self.n, fmt, capi.LL_HOST, float(time_stamp), C.byref(ns)))
        return ns.value

    def extract_from_pointcloud2(self, data: bytes, n_points: int, time_stamp: float) -> int:
        """Same, from the raw payload of a sensor_msgs/PointCloud2 (layout set with Context.set_point_layout): replaces pcl::fromROSMsg +
        extract_laser_features (laser_feature_extractor.hpp:275,285); the payload is unpacked on the device."""
        buf = np.frombuffer(data, dtype=np.uint8)
        self.n = int(n_points)
        ns = C.c_int(0)
        self.ctx.check(self.ctx._lib.ll_extract(self.ctx.h, buf.ctypes.data, self.n, capi.LL_FMT_STRIDED, capi.LL_HOST, float(time_stamp), C.byref(ns)))
        return ns.value

    def get_features(self, minimum_blur: float = 0.0, maximum_blur: float = 0.3):
        n = self.n
        c = np.empty((n, 4), np.float32)
        s = np.empty((n, 4), np.float32)
        f = np.empty((n, 4), np.float32)
        nc, ns, nf = C.c_size_t(), C.c_size_t(), C.c_size_t()
        self.ctx.check(self.ctx._lib.ll_get_features(self.ctx.h, minimum_blur, maximum_blur, c.ctypes.data, C.byref(nc), s.ctypes.data, C.byref(ns),
                                                     f.ctypes.data, C.byref(nf)))
        return c[:nc.value].copy(), s[:ns.value].copy(), f[:nf.value].copy()

    def piece_bounds(self, pieces: int):
        a = np.empty(pieces, np.float32)
        b = np.empty(pieces, np.float32)
        self.ctx.check(self.ctx._lib.ll_piece_bounds(self.ctx.h, pieces, a.ctypes.data, b.ctypes.data))
        return a, b

    def point_info(self):
        n = self.n
        o = dict(pt_type=np.empty(n, np.int32), pt_label=np.empty(n, np.int32), curvature=np.empty(n, np.float32), view_angle=np.empty(n, np.float32),
                 depth_sq2=np.empty(n, np.float32), time_stamp=np.empty(n, np.float32), polar_dis_sq2=np.empty(n, np.float32), polar_direction=np.empty(n, np.int32))
        self.ctx.check(self.ctx._lib.ll_extract_point_info(self.ctx.h, *[o[k].ctypes.data for k in
                                                                         ("pt_type", "pt_label", "curvature", "view_angle", "depth_sq2", "time_stamp", "polar_dis_sq2", "polar_direction")]))
        return o

    def split_idx(self):
        buf = np.empty(self.n + 1, np.int32)
        m = C.c_int(0)
        self.ctx.check(self.ctx._lib.ll_extract_split_idx(self.ctx.h, buf.ctypes.data, buf.shape[0], C.byref(m)))
        return buf[:m.value].copy()


def voxel_grid_filter(ctx: Context, cloud, leaf: float):
    """pcl::VoxelGrid<PointXYZI>::setLeafSize(leaf,leaf,leaf) + filter."""
    pts, fmt = _pts(cloud)
    out = np.empty((pts.shape[0], 4), np.float32)
    m = C.c_size_t(0)
    ctx.check(ctx._lib.ll_voxel_downsample(ctx.h, pts.ctypes.data, pts.shape[0], fmt, capi.LL_HOST, leaf, out.ctypes.data, C.byref(m)))
    return out[:m.value].copy()


class Map:
    """The match-map snapshot: two world-frame clouds + their exact-kNN indices (m_kdtree_{corner,surf}_from_map_last)."""

    def __init__(self, ctx: Context, corner, surf, rank: int = 0, world: int = 1, cell_size: float = 2.0):
        self.ctx = ctx
        c, fmt = _pts(corner)
        s, fmt2 = _pts(surf)
        assert fmt == fmt2
        h = C.c_void_p()
        if world > 1:
            st = ctx._lib.ll_map_build_sharded(ctx.h, c.ctypes.data, c.shape[0], s.ctypes.data, s.shape[0], fmt, capi.LL_HOST, rank, world, cell_size,
                                               2.0 ** 0.5, 50.0 ** 0.5, C.byref(h))
        else:
            st = ctx._lib.ll_map_build(ctx.h, c.ctypes.data, c.shape[0], s.ctypes.data, s.shape[0], fmt, capi.LL_HOST, C.byref(h))
        ctx.check(st)
        self.h = h

    def size(self, which):
        return int(self.ctx._lib.ll_map_size(self.h, which))

    def shard_info(self):
        """(ShardInfo, owner table [dims z,y,x] int32) of a sharded snapshot (ll_map_shard_info)."""
        info = capi.ShardInfo()
        self.ctx.check(self.ctx._lib.ll_map_shard_info(self.h, C.byref(info), None, 0))
        owner = np.zeros(int(info.dims[0]) * int(info.dims[1]) * int(info.dims[2]), np.int32)
        self.ctx.check(self.ctx._lib.ll_map_shard_info(self.h, C.byref(info), owner.ctypes.data, owner.shape[0]))
        return info, owner

    def nearestKSearch(self, which: int, queries_world):
        """k = 5 search of either tree; returns (indices [nq,5] int32, squared distances [nq,5] float32)."""
        q = np.ascontiguousarray(queries_world, np.float32)
        idx = np.empty((q.shape[0], 5), np.int32)
        d2 = np.empty((q.shape[0], 5), np.float32)
        self.ctx.check(self.ctx._lib.ll_knn(self.ctx.h, self.h, which, q.ctypes.data, q.shape[0], idx.ctypes.data, d2.ctypes.data))
        return idx, d2

    def release(self):
        if getattr(self, "h", None):
            self.ctx._lib.ll_map_release(self.h)
            self.h = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class Point_cloud_registration:
    """Mirror of class Point_cloud_registration (point_cloud_registration.hpp:38). Quaternions are (w,x,y,z)."""

    def __init__(self, ctx: Context, **state):
        self.ctx = ctx
        self.state = capi.default_reg_state(**state)
        self.result = capi.RegResult()

    # the members init_pointcloud_registration writes (laser_mapping.hpp:1266-1297) are fields of self.state
    def set_pose(self, q_wxyz, t):
        self.state.q_w_last[:] = list(q_wxyz)
        self.state.t_w_last[:] = list(t)
        self.state.q_w_curr[:] = list(q_wxyz)
        self.state.t_w_curr[:] = list(t)

    def find_out_incremental_transfrom(self, match_map: Map, laserCloudCornerStack, laserCloudSurfStack) -> int:
        c, fmt = _pts(laserCloudCornerStack)
        s, _ = _pts(laserCloudSurfStack)
        self.ctx.check(self.ctx._lib.ll_register(self.ctx.h, match_map.h, c.ctypes.data, c.shape[0], s.ctypes.data, s.shape[0], fmt, capi.LL_HOST,
                                                 C.byref(self.state), C.byref(self.result)))
        r = self.result
        self.m_q_w_curr, self.m_t_w_curr = np.array(r.q_w_curr), np.array(r.t_w_curr)
        self.m_q_w_incre, self.m_t_w_incre = np.array(r.q_w_incre), np.array(r.t_w_incre)
        self.m_inlier_threshold = r.inlier_threshold
        return r.status

    def pointcloudAssociateToMap(self, pc_in, q_wxyz=None, t=None):
        q = np.asarray(self.m_q_w_curr if q_wxyz is None else q_wxyz, np.float64)
        t = np.asarray(self.m_t_w_curr if t is None else t, np.float64)
        p, fmt = _pts(pc_in)
        out = np.empty((p.shape[0], 4), np.float32)
        self.ctx.check(self.ctx._lib.ll_transform(self.ctx.h, q.ctypes.data, t.ctypes.data, p.ctypes.data, p.shape[0], fmt, capi.LL_HOST, out.ctypes.data))
        return out

    # ---- step-by-step parity hooks
    def build_blocks(self, match_map: Map, corner, surf):
        c, fmt = _pts(corner)
        s, _ = _pts(surf)
        M = c.shape[0] + s.shape[0]
        typ = np.zeros(M, np.int32)
        a3 = np.zeros((M, 3))
        v3 = np.zeros((M, 3))
        ca, sa = C.c_int(), C.c_int()
        self.ctx.check(self.ctx._lib.ll_build_blocks(self.ctx.h, match_map.h, c.ctypes.data, c.shape[0], s.ctypes.data, s.shape[0], fmt, capi.LL_HOST, C.byref(self.state),
                                                     typ.ctypes.data, a3.ctypes.data, v3.ctypes.data, C.byref(ca), C.byref(sa)))
        return typ, a3, v3, ca.value, sa.value

    def debug_knn_blocks(self, match_map: Map, corner, surf, icp_iter: int = 0, seeds=None):
        """One ICP iteration's kNN + residual-block launch as ll_register runs it (the context's kernel variant), at ICP iteration icp_iter and
        with seeds [M,5] int32 (-1 = none; None = no seeds).  Returns (idx5 [M,5] int32, d5 [M,5] float32, type, a3, v3, tma_variant); a row the
        kernel leaves inactive keeps its seeds, with NaN distances."""
        c, fmt = _pts(corner)
        s, _ = _pts(surf)
        M = c.shape[0] + s.shape[0]
        sd = None
        if seeds is not None:
            sd = np.ascontiguousarray(seeds, np.int32)
            assert sd.shape == (M, 5)
        idx = np.empty((M, 5), np.int32)
        d2 = np.empty((M, 5), np.float32)
        typ = np.zeros(M, np.int32)
        a3 = np.zeros((M, 3))
        v3 = np.zeros((M, 3))
        tma = C.c_int(-1)
        self.ctx.check(self.ctx._lib.ll_debug_knn_blocks(self.ctx.h, match_map.h, c.ctypes.data, c.shape[0], s.ctypes.data, s.shape[0], fmt, capi.LL_HOST,
                                                         C.byref(self.state), int(icp_iter), None if sd is None else sd.ctypes.data, idx.ctypes.data,
                                                         d2.ctypes.data, typ.ctypes.data, a3.ctypes.data, v3.ctypes.data, C.byref(tma)))
        return idx, d2, typ, a3, v3, tma.value

    def normal_equations(self, x7):
        x = np.ascontiguousarray(x7, np.float64)
        out = np.zeros(28)
        self.ctx.check(self.ctx._lib.ll_normal_equations(self.ctx.h, x.ctypes.data, out.ctypes.data))
        H = np.zeros((6, 6))
        k = 0
        for i in range(6):
            for j in range(i, 6):
                H[i, j] = H[j, i] = out[k]
                k += 1
        return H, out[21:27].copy(), out[27]

    def solve(self, x7, max_iterations):
        x = np.array(x7, np.float64)
        ic, fc, it = C.c_double(), C.c_double(), C.c_int()
        self.ctx.check(self.ctx._lib.ll_solve(self.ctx.h, max_iterations, x.ctypes.data, C.byref(ic), C.byref(fc), C.byref(it)))
        return x, ic.value, fc.value, it.value


def scan_to_pose(ctx: Context, match_map: Map, raw, stamp, pipeline: capi.PipelineCfg, state: capi.RegState, where=capi.LL_HOST, n=None, fmt=None):
    """Whole per-scan step: raw scan -> features -> VoxelGrid x2 -> registration (ll_scan_to_pose)."""
    if where == capi.LL_HOST:
        pts, fmt = _pts(raw)
        ptr, n = pts.ctypes.data, pts.shape[0]
    else:
        ptr = int(raw)
    res = capi.RegResult()
    nc, ns = C.c_int(), C.c_int()
    ctx.check(ctx._lib.ll_scan_to_pose(ctx.h, match_map.h, ptr, n, fmt, where, float(stamp), C.byref(pipeline), C.byref(state), C.byref(res), C.byref(nc), C.byref(ns)))
    return res, nc.value, ns.value


def frame_to_pose(ctx: Context, match_map: Map, heads, stamps, pipeline: capi.PipelineCfg, state: capi.RegState, where=capi.LL_HOST, ns=None, fmt=None):
    """Multi-head frame (Mid-100: three Mid-40 heads): one extractor over the heads in turn, feature clouds summed, VoxelGrids, registration
    (ll_frame_to_pose; laser_feature_extractor.hpp:303-380).  heads: list of [n,4] arrays (LL_HOST) or of device pointers (LL_DEVICE, with ns)."""
    k = len(heads)
    if where == capi.LL_HOST:
        arrs = [_pts(h) for h in heads]
        fmt = arrs[0][1]
        ptrs = (C.c_void_p * k)(*[a.ctypes.data for a, _ in arrs])
        sizes = (C.c_size_t * k)(*[a.shape[0] for a, _ in arrs])
    else:
        ptrs = (C.c_void_p * k)(*[int(h) for h in heads])
        sizes = (C.c_size_t * k)(*[int(n) for n in ns])
    st = (C.c_double * k)(*[float(t) for t in stamps])
    res = capi.RegResult()
    nc, nsf = C.c_int(), C.c_int()
    ctx.check(ctx._lib.ll_frame_to_pose(ctx.h, match_map.h, k, ptrs, sizes, fmt, where, st, C.byref(pipeline), C.byref(state), C.byref(res), C.byref(nc), C.byref(nsf)))
    return res, nc.value, nsf.value


def features_to_pointcloud2(ctx: Context, which: int) -> bytes:
    """pcl::toROSMsg of the last registration's corner (0) / surface (1) features, in the layout of Context.set_point_layout (ll_features_to_pointcloud2)."""
    n = C.c_size_t()
    ctx.check(ctx._lib.ll_features_to_pointcloud2(ctx.h, which, None, 0, C.byref(n)))
    step = ctx._layout_step if hasattr(ctx, "_layout_step") else 16
    buf = np.zeros(n.value * step, np.uint8)
    if n.value:
        ctx.check(ctx._lib.ll_features_to_pointcloud2(ctx.h, which, buf.ctypes.data, buf.shape[0], C.byref(n)))
    return buf.tobytes()


class Scene_alignment:
    """Mirror of Scene_alignment::find_tranfrom_of_two_mappings from the point where the four feature clouds exist
    (/root/reference/source/scene_alignment.hpp:269-353): coarse-to-fine registration of keyframe b's features onto keyframe a's."""

    def __init__(self, ctx: Context, line_res: float = 0.4, plane_res: float = 0.4, **kw):
        self.ctx = ctx
        self.cfg = capi.AlignCfg()
        ctx._lib.ll_align_cfg_default(C.byref(self.cfg))
        self.cfg.line_res, self.cfg.plane_res = line_res, plane_res
        for k, v in kw.items():
            setattr(self.cfg, k, v)

    def find_tranfrom_of_two_mappings(self, source_line, source_plane, target_line, target_plane, t_init=(0.0, 0.0, 0.0)):
        sl, fmt = _pts(source_line)
        sp, _ = _pts(source_plane)
        tl, _ = _pts(target_line)
        tp, _ = _pts(target_plane)
        self.cfg.t_init[:] = list(t_init)
        res, runs = capi.RegResult(), C.c_int()
        self.ctx.check(self.ctx._lib.ll_scene_align(self.ctx.h, sl.ctypes.data, sl.shape[0], sp.ctypes.data, sp.shape[0], tl.ctypes.data, tl.shape[0], tp.ctypes.data, tp.shape[0],
                                                    fmt, capi.LL_HOST, C.byref(self.cfg), C.byref(res), C.byref(runs)))
        self.m_q_w_curr, self.m_t_w_curr = np.array(res.q_w_curr), np.array(res.t_w_curr)
        self.scales_run = runs.value
        return res


class Points_cloud_map:
    """Device-resident voxel-cell map as the matching path uses it (Points_cloud_map<float>, /root/reference/source/cell_map_keyframe.hpp:264;
    append_cloud :619, find_cells_in_radius :761; the consumer is update_buff_for_matching, /root/reference/source/laser_mapping.hpp:471-516)."""

    def __init__(self, ctx: Context, resolution: float = 1.0, revisit_threshold: int = 2000, max_cells: int = 0):
        self.ctx = ctx
        h = C.c_void_p()
        ctx.check(ctx._lib.ll_cellmap_create(ctx.h, float(resolution), int(revisit_threshold), int(max_cells), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.ctx._lib.ll_cellmap_release(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, store_points: int, scan_points: int = 0):
        """Allocate now for that many stored points (and appends of up to scan_points): nothing is reallocated below that."""
        self.ctx.check(self.ctx._lib.ll_cellmap_reserve(self.ctx.h, self.h, int(store_points), int(scan_points)))

    def append_cloud(self, pts):
        pts, fmt = _pts(pts)
        self.ctx.check(self.ctx._lib.ll_cellmap_append(self.ctx.h, self.h, pts.ctypes.data, pts.shape[0], fmt, capi.LL_HOST))

    def stats(self):
        c, p, f = C.c_int(), C.c_int(), C.c_int()
        self.ctx.check(self.ctx._lib.ll_cellmap_stats(self.ctx.h, self.h, C.byref(c), C.byref(p), C.byref(f)))
        return c.value, p.value, f.value

    def get_cells_size(self) -> int:
        return self.stats()[0]

    def assemble(self, q_w_curr, t_w_curr, search_range=100.0, fov_angle=45.0, leaf=0.4, replace=True):
        """cells in radius + if_pt_in_fov + per-cell VoxelGrid (+ replace) -> (n x 4 float32 cloud, cells in the FOV)."""
        q = np.ascontiguousarray(q_w_curr, np.float64)
        t = np.ascontiguousarray(t_w_curr, np.float64)
        cap = max(self.stats()[1], 1)
        out = np.empty((cap, 4), np.float32)
        n, nf, dev = C.c_size_t(), C.c_int(), C.c_void_p()
        self.ctx.check(self.ctx._lib.ll_cellmap_assemble(self.ctx.h, self.h, q.ctypes.data, t.ctypes.data, float(search_range), float(fov_angle), float(leaf), int(bool(replace)),
                                                         out.ctypes.data, cap, C.byref(n), C.byref(nf), C.byref(dev)))
        return out[:n.value].copy(), nf.value


class Laser_mapping:
    """Streaming odometry: one call per raw scan (Laser_mapping::process_new_scan, /root/reference/source/laser_mapping.hpp:1316-1521, with the
    match-map refresh of update_buff_for_matching :460-566 in matching_mode 1).  All state stays on the device."""

    def __init__(self, ctx: Context, **kw):
        self.ctx = ctx
        cfg = capi.MapperConfig()
        ctx._lib.ll_mapper_config_default(C.byref(cfg))
        reg = kw.pop("reg", None)
        pipeline = kw.pop("pipeline", None)
        if reg is not None:
            cfg.reg = reg
        if pipeline is not None:
            cfg.pipeline = pipeline
        for k, v in kw.items():
            if not hasattr(cfg, k):
                raise AttributeError(k)
            setattr(cfg, k, v)
        self.cfg = cfg
        h = C.c_void_p()
        ctx.check(ctx._lib.ll_mapper_create(ctx.h, C.byref(cfg), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            self.ctx._lib.ll_mapper_release(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process_new_scan(self, raw, stamp, where=capi.LL_HOST, n=None, fmt=None):
        if where == capi.LL_HOST:
            pts, fmt = _pts(raw)
            ptr, n = pts.ctypes.data, pts.shape[0]
        else:
            ptr = int(raw)
        res, stats = capi.RegResult(), capi.MapperStats()
        self.ctx.check(self.ctx._lib.ll_mapper_process_scan(self.h, ptr, n, fmt, where, float(stamp), C.byref(res), C.byref(stats)))
        return res, stats

    def pose(self):
        q, t, f = np.empty(4), np.empty(3), C.c_int()
        self.ctx.check(self.ctx._lib.ll_mapper_pose(self.h, q.ctypes.data, t.ctypes.data, C.byref(f)))
        return q, t, f.value
