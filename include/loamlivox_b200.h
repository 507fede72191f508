/* loamlivox_b200.h — C-ABI of the B200-native scan-to-map registration hot path of hku-mars/loam_livox.
 *
 * Plain C, POD structs, caller-owned memory, opaque handles, int status (0 = OK, <0 = error, never throws).
 * No global state; distinct ll_ctx objects may be used from distinct threads concurrently (one CUDA stream each),
 * which is how the reference calls the path (one Point_cloud_registration per std::async worker,
 * /root/reference/source/laser_mapping.hpp:1348,1737-1742).
 *
 * The reference has no plugin/FFI layer; the boundary is the three C++ call seams SURVEY.md §8(b) lists.
 * Each entry point below names the reference call it replaces.  Quaternions are (w,x,y,z) unless noted.
 */
#ifndef LOAMLIVOX_B200_H
#define LOAMLIVOX_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- point formats -------------------------------------------------------------------------------- */
typedef struct { float x, y, z, intensity; } ll_point;                   /* 16 B, the device format     */
typedef struct { float x, y, z, _pad0, intensity, _pad1, _pad2, _pad3; } ll_pcl_xyzi; /* == pcl::PointXYZI (32 B),
                                               the reference's PointType: /root/reference/include/tools/common.h:9 */
enum { LL_FMT_XYZI16 = 0, LL_FMT_PCL32 = 1, LL_FMT_STRIDED = 2 /* records described by ll_set_point_layout, e.g. a sensor_msgs/PointCloud2 payload */ };
enum { LL_HOST = 0, LL_DEVICE = 1 };           /* where an input pointer lives                           */

/* ---- status codes --------------------------------------------------------------------------------- */
enum {
  LL_OK = 0,
  LL_ERR_INVALID = -1,    /* bad argument                                                              */
  LL_ERR_CUDA = -2,       /* CUDA runtime error (ll_last_error has the text)                           */
  LL_ERR_CAPACITY = -3,   /* input larger than the context was created for                             */
  LL_ERR_NO_BLOCKS = -4,  /* no residual block survived the gates (reference would dereference an empty
                             std::set at point_cloud_registration.hpp:160)                              */
  LL_ERR_CAP_BINDS = -5   /* no longer returned (kept for ABI stability): the residual-block cap (:232-238,:339-345,:434-458) is implemented,
                             see ll_reg_state::rng_seed */
};

/* ---- pt_type / pt_label bit masks (livox_feature_extractor.hpp:82-103) --------------------------- */
enum { LL_PT_NORMAL = 0, LL_PT_000 = 1, LL_PT_TOO_NEAR = 2, LL_PT_REFLECTIVITY_LOW = 4, LL_PT_REFLECTIVITY_HIGH = 8,
       LL_PT_CIRCLE_EDGE = 16, LL_PT_NAN = 32, LL_PT_SMALL_VIEW_ANGLE = 64 };
enum { LL_LABEL_INVALID = -1, LL_LABEL_UNLABELED = 0, LL_LABEL_CORNER = 1, LL_LABEL_SURFACE = 2, LL_LABEL_NEAR_NAN = 4,
       LL_LABEL_NEAR_ZERO = 8 };

typedef struct ll_ctx ll_ctx;
typedef struct ll_map ll_map;

/* Context configuration.  The extractor fields are the ones Laser_feature writes into Livox_laser
 * (laser_feature_extractor.hpp:152-154,854,859); capacities size the device arenas once. */
typedef struct {
  float corner_curvature;     /* feature_extraction/corner_curvature   (YAML 0.1)   */
  float surface_curvature;    /* feature_extraction/surface_curvature  (YAML 0.005) */
  float minimum_view_angle;   /* feature_extraction/minimum_view_angle (YAML 5)     */
  float livox_min_dis;        /* feature_extraction/livox_min_dis      (0.1)        */
  float livox_min_sigma;      /* feature_extraction/livox_min_sigma    (7e-4)       */
  float max_fov_deg;          /* Livox_laser::max_fov (17)                          */
  float time_interval_pts;    /* Livox_laser::m_time_internal_pts (1e-5)            */
  int   max_scan_points;      /* capacity: raw points per scan                      */
  int   max_features;         /* capacity: corner + surface features per registration */
} ll_config;
void ll_config_default(ll_config* cfg);

int  ll_ctx_create(const ll_config* cfg, int device, ll_ctx** out);
void ll_ctx_destroy(ll_ctx* ctx);
/* Optional: run one toy registration now, so that the module loads and the first cooperative launch CUDA defers to first use (1 - 70 ms on a B200 box)
 * do not land in the first registered scan.  ll_mapper_create calls it; nothing else depends on it. */
int  ll_ctx_warmup(ll_ctx* ctx);
const char* ll_last_error(const ll_ctx* ctx);
/* CUDA stream of the context as a cudaStream_t cast to void* (all work of a context is enqueued on it). */
void* ll_ctx_stream(ll_ctx* ctx);
int  ll_ctx_sync(ll_ctx* ctx);

/* ---- S1: feature extraction ------------------------------------------------------------------------ */
/* Replaces Livox_laser::extract_laser_features (livox_feature_extractor.hpp:722-766; projection_scan_3d_2d
 * :458-607, compute_features :361-455, split_laser_scan :657-719).  `raw` is one sensor frame in scan order.
 * *n_scans receives laserCloudScans.size() (the caller drops the frame when it is <= 5,
 * laser_feature_extractor.hpp:287).  Per-scan state stays on the device for ll_get_features. */
int ll_extract(ll_ctx* ctx, const void* raw, size_t n, int fmt, int where, double stamp, int* n_scans);
/* Forget the cross-scan state of the extractor (m_first_receive_time, m_last_maximum_time_stamp): a fresh Livox_laser object. */
int ll_extract_reset(ll_ctx* ctx);
/* Piece bounds of laser_feature_extractor.hpp:313-323 (fraction of the frame covered by each piece). */
int ll_piece_bounds(ll_ctx* ctx, int pieces, float* start, float* end);
/* Replaces Livox_laser::get_features (livox_feature_extractor.hpp:219-272).  Host outputs, each sized n. */
int ll_get_features(ll_ctx* ctx, float minimum_blur, float maximum_blur, ll_point* corners, size_t* n_corners,
                    ll_point* surface, size_t* n_surface, ll_point* full, size_t* n_full);
/* Debug/parity view of the per-point state (Pt_infos, livox_feature_extractor.hpp:118-133); any pointer may be NULL. */
int ll_extract_point_info(ll_ctx* ctx, int32_t* pt_type, int32_t* pt_label, float* curvature, float* view_angle,
                          float* depth_sq2, float* time_stamp, float* polar_dis_sq2, int32_t* polar_direction);
int ll_extract_split_idx(ll_ctx* ctx, int32_t* out, int cap, int* n_out);

/* ---- a5: voxel-grid down-sampling ------------------------------------------------------------------ */
/* Replaces pcl::VoxelGrid<PointXYZI>::filter at laser_feature_extractor.hpp:372-380 and
 * laser_mapping.hpp:491,509,533-537,1367-1373,1434-1437.  `out` must hold n points. */
int ll_voxel_downsample(ll_ctx* ctx, const void* in, size_t n, int fmt, int where, float leaf, ll_point* out, size_t* n_out);

/* ---- S2: map snapshot + index ---------------------------------------------------------------------- */
/* Replaces pcl::KdTreeFLANN::setInputCloud x2 in Laser_mapping::update_buff_for_matching
 * (laser_mapping.hpp:544-545) and in the 4-argument registration overload (point_cloud_registration.hpp:596-597).
 * The two world-frame clouds are copied to HBM and indexed; the handle is immutable and may be shared. */
int  ll_map_build(ll_ctx* ctx, const void* corner, size_t n_corner, const void* surf, size_t n_surf, int fmt, int where, ll_map** out);
/* Re-index an existing snapshot in place, reusing its device buffers (the per-scan refresh, laser_mapping.hpp:533-545). Not concurrent with searches of `map`. */
int  ll_map_rebuild(ll_ctx* ctx, ll_map* map, const void* corner, size_t nc, const void* surf, size_t ns, int fmt, int where);
void ll_map_release(ll_map* map);
size_t ll_map_size(const ll_map* map, int which /*0 corner, 1 surface*/);
/* Multi-GPU (config C4): every rank is given the same two clouds and keeps (copies to HBM and indexes) only its shard: the points of the cells
 * it owns plus every point within halo_corner / halo_surf metres of one of those cells.  Cells are cubes of cell_size metres on a grid over the
 * bounding box of the whole map; in Morton order they are cut into `world` contiguous ranges of (nearly) equal point count, rank r owns range r;
 * border cells extend outwards without bound.  With halo >= sqrt(maximum_dis_line_for_match) (1.42 m) and sqrt(maximum_dis_plane_for_match)
 * (7.07 m) -- the squared-distance gates of point_cloud_registration.hpp:64-65,254,353 -- every accepted correspondence has exactly the neighbours
 * a search of the whole map finds (ll_register refuses gates wider than the halo).  ll_register on a sharded map emits residual blocks only for the
 * features whose cell (at the current pose) this rank owns and all-reduces the normal equations inside the solver kernel (ll_comm_*).
 * Indices returned by ll_knn on a sharded map refer to the shard's own compacted clouds. */
int  ll_map_build_sharded(ll_ctx* ctx, const void* corner, size_t n_corner, const void* surf, size_t n_surf, int fmt, int where,
                          int rank, int world, float cell_size, float halo_corner, float halo_surf, ll_map** out);
typedef struct { int rank, world; float cell_size, halo_corner, halo_surf; float origin[3]; int dims[3]; long long kept_corner, kept_surf, total_corner, total_surf; } ll_shard_info;
/* Grid, halo and shard sizes of a map; owner_out (dims[0]*dims[1]*dims[2] ints, x fastest; may be NULL) receives the rank owning every cell. */
int  ll_map_shard_info(const ll_map* map, ll_shard_info* info, int* owner_out, size_t owner_cap);
/* The partition rule alone (pure host code): points per cell in, owner per cell out. */
int  ll_shard_plan(const int* cell_counts, const int dims[3], int world, int* owner_out);

/* Parity hook for pcl::KdTreeFLANN::nearestKSearch(k = 5) (point_cloud_registration.hpp:249,351): world-frame
 * queries in, 5 indices (into the cloud given to ll_map_build, -1 when fewer exist) and float squared distances out. */
int ll_knn(ll_ctx* ctx, const ll_map* map, int which, const ll_point* queries, size_t nq, int32_t* idx5, float* sqdist5);

/* ---- S3: registration ------------------------------------------------------------------------------ */
/* Inputs of Point_cloud_registration: exactly what Laser_mapping::init_pointcloud_registration copies
 * (laser_mapping.hpp:1266-1297) plus the members Scene_alignment pokes (scene_alignment.hpp:233-243,292-306). */
typedef struct {
  int    if_motion_deblur;                /* m_if_motion_deblur: *_mb functors + interpolated matching */
  int    current_frame_index;             /* m_current_frame_index                                     */
  int    mapping_init_accumulate_frames;  /* m_mapping_init_accumulate_frames                          */
  int    icp_max_iterations;              /* m_para_icp_max_iterations                                 */
  int    cere_max_iterations;             /* m_para_cere_max_iterations                                */
  int    cere_prerun_times;               /* m_para_cere_prerun_times (2)                              */
  int    icp_plane, icp_line;             /* ICP_PLANE, ICP_LINE                                       */
  int    maximum_allow_residual_block;    /* m_maximum_allow_residual_block: features are pre-skipped when their class has more than 2 x this
                                             (:232-238,:339-345) and blocks dropped with probability 1 - cap/M when M exceed it (:434-458)     */
  int    rng_seed;                        /* seed of the counter-based generator that replaces the reference's std::random_device-seeded
                                             m_rand_float (tools_random.hpp:18-25): same seed, same kept blocks, on any GPU count             */
  double para_max_angular_rate;           /* m_para_max_angular_rate (deg, reject gate)                */
  double para_max_speed;                  /* m_para_max_speed (bound on |t_incre[j]|)                  */
  double max_final_cost;                  /* m_max_final_cost                                          */
  double minimum_pt_time_stamp, maximum_pt_time_stamp;
  double minimum_icp_R_diff, minimum_icp_T_diff;
  double inliner_dis, inlier_ratio;       /* m_inliner_dis (0.02), m_inlier_ratio (0.80)               */
  double maximum_dis_plane_for_match;     /* 50.0, compared with a SQUARED distance (:353)             */
  double maximum_dis_line_for_match;      /* 2.0,  compared with a SQUARED distance (:254)             */
  double huber_a;                         /* ceres::HuberLoss(0.1) (:220)                              */
  double q_w_last[4], t_w_last[3];        /* m_q_w_last, m_t_w_last                                    */
  double q_w_curr[4], t_w_curr[3];        /* m_q_w_curr, m_t_w_curr                                    */
  double para_buffer_incremental[7];      /* m_para_buffer_incremental: q (x,y,z,w) then t             */
} ll_reg_state;
/* performance_precision.yaml + launch/rosbag.launch values, EXCEPT the two knobs SURVEY.md 8(d) raises for the 30k-feature benchmark scans:
 * maximum_allow_residual_block = 1e6 (no random drop) and max_final_cost = 1e9 (the shipped 2.0 assumes <= 200 blocks). */
void ll_reg_state_default(ll_reg_state* s);
/* The shipped values exactly: config/performance_precision.yaml (realtime = 0: cap 200) or performance_realtime.yaml (realtime = 1: cap 150),
 * max_allow_final_cost 2.0, launch/rosbag.launch:9-11 (20 deg, 0.3 m). */
void ll_reg_state_yaml(ll_reg_state* s, int realtime);
/* The uniform float in [0,1) the cap draws for (seed, ICP iteration, stream 0 corner pre-skip / 1 surface pre-skip / 2 drop, index). */
float ll_cap_uniform(int seed, int icp_iteration, int stream, int index);

typedef struct {
  int    status;                 /* return value of find_out_incremental_transfrom: 1 accepted or skipped, 0 rejected */
  int    registered;             /* 1 when the ICP branch ran (:199)                                    */
  int    num_residual_blocks;    /* summary.num_residual_blocks of the last solve                       */
  int    icp_iterations, corner_used, surf_used;
  int    total_lm_iterations, total_evaluations;
  double q_w_curr[4], t_w_curr[3];   /* m_q_w_curr, m_t_w_curr                                          */
  double q_w_incre[4], t_w_incre[3]; /* m_q_w_incre (w,x,y,z), m_t_w_incre                              */
  double inlier_threshold;       /* m_inlier_threshold after the final/initial cost rescale (:559)      */
  double final_cost, initial_cost;
  double angular_diff, t_diff;   /* m_angular_diff (deg), m_t_diff                                      */
  float  gpu_ms_total, gpu_ms_knn;  /* CUDA-event timings of this call; gpu_ms_knn = first kNN launch     */
  float  gpu_ms_knn_all, gpu_ms_solve_all, gpu_ms_select_all, gpu_ms_sort; /* sums over the ICP iterations */
} ll_reg_result;

/* Replaces Point_cloud_registration::find_out_incremental_transfrom (point_cloud_registration.hpp:163-583):
 * ICP outer loop; per iteration pointAssociateToMap + 5-NN of every feature (:230-432), gates, residual blocks,
 * Solve #1 (2 iterations), inlier selection (:476-499), Solve #2, pose composition, termination (:514-531), reject
 * gate (:561-573).  Returns LL_OK and fills `out` (out->status carries the reference's 0/1); <0 on error. */
int ll_register(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t n_corner, const void* scan_surf, size_t n_surf,
                int fmt, int where, const ll_reg_state* in, ll_reg_result* out);

/* Step-by-step parity hooks (tests): one ICP iteration's residual blocks at the pose in `in`
 * (type 0 invalid / 1 line / 2 plane, a[3], v[3] per slot; slots = corner features then surface features) ... */
int ll_build_blocks(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t n_corner, const void* scan_surf, size_t n_surf,
                    int fmt, int where, const ll_reg_state* in, int32_t* type, double* a3, double* v3, int* corner_avail, int* surf_avail);
/* ... and the same launch as one ICP iteration of ll_register runs it (the kNN kernel variant the context selected, LL_KNN_TMA=1 at
 * ll_ctx_create), at ICP iteration icp_iter (the residual-block cap's pre-skip draws) and with caller-chosen seeds: seeds_in [M x 5] are the
 * neighbour ids a search starts from (-1 = none; NULL = all -1), as the previous ICP iteration leaves them.  Out: idx5 / d5 [M x 5] the
 * neighbour ids (-1 when fewer exist) and fp32 squared distances, type / a3 / v3 the slots as ll_build_blocks, *tma_variant = 1 when the
 * TMA-staged kernel ran.  A row the kernel leaves inactive (pre-skipped, non-finite or not owned) keeps its input seeds, with NaN distances. */
int ll_debug_knn_blocks(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t n_corner, const void* scan_surf, size_t n_surf, int fmt, int where,
                        const ll_reg_state* in, int icp_iter, const int32_t* seeds_in, int32_t* idx5, float* d5, int32_t* type, double* a3, double* v3,
                        int* tma_variant);
/* ... and the loss-corrected normal equations at x (q x,y,z,w ; t): out28 = 21 upper-triangular JtJ (row-major), 6 Jtr, cost. */
int ll_normal_equations(ll_ctx* ctx, const double x[7], double out28[28]);
/* ... and one ceres::Solve-equivalent on the blocks currently resident (max_iterations as in Solver::Options). */
int ll_solve(ll_ctx* ctx, int max_iterations, double x_io[7], double* initial_cost, double* final_cost, int* iterations);

/* ---- N4: loop-closure reuse of S3 ----------------------------------------------------------------------- */
/* Replaces Scene_alignment::find_tranfrom_of_two_mappings (scene_alignment.hpp:269-353) from the point where the four feature clouds exist:
 * three coarse-to-fine registrations (leaf x8, x4, x1; twice the ICP iterations at the finest) of the target keyframe's features against the source
 * keyframe's, ICP_LINE = 0, on one persistent registration object (increment and pose carry over between scales, :233-243,292-306).
 * out = the state after the last scale run (q_w_curr / t_w_curr = the transform of keyframe b into keyframe a; inlier_threshold = the score
 * Scene_alignment returns).  *scales_run <= 3 (stops early when inlier_threshold > 2 x accepted_threshold, :349-350). */
typedef struct {
  float  line_res, plane_res;          /* Scene_alignment::m_line_res / m_plane_res (0.4 / 0.4, :27-28)                                  */
  int    maximum_icp_iteration;        /* m_maximum_icp_iteration (10, :35)                                                              */
  int    maximum_residual_block;       /* m_para_scene_alignments_maximum_residual_block (5000, :34)                                     */
  float  accepted_threshold;           /* m_accepted_threshold (0.2, :36)                                                                */
  int    rng_seed;                     /* see ll_reg_state::rng_seed                                                                      */
  double t_init[3];                    /* keyframe_a->get_center() - keyframe_b->get_center() (:303)                                     */
} ll_align_cfg;
void ll_align_cfg_default(ll_align_cfg* cfg);
int  ll_scene_align(ll_ctx* ctx, const void* source_line, size_t n_sl, const void* source_plane, size_t n_sp, const void* target_line, size_t n_tl,
                    const void* target_plane, size_t n_tp, int fmt, int where, const ll_align_cfg* cfg, ll_reg_result* out, int* scales_run);

/* ---- a7: pointAssociateToMap over a cloud ----------------------------------------------------------- */
/* Replaces Point_cloud_registration::pointcloudAssociateToMap (point_cloud_registration.hpp:673-685, non-deblur
 * branch of :622-661): p_w = q*p + t in fp64, stored as fp32, intensity passed through. */
int ll_transform(ll_ctx* ctx, const double q_wxyz[4], const double t[3], const void* in, size_t n, int fmt, int where, ll_point* out);

/* ---- whole per-scan step (what Laser_feature::laserCloudHandler + Laser_mapping::process_new_scan do) ------ */
typedef struct {
  int   pieces;               /* common/piecewise_number; only piece 0 is registered (odom_mode 0, :385)    */
  int   use_piece;            /* which piece's features to register (0)                                      */
  float extractor_leaf_corner;/* laser_feature_extractor.hpp:193 (line_res)                                  */
  float extractor_leaf_surf;  /* laser_feature_extractor.hpp:192 (plane_res / 2)                             */
  float mapping_leaf_corner;  /* laser_mapping.hpp:1367-1373 (line_res)                                      */
  float mapping_leaf_surf;    /* (plane_res)                                                                 */
  int   whole_frame;          /* 1: ignore pieces, use min_blur = 0, max_blur = 1                            */
} ll_pipeline_cfg;
/* raw scan -> features -> VoxelGrid x2 -> registration against `map`, without leaving the device. */
int ll_scan_to_pose(ll_ctx* ctx, const ll_map* map, const void* raw, size_t n, int fmt, int where, double stamp,
                    const ll_pipeline_cfg* pc, const ll_reg_state* in, ll_reg_result* out, int* n_corner_used, int* n_surf_used);

/* Multi-head frames (Mid-100 = three Mid-40 heads, launch/rosbag_mid100.launch:6): ONE extractor handles the heads in turn and the per-piece feature
 * clouds of the heads are summed before the VoxelGrids (laser_feature_extractor.hpp:303-380, 339-389); then as ll_scan_to_pose.  raws / ns / stamps have n_heads
 * entries (<= 8); the context's max_scan_points must cover the whole frame.  A head whose frame has <= 5 petals contributes nothing (:287). */
int ll_frame_to_pose(ll_ctx* ctx, const ll_map* map, int n_heads, const void* const* raws, const size_t* ns, int fmt, int where, const double* stamps,
                     const ll_pipeline_cfg* pc, const ll_reg_state* in, ll_reg_result* out, int* n_corner_used, int* n_surf_used);

/* ---- a14: device-resident voxel-cell map (matching_mode 1) ---------------------------------------------- */
/* Replaces Points_cloud_map<float> as the matching path uses it (cell_map_keyframe.hpp:476-1000): `resolution` is what
 * Laser_mapping passes to set_resolution (1.0 => 0.5 m cells, :674-679), `revisit_threshold` = m_minimum_revisit_threshold
 * (common/threshold_cell_revisit).  max_cells sizes the hash table (0 = 1 Mi cells). */
typedef struct ll_cellmap ll_cellmap;
int  ll_cellmap_create(ll_ctx* ctx, float resolution, int revisit_threshold, int max_cells, ll_cellmap** out);
void ll_cellmap_release(ll_cellmap* map);
/* Points_cloud_map::append_cloud (cell_map_keyframe.hpp:619-672; first call = set_point_cloud :578-617). xyz only. */
int  ll_cellmap_append(ll_ctx* ctx, ll_cellmap* map, const void* pts, size_t n, int fmt, int where);
/* update_buff_for_matching, matching_mode 1, for one of the two maps (laser_mapping.hpp:475-516): find_cells_in_radius(t, search_range)
 * (cell_map_keyframe.hpp:761-788) + if_pt_in_fov (laser_mapping.hpp:310-324) + per-cell VoxelGrid(leaf) + optional down-sample-and-replace
 * (m_down_sample_replace).  The concatenated cloud stays on the device (*out_dev, valid until the next call on this map) and is copied to
 * out_host (cap points) when out_host != NULL.  Cells are visited in ascending (k, j, i) index order (the PCL octree order is unspecified). */
int  ll_cellmap_assemble(ll_ctx* ctx, ll_cellmap* map, const double q_w_curr[4], const double t_w_curr[3], float search_range, float fov_deg, float leaf,
                         int down_sample_replace, ll_point* out_host, size_t cap, size_t* n_out, int* cells_in_fov, const ll_point** out_dev);
/* Allocate now for `store_points` stored points and appends of up to `scan_points`: no allocation afterwards while the store stays below that. */
int  ll_cellmap_reserve(ll_ctx* ctx, ll_cellmap* map, size_t store_points, size_t scan_points);
int  ll_cellmap_stats(ll_ctx* ctx, ll_cellmap* map, int* cells, int* stored_points, int* frame_idx);

/* ---- streaming odometry: Laser_mapping::process_new_scan + update_buff_for_matching (matching_mode 0 and 1) ------------------------- */
typedef struct {
  float line_resolution, plane_resolution;      /* feature_extraction/mapping_{line,plane}_resolution (laser_mapping.hpp:661-662)          */
  float cell_resolution;                        /* m_pt_cell_resolution (1.0 => 0.5 m cells)                                               */
  int   threshold_cell_revisit;                 /* common/threshold_cell_revisit                                                           */
  float maximum_search_range_corner, maximum_search_range_surface, maximum_in_fov_angle;   /* mapping/... (:691-695)                      */
  int   down_sample_replace;                    /* m_down_sample_replace (:277)                                                            */
  int   max_cells;                              /* hash-table sizing of each cell map (0 = 1 Mi cells)                                     */
  int   matching_mode;                          /* mapping/matching_mode (:689): 0 = sliding window of the last maximum_history_size feature clouds
                                                   (:518-531,1439-1478; what both shipped YAMLs select), 1 = cells in range and in the FOV (:471-516)   */
  int   maximum_history_size;                   /* mapping/maximum_histroy_buffer (:687; YAML 400 / 200)                                   */
  int   reserve_map_points;                     /* device memory reserved at creation, per feature kind, for the match map (history window / assembled
                                                   cells, its VoxelGrid, snapshot and index): nothing is reallocated while the map stays below it
                                                   (default 4 Mi points >= maximum_history_size x down-sampled features per scan; 0 = grow on
                                                   demand, by doubling)                                                                     */
  int   reserve_store_points;                   /* same for each cell map's point store (default 4 Mi points; the store of mode 0 only ever grows) */
  ll_pipeline_cfg pipeline;                     /* feature-extraction glue (leaves, pieces)                                                */
  ll_reg_state reg;                             /* registration parameters; the poses in it are the initial pose                           */
} ll_mapper_config;
typedef struct { int n_corner, n_surf, map_corner, map_surf, cells_in_fov_corner, cells_in_fov_surf, appended_corner, appended_surf;
                 float ms_front_end, ms_refresh, ms_register, ms_append; /* host wall clock per phase, syncs included */ } ll_mapper_stats;
typedef struct ll_mapper ll_mapper;
void ll_mapper_config_default(ll_mapper_config* cfg);
int  ll_mapper_create(ll_ctx* ctx, const ll_mapper_config* cfg, ll_mapper** out);
void ll_mapper_release(ll_mapper* mapper);
/* One raw scan through process_new_scan (laser_mapping.hpp:1316-1521): features, match-map refresh from the cell maps, registration
 * (out->status 1 accepted/skipped, 0 rejected and discarded), world-frame features appended to the cell maps, pose adopted. */
int  ll_mapper_process_scan(ll_mapper* mapper, const void* raw, size_t n, int fmt, int where, double stamp, ll_reg_result* out, ll_mapper_stats* stats);
int  ll_mapper_pose(const ll_mapper* mapper, double q_wxyz[4], double t[3], int* frame_index);

/* ---- wire formats (SURVEY 8(f) N3) ---------------------------------------------------------------------------------------------- */
/* Layout of one point record of an LL_FMT_STRIDED input: what pcl::fromROSMsg (laser_feature_extractor.hpp:275) resolves by field name from a
 * sensor_msgs/PointCloud2 (point_step, the offsets of the little-endian fields x, y, z, intensity and intensity's datatype).  The payload is
 * copied to the device as it is and unpacked there into 16-byte points; n = width * height. */
enum { LL_I_NONE = 0, LL_I_FLOAT32 = 7, LL_I_UINT8 = 2, LL_I_UINT16 = 4 };   /* = sensor_msgs/PointField datatype codes (0: no intensity field -> 0.0) */
typedef struct { int point_step, offset_x, offset_y, offset_z, offset_intensity, intensity_datatype; } ll_point_layout;
int  ll_set_point_layout(ll_ctx* ctx, const ll_point_layout* layout);
/* The output side (pcl::toROSMsg, laser_feature_extractor.hpp:367-384): the feature cloud of the last registration on this context (which = 0 corners,
 * 1 surfaces; what the feature node publishes on /pc2_corners, /pc2_surface) packed on the device into PointCloud2 records of the layout above.
 * out_host may be NULL to query *n_points first. */
int  ll_features_to_pointcloud2(ll_ctx* ctx, int which, void* out_host, size_t cap_bytes, size_t* n_points);
/* One accepted scan in the format of the reference's poses.log (laser_mapping.hpp:1506-1511; the Ceres BriefReport line is not reproduced).
 * Returns the number of characters written (excluding the terminating 0), or -1 when cap is too small. */
int  ll_format_pose_log(const ll_reg_result* r, char* buf, size_t cap);

/* Size of the registration-state snapshot copied to the host once per ICP iteration (for traffic accounting). */
int  ll_state_snapshot_bytes(void);
/* Diagnostics: cycle counters of the solver's master CTA over the last registration: eval, wait-for-slowest-CTA, grid reduce, lm_step, publish, #evaluations, staging, epilogue. */
int  ll_debug_solver_cycles(ll_ctx* ctx, long long out16[16]);   /* [8..12]: fused K10 section: L1 + insert, barrier, select, barrier, drop */

/* ---- device-to-device forms used when chaining stages without leaving the GPU (outputs in caller-provided device buffers) ------------- */
int ll_voxel_downsample_dev(ll_ctx* ctx, const ll_point* in_dev, size_t n, float leaf, ll_point* out_dev, size_t* n_out);
int ll_transform_dev(ll_ctx* ctx, const double q_wxyz[4], const double t[3], const ll_point* in_dev, size_t n, ll_point* out_dev);
/* Device pointers to the features of the last ll_register / ll_scan_to_pose on this context (scan frame, corners then surfaces). */
int ll_last_features_dev(ll_ctx* ctx, const ll_point** corner_dev, size_t* n_corner, const ll_point** surf_dev, size_t* n_surf);

/* ---- multi-GPU ------------------------------------------------------------------------------------- */
/* One process per GPU.  The 28-double normal equations (+4 counters) are all-reduced inside the solver kernel
 * through peer-mapped staging buffers (CUDA IPC over NVLink); the host only exchanges the IPC handles once. */
#define LL_IPC_HANDLE_BYTES 64
int ll_comm_local_handle(ll_ctx* ctx, unsigned char handle[LL_IPC_HANDLE_BYTES]);
int ll_comm_connect(ll_ctx* ctx, int rank, int world, const unsigned char* all_handles /* world x LL_IPC_HANDLE_BYTES */);

/* number of kernel launches issued by this context since creation (bench.py's gpu_launches) */
uint64_t ll_launch_count(const ll_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* LOAMLIVOX_B200_H */
