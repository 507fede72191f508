// C-ABI of libloamlivox_b200.so (see include/loamlivox_b200.h) and the host-side ICP driver.
//
// Host logic restated from Point_cloud_registration::find_out_incremental_transfrom
// (/root/reference/source/point_cloud_registration.hpp:163-583): the gate at :199, the ICP loop :211-532 (the per-iteration work is
// four kernels: kNN+blocks, solve #1, inlier select, solve #2 + pose/termination), the threshold rescale :559 and the reject gate :561-573.
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <cstdio>
#include "common.cuh"
#include "kernels.cuh"

int launch_inlier_select(ll_ctx* ctx, const double* d_l1, int M, double ratio, double* d_sorted, double* d_unique, int* d_n_unique);

static inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

int reg_arrays(ll_ctx* ctx, int M, RegArrays* A) {
  int cap = M > ctx->cfg.max_features ? M : ctx->cfg.max_features;
  int scap = ctx->cfg.max_scan_points > cap ? ctx->cfg.max_scan_points : cap;
  size_t bytes = align256((size_t)cap * 16) * 2 + align256((size_t)cap * 24) + align256((size_t)cap * 8 + 64) * 3 + align256((size_t)ctx->num_sms * 32 * 8) + 4096 +
                 align256((size_t)cap * 20) * 2 + align256((size_t)cap * 4) * 2 + align256((size_t)scap * 16) * 4;
  LL_CUDA(ctx, ctx->reg_buf.reserve(bytes));
  char* p = ctx->reg_buf.as<char>();
  auto take = [&](size_t b) { char* r = p; p += align256(b); return r; };
  A->cap = cap;
  A->feat = (float4*)take((size_t)cap * 16); A->blk_a = (float4*)take((size_t)cap * 16); A->blk_v = (double*)take((size_t)cap * 24);
  A->l1 = (double*)take((size_t)cap * 8); A->l1_sorted = (double*)take((size_t)cap * 8 + 64); A->l1_unique = (double*)take((size_t)cap * 8);
  A->partials = (double*)take((size_t)ctx->num_sms * 32 * 8);
  A->n_unique = (int*)take(256); A->counts = (int*)take(256); A->bounds = (float*)take(256); A->pose_tmp = (double*)take(256);
  A->knn_idx = (int*)take((size_t)cap * 20); A->knn_d = (float*)take((size_t)cap * 20); A->perm = (int*)take((size_t)cap * 4);
  A->tmp_a = (float4*)take((size_t)scap * 16); A->tmp_b = (float4*)take((size_t)scap * 16); A->tmp_c = (float4*)take((size_t)scap * 16); A->tmp_d = (float4*)take((size_t)scap * 16);
  return LL_OK;
}

extern "C" {

void ll_config_default(ll_config* c) {
  c->corner_curvature = 0.1f; c->surface_curvature = 0.005f; c->minimum_view_angle = 5.0f; c->livox_min_dis = 0.1f; c->livox_min_sigma = 7e-4f;
  c->max_fov_deg = 17.0f; c->time_interval_pts = 1.0e-5f; c->max_scan_points = 400000; c->max_features = 400000;
}
void ll_reg_state_default(ll_reg_state* s) {
  memset(s, 0, sizeof(*s));
  s->if_motion_deblur = 0; s->current_frame_index = 1000; s->mapping_init_accumulate_frames = 50; s->icp_max_iterations = 15; s->cere_max_iterations = 50; s->cere_prerun_times = 2;
  s->icp_plane = 1; s->icp_line = 1; s->maximum_allow_residual_block = 1000000;
  s->para_max_angular_rate = 20.0; s->para_max_speed = 0.3; s->max_final_cost = 1.0e9; s->minimum_pt_time_stamp = 0.0; s->maximum_pt_time_stamp = 0.1;
  s->minimum_icp_R_diff = 0.01; s->minimum_icp_T_diff = 0.01; s->inliner_dis = 0.02; s->inlier_ratio = 0.80; s->maximum_dis_plane_for_match = 50.0; s->maximum_dis_line_for_match = 2.0; s->huber_a = 0.1;
  s->q_w_last[0] = 1; s->q_w_curr[0] = 1; s->para_buffer_incremental[3] = 1;
}

void ll_reg_state_yaml(ll_reg_state* s, int realtime) {
  ll_reg_state_default(s);
  s->maximum_allow_residual_block = realtime ? 150 : 200;   // config/performance_realtime.yaml:23 / performance_precision.yaml:23
  s->max_final_cost = 2.0;                                  // optimization/max_allow_final_cost
}
float ll_cap_uniform(int seed, int icp_iteration, int stream, int index) { return ll_cap_uniform_f(seed, icp_iteration, stream, index); }

int ll_ctx_create(const ll_config* cfg, int device, ll_ctx** out) {
  if (!out) return LL_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return LL_ERR_CUDA;   // no silent CPU fallback: the CUDA path is the product
  if (device < 0 || device >= ndev) return LL_ERR_INVALID;
  // ex_scatter_kernel packs the three running counts of get_features in 21 bits each; the cap on a scan is therefore 2^21 - 1 points
  if (cfg && (cfg->max_scan_points < 1 || cfg->max_scan_points >= (1 << 21) || cfg->max_features < 1)) return LL_ERR_INVALID;
  ll_ctx* ctx = new ll_ctx();
  ctx->device = device;
  if (cfg) ctx->cfg = *cfg; else ll_config_default(&ctx->cfg);
  { const char* e = getenv("LL_KNN_TMA"); ctx->knn_tma = (e && e[0] == '1') ? 1 : 0; }
  // every call is checked: the first failure wins and the half-built context is torn down by ll_ctx_destroy (which tolerates null members)
  cudaError_t e = cudaSetDevice(device);
  auto ok = [&](cudaError_t r) { if (e == cudaSuccess && r != cudaSuccess) e = r; };
  cudaDeviceProp prop; ok(cudaGetDeviceProperties(&prop, device)); ctx->num_sms = prop.multiProcessorCount;
  ok(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  ok(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
  ok(cudaStreamCreateWithFlags(&ctx->stream3, cudaStreamNonBlocking));
  ok(cudaEventCreateWithFlags(&ctx->ev_fork3, cudaEventDisableTiming)); ok(cudaEventCreateWithFlags(&ctx->ev_join3, cudaEventDisableTiming));
  ok(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming)); ok(cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
  ok(cudaEventCreateWithFlags(&ctx->ev_it[0], cudaEventDisableTiming)); ok(cudaEventCreateWithFlags(&ctx->ev_it[1], cudaEventDisableTiming));
  ok(cudaEventCreate(&ctx->ev0)); ok(cudaEventCreate(&ctx->ev1)); ok(cudaEventCreate(&ctx->ev2)); ok(cudaEventCreate(&ctx->ev3));
  for (int i = 0; i < 5 * 16 + 2; i++) ok(cudaEventCreate(&ctx->evp[i]));
  ctx->pinned_cap = 1 << 16; ok(cudaHostAlloc(&ctx->pinned, ctx->pinned_cap, cudaHostAllocDefault));
  void* dreg = nullptr; ok(cudaMalloc(&dreg, sizeof(RegDevState))); if (dreg) ok(cudaMemset(dreg, 0, sizeof(RegDevState))); ctx->d_reg = (RegDevState*)dreg;
  if (e == cudaSuccess && solve_prepare(ctx) != LL_OK) e = cudaErrorUnknown;   // per-function attributes of the solver kernels (no process-global flag: contexts are created from any thread)
  if (e != cudaSuccess) { cudaGetLastError(); ll_ctx_destroy(ctx); return LL_ERR_CUDA; }
  *out = ctx; return LL_OK;
}
void ll_ctx_destroy(ll_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream); if (ctx->stream2) cudaStreamSynchronize(ctx->stream2); if (ctx->stream3) cudaStreamSynchronize(ctx->stream3);
  ctx->scratch3.release(); if (ctx->stream3) cudaStreamDestroy(ctx->stream3); if (ctx->ev_fork3) cudaEventDestroy(ctx->ev_fork3); if (ctx->ev_join3) cudaEventDestroy(ctx->ev_join3);
  if (ctx->fg.exec) cudaGraphExecDestroy(ctx->fg.exec);
  ctx->scratch2.release(); ctx->scratch_fe.release(); if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork); if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
  for (int i = 0; i < 2; i++) if (ctx->ev_it[i]) cudaEventDestroy(ctx->ev_it[i]);
  ctx->scratch.release(); ctx->stage_in.release(); ctx->extract_buf.release(); ctx->feat_buf.release(); ctx->reg_buf.release();
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->d_reg) cudaFree(ctx->d_reg);
  if (ctx->d_sync) cudaFree(ctx->d_sync);
  if (ctx->comm_local) cudaFree(ctx->comm_local);
  for (int i = 0; i < 8; i++) if (ctx->comm_peers[i] && i != ctx->rank) cudaIpcCloseMemHandle(ctx->comm_peers[i]);
  for (int i = 0; i < 5 * 16 + 2; i++) if (ctx->evp[i]) cudaEventDestroy(ctx->evp[i]);
  if (ctx->ev0) cudaEventDestroy(ctx->ev0); if (ctx->ev1) cudaEventDestroy(ctx->ev1); if (ctx->ev2) cudaEventDestroy(ctx->ev2); if (ctx->ev3) cudaEventDestroy(ctx->ev3);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}
const char* ll_last_error(const ll_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
void* ll_ctx_stream(ll_ctx* ctx) { return (void*)ctx->stream; }
int ll_ctx_sync(ll_ctx* ctx) { cudaSetDevice(ctx->device); LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); return LL_OK; }
uint64_t ll_launch_count(const ll_ctx* ctx) { return ctx->launches; }

// ---------------------------------------------------------------------------------------------- S1
// Host half of extract_laser_features: time-stamp bookkeeping (:724-736), upload, scan time to the device.
static int extract_prepare(ll_ctx* ctx, const void* raw, size_t n, int fmt, int where, double stamp) {
  if ((int)n > ctx->cfg.max_scan_points) { ctx->set_error("scan larger than max_scan_points"); return LL_ERR_CAPACITY; }
  ExtractState& e = ctx->ex;
  LL_TRY(extract_reserve(ctx, ctx->cfg.max_scan_points));
  if (stamp <= 0.0000001 || (stamp < e.last_maximum_time_stamp)) e.current_time = e.last_maximum_time_stamp; else e.current_time = stamp - e.first_receive_time;
  if (e.first_receive_time <= 0) e.first_receive_time = stamp;
  e.n = (int)n;
  if (n > 0) e.last_maximum_time_stamp = (double)(float)(e.current_time + (double)(((float)(n - 1)) * ctx->cfg.time_interval_pts));
  LL_TRY(upload_cloud(ctx, raw, n, fmt, where, e.raw));
  double* h = (double*)((char*)ctx->pinned + 49152); *h = e.current_time;
  LL_CUDA(ctx, cudaMemcpyAsync(e.d_time, h, sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  return LL_OK;
}
static int extract_enqueue(ll_ctx* ctx) {
  ExtractState& e = ctx->ex;
  if (e.n >= 5) LL_TRY(launch_extract(ctx, e.n));
  else LL_CUDA(ctx, cudaMemsetAsync(e.d_meta, 0, 16, ctx->stream));
  return LL_OK;
}
int ll_extract(ll_ctx* ctx, const void* raw, size_t n, int fmt, int where, double stamp, int* n_scans) {
  if (!ctx || (!raw && n)) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  ExtractState& e = ctx->ex;
  LL_TRY(extract_prepare(ctx, raw, n, fmt, where, stamp));
  LL_TRY(extract_enqueue(ctx));
  if (n_scans) {
    int* h = (int*)ctx->pinned;
    LL_CUDA(ctx, cudaMemcpyAsync(h, e.d_meta, 3 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *n_scans = h[1];
  }
  return LL_OK;
}
int ll_extract_reset(ll_ctx* ctx) {
  if (!ctx) return LL_ERR_INVALID;
  ctx->ex.first_receive_time = -1; ctx->ex.current_time = 0; ctx->ex.last_maximum_time_stamp = 0; ctx->ex.n = 0;
  return LL_OK;
}
int ll_piece_bounds(ll_ctx* ctx, int pieces, float* start, float* end) {
  if (!ctx || pieces < 1 || pieces > 16) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  RegArrays A; LL_TRY(reg_arrays(ctx, 0, &A));
  LL_TRY(launch_piece_bounds(ctx, pieces, A.bounds));
  float* h = (float*)ctx->pinned;
  LL_CUDA(ctx, cudaMemcpyAsync(h, A.bounds, 2 * pieces * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < pieces; i++) { start[i] = h[2 * i]; end[i] = h[2 * i + 1]; }
  return LL_OK;
}
int ll_get_features(ll_ctx* ctx, float minimum_blur, float maximum_blur, ll_point* corners, size_t* n_corners, ll_point* surface, size_t* n_surface, ll_point* full, size_t* n_full) {
  if (!ctx) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  RegArrays A; LL_TRY(reg_arrays(ctx, 0, &A));
  LL_TRY(launch_get_features(ctx, nullptr, minimum_blur, maximum_blur, A.tmp_a, A.tmp_b, A.tmp_c, A.counts));
  int* h = (int*)ctx->pinned;
  LL_CUDA(ctx, cudaMemcpyAsync(h, A.counts, 3 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  int nc = ctx->ex.n ? h[0] : 0, ns = ctx->ex.n ? h[1] : 0, nf = ctx->ex.n ? h[2] : 0;
  if (corners && nc) LL_CUDA(ctx, cudaMemcpyAsync(corners, A.tmp_a, (size_t)nc * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (surface && ns) LL_CUDA(ctx, cudaMemcpyAsync(surface, A.tmp_b, (size_t)ns * 16, cudaMemcpyDeviceToHost, ctx->stream));
  if (full && nf) LL_CUDA(ctx, cudaMemcpyAsync(full, A.tmp_c, (size_t)nf * 16, cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (n_corners) *n_corners = nc; if (n_surface) *n_surface = ns; if (n_full) *n_full = nf;
  return LL_OK;
}
int ll_extract_point_info(ll_ctx* ctx, int32_t* pt_type, int32_t* pt_label, float* curvature, float* view_angle, float* depth_sq2, float* time_stamp, float* polar_dis_sq2, int32_t* polar_direction) {
  if (!ctx) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  ExtractState& e = ctx->ex; size_t n = e.n; cudaStream_t s = ctx->stream;
  if (pt_type) LL_CUDA(ctx, cudaMemcpyAsync(pt_type, e.pt_type, n * 4, cudaMemcpyDeviceToHost, s));
  if (pt_label) LL_CUDA(ctx, cudaMemcpyAsync(pt_label, e.pt_label, n * 4, cudaMemcpyDeviceToHost, s));
  if (curvature) LL_CUDA(ctx, cudaMemcpyAsync(curvature, e.curvature, n * 4, cudaMemcpyDeviceToHost, s));
  if (view_angle) LL_CUDA(ctx, cudaMemcpyAsync(view_angle, e.view_angle, n * 4, cudaMemcpyDeviceToHost, s));
  if (depth_sq2) LL_CUDA(ctx, cudaMemcpyAsync(depth_sq2, e.depth_sq2, n * 4, cudaMemcpyDeviceToHost, s));
  if (time_stamp) LL_CUDA(ctx, cudaMemcpyAsync(time_stamp, e.time_stamp, n * 4, cudaMemcpyDeviceToHost, s));
  if (polar_dis_sq2) LL_CUDA(ctx, cudaMemcpyAsync(polar_dis_sq2, e.polar_dis_sq2, n * 4, cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaStreamSynchronize(s));
  if (polar_direction) {
    std::vector<int8_t> tmp(n);
    LL_CUDA(ctx, cudaMemcpy(tmp.data(), e.polar_dir, n, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; i++) polar_direction[i] = tmp[i];
  }
  return LL_OK;
}
int ll_extract_split_idx(ll_ctx* ctx, int32_t* out, int cap, int* n_out) {
  if (!ctx) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  int meta[3] = {0, 0, 0};
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  LL_CUDA(ctx, cudaMemcpy(meta, ctx->ex.d_meta, sizeof(meta), cudaMemcpyDeviceToHost));
  int m = meta[0] < cap ? meta[0] : cap;
  if (m > 0) LL_CUDA(ctx, cudaMemcpy(out, ctx->ex.split_idx, (size_t)m * 4, cudaMemcpyDeviceToHost));
  if (n_out) *n_out = meta[0];
  return LL_OK;
}

// ---------------------------------------------------------------------------------------------- a5 / a7
int ll_voxel_downsample(ll_ctx* ctx, const void* in, size_t n, int fmt, int where, float leaf, ll_point* out, size_t* n_out) {
  if (!ctx || !n_out || !(leaf > 0.f)) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  *n_out = 0; if (n == 0) return LL_OK;
  LL_CUDA(ctx, ctx->feat_buf.reserve(align256(n * 16) * 2 + 512));
  float4* d_in = ctx->feat_buf.as<float4>(); float4* d_out = (float4*)((char*)d_in + align256(n * 16)); int* d_n = (int*)((char*)d_out + align256(n * 16));
  LL_TRY(upload_cloud(ctx, in, n, fmt, where, d_in));
  LL_TRY(launch_voxel_grid(ctx, d_in, (int)n, nullptr, leaf, d_out, d_n));
  int* h = (int*)ctx->pinned;
  LL_CUDA(ctx, cudaMemcpyAsync(h, d_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *n_out = (size_t)h[0];
  if (out && h[0] > 0) { LL_CUDA(ctx, cudaMemcpyAsync(out, d_out, (size_t)h[0] * 16, cudaMemcpyDeviceToHost, ctx->stream)); LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream)); }
  return LL_OK;
}
int ll_transform(ll_ctx* ctx, const double q[4], const double t[3], const void* in, size_t n, int fmt, int where, ll_point* out) {
  if (!ctx || !q || !t) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (n == 0) return LL_OK;
  LL_CUDA(ctx, ctx->feat_buf.reserve(align256(n * 16) * 2 + 512));
  float4* d_in = ctx->feat_buf.as<float4>(); float4* d_out = (float4*)((char*)d_in + align256(n * 16)); double* d_pose = (double*)((char*)d_out + align256(n * 16));
  double* h = (double*)ctx->pinned; for (int k = 0; k < 4; k++) h[k] = q[k]; for (int k = 0; k < 3; k++) h[4 + k] = t[k];
  LL_CUDA(ctx, cudaMemcpyAsync(d_pose, h, 7 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  LL_TRY(upload_cloud(ctx, in, n, fmt, where, d_in));
  LL_TRY(launch_transform(ctx, d_pose, d_in, (int)n, d_out));
  LL_CUDA(ctx, cudaMemcpyAsync(out, d_out, n * 16, cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return LL_OK;
}

int ll_voxel_downsample_dev(ll_ctx* ctx, const ll_point* in_dev, size_t n, float leaf, ll_point* out_dev, size_t* n_out) {
  if (!ctx || !n_out || !(leaf > 0.f)) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  *n_out = 0; if (n == 0) return LL_OK;
  LL_CUDA(ctx, ctx->feat_buf.reserve(512));
  int* d_n = ctx->feat_buf.as<int>();
  LL_TRY(launch_voxel_grid(ctx, (const float4*)in_dev, (int)n, nullptr, leaf, (float4*)out_dev, d_n));
  int* h = (int*)ctx->pinned;
  LL_CUDA(ctx, cudaMemcpyAsync(h, d_n, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *n_out = (size_t)h[0];
  return LL_OK;
}
int ll_transform_dev(ll_ctx* ctx, const double q[4], const double t[3], const ll_point* in_dev, size_t n, ll_point* out_dev) {
  if (!ctx || !q || !t) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (n == 0) return LL_OK;
  LL_CUDA(ctx, ctx->feat_buf.reserve(512));
  double* d_pose = (double*)((char*)ctx->feat_buf.p + 256);
  double* h = (double*)((char*)ctx->pinned + 1024); for (int k = 0; k < 4; k++) h[k] = q[k]; for (int k = 0; k < 3; k++) h[4 + k] = t[k];
  LL_CUDA(ctx, cudaMemcpyAsync(d_pose, h, 7 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
  LL_TRY(launch_transform(ctx, d_pose, (const float4*)in_dev, (int)n, (float4*)out_dev));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return LL_OK;
}
int ll_last_features_dev(ll_ctx* ctx, const ll_point** corner_dev, size_t* n_corner, const ll_point** surf_dev, size_t* n_surf) {
  if (!ctx) return LL_ERR_INVALID;
  RegArrays A; LL_TRY(reg_arrays(ctx, 0, &A));
  if (corner_dev) *corner_dev = (const ll_point*)A.feat; if (n_corner) *n_corner = (size_t)ctx->last_nc;
  if (surf_dev) *surf_dev = (const ll_point*)(A.feat + ctx->last_nc); if (n_surf) *n_surf = (size_t)ctx->last_ns;
  return LL_OK;
}

// ---------------------------------------------------------------------------------------------- S2
static int map_index(ll_ctx* ctx, ll_map* m, const void* corner, size_t nc, const void* surf, size_t ns, int fmt, int where) {
  // device clouds already in the library's layout are indexed where they lie (the tree keeps its own source-order copy)
  const bool in_place = where == LL_DEVICE && fmt == LL_FMT_XYZI16;
  const float4* d_c = (const float4*)corner; const float4* d_s = (const float4*)surf;
  int st = LL_OK;
  if (!in_place) {
    LL_CUDA(ctx, ctx->feat_buf.reserve(align256(nc * 16) + align256(ns * 16) + 512));
    float4* b = ctx->feat_buf.as<float4>(); d_c = b; d_s = (const float4*)((char*)b + align256(nc * 16));
    st = upload_cloud(ctx, corner, nc, fmt, where, (float4*)d_c);
    if (st == LL_OK) st = upload_cloud(ctx, surf, ns, fmt, where, (float4*)d_s);
    if (st != LL_OK) return st;
  }
  // the two indices side by side: corner on the side stream with its own scratch, surface on the context's stream
  cudaStream_t s = ctx->stream;
  LL_CUDA(ctx, cudaEventRecord(ctx->ev_fork, s));
  LL_CUDA(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
  st = build_bucket_tree_on(ctx, ctx->stream2, ctx->scratch2, d_c, (int)nc, &m->corner);
  const int st2 = build_bucket_tree_on(ctx, s, ctx->scratch, d_s, (int)ns, &m->surf);
  LL_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));
  LL_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev_join, 0));
  if (st == LL_OK) st = st2;
  // host inputs may be freed by the caller as soon as this returns; device inputs are consumed in stream order (the per-scan refresh never waits)
  if (st == LL_OK && where == LL_HOST && cudaStreamSynchronize(s) != cudaSuccess) st = LL_ERR_CUDA;
  return st;
}
static int map_build_common(ll_ctx* ctx, const void* corner, size_t nc, const void* surf, size_t ns, int fmt, int where, ll_map** out) {
  if (!ctx || !out) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  ll_map* m = new ll_map(); m->device = ctx->device;
  int st = map_index(ctx, m, corner, nc, surf, ns, fmt, where);
  if (st != LL_OK) { m->corner.storage.release(); m->surf.storage.release(); delete m; return st; }
  *out = m; return LL_OK;
}
// Re-index an existing snapshot in place (device buffers are reused when large enough): the per-scan refresh of
// update_buff_for_matching (laser_mapping.hpp:544-545) without an allocation per scan.  The caller must not be searching `map` concurrently.
int ll_map_rebuild(ll_ctx* ctx, ll_map* map, const void* corner, size_t nc, const void* surf, size_t ns, int fmt, int where) {
  if (!ctx || !map) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  return map_index(ctx, map, corner, nc, surf, ns, fmt, where);
}
int ll_map_build(ll_ctx* ctx, const void* corner, size_t nc, const void* surf, size_t ns, int fmt, int where, ll_map** out) {
  return map_build_common(ctx, corner, nc, surf, ns, fmt, where, out);
}
void ll_map_release(ll_map* map) {
  if (!map) return;
  cudaSetDevice(map->device);
  map->corner.storage.release(); map->surf.storage.release(); map->shard_owner.release(); delete map;
}
size_t ll_map_size(const ll_map* map, int which) { return map ? (size_t)(which == 0 ? map->corner.n : map->surf.n) : 0; }

int ll_knn(ll_ctx* ctx, const ll_map* map, int which, const ll_point* queries, size_t nq, int32_t* idx5, float* sqdist5) {
  if (!ctx || !map) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (nq == 0) return LL_OK;
  LL_CUDA(ctx, ctx->feat_buf.reserve(align256(nq * 16) + align256(nq * 20) * 2));
  float4* d_q = ctx->feat_buf.as<float4>(); int* d_idx = (int*)((char*)d_q + align256(nq * 16)); float* d_d = (float*)((char*)d_idx + align256(nq * 20));
  LL_CUDA(ctx, cudaMemcpyAsync(d_q, queries, nq * 16, cudaMemcpyHostToDevice, ctx->stream));
  LL_TRY(launch_knn_query(ctx, which == 0 ? map->corner : map->surf, d_q, (int)nq, d_idx, d_d));
  LL_CUDA(ctx, cudaMemcpyAsync(idx5, d_idx, nq * 20, cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaMemcpyAsync(sqdist5, d_d, nq * 20, cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return LL_OK;
}

// ---------------------------------------------------------------------------------------------- S3
static void fill_state(RegDevState* h, const ll_reg_state* in) {
  memset(h, 0, sizeof(RegDevState));
  for (int k = 0; k < 4; k++) { h->pose_curr[k] = in->q_w_curr[k]; h->pose_last[k] = in->q_w_last[k]; }
  for (int k = 0; k < 3; k++) { h->pose_curr[4 + k] = in->t_w_curr[k]; h->pose_last[4 + k] = in->t_w_last[k]; }
  for (int k = 0; k < 7; k++) h->x[k] = in->para_buffer_incremental[k];
  h->q_last_opt[0] = 1.0;
  h->bound = (double)(float)in->para_max_speed; h->huber_a = in->huber_a; h->inliner_dis = in->inliner_dis; h->inlier_ratio = in->inlier_ratio;
  h->min_icp_R = in->minimum_icp_R_diff; h->min_icp_T = in->minimum_icp_T_diff;
  h->cap = in->maximum_allow_residual_block; h->rng_seed = in->rng_seed;
  h->if_motion_deblur = in->if_motion_deblur ? 1 : 0; h->min_ts = in->minimum_pt_time_stamp; h->max_ts = in->maximum_pt_time_stamp;   // interp_* = 0: reset_incremtal_parameter (:120-125)
}
static KnnBlocksArgs knn_args(ll_ctx* ctx, const ll_map* map, const RegArrays& A, int nc, int ns, const ll_reg_state* in, bool debug) {
  KnnBlocksArgs a; a.corner = make_view(map->corner); a.surf = make_view(map->surf); a.feat = A.feat; a.n_corner = nc; a.n_surf = ns;
  a.pose = ctx->d_reg->pose_curr; a.max_dis_line = in->maximum_dis_line_for_match; a.max_dis_plane = in->maximum_dis_plane_for_match;
  a.icp_line = in->icp_line; a.icp_plane = in->icp_plane; a.blk_a = A.blk_a; a.blk_v = A.blk_v;
  a.corner_avail = &ctx->d_reg->corner_avail; a.surf_avail = &ctx->d_reg->surf_avail; a.n_blocks = &ctx->d_reg->n_blocks;
  a.cap = in->maximum_allow_residual_block; a.rng_seed = in->rng_seed;
  a.seed_ids = A.knn_idx; a.knn_d = debug ? A.knn_d : nullptr; a.perm = A.perm;
  ctx->solve_world = (map->world > 1 && ctx->world > 1) ? ctx->world : 1;   // replicas of the whole map never exchange anything
  a.st = ctx->d_reg; a.deblur = in->if_motion_deblur ? 1 : 0; ctx->reg_deblur = a.deblur;
  a.rank = map->rank; a.world = map->world; a.grid = map->grid; a.shard_owner = (const int*)map->shard_owner.p;
  return a;
}
static SolveArgs solve_args(ll_ctx* ctx, const RegArrays& A, int M, int mode, int max_iter) {
  SolveArgs s; s.st = ctx->d_reg; s.sync = ctx->d_sync; s.feat = A.feat; s.blk_a = A.blk_a; s.blk_v = A.blk_v; s.l1 = A.l1; s.l1_sorted_unique = A.l1_unique; s.d_n_unique = A.n_unique;
  s.partials = A.partials; s.M = M; s.max_iterations = max_iter; s.mode = mode; s.rank = ctx->rank; s.world = ctx->solve_world; s.comm_local = (double*)ctx->comm_local;
  for (int i = 0; i < 8; i++) s.comm_peer[i] = (double*)ctx->comm_peers[i];
  s.cap_check = 0; s.deblur = ctx->reg_deblur; s.prerun_iterations = 0; s.table = nullptr; s.table_mask = 0; s.uniq = nullptr; s.n_uniq = nullptr;
  return s;
}

}  // extern "C"

// Registration on features already resident in A.feat (device). Core of ll_register / ll_scan_to_pose.
int register_device(ll_ctx* ctx, const ll_map* map, const RegArrays& A, int nc, int ns, const ll_reg_state* in, ll_reg_result* out) {
  cudaStream_t s = ctx->stream;
  memset(out, 0, sizeof(*out));
  out->status = 1;
  for (int k = 0; k < 4; k++) { out->q_w_curr[k] = in->q_w_curr[k]; out->q_w_incre[k] = k == 0 ? in->para_buffer_incremental[3] : in->para_buffer_incremental[k - 1]; }
  for (int k = 0; k < 3; k++) { out->t_w_curr[k] = in->t_w_curr[k]; out->t_w_incre[k] = in->para_buffer_incremental[4 + k]; }
  // gate (:199): CORNER_MIN_MAP_NUM 0, SURFACE_MIN_MAP_NUM 50
  if (!(map->corner.n_src > 0 && map->surf.n_src > 50 && in->current_frame_index > in->mapping_init_accumulate_frames)) return LL_OK;
  const int M = nc + ns;
  ctx->last_nc = nc; ctx->last_ns = ns;
  const int cap_check = M > in->maximum_allow_residual_block ? 1 : 0;   // fewer slots than the cap: neither the pre-skip nor the drop rule can fire
  if (M == 0) { ctx->set_error("no features"); return LL_ERR_NO_BLOCKS; }
  RegDevState* h = (RegDevState*)ctx->pinned;
  fill_state(h, in);
  LL_CUDA(ctx, cudaMemcpyAsync(ctx->d_reg, h, sizeof(RegDevState), cudaMemcpyHostToDevice, s));
  LL_CUDA(ctx, cudaEventRecord(ctx->ev0, s));
  out->registered = 1;
  KnnBlocksArgs ka = knn_args(ctx, map, A, nc, ns, in, false);
  LL_CUDA(ctx, cudaMemsetAsync(A.knn_idx, 0xff, (size_t)M * LL_KNN * 4, s));   // no seeds for the first ICP iteration
  LL_CUDA(ctx, cudaEventRecord(ctx->evp[80], s));
  LL_TRY(launch_query_sort(ctx, ka, A.perm));   // spatial tiles of features (Hilbert order at the initial pose)
  LL_CUDA(ctx, cudaEventRecord(ctx->evp[81], s));
  int iter = 0; RegDevState* hs = (RegDevState*)((char*)ctx->pinned + align256(sizeof(RegDevState)));
  const bool sharded = ctx->world > 1 && map->world > 1;
  if (sharded && (map->world != ctx->world || map->rank != ctx->rank)) { ctx->set_error("map shard and context disagree on rank/world"); return LL_ERR_INVALID; }
  // (the shard was built with halo * 1.0001 + 1 mm, shard.cu: a halo handed over as the float nearest to sqrt(gate) must pass)
  if (map->world > 1 && (std::sqrt(in->maximum_dis_line_for_match) > (double)map->halo[0] * 1.0001 + 1e-3 || std::sqrt(in->maximum_dis_plane_for_match) > (double)map->halo[1] * 1.0001 + 1e-3)) {
    ctx->set_error("match gates wider than the halo this shard was built with: owner + halo search would no longer be exact"); return LL_ERR_INVALID;
  }
  if (map->world > 1 && ctx->world != map->world) { ctx->set_error("a sharded map needs a context connected to the same number of ranks (ll_comm_connect)"); return LL_ERR_INVALID; }
  if (sharded && M > ctx->cfg.max_features) { ctx->set_error("more features than max_features (exchange buffer)"); return LL_ERR_CAPACITY; }
  double* x_l1 = sharded ? (double*)((char*)ctx->comm_local + LL_COMM_X_OFF) : nullptr;
  unsigned set_cap = 1024; while (set_cap < (unsigned)(2 * M)) set_cap <<= 1;   // hash set of the L1 norms (K10)
  LL_CUDA(ctx, ctx->scratch.reserve((size_t)set_cap * 8 + 256));
  // One ICP iteration's device work + a snapshot of the 1.7 KB state into pinned slot `it & 1`.
  RegDevState* slots[2] = {hs, (RegDevState*)((char*)hs + align256(sizeof(RegDevState)))};
  auto enqueue_iteration = [&](int it) -> int {
    cudaEvent_t* e = it < 16 ? &ctx->evp[5 * it] : nullptr;
    LL_CUDA(ctx, cudaMemsetAsync(&ctx->d_reg->corner_avail, 0, 3 * sizeof(int), s));   // corner_avail, surf_avail, n_blocks
    if (sharded) LL_CUDA(ctx, cudaMemsetAsync(x_l1, 0xff, (size_t)M * sizeof(double), s));   // NaN = nobody owns a block here (peers fill it after solve #1)
    if (it == 0) LL_CUDA(ctx, cudaEventRecord(ctx->ev1, s));
    if (e) LL_CUDA(ctx, cudaEventRecord(e[0], s));
    LL_TRY(launch_knn_blocks(ctx, ka));
    if (e) LL_CUDA(ctx, cudaEventRecord(e[1], s));
    if (it == 0) LL_CUDA(ctx, cudaEventRecord(ctx->ev2, s));
    if (!sharded) {
      // one launch: solve #1 -> L1 norms -> de-duplication + order statistic -> outlier drop -> solve #2 -> pose (lm_solve_kernel, mode 4)
      SolveArgs sa = solve_args(ctx, A, M, 4, in->cere_max_iterations);
      sa.prerun_iterations = in->cere_prerun_times; sa.table = (unsigned long long*)ctx->scratch.p; sa.table_mask = set_cap - 1;
      sa.n_uniq = (int*)A.l1_sorted; sa.uniq = A.l1_sorted + 2; sa.cap_check = cap_check;
      if (e) { LL_CUDA(ctx, cudaEventRecord(e[2], s)); LL_CUDA(ctx, cudaEventRecord(e[3], s)); }
      LL_TRY(launch_solve(ctx, sa));
    } else {
      if (cap_check) LL_TRY(launch_count_exchange(ctx));
      { SolveArgs sa = solve_args(ctx, A, M, 0, in->cere_prerun_times); sa.cap_check = cap_check; LL_TRY(launch_solve(ctx, sa)); }
      if (e) LL_CUDA(ctx, cudaEventRecord(e[2], s));
      LL_TRY(launch_l1_exchange(ctx, A.l1, M));
      LL_TRY(launch_inlier_select(ctx, x_l1, M, in->inlier_ratio, A.l1_sorted, A.l1_unique, A.n_unique));
      if (e) LL_CUDA(ctx, cudaEventRecord(e[3], s));
      { SolveArgs sa = solve_args(ctx, A, M, 1, in->cere_max_iterations); sa.cap_check = cap_check; LL_TRY(launch_solve(ctx, sa)); }
    }
    if (e) LL_CUDA(ctx, cudaEventRecord(e[4], s));
    LL_CUDA(ctx, cudaMemcpyAsync(slots[it & 1], ctx->d_reg, sizeof(RegDevState), cudaMemcpyDeviceToHost, s));
    LL_CUDA(ctx, cudaEventRecord(ctx->ev_it[it & 1], s));
    return LL_OK;
  };
  // The host stays one iteration ahead: iteration k+1 is enqueued before iteration k's state is read back, so the GPU never waits for the
  // PCIe round trip of the termination test.  The kernels of an iteration enqueued after the loop has ended return at once (st->icp_done).
  const bool speculate = !sharded;
  LL_TRY(enqueue_iteration(0));
  for (iter = 0; iter < in->icp_max_iterations; iter++) {
    if (speculate && iter + 1 < in->icp_max_iterations) LL_TRY(enqueue_iteration(iter + 1));
    LL_CUDA(ctx, cudaEventSynchronize(ctx->ev_it[iter & 1]));
    hs = slots[iter & 1];
    if (hs->lm.termination == -1) {   // the iteration enqueued ahead returns at once (icp_done is set on the device); drain it before the arena is reused
      cudaStreamSynchronize(s); ctx->set_error("no residual block survived the gates / cap / inlier selection"); return LL_ERR_NO_BLOCKS;
    }
    if (hs->icp_done) break;
    if (!speculate && iter + 1 < in->icp_max_iterations) LL_TRY(enqueue_iteration(iter + 1));
  }
  LL_CUDA(ctx, cudaEventRecord(ctx->ev3, s));
  LL_CUDA(ctx, cudaEventSynchronize(ctx->ev3));
  cudaEventElapsedTime(&out->gpu_ms_total, ctx->ev0, ctx->ev3); cudaEventElapsedTime(&out->gpu_ms_knn, ctx->ev1, ctx->ev2);
  cudaEventElapsedTime(&out->gpu_ms_sort, ctx->evp[80], ctx->evp[81]);
  { const int done_iters = (iter < in->icp_max_iterations ? iter + 1 : in->icp_max_iterations);
    for (int i = 0; i < done_iters && i < 16; i++) { float a = 0, b = 0, c = 0, d = 0; cudaEvent_t* e = &ctx->evp[5 * i];
      cudaEventElapsedTime(&a, e[0], e[1]); cudaEventElapsedTime(&b, e[1], e[2]); cudaEventElapsedTime(&c, e[2], e[3]); cudaEventElapsedTime(&d, e[3], e[4]);
      out->gpu_ms_knn_all += a; out->gpu_ms_solve_all += b + d; out->gpu_ms_select_all += c; } }
  out->icp_iterations = (iter + 1 < in->icp_max_iterations) ? iter + 1 : in->icp_max_iterations;
  out->corner_used = hs->corner_avail; out->surf_used = hs->surf_avail; out->num_residual_blocks = hs->num_residual_blocks;
  out->total_lm_iterations = hs->total_lm_iterations; out->total_evaluations = hs->total_evaluations;
  for (int k = 0; k < 4; k++) out->q_w_curr[k] = hs->pose_curr[k];
  for (int k = 0; k < 3; k++) out->t_w_curr[k] = hs->pose_curr[4 + k];
  out->q_w_incre[0] = hs->x[3]; out->q_w_incre[1] = hs->x[0]; out->q_w_incre[2] = hs->x[1]; out->q_w_incre[3] = hs->x[2];
  for (int k = 0; k < 3; k++) out->t_w_incre[k] = hs->x[4 + k];
  out->final_cost = hs->final_cost; out->initial_cost = hs->initial_cost; out->angular_diff = hs->angular_diff; out->t_diff = hs->t_diff;
  out->inlier_threshold = hs->inlier_threshold * hs->final_cost / hs->initial_cost;   // :559
  const float minimize_cost = (float)hs->final_cost;
  if (hs->angular_diff > (double)(float)in->para_max_angular_rate || minimize_cost > (float)in->max_final_cost) {   // :561-573
    out->status = 0;
    for (int k = 0; k < 4; k++) out->q_w_curr[k] = in->q_w_last[k];
    for (int k = 0; k < 3; k++) out->t_w_curr[k] = in->t_w_last[k];
  }
  return LL_OK;
}

extern "C" {

int ll_register(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t nc, const void* scan_surf, size_t ns, int fmt, int where, const ll_reg_state* in, ll_reg_result* out) {
  if (!ctx || !map || !in || !out) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if ((int)(nc + ns) > ctx->cfg.max_features) { ctx->set_error("more features than max_features"); return LL_ERR_CAPACITY; }
  RegArrays A; LL_TRY(reg_arrays(ctx, (int)(nc + ns), &A));
  LL_TRY(upload_cloud(ctx, scan_corner, nc, fmt, where, A.feat));
  LL_TRY(upload_cloud(ctx, scan_surf, ns, fmt, where, A.feat + nc));
  return register_device(ctx, map, A, (int)nc, (int)ns, in, out);
}

// One tiny registration (three planes and two edges: 1240 map points, 310 features) through the whole device path, result discarded.  It pays -- once, at a
// time of the caller's choosing -- what CUDA defers to first use: the module loads of the kNN / solver / sort kernels and the first cooperative launch
// (1 - 70 ms on the GPU boxes, measured as the first registered scan of a stream: profiles/r2/c3_first_registration.txt).  ll_mapper_create calls it.
int ll_ctx_warmup(ll_ctx* ctx) {
  if (!ctx) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  std::vector<ll_point> surf, corner, fs, fc;
  auto add = [](std::vector<ll_point>& v, float x, float y, float z) { ll_point p; p.x = x; p.y = y; p.z = z; p.intensity = 0.f; v.push_back(p); };
  for (int i = 0; i < 20; i++) for (int j = 0; j < 20; j++) {
    const float u = 0.1f * i + 0.013f * (j % 3), v = 0.1f * j + 0.007f * (i % 5);
    add(surf, 1.f + u, -1.f + v, 0.f); add(surf, 1.f + u, 1.2f, 0.05f + v); add(surf, 3.2f, -1.f + u, 0.05f + v);
    if ((i * 20 + j) % 4 == 0) { add(fs, 1.f + u + 0.004f, -1.f + v - 0.003f, 0.006f); add(fs, 1.f + u, 1.195f, 0.05f + v); add(fs, 3.194f, -1.f + u, 0.05f + v); }
  }
  for (int k = 0; k < 20; k++) { add(corner, 3.2f, 1.2f, 0.1f * k); add(corner, 1.f + 0.1f * k, 1.2f, 0.f); if (k % 4 == 0) { add(fc, 3.195f, 1.197f, 0.1f * k + 0.02f); add(fc, 1.02f + 0.1f * k, 1.196f, 0.004f); } }
  if ((int)(fc.size() + fs.size()) > ctx->cfg.max_features) return LL_OK;   // a context sized for less than the toy problem: nothing to warm
  ll_map* m = nullptr;
  int st = ll_map_build(ctx, corner.data(), corner.size(), surf.data(), surf.size(), LL_FMT_XYZI16, LL_HOST, &m);
  if (st == LL_OK) {
    ll_reg_state rs; ll_reg_state_default(&rs); rs.current_frame_index = rs.mapping_init_accumulate_frames + 1;
    ll_reg_result r;
    st = ll_register(ctx, m, fc.data(), fc.size(), fs.data(), fs.size(), LL_FMT_XYZI16, LL_HOST, &rs, &r);
    if (st == LL_ERR_NO_BLOCKS) st = LL_OK;   // (nothing here depends on the outcome of the toy problem)
  }
  if (m) ll_map_release(m);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return LL_ERR_CUDA;
  return st;
}

// One ICP iteration's kNN + residual-block launch at the pose in `in`, ICP iteration icp_iter, seeded with seeds_in ([M x 5], NULL = no seeds),
// followed by the read-back of the slots; idx5 / d5 (may be NULL) receive the search's neighbour ids and squared distances.
static int blocks_hook(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t nc, const void* scan_surf, size_t ns, int fmt, int where, const ll_reg_state* in,
                       int icp_iter, const int32_t* seeds_in, int32_t* idx5, float* d5, int32_t* type, double* a3, double* v3, int* corner_avail, int* surf_avail) {
  if (!ctx || !map || !in) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const int M = (int)(nc + ns);
  if (M > ctx->cfg.max_features) return LL_ERR_CAPACITY;
  RegArrays A; LL_TRY(reg_arrays(ctx, M, &A));
  cudaStream_t s = ctx->stream;
  LL_TRY(upload_cloud(ctx, scan_corner, nc, fmt, where, A.feat));
  LL_TRY(upload_cloud(ctx, scan_surf, ns, fmt, where, A.feat + nc));
  RegDevState* h = (RegDevState*)ctx->pinned; fill_state(h, in);
  h->icp_iter = icp_iter;   // the cap's pre-skip draws depend on the ICP iteration
  LL_CUDA(ctx, cudaMemcpyAsync(ctx->d_reg, h, sizeof(RegDevState), cudaMemcpyHostToDevice, s));
  const size_t row_bytes = (size_t)M * LL_KNN * 4;
  if (seeds_in) { if (M > 0) LL_CUDA(ctx, cudaMemcpyAsync(A.knn_idx, seeds_in, row_bytes, cudaMemcpyHostToDevice, s)); }
  else LL_CUDA(ctx, cudaMemsetAsync(A.knn_idx, 0xff, row_bytes, s));
  LL_CUDA(ctx, cudaMemsetAsync(A.knn_d, 0xff, row_bytes, s));   // NaN: rows the kernel leaves inactive keep it
  { KnnBlocksArgs ka = knn_args(ctx, map, A, (int)nc, (int)ns, in, true); LL_TRY(launch_query_sort(ctx, ka, A.perm)); LL_TRY(launch_knn_blocks(ctx, ka)); }
  std::vector<float4> ba(M); std::vector<double> bv((size_t)M * 3);
  int cnt[2];
  LL_CUDA(ctx, cudaMemcpyAsync(ba.data(), A.blk_a, (size_t)M * 16, cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaMemcpyAsync(bv.data(), A.blk_v, (size_t)M * 24, cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaMemcpyAsync(cnt, &ctx->d_reg->corner_avail, 8, cudaMemcpyDeviceToHost, s));
  if (idx5 && M > 0) LL_CUDA(ctx, cudaMemcpyAsync(idx5, A.knn_idx, row_bytes, cudaMemcpyDeviceToHost, s));
  if (d5 && M > 0) LL_CUDA(ctx, cudaMemcpyAsync(d5, A.knn_d, row_bytes, cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaStreamSynchronize(s));
  for (int i = 0; i < M; i++) {
    int t; memcpy(&t, &ba[i].w, 4);
    if (type) type[i] = t;
    if (a3) { a3[3 * i] = ba[i].x; a3[3 * i + 1] = ba[i].y; a3[3 * i + 2] = ba[i].z; }
    if (v3) { v3[3 * i] = bv[3 * i]; v3[3 * i + 1] = bv[3 * i + 1]; v3[3 * i + 2] = bv[3 * i + 2]; }
  }
  if (corner_avail) *corner_avail = cnt[0]; if (surf_avail) *surf_avail = cnt[1];
  ctx->hook_slots = M;   // slot count for ll_normal_equations / ll_solve
  return LL_OK;
}
int ll_build_blocks(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t nc, const void* scan_surf, size_t ns, int fmt, int where, const ll_reg_state* in,
                    int32_t* type, double* a3, double* v3, int* corner_avail, int* surf_avail) {
  return blocks_hook(ctx, map, scan_corner, nc, scan_surf, ns, fmt, where, in, 0, nullptr, nullptr, nullptr, type, a3, v3, corner_avail, surf_avail);
}
int ll_debug_knn_blocks(ll_ctx* ctx, const ll_map* map, const void* scan_corner, size_t nc, const void* scan_surf, size_t ns, int fmt, int where,
                        const ll_reg_state* in, int icp_iter, const int32_t* seeds_in, int32_t* idx5, float* d5, int32_t* type, double* a3, double* v3,
                        int* tma_variant) {
  const int st = blocks_hook(ctx, map, scan_corner, nc, scan_surf, ns, fmt, where, in, icp_iter, seeds_in, idx5, d5, type, a3, v3, nullptr, nullptr);
  if (st == LL_OK && tma_variant) *tma_variant = ctx->knn_tma;
  return st;
}
int ll_normal_equations(ll_ctx* ctx, const double x[7], double out28[28]) {
  if (!ctx || !x || !out28) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const int M = ctx->hook_slots;
  RegArrays A; LL_TRY(reg_arrays(ctx, M, &A));
  cudaStream_t s = ctx->stream;
  LL_CUDA(ctx, cudaMemcpyAsync(ctx->d_reg->x, x, 7 * sizeof(double), cudaMemcpyHostToDevice, s));
  LL_TRY(launch_solve(ctx, solve_args(ctx, A, M, 3, 0)));
  RegDevState* hs = (RegDevState*)((char*)ctx->pinned + align256(sizeof(RegDevState)));
  LL_CUDA(ctx, cudaMemcpyAsync(hs, ctx->d_reg, sizeof(RegDevState), cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaStreamSynchronize(s));
  for (int i = 0; i < 21; i++) out28[i] = hs->lm.H[i];
  for (int i = 0; i < 6; i++) out28[21 + i] = hs->lm.g[i];
  out28[27] = hs->lm.x_cost;
  return LL_OK;
}
int ll_solve(ll_ctx* ctx, int max_iterations, double x_io[7], double* initial_cost, double* final_cost, int* iterations) {
  if (!ctx || !x_io) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const int M = ctx->hook_slots;
  RegArrays A; LL_TRY(reg_arrays(ctx, M, &A));
  cudaStream_t s = ctx->stream;
  LL_CUDA(ctx, cudaMemcpyAsync(ctx->d_reg->x, x_io, 7 * sizeof(double), cudaMemcpyHostToDevice, s));
  LL_TRY(launch_solve(ctx, solve_args(ctx, A, M, 2, max_iterations)));
  RegDevState* hs = (RegDevState*)((char*)ctx->pinned + align256(sizeof(RegDevState)));
  LL_CUDA(ctx, cudaMemcpyAsync(hs, ctx->d_reg, sizeof(RegDevState), cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaStreamSynchronize(s));
  for (int k = 0; k < 7; k++) x_io[k] = hs->x[k];
  if (initial_cost) *initial_cost = hs->lm.initial_cost; if (final_cost) *final_cost = hs->lm.final_cost; if (iterations) *iterations = hs->lm.iteration;
  return LL_OK;
}

int ll_set_point_layout(ll_ctx* ctx, const ll_point_layout* L) {
  if (!ctx || !L) return LL_ERR_INVALID;
  const int isz = L->intensity_datatype == LL_I_FLOAT32 ? 4 : L->intensity_datatype == LL_I_UINT16 ? 2 : L->intensity_datatype == LL_I_UINT8 ? 1 : 0;
  if (L->intensity_datatype != LL_I_NONE && isz == 0) { ctx->set_error("unsupported intensity datatype"); return LL_ERR_INVALID; }
  const int offs[3] = {L->offset_x, L->offset_y, L->offset_z};
  for (int k = 0; k < 3; k++) if (offs[k] < 0 || offs[k] + 4 > L->point_step) { ctx->set_error("field outside the point record"); return LL_ERR_INVALID; }
  if (isz && (L->offset_intensity < 0 || L->offset_intensity + isz > L->point_step)) { ctx->set_error("intensity outside the point record"); return LL_ERR_INVALID; }
  ctx->layout = *L;
  return LL_OK;
}
// pcl::toROSMsg for the feature clouds the feature node publishes (laser_feature_extractor.hpp:367-384): the features of the last ll_scan_to_pose /
// ll_register / ll_frame_to_pose on this context (which = 0 corners, 1 surfaces; scan frame) as PointCloud2 records in the layout of ll_set_point_layout.
int ll_features_to_pointcloud2(ll_ctx* ctx, int which, void* out_host, size_t cap_bytes, size_t* n_points) {
  if (!ctx || !n_points || (which != 0 && which != 1)) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  RegArrays A; LL_TRY(reg_arrays(ctx, 0, &A));
  const int n = which == 0 ? ctx->last_nc : ctx->last_ns;
  const float4* src = which == 0 ? A.feat : A.feat + ctx->last_nc;
  *n_points = (size_t)n;
  const size_t bytes = (size_t)n * (size_t)ctx->layout.point_step;
  if (!out_host || n == 0) return LL_OK;
  if (cap_bytes < bytes) { ctx->set_error("output buffer smaller than n * point_step"); return LL_ERR_CAPACITY; }
  LL_CUDA(ctx, ctx->stage_in.reserve(bytes));
  LL_TRY(launch_pack_strided(ctx, src, n, ctx->stage_in.as<unsigned char>()));
  LL_CUDA(ctx, cudaMemcpyAsync(out_host, ctx->stage_in.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return LL_OK;
}
int ll_format_pose_log(const ll_reg_result* r, char* buf, size_t cap) {
  if (!r || !buf) return -1;
  const int n = snprintf(buf, cap, "--------------------\nCurr_Q = %f,%f,%f,%f\r\nCurr_T = %f,%f,%f\r\nIncre_Q = %f,%f,%f,%f\r\nIncre_T = %f,%f,%f\r\nCost=%f,blk_size = %d \r\n",
                         r->q_w_curr[0], r->q_w_curr[1], r->q_w_curr[2], r->q_w_curr[3], r->t_w_curr[0], r->t_w_curr[1], r->t_w_curr[2],
                         r->q_w_incre[0], r->q_w_incre[1], r->q_w_incre[2], r->q_w_incre[3], r->t_w_incre[0], r->t_w_incre[1], r->t_w_incre[2],
                         r->final_cost, r->num_residual_blocks);
  return (n < 0 || (size_t)n >= cap) ? -1 : n;
}
// Bytes read back per ICP iteration (the device-side registration state snapshot): what bench.py counts as d2h traffic.
int ll_state_snapshot_bytes(void) { return (int)sizeof(RegDevState); }
// Diagnostics: the master CTA's cycle counters of the last registration (kernels.cuh: RegDevState::prof).
int ll_debug_solver_cycles(ll_ctx* ctx, long long out8[16]) {
  if (!ctx || !out8) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  LL_CUDA(ctx, cudaMemcpyAsync(out8, ctx->d_reg->prof, 16 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  LL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return LL_OK;
}

// ---------------------------------------------------------------------------------------------- whole per-scan step
}  // extern "C"

// Laser_feature::laserCloudHandler for one frame, on the device: extraction, piece bounds, get_features, the extractor's VoxelGrids
// (laser_feature_extractor.hpp:285-380) and the mapping node's input VoxelGrids (laser_mapping.hpp:1367-1373).  Leaves the features in
// A.feat (corners then surfaces).  *dropped = 1 when the frame has <= 5 petals (:287).
// Everything of the front end that is enqueued on the device, in the order the reference runs it; counts land in pinned memory.
static int front_end_enqueue(ll_ctx* ctx, const ll_pipeline_cfg* pc, const RegArrays& A, int ncap) {
  cudaStream_t s = ctx->stream;
  const bool petals_aside = pc->whole_frame && ctx->ex.n >= 5;   // nothing downstream of get_features reads the petal bookkeeping then
  if (petals_aside) {
    LL_TRY(launch_extract_points(ctx, ctx->ex.n));
    LL_CUDA(ctx, cudaEventRecord(ctx->ev_fork3, s));
    LL_CUDA(ctx, cudaStreamWaitEvent(ctx->stream3, ctx->ev_fork3, 0));
    LL_TRY(launch_extract_petals(ctx, ctx->ex.n, ctx->stream3, ctx->scratch3));
    LL_CUDA(ctx, cudaEventRecord(ctx->ev_join3, ctx->stream3));
  } else LL_TRY(extract_enqueue(ctx));
  const float* d_bounds = nullptr;
  if (!pc->whole_frame) { LL_TRY(launch_piece_bounds(ctx, pc->pieces, A.bounds)); d_bounds = A.bounds + 2 * pc->use_piece; }
  LL_TRY(launch_get_features(ctx, d_bounds, 0.f, 1.f, A.tmp_a, A.tmp_b, nullptr, A.counts));
  int* cnt = A.counts;   // [0] corners [1] surf [2] full [4..7] VoxelGrid outputs
  // corner chain on the side stream, surface chain on the main stream (laser_feature_extractor.hpp:372-380 then laser_mapping.hpp:1367-1373)
  LL_CUDA(ctx, cudaEventRecord(ctx->ev_fork, s));
  LL_CUDA(ctx, cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
  LL_TRY(launch_voxel_grid_on(ctx, ctx->stream2, ctx->scratch2, A.tmp_a, ncap, cnt + 0, pc->extractor_leaf_corner, A.tmp_d, cnt + 4));
  LL_TRY(launch_voxel_grid_on(ctx, ctx->stream2, ctx->scratch2, A.tmp_d, ncap, cnt + 4, pc->mapping_leaf_corner, A.tmp_a, cnt + 5));
  LL_CUDA(ctx, cudaEventRecord(ctx->ev_join, ctx->stream2));
  LL_TRY(launch_voxel_grid(ctx, A.tmp_b, ncap, cnt + 1, pc->extractor_leaf_surf, A.tmp_c, cnt + 6));
  LL_TRY(launch_voxel_grid(ctx, A.tmp_c, ncap, cnt + 6, pc->mapping_leaf_surf, A.tmp_b, cnt + 7));
  LL_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev_join, 0));
  if (petals_aside) LL_CUDA(ctx, cudaStreamWaitEvent(s, ctx->ev_join3, 0));
  int* h = (int*)ctx->pinned + 8192;
  LL_CUDA(ctx, cudaMemcpyAsync(h, cnt, 12 * sizeof(int), cudaMemcpyDeviceToHost, s));   // [10], [11]: min / max time stamp of the full cloud
  LL_CUDA(ctx, cudaMemcpyAsync(h + 12, ctx->ex.d_meta, 12, cudaMemcpyDeviceToHost, s));
  return LL_OK;
}

int scan_front_end(ll_ctx* ctx, const void* raw, size_t n, int fmt, int where, double stamp, const ll_pipeline_cfg* pc, const RegArrays& A, int* nc_out, int* ns_out, int* dropped) {
  cudaStream_t s = ctx->stream;
  LL_TRY(extract_prepare(ctx, raw, n, fmt, where, stamp));
  const int ncap = (int)n;
  // the front end runs on its own scratch arena (swapped in under the usual name for the duration of this function)
  struct ScratchSwap { ll_ctx* c; ScratchSwap(ll_ctx* c_) : c(c_) { DevBuf t = c->scratch; c->scratch = c->scratch_fe; c->scratch_fe = t; }
                       ~ScratchSwap() { DevBuf t = c->scratch; c->scratch = c->scratch_fe; c->scratch_fe = t; } } swap_guard(ctx);
  ll_ctx::FrontGraph& g = ctx->fg;
  void* bufs[6] = {ctx->extract_buf.p, ctx->reg_buf.p, ctx->scratch.p, ctx->scratch2.p, (void*)(size_t)ctx->scratch.cap, ctx->scratch3.p};
  const bool same = g.n == n && memcmp(&g.pc, pc, sizeof(*pc)) == 0 && memcmp(g.bufs, bufs, sizeof(bufs)) == 0;
  if (same && g.exec) {
    LL_CUDA(ctx, cudaGraphLaunch(g.exec, s));
    ctx->launches += g.launches;
  } else if (same && g.warm && n >= 5) {
    // second call with this shape: every arena has its final size, so nothing allocates while the stream is being captured
    if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    const uint64_t l0 = ctx->launches;
    cudaGraph_t graph = nullptr;
    LL_CUDA(ctx, cudaStreamBeginCapture(s, cudaStreamCaptureModeRelaxed));
    const int st = front_end_enqueue(ctx, pc, A, ncap);
    const cudaError_t ce = cudaStreamEndCapture(s, &graph);
    void* after[6] = {ctx->extract_buf.p, ctx->reg_buf.p, ctx->scratch.p, ctx->scratch2.p, (void*)(size_t)ctx->scratch.cap, ctx->scratch3.p};
    if (st != LL_OK || ce != cudaSuccess || memcmp(after, bufs, sizeof(bufs)) != 0) {   // should not happen: fall back to eager launches
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError(); g.warm = false; g.n = 0;
      LL_TRY(front_end_enqueue(ctx, pc, A, ncap));
    } else {
      g.launches = ctx->launches - l0;
      LL_CUDA(ctx, cudaGraphInstantiate(&g.exec, graph, 0));
      cudaGraphDestroy(graph);
      LL_CUDA(ctx, cudaGraphLaunch(g.exec, s));
    }
  } else {
    if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
    LL_TRY(front_end_enqueue(ctx, pc, A, ncap));
    void* after[6] = {ctx->extract_buf.p, ctx->reg_buf.p, ctx->scratch.p, ctx->scratch2.p, (void*)(size_t)ctx->scratch.cap, ctx->scratch3.p};
    g.n = n; g.pc = *pc; memcpy(g.bufs, after, sizeof(after)); g.warm = true;
  }
  LL_CUDA(ctx, cudaStreamSynchronize(s));
  int* h = (int*)ctx->pinned + 8192;
  const int nc = h[5], ns = h[7], meta_scans = h[13];
  { int lo = h[10], hi = h[11]; lo = lo >= 0 ? lo : lo ^ 0x7fffffff; hi = hi >= 0 ? hi : hi ^ 0x7fffffff; memcpy(&ctx->last_full_min_t, &lo, 4); memcpy(&ctx->last_full_max_t, &hi, 4); }
  *nc_out = nc; *ns_out = ns;
  *dropped = (meta_scans <= 5 && !pc->whole_frame) ? 1 : 0;
  if (*dropped) return LL_OK;
  if (nc + ns > ctx->cfg.max_features) { ctx->set_error("more features than max_features"); return LL_ERR_CAPACITY; }
  LL_CUDA(ctx, cudaMemcpyAsync(A.feat, A.tmp_a, (size_t)nc * 16, cudaMemcpyDeviceToDevice, s));
  LL_CUDA(ctx, cudaMemcpyAsync(A.feat + nc, A.tmp_b, (size_t)ns * 16, cudaMemcpyDeviceToDevice, s));
  return LL_OK;
}

extern "C" int ll_scan_to_pose(ll_ctx* ctx, const ll_map* map, const void* raw, size_t n, int fmt, int where, double stamp, const ll_pipeline_cfg* pc, const ll_reg_state* in,
                    ll_reg_result* out, int* n_corner_used, int* n_surf_used) {
  if (!ctx || !map || !pc || !in || !out) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  RegArrays A; LL_TRY(reg_arrays(ctx, 0, &A));
  int nc = 0, ns = 0, dropped = 0;
  LL_TRY(scan_front_end(ctx, raw, n, fmt, where, stamp, pc, A, &nc, &ns, &dropped));
  if (n_corner_used) *n_corner_used = nc; if (n_surf_used) *n_surf_used = ns;
  if (dropped) { memset(out, 0, sizeof(*out)); out->status = 1; ctx->set_error("frame dropped: <= 5 petals"); return LL_OK; }
  return register_device(ctx, map, A, nc, ns, in, out);
}

// Multi-head frame (Mid-100: three Mid-40 heads, launch/rosbag_mid100.launch): Laser_feature::laserCloudHandler runs ONE Livox_laser object over
// the heads in turn and sums their per-piece feature clouds before the VoxelGrids (laser_feature_extractor.hpp:303-380); the mapping node then sees
// one merged feature pair (laser_mapping.hpp:1367-1405).  Heads whose frame has <= 5 petals contribute nothing (:287).
extern "C" int ll_frame_to_pose(ll_ctx* ctx, const ll_map* map, int n_heads, const void* const* raws, const size_t* ns, int fmt, int where, const double* stamps,
                     const ll_pipeline_cfg* pc, const ll_reg_state* in, ll_reg_result* out, int* n_corner_used, int* n_surf_used) {
  if (!ctx || !map || !pc || !in || !out || !raws || !ns || !stamps || n_heads < 1 || n_heads > 8) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  cudaStream_t s = ctx->stream;
  size_t total = 0; for (int h = 0; h < n_heads; h++) total += ns[h];
  if ((int)total > ctx->cfg.max_scan_points) { ctx->set_error("frame (all heads) larger than max_scan_points"); return LL_ERR_CAPACITY; }
  RegArrays A; LL_TRY(reg_arrays(ctx, 0, &A));
  int acc_c = 0, acc_s = 0;
  int* hc = (int*)ctx->pinned + 8192;
  for (int h = 0; h < n_heads; h++) {
    LL_TRY(extract_prepare(ctx, raws[h], ns[h], fmt, where, stamps[h]));
    LL_TRY(extract_enqueue(ctx));
    const float* d_bounds = nullptr;
    if (!pc->whole_frame) { LL_TRY(launch_piece_bounds(ctx, pc->pieces, A.bounds)); d_bounds = A.bounds + 2 * pc->use_piece; }
    LL_TRY(launch_get_features(ctx, d_bounds, 0.f, 1.f, A.tmp_a + acc_c, A.tmp_b + acc_s, nullptr, A.counts));
    LL_CUDA(ctx, cudaMemcpyAsync(hc, A.counts, 3 * sizeof(int), cudaMemcpyDeviceToHost, s));
    LL_CUDA(ctx, cudaMemcpyAsync(hc + 4, ctx->ex.d_meta, 12, cudaMemcpyDeviceToHost, s));
    LL_CUDA(ctx, cudaStreamSynchronize(s));
    if (ns[h] >= 5 && (hc[5] > 5 || pc->whole_frame)) { acc_c += hc[0]; acc_s += hc[1]; }   // hc[5] = meta[1] = laserCloudScans.size()
  }
  int* cnt = A.counts;   // [4..7] VoxelGrid outputs
  LL_TRY(launch_voxel_grid(ctx, A.tmp_a, acc_c, nullptr, pc->extractor_leaf_corner, A.tmp_d, cnt + 4));
  LL_TRY(launch_voxel_grid(ctx, A.tmp_d, acc_c > 0 ? acc_c : 0, cnt + 4, pc->mapping_leaf_corner, A.tmp_a, cnt + 5));
  LL_TRY(launch_voxel_grid(ctx, A.tmp_b, acc_s, nullptr, pc->extractor_leaf_surf, A.tmp_c, cnt + 6));
  LL_TRY(launch_voxel_grid(ctx, A.tmp_c, acc_s > 0 ? acc_s : 0, cnt + 6, pc->mapping_leaf_surf, A.tmp_b, cnt + 7));
  LL_CUDA(ctx, cudaMemcpyAsync(hc, cnt, 8 * sizeof(int), cudaMemcpyDeviceToHost, s));
  LL_CUDA(ctx, cudaStreamSynchronize(s));
  const int nc = hc[5], nsf = hc[7];
  if (n_corner_used) *n_corner_used = nc; if (n_surf_used) *n_surf_used = nsf;
  if (nc + nsf > ctx->cfg.max_features) { ctx->set_error("more features than max_features"); return LL_ERR_CAPACITY; }
  LL_CUDA(ctx, cudaMemcpyAsync(A.feat, A.tmp_a, (size_t)nc * 16, cudaMemcpyDeviceToDevice, s));
  LL_CUDA(ctx, cudaMemcpyAsync(A.feat + nc, A.tmp_b, (size_t)nsf * 16, cudaMemcpyDeviceToDevice, s));
  return register_device(ctx, map, A, nc, nsf, in, out);
}

extern "C" {

// ---------------------------------------------------------------------------------------------- multi-GPU
int ll_comm_local_handle(ll_ctx* ctx, unsigned char handle[LL_IPC_HANDLE_BYTES]) {
  if (!ctx) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  const size_t comm_bytes = LL_COMM_X_OFF + (size_t)ctx->cfg.max_features * sizeof(double);
  if (!ctx->comm_local) { LL_CUDA(ctx, cudaMalloc(&ctx->comm_local, comm_bytes)); LL_CUDA(ctx, cudaMemset(ctx->comm_local, 0, comm_bytes)); }
  cudaIpcMemHandle_t h; LL_CUDA(ctx, cudaIpcGetMemHandle(&h, ctx->comm_local));
  static_assert(sizeof(cudaIpcMemHandle_t) <= LL_IPC_HANDLE_BYTES, "ipc handle size");
  memset(handle, 0, LL_IPC_HANDLE_BYTES); memcpy(handle, &h, sizeof(h));
  return LL_OK;
}
int ll_comm_connect(ll_ctx* ctx, int rank, int world, const unsigned char* all) {
  if (!ctx || world < 1 || world > 8 || rank < 0 || rank >= world) return LL_ERR_INVALID;
  cudaSetDevice(ctx->device);
  if (!ctx->comm_local) { ctx->set_error("call ll_comm_local_handle first"); return LL_ERR_INVALID; }
  ctx->rank = rank; ctx->world = world;
  for (int p = 0; p < world; p++) {
    if (p == rank) { ctx->comm_peers[p] = ctx->comm_local; continue; }
    cudaIpcMemHandle_t h; memcpy(&h, all + (size_t)p * LL_IPC_HANDLE_BYTES, sizeof(h));
    LL_CUDA(ctx, cudaIpcOpenMemHandle(&ctx->comm_peers[p], h, cudaIpcMemLazyEnablePeerAccess));
  }
  return LL_OK;
}
}  // extern "C"
