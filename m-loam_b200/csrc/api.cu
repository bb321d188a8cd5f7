// api.cu — the C ABI declared in include/mloam_b200.h: context, host<->device staging, and the
// orchestrators (scan2MapOptimization, the per-sweep frame) expressed as kernel sequences on one stream.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "ctx.h"
#include "host_util.h"

using namespace mloam;

namespace mloam {

ProfScope::ProfScope(Ctx *ctx, const char *nm) : c(ctx), name(nm) {
  if (!c->prof_on) return;
  auto get = [&]() {
    cudaEvent_t e;
    if (!c->evt_pool.empty()) {
      e = c->evt_pool.back();
      c->evt_pool.pop_back();
    } else {
      cudaEventCreate(&e);
    }
    return e;
  };
  a = get();
  b = get();
  cudaEventRecord(a, c->stream);
}
ProfScope::~ProfScope() {
  if (!a) return;
  cudaEventRecord(b, c->stream);
  c->pending.push_back(Ctx::PendingEvt{name, a, b});
}
void prof_collect(Ctx *c) {
  for (auto &p : c->pending) {
    float ms = 0.f;
    if (cudaEventSynchronize(p.b) == cudaSuccess && cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
      ProfSlot &s = c->prof[p.name];
      s.ms += ms;
      s.launches += 1;
    }
    c->evt_pool.push_back(p.a);
    c->evt_pool.push_back(p.b);
  }
  c->pending.clear();
}

}  // namespace mloam

extern "C" {

const char *mloam_version(void) { return "mloam_b200 0.1 (sm_100a)"; }

void mloam_default_params(mloam_params_t *p) {
  memset(p, 0, sizeof(*p));
  p->n_scans = 64;
  p->distance_sq_threshold = 25.0f;  // config_realvehicle_hercules.yaml:103
  p->nearby_scan = 2.5f;             // :104
  p->min_match_sq_dis = 1.0f;        // :110
  p->min_plane_dis = 0.2f;           // :111
  p->n_neigh = 5;
  p->check_fov = 0;
  p->point_plane_factor = 1;
  p->point_edge_factor = 1;
  p->huber_a = 0.1;
  p->eig_thre = 100.0;               // MAP_EIG_THRE :140
  p->cov_trace = 0.0075;             // 3 * 0.0025 (:160-168)
  p->max_outer = 2;
  p->max_inner = 30;
  p->map_cell = 0.0f;
  p->corner_leaf = 0.2f;             // MAP_CORNER_RES :136
  p->surf_leaf = 0.4f;               // MAP_SURF_RES :137
  p->gf_method = 0, p->gf_ratio = 1.0f, p->gf_seed = 0;  // wo_gf
}

int mloam_ctx_create(int device, const mloam_params_t *params, mloam_ctx_t **out) {
  if (!out) return MLOAM_E_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) return MLOAM_E_NO_DEVICE;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MLOAM_E_NO_DEVICE;
  if (prop.major != 10) {
    fprintf(stderr, "mloam_b200: device %d is sm_%d%d; this library carries sm_100a code only\n", device, prop.major,
            prop.minor);
    return MLOAM_E_NO_DEVICE;
  }
  if (cudaSetDevice(device) != cudaSuccess) return MLOAM_E_NO_DEVICE;
  mloam_ctx *h = new (std::nothrow) mloam_ctx();
  if (!h) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if (params) c->params = *params;
  else mloam_default_params(&c->params);
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_maps, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream3, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_fork3, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join3, cudaEventDisableTiming) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream4, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&c->stream5, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_fork4, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join4, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_fork5, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join5, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_next, cudaEventDisableTiming) != cudaSuccess ||
      cudaMallocHost(&c->pinned, kPinnedBytes) != cudaSuccess || c->lm_state.reserve(sizeof(LMState) + 64) != cudaSuccess ||
      c->scratch[7].reserve(4096) != cudaSuccess) {
    delete h;
    return MLOAM_E_CUDA;
  }
  c->pinned_cap = kPinnedBytes;
  memset(c->pinned, 0, kPinnedBytes);
  cudaMemset(c->scratch[7].p, 0, 4096);
  if (const char *e = getenv("MLOAM_DISABLE_GRAPHS")) c->use_graphs = (e[0] == '0' || e[0] == '\0') ? 1 : 0;
  if (const char *e = getenv("MLOAM_KNN_TRACE")) c->knn_trace_on = e[0] == '1';
  if (const char *e = getenv("MLOAM_KNN_MB")) {
    const int v = atoi(e);
    if (v >= 2 && v <= 4) c->knn_min_blocks = v;
  }
  if (const char *e = getenv("MLOAM_KNN_TMA_MIN")) c->knn_tma_min = (unsigned)strtoul(e, nullptr, 10);
  if (const char *e = getenv("MLOAM_LOOKAHEAD")) c->use_lookahead = (e[0] == '0') ? 0 : 1;
  if (const char *e = getenv("MLOAM_STAMP")) c->stamp_on = e[0] == '1';
  if (const char *e = getenv("MLOAM_FUSE_ITER")) c->fuse_iter = (e[0] == '0') ? 0 : 1;
  if (const char *e = getenv("MLOAM_DISABLE_SEEDS")) c->use_seeds = (e[0] == '0' || e[0] == '\0') ? 1 : 0;
  *out = h;
  return MLOAM_OK;
}

void mloam_ctx_destroy(mloam_ctx_t *h) {
  if (!h) return;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  mloam_comm_destroy(h);
  for (auto &g : c->graphs)
    if (g.exec) cudaGraphExecDestroy(g.exec);
  c->graphs.clear();
  prof_collect(c);
  for (auto e : c->evt_pool) cudaEventDestroy(e);
  for (auto &m : c->maps) {
    m.sorted.release(), m.orig.release(), m.cells.release(), m.rank_of.release(), m.tile_sums.release(), m.hdr.release();
  }
  for (int i = 0; i < 4; i++) c->scan_pts[i].release(), c->feat_valid[i].release(), c->feat_coeff[i].release(), c->feat_nn[i].release(), c->knn_pos[i].release(), c->knn_changed[i].release(), c->knn_anchor[i].release(), c->knn_heavy[i].release();
  for (int i = 0; i < 2; i++) c->gf_work[i].release();
  c->knn_heavy_list.release(), c->knn_trace.release();
  c->partials.release(), c->lm_state.release();
  for (auto &s : c->scratch) s.release();
  c->frame_main.release(), c->frame_alt.release(), c->next_in.release(), c->stamps.release();
  if (c->pinned) cudaFreeHost(c->pinned);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  if (c->stream2) cudaStreamSynchronize(c->stream2), cudaStreamDestroy(c->stream2);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->ev_maps) cudaEventDestroy(c->ev_maps);
  if (c->stream3) cudaStreamSynchronize(c->stream3), cudaStreamDestroy(c->stream3);
  if (c->ev_fork3) cudaEventDestroy(c->ev_fork3);
  if (c->ev_join3) cudaEventDestroy(c->ev_join3);
  if (c->stream4) cudaStreamSynchronize(c->stream4), cudaStreamDestroy(c->stream4);
  if (c->stream5) cudaStreamSynchronize(c->stream5), cudaStreamDestroy(c->stream5);
  for (cudaEvent_t ev : {c->ev_fork4, c->ev_join4, c->ev_fork5, c->ev_join5, c->ev_next})
    if (ev) cudaEventDestroy(ev);
  delete h;
}

int mloam_set_params(mloam_ctx_t *h, const mloam_params_t *p) {
  if (!h || !p) return MLOAM_E_INVALID;
  if (p->n_neigh != 5 && p->n_neigh != 10) return fail(&h->c, MLOAM_E_INVALID, "n_neigh must be 5 or 10");
  h->c.params = *p;
  h->c.prefetched.valid = false;  // look-ahead features were extracted under the previous parameters
  return MLOAM_OK;
}

int mloam_set_stream(mloam_ctx_t *h, void *s) {
  if (!h) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaStreamSynchronize(c->stream);
  if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
  c->stream = (cudaStream_t)s;
  c->own_stream = false;
  return MLOAM_OK;
}

int mloam_sync(mloam_ctx_t *h) {
  if (!h) return MLOAM_E_INVALID;
  MLOAM_CUDA_OK(&h->c, cudaStreamSynchronize(h->c.stream));
  return MLOAM_OK;
}
const char *mloam_last_error(mloam_ctx_t *h) { return h ? h->c.err.c_str() : "null context"; }
long long mloam_launch_count(mloam_ctx_t *h) { return h ? h->c.launches : 0; }

int mloam_profile_enable(mloam_ctx_t *h, int on) {
  if (!h) return MLOAM_E_INVALID;
  h->c.prof_on = on != 0;
  return MLOAM_OK;
}
int mloam_profile_get(mloam_ctx_t *h, const char *name, double *ms_total, long long *launches) {
  if (!h || !name) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaStreamSynchronize(c->stream);
  prof_collect(c);
  if (!strcmp(name, "graph_capture_failures")) {  // frames that ran on the stream path because their graph capture failed
    if (ms_total) *ms_total = 0.0;
    if (launches) *launches = c->graph_capture_failures;
    return MLOAM_OK;
  }
  // query counts / SM cycles of the matcher's search paths (k_match_knn), reported through `launches`
  if (!strncmp(name, "knn_slow_rec", 12) && name[12] >= '0' && name[12] <= '9') {
    long long v = 0;
    MLOAM_CUDA_OK(c, cudaMemcpy(&v, c->scratch[7].as<char>() + kKnnPathStatsOffset + 160 + 8 * (size_t)(name[12] - '0'), 8, cudaMemcpyDeviceToHost));
    if (ms_total) *ms_total = 0.0;
    if (launches) *launches = v;
    return MLOAM_OK;
  }
  static const char *kBlind[8] = {"knn_blind_cycles_coarse", "knn_blind_cycles_ring1", "knn_blind_cycles_finish", "knn_blind_ring1_points",
                                  "knn_blind_finish_points", "knn_blind_finish_blocks", "knn_blind_finish_cells", "knn_blind_finish_queries"};
  for (int k = 0; k < 8; k++)
    if (!strcmp(name, kBlind[k])) {
      unsigned long long v = 0;
      MLOAM_CUDA_OK(c, cudaMemcpy(&v, c->scratch[7].as<char>() + kKnnPathStatsOffset + 96 + 8 * (size_t)k, 8, cudaMemcpyDeviceToHost));
      if (ms_total) *ms_total = 0.0;
      if (launches) *launches = (long long)v;
      return MLOAM_OK;
    }
  static const char *kPaths[12] = {"knn_keep_matched", "knn_keep_rejected", "knn_ball", "knn_blind", "knn_max_query_cycles",
                                   "knn_queries_over_32k_cycles", "knn_queries_over_64k_cycles", "knn_cycles_keep_matched",
                                   "knn_cycles_keep_rejected", "knn_cycles_ball", "knn_cycles_blind", "knn_slowest_query"};
  for (int k = 0; k < 12; k++)
    if (!strcmp(name, kPaths[k])) {
      unsigned long long v = 0;
      const size_t off = kKnnPathStatsOffset + (k < 7 ? 4 * (size_t)k : 32 + 8 * (size_t)(k - 7));
      MLOAM_CUDA_OK(c, cudaMemcpy(&v, c->scratch[7].as<char>() + off, k < 7 ? 4 : 8, cudaMemcpyDeviceToHost));
      if (ms_total) *ms_total = 0.0;
      if (launches) *launches = (long long)v;
      return MLOAM_OK;
    }
  auto it = c->prof.find(name);
  if (ms_total) *ms_total = it == c->prof.end() ? 0.0 : it->second.ms;
  if (launches) *launches = it == c->prof.end() ? 0 : it->second.launches;
  return MLOAM_OK;
}
int mloam_profile_reset(mloam_ctx_t *h) {
  if (!h) return MLOAM_E_INVALID;
  cudaStreamSynchronize(h->c.stream);
  prof_collect(&h->c);
  cudaMemset(h->c.scratch[7].as<char>() + kKnnPathStatsOffset, 0, 256);
  h->c.prof.clear();
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ maps / kNN
int mloam_map_build_device(mloam_ctx_t *h, int slot, const mloam_point_t *d_pts, int m, float cell) {
  if (!h) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  return map_build_device(c, slot, reinterpret_cast<const float4 *>(d_pts), m, pick_cell(c, cell));
}

int mloam_map_build(mloam_ctx_t *h, int slot, const mloam_point_t *h_pts, int m, float cell) {
  if (!h || (!h_pts && m > 0) || m < 0) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  DevBuf &stage = c->scratch[0];
  MLOAM_CUDA_OK(c, stage.reserve(sizeof(float4) * (size_t)(m + 1)));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(stage.p, h_pts, sizeof(float4) * (size_t)m, cudaMemcpyHostToDevice, c->stream));
  return map_build_device(c, slot, stage.as<float4>(), m, pick_cell(c, cell));
}

__global__ void k_stamp(unsigned long long *slot) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  *slot = t;
}
}  // extern "C" (reopened below)
namespace mloam {
void stamp(Ctx *c, const char *label) {
  if (!c->stamp_on || c->stamp_mute || c->stamp_n >= 256) return;
  if (c->stamps.reserve(256 * sizeof(unsigned long long)) != cudaSuccess) return;
  if ((int)c->stamp_labels.size() <= c->stamp_n) c->stamp_labels.resize(c->stamp_n + 1);
  c->stamp_labels[c->stamp_n] = label;
  k_stamp<<<1, 1, 0, c->stream>>>(c->stamps.as<unsigned long long>() + c->stamp_n);
  c->stamp_n++;
}
}  // namespace mloam
extern "C" {
// Diagnosis only: the globaltimer stamps [ns] of the last frame (MLOAM_STAMP=1) and their labels.
int mloam_debug_stamps(mloam_ctx_t *h, unsigned long long *out_ns, int cap, int *n) {
  if (!h || !out_ns || !n) return MLOAM_E_INVALID;
  cudaSetDevice(h->c.device);
  *n = h->c.stamp_n < cap ? h->c.stamp_n : cap;
  if (*n <= 0) return MLOAM_OK;
  if (cudaStreamSynchronize(h->c.stream) != cudaSuccess) return MLOAM_E_CUDA;
  return cudaMemcpy(out_ns, h->c.stamps.p, sizeof(unsigned long long) * (size_t)*n, cudaMemcpyDeviceToHost) == cudaSuccess ? MLOAM_OK : MLOAM_E_CUDA;
}
const char *mloam_debug_stamp_label(mloam_ctx_t *h, int i) {
  if (!h || i < 0 || i >= (int)h->c.stamp_labels.size()) return "";
  return h->c.stamp_labels[i].c_str();
}

// Diagnosis only (not part of include/mloam_b200.h): per-query words of the last traced k_match_knn launch.
int mloam_debug_knn_trace(mloam_ctx_t *h, unsigned *out, int n_queries) {
  if (!h || !out || n_queries <= 0 || h->c.knn_trace.cap < 16 * (size_t)n_queries) return MLOAM_E_INVALID;  // n_queries may include the timeline tail
  cudaSetDevice(h->c.device);
  if (cudaStreamSynchronize(h->c.stream) != cudaSuccess) return MLOAM_E_CUDA;
  return cudaMemcpy(out, h->c.knn_trace.p, 16 * (size_t)n_queries, cudaMemcpyDeviceToHost) == cudaSuccess ? MLOAM_OK : MLOAM_E_CUDA;
}

int mloam_map_size(mloam_ctx_t *h, int slot) {
  if (!h || slot < 0 || slot >= MLOAM_NUM_MAPS || !h->c.maps[slot].built) return -1;
  return h->c.maps[slot].m;
}

int mloam_knn(mloam_ctx_t *h, int slot, const mloam_point_t *h_q, int nq, const double *pose7, int k, float max_sqdist,
              int *h_idx, float *h_sqdist) {
  if (!h || nq < 0 || (nq > 0 && (!h_q || !h_idx || !h_sqdist))) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  if (nq == 0) return MLOAM_OK;
  MLOAM_CUDA_OK(c, c->scratch[1].reserve(sizeof(float4) * (size_t)nq));
  MLOAM_CUDA_OK(c, c->scratch[2].reserve(sizeof(int) * (size_t)nq * k));
  MLOAM_CUDA_OK(c, c->scratch[3].reserve(sizeof(float) * (size_t)nq * k));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scratch[1].p, h_q, sizeof(float4) * (size_t)nq, cudaMemcpyHostToDevice, c->stream));
  double *d_pose = nullptr;
  if (pose7) {
    int rc = upload_pose(c, pose7, &d_pose);
    if (rc) return rc;
  }
  int rc = knn_device(c, slot, c->scratch[1].as<float4>(), nq, d_pose, k, max_sqdist, c->scratch[2].as<int>(),
                      c->scratch[3].as<float>());
  if (rc) return rc;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_idx, c->scratch[2].p, sizeof(int) * (size_t)nq * k, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_sqdist, c->scratch[3].p, sizeof(float) * (size_t)nq * k, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ matching
int mloam_match_from_map(mloam_ctx_t *h, int slot, int type, const mloam_point_t *h_pts, int n, const double *pose7,
                         unsigned char *h_valid, double *h_coeffs, int *h_nn) {
  if (!h || n < 0 || !pose7 || (n > 0 && (!h_pts || !h_valid || !h_coeffs))) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  if (n == 0) return MLOAM_OK;
  const int t = type == 's' ? 1 : 0;
  const int K = c->params.n_neigh;
  MLOAM_CUDA_OK(c, c->scan_pts[t].reserve(sizeof(float4) * (size_t)n));
  int rc = reserve_feat(c, t, n);
  if (rc) return rc;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[t].p, h_pts, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  double *d_pose;
  rc = upload_pose(c, pose7, &d_pose);
  if (rc) return rc;
  rc = match_from_map_device(c, slot, type, c->scan_pts[t].as<float4>(), n, nullptr, d_pose, match_cfg(c),
                             c->feat_valid[t].as<unsigned char>(), c->feat_coeff[t].as<float>(), c->feat_nn[t].as<int>());
  if (rc) return rc;
  std::vector<float> cf((size_t)n * 6);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_valid, c->feat_valid[t].p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(cf.data(), c->feat_coeff[t].p, sizeof(float) * 6 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  if (h_nn)
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_nn, c->feat_nn[t].p, sizeof(int) * (size_t)K * n, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (size_t i = 0; i < (size_t)n * 6; i++) h_coeffs[i] = (double)cf[i];
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ factors
int mloam_factor_evaluate(mloam_ctx_t *h, int kind, int n, const double *h_points, const double *h_coeffs,
                          const double *h_sqrt_info, const double *h_params, double *h_residuals, double *h_jacobians) {
  if (!h || n < 0 || kind < 0 || kind > 4 || (n > 0 && (!h_points || !h_coeffs || !h_params || !h_residuals)))
    return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  if (n == 0) return MLOAM_OK;
  const int rows = kind == 2 ? 3 : 1;
  const int cols = kind >= 3 ? 21 : 7;
  const int np = kind >= 3 ? 21 : 7;
  DevBuf &dp = c->scratch[1], &dc = c->scratch[2], &ds = c->scratch[3], &dr = c->scratch[4], &dj = c->scratch[5], &dx = c->scratch[6];
  MLOAM_CUDA_OK(c, dp.reserve(sizeof(double) * 3 * (size_t)n));
  MLOAM_CUDA_OK(c, dc.reserve(sizeof(double) * 6 * (size_t)n));
  MLOAM_CUDA_OK(c, ds.reserve(sizeof(double) * (size_t)n));
  MLOAM_CUDA_OK(c, dr.reserve(sizeof(double) * rows * (size_t)n));
  MLOAM_CUDA_OK(c, dj.reserve(sizeof(double) * rows * cols * (size_t)n));
  MLOAM_CUDA_OK(c, dx.reserve(sizeof(double) * 32));
  cudaStream_t st = c->stream;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(dp.p, h_points, sizeof(double) * 3 * (size_t)n, cudaMemcpyHostToDevice, st));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(dc.p, h_coeffs, sizeof(double) * 6 * (size_t)n, cudaMemcpyHostToDevice, st));
  if (h_sqrt_info) MLOAM_CUDA_OK(c, cudaMemcpyAsync(ds.p, h_sqrt_info, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(dx.p, h_params, sizeof(double) * np, cudaMemcpyHostToDevice, st));
  int rc = factor_evaluate_device(c, kind, n, dp.as<double>(), dc.as<double>(), h_sqrt_info ? ds.as<double>() : nullptr,
                                  dx.as<double>(), dr.as<double>(), h_jacobians ? dj.as<double>() : nullptr);
  if (rc) return rc;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_residuals, dr.p, sizeof(double) * rows * (size_t)n, cudaMemcpyDeviceToHost, st));
  if (h_jacobians)
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_jacobians, dj.p, sizeof(double) * rows * cols * (size_t)n, cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  return MLOAM_OK;
}

int mloam_normal_equations(mloam_ctx_t *h, int n, const unsigned char *h_types, const double *h_points, const double *h_coeffs,
                           double sqrt_info, double huber_a, const double *pose7, double *H36, double *g6, double *cost) {
  if (!h || n < 0 || !pose7 || !H36 || !g6 || !cost || (n > 0 && (!h_types || !h_points || !h_coeffs))) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  // The reference's PointPlaneFeature carries float-valued point_/coeffs_ (feature_extract.hpp:771-781,872-875):
  // pack into the device feature format (float4 point, float[6] coefficients), one set per factor type.
  std::vector<float4> pts[2];
  std::vector<float> cf[2];
  for (int i = 0; i < n; i++) {
    const int t = h_types[i] == 's' ? 1 : 0;
    pts[t].push_back(make_float4((float)h_points[i * 3], (float)h_points[i * 3 + 1], (float)h_points[i * 3 + 2], 0.f));
    for (int k = 0; k < 6; k++) cf[t].push_back((float)h_coeffs[(size_t)i * 6 + k]);
  }
  FeatSet sets[2];
  for (int t = 0; t < 2; t++) {
    const int nt = (int)pts[t].size();
    MLOAM_CUDA_OK(c, c->scan_pts[t].reserve(sizeof(float4) * (size_t)(nt + 1)));
    int rc = reserve_feat(c, t, nt);
    if (rc) return rc;
    if (nt > 0) {
      MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[t].p, pts[t].data(), sizeof(float4) * nt, cudaMemcpyHostToDevice, c->stream));
      MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->feat_coeff[t].p, cf[t].data(), sizeof(float) * 6 * nt, cudaMemcpyHostToDevice, c->stream));
      MLOAM_CUDA_OK(c, cudaMemsetAsync(c->feat_valid[t].p, 1, nt, c->stream));
    }
    sets[t] = FeatSet{c->scan_pts[t].as<float4>(), c->feat_valid[t].as<unsigned char>(), c->feat_coeff[t].as<float>(), nt, t, nullptr};
  }
  double *d_pose;
  int rc = upload_pose(c, pose7, &d_pose);
  if (rc) return rc;
  MLOAM_CUDA_OK(c, c->scratch[6].reserve(sizeof(double) * 32));
  rc = linearize_device(c, sets, 2, SolveCfg{sqrt_info, huber_a, 0.0, false}, kEvalAtPose, d_pose, c->scratch[6].as<double>());
  if (rc) return rc;
  double *ne = reinterpret_cast<double *>(c->pinned) + 64;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(ne, c->scratch[6].p, sizeof(double) * 30, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  int q = 0;
  for (int i = 0; i < 6; i++)
    for (int j = i; j < 6; j++) H36[i * 6 + j] = H36[j * 6 + i] = ne[q++];
  for (int k = 0; k < 6; k++) g6[k] = ne[21 + k];
  *cost = ne[27];
  return MLOAM_OK;
}

__global__ void k_pose_plus(const double *x, const double *d, const double *V, double *out) {
  if (threadIdx.x == 0) mloam::pose_plus(x, d, V, out);
}
int mloam_pose_plus(mloam_ctx_t *h, const double *x7, const double *delta6, const double *V36, double *out7) {
  if (!h || !x7 || !delta6 || !out7) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  double *stage = reinterpret_cast<double *>(c->pinned) + 128;
  for (int k = 0; k < 7; k++) stage[k] = x7[k];
  for (int k = 0; k < 6; k++) stage[8 + k] = delta6[k];
  for (int k = 0; k < 36; k++) stage[16 + k] = V36 ? V36[k] : (k % 7 == 0 ? 1.0 : 0.0);
  MLOAM_CUDA_OK(c, c->scratch[6].reserve(sizeof(double) * 64));
  double *d = c->scratch[6].as<double>();
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d, stage, sizeof(double) * 52, cudaMemcpyHostToDevice, c->stream));
  k_pose_plus<<<1, 32, 0, c->stream>>>(d, d + 8, d + 16, d + 56);
  c->launches++;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(stage + 56, d + 56, sizeof(double) * 7, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 7; k++) out7[k] = stage[56 + k];
  return MLOAM_OK;
}

}  // extern "C"
