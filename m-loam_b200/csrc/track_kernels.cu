// track_kernels.cu — scan-to-scan association and LidarTracker::trackCloud.
//
//   k_match_scan<SURF>  FeatureExtract::matchCornerFromScan / matchSurfFromScan (feature_extract.hpp:131-376):
//                       one warp per feature: TransformToStart (s = 1), exact 1-NN in the voxel-hash of the
//                       previous sweep's features, then the reference's walk over the ARRAY ORDER of the previous
//                       cloud for the nearest point(s) on neighbouring rings (|ring diff| <= NEARBY_SCAN) — 32
//                       array slots per step, ballot for the first slot that ends the walk, warp-min on
//                       (distance, visiting order) so ties resolve exactly as the sequential `<` loop does.
//   track_cloud_device  lidar_tracker.cpp:23-129: 2 outer rounds x (match, Huber(0.1), <= 4 LM iterations),
//                       "less than 10 correspondences" skip, on the device-resident LM state of solve_kernels.cu.
#include "ctx.h"
#include "host_util.h"
#include "knn.cuh"

namespace mloam {

constexpr int TWARPS = 8;

__device__ __forceinline__ float sqr3(float a, float b, float c) { return a * a + b * b + c * c; }  // common::sqrSum

// Walk one direction.  best2/best3: running (d2 bits << 32 | visit order) keys; j2/j3 the matching array indices.
// SURF = false: only `best2` (other-ring candidate) is used (matchCornerFromScan).
template <bool SURF>
__device__ __forceinline__ void walk(const float4 *__restrict__ scan, int m, int closest, int ring, float nearby, float thr,
                                     float sx, float sy, float sz, int dir, int lane, unsigned &order, unsigned long long &best2,
                                     int &j2, unsigned long long &best3, int &j3) {
  for (int base = 1;; base += 32) {
    const int step = base + lane;
    const int j = closest + dir * step;
    const bool inb = dir > 0 ? (j < m) : (j >= 0);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (inb) v = __ldg(scan + j);
    const int rj = (int)v.w;
    // "if not in nearby scans, end the loop" (:171-172 / :191-192 / :307-308 / :330-331): int vs (int + float)
    const bool brk = !inb || (dir > 0 ? ((float)rj > (float)ring + nearby) : ((float)rj < (float)ring - nearby));
    const unsigned mb = __ballot_sync(MLOAM_FULL_MASK, brk);
    const unsigned live = mb ? ((1u << (__ffs(mb) - 1)) - 1u) : 0xffffffffu;  // slots before the first break
    const bool on = (live >> lane) & 1u;
    const float d = sqr3(v.x - sx, v.y - sy, v.z - sz);
    const unsigned long long key = ((unsigned long long)__float_as_uint(d) << 32) | (order + (unsigned)(step - 1));
    if (!SURF) {
      // corner: skip same-side rings (:168-169 `<= ring` going up, :188-189 `>= ring` going down)
      const bool cand = on && (dir > 0 ? (rj > ring) : (rj < ring)) && d < thr;
      const unsigned long long k = warp_min_u64(cand ? key : MLOAM_KEY_NONE);
      if (k < best2) {
        best2 = k;
        const unsigned owner = __ballot_sync(MLOAM_FULL_MASK, cand && key == k);
        j2 = __shfl_sync(MLOAM_FULL_MASK, j, __ffs(owner) - 1);
      }
    } else {
      // surf: same-or-near-side ring -> ind2, the other side -> ind3 (:313-323 / :336-346)
      const bool same = dir > 0 ? (rj <= ring) : (rj >= ring);
      const bool c2 = on && same && d < thr, c3 = on && !same && d < thr;
      const unsigned long long k2 = warp_min_u64(c2 ? key : MLOAM_KEY_NONE);
      if (k2 < best2) {
        best2 = k2;
        const unsigned owner = __ballot_sync(MLOAM_FULL_MASK, c2 && key == k2);
        j2 = __shfl_sync(MLOAM_FULL_MASK, j, __ffs(owner) - 1);
      }
      const unsigned long long k3 = warp_min_u64(c3 ? key : MLOAM_KEY_NONE);
      if (k3 < best3) {
        best3 = k3;
        const unsigned owner = __ballot_sync(MLOAM_FULL_MASK, c3 && key == k3);
        j3 = __shfl_sync(MLOAM_FULL_MASK, j, __ffs(owner) - 1);
      }
    }
    if (mb) {
      order += (unsigned)(base + (__ffs(mb) - 1) - 1);
      break;
    }
  }
}

template <bool SURF>
__global__ void __launch_bounds__(TWARPS * 32)
    k_match_scan(MapView map, const float4 *__restrict__ pts, int n, const double *__restrict__ pose7, float dist_sq_thr, float nearby,
                 unsigned char *__restrict__ valid, float *__restrict__ coeff, int *__restrict__ nn, unsigned tma_min) {
  __shared__ KnnSmem ksm[TWARPS];
  const int lane = threadIdx.x & 31;
  KnnSmem &ks = ksm[threadIdx.x >> 5];
  knn_smem_init(ks, lane, tma_min);
  const GridP g = load_grid(map);
  PoseD T = pose_from_param(pose7);
  T.q = qnormalized(T.q);  // Pose(q, t) normalises (pose.cpp:34-41; lidar_tracker.cpp:54-55)
  for (int i = blockIdx.x * TWARPS + (threadIdx.x >> 5); i < n; i += gridDim.x * TWARPS) {
    const float4 p = __ldg(pts + i);
    const float3 sel = associate(T, p.x, p.y, p.z);  // TransformToStart, b_distortion = false (utility.h:55-77)
    Best best;
    warp_knn<1, true>(map, g, ks, sel.x, sel.y, sel.z, dist_sq_thr, lane, best);
    const unsigned long long k0 = best_key(best, 0);
    bool ok = k0 != MLOAM_KEY_NONE && key_d2(k0) < dist_sq_thr;  // :158 / :296
    float out[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    int closest = -1, j2 = -1, j3 = -1;
    if (ok) {
      closest = (int)(unsigned)(k0 & 0xffffffffu);
      const float4 c = __ldg(map.orig + closest);
      const int ring = (int)c.w;
      // running minima start at DISTANCE_SQ_THRESHOLD (:163 / :301): candidates must be strictly below it
      unsigned long long best2 = MLOAM_KEY_NONE, best3 = MLOAM_KEY_NONE;
      unsigned order = 0;
      walk<SURF>(map.orig, map.m, closest, ring, nearby, dist_sq_thr, sel.x, sel.y, sel.z, +1, lane, order, best2, j2, best3, j3);
      walk<SURF>(map.orig, map.m, closest, ring, nearby, dist_sq_thr, sel.x, sel.y, sel.z, -1, lane, order, best2, j2, best3, j3);
      if (!SURF) {
        ok = j2 >= 0;
        if (ok) {
          const float4 b = __ldg(map.orig + j2);
          out[0] = c.x, out[1] = c.y, out[2] = c.z, out[3] = b.x, out[4] = b.y, out[5] = b.z;  // :255-261
        }
      } else {
        ok = j2 >= 0 && j3 >= 0;
        if (ok) {  // :351-366, Vector3f arithmetic
          const float4 l = __ldg(map.orig + j2), mm = __ldg(map.orig + j3);
          const float ax = c.x - l.x, ay = c.y - l.y, az = c.z - l.z;
          const float bx = c.x - mm.x, by = c.y - mm.y, bz = c.z - mm.z;
          float wx = ay * bz - az * by, wy = az * bx - ax * bz, wz = ax * by - ay * bx;
          const float nrm = sqrtf(wx * wx + wy * wy + wz * wz);
          wx = wx / nrm, wy = wy / nrm, wz = wz / nrm;
          out[0] = wx, out[1] = wy, out[2] = wz, out[3] = -(wx * c.x + wy * c.y + wz * c.z);
        }
      }
    }
    if (lane == 0) {
      valid[i] = ok ? 1 : 0;
#pragma unroll
      for (int k = 0; k < 6; k++) coeff[(size_t)i * 6 + k] = ok ? out[k] : 0.f;
      if (nn) nn[(size_t)i * 3 + 0] = ok ? closest : -1, nn[(size_t)i * 3 + 1] = ok ? j2 : -1, nn[(size_t)i * 3 + 2] = ok ? j3 : -1;
    }
  }
}

int match_from_scan_device(Ctx *c, int slot, int type, const float4 *d_pts, int n, const double *d_pose7, unsigned char *d_valid,
                           float *d_coeff, int *d_nn3) {
  if (slot < 0 || slot >= MLOAM_NUM_MAPS || !c->maps[slot].built) {
    c->err = "match_from_scan: map slot not built";
    return MLOAM_E_STATE;
  }
  if (n <= 0) return MLOAM_OK;
  ProfScope ps(c, "match_scan");
  MapView mv = c->maps[slot].view();
  int nb = (n + TWARPS - 1) / TWARPS;
  if (nb > 8 * c->sm_count) nb = 8 * c->sm_count;
  const float thr = c->params.distance_sq_threshold, nearby = c->params.nearby_scan;
  if (type == 's') k_match_scan<true><<<nb, TWARPS * 32, 0, c->stream>>>(mv, d_pts, n, d_pose7, thr, nearby, d_valid, d_coeff, d_nn3, c->knn_tma_min);
  else k_match_scan<false><<<nb, TWARPS * 32, 0, c->stream>>>(mv, d_pts, n, d_pose7, thr, nearby, d_valid, d_coeff, d_nn3, c->knn_tma_min);
  c->launches++;
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

// LidarTracker::trackCloud, lidar_tracker.cpp:23-129.  All four clouds are device pointers.
int track_cloud_device(Ctx *c, const float4 *d_prev_less_sharp, int n_pls, const float4 *d_prev_less_flat, int n_plf,
                       const float4 *d_cur_sharp, int n_cs, const float4 *d_cur_flat, int n_cf, const double *pose_ini7,
                       double *pose_out7, mloam_solve_stats_t *stats) {
  if (stats) memset(stats, 0, sizeof(*stats));
  // :27-34 kd-trees over the previous sweep's less-sharp / less-flat features.  Cell 1.3 m: the nearest neighbour of a tracked
  // feature is almost always inside the 27-cell neighbourhood; the shells of knn.cuh cover the rest of the 5 m ball.
  const float cell = fmaxf(0.26f, sqrtf(c->params.distance_sq_threshold) * 0.26f);
  int rc = map_build_device(c, MLOAM_MAP_SCAN_CORNER, d_prev_less_sharp, n_pls, cell);
  if (rc) return rc;
  rc = map_build_device(c, MLOAM_MAP_SCAN_SURF, d_prev_less_flat, n_plf, cell);
  if (rc) return rc;
  rc = reserve_feat(c, 0, n_cs);
  if (rc) return rc;
  rc = reserve_feat(c, 1, n_cf);
  if (rc) return rc;
  const int max_outer = 2, max_inner = 4;  // :44, :114
  // Huber 0.1 (:47); evalDegenracy is commented out in trackCloud (:101-108)
  const SolveCfg cfg{1.0, 0.1, 0.0, false};
  rc = lm_init_state(c, pose_ini7, max_inner, 10);  // :64-68
  if (rc) return rc;
  LMState *st = c->lm_state.as<LMState>();
  int *h_done = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 2048);
  FeatSet sets[2] = {FeatSet{d_cur_sharp, c->feat_valid[0].as<unsigned char>(), c->feat_coeff[0].as<float>(), n_cs, 2, nullptr},
                     FeatSet{d_cur_flat, c->feat_valid[1].as<unsigned char>(), c->feat_coeff[1].as<float>(), n_cf, 1, nullptr}};
  for (int outer = 0; outer < max_outer && rc == MLOAM_OK; outer++) {
    rc = match_from_scan_device(c, MLOAM_MAP_SCAN_CORNER, 'c', d_cur_sharp, n_cs, st->x, c->feat_valid[0].as<unsigned char>(),
                                c->feat_coeff[0].as<float>(), nullptr);
    if (rc) break;
    rc = match_from_scan_device(c, MLOAM_MAP_SCAN_SURF, 's', d_cur_flat, n_cf, st->x, c->feat_valid[1].as<unsigned char>(),
                                c->feat_coeff[1].as<float>(), nullptr);
    if (rc) break;
    rc = linearize_device(c, sets, 2, cfg, kEvalBegin);
    if (rc) break;
    for (int it = 0; it < max_inner; it++) {
      rc = linearize_device(c, sets, 2, cfg, kEvalCandidate);
      if (rc) break;
      if (cudaMemcpyAsync(h_done, &st->done, sizeof(int), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
          cudaStreamSynchronize(c->stream) != cudaSuccess) {
        c->err = "track_cloud: done-flag read-back failed";
        rc = MLOAM_E_CUDA;
        break;
      }
      if (*h_done) break;
    }
  }
  if (rc) return rc;
  LMState *hs = reinterpret_cast<LMState *>(reinterpret_cast<char *>(c->pinned) + 4096);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hs, st, sizeof(LMState), cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  // :126-128 Pose(q, t) normalises
  const Q4 q = qnormalized(Q4{hs->x[3], hs->x[4], hs->x[5], hs->x[6]});
  pose_out7[0] = hs->x[0], pose_out7[1] = hs->x[1], pose_out7[2] = hs->x[2];
  pose_out7[3] = q.x, pose_out7[4] = q.y, pose_out7[5] = q.z, pose_out7[6] = q.w;
  if (stats) {
    stats->ran = 1;
    stats->n_corner = hs->n_valid[0], stats->n_surf = hs->n_valid[1];
    stats->lm_iterations = hs->total_iterations;
    stats->termination = hs->termination;
    stats->final_cost = hs->cost;
    stats->n_corner_in = n_cs, stats->n_surf_in = n_cf;
  }
  return MLOAM_OK;
}

}  // namespace mloam

using namespace mloam;

extern "C" {

int mloam_track_cloud(mloam_ctx_t *h, const mloam_point_t *h_prev_less_sharp, int n_pls, const mloam_point_t *h_prev_less_flat,
                      int n_plf, const mloam_point_t *h_cur_sharp, int n_cs, const mloam_point_t *h_cur_flat, int n_cf,
                      const double *pose_ini7, double *pose_out7, mloam_solve_stats_t *stats) {
  if (!h || !pose_ini7 || !pose_out7 || n_pls < 0 || n_plf < 0 || n_cs < 0 || n_cf < 0) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  const int ns[4] = {n_pls, n_plf, n_cs, n_cf};
  const mloam_point_t *hp[4] = {h_prev_less_sharp, h_prev_less_flat, h_cur_sharp, h_cur_flat};
  float4 *dp[4];
  DevBuf *bufs[4] = {&c->scratch[0], &c->scratch[1], &c->scan_pts[0], &c->scan_pts[1]};
  for (int k = 0; k < 4; k++) {
    if (ns[k] > 0 && !hp[k]) return MLOAM_E_INVALID;
    MLOAM_CUDA_OK(c, bufs[k]->reserve(sizeof(float4) * (size_t)(ns[k] + 1)));
    dp[k] = bufs[k]->as<float4>();
    if (ns[k] > 0) MLOAM_CUDA_OK(c, cudaMemcpyAsync(dp[k], hp[k], sizeof(float4) * (size_t)ns[k], cudaMemcpyHostToDevice, c->stream));
  }
  return track_cloud_device(c, dp[0], n_pls, dp[1], n_plf, dp[2], n_cs, dp[3], n_cf, pose_ini7, pose_out7, stats);
}

// FeatureExtract::matchCornerFromScan / matchSurfFromScan against map slot `slot` (built from the previous sweep's
// features with mloam_map_build).  nn3 (nullable): [closest, ind2, ind3] per query.
int mloam_match_from_scan(mloam_ctx_t *h, int slot, int type, const mloam_point_t *h_pts, int n, const double *pose7,
                          unsigned char *h_valid, double *h_coeffs, int *h_nn3) {
  if (!h || n < 0 || !pose7 || (n > 0 && (!h_pts || !h_valid || !h_coeffs))) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  if (n == 0) return MLOAM_OK;
  const int t = type == 's' ? 1 : 0;
  MLOAM_CUDA_OK(c, c->scan_pts[t].reserve(sizeof(float4) * (size_t)n));
  int rc = reserve_feat(c, t, n);
  if (rc) return rc;
  MLOAM_CUDA_OK(c, c->scratch[3].reserve(sizeof(int) * 3 * (size_t)n));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[t].p, h_pts, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  double *d_pose;
  rc = upload_pose(c, pose7, &d_pose);
  if (rc) return rc;
  rc = match_from_scan_device(c, slot, type, c->scan_pts[t].as<float4>(), n, d_pose, c->feat_valid[t].as<unsigned char>(),
                              c->feat_coeff[t].as<float>(), c->scratch[3].as<int>());
  if (rc) return rc;
  std::vector<float> cf((size_t)n * 6);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_valid, c->feat_valid[t].p, (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(cf.data(), c->feat_coeff[t].p, sizeof(float) * 6 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  if (h_nn3) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_nn3, c->scratch[3].p, sizeof(int) * 3 * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (size_t i = 0; i < (size_t)n * 6; i++) h_coeffs[i] = (double)cf[i];
  return MLOAM_OK;
}

}  // extern "C"
