// pipeline.cu — the orchestrators of the hot path as kernel sequences on the context stream:
//   scan2MapOptimization  (lidar_mapper_keyframe.cpp:423-639, gf_method wo_gf)
//   the per-sweep frame   (extractCloud -> downsampleCurrentScan -> scan2MapOptimization)
// plus the host-buffer entry points of extraction and the voxel filters.
//
// Feature counts produced on the device (extraction, voxel filters) are consumed on the device: kernels are
// sized for the host-known upper bound and read the true count from HBM, so a frame with max_inner == 1 runs
// without a single host round trip until the final pose read-back.
#include <cstdio>
#include <cstring>

#include "ctx.h"
#include "host_util.h"

using namespace mloam;

namespace {

typedef Ctx::ScanRef ScanRef;

// Enqueue the whole solve on the context stream (no host synchronisation when max_inner == 1, so the sequence can be
// captured into a CUDA graph); scan2map_finish() waits and unpacks.  c->s2m_ran tells finish whether the gate passed.
int scan2map_enqueue(Ctx *c, const ScanRef &S, const double *pose_init7) {
  const mloam_params_t &P = c->params;
  c->s2m_ran = 0;
  const MapStorage &MS = c->maps[MLOAM_MAP_SURF], &MC = c->maps[MLOAM_MAP_CORNER];
  if (!MS.built || !MC.built) return fail(c, MLOAM_E_STATE, "scan2map: build MLOAM_MAP_SURF and MLOAM_MAP_CORNER first");
  if (!((MS.m > 50) && (MC.m > 10))) return MLOAM_OK;  // lidar_mapper_keyframe.cpp:429 ("Map surf num is not enough")
  c->s2m_ran = 1;
  // Collective solve: the gate above depends on the replicated maps only, so every rank takes the same branch; from here on
  // every rank enqueues the same number of LM evaluations (max_outer x (1 + max_inner) with max_inner == 1; with max_inner > 1
  // the done flag all ranks poll is the identical, summed state).  Per-rank solves (tracker, odometry) are not collective.
  const SolveCfg solve{map_sqrt_info(P.cov_trace), P.huber_a, P.eig_thre, true};
  int rc = reserve_feat(c, 0, S.n_corner);
  if (rc) return rc;
  rc = reserve_feat(c, 1, S.n_surf);
  if (rc) return rc;
  rc = lm_init_state(c, pose_init7, P.max_inner, 0);
  if (rc) return rc;
  LMState *st = c->lm_state.as<LMState>();
  const double *d_pose = st->x;  // first member
  const MatchCfg cfg = match_cfg(c);
  int *h_done = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 2048);
  const int nc_use = P.point_edge_factor ? S.n_corner : 0, ns_use = P.point_plane_factor ? S.n_surf : 0;
  FeatSet sets[2] = {
      FeatSet{S.corner, c->feat_valid[0].as<unsigned char>(), c->feat_coeff[0].as<float>(), nc_use, 0, S.d_n_corner, S.sinfo_corner},
      FeatSet{S.surf, c->feat_valid[1].as<unsigned char>(), c->feat_coeff[1].as<float>(), ns_use, 1, S.d_n_surf, S.sinfo_surf}};
  // without good-feature selection nothing reads the fit before the solve: its launch folds into the first evaluation
  PendingFit fit;
  PendingFit *const defer = (c->fuse_iter && P.gf_method == 0) ? &fit : nullptr;
  for (int outer = 0; outer < P.max_outer; outer++) {
    // :503-532  match corner then surf at pose_wmap_curr (wo_gf: every feature)
    {
      // From the second iteration on the same features meet the same maps at a slightly moved pose: the previous
      // neighbour lists seed the search (exact, see knn.cuh) and unchanged lists keep their line / plane fit.
      const int seeded = (outer > 0 && c->use_seeds) ? 1 : 0;
      MatchJob jobs[2] = {
          MatchJob{MLOAM_MAP_CORNER, 'c', S.corner, nc_use, S.d_n_corner, c->feat_valid[0].as<unsigned char>(),
                   c->feat_coeff[0].as<float>(), nullptr, seeded},
          MatchJob{MLOAM_MAP_SURF, 's', S.surf, ns_use, S.d_n_surf, c->feat_valid[1].as<unsigned char>(),
                   c->feat_coeff[1].as<float>(), nullptr, seeded}};
      rc = match_pair_device(c, jobs, 2, d_pose, cfg, 0, defer);
      if (rc) return rc;
      stamp(c, "match");
    }
    // goodFeatureMatching (:503-532 with FLAGS_gf_method != wo_gf): select gf_ratio of the features per set, on the device;
    // the solve below only sees the selected ones.  Corner first, then surf, as in the reference.
    sets[0].mask = sets[1].mask = nullptr;
    if (P.gf_method != 0) {
      // the two selections are independent single-CTA chains: corner on the side stream next to surf (also inside a captured graph)
      const bool fork_gf = !c->prof_on && sets[0].n > 0 && sets[1].n > 0;
      if (fork_gf) {
        MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_fork3, c->stream));
        MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream3, c->ev_fork3, 0));
      }
      for (int t = 0; t < 2; t++) {
        if (sets[t].n <= 0) continue;
        unsigned char *mask = nullptr;
        cudaStream_t main_stream = c->stream;
        if (fork_gf && t == 0) c->stream = c->stream3;
        rc = gf_select_set_device(c, t, sets[t], d_pose, solve.sqrt_info, P.gf_method, (double)P.gf_ratio,
                                  (unsigned long long)P.gf_seed + 2ull * (unsigned long long)outer + (unsigned long long)t, &mask);
        c->stream = main_stream;
        if (rc) return rc;
        if (fork_gf && t == 0) MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_join3, c->stream3));
        sets[t].mask = mask;
      }
      if (fork_gf) MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream, c->ev_join3, 0));
    }
    // :537-582 residual blocks + Evaluate -> J^T J -> evalDegenracy, and iteration 0 of ceres::Solve.  The device
    // only needs the degeneracy decision; scan2map_finish fills in the eigenvalue report of the last iteration.
    if (P.gf_method != 0) stamp(c, "gf");
    // max_inner == 1: the candidate of the one LM iteration is evaluated in the same launch
    bool second_done = false;
    rc = linearize_device(c, sets, 2, solve, kEvalBegin, nullptr, nullptr, defer, c->fuse_iter && P.max_inner == 1, &second_done);
    if (rc) return rc;
    stamp(c, second_done ? "linearize x2" : "linearize");
    // :586-596 ceres::Solve, at most max_inner LM iterations; the device raises `done`
    for (int it = 0; it < P.max_inner && !second_done; it++) {
      rc = linearize_device(c, sets, 2, solve, kEvalCandidate);
      if (rc) return rc;
      stamp(c, "linearize (candidate)");
      if (P.max_inner > 1) {
        MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_done, &st->done, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
        if (*h_done) break;
      }
    }
  }
  char *pin = reinterpret_cast<char *>(c->pinned);
  LMState *hs = reinterpret_cast<LMState *>(pin + 4096);
  int *h_cnt = reinterpret_cast<int *>(pin + 3072);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hs, st, sizeof(LMState), cudaMemcpyDeviceToHost, c->stream));
  if (S.d_n_surf) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_cnt, S.d_n_surf, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if (S.d_n_corner) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_cnt + 1, S.d_n_corner, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  return MLOAM_OK;
}

int scan2map_finish(Ctx *c, const ScanRef &S, const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  if (stats) memset(stats, 0, sizeof(*stats));
  for (int k = 0; k < 7; k++) pose_out7[k] = pose_init7[k];
  if (!c->s2m_ran) return MLOAM_OK;
  char *pin = reinterpret_cast<char *>(c->pinned);
  const LMState *hs = reinterpret_cast<const LMState *>(pin + 4096);
  int *h_cnt = reinterpret_cast<int *>(pin + 3072);
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  if (!S.d_n_surf) h_cnt[0] = S.n_surf;
  if (!S.d_n_corner) h_cnt[1] = S.n_corner;
  for (int k = 0; k < 7; k++) pose_out7[k] = hs->x[k];
  if (hs->termination == 9) {  // the peer-memory exchange timed out or the ranks lost lock-step: the summed state is not trustworthy
    for (int k = 0; k < 7; k++) pose_out7[k] = pose_init7[k];
    if (stats) stats->ran = 1, stats->termination = 9;
    return fail(c, MLOAM_E_NCCL, "scan2map: peer-memory exchange failed (a rank did not arrive or the ranks lost lock-step); "
                                  "call mloam_comm_p2p_reset on every rank behind a barrier");
  }
  if (hs->termination == 8) {  // k_linearize's grid barrier gave up: a block of the grid never became resident within ~2 s
    for (int k = 0; k < 7; k++) pose_out7[k] = pose_init7[k];
    if (stats) stats->ran = 1, stats->termination = 8;
    return fail(c, MLOAM_E_STATE, "scan2map: the two-evaluation launch timed out at its grid barrier (GPU shared with a kernel that never "
                                   "yields?); set MLOAM_FUSE_ITER=0 to use one launch per evaluation");
  }
  if (c->prof_on) {  // device-side cycle counters of the fused LM tail, reported next to the event-timed stages
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->device);
    if (khz > 0) {
      c->prof["lm_tail_reduce"].ms += (double)hs->dbg_cycles[0] / khz, c->prof["lm_tail_reduce"].launches += hs->dbg_cycles[2];
      c->prof["lm_tail_advance"].ms += (double)hs->dbg_cycles[1] / khz, c->prof["lm_tail_advance"].launches += hs->dbg_cycles[2];
    }
  }
  if (stats) {
    stats->ran = 1;
    stats->n_corner = hs->n_valid[0], stats->n_surf = hs->n_valid[1];
    stats->lm_iterations = hs->total_iterations;
    stats->degenerate = hs->is_degenerate;
    stats->termination = hs->termination;
    stats->final_cost = hs->cost;
    memcpy(stats->eig, hs->eig, sizeof(stats->eig));
    memcpy(stats->H, hs->H0, sizeof(stats->H));
    // evalDegenracy's eigenvalues (lidar_mapper_keyframe.cpp:1172-1204): the device decides degeneracy with a
    // Cholesky test of H - thre*I and only runs the eigen-solver when that fails; the report of a healthy Solve is
    // computed here from the same H.
    if (!hs->is_degenerate && !hs->skipped && hs->rows > 0 && c->params.eig_thre > 0.0) eig_report_host(hs->H0, stats->eig);
    stats->n_surf_in = h_cnt[0], stats->n_corner_in = h_cnt[1];
  }
  return MLOAM_OK;
}

int scan2map_run(Ctx *c, const ScanRef &S, const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  int rc = scan2map_enqueue(c, S, pose_init7);
  if (rc) return rc;
  return scan2map_finish(c, S, pose_init7, pose_out7, stats);
}

// Device buffers of one frame: feature sets of extractCloud + the down-sampled scans fed to matching.
struct FrameBufs {
  ExtractOut ex;
  float4 *corner_ds, *surf_ds;
  int *n_corner_ds, *n_surf_ds;  // device counts
};
int frame_bufs(Ctx *c, int n, FrameBufs *F, int parity = 0) {
  DevBuf &B = parity ? c->frame_alt : c->frame_main;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  };
  const size_t N1 = (size_t)n + 16;
  const size_t o_sharp = take(16 * N1), o_less = take(16 * N1), o_flat = take(16 * N1), o_lflat = take(16 * N1);
  const size_t o_cds = take(16 * N1), o_sds = take(16 * N1), o_cnt = take(64);
  MLOAM_CUDA_OK(c, B.reserve(off));
  char *p = B.as<char>();
  F->ex.sharp = reinterpret_cast<float4 *>(p + o_sharp), F->ex.less_sharp = reinterpret_cast<float4 *>(p + o_less);
  F->ex.flat = reinterpret_cast<float4 *>(p + o_flat), F->ex.less_flat = reinterpret_cast<float4 *>(p + o_lflat);
  F->corner_ds = reinterpret_cast<float4 *>(p + o_cds), F->surf_ds = reinterpret_cast<float4 *>(p + o_sds);
  int *cnt = reinterpret_cast<int *>(p + o_cnt);
  F->ex.counts = cnt;  // [0..3]
  F->n_corner_ds = cnt + 4, F->n_surf_ds = cnt + 5;
  return MLOAM_OK;
}

bool frame_has_prefetched(const Ctx *c, const void *key_ptr, int n, int n_scans) {
  const Ctx::Features &f = c->prefetched;
  return f.valid && c->use_lookahead && !c->prof_on && f.key_ptr == key_ptr && f.n == n && f.n_scans == n_scans;
}

// extractCloud + (multi-LiDAR merge | base-frame transform) + downsampleCurrentScan of one sweep on c->stream, into half `parity` of the
// feature double buffer.  `side` / ev_fork_v / ev_join_v: the stream and events of the corner-filter fork.
int features_enqueue(Ctx *c, const float4 *d_cloud, int n, const int *d_scan_start, const int *d_scan_end, int n_scans, int parity,
                     cudaStream_t side, cudaEvent_t ev_fork_v, cudaEvent_t ev_join_v, ScanRef *S_out) {
  const mloam_params_t &P = c->params;
  FrameBufs F;
  int rc = frame_bufs(c, n, &F, parity);
  if (rc) return rc;
  rc = extract_device(c, d_cloud, n, d_scan_start, d_scan_end, n_scans, F.ex, nullptr, nullptr);
  if (rc) return rc;
  stamp(c, "extract");
  const int less_cap = n < 120 * n_scans ? n : 120 * n_scans;  // <= 20 less-sharp picks x 6 sectors per ring
  if (c->n_lidars > 1 || c->lidar_merge) {
    // batched sweeps of several LiDARs: features of LiDAR l go to the base frame with its extrinsic, intensity = l
    // (transformCloudFeature, visualization.cpp:40-52), LiDAR after LiDAR as pubPointCloud's `+=` (:93-104)
    if (n_scans % c->n_lidars != 0) return fail(c, MLOAM_E_INVALID, "frame: n_scans must be n_lidars x rings per LiDAR");
    float *stage = reinterpret_cast<float *>(reinterpret_cast<char *>(c->pinned) + 12288);
    for (int l = 0; l < c->n_lidars; l++) {
      const double *e = c->lidar_ext[l];
      const M33 R = qmat(qnormalized(Q4{e[3], e[4], e[5], e[6]}));  // Pose(q, t): q normalised, T_ = [R | t] (pose.cpp:34-41), cast<float>
      for (int r = 0; r < 3; r++) {
        for (int k = 0; k < 3; k++) stage[12 * l + 4 * r + k] = (float)R.m[3 * r + k];
        stage[12 * l + 4 * r + 3] = (float)e[r];
      }
    }
    float *d_ext12 = reinterpret_cast<float *>(c->scratch[7].as<char>() + 1024);
    int *d_off = reinterpret_cast<int *>(c->scratch[7].as<char>() + 2048);
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_ext12, stage, sizeof(float) * 12 * c->n_lidars, cudaMemcpyHostToDevice, c->stream));
    rc = merge_lidars_device(c, F.ex, less_cap, n, c->n_lidars, n_scans / c->n_lidars, d_ext12, d_off);
    if (rc) return rc;
  } else if (c->has_ext) {  // features are handed to the mapper in the base frame
    double *stage = reinterpret_cast<double *>(c->pinned) + 32;
    for (int k = 0; k < 7; k++) stage[k] = c->ext[k];
    double *d_ext = c->scratch[7].as<double>() + 32;
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_ext, stage, 7 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    rc = transform_points_device(c, F.ex.less_sharp, less_cap, F.ex.counts + 1, d_ext);
    if (rc) return rc;
    rc = transform_points_device(c, F.ex.less_flat, n, F.ex.counts + 3, d_ext);
    if (rc) return rc;
  }
  // downsampleCurrentScan, lidar_mapper_keyframe.cpp:356-364 (VoxelGridCovarianceMLOAM<PointI>: xyz mean, last intensity)
  // The two filters are independent chains of small kernels: the corner one runs on a second side stream next to the
  // surf one (own scratch slot), also inside a captured graph; with stage profiling on they stay serial.
  const bool fork_voxel = !c->prof_on;
  if (fork_voxel) {
    MLOAM_CUDA_OK(c, cudaEventRecord(ev_fork_v, c->stream));
    MLOAM_CUDA_OK(c, cudaStreamWaitEvent(side, ev_fork_v, 0));
    cudaStream_t main_stream = c->stream;
    c->stream = side;
    rc = voxel_downsample_device(c, F.ex.less_sharp, less_cap, F.ex.counts + 1, P.corner_leaf, 1, F.corner_ds, F.n_corner_ds, 8);
    c->stream = main_stream;
    if (rc) return rc;
    MLOAM_CUDA_OK(c, cudaEventRecord(ev_join_v, side));
  } else {
    rc = voxel_downsample_device(c, F.ex.less_sharp, less_cap, F.ex.counts + 1, P.corner_leaf, 1, F.corner_ds, F.n_corner_ds, 8);
    if (rc) return rc;
  }
  rc = voxel_downsample_device(c, F.ex.less_flat, n, F.ex.counts + 3, P.surf_leaf, 1, F.surf_ds, F.n_surf_ds, 9);
  if (rc) return rc;
  if (fork_voxel) MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream, ev_join_v, 0));
  stamp(c, "voxel (surf; corner on the side stream)");
  ScanRef S{F.surf_ds, n, F.n_surf_ds, F.corner_ds, less_cap, F.n_corner_ds};
  *S_out = S;
  return MLOAM_OK;
}

int frame_enqueue(Ctx *c, const float4 *d_cloud, int n, const int *d_scan_start, const int *d_scan_end, int n_scans,
                  const float4 *d_surf_map, int n_surf_map, const float4 *d_corner_map, int n_corner_map, int rebuild_maps,
                  const double *pose_init7, ScanRef *S_out) {
  int rc;
  bool forked = false;
  if (rebuild_maps) {  // lidar_mapper_keyframe.cpp:433-434 (every frame in the reference)
    // The two submap builds do not depend on the sweep: they run on a forked side stream, concurrently with
    // extraction + scan down-sampling, and join right before matching (also inside a captured graph).
    // With stage profiling on the branch stays on the main stream so that per-stage event times do not overlap.
    forked = !c->prof_on;
    if (!forked) {
      if (c->maps_pending) MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream, c->ev_maps, 0));
      rc = map_build_device(c, MLOAM_MAP_SURF, d_surf_map, n_surf_map, pick_cell(c, 0.f));
      if (rc == MLOAM_OK) rc = map_build_device(c, MLOAM_MAP_CORNER, d_corner_map, n_corner_map, pick_cell(c, 0.f));
      if (rc) return rc;
    }
  }
  if (forked) {
    MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_fork, c->stream));
    MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream2, c->ev_fork, 0));
    if (c->maps_pending) {
      // mloam_frame copied the submaps on stream2 outside of any capture: inside a captured graph the branch waits
      // on that record as an external event node; on the plain stream path stream2 is already ordered after it.
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      MLOAM_CUDA_OK(c, cudaStreamIsCapturing(c->stream2, &cs));
      if (cs == cudaStreamCaptureStatusActive) MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream2, c->ev_maps, cudaEventWaitExternal));
    }
    cudaStream_t main_stream = c->stream;
    c->stream = c->stream2;
    rc = map_build_device(c, MLOAM_MAP_SURF, d_surf_map, n_surf_map, pick_cell(c, 0.f));
    if (rc == MLOAM_OK) rc = map_build_device(c, MLOAM_MAP_CORNER, d_corner_map, n_corner_map, pick_cell(c, 0.f));
    c->stream = main_stream;
    if (rc) return rc;
    MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_join, c->stream2));
  }
  c->stamp_n = 0;
  stamp(c, "start");
  // features of this sweep: extracted while the previous frame was solved (look-ahead), or now
  ScanRef S{};
  int parity = c->frame_parity;
  const void *key_now = c->cloud_key ? c->cloud_key : static_cast<const void *>(d_cloud);
  const bool have = frame_has_prefetched(c, key_now, n, n_scans);
  if (have) {
    S = c->prefetched.S, parity = c->prefetched.parity;
  } else {
    rc = features_enqueue(c, d_cloud, n, d_scan_start, d_scan_end, n_scans, parity, c->stream3, c->ev_fork3, c->ev_join3, &S);
    if (rc) return rc;
  }
  c->prefetched.valid = false;
  c->frame_parity = parity ^ 1;
  // look-ahead: the announced next sweep goes through the same steps on stream4 into the other half while this frame is matched
  // and solved (the extraction scratch is shared with the block above, hence the fork AFTER it)
  bool ahead = false;
  Ctx::Features nf{};
  if (c->next.set && c->use_lookahead && !c->prof_on) {
    const Ctx::NextSweep nx = c->next;
    MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_fork4, c->stream));
    MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream4, c->ev_fork4, 0));
    if (c->next_pending) {  // mloam_frame copied the next sweep on stream4 outside of any capture (as ev_maps above)
      cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
      MLOAM_CUDA_OK(c, cudaStreamIsCapturing(c->stream4, &cs));
      if (cs == cudaStreamCaptureStatusActive) MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream4, c->ev_next, cudaEventWaitExternal));
    }
    cudaStream_t main_stream = c->stream;
    c->stream = c->stream4;
    c->stamp_mute = true;
    ScanRef Sn{};
    rc = features_enqueue(c, nx.d_cloud, nx.n, nx.d_scan_start, nx.d_scan_end, nx.n_scans, parity ^ 1, c->stream5, c->ev_fork5, c->ev_join5, &Sn);
    c->stamp_mute = false;
    c->stream = main_stream;
    if (rc) return rc;
    MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_join4, c->stream4));
    ahead = true;
    nf.valid = true, nf.host = nx.host, nf.key_ptr = nx.key_ptr, nf.n = nx.n, nf.n_scans = nx.n_scans, nf.parity = parity ^ 1, nf.S = Sn;
  }
  c->next.set = false;
  stamp(c, have ? "features (prefetched)" : "extract + voxel");
  if (forked) MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream, c->ev_join, 0));  // join the map-build branch
  if (forked) stamp(c, "map build join");
  *S_out = S;
  rc = scan2map_enqueue(c, S, pose_init7);
  if (rc) return rc;
  if (ahead) {  // the frame ends when both branches have: the features of the next sweep are complete when this call returns
    MLOAM_CUDA_OK(c, cudaStreamWaitEvent(c->stream, c->ev_join4, 0));
    stamp(c, "look-ahead join");
    c->prefetched = nf;
  }
  return MLOAM_OK;
}

// A sweep announced from HOST memory goes up on stream4 right away (outside of any capture); the look-ahead branch of the frame
// waits on ev_next.  stream4's previous work — the look-ahead of the previous frame, which read next_in — was joined by that frame.
int stage_next_sweep(Ctx *c) {
  if (!c->next.set || !c->next.host || !c->use_lookahead || c->prof_on) return MLOAM_OK;
  const int n = c->next.n, ns = c->next.n_scans;
  DevBuf &in = c->next_in;
  MLOAM_CUDA_OK(c, in.reserve(sizeof(float4) * (size_t)n + 1024 + 8 * (size_t)ns));
  float4 *d_cloud = in.as<float4>();
  int *d_ss = reinterpret_cast<int *>(in.as<char>() + sizeof(float4) * (size_t)n + 256);
  int *d_se = d_ss + ns;
  // ScanInfo goes through the context's pinned block: an async copy from pageable memory would block the host behind the sweep's copy
  int *pin = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + kPinnedScanInfoNext);
  std::memcpy(pin, c->next_host_ss, sizeof(int) * ns), std::memcpy(pin + MLOAM_MAX_RINGS, c->next_host_se, sizeof(int) * ns);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_ss, pin, sizeof(int) * ns, cudaMemcpyHostToDevice, c->stream4));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_se, pin + MLOAM_MAX_RINGS, sizeof(int) * ns, cudaMemcpyHostToDevice, c->stream4));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_cloud, c->next.key_ptr, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, c->stream4));
  MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_next, c->stream4));
  c->next.d_cloud = d_cloud, c->next.d_scan_start = d_ss, c->next.d_scan_end = d_se;
  c->next_pending = true;
  return MLOAM_OK;
}

unsigned long long fnv1a(unsigned long long h, const void *p, size_t n) {
  const unsigned char *b = static_cast<const unsigned char *>(p);
  for (size_t i = 0; i < n; i++) h = (h ^ b[i]) * 1099511628211ull;
  return h;
}

// One frame.  With max_inner == 1 the ~60 launches of a frame form a fixed sequence that depends on the host only
// through the pose guess (staged in pinned memory) — it is captured once per (buffers, sizes, parameters) into a CUDA
// graph and replayed: the first call with a new key runs on the stream (and performs every allocation), the second
// captures + instantiates, later ones replay.  Profiling, multi-GPU (NCCL on the stream) and max_inner > 1 (the host
// polls the LM done flag) use the plain stream path.
int frame_run(Ctx *c, const float4 *d_cloud, int n, const int *d_scan_start, const int *d_scan_end, int n_scans,
              const float4 *d_surf_map, int n_surf_map, const float4 *d_corner_map, int n_corner_map, int rebuild_maps,
              const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  ScanRef S{};
  const bool can_graph = c->use_graphs && c->params.max_inner == 1 && !c->prof_on && (!c->nccl_comm || c->p2p_on);
  if (can_graph) {
    unsigned long long key = 1469598103934665603ull;
    const void *ptrs[5] = {d_cloud, d_scan_start, d_scan_end, d_surf_map, d_corner_map};
    const int ints[7] = {n, n_scans, n_surf_map, n_corner_map, rebuild_maps, c->has_ext ? 1 : 0, c->maps_pending ? 1 : 0};
    key = fnv1a(key, ptrs, sizeof(ptrs));
    key = fnv1a(key, ints, sizeof(ints));
    if (rebuild_maps && !(c->params.map_cell > 0.f)) {  // the auto cell edges are kernel arguments of the captured build
      const float cells[2] = {c->maps[MLOAM_MAP_SURF].auto_cell_pick(c->pinned, MLOAM_MAP_SURF),
                              c->maps[MLOAM_MAP_CORNER].auto_cell_pick(c->pinned, MLOAM_MAP_CORNER)};
      key = fnv1a(key, cells, sizeof(cells));
    }
    key = fnv1a(key, &c->params, sizeof(c->params));
    key = fnv1a(key, c->ext, sizeof(c->ext));
    key = fnv1a(key, &c->n_lidars, sizeof(c->n_lidars));
    key = fnv1a(key, &c->lidar_merge, sizeof(c->lidar_merge));
    key = fnv1a(key, c->lidar_ext, sizeof(double) * 7 * (size_t)c->n_lidars);
    key = fnv1a(key, &c->stream, sizeof(c->stream));
    {  // look-ahead: which half holds this sweep's features (or that they are extracted now), and the announced next sweep
      const void *key_now = c->cloud_key ? c->cloud_key : static_cast<const void *>(d_cloud);
      const bool have = frame_has_prefetched(c, key_now, n, n_scans);
      const bool ahead = c->next.set && c->use_lookahead;
      const int la[8] = {have ? 1 : 0, have ? c->prefetched.parity : c->frame_parity, ahead ? 1 : 0, ahead ? c->next.n : 0, ahead ? c->next.n_scans : 0,
                         (ahead && c->next.host) ? 1 : 0, (ahead && c->next_pending) ? 1 : 0, c->stamp_on ? 1 : 0};
      const void *lp[5] = {key_now, ahead ? c->next.key_ptr : nullptr, ahead ? static_cast<const void *>(c->next.d_cloud) : nullptr,
                           ahead ? static_cast<const void *>(c->next.d_scan_start) : nullptr, ahead ? static_cast<const void *>(c->next.d_scan_end) : nullptr};
      key = fnv1a(key, la, sizeof(la));
      key = fnv1a(key, lp, sizeof(lp));
    }
    Ctx::GraphEntry *e = nullptr;
    for (auto &g : c->graphs)
      if (g.key == key) e = &g;
    if (e && e->exec && e->epoch == alloc_epoch()) {
      double *stage = reinterpret_cast<double *>(c->pinned);
      for (int k = 0; k < 7; k++) stage[k] = pose_init7[k];  // the captured H2D node reads this at execution time
      if (c->has_ext)
        for (int k = 0; k < 7; k++) stage[32 + k] = c->ext[k];
      MLOAM_CUDA_OK(c, cudaGraphLaunch(e->exec, c->stream));
      c->launches += e->launches;
      c->s2m_ran = e->s2m_ran;
      // the state transitions frame_enqueue makes at capture time
      c->frame_parity = (frame_has_prefetched(c, c->cloud_key ? c->cloud_key : static_cast<const void *>(d_cloud), n, n_scans) ? c->prefetched.parity : c->frame_parity) ^ 1;
      c->prefetched = e->prefetched_out;
      c->next.set = false;
      return scan2map_finish(c, e->S, pose_init7, pose_out7, stats);
    }
    if (e && e->seen >= 1) {  // second sighting: capture
      if (e->exec) cudaGraphExecDestroy(e->exec), e->exec = nullptr;
      const long long l0 = c->launches;
      const unsigned long long ep0 = alloc_epoch();
      cudaGraph_t graph = nullptr;
      const Ctx::Features pf0 = c->prefetched;  // frame_enqueue consumes these: put them back when the capture fails
      const Ctx::NextSweep nx0 = c->next;
      const int par0 = c->frame_parity;
      MLOAM_CUDA_OK(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      int rc = frame_enqueue(c, d_cloud, n, d_scan_start, d_scan_end, n_scans, d_surf_map, n_surf_map, d_corner_map, n_corner_map,
                             rebuild_maps, pose_init7, &S);
      cudaError_t ce = cudaStreamEndCapture(c->stream, &graph);
      if (rc == MLOAM_OK && ce == cudaSuccess && graph && ep0 == alloc_epoch() &&
          cudaGraphInstantiate(&e->exec, graph, 0) == cudaSuccess) {
        e->launches = (int)(c->launches - l0), e->epoch = ep0, e->S = S, e->s2m_ran = c->s2m_ran;
        e->prefetched_out = c->prefetched;
        c->launches = l0;
        cudaGraphDestroy(graph);
        MLOAM_CUDA_OK(c, cudaGraphLaunch(e->exec, c->stream));
        c->launches += e->launches;
        return scan2map_finish(c, S, pose_init7, pose_out7, stats);
      }
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      e->exec = nullptr, e->seen = 0;  // capture failed (e.g. a buffer had to grow, which is illegal while capturing): run this frame on
      c->launches = l0;                // the plain stream path below — it performs the allocation — and capture at a later sighting
      c->graph_capture_failures++;
      c->prefetched = pf0, c->next = nx0, c->frame_parity = par0;
    } else if (!e) {
      if (c->graphs.size() >= 96) {
        if (c->graphs.front().exec) cudaGraphExecDestroy(c->graphs.front().exec);
        c->graphs.erase(c->graphs.begin());
      }
      Ctx::GraphEntry g;
      g.key = key, g.seen = 1;
      c->graphs.push_back(g);
    }
  }
  int rc = frame_enqueue(c, d_cloud, n, d_scan_start, d_scan_end, n_scans, d_surf_map, n_surf_map, d_corner_map, n_corner_map,
                         rebuild_maps, pose_init7, &S);
  if (rc) return rc;
  return scan2map_finish(c, S, pose_init7, pose_out7, stats);
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------ scan2map
int mloam_scan2map_device(mloam_ctx_t *h, const mloam_point_t *d_surf_scan, int n_surf, const mloam_point_t *d_corner_scan,
                          int n_corner, const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  if (!h || !pose_init7 || !pose_out7 || n_surf < 0 || n_corner < 0) return MLOAM_E_INVALID;
  cudaSetDevice(h->c.device);
  ScanRef S{reinterpret_cast<const float4 *>(d_surf_scan), n_surf, nullptr, reinterpret_cast<const float4 *>(d_corner_scan), n_corner,
            nullptr};
  return scan2map_run(&h->c, S, pose_init7, pose_out7, stats);
}

int mloam_scan2map(mloam_ctx_t *h, const mloam_point_t *h_surf_scan, int n_surf, const mloam_point_t *h_corner_scan, int n_corner,
                   const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  if (!h || !pose_init7 || !pose_out7 || n_surf < 0 || n_corner < 0) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  MLOAM_CUDA_OK(c, c->scan_pts[0].reserve(sizeof(float4) * (size_t)(n_corner + 1)));
  MLOAM_CUDA_OK(c, c->scan_pts[1].reserve(sizeof(float4) * (size_t)(n_surf + 1)));
  if (n_corner > 0)
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[0].p, h_corner_scan, sizeof(float4) * (size_t)n_corner, cudaMemcpyHostToDevice, c->stream));
  if (n_surf > 0)
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[1].p, h_surf_scan, sizeof(float4) * (size_t)n_surf, cudaMemcpyHostToDevice, c->stream));
  ScanRef S{c->scan_pts[1].as<float4>(), n_surf, nullptr, c->scan_pts[0].as<float4>(), n_corner, nullptr};
  return scan2map_run(c, S, pose_init7, pose_out7, stats);
}

// scan2MapOptimization with with_ua = true (lidar_mapper_keyframe.cpp:541-545,556-560): every residual is weighted by
// sqrt_info of its scan point's covariance (PointIWithCov::cov_vec, float[6] per point, from mloam_point_uncertainty).
int mloam_scan2map_ua(mloam_ctx_t *h, const mloam_point_t *h_surf_scan, int n_surf, const float *h_surf_cov6,
                      const mloam_point_t *h_corner_scan, int n_corner, const float *h_corner_cov6, const double *pose_init7,
                      double *pose_out7, mloam_solve_stats_t *stats) {
  if (!h || !pose_init7 || !pose_out7 || n_surf < 0 || n_corner < 0 || (n_surf > 0 && (!h_surf_scan || !h_surf_cov6)) ||
      (n_corner > 0 && (!h_corner_scan || !h_corner_cov6)))
    return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  cudaStream_t st = c->stream;
  const int ns[2] = {n_corner, n_surf};
  const mloam_point_t *hp[2] = {h_corner_scan, h_surf_scan};
  const float *hc[2] = {h_corner_cov6, h_surf_cov6};
  DevBuf *cov[2] = {&c->scratch[1], &c->scratch[2]}, *sin[2] = {&c->scratch[3], &c->scratch[4]};
  for (int t = 0; t < 2; t++) {
    MLOAM_CUDA_OK(c, c->scan_pts[t].reserve(sizeof(float4) * (size_t)(ns[t] + 1)));
    MLOAM_CUDA_OK(c, cov[t]->reserve(sizeof(float) * 6 * (size_t)(ns[t] + 1)));
    MLOAM_CUDA_OK(c, sin[t]->reserve(sizeof(double) * (size_t)(ns[t] + 1)));
    if (ns[t] > 0) {
      MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[t].p, hp[t], sizeof(float4) * (size_t)ns[t], cudaMemcpyHostToDevice, st));
      MLOAM_CUDA_OK(c, cudaMemcpyAsync(cov[t]->p, hc[t], sizeof(float) * 6 * (size_t)ns[t], cudaMemcpyHostToDevice, st));
      int rc = sqrt_info_device(c, cov[t]->as<float>(), ns[t], sin[t]->as<double>());
      if (rc) return rc;
    }
  }
  ScanRef S{c->scan_pts[1].as<float4>(), n_surf, nullptr, c->scan_pts[0].as<float4>(), n_corner, nullptr, sin[1]->as<double>(),
            sin[0]->as<double>()};
  return scan2map_run(c, S, pose_init7, pose_out7, stats);
}

// ------------------------------------------------------------------------------------------ extractCloud
int mloam_extract_features(mloam_ctx_t *h, const mloam_point_t *h_cloud, int n, const int *h_scan_start, const int *h_scan_end,
                           int n_scans, mloam_features_t *out) {
  if (!h || !out || n < 0 || n_scans <= 0 || n_scans > MLOAM_MAX_RINGS || (n > 0 && !h_cloud) || !h_scan_start || !h_scan_end)
    return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  out->n_sharp = out->n_less_sharp = out->n_flat = out->n_less_flat = 0;
  if (n == 0) return MLOAM_OK;
  c->prefetched.valid = false;  // this call reuses half 0 of the frame feature buffers
  FrameBufs F;
  int rc = frame_bufs(c, n, &F);
  if (rc) return rc;
  DevBuf &in = c->scratch[0];
  MLOAM_CUDA_OK(c, in.reserve(sizeof(float4) * (size_t)n + 1024 + 8 * (size_t)n_scans));
  float4 *d_cloud = in.as<float4>();
  int *d_ss = reinterpret_cast<int *>(in.as<char>() + sizeof(float4) * (size_t)n + 256);
  int *d_se = d_ss + n_scans;
  cudaStream_t st = c->stream;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_cloud, h_cloud, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, st));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_ss, h_scan_start, sizeof(int) * n_scans, cudaMemcpyHostToDevice, st));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_se, h_scan_end, sizeof(int) * n_scans, cudaMemcpyHostToDevice, st));
  rc = extract_device(c, d_cloud, n, d_ss, d_se, n_scans, F.ex, nullptr, nullptr);
  if (rc) return rc;
  int *hc = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 3072);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hc, F.ex.counts, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hc + 4, c->d_extract_status, sizeof(int), cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  if (hc[4] != 0)
    return fail(c, MLOAM_E_INVALID, "extract: a ring exceeds the on-chip window (12288 points) or ScanInfo is out of range");
  if (hc[0] > out->cap || hc[1] > out->cap || hc[2] > out->cap || hc[3] > out->cap)
    return fail(c, MLOAM_E_INVALID, "extract: output capacity too small");
  out->n_sharp = hc[0], out->n_less_sharp = hc[1], out->n_flat = hc[2], out->n_less_flat = hc[3];
  if (out->corner_points_sharp && hc[0])
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(out->corner_points_sharp, F.ex.sharp, sizeof(float4) * hc[0], cudaMemcpyDeviceToHost, st));
  if (out->corner_points_less_sharp && hc[1])
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(out->corner_points_less_sharp, F.ex.less_sharp, sizeof(float4) * hc[1], cudaMemcpyDeviceToHost, st));
  if (out->surf_points_flat && hc[2])
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(out->surf_points_flat, F.ex.flat, sizeof(float4) * hc[2], cudaMemcpyDeviceToHost, st));
  if (out->surf_points_less_flat && hc[3])
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(out->surf_points_less_flat, F.ex.less_flat, sizeof(float4) * hc[3], cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  return MLOAM_OK;
}

int mloam_extract_debug(mloam_ctx_t *h, float *h_curvature, int *h_label, int n) {
  if (!h || n < 0) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  // layout of extract_device(): curvature at offset 0, label after it (both 4*(n+16) rounded to 256)
  const size_t blk = (4 * ((size_t)n + 16) + 255) & ~(size_t)255;
  if (c->scratch[4].cap < 2 * blk) return fail(c, MLOAM_E_STATE, "extract_debug: no extraction of this size has run");
  const char *p = c->scratch[4].as<char>();
  if (h_curvature) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_curvature, p, sizeof(float) * n, cudaMemcpyDeviceToHost, c->stream));
  if (h_label) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_label, p + blk, sizeof(int) * n, cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ range image
int mloam_project_cloud(mloam_ctx_t *h, const mloam_point_t *h_cloud, int n, int vertical_scans, int horizon_scans, double roi_range,
                        mloam_point_t *h_out, int *n_out, int *h_scan_start, int *h_scan_end) {
  if (!h || n < 0 || !n_out || !h_scan_start || !h_scan_end || (n > 0 && (!h_cloud || !h_out))) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  *n_out = 0;
  if (vertical_scans != 16 && vertical_scans != 32 && vertical_scans != 64)
    return fail(c, MLOAM_E_INVALID, "project_cloud: vertical_scans must be 16, 32 or 64 (ImageSegmenter::setParameter)");
  if (horizon_scans <= 0) return MLOAM_E_INVALID;
  if (n == 0) {  // image_segmenter.hpp:381-387 on an empty cloud
    for (int i = 0; i < vertical_scans; i++) h_scan_start[i] = 5, h_scan_end[i] = -6;
    return MLOAM_OK;
  }
  DevBuf &in = c->scratch[0], &outb = c->scratch[1];
  MLOAM_CUDA_OK(c, in.reserve(sizeof(float4) * (size_t)n));
  MLOAM_CUDA_OK(c, outb.reserve(sizeof(float4) * (size_t)n + 1024));
  cudaStream_t st = c->stream;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(in.p, h_cloud, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, st));
  int *d_meta = reinterpret_cast<int *>(outb.as<char>() + sizeof(float4) * (size_t)n);  // [0] count, [64..] start, [128..] end
  int rc = project_cloud_device(c, in.as<float4>(), n, vertical_scans, horizon_scans, roi_range, outb.as<float4>(), d_meta + 64, d_meta + 128,
                                d_meta);
  if (rc) return rc;
  int *hc = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 3072);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hc, d_meta, sizeof(int) * 192, cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  *n_out = hc[0];
  std::memcpy(h_scan_start, hc + 64, sizeof(int) * vertical_scans), std::memcpy(h_scan_end, hc + 128, sizeof(int) * vertical_scans);
  if (hc[0] > 0) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_out, outb.p, sizeof(float4) * (size_t)hc[0], cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ voxel grid
int mloam_voxel_downsample(mloam_ctx_t *h, const mloam_point_t *h_in, int n, float leaf, int intensity_last, mloam_point_t *h_out,
                           int *n_out) {
  if (!h || n < 0 || !n_out || (n > 0 && (!h_in || !h_out)) || !(leaf > 0.f)) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  *n_out = 0;
  if (n == 0) return MLOAM_OK;
  DevBuf &in = c->scratch[0], &outb = c->scratch[1];
  MLOAM_CUDA_OK(c, in.reserve(sizeof(float4) * (size_t)n));
  MLOAM_CUDA_OK(c, outb.reserve(sizeof(float4) * (size_t)n + 256));
  cudaStream_t st = c->stream;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(in.p, h_in, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, st));
  int *d_cnt = reinterpret_cast<int *>(outb.as<char>() + sizeof(float4) * (size_t)n);
  int rc = voxel_downsample_device(c, in.as<float4>(), n, nullptr, leaf, intensity_last, outb.as<float4>(), d_cnt, 5);
  if (rc) return rc;
  int *hc = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 3072);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hc, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  *n_out = hc[0];
  if (hc[0] > 0) MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_out, outb.p, sizeof(float4) * (size_t)hc[0], cudaMemcpyDeviceToHost, st));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(st));
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ frame
int mloam_frame_device(mloam_ctx_t *h, const mloam_point_t *d_cloud, int n, const int *d_scan_start, const int *d_scan_end, int n_scans,
                       const mloam_point_t *d_surf_map, int n_surf_map, const mloam_point_t *d_corner_map, int n_corner_map,
                       int rebuild_maps, const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  if (!h || !pose_init7 || !pose_out7 || n <= 0 || !d_cloud || !d_scan_start || !d_scan_end) return MLOAM_E_INVALID;
  cudaSetDevice(h->c.device);
  Ctx *c = &h->c;
  int rc = stage_next_sweep(c);
  if (rc) return rc;
  rc = frame_run(c, reinterpret_cast<const float4 *>(d_cloud), n, d_scan_start, d_scan_end, n_scans,
                 reinterpret_cast<const float4 *>(d_surf_map), n_surf_map, reinterpret_cast<const float4 *>(d_corner_map),
                 n_corner_map, rebuild_maps, pose_init7, pose_out7, stats);
  c->next_pending = false, c->next.set = false;
  return rc;
}

// Look-ahead: announce the sweep of the NEXT mloam_frame* call.  While the coming frame is matched and solved, that sweep is extracted
// and down-sampled on a side stream (in the reference the two stages run in different nodes, estimator -> lidar_mapper); the next
// call finds its features ready when it passes the same pointer (and sizes) — otherwise it extracts as usual.  One announcement is
// consumed by one frame; results are identical with or without it.
int mloam_frame_set_next_device(mloam_ctx_t *h, const mloam_point_t *d_cloud, int n, const int *d_scan_start, const int *d_scan_end, int n_scans) {
  if (!h) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  c->next = Ctx::NextSweep{};
  if (!d_cloud || n <= 0) return MLOAM_OK;  // withdraw
  if (!d_scan_start || !d_scan_end || n_scans <= 0 || n_scans > MLOAM_MAX_RINGS) return MLOAM_E_INVALID;
  c->next.set = true, c->next.host = false, c->next.key_ptr = d_cloud, c->next.d_cloud = reinterpret_cast<const float4 *>(d_cloud);
  c->next.d_scan_start = d_scan_start, c->next.d_scan_end = d_scan_end, c->next.n = n, c->next.n_scans = n_scans;
  return MLOAM_OK;
}
int mloam_frame_set_next(mloam_ctx_t *h, const mloam_point_t *h_cloud, int n, const int *h_scan_start, const int *h_scan_end, int n_scans) {
  if (!h) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  c->next = Ctx::NextSweep{};
  if (!h_cloud || n <= 0) return MLOAM_OK;  // withdraw
  if (!h_scan_start || !h_scan_end || n_scans <= 0 || n_scans > MLOAM_MAX_RINGS) return MLOAM_E_INVALID;
  c->next.set = true, c->next.host = true, c->next.key_ptr = h_cloud, c->next.n = n, c->next.n_scans = n_scans;
  c->next_host_ss = h_scan_start, c->next_host_se = h_scan_end;
  return MLOAM_OK;
}

int mloam_frame(mloam_ctx_t *h, const mloam_point_t *h_cloud, int n, const int *h_scan_start, const int *h_scan_end, int n_scans,
                const mloam_point_t *h_surf_map, int n_surf_map, const mloam_point_t *h_corner_map, int n_corner_map, int rebuild_maps,
                const double *pose_init7, double *pose_out7, mloam_solve_stats_t *stats) {
  if (!h || !pose_init7 || !pose_out7 || n <= 0 || !h_cloud || !h_scan_start || !h_scan_end || n_scans <= 0 || n_scans > MLOAM_MAX_RINGS)
    return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  cudaStream_t st = c->stream;
  DevBuf &in = c->scratch[0];
  MLOAM_CUDA_OK(c, in.reserve(sizeof(float4) * (size_t)n + 1024 + 8 * (size_t)n_scans));
  float4 *d_cloud = in.as<float4>();
  int *d_ss = reinterpret_cast<int *>(in.as<char>() + sizeof(float4) * (size_t)n + 256);
  int *d_se = d_ss + n_scans;
  // the sweep was announced with the previous frame and its features are ready (look-ahead): nothing to copy
  const bool have = c->prefetched.host && frame_has_prefetched(c, h_cloud, n, n_scans);
  if (!have) {
    int *pin = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + kPinnedScanInfo);
    std::memcpy(pin, h_scan_start, sizeof(int) * n_scans), std::memcpy(pin + MLOAM_MAX_RINGS, h_scan_end, sizeof(int) * n_scans);
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_ss, pin, sizeof(int) * n_scans, cudaMemcpyHostToDevice, st));
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_se, pin + MLOAM_MAX_RINGS, sizeof(int) * n_scans, cudaMemcpyHostToDevice, st));
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_cloud, h_cloud, sizeof(float4) * (size_t)n, cudaMemcpyHostToDevice, st));
  }
  {
    const int rc_next = stage_next_sweep(c);
    if (rc_next) return rc_next;
  }
  const float4 *d_sm = nullptr, *d_cm = nullptr;
  if (rebuild_maps) {
    if (!h_surf_map || !h_corner_map || n_surf_map < 0 || n_corner_map < 0) return MLOAM_E_INVALID;
    DevBuf &ms = c->scratch[1], &mc = c->scratch[2];
    MLOAM_CUDA_OK(c, ms.reserve(sizeof(float4) * (size_t)(n_surf_map + 1)));
    MLOAM_CUDA_OK(c, mc.reserve(sizeof(float4) * (size_t)(n_corner_map + 1)));
    // The submaps (16 B/point, ~8x the sweep) go up on the side stream so that the copy overlaps extraction and scan
    // down-sampling of the sweep; the map-build branch of frame_enqueue is ordered after ev_maps.
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(ms.p, h_surf_map, sizeof(float4) * (size_t)n_surf_map, cudaMemcpyHostToDevice, c->stream2));
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(mc.p, h_corner_map, sizeof(float4) * (size_t)n_corner_map, cudaMemcpyHostToDevice, c->stream2));
    MLOAM_CUDA_OK(c, cudaEventRecord(c->ev_maps, c->stream2));
    c->maps_pending = true;
    d_sm = ms.as<float4>(), d_cm = mc.as<float4>();
  }
  c->cloud_key = h_cloud;
  const int rc = frame_run(c, d_cloud, n, d_ss, d_se, n_scans, d_sm, n_surf_map, d_cm, n_corner_map, rebuild_maps, pose_init7, pose_out7, stats);
  c->cloud_key = nullptr;
  c->maps_pending = false, c->next_pending = false, c->next.set = false;
  return rc;
}

int mloam_set_lidars(mloam_ctx_t *h, int n_lidars, const double *ext7) {
  if (!h || n_lidars < 1 || n_lidars > MLOAM_MAX_LIDARS || (n_lidars > 1 && !ext7)) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  c->n_lidars = n_lidars;
  c->prefetched.valid = false;  // look-ahead features were merged with the previous extrinsics
  c->lidar_merge = ext7 != nullptr;  // also for ONE LiDAR with an extrinsic: same float transform + laser id as in a rig
  for (int l = 0; l < n_lidars; l++)
    for (int k = 0; k < 7; k++) c->lidar_ext[l][k] = ext7 ? ext7[7 * l + k] : (k == 6 ? 1.0 : 0.0);
  return MLOAM_OK;
}

int mloam_set_extrinsic(mloam_ctx_t *h, const double *ext7) {
  if (!h) return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  c->has_ext = ext7 != nullptr;
  c->prefetched.valid = false;
  for (int k = 0; k < 7; k++) c->ext[k] = ext7 ? ext7[k] : (k == 6 ? 1.0 : 0.0);
  return MLOAM_OK;
}

}  // extern "C"
