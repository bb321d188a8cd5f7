// ctx.h — host-side context behind the C ABI (include/mloam_b200.h) and the kernel launchers.
#pragma once
#include <cuda_runtime.h>
#include <map>
#include <string>
#include <vector>

#include "../../include/mloam_b200.h"
#include "common.cuh"

namespace mloam {

// Bumped whenever a device buffer is (re)allocated: captured CUDA graphs hold raw pointers and are re-captured
// when the epoch they were recorded in is over.
inline unsigned long long &alloc_epoch() {
  static unsigned long long e = 0;
  return e;
}

// Input / output of the per-feature line / plane fit (match_fit.cuh)
struct FitSet {
  const float4 *sorted;  // MapView::sorted of the set's map
  const float4 *pts;
  int n;
  const int *d_n;
  const int *pos;        // n * K from k_match_knn
  unsigned char *valid;  // out
  float *coeff;          // out: n * 6
  int *nn;               // out (nullable): n * K original map indices
  int is_plane;
  const unsigned char *changed;  // nullable: 0 -> same neighbours as the previous iteration, valid/coeff already hold the fit
};
// A fit whose launch the matcher left to the first evaluation of the solve (k_linearize pass 0): filled by
// match_pair_device, handed by the caller to the linearize_device that begins the solve
struct PendingFit {
  FitSet set[2];
  int K = 0;  // 0: nothing pending
  float min_plane_dis = 0.f;
  int check_fov = 0;
};

// Grow-only device buffer (cudaMalloc only when capacity is exceeded; steady-state frames allocate nothing).
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    size_t want = bytes + bytes / 4 + 256;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    alloc_epoch()++;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T *as() const {
    return reinterpret_cast<T *>(p);
  }
};

#define MLOAM_MAX_RINGS 1024  // rings of one (possibly multi-LiDAR) extraction
#define MLOAM_MAX_LIDARS 16

constexpr size_t kMapStatsOffset = 16384;  // pinned: 64 B per map slot, the GridHdr head of the slot's last build (auto cell)

struct MapStorage {
  DevBuf sorted, orig, cells, rank_of, tile_sums, hdr;
  unsigned capacity = 0;  // cells the dense grid may use (4 B each)
  int m = 0;
  float cell = 0.f;       // requested cell edge of the last build (the device may have coarsened it: GridHdr::level)
  float auto_cell = 0.25f;  // map_cell <= 0: cell edge picked from the occupancy statistics of the previous build
  bool built = false;
  MapView view() const {
    MapView v;
    v.sorted = sorted.as<float4>();
    v.orig = orig.as<float4>();
    v.cell_start = cells.as<unsigned>();
    v.hdr = hdr.as<GridHdr>();
    v.m = m;
    return v;
  }
  // Sticky auto cell: a cell edge that gives a few points per occupied cell lets the 3x3x3 neighbourhood of a query
  // hold its K neighbours (knn.cuh ring 1).  Decided from the header the previous build of this slot copied to pinned
  // memory (possibly one build stale — it only steers speed, never results).  Power-of-two edges only.
  float auto_cell_pick(const void *pinned, int slot) {
    if (built && pinned) {
      const GridHdr *h = reinterpret_cast<const GridHdr *>(reinterpret_cast<const char *>(pinned) + kMapStatsOffset + 64 * slot);
      if (h->n_occupied > 0 && h->n_sorted > 0 && h->cell > 0.f) {
        const float avg = (float)h->n_sorted / (float)h->n_occupied;
        float cur = h->cell;
        if (avg < 2.5f && cur < 1.0f) cur *= 2.0f;
        else if (avg > 40.0f && cur > 0.125f) cur *= 0.5f;
        auto_cell = cur;
      }
    }
    return auto_cell;
  }
};

constexpr size_t kPinnedScanInfo = 32768, kPinnedScanInfoNext = 40960;  // 2 x MLOAM_MAX_RINGS ints each inside Ctx::pinned (ScanInfo staging of mloam_frame / of the announced sweep)
constexpr size_t kKnnPathStatsOffset = 3072;  // 64 B of matcher counters inside Ctx::scratch[7] (zeroed at creation / profile reset)

struct ProfSlot {
  double ms = 0;
  long long launches = 0;
};

// Parameters the kernels need, flattened from mloam_params_t.
struct MatchCfg {
  float min_match_sq_dis, min_plane_dis;
  int n_neigh, check_fov;
};

struct Ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = true;
  cudaStream_t stream2 = nullptr;        // side stream: submap upload + build run concurrently with extraction
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  cudaStream_t stream3 = nullptr;        // side stream: corner-scan voxel filter next to the surf-scan one
  cudaEvent_t ev_fork3 = nullptr, ev_join3 = nullptr;
  cudaEvent_t ev_maps = nullptr;         // recorded on stream2 after the host API's submap H2D copies
  bool maps_pending = false;             // the map-build branch must wait on ev_maps (external to a captured graph)
  mloam_params_t params;
  std::string err;
  long long launches = 0;

  MapStorage maps[MLOAM_NUM_MAPS];

  // scan features (device copies when the caller passes host buffers)
  DevBuf scan_pts[4];             // [0] corner, [1] surf
  DevBuf feat_valid[4];           // unsigned char per query
  DevBuf feat_coeff[4];           // float[6] per query
  DevBuf feat_nn[4];              // int[n_neigh] per query (optional)
  DevBuf knn_pos[4];              // int[n_neigh] per query: neighbour positions handed from k_match_knn to k_match_fit
  DevBuf knn_changed[4];          // unsigned char per query: neighbour list differs from the previous iteration's
  DevBuf knn_anchor[4];           // float4 per query: position of its last real search + tolerated displacement
  DevBuf gf_work[2];              // good-feature selection scratch per set (Jacobian rows, pool tree, mask, ...)
  DevBuf knn_heavy[4];            // 2 x unsigned char per query: "needed a real search" verdicts of the last two launches
  DevBuf knn_heavy_list;          // 3 rotating counters + 2 lists of feature indices that needed a real search (match_kernels.cu HeavyQ)
  int knn_rot = 0;                // launch ordinal inside the current solve (rotation of the heavy lists / counters)
  int knn_parity = 0;             // which half of knn_heavy the next seeded launch reads
  DevBuf partials;                // per-block packed normal equations
  DevBuf lm_state;                // LMState
  void *ticket_zeroed_for = nullptr;  // partials allocation whose last-block ticket has been zeroed
  DevBuf scratch[10];             // general scratch (knn outputs, factor batches, extraction, voxel)
  void *pinned = nullptr;         // pinned host staging (LMState mirror + small results)
  size_t pinned_cap = 0;

  // profiling with CUDA events on `stream`
  bool prof_on = false;
  std::map<std::string, ProfSlot> prof;
  struct PendingEvt {
    std::string name;
    cudaEvent_t a, b;
  };
  std::vector<PendingEvt> pending;
  std::vector<cudaEvent_t> evt_pool;

  // NCCL (multi-GPU); opaque here
  void *d_ring_stage = nullptr;     // RingStage[n_scans] of the last extraction (extract_kernels.cu)
  int *d_ring_cnt = nullptr;        // per-ring less-flat centroid counts of the last extraction
  int *d_extract_status = nullptr;  // device flag of the last extraction (1: ring window overflow / bad ScanInfo)
  // CUDA-graph cache of whole frames (pipeline.cu frame_run)
  struct ScanRef {
    const float4 *surf;
    int n_surf;            // count or upper bound
    const int *d_n_surf;   // nullable device-side count
    const float4 *corner;
    int n_corner;
    const int *d_n_corner;
    const double *sinfo_surf, *sinfo_corner;  // nullable per-feature sqrt_info (uncertainty-aware mapping)
  };
  // Sweep look-ahead (mloam_frame_set_next*): while frame k is matched and solved, the features of sweep k+1 are extracted and
  // down-sampled on a side stream into the other half of a double buffer — the reference runs the two stages in different nodes
  // (estimator -> lidar_mapper), so they overlap there too.  `Features` describes one half.
  struct Features {
    bool valid = false;
    bool host = false;          // key_ptr is a host pointer (mloam_frame) / a device pointer (mloam_frame_device)
    const void *key_ptr = nullptr;
    int n = 0, n_scans = 0, parity = 0;
    ScanRef S{};
  };
  struct NextSweep {
    bool set = false, host = false;
    const void *key_ptr = nullptr;      // what the caller will pass as the cloud of the next frame
    const float4 *d_cloud = nullptr;    // where the sweep is (or will be, after the pending H2D) on the device
    const int *d_scan_start = nullptr, *d_scan_end = nullptr;
    int n = 0, n_scans = 0;
  };
  Features prefetched;             // features of the sweep announced with the previous frame, ready when that frame returned
  NextSweep next;                  // announced for the frame being enqueued (consumed by it)
  const void *cloud_key = nullptr; // mloam_frame: the HOST pointer of the sweep being processed (look-ahead matches on it)
  const int *next_host_ss = nullptr, *next_host_se = nullptr;  // ScanInfo of a sweep announced from host memory
  bool next_pending = false;       // its H2D copy was enqueued on stream4 outside of any capture (ev_next)
  int frame_parity = 0;
  int use_lookahead = 1;           // MLOAM_LOOKAHEAD=0: announcements are ignored
  bool stamp_mute = false;
  DevBuf frame_main, frame_alt, next_in;  // the two halves of the frame feature double buffer; the announced sweep's staging
  cudaStream_t stream4 = nullptr, stream5 = nullptr;  // look-ahead extraction and its corner-voxel fork
  cudaEvent_t ev_fork4 = nullptr, ev_join4 = nullptr, ev_fork5 = nullptr, ev_join5 = nullptr, ev_next = nullptr;
  struct GraphEntry {
    unsigned long long key = 0, epoch = 0;
    cudaGraphExec_t exec = nullptr;
    int launches = 0, seen = 0, s2m_ran = 0;
    ScanRef S{};
    Features prefetched_out{};     // what the frame leaves in Ctx::prefetched
  };
  std::vector<GraphEntry> graphs;
  bool smem_opt_in_gf = false;     // k_gf_select's 200 KB pool
  bool smem_opt_in[3] = {false, false, false};  // >48 KB dynamic shared memory enabled for k_voxel_small / k_ring_pick / k_ring_voxel
  long long graph_capture_failures = 0;  // frames that fell back to the stream path because their capture failed (mloam_profile_get "graph_capture_failures")
  int use_graphs = 1;
  unsigned knn_tma_min = 8;        // kNN staging: runs of >= this many points use TMA bulk copies, shorter ones 16 B loads (MLOAM_KNN_TMA_MIN)
  DevBuf knn_trace;                // MLOAM_KNN_TRACE=1: 4 words per query of the last k_match_knn launch (diagnosis, tools/knn_micro.py)
  bool knn_trace_on = false;
  // MLOAM_STAMP=1 (diagnosis, tools/stamp_frame.py): one-thread kernels that write %globaltimer between the stages of a frame, so that
  // the stage times of a GRAPH REPLAY can be read (the event scopes of mloam_profile_enable force the stream path and add launch gaps)
  bool stamp_on = false;
  DevBuf stamps;
  int stamp_n = 0;
  std::vector<std::string> stamp_labels;
  int knn_min_blocks = 4;          // k_match_knn variant: resident CTAs per SM it is compiled for (MLOAM_KNN_MB = 2 | 3 | 4)
  int use_seeds = 1;               // seed the kNN of re-association iterations > 0 with the previous neighbour lists
  int s2m_ran = 0;
  int fuse_iter = 1;               // scan2map: fit inside the first evaluation + both evaluations of an LM iteration in ONE launch
                                   // (grid barrier between them); MLOAM_FUSE_ITER=0 restores the three launches
  bool lidar_merge = false;        // mloam_set_lidars was given extrinsics: features go through the rig merge (also for one LiDAR)
  int n_lidars = 1;                // LiDARs batched into one frame of this context (mloam_set_lidars)
  double lidar_ext[MLOAM_MAX_LIDARS][7];  // their sensor -> base extrinsics
  bool has_ext = false;            // sensor -> base extrinsic applied to extracted features (frame path)
  double ext[7] = {0, 0, 0, 0, 0, 0, 1};
  void *nccl_comm = nullptr;
  int nranks = 1, rank = 0;
  // peer-memory exchange of the packed normal equations (comm.cu, solve_kernels.cu lm_tail): every rank's exchange
  // buffer is mapped into every other rank through CUDA IPC; p2p_on replaces the NCCL all-reduce + two extra launches
  // by stores / polls over NVLink inside the k_linearize tail
  void *p2p_local = nullptr;
  void *p2p_peer[MLOAM_P2P_MAX_RANKS] = {nullptr};
  void *p2p_view = nullptr;        // device copy of the P2PView the kernels read
  bool p2p_on = false;
};

// RAII-less helper: bracket a kernel (or a few) with events when profiling is on.
struct ProfScope {
  Ctx *c;
  cudaEvent_t a = nullptr, b = nullptr;
  const char *name;
  ProfScope(Ctx *ctx, const char *nm);
  ~ProfScope();
};
void prof_collect(Ctx *c);

#define MLOAM_CUDA_OK(ctx, expr)                                                                      \
  do {                                                                                                \
    cudaError_t _e = (expr);                                                                          \
    if (_e != cudaSuccess) {                                                                          \
      (ctx)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                                \
      return MLOAM_E_CUDA;                                                                            \
    }                                                                                                 \
  } while (0)

// ---------------------------------------------------------------- launchers (one per .cu)
// map_kernels.cu
int map_build_device(Ctx *c, int slot, const float4 *d_pts, int m, float cell);
int knn_device(Ctx *c, int slot, const float4 *d_q, int nq, const double *d_pose7_or_null, int k, float max_sqdist,
               int *d_idx, float *d_sqd);
// type 'c' / 's'.  d_pose7 device pointer to 7 doubles.  Outputs: valid[n], coeff[n*6] float, nn[n*n_neigh] (nullable)
// d_n (nullable): device-side feature count, n is then the launch upper bound.
int match_from_map_device(Ctx *c, int slot, int type, const float4 *d_pts, int n, const int *d_n, const double *d_pose7,
                          const MatchCfg &cfg, unsigned char *d_valid, float *d_coeff, int *d_nn);

// match_kernels.cu: one kNN launch + one fit launch over up to two feature sets
struct MatchJob {
  int slot;                 // map slot
  int type;                 // 'c' (line fit) | 's' (plane fit)
  const float4 *pts;        // sensor-frame features
  int n;                    // count / upper bound
  const int *d_n;           // nullable device-side count
  unsigned char *valid;     // out
  float *coeff;             // out, n * 6
  int *nn;                  // out, nullable, n * n_neigh original indices
  int seeded;               // 1: same features against the same map as the previous call with this job index — its neighbour
                            // lists (Ctx::knn_pos) seed the search and unchanged lists keep their fit
};
// buf_base: which pair of the context's per-set buffers (knn_pos / knn_anchor / ...) the jobs use: 0 (sets 0, 1) or 2 (sets 2, 3)
// defer (nullable): when no job asks for neighbour lists, skip the fit launch and describe the fit in *defer for the
// linearize_device that begins the solve; otherwise the fit is launched here and defer->K is 0
int match_pair_device(Ctx *c, const MatchJob *jobs, int n_jobs, const double *d_pose7, const MatchCfg &cfg, int buf_base = 0,
                      PendingFit *defer = nullptr);

// track_kernels.cu
int match_from_scan_device(Ctx *c, int slot, int type, const float4 *d_pts, int n, const double *d_pose7, unsigned char *d_valid,
                           float *d_coeff, int *d_nn3);
int track_cloud_device(Ctx *c, const float4 *d_prev_less_sharp, int n_pls, const float4 *d_prev_less_flat, int n_plf,
                       const float4 *d_cur_sharp, int n_cs, const float4 *d_cur_flat, int n_cf, const double *pose_ini7,
                       double *pose_out7, mloam_solve_stats_t *stats);

// solve_kernels.cu
struct FeatSet {
  const float4 *pts;           // sensor-frame points
  const unsigned char *valid;
  const float *coeff;          // float[6]
  int n;                       // count, or launch upper bound when d_n is set
  int is_plane;                // 1: LidarMapPlaneNormFactor, 0: LidarMapEdgeFactor
  const int *d_n;              // nullable device-side count
  const double *sinfo;         // nullable per-feature sqrt_info (with_ua: lidar_map_factor.hpp:34,41 on the point's covariance)
  const unsigned char *mask;   // nullable: only features with mask[i] != 0 enter (good-feature selection)
};
// Settings fixed for the length of one solve
struct SolveCfg {
  double sqrt_info;  // weight of a feature without a per-feature sqrt_info
  double huber_a;    // HuberLoss scale
  double eig_thre;   // evalDegenracy: directions of H with an eigenvalue below it are not updated (0: no test)
  bool collective;   // every rank runs this solve in lock-step: the normal equations are summed over the ranks
};
// What linearize_device evaluates and which LM step follows (the value is lm_tail's mode)
enum LinEval {
  kEvalAtPose = 0,     // at d_pose7; no step (the packed normal equations go to d_out30 if non-null)
  kEvalBegin = 1,      // at LMState::x; begins the Solve
  kEvalCandidate = 2,  // at LMState::xc; accepts or rejects the candidate (nothing happens once the Solve is done)
};
// Accumulate loss-corrected normal equations of both feature sets into c->partials, then run the LM step of `eval`.
// fit (nullable, kEvalBegin): the matcher's deferred fit, run by the evaluation at x.  two_pass: also evaluate the
// candidate of the step in the same launch when the tail runs fused; *two_pass_done (nullable) tells whether it did.
int linearize_device(Ctx *c, const FeatSet *sets, int n_sets, const SolveCfg &cfg, LinEval eval, const double *d_pose7 = nullptr,
                     double *d_out30 = nullptr, const PendingFit *fit = nullptr, bool two_pass = false, bool *two_pass_done = nullptr);
// min_corr: a Solve with fewer matched features is skipped
int lm_init_state(Ctx *c, const double *pose7_host, int max_inner, int min_corr);
void eig_report_host(const double *H36, double *w6);  // ascending eigenvalues of a symmetric 6x6 (host side)
int factor_evaluate_device(Ctx *c, int kind, int n, const double *d_points, const double *d_coeffs, const double *d_sqrt_info,
                           const double *d_params, double *d_res, double *d_jac);

// in place: p <- T * p for the first min(n, *d_n) points (pointAssociateToMap, utility.h:103-117); d_pose7 on device
int transform_points_device(Ctx *c, float4 *d_pts, int n, const int *d_n, const double *d_pose7);

// gf_kernels.cu: good-feature selection of one matched feature set on the device (goodFeatureMatching inside
// scan2MapOptimization): Jacobian rows + selection, result as a 0/1 mask over the features (set index t: 0 corner, 1 surf)
int gf_select_set_device(Ctx *c, int t, const FeatSet &fs, const double *d_pose7, double default_sinfo, int method, double gf_ratio,
                         unsigned long long seed, unsigned char **d_mask_out);

// uct_kernels.cu: per-point sqrt_info from PointIWithCov::cov_vec (float[6] per point)
int sqrt_info_device(Ctx *c, const float *d_cov6, int n, double *d_sinfo);

// comm.cu: in-place sum over ranks on the context stream (no-op without a communicator)
int comm_allreduce_doubles(Ctx *c, double *d_buf, int count);

// extract_kernels.cu
struct ExtractOut {
  float4 *sharp, *less_sharp, *flat, *less_flat;  // device buffers, capacity n each
  int *counts;                                     // device int[4]
};
int extract_device(Ctx *c, const float4 *d_cloud, int n, const int *d_scan_start, const int *d_scan_end, int n_scans,
                   ExtractOut out, float *d_curv_or_null, int *d_label_or_null);
// in place: segment l of d_pts (points [d_off[l], d_off[l + 1])) <- float 3x4 matrix l times the point, intensity kept
void stamp(Ctx *c, const char *label);  // api.cu
int project_cloud_device(Ctx *c, const float4 *d_in, int n, int vertical_scans, int horizon_scans, double roi_range, float4 *d_out,
                         int *d_scan_start, int *d_scan_end, int *d_n_out);
int transform_segments_device(Ctx *c, float4 *d_pts, int n, const int *d_off, int n_seg, const float *d_mat12);
// VoxelGridCovarianceMLOAM<PointIWithCov>::filter: covariance-weighted merge per voxel (cov6 + trace per point in and out)
int voxel_downsample_cov_device(Ctx *c, const float4 *d_in, const float *d_cov6, const float *d_trace, int n, const int *d_n_in, float leaf,
                                float trace_threshold, float4 *d_out, float *d_cov6_out, float *d_trace_out, int *d_n_out, int work_slot = 5);
// exclusive scan of ints on the context stream (extract_kernels.cu); tmp holds ceil(n / 2048) ints
void scan_exclusive(Ctx *c, const int *d_in, int *d_out, int n, int *d_tmp, int *d_total);
// After a batched extraction over the concatenated sweeps of n_lidars LiDARs: move the less-sharp / less-flat features of LiDAR l into
// the base frame with its float 3x4 extrinsic d_ext12[l] and set intensity = l (transformCloudFeature, visualization.cpp:40-52).
// d_off: scratch for 2 x (n_lidars + 1) ints.
int merge_lidars_device(Ctx *c, ExtractOut out, int n_cap_less, int n_cap_lflat, int n_lidars, int rings_per_lidar, const float *d_ext12,
                        int *d_off);
// d_n_in (nullable): device-side input count (n is then the upper bound the kernels are sized for).
int voxel_downsample_device(Ctx *c, const float4 *d_in, int n, const int *d_n_in, float leaf, int intensity_last, float4 *d_out,
                            int *d_n_out, int work_slot = 5);

}  // namespace mloam

struct mloam_ctx {
  mloam::Ctx c;
};
