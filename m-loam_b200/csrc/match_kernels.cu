// match_kernels.cu — FeatureExtract::matchCornerFromMap / matchSurfFromMap (feature_extract.hpp:378-643;
// per-point forms :645-883) as two kernels:
//
//   k_match_knn  one WARP per feature: pointAssociateToMap + exact K-nearest search in the dense voxel grid
//                (knn.cuh) + the distance gate sqdist[K-1] < MIN_MATCH_SQ_DIS.  Corner and surf features share one
//                launch; the features that needed a real search in the previous iteration are scheduled first (HeavyQ),
//                so long queries — features in sparse regions — do not form the tail of the launch.  Output: K neighbour positions per feature (20 B).
//   k_match_fit  one THREAD per feature: gathers the K neighbours (5 x 16 B), fits the line (mean + scatter +
//                3x3 eigen) or the plane (5x3 column-pivoted QR), applies the lambda / plane-distance / FOV gates
//                and writes valid + coefficients.  Running the fit one-thread-per-feature instead of redundantly
//                in all 32 lanes of the search warp removes ~1/3 of the matcher's warp instructions and halves its
//                register footprint.  The per-feature routine lives in match_fit.cuh; scan2map without good-feature
//                selection defers it into the first evaluation of the solve (k_linearize), so that a GN iteration is
//                two launches.
#include <cstdlib>

#include "ctx.h"
#include "fit.cuh"
#include "knn.cuh"
#include "match_fit.cuh"

namespace mloam {

constexpr int MWARPS = 8;  // warps per CTA in k_match_knn

struct KnnSet {
  MapView map;
  const float4 *pts;   // sensor-frame features
  int n;               // count, or launch upper bound when d_n is set
  const int *d_n;      // nullable device-side count
  int *pos;            // out: n * K positions into map.sorted (-1: gate failed); in: the previous result when seeded
  int seeded;          // pos holds this set's result of the previous re-association iteration on the SAME map
  unsigned char *changed;  // out (nullable): 1 when the neighbour list differs from the seed (or there was none)
  float4 *anchor;      // per feature: map-frame position of its last real search + the displacement it tolerates
  const unsigned char *heavy_in;  // nullable: 1 where the previous launch had to search (ball / blind) — those go first
  unsigned char *heavy_out;       // this launch's verdict, for the next one
};

// Scheduling of the searches inside a launch.  Queries differ by 10x in cost (a kept neighbour list: ~2.5k cycles, a
// real search: 10-30k) and a launch is only as fast as its slowest warp, so the few features that needed a real search
// in the previous re-association iteration are listed (atomic append — a few dozen per launch, not one atomic per
// query: 20k increments of ONE address cost ~1 ns each at the L2 and were the longest part of the launch) and taken
// first, one per warp; everything else is a static stride.  cnt[3] rotates: a launch reads cnt_in, appends to cnt_out
// and clears cnt_zero for the launch after the next.
struct HeavyQ {
  const int *list_in;   // nullable (first iteration): global feature indices (corner set first)
  const int *cnt_in;
  int *list_out;
  int *cnt_out;
  int *cnt_zero;
};

// MB: resident CTAs per SM the kernel is compiled for (register budget 65536 / (256 * MB)).  The search is a chain of
// dependent warp-wide operations (prefix loads -> point loads -> REDUX / ballot / shuffle rounds): issue slots are only
// filled when many warps are resident, so the default trades a few spilled registers for twice the warps.
template <int K, int MB>
__global__ void __launch_bounds__(MWARPS * 32, MB)
    k_match_knn(KnnSet a, KnnSet b, const double *__restrict__ pose7, float min_match_sq_dis, HeavyQ hq,
                unsigned *__restrict__ path_stats, unsigned tma_min, unsigned *__restrict__ trace) {
  __shared__ KnnSmem ksm[MWARPS];
  const int lane = threadIdx.x & 31;
  KnnSmem &ks = ksm[threadIdx.x >> 5];
  unsigned long long t_enter = 0ull;
  if (trace) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_enter));
  knn_smem_init(ks, lane, tma_min);
  __shared__ GridP s_grid[2];
  __shared__ PoseD s_pose;
  if (threadIdx.x == 0) s_grid[0] = load_grid(a.map), s_grid[1] = load_grid(b.map), s_pose = pose_from_param(pose7);
  __syncthreads();
  const int na = a.d_n ? min(a.n, *a.d_n) : a.n;
  const int nb = b.d_n ? min(b.n, *b.d_n) : b.n;
  const int n = na + nb;
  // Schedule: first the listed heavy features of the previous launch (one per warp), then a static stride over the rest.
  const int gw = blockIdx.x * MWARPS + (threadIdx.x >> 5), n_warps = gridDim.x * MWARPS;
  if (hq.cnt_zero && gw == 0 && lane == 0) *hq.cnt_zero = 0;
  const bool listed = hq.list_in != nullptr;
  const int n_heavy = listed ? min(__ldg(hq.cnt_in), n) : 0;
  const int it_a = n_heavy > gw ? (n_heavy - gw + n_warps - 1) / n_warps : 0;
  const int it_b = n > gw ? (n - gw + n_warps - 1) / n_warps : 0;
#pragma unroll 1
  for (int it = 0; it < it_a + it_b; it++) {
    int i;
    if (it < it_a) {
      i = __ldg(hq.list_in + gw + it * n_warps);
    } else {
      i = gw + (it - it_a) * n_warps;
      if (listed) {  // listed ones have been done above
        const unsigned char *hin = i < na ? a.heavy_in : b.heavy_in;
        if (hin && hin[i < na ? i : i - na]) continue;
      }
    }
    const float4 p = __ldg(i < na ? a.pts + i : b.pts + (i - na));
    const bool in_a = i < na;
    const int j = in_a ? i : i - na;
    const long long t_query = (path_stats || trace) ? clock64() : 0ll;
    int path = 3;  // 0 keep (matched), 1 keep (rejected), 2 ball, 3 blind
    const float3 sel = associate(s_pose, p.x, p.y, p.z);  // pointAssociateToMap, utility.h:103-117
    const GridP &g = s_grid[in_a ? 0 : 1];
    Best best;  // selection width K + 1: lane K holds the nearest scanned point outside the K-set (feeds the anchor's slack)
    int *const pos_out = (in_a ? a.pos : b.pos) + (size_t)j * K;
    const int seeded = in_a ? a.seeded : b.seeded;
    unsigned char *const changed = in_a ? a.changed : b.changed;
    float4 *const anchor = (in_a ? a.anchor : b.anchor) + j;
    // Temporal coherence between re-association iterations (all three shortcuts are exact, see knn.cuh):
    //   keep    the query moved less than the anchor's slack since its last real search: the K-set cannot have
    //           changed, only its order — recompute the K distances and re-rank (no cell probes, no scan)
    //   ball    otherwise the previous neighbours bound the search ball around the moved query
    //   blind   no previous neighbours (or a ball of more than 32 cells)
    int prev = -1, newpos = -1;
    bool done = false;
    float r2 = 3.0e38f;
    if (seeded) {
      if (lane < K) prev = pos_out[lane];
      const float4 an = *anchor;
      const float mx = sel.x - an.x, my = sel.y - an.y, mz = sel.z - an.z;
      const float moved = sqrtf(mx * mx + my * my + mz * mz);
      const bool within = an.w > 0.0f && moved + 2e-5f < an.w;
      if (__shfl_sync(MLOAM_FULL_MASK, prev, 0) < 0) {
        // rejected last time with the K-th neighbour at least radius + an.w away from the anchor: still rejected
        if (within) {
          done = true;
          path = 1;
        }
      } else {
        unsigned long long key = MLOAM_KEY_NONE;
        unsigned d2b = 0u;
        if (lane < K) {
          const float4 v = __ldg((in_a ? a.map.sorted : b.map.sorted) + prev);
          const float ex = v.x - sel.x, ey = v.y - sel.y, ez = v.z - sel.z;
          d2b = __float_as_uint(ex * ex + ey * ey + ez * ez);  // non-negative floats order like their bit patterns
          key = ((unsigned long long)d2b << 32) | (unsigned)__float_as_int(v.w);
        }
        r2 = __uint_as_float(__reduce_max_sync(MLOAM_FULL_MASK, d2b));
        if (within) {
          int rank = 0;
#pragma unroll
          for (int k = 0; k < K; k++) {
            const unsigned long long other = __shfl_sync(MLOAM_FULL_MASK, key, k);
            if (other < key) rank++;
          }
#pragma unroll
          for (int k = 0; k < K; k++) {
            const int rk = __shfl_sync(MLOAM_FULL_MASK, rank, k), pk = __shfl_sync(MLOAM_FULL_MASK, prev, k);
            if (rk == lane) newpos = pk;
          }
          if (!(r2 < min_match_sq_dis)) {  // :407,571,667,814 — the slack of a match says nothing about a rejection
            newpos = -1;
            if (lane == 0) *anchor = make_float4(sel.x, sel.y, sel.z, 0.0f);
          }
          done = true;
          path = 0;
        }
      }
    }
    if (!done) {
      float explored = 0.0f;
      bool found = false;
      if (r2 < min_match_sq_dis)
        found = warp_knn_seeded<K, K + 1>(in_a ? a.map : b.map, g, ks, sel.x, sel.y, sel.z, r2, 0.1f * g.cell,
                                             lane, best, &explored);
      if (!found) {
        KnnDbg dbg = {0, 0, 0, 0, 0, 0};
        const long long t_blind = (path_stats || trace) ? clock64() : 0ll;
        warp_knn<K, true, K + 1>(in_a ? a.map : b.map, g, ks, sel.x, sel.y, sel.z, min_match_sq_dis, lane, best, &explored, 0.05f,
                                 (path_stats || trace) ? &dbg : nullptr);
        if (trace && lane == 0) {
          unsigned *tr = trace + 4 * (size_t)((in_a ? 0 : na) + j);
          tr[1] = (unsigned)dbg.t_ring1, tr[2] = (unsigned)dbg.t_ball, tr[3] = ((unsigned)dbg.ring1_pts << 20) | ((unsigned)(dbg.ball_pts & 0xfff) << 8) | (unsigned)(dbg.ball_steps & 0xff);
        }
        if (path_stats && lane == 0) {
          unsigned long long *q = reinterpret_cast<unsigned long long *>(path_stats + 24);
          atomicAdd(q + 0, 0ull), atomicAdd(q + 1, (unsigned long long)dbg.t_ring1);
          atomicAdd(q + 2, (unsigned long long)dbg.t_ball), atomicAdd(q + 3, (unsigned long long)dbg.ring1_pts);
          atomicAdd(q + 4, (unsigned long long)dbg.ball_pts), atomicAdd(q + 5, (unsigned long long)dbg.ball_steps);
          atomicAdd(q + 6, (unsigned long long)dbg.ball_rows), atomicAdd(q + 7, dbg.t_ball ? 1ull : 0ull);
          const long long dt_blind = clock64() - t_blind;
          if (dt_blind > 90000) {  // a record of one very slow blind query (benign race: any of them will do)
            long long *rec = reinterpret_cast<long long *>(path_stats + 40);
            rec[0] = dt_blind, rec[1] = 0, rec[2] = dbg.t_ring1, rec[3] = dbg.t_ball, rec[4] = dbg.ring1_pts;
            rec[5] = dbg.ball_pts, rec[6] = dbg.ball_rows, rec[7] = dbg.ball_steps, rec[8] = (in_a ? 0 : 1) * 1000000 + j;
            rec[9] = (long long)(t_blind - t_query);
          }
        }
      }
      path = found ? 2 : 3;
      const unsigned long long kK = best_key(best, K - 1), kK1 = best_key(best, K);
      const bool ok = kK != MLOAM_KEY_NONE && key_d2(kK) < min_match_sq_dis;  // :407,571,667,814
      newpos = (ok && lane < K) ? best.pos : -1;
      // anchor: K-set members are within rK of this position, everything else at least lb away
      float slack = 0.0f;
      if (ok) {
        const float rK = sqrtf(key_d2(kK));
        float lb = explored;
        if (kK1 != MLOAM_KEY_NONE) lb = fminf(lb, sqrtf(key_d2(kK1)));
        slack = 0.5f * (lb - rK) - 2e-5f;
      } else {
        // rejected: the K-th neighbour is at least lbK away; while the query stays within lbK - radius of here the
        // verdict stands
        float lbK = explored;
        if (kK != MLOAM_KEY_NONE) lbK = fminf(lbK, sqrtf(key_d2(kK)));
        slack = lbK - sqrtf(min_match_sq_dis) - 2e-5f;
      }
      if (lane == 0) *anchor = make_float4(sel.x, sel.y, sel.z, slack);
    }
    if (lane < K) pos_out[lane] = newpos;
    if (changed) {
      const bool diff = __any_sync(MLOAM_FULL_MASK, lane < K && (!seeded || newpos != prev));
      if (lane == 0) changed[j] = diff ? 1 : 0;
    }
    if (path_stats && lane == 0) {  // stage profiling: queries and SM cycles per search path, slowest single query
      const unsigned long long dt = (unsigned long long)(clock64() - t_query);
      atomicAdd(path_stats + path, 1u);
      atomicAdd(reinterpret_cast<unsigned long long *>(path_stats + 8) + path, dt);
      atomicMax(path_stats + 4, (unsigned)(dt > 0xffffffffull ? 0xffffffffull : dt));
      if (dt > 32768ull) atomicAdd(path_stats + 5, 1u);
      if (dt > 65536ull) atomicAdd(path_stats + 6, 1u);
      // slowest query: cycles << 32 | path << 30 | set << 29 | feature index
      atomicMax(reinterpret_cast<unsigned long long *>(path_stats + 16),
                (dt << 32) | ((unsigned long long)path << 30) | ((unsigned long long)(in_a ? 0 : 1) << 29) | (unsigned)(j & 0x1fffffff));
    }
    if (trace && lane == 0) trace[4 * (size_t)((in_a ? 0 : na) + j)] = (unsigned)(clock64() - t_query) | ((unsigned)path << 30);
    unsigned char *const hout = in_a ? a.heavy_out : b.heavy_out;
    if (hout && lane == 0) {
      hout[j] = path >= 2 ? 1 : 0;
      if (path >= 2 && hq.list_out) hq.list_out[atomicAdd(hq.cnt_out, 1)] = i;
    }
  }
  if (trace && lane == 0) {  // per-warp timeline after the per-query words: [enter, first query, exit] in ns
    unsigned long long t_exit;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_exit));
    unsigned long long *w = reinterpret_cast<unsigned long long *>(trace + 4 * (size_t)(a.n + b.n + 1)) + 2 * (size_t)(blockIdx.x * MWARPS + (threadIdx.x >> 5));
    w[0] = t_enter, w[1] = t_exit;
  }
}

template <int K>
__global__ void __launch_bounds__(128) k_match_fit(FitSet a, FitSet b, const double *__restrict__ pose7, float min_plane_dis, int check_fov) {
  const int na = a.d_n ? min(a.n, *a.d_n) : a.n;
  const int nb = b.d_n ? min(b.n, *b.d_n) : b.n;
  const PoseD T = pose_from_param(pose7);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < na + nb; i += gridDim.x * blockDim.x) {
    if (i < na) fit_one<K>(a, i, T, min_plane_dis, check_fov);
    else fit_one<K>(b, i - na, T, min_plane_dis, check_fov);
  }
}

// ------------------------------------------------------------------------------------------------ launchers
// Match up to two feature sets (corner against MLOAM_MAP_CORNER-like slot, surf against a surf slot) in one
// kNN launch + one fit launch.  Sets with n == 0 are skipped.
int match_pair_device(Ctx *c, const MatchJob *jobs, int n_jobs, const double *d_pose7, const MatchCfg &cfg, int buf_base, PendingFit *defer) {
  if (defer) defer->K = 0;
  if (n_jobs < 1 || n_jobs > 2 || (buf_base != 0 && buf_base != 2)) {
    c->err = "match: 1 or 2 jobs";
    return MLOAM_E_INVALID;
  }
  if (cfg.n_neigh != 5 && cfg.n_neigh != 10) {
    c->err = "match_from_map: n_neigh must be 5 or 10";
    return MLOAM_E_INVALID;
  }
  const int K = cfg.n_neigh;
  KnnSet ks[2];
  FitSet fs[2];
  int n_upper = 0;
  bool flip = false;
  for (int t = 0; t < 2; t++) {
    KnnSet &k = ks[t];
    FitSet &f = fs[t];
    memset(&k, 0, sizeof(k));
    memset(&f, 0, sizeof(f));
    if (t >= n_jobs || jobs[t].n <= 0) continue;
    const MatchJob &J = jobs[t];
    if (J.slot < 0 || J.slot >= MLOAM_NUM_MAPS || !c->maps[J.slot].built) {
      c->err = "match_from_map: map slot not built";
      return MLOAM_E_STATE;
    }
    if (J.type != 'c' && J.type != 's') {
      c->err = "match_from_map: type must be 'c' or 's'";
      return MLOAM_E_INVALID;
    }
    DevBuf &pb = c->knn_pos[buf_base + t];
    MLOAM_CUDA_OK(c, pb.reserve(sizeof(int) * (size_t)K * (size_t)(J.n + 1)));
    k.map = c->maps[J.slot].view();
    DevBuf &cb = c->knn_changed[buf_base + t];
    MLOAM_CUDA_OK(c, cb.reserve((size_t)(J.n + 1)));
    k.pts = J.pts, k.n = J.n, k.d_n = J.d_n, k.pos = pb.as<int>();
    DevBuf &ab = c->knn_anchor[buf_base + t];
    MLOAM_CUDA_OK(c, ab.reserve(sizeof(float4) * (size_t)(J.n + 1)));
    k.seeded = J.seeded, k.changed = cb.as<unsigned char>(), k.anchor = ab.as<float4>();
    // search verdicts ("had to search") alternate between two halves from launch to launch: read the previous, write the next
    DevBuf &hb = c->knn_heavy[buf_base + t];
    const size_t half = ((size_t)J.n + 256) & ~(size_t)255;
    MLOAM_CUDA_OK(c, hb.reserve(2 * half));
    k.heavy_in = J.seeded ? hb.as<unsigned char>() + half * (size_t)c->knn_parity : nullptr;
    k.heavy_out = hb.as<unsigned char>() + half * (size_t)(J.seeded ? (c->knn_parity ^ 1) : c->knn_parity);
    flip = flip || J.seeded;
    f.changed = (J.seeded && !J.nn) ? cb.as<unsigned char>() : nullptr;
    f.sorted = k.map.sorted, f.pts = J.pts, f.n = J.n, f.d_n = J.d_n, f.pos = pb.as<int>();
    f.valid = J.valid, f.coeff = J.coeff, f.nn = J.nn, f.is_plane = J.type == 's' ? 1 : 0;
    n_upper += J.n;
  }
  if (n_upper <= 0) return MLOAM_OK;
  // heavy list of the launch: 2 lists x n_upper ints + 3 rotating counters (zeroed with the buffer, and again by the
  // non-seeded launch that starts a solve, where the rotation restarts)
  HeavyQ hq{nullptr, nullptr, nullptr, nullptr, nullptr};
  {
    DevBuf &hl = c->knn_heavy_list;
    const size_t ints = 2 * ((size_t)n_upper + 64) + 16;
    if (hl.cap < sizeof(int) * ints) {
      MLOAM_CUDA_OK(c, hl.reserve(sizeof(int) * ints));
      MLOAM_CUDA_OK(c, cudaMemsetAsync(hl.p, 0, hl.cap, c->stream));
    }
    int *cnt = hl.as<int>();                 // [0..2] counters
    int *lists = hl.as<int>() + 16;
    const size_t half_l = (size_t)n_upper + 64;
    if (!flip) {                              // a non-seeded launch starts a solve: the rotation restarts with clean counters
      c->knn_rot = 0;
      MLOAM_CUDA_OK(c, cudaMemsetAsync(cnt, 0, 3 * sizeof(int), c->stream));
    }
    const int k = c->knn_rot;
    if (flip) hq.list_in = lists + half_l * (size_t)(k & 1), hq.cnt_in = cnt + k % 3;
    hq.list_out = lists + half_l * (size_t)((k + 1) & 1), hq.cnt_out = cnt + (k + 1) % 3, hq.cnt_zero = cnt + (k + 2) % 3;
    c->knn_rot = k + 1;
  }
  if (flip) c->knn_parity ^= 1;
  cudaStream_t st = c->stream;
  {
    ProfScope ps(c, "match");
    // with stage profiling on: how many queries took the keep (matched / rejected), ball and blind paths
    unsigned *path_stats = (c->prof_on && !getenv("MLOAM_KNN_NO_STATS")) ? reinterpret_cast<unsigned *>(c->scratch[7].as<char>() + kKnnPathStatsOffset) : nullptr;
    unsigned *trace = nullptr;
    if (c->knn_trace_on) {
      MLOAM_CUDA_OK(c, c->knn_trace.reserve(16 * (size_t)(n_upper + 1) + 16 * 8 * 4 * 148 + 64));
      MLOAM_CUDA_OK(c, cudaMemsetAsync(c->knn_trace.p, 0, 16 * (size_t)(n_upper + 1) + 16 * 8 * 4 * 148, st));
      trace = c->knn_trace.as<unsigned>();
    }
    const int mb = c->knn_min_blocks;
    int nb = (n_upper + MWARPS - 1) / MWARPS;
    if (nb > mb * c->sm_count) nb = mb * c->sm_count;  // all CTAs resident; warps pull / stride over the features
#define MLOAM_LAUNCH_KNN(KK, MBB) \
  k_match_knn<KK, MBB><<<nb, MWARPS * 32, 0, st>>>(ks[0], ks[1], d_pose7, cfg.min_match_sq_dis, hq, path_stats, c->knn_tma_min, trace)
    if (K == 5) {
      if (mb == 2) MLOAM_LAUNCH_KNN(5, 2);
      else if (mb == 3) MLOAM_LAUNCH_KNN(5, 3);
      else MLOAM_LAUNCH_KNN(5, 4);
    } else {
      if (mb == 2) MLOAM_LAUNCH_KNN(10, 2);
      else if (mb == 3) MLOAM_LAUNCH_KNN(10, 3);
      else MLOAM_LAUNCH_KNN(10, 4);
    }
#undef MLOAM_LAUNCH_KNN
    c->launches++;
  }
  if (defer && !fs[0].nn && !fs[1].nn) {
    defer->set[0] = fs[0], defer->set[1] = fs[1];
    defer->K = K, defer->min_plane_dis = cfg.min_plane_dis, defer->check_fov = cfg.check_fov;
  } else {
    ProfScope ps(c, "fit");
    int nb = (n_upper + 127) / 128;
    if (nb > 4 * c->sm_count) nb = 4 * c->sm_count;
    if (K == 5) k_match_fit<5><<<nb, 128, 0, st>>>(fs[0], fs[1], d_pose7, cfg.min_plane_dis, cfg.check_fov);
    else k_match_fit<10><<<nb, 128, 0, st>>>(fs[0], fs[1], d_pose7, cfg.min_plane_dis, cfg.check_fov);
    c->launches++;
  }
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

int match_from_map_device(Ctx *c, int slot, int type, const float4 *d_pts, int n, const int *d_n, const double *d_pose7,
                          const MatchCfg &cfg, unsigned char *d_valid, float *d_coeff, int *d_nn) {
  MatchJob j{slot, type, d_pts, n, d_n, d_valid, d_coeff, d_nn, 0};
  return match_pair_device(c, &j, 1, d_pose7, cfg);
}

}  // namespace mloam
