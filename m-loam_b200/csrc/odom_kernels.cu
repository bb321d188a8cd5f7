// odom_kernels.cu — the odometry node's local-map residuals (Estimator::optimizeMap, estimator.cpp:687-848):
// LidarPureOdom{PlaneNorm,Edge}Factor on the pose chain (pose_pivot [constant], pose_i, ext_n), Huber(1.0),
// ceres::Solve(DENSE_SCHUR, NUM_ITERATIONS).  Each feature emits one row over the FREE blocks:
//   1x6  (pose_i free, ext constant: ESTIMATE_EXTRINSIC == 0, estimator.cpp:640,794-848)
//   1x6  (ext free only)
//   1x12 [J_pose_i | J_ext]  (both free: the calibration row of BASELINE.json's north star)
// k_odom_linearize<D>: one thread per feature computes (r, row); the D(D+1)/2 + D + 2 packed sums are reduced
// element by element with warp shuffles into a per-warp shared-memory accumulator (a 1x12 row would need 92 fp64
// accumulators per thread otherwise), summed across warps in fixed order, one partial per CTA — no atomics.
// k_odom_lm<D>: fixed-order partial sum + the same Levenberg-Marquardt state machine as solve_kernels.cu's k_lm,
// generalised to D = 6 or 12 (two 6-dof blocks, PoseLocalParameterization::Plus per block).
#include "ctx.h"
#include "factors.cuh"
#include "host_util.h"

namespace mloam {

constexpr int OD_THREADS = 256;

template <int D>
struct OdPack {
  static constexpr int NH = D * (D + 1) / 2;
  static constexpr int N = NH + D + 2;  // H upper | g | cost | rows
};

struct OdomState {
  double xr[7];                // calibration frame: extrinsic of the reference LiDAR (constant, estimator.cpp:642)
  double xp[7], xi[7], xe[7];  // pivot (constant), pose_i, ext: accepted
  double xic[7], xec[7];       // candidates
  double H[144], g[12], cost;
  double scale[12], diag[12];
  double radius, decrease_factor, model_cost_change, x_norm, initial_cost;
  int free_mask;               // bit 0: pose_i free, bit 1: ext free
  int reuse_diagonal, iteration, num_invalid, done, termination, total_iterations, rows, max_inner, pad;
};

// Row kinds.  0: LidarPureOdom* on (pivot, pose_i, ext) with the free blocks of OdomState::free_mask (mloam_odom_solve).
// Calibration frame (D = 12, state [pose_i | ext_cal]; Estimator::optimizeMap with ESTIMATE_EXTRINSIC == 1, estimator.cpp:687-787):
// 1: LidarPureOdom* of the REFERENCE LiDAR on (pivot, pose_i, ext_ref constant) -> columns 0..5;
// 2: LidarOnlineCalib* of the calibrated LiDAR on ext_cal (lidar_online_calib_factor.hpp:24-227) -> columns 6..11.
constexpr int OD_SETS = 4;
struct OdomSets {
  const float4 *pts[OD_SETS];
  const float *coeff[OD_SETS];
  const unsigned char *valid[OD_SETS];  // nullable: all valid
  int n[OD_SETS];
  int is_plane[OD_SETS];
  int kind[OD_SETS];
  double sqrt_info, huber_a;
};

template <int D>
__global__ void __launch_bounds__(OD_THREADS) k_odom_linearize(OdomSets a, const OdomState *st, int use_candidate, double *__restrict__ partials) {
  constexpr int N = OdPack<D>::N, NH = OdPack<D>::NH;
  __shared__ double acc[OD_THREADS / 32][N];
  if (use_candidate && st->done) return;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  for (int k = lane; k < N; k += 32) acc[wid][k] = 0.0;
  __syncwarp();
  const Chain ch = make_chain(st->xp, use_candidate ? st->xic : st->xi, use_candidate ? st->xec : st->xe);
  const Chain ch_ref = make_chain(st->xp, use_candidate ? st->xic : st->xi, st->xr);
  const PoseR p_cal = make_poser(use_candidate ? st->xec : st->xe);
  const int fm = st->free_mask;
  for (int s = 0; s < OD_SETS; s++) {
    const int n = a.n[s];
    if (n <= 0) continue;
    const int kind = a.kind[s];
    // all lanes of a warp iterate together (the shuffles below need them); out-of-range lanes contribute zeros
    for (int base = (blockIdx.x * (OD_THREADS / 32) + wid) * 32; base < n; base += gridDim.x * OD_THREADS) {
      const int i = base + lane;
      double row[D];
#pragma unroll
      for (int k = 0; k < D; k++) row[k] = 0.0;
      double r = 0.0, rho = 0.0, one = 0.0;
      if (i < n && (!a.valid[s] || a.valid[s][i])) {
        const float4 pf = __ldg(a.pts[s] + i);
        const D3 p{(double)pf.x, (double)pf.y, (double)pf.z};
        const float *cf = a.coeff[s] + (size_t)i * 6;
        double Ji[6], Je[6];
        const D3 c0{(double)cf[0], (double)cf[1], (double)cf[2]}, c1{(double)cf[3], (double)cf[4], (double)cf[5]};
        if (kind == 2) {  // LidarOnlineCalib*: the map factor with T = ext_cal, sqrt_info as given
#pragma unroll
          for (int k = 0; k < 6; k++) Ji[k] = 0.0;
          r = a.is_plane[s] ? plane_factor(p_cal, p, c0, (double)cf[3], a.sqrt_info, Je, true) : edge_factor(p_cal, p, c0, c1, a.sqrt_info, Je, true);
        } else {
          const Chain &cc = kind == 1 ? ch_ref : ch;
          if (a.is_plane[s]) r = odom_plane_factor(cc, p, c0, (double)cf[3], a.sqrt_info, nullptr, Ji, Je);
          else r = odom_edge_factor(cc, p, c0, c1, a.sqrt_info, nullptr, Ji, Je);
          if (kind == 1) {
#pragma unroll
            for (int k = 0; k < 6; k++) Je[k] = 0.0;  // the reference LiDAR's extrinsic is a constant block
          }
        }
        double rho1;
        huber(a.huber_a, r * r, &rho, &rho1);
        const double sc = sqrt(rho1);
        r = sc * r;
        if (D == 12) {
#pragma unroll
          for (int k = 0; k < 6; k++) row[k] = sc * Ji[k], row[6 + k] = sc * Je[k];
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) row[k] = sc * ((fm & 1) ? Ji[k] : Je[k]);
        }
        one = 1.0;
      }
      // element-wise warp reduction into the warp's accumulator (lane 0 adds; order fixed => deterministic)
      int q = 0;
#pragma unroll
      for (int i0 = 0; i0 < D; i0++) {
#pragma unroll
        for (int j0 = i0; j0 < D; j0++) {
          double v = row[i0] * row[j0];
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(MLOAM_FULL_MASK, v, o);
          if (lane == 0) acc[wid][q] += v;
          q++;
        }
      }
#pragma unroll
      for (int k = 0; k < D + 2; k++) {
        double v = k < D ? row[k] * r : (k == D ? 0.5 * rho : one);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(MLOAM_FULL_MASK, v, o);
        if (lane == 0) acc[wid][NH + k] += v;
      }
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < N; k += OD_THREADS) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < OD_THREADS / 32; w++) v += acc[w][k];
    partials[(size_t)blockIdx.x * N + k] = v;
  }
}

// ------------------------------------------------------------------------------------------ LM (D = 6 | 12)
template <int D>
__device__ bool chol_d(double *A) {
  for (int j = 0; j < D; j++) {
    double d = A[j * D + j];
    for (int k = 0; k < j; k++) d -= A[j * D + k] * A[j * D + k];
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    A[j * D + j] = d;
    for (int i = j + 1; i < D; i++) {
      double s = A[i * D + j];
      for (int k = 0; k < j; k++) s -= A[i * D + k] * A[j * D + k];
      A[i * D + j] = s / d;
    }
  }
  return true;
}
template <int D>
__device__ void chol_solve_d(const double *L, const double *b, double *x) {
  double y[D];
  for (int i = 0; i < D; i++) {
    double s = b[i];
    for (int k = 0; k < i; k++) s -= L[i * D + k] * y[k];
    y[i] = s / L[i * D + i];
  }
  for (int i = D - 1; i >= 0; i--) {
    double s = y[i];
    for (int k = i + 1; k < D; k++) s -= L[k * D + i] * x[k];
    x[i] = s / L[i * D + i];
  }
}

__device__ constexpr double kOdMinDiag = 1e-6, kOdMaxDiag = 1e32, kOdMaxRadius = 1e16;
__device__ constexpr double kOdFuncTol = 1e-6, kOdParamTol = 1e-8, kOdGradTol = 1e-10, kOdMinRel = 1e-3;

// x (+) delta over the free blocks (identity V_update: the odometry's per-block degeneracy remap, estimator.cpp:1610-1635,
// is not applied here — next tier)
template <int D>
__device__ void od_plus(const OdomState *st, const double *delta, double *xi_out, double *xe_out) {
  const double I6[36] = {1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1, 0, 0, 0, 0, 0, 0, 1};
  for (int k = 0; k < 7; k++) xi_out[k] = st->xi[k], xe_out[k] = st->xe[k];
  if (D == 12) {
    pose_plus(st->xi, delta, I6, xi_out);
    pose_plus(st->xe, delta + 6, I6, xe_out);
  } else if (st->free_mask & 1) {
    pose_plus(st->xi, delta, I6, xi_out);
  } else {
    pose_plus(st->xe, delta, I6, xe_out);
  }
}
template <int D>
__device__ double od_xnorm(const OdomState *st, const double *xi, const double *xe) {
  double s = 0;
  if (D == 12 || (st->free_mask & 1))
    for (int k = 0; k < 7; k++) s += xi[k] * xi[k];
  if (D == 12 || (st->free_mask & 2))
    for (int k = 0; k < 7; k++) s += xe[k] * xe[k];
  return sqrt(s);
}
template <int D>
__device__ double od_grad_max(const OdomState *st) {
  double neg[D], xi[7], xe[7];
  for (int j = 0; j < D; j++) neg[j] = -st->g[j];
  od_plus<D>(st, neg, xi, xe);
  double m = 0;
  for (int k = 0; k < 7; k++) m = fmax(m, fmax(fabs(st->xi[k] - xi[k]), fabs(st->xe[k] - xe[k])));
  return m;
}
template <int D>
__device__ void od_compute_step(OdomState *st) {
  while (true) {
    if (st->iteration >= st->max_inner) {
      st->done = 1, st->termination = 0;
      return;
    }
    double Hs[D * D], gs[D], A[D * D], step[D];
    for (int a = 0; a < D; a++) {
      gs[a] = st->scale[a] * st->g[a];
      for (int b = 0; b < D; b++) Hs[a * D + b] = st->scale[a] * st->H[a * D + b] * st->scale[b];
    }
    if (!st->reuse_diagonal)
      for (int j = 0; j < D; j++) st->diag[j] = fmin(fmax(Hs[j * D + j], kOdMinDiag), kOdMaxDiag);
    for (int i = 0; i < D * D; i++) A[i] = Hs[i];
    for (int j = 0; j < D; j++) {
      const double l = sqrt(st->diag[j] / st->radius);
      A[j * D + j] += l * l;
    }
    bool ok = chol_d<D>(A);
    if (ok) {
      chol_solve_d<D>(A, gs, step);
      for (int j = 0; j < D; j++) {
        step[j] = -step[j];
        if (!isfinite(step[j])) ok = false;
      }
    }
    st->reuse_diagonal = 1;
    st->iteration++;
    st->total_iterations++;
    double mcc = 0;
    if (ok) {
      double sg = 0, sHs = 0;
      for (int a = 0; a < D; a++) {
        sg += step[a] * gs[a];
        double t = 0;
        for (int b = 0; b < D; b++) t += Hs[a * D + b] * step[b];
        sHs += step[a] * t;
      }
      mcc = -(sg + 0.5 * sHs);
      if (mcc < 0) ok = false;
    }
    if (!ok) {
      if (++st->num_invalid >= 5) {
        st->done = 1, st->termination = 4;
        return;
      }
      st->radius *= 0.5;
      continue;
    }
    st->num_invalid = 0;
    double delta[D];
    for (int j = 0; j < D; j++) delta[j] = step[j] * st->scale[j];
    od_plus<D>(st, delta, st->xic, st->xec);
    st->model_cost_change = mcc;
    return;
  }
}

template <int D>
__global__ void __launch_bounds__(OD_THREADS) k_odom_lm(const double *__restrict__ partials, int n_blocks, OdomState *st, int mode) {
  constexpr int N = OdPack<D>::N, NH = OdPack<D>::NH;
  __shared__ double ne[N];
  for (int k = threadIdx.x; k < N; k += OD_THREADS) {
    double v = 0.0;
    for (int b = 0; b < n_blocks; b++) v += partials[(size_t)b * N + k];
    ne[k] = v;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double H[D * D], g[D];
  int q = 0;
  for (int i = 0; i < D; i++)
    for (int j = i; j < D; j++) H[i * D + j] = H[j * D + i] = ne[q++];
  for (int k = 0; k < D; k++) g[k] = ne[NH + k];
  const double cost = ne[NH + D];
  if (mode == 1) {
    for (int i = 0; i < D * D; i++) st->H[i] = H[i];
    for (int i = 0; i < D; i++) st->g[i] = g[i];
    st->cost = st->initial_cost = cost;
    st->rows = (int)ne[NH + D + 1];
    st->x_norm = od_xnorm<D>(st, st->xi, st->xe);
    for (int j = 0; j < D; j++) st->scale[j] = 1.0 / (1.0 + sqrt(H[j * D + j]));
    st->radius = 1e4, st->decrease_factor = 2.0, st->reuse_diagonal = 0;
    st->iteration = 0, st->num_invalid = 0, st->done = 0, st->termination = 0;
    for (int k = 0; k < 7; k++) st->xic[k] = st->xi[k], st->xec[k] = st->xe[k];
    if (od_grad_max<D>(st) <= kOdGradTol) {
      st->done = 1, st->termination = 3;
      return;
    }
    od_compute_step<D>(st);
    return;
  }
  if (st->done) return;
  double sn = 0;
  for (int k = 0; k < 7; k++)
    sn += (st->xi[k] - st->xic[k]) * (st->xi[k] - st->xic[k]) + (st->xe[k] - st->xec[k]) * (st->xe[k] - st->xec[k]);
  sn = sqrt(sn);
  if (sn <= kOdParamTol * (st->x_norm + kOdParamTol)) {
    st->done = 1, st->termination = 2;
    return;
  }
  const double cost_change = st->cost - cost;
  if (fabs(cost_change) <= kOdFuncTol * st->cost) {
    st->done = 1, st->termination = 1;
    return;
  }
  const double rel = cost_change / st->model_cost_change;
  if (rel > kOdMinRel) {
    const double t = 2.0 * rel - 1.0;
    st->radius = fmin(kOdMaxRadius, st->radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
    st->decrease_factor = 2.0;
    st->reuse_diagonal = 0;
    for (int k = 0; k < 7; k++) st->xi[k] = st->xic[k], st->xe[k] = st->xec[k];
    st->x_norm = od_xnorm<D>(st, st->xi, st->xe);
    for (int i = 0; i < D * D; i++) st->H[i] = H[i];
    for (int i = 0; i < D; i++) st->g[i] = g[i];
    st->cost = cost;
    if (od_grad_max<D>(st) <= kOdGradTol) {
      st->done = 1, st->termination = 3;
      return;
    }
  } else {
    st->radius = st->radius / st->decrease_factor;
    st->decrease_factor *= 2.0;
    st->reuse_diagonal = 1;
  }
  od_compute_step<D>(st);
}

__global__ void k_odom_init(OdomState *st, const double *x21, int free_mask, int max_inner, const double *xr7 = nullptr) {
  if (threadIdx.x == 0) {
    for (int k = 0; k < 7; k++) st->xp[k] = x21[k], st->xi[k] = st->xic[k] = x21[7 + k], st->xe[k] = st->xec[k] = x21[14 + k];
    for (int k = 0; k < 7; k++) st->xr[k] = xr7 ? xr7[k] : (k == 6 ? 1.0 : 0.0);
    st->free_mask = free_mask, st->max_inner = max_inner;
    st->done = 0, st->termination = 0, st->total_iterations = 0, st->iteration = 0, st->rows = 0, st->cost = st->initial_cost = 0;
  }
}

template <int D>
static int odom_solve_run(Ctx *c, const OdomSets &sets, OdomState *st, int max_inner, int nb, double *partials) {
  int *h_done = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 2048);
  k_odom_linearize<D><<<nb, OD_THREADS, 0, c->stream>>>(sets, st, 0, partials);
  k_odom_lm<D><<<1, OD_THREADS, 0, c->stream>>>(partials, nb, st, 1);
  c->launches += 2;
  for (int it = 0; it < max_inner; it++) {
    k_odom_linearize<D><<<nb, OD_THREADS, 0, c->stream>>>(sets, st, 1, partials);
    k_odom_lm<D><<<1, OD_THREADS, 0, c->stream>>>(partials, nb, st, 2);
    c->launches += 2;
    MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_done, &st->done, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
    if (*h_done) break;
  }
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

// ------------------------------------------------------------------------------------------ calibration frame
// poses the two feature groups are matched at (buildCalibMap, estimator.cpp:1086-1090,1135-1149):
//   reference LiDAR, frame i:   pose_local = pivot^-1 * pose_i * ext_ref
//   calibrated LiDAR, pivot:    pose_local = pivot^-1 * pivot * ext_cal = ext_cal
__global__ void k_calib_poses(const OdomState *st, double *pose_a7, double *pose_b7) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const PoseD P = pose_from_param(st->xp), I = pose_from_param(st->xi), R = pose_from_param(st->xr);
  const Q4 qpi = qconj(qnormalized(P.q));
  // pivot^-1 * (pose_i * ext_ref)
  const Q4 q_ir = qmul(I.q, R.q);
  const D3 t_ir = qrot(I.q, R.t) + I.t;
  const Q4 q = qnormalized(qmul(qpi, q_ir));
  const D3 t = qrot(qpi, t_ir - P.t);
  pose_a7[0] = t.x, pose_a7[1] = t.y, pose_a7[2] = t.z, pose_a7[3] = q.x, pose_a7[4] = q.y, pose_a7[5] = q.z, pose_a7[6] = q.w;
  for (int k = 0; k < 7; k++) pose_b7[k] = st->xe[k];
}

template <int D>
__global__ void k_odom_sum_partials(const double *__restrict__ partials, int n_blocks, double *__restrict__ out) {
  constexpr int N = OdPack<D>::N;
  for (int k = threadIdx.x; k < N; k += blockDim.x) {
    double v = 0.0;
    for (int b = 0; b < n_blocks; b++) v += partials[(size_t)b * N + k];
    out[k] = v;
  }
}

// One evaluation of the 12-dof calibration problem + LM state machine step; with a communicator the packed normal
// equations (78 + 12 + 2 doubles) are summed over the ranks first — the path's one collective (SURVEY.md 8e).
static int calib_eval(Ctx *c, const OdomSets &sets, OdomState *st, int nb, double *partials, int use_candidate, int lm_mode) {
  constexpr int N = OdPack<12>::N;
  k_odom_linearize<12><<<nb, OD_THREADS, 0, c->stream>>>(sets, st, use_candidate, partials);
  c->launches++;
  if (c->nccl_comm) {
    double *ne = partials + (size_t)N * (nb + 1);
    k_odom_sum_partials<12><<<1, 128, 0, c->stream>>>(partials, nb, ne);
    c->launches++;
    int rc = comm_allreduce_doubles(c, ne, N);
    if (rc) return rc;
    k_odom_lm<12><<<1, OD_THREADS, 0, c->stream>>>(ne, 1, st, lm_mode);
  } else {
    k_odom_lm<12><<<1, OD_THREADS, 0, c->stream>>>(partials, nb, st, lm_mode);
  }
  c->launches++;
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

}  // namespace mloam

using namespace mloam;

// Estimator::optimizeMap with ESTIMATE_EXTRINSIC == 1 for one frame i and one calibrated LiDAR (estimator.cpp:687-787), the
// matching of buildCalibMap (:1135-1149) redone at every outer iteration: see include/mloam_b200.h.
extern "C" int mloam_calib_frame(mloam_ctx_t *h, const mloam_point_t *h_surf_ref, int n_surf_ref, const mloam_point_t *h_corner_ref,
                                 int n_corner_ref, const mloam_point_t *h_surf_cal, int n_surf_cal, const mloam_point_t *h_corner_cal,
                                 int n_corner_cal, const double *pose_pivot7, double *pose_i7, const double *ext_ref7, double *ext_cal7,
                                 int max_outer, int max_inner, double huber_a, int own_cal_maps, mloam_solve_stats_t *stats) {
  if (!h || !pose_pivot7 || !pose_i7 || !ext_ref7 || !ext_cal7 || n_surf_ref < 0 || n_corner_ref < 0 || n_surf_cal < 0 || n_corner_cal < 0 ||
      max_outer < 1 || max_inner < 1)
    return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  if (stats) memset(stats, 0, sizeof(*stats));
  const MapStorage *M = c->maps;
  if (!M[MLOAM_MAP_SURF].built || !M[MLOAM_MAP_CORNER].built) return fail(c, MLOAM_E_STATE, "calib_frame: build the local maps first");
  if (own_cal_maps && !(M[MLOAM_MAP_SCAN_SURF].built && M[MLOAM_MAP_SCAN_CORNER].built))
    return fail(c, MLOAM_E_STATE, "calib_frame: own_cal_maps needs MLOAM_MAP_SCAN_SURF / MLOAM_MAP_SCAN_CORNER built");
  const int cal_surf = own_cal_maps ? MLOAM_MAP_SCAN_SURF : MLOAM_MAP_SURF, cal_corner = own_cal_maps ? MLOAM_MAP_SCAN_CORNER : MLOAM_MAP_CORNER;
  // sets: 0 corner_ref, 1 surf_ref, 2 corner_cal, 3 surf_cal
  const mloam_point_t *hp[4] = {h_corner_ref, h_surf_ref, h_corner_cal, h_surf_cal};
  const int ns[4] = {n_corner_ref, n_surf_ref, n_corner_cal, n_surf_cal};
  int n_max = 1;
  for (int t = 0; t < 4; t++) {
    if (ns[t] > 0 && !hp[t]) return MLOAM_E_INVALID;
    MLOAM_CUDA_OK(c, c->scan_pts[t].reserve(sizeof(float4) * (size_t)(ns[t] + 1)));
    int rc = reserve_feat(c, t, ns[t]);
    if (rc) return rc;
    if (ns[t] > 0) MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[t].p, hp[t], sizeof(float4) * (size_t)ns[t], cudaMemcpyHostToDevice, c->stream));
    n_max = ns[t] > n_max ? ns[t] : n_max;
  }
  int nb = (n_max + OD_THREADS - 1) / OD_THREADS;
  nb = nb < 1 ? 1 : (nb > c->sm_count ? c->sm_count : nb);
  MLOAM_CUDA_OK(c, c->scratch[6].reserve(sizeof(OdomState) + 512 + sizeof(double) * 96 * (size_t)(nb + 3)));
  OdomState *st = c->scratch[6].as<OdomState>();
  double *partials = reinterpret_cast<double *>(c->scratch[6].as<char>() + ((sizeof(OdomState) + 255) & ~(size_t)255));
  double *stage = reinterpret_cast<double *>(c->pinned) + 200;
  for (int k = 0; k < 7; k++) stage[k] = pose_pivot7[k], stage[7 + k] = pose_i7[k], stage[14 + k] = ext_cal7[k], stage[21 + k] = ext_ref7[k];
  double *d_x = c->scratch[7].as<double>() + 64;  // 28 doubles; the two match poses follow at + 96 / + 104
  double *d_pose_a = c->scratch[7].as<double>() + 96, *d_pose_b = c->scratch[7].as<double>() + 104;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_x, stage, 28 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  k_odom_init<<<1, 32, 0, c->stream>>>(st, d_x, 3, max_inner, d_x + 21);
  c->launches++;
  OdomSets sets;
  memset(&sets, 0, sizeof(sets));
  for (int t = 0; t < 4; t++) {
    sets.pts[t] = c->scan_pts[t].as<float4>(), sets.coeff[t] = c->feat_coeff[t].as<float>(), sets.valid[t] = c->feat_valid[t].as<unsigned char>();
    sets.n[t] = ns[t], sets.is_plane[t] = t & 1, sets.kind[t] = t < 2 ? 1 : 2;
  }
  sets.sqrt_info = 1.0, sets.huber_a = huber_a;  // factors are built with s = 1.0 (estimator.cpp:696,733); Huber(1.0) (:602)
  MatchCfg cfg_ref{c->params.min_match_sq_dis, c->params.min_plane_dis, 5, 1};   // n_neigh 5, CHECK_FOV true (estimator.cpp:1135-1142)
  MatchCfg cfg_cal{c->params.min_match_sq_dis, c->params.min_plane_dis, 10, 1};  // n_neigh 10 for the other LiDARs
  int *h_done = reinterpret_cast<int *>(reinterpret_cast<char *>(c->pinned) + 2048);
  int rc = MLOAM_OK;
  for (int outer = 0; outer < max_outer && rc == MLOAM_OK; outer++) {
    k_calib_poses<<<1, 32, 0, c->stream>>>(st, d_pose_a, d_pose_b);
    c->launches++;
    if (n_corner_ref + n_surf_ref > 0) {
      MatchJob jobs[2] = {MatchJob{MLOAM_MAP_CORNER, 'c', sets.pts[0], ns[0], nullptr, c->feat_valid[0].as<unsigned char>(), c->feat_coeff[0].as<float>(), nullptr, 0},
                          MatchJob{MLOAM_MAP_SURF, 's', sets.pts[1], ns[1], nullptr, c->feat_valid[1].as<unsigned char>(), c->feat_coeff[1].as<float>(), nullptr, 0}};
      rc = match_pair_device(c, jobs, 2, d_pose_a, cfg_ref, 0);
      if (rc) break;
    }
    if (n_corner_cal + n_surf_cal > 0) {
      MatchJob jobs[2] = {MatchJob{cal_corner, 'c', sets.pts[2], ns[2], nullptr, c->feat_valid[2].as<unsigned char>(), c->feat_coeff[2].as<float>(), nullptr, 0},
                          MatchJob{cal_surf, 's', sets.pts[3], ns[3], nullptr, c->feat_valid[3].as<unsigned char>(), c->feat_coeff[3].as<float>(), nullptr, 0}};
      rc = match_pair_device(c, jobs, 2, d_pose_b, cfg_cal, 2);
      if (rc) break;
    }
    rc = calib_eval(c, sets, st, nb, partials, 0, 1);
    for (int it = 0; it < max_inner && rc == MLOAM_OK; it++) {
      rc = calib_eval(c, sets, st, nb, partials, 1, 2);
      if (rc == MLOAM_OK && max_inner > 1) {
        MLOAM_CUDA_OK(c, cudaMemcpyAsync(h_done, &st->done, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
        if (*h_done) break;
      }
    }
  }
  if (rc) return rc;
  OdomState *hs = reinterpret_cast<OdomState *>(reinterpret_cast<char *>(c->pinned) + 8192);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hs, st, sizeof(OdomState), cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 7; k++) pose_i7[k] = hs->xi[k], ext_cal7[k] = hs->xe[k];
  if (stats) {
    stats->ran = 1, stats->lm_iterations = hs->total_iterations, stats->termination = hs->termination, stats->final_cost = hs->cost;
    stats->n_surf = hs->rows;  // residual rows of the last evaluation, all ranks
    stats->n_surf_in = n_surf_ref + n_surf_cal, stats->n_corner_in = n_corner_ref + n_corner_cal;
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 6; j++) stats->H[i * 6 + j] = hs->H[i * 12 + j];  // pose block
  }
  return MLOAM_OK;
}

extern "C" int mloam_odom_solve(mloam_ctx_t *h, int n, const unsigned char *h_types, const double *h_points, const double *h_coeffs,
                                const double *pose_pivot7, double *pose_i7, double *ext7, int free_mask, int max_iterations,
                                double huber_a, double sqrt_info, mloam_solve_stats_t *stats) {
  if (!h || n < 0 || !pose_pivot7 || !pose_i7 || !ext7 || free_mask < 1 || free_mask > 3 || (n > 0 && (!h_types || !h_points || !h_coeffs)))
    return MLOAM_E_INVALID;
  Ctx *c = &h->c;
  cudaSetDevice(c->device);
  if (stats) memset(stats, 0, sizeof(*stats));
  // PointPlaneFeature carries float-valued point_/coeffs_ (feature_extract.hpp:771-781,872-875): device feature format
  std::vector<float4> pts[2];
  std::vector<float> cf[2];
  for (int i = 0; i < n; i++) {
    const int t = h_types[i] == 's' ? 1 : 0;
    pts[t].push_back(make_float4((float)h_points[i * 3], (float)h_points[i * 3 + 1], (float)h_points[i * 3 + 2], 0.f));
    for (int k = 0; k < 6; k++) cf[t].push_back((float)h_coeffs[(size_t)i * 6 + k]);
  }
  OdomSets sets;
  memset(&sets, 0, sizeof(sets));
  int n_max = 0;
  for (int t = 0; t < 2; t++) {
    const int nt = (int)pts[t].size();
    MLOAM_CUDA_OK(c, c->scan_pts[t].reserve(sizeof(float4) * (size_t)(nt + 1)));
    int rc = reserve_feat(c, t, nt);
    if (rc) return rc;
    if (nt > 0) {
      MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->scan_pts[t].p, pts[t].data(), sizeof(float4) * nt, cudaMemcpyHostToDevice, c->stream));
      MLOAM_CUDA_OK(c, cudaMemcpyAsync(c->feat_coeff[t].p, cf[t].data(), sizeof(float) * 6 * nt, cudaMemcpyHostToDevice, c->stream));
    }
    sets.pts[t] = c->scan_pts[t].as<float4>(), sets.coeff[t] = c->feat_coeff[t].as<float>(), sets.n[t] = nt, sets.is_plane[t] = t;
    n_max = nt > n_max ? nt : n_max;
  }
  sets.sqrt_info = sqrt_info, sets.huber_a = huber_a;
  const int D = free_mask == 3 ? 12 : 6;
  int nb = (n_max + OD_THREADS - 1) / OD_THREADS;
  nb = nb < 1 ? 1 : (nb > c->sm_count ? c->sm_count : nb);
  MLOAM_CUDA_OK(c, c->scratch[6].reserve(sizeof(OdomState) + 512 + sizeof(double) * 96 * (size_t)(nb + 1)));
  OdomState *st = c->scratch[6].as<OdomState>();
  double *partials = reinterpret_cast<double *>(c->scratch[6].as<char>() + ((sizeof(OdomState) + 255) & ~(size_t)255));
  double *stage = reinterpret_cast<double *>(c->pinned) + 200;
  for (int k = 0; k < 7; k++) stage[k] = pose_pivot7[k], stage[7 + k] = pose_i7[k], stage[14 + k] = ext7[k];
  double *d_x = c->scratch[7].as<double>() + 64;
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_x, stage, 21 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  k_odom_init<<<1, 32, 0, c->stream>>>(st, d_x, free_mask, max_iterations);
  c->launches++;
  int rc = D == 12 ? odom_solve_run<12>(c, sets, st, max_iterations, nb, partials) : odom_solve_run<6>(c, sets, st, max_iterations, nb, partials);
  if (rc) return rc;
  OdomState *hs = reinterpret_cast<OdomState *>(reinterpret_cast<char *>(c->pinned) + 8192);
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(hs, st, sizeof(OdomState), cudaMemcpyDeviceToHost, c->stream));
  MLOAM_CUDA_OK(c, cudaStreamSynchronize(c->stream));
  for (int k = 0; k < 7; k++) pose_i7[k] = hs->xi[k], ext7[k] = hs->xe[k];
  if (stats) {
    stats->ran = 1, stats->lm_iterations = hs->total_iterations, stats->termination = hs->termination;
    stats->final_cost = hs->cost, stats->n_surf = (int)pts[1].size(), stats->n_corner = (int)pts[0].size();
    for (int i = 0; i < 6; i++)
      for (int j = 0; j < 6; j++) stats->H[i * 6 + j] = hs->H[i * D + j];  // leading 6x6 block
  }
  return MLOAM_OK;
}
