// solve_kernels.cu — residual/Jacobian evaluation, J^T J / J^T r reduction and the device-resident
// Levenberg-Marquardt state machine that replaces ceres::Solve for the single-pose problems of the path
// (lidar_mapper_keyframe.cpp:537-596, lidar_tracker.cpp:70-120).
//
//   k_linearize : one thread per feature -> (r, 1x6 row) in double, Huber corrector, per-thread packed
//                 upper-triangular J^T J (21) + J^T r (6) + cost + row counts, 31-exchange butterfly over the 30
//                 components -> shared-memory cross-warp sum -> one partial per block (deterministic: no atomics).
//                 The block that finishes last (ticket) runs lm_tail: fixed-order sum of the block partials, optional
//                 peer-memory exchange with the other GPUs' sums, and the LM state machine (Jacobi scaling, LM diagonal,
//                 6x6 Cholesky, step acceptance, radius update, tolerances, degeneracy remap) on a shared-memory copy of
//                 the device-resident state — the host only reads the final state back.
//   k_lm        : the same tail as a stand-alone kernel (NCCL path, mloam_normal_equations).
#include "ctx.h"
#include "factors.cuh"
#include "match_fit.cuh"

namespace mloam {

constexpr int NE_H = 21, NE_G = 6;
constexpr int NE_PACK = 30;  // 21 H upper | 6 g | cost | rows(set 0) | rows(set 1)
constexpr int LIN_THREADS = 256;
constexpr int LM_THREADS = 256;

struct FeatSetDev {
  const float4 *pts;
  const unsigned char *valid;
  const float *coeff;
  int n;
  int is_plane;
  const int *d_n;
  const double *sinfo;
  const unsigned char *mask;
};
struct LinArgs {
  FeatSetDev set[2];
  int n_sets;
  double sqrt_info, huber_a;
  const double *pose;      // where pass 0 evaluates: an explicit pose, LMState::x or LMState::xc (7 doubles)
  const int *done;         // candidate evaluation: LMState::done (a terminated Solve has nothing to evaluate), else null
  // fused LM tail (single GPU): the block that finishes last reduces the partials and advances the state machine
  int lm_mode;             // 1 | 2, or 0: no tail (partials only)
  double eig_thre;
  unsigned *ticket;        // zero between launches
  LMState *state_rw;
  const P2PView *p2p;      // device copy of the peer-memory view, or null: sum the packed normal equations over the ranks
  // two_pass (needs the fused tail): the evaluation at x, the LM step, and the evaluation at the candidate xc in ONE launch.  The
  // blocks wait at a grid barrier (generation word next to the ticket) for the block that ran the tail; every block of the grid
  // is resident (<= 64 blocks of 256 threads, one per SM).
  int two_pass;
  // deferred fit (KFIT > 0): the thread that evaluates a feature first fits its line / plane from the matcher's neighbour list
  FitSet fit[2];
  float fit_min_plane_dis;
  int fit_check_fov;
};

__device__ __noinline__ void lm_tail(const double *partials, int n_blocks, LMState *gst, int mode, double eig_thre, double *out_ne,
                                     const P2PView *p2p);

template <int KFIT>
__global__ void __launch_bounds__(LIN_THREADS) k_linearize(LinArgs a, double *__restrict__ partials) {
  __shared__ double sm[LIN_THREADS / 32][NE_PACK];
  __shared__ bool is_last;
  __shared__ int barrier_failed;
  if (a.done && *a.done) return;  // Solve already terminated: nothing to evaluate
  volatile unsigned *const gen = a.ticket + 1;
  const unsigned gen0 = a.two_pass ? *gen : 0u;  // read before this block's ticket: the release cannot have happened yet
#pragma unroll 1
  for (int pass = 0; pass < (a.two_pass ? 2 : 1); pass++) {
  double xs[7];
  if (pass == 0) {
#pragma unroll
    for (int k = 0; k < 7; k++) xs[k] = a.pose[k];
  } else {
    // grid barrier: the block that ran the tail of pass 0 publishes the state and bumps the generation word
    if (threadIdx.x == 0) {
      barrier_failed = 0;
      const long long w0 = clock64();
      while (*gen == gen0) {
        if (clock64() - w0 > 4000000000ll) {  // ~2 s: a block of this grid never became resident
          barrier_failed = 1;
          break;
        }
      }
      __threadfence();
    }
    __syncthreads();
    if (barrier_failed) {
      if (threadIdx.x == 0) a.state_rw->termination = 8, a.state_rw->done = 1;
      return;
    }
    if (__ldcg(&a.state_rw->done)) return;  // the step of pass 0 ended the Solve (tolerance, too few rows, invalid steps)
#pragma unroll
    for (int k = 0; k < 7; k++) xs[k] = __ldcg(&a.state_rw->xc[k]);  // L2: this SM's L1 may hold the line from pass 0
  }
  const PoseR P = make_poser(xs);
  double acc[NE_PACK];
#pragma unroll
  for (int k = 0; k < NE_PACK; k++) acc[k] = 0.0;
  for (int s = 0; s < a.n_sets; s++) {
    const FeatSetDev fs = a.set[s];
    const int fn = fs.d_n ? min(fs.n, *fs.d_n) : fs.n;
    // Both sets keep their features at the low indices of a much larger launch bound: the second set is handed out from
    // the last thread downwards, so that a thread evaluates one feature of either set instead of one of each.
    const int G = gridDim.x * blockDim.x, gid = blockIdx.x * blockDim.x + threadIdx.x;
    for (int i = (s & 1) ? G - 1 - gid : gid; i < fn; i += G) {
      if (KFIT > 0 && pass == 0 && a.fit[s].pos) {  // deferred fit: this thread is the only one that touches feature i
        const PoseD T = pose_from_param(xs);
        fit_one<(KFIT > 0 ? KFIT : 5)>(a.fit[s], i, T, a.fit_min_plane_dis, a.fit_check_fov);
      }
      if (!fs.valid[i] || (fs.mask && !fs.mask[i])) continue;
      const float4 pf = __ldg(fs.pts + i);
      const D3 p{(double)pf.x, (double)pf.y, (double)pf.z};
      const float *cf = fs.coeff + (size_t)i * 6;
      double J[6];
      double r;
      if (fs.is_plane == 2) {
        // LidarScanEdgeFactorVector (tracker, lidar_tracker.cpp:89): one 3-row residual BLOCK, the loss acts on
        // its squared norm (Ceres applies rho per block)
        double r3[3], J3[18];
        edge_vector_factor(P, p, D3{(double)cf[0], (double)cf[1], (double)cf[2]}, D3{(double)cf[3], (double)cf[4], (double)cf[5]}, r3,
                           J3, true);
        double rho, rho1;
        huber(a.huber_a, r3[0] * r3[0] + r3[1] * r3[1] + r3[2] * r3[2], &rho, &rho1);
        const double sc = sqrt(rho1);
#pragma unroll
        for (int m = 0; m < 3; m++) {
          const double rm = sc * r3[m];
          double Jm[6];
#pragma unroll
          for (int k = 0; k < 6; k++) Jm[k] = sc * J3[m * 6 + k];
          int q = 0;
#pragma unroll
          for (int i0 = 0; i0 < 6; i0++)
#pragma unroll
            for (int j0 = i0; j0 < 6; j0++) acc[q++] += Jm[i0] * Jm[j0];
#pragma unroll
          for (int k = 0; k < 6; k++) acc[NE_H + k] += Jm[k] * rm;
        }
        acc[NE_H + NE_G] += 0.5 * rho;
        if (s == 0) acc[NE_H + NE_G + 1] += 1.0;
        else acc[NE_H + NE_G + 2] += 1.0;
        continue;
      }
      const double si = fs.sinfo ? fs.sinfo[i] : a.sqrt_info;  // per-feature weight when mapping is uncertainty-aware
      if (fs.is_plane) {
        r = plane_factor(P, p, D3{(double)cf[0], (double)cf[1], (double)cf[2]}, (double)cf[3], si, J, true);
      } else {
        r = edge_factor(P, p, D3{(double)cf[0], (double)cf[1], (double)cf[2]}, D3{(double)cf[3], (double)cf[4], (double)cf[5]},
                        si, J, true);
      }
      double rho, rho1;
      huber(a.huber_a, r * r, &rho, &rho1);
      const double sc = sqrt(rho1);
      r = sc * r;
#pragma unroll
      for (int k = 0; k < 6; k++) J[k] = sc * J[k];
      int q = 0;
#pragma unroll
      for (int i0 = 0; i0 < 6; i0++)
#pragma unroll
        for (int j0 = i0; j0 < 6; j0++) acc[q++] += J[i0] * J[j0];
#pragma unroll
      for (int k = 0; k < 6; k++) acc[NE_H + k] += J[k] * r;
      acc[NE_H + NE_G] += 0.5 * rho;
      if (s == 0) acc[NE_H + NE_G + 1] += 1.0;
      else acc[NE_H + NE_G + 2] += 1.0;
    }
  }
  // Warp reduction of all 30 components at once (fixed butterfly, 31 exchanges instead of 30 x 5): at offset o a lane
  // keeps the half of its remaining components selected by its bit o and adds the partner's partial sums of that
  // half; after offsets 16..1 lane L holds the warp total of component L.
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  {
    double v[32];
#pragma unroll
    for (int k = 0; k < 32; k++) v[k] = k < NE_PACK ? acc[k] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const bool upper = (lane & o) != 0;
#pragma unroll
      for (int k = 0; k < o; k++) {
        const double send = upper ? v[k] : v[k + o];
        const double keep = upper ? v[k + o] : v[k];
        v[k] = keep + __shfl_xor_sync(MLOAM_FULL_MASK, send, o);
      }
    }
    if (lane < NE_PACK) sm[wid][lane] = v[0];
  }
  __syncthreads();
  if (threadIdx.x < NE_PACK) {
    double v = 0.0;
#pragma unroll
    for (int w = 0; w < LIN_THREADS / 32; w++) v += sm[w][threadIdx.x];
    partials[(size_t)blockIdx.x * NE_PACK + threadIdx.x] = v;
  }
  if (a.lm_mode == 0) return;
  // ---- fused tail: the last block to arrive sums the partials in block order (so the result does not depend on
  // which block that is) and runs the LM step that a separate k_lm launch used to do.
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) {
    if (a.two_pass && pass == 0) continue;  // on to the barrier of pass 1
    return;
  }
  __threadfence();
  lm_tail(partials, (int)gridDim.x, a.state_rw, pass == 0 ? a.lm_mode : 2, a.eig_thre, nullptr, a.p2p);
  __threadfence();  // the state (written by all threads of this block) before the ticket reset and the release
  __syncthreads();
  if (threadIdx.x == 0) {
    *a.ticket = 0u;
    if (a.two_pass && pass == 0) {
      __threadfence();
      atomicAdd(a.ticket + 1, 1u);  // release the grid into pass 1
    }
  }
  }
}

// ---------------------------------------------------------------------------------------- small dense (device)
__host__ __device__ void eig_sym6(const double *Ain, double *w, double *V) {
  const int N = 6;
  double a[36], v[36];
  for (int i = 0; i < 36; i++) a[i] = Ain[i], v[i] = (i % 7 == 0) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0, diag = 0;
    for (int i = 0; i < N; i++) {
      diag += fabs(a[i * N + i]);
      for (int j = i + 1; j < N; j++) off += fabs(a[i * N + j]);
    }
    if (off <= 1e-22 * diag || off == 0.0) break;
    for (int p = 0; p < N - 1; p++)
      for (int q = p + 1; q < N; q++) {
        const double apq = a[p * N + q];
        if (apq == 0.0) continue;
        const double theta = (a[q * N + q] - a[p * N + p]) / (2.0 * apq);
        double t = 1.0 / (fabs(theta) + sqrt(theta * theta + 1.0));
        if (theta < 0.0) t = -t;
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        a[p * N + p] -= t * apq;
        a[q * N + q] += t * apq;
        a[p * N + q] = a[q * N + p] = 0.0;
        for (int r = 0; r < N; r++) {
          if (r == p || r == q) continue;
          const double arp = a[r * N + p], arq = a[r * N + q];
          a[r * N + p] = a[p * N + r] = c * arp - s * arq;
          a[r * N + q] = a[q * N + r] = s * arp + c * arq;
        }
        for (int k = 0; k < N; k++) {
          const double vkp = v[k * N + p], vkq = v[k * N + q];
          v[k * N + p] = c * vkp - s * vkq;
          v[k * N + q] = s * vkp + c * vkq;
        }
      }
  }
  int idx[6] = {0, 1, 2, 3, 4, 5};
  for (int i = 1; i < N; i++) {  // stable insertion sort, ascending
    int k = idx[i], j = i - 1;
    while (j >= 0 && a[idx[j] * N + idx[j]] > a[k * N + k]) idx[j + 1] = idx[j], j--;
    idx[j + 1] = k;
  }
  for (int j = 0; j < N; j++) {
    w[j] = a[idx[j] * N + idx[j]];
    for (int k = 0; k < N; k++) V[k * N + j] = v[k * N + idx[j]];
  }
}

// Eigenvalue report of a non-degenerate Solve, filled in by the host from the read-back H0 (the device only runs the
// 6x6 Jacobi solver when the Cholesky test says a direction is degenerate — a ~10^5-cycle single-thread job).
void eig_report_host(const double *H36, double *w6) {
  double V[36];
  eig_sym6(H36, w6, V);
}

// In-place lower Cholesky factor of a 6x6; inv_diag[j] = 1 / L[j][j].  One square root and one division per column:
// the off-diagonal entries are scaled by the reciprocal (double division is a ~100-cycle software sequence and this
// runs on a single thread between two grid-wide kernels).
__device__ __forceinline__ bool chol6(double *A, double *inv_diag) {
  constexpr int N = 6;
#pragma unroll
  for (int j = 0; j < N; j++) {
    double d = A[j * N + j];
#pragma unroll
    for (int k = 0; k < j; k++) d -= A[j * N + k] * A[j * N + k];
    if (!(d > 0.0)) return false;
    d = sqrt(d);
    A[j * N + j] = d;
    const double inv = 1.0 / d;
    inv_diag[j] = inv;
#pragma unroll
    for (int i = j + 1; i < N; i++) {
      double s = A[i * N + j];
#pragma unroll
      for (int k = 0; k < j; k++) s -= A[i * N + k] * A[j * N + k];
      A[i * N + j] = s * inv;
    }
  }
  return true;
}
__device__ __forceinline__ void chol6_solve(const double *L, const double *inv_diag, const double *b, double *x) {
  constexpr int N = 6;
  double y[6];
#pragma unroll
  for (int i = 0; i < N; i++) {
    double s = b[i];
#pragma unroll
    for (int k = 0; k < i; k++) s -= L[i * N + k] * y[k];
    y[i] = s * inv_diag[i];
  }
#pragma unroll
  for (int i = N - 1; i >= 0; i--) {
    double s = y[i];
#pragma unroll
    for (int k = i + 1; k < N; k++) s -= L[k * N + i] * x[k];
    x[i] = s * inv_diag[i];
  }
}

// Ceres defaults the reference relies on (never overridden in-tree; SURVEY.md §8c)
__device__ constexpr double kMinDiag = 1e-6, kMaxDiag = 1e32, kMaxRadius = 1e16;
__device__ constexpr double kFuncTol = 1e-6, kParamTol = 1e-8, kGradTol = 1e-10, kMinRelDecrease = 1e-3;

__device__ double gradient_max_norm(const LMState *st) {
  double neg[6], xp[7];
  for (int j = 0; j < 6; j++) neg[j] = -st->g[j];
  pose_plus(st->x, neg, st->V_update, xp);
  double m = 0;
  for (int k = 0; k < 7; k++) m = fmax(m, fabs(st->x[k] - xp[k]));
  return m;
}

// LevenbergMarquardtStrategy::ComputeStep + the invalid-step loop of TrustRegionMinimizer.
__device__ void lm_compute_step(LMState *st) {
  while (true) {
    if (st->iteration >= st->max_inner) {
      st->done = 1, st->termination = 0;
      return;
    }
    double Hs[36], gs[6], A[36], step[6];
#pragma unroll
    for (int a = 0; a < 6; a++) {
      gs[a] = st->scale[a] * st->g[a];
#pragma unroll
      for (int b = 0; b < 6; b++) Hs[a * 6 + b] = st->scale[a] * st->H[a * 6 + b] * st->scale[b];
    }
    if (!st->reuse_diagonal) {
#pragma unroll
      for (int j = 0; j < 6; j++) st->diag[j] = fmin(fmax(Hs[j * 6 + j], kMinDiag), kMaxDiag);
    }
#pragma unroll
    for (int i = 0; i < 36; i++) A[i] = Hs[i];
#pragma unroll
    for (int j = 0; j < 6; j++) {
      const double l = sqrt(st->diag[j] / st->radius);
      A[j * 6 + j] += l * l;
    }
    double inv_diag[6];
    bool ok = chol6(A, inv_diag);
    if (ok) {
      chol6_solve(A, inv_diag, gs, step);
#pragma unroll
      for (int j = 0; j < 6; j++) {
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
#pragma unroll
      for (int a = 0; a < 6; a++) {
        sg += step[a] * gs[a];
        double t = 0;
#pragma unroll
        for (int b = 0; b < 6; b++) t += Hs[a * 6 + b] * step[b];
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
      st->reuse_diagonal = 1;
      continue;
    }
    st->num_invalid = 0;
    double delta[6];
#pragma unroll
    for (int j = 0; j < 6; j++) delta[j] = step[j] * st->scale[j];
    pose_plus(st->x, delta, st->V_update, st->xc);
    st->model_cost_change = mcc;
    return;
  }
}

__device__ void unpack_ne(const double *ne, double *H, double *g) {
  int q = 0;
  for (int i = 0; i < 6; i++)
    for (int j = i; j < 6; j++) {
      H[i * 6 + j] = ne[q];
      H[j * 6 + i] = ne[q];
      q++;
    }
  for (int k = 0; k < 6; k++) g[k] = ne[NE_H + k];
}

// One thread advances the state machine on a shared-memory copy of the state (lm_tail stages it in and out).
// mode 1: begin a Solve with the evaluation at x.  mode 2: digest the evaluation at xc.
__device__ void lm_advance(LMState *st, const double *ne, int mode, double eig_thre) {
  double H[36], g[6];
  unpack_ne(ne, H, g);
  const double cost = ne[NE_H + NE_G];
  if (mode == 1) {
    for (int i = 0; i < 36; i++) st->H[i] = H[i], st->H0[i] = H[i];
    for (int i = 0; i < 6; i++) st->g[i] = g[i];
    st->cost = cost;
    st->initial_cost = cost;
    st->n_valid[0] = (int)ne[NE_H + NE_G + 1];
    st->n_valid[1] = (int)ne[NE_H + NE_G + 2];
    st->rows = st->n_valid[0] + st->n_valid[1];
    st->skipped = 0;
    if (st->rows < st->min_corr) {  // "less correspondence": the outer iteration is skipped, pose untouched
      st->done = 1, st->termination = 5, st->skipped = 1;
      for (int k = 0; k < 7; k++) st->xc[k] = st->x[k];
      return;
    }
    // PoseLocalParameterization::setParameter + evalDegenracy (lidar_mapper_keyframe.cpp:1172-1204)
    for (int i = 0; i < 36; i++) st->V_update[i] = (i % 7 == 0) ? 1.0 : 0.0;
    st->is_degenerate = 0;
    for (int i = 0; i < 6; i++) st->eig[i] = 0.0;
    // lambda_min(H) > eig_thre  <=>  H - eig_thre*I is positive definite: one 6x6 Cholesky decides the common,
    // non-degenerate case; the Jacobi eigen-solver only runs when a direction is (nearly) degenerate.
    bool need_eig = st->rows > 0 && eig_thre > 0.0;
    if (need_eig) {
      double S[36];
      for (int i = 0; i < 36; i++) S[i] = H[i] - ((i % 7 == 0) ? eig_thre : 0.0);
      double inv_diag[6];
      if (chol6(S, inv_diag)) need_eig = false;
    }
    if (need_eig) {
      double w[6], Vf[36], Vp[36];
      eig_sym6(H, w, Vf);
      for (int i = 0; i < 36; i++) Vp[i] = Vf[i];
      for (int j = 0; j < 6; j++) {
        if (w[j] < eig_thre) {
          for (int k = 0; k < 6; k++) Vp[k * 6 + j] = 0.0;
          st->is_degenerate = 1;
        } else {
          break;
        }
      }
      for (int i = 0; i < 6; i++) st->eig[i] = w[i];
      if (st->is_degenerate)
        for (int i = 0; i < 6; i++)
          for (int j = 0; j < 6; j++) {
            double s = 0;
            for (int k = 0; k < 6; k++) s += Vf[i * 6 + k] * Vp[j * 6 + k];
            st->V_update[i * 6 + j] = s;
          }
    }
    // Compiler barrier: the state is re-read from shared memory below instead of being held in registers across the
    // degeneracy test (which would add spills to lm_tail and stack to every kernel that calls it).
    asm volatile("" ::: "memory");
    double xn = 0;
    for (int k = 0; k < 7; k++) xn += st->x[k] * st->x[k];
    st->x_norm = sqrt(xn);
    for (int j = 0; j < 6; j++) st->scale[j] = 1.0 / (1.0 + sqrt(H[j * 6 + j]));
    st->radius = 1e4, st->decrease_factor = 2.0, st->reuse_diagonal = 0;
    st->iteration = 0, st->num_invalid = 0, st->done = 0, st->termination = 0;
    for (int k = 0; k < 7; k++) st->xc[k] = st->x[k];
    if (gradient_max_norm(st) <= kGradTol) {
      st->done = 1, st->termination = 3;
      return;
    }
    lm_compute_step(st);
    return;
  }
  // mode 2
  if (st->done) return;
  double sn = 0;
  for (int k = 0; k < 7; k++) sn += (st->x[k] - st->xc[k]) * (st->x[k] - st->xc[k]);
  sn = sqrt(sn);
  if (sn <= kParamTol * (st->x_norm + kParamTol)) {
    st->done = 1, st->termination = 2;
    return;
  }
  const double cost_change = st->cost - cost;
  if (fabs(cost_change) <= kFuncTol * st->cost) {
    st->done = 1, st->termination = 1;
    return;
  }
  const double rel = cost_change / st->model_cost_change;
  if (rel > kMinRelDecrease) {
    const double t = 2.0 * rel - 1.0;
    st->radius = st->radius / fmax(1.0 / 3.0, 1.0 - t * t * t);
    st->radius = fmin(kMaxRadius, st->radius);
    st->decrease_factor = 2.0;
    st->reuse_diagonal = 0;
    double xn = 0;
    for (int k = 0; k < 7; k++) st->x[k] = st->xc[k], xn += st->xc[k] * st->xc[k];
    st->x_norm = sqrt(xn);
    for (int i = 0; i < 36; i++) st->H[i] = H[i];
    for (int i = 0; i < 6; i++) st->g[i] = g[i];
    st->cost = cost;
    if (gradient_max_norm(st) <= kGradTol) {
      st->done = 1, st->termination = 3;
      return;
    }
  } else {
    st->radius = st->radius / st->decrease_factor;
    st->decrease_factor *= 2.0;
    st->reuse_diagonal = 1;
  }
  lm_compute_step(st);
}

// Called by all LM_THREADS threads of one block.  Block partials -> packed normal equations in a fixed order
// (deterministic): warp w sums blocks w, w+8, ... for component `lane`, then the 8 warp sums are added in warp order.
// The LM state lives in global memory between launches; it is staged through shared memory here because the
// single-threaded state machine touches it a few hundred times (each a dependent L2 round trip otherwise).
//
// Multi-GPU (p2p != nullptr): one LiDAR per GPU, the LM step needs the SUM of every rank's normal equations.  The
// reduction, the exchange and the step are one kernel: this block stores its 30 doubles into slot[rank] of every
// rank's exchange buffer (peer stores over NVLink), raises its flag there, polls its own buffer until all ranks'
// flags carry this exchange's epoch, and adds the slots in rank order — the same order on every rank, so all ranks
// advance bit-identical states.  Slots and flags are double-buffered by the parity of the epoch: a rank can only be
// one exchange ahead of the slowest one, so a slot is never overwritten before it has been read.
__device__ __noinline__ void lm_tail(const double *partials, int n_blocks, LMState *gst, int mode, double eig_thre, double *out_ne,
                                     const P2PView *p2p) {
  __shared__ double ne[NE_PACK];
  __shared__ unsigned long long p2p_epoch;
  __shared__ int p2p_timeout;
  __shared__ double wsum[LM_THREADS / 32][32];
  __shared__ LMState s;
  static_assert(sizeof(LMState) % 8 == 0, "LMState is staged as 8-byte words");
  constexpr int kWords = (int)(sizeof(LMState) / 8);
  const long long t0 = clock64();
  if (mode != 0) {
    const unsigned long long *src = reinterpret_cast<const unsigned long long *>(gst);
    unsigned long long *dst = reinterpret_cast<unsigned long long *>(&s);
    for (int k = threadIdx.x; k < kWords; k += LM_THREADS) dst[k] = __ldcg(src + k);
  }
  {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    constexpr int S = LM_THREADS / 32;
    double v = 0.0;
    if (lane < NE_PACK) {
      const double *p = partials + lane;
      int b = w;
      for (; b + 7 * S < n_blocks; b += 8 * S) {  // eight loads in flight, same summation order
        double t[8];
#pragma unroll
        for (int u = 0; u < 8; u++) t[u] = __ldcg(p + (size_t)(b + u * S) * NE_PACK);
#pragma unroll
        for (int u = 0; u < 8; u++) v += t[u];
      }
      for (; b < n_blocks; b += S) v += __ldcg(p + (size_t)b * NE_PACK);
    }
    wsum[w][lane] = v;
    __syncthreads();
    if (threadIdx.x < NE_PACK) {
      double t = 0.0;
#pragma unroll
      for (int ww = 0; ww < S; ww++) t += wsum[ww][threadIdx.x];
      ne[threadIdx.x] = t;
      if (out_ne) out_ne[threadIdx.x] = t;
    }
  }
  __syncthreads();
  if (mode == 0) return;
  if (p2p) {
    const int N = p2p->nranks, me = p2p->rank;
    if (threadIdx.x == 0) p2p_epoch = *p2p->epoch, p2p_timeout = 0;
    __syncthreads();
    const unsigned long long ep = p2p_epoch;
    const int par = (int)(ep & 1ull);
    const unsigned target = (unsigned)(ep + 1ull);
    if (threadIdx.x < NE_PACK)
      for (int q = 0; q < N; q++) reinterpret_cast<volatile double *>(p2p->slots[q])[(par * MLOAM_P2P_MAX_RANKS + me) * 32 + threadIdx.x] = ne[threadIdx.x];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < N) {
      *reinterpret_cast<volatile unsigned *>(p2p->flags[threadIdx.x] + par * MLOAM_P2P_MAX_RANKS + me) = target;  // notify rank threadIdx.x
      volatile unsigned *mine = reinterpret_cast<volatile unsigned *>(p2p->flags[me] + par * MLOAM_P2P_MAX_RANKS + threadIdx.x);
      const long long w0 = clock64();
      while (true) {
        const unsigned v = *mine;
        if (v == target) break;
        if ((int)(v - target) > 0) {  // the peer is AHEAD of this exchange: the ranks lost lock-step, its slot holds a later sum
          p2p_timeout = 2;
          break;
        }
        if (clock64() - w0 > 6000000000ll) {  // ~3 s: a peer never showed up
          p2p_timeout = 1;
          break;
        }
      }
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x < NE_PACK) {
      double t = 0.0;
      for (int q = 0; q < N; q++) t += reinterpret_cast<volatile double *>(p2p->slots[me])[(par * MLOAM_P2P_MAX_RANKS + q) * 32 + threadIdx.x];
      ne[threadIdx.x] = t;
    }
    if (threadIdx.x == 0) *p2p->epoch = ep + 1ull;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    const long long t1 = clock64();
    lm_advance(&s, ne, mode, eig_thre);
    if (p2p && p2p_timeout) s.done = 1, s.termination = 9;  // exchange failed: the state is not trustworthy
    s.dbg_cycles[0] += t1 - t0, s.dbg_cycles[1] += clock64() - t1, s.dbg_cycles[2] += 1;
  }
  __syncthreads();
  {
    const unsigned long long *src = reinterpret_cast<const unsigned long long *>(&s);
    unsigned long long *dst = reinterpret_cast<unsigned long long *>(gst);
    for (int k = threadIdx.x; k < kWords; k += LM_THREADS) dst[k] = src[k];
  }
}

__global__ void __launch_bounds__(LM_THREADS) k_lm(const double *__restrict__ partials, int n_blocks, LMState *st, int mode, double eig_thre,
                                                  double *__restrict__ out_ne) {
  lm_tail(partials, n_blocks, st, mode, eig_thre, out_ne, nullptr);
}

__global__ void k_lm_init(LMState *st, const double *pose7, int max_inner, int min_corr) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    for (int k = 0; k < 7; k++) st->x[k] = pose7[k], st->xc[k] = pose7[k];
    st->max_inner = max_inner;
    st->min_corr = min_corr, st->skipped = 0;
    st->done = 0, st->termination = 0, st->total_iterations = 0, st->iteration = 0;
    st->is_degenerate = 0, st->rows = 0, st->n_valid[0] = st->n_valid[1] = 0;
    st->cost = 0, st->initial_cost = 0;
    for (int i = 0; i < 36; i++) st->V_update[i] = (i % 7 == 0) ? 1.0 : 0.0, st->H0[i] = 0, st->H[i] = 0;
    for (int i = 0; i < 6; i++) st->eig[i] = 0, st->g[i] = 0;
    for (int i = 0; i < 4; i++) st->dbg_cycles[i] = 0;
  }
}

int lm_init_state(Ctx *c, const double *pose7_host, int max_inner, int min_corr) {
  MLOAM_CUDA_OK(c, c->lm_state.reserve(sizeof(LMState) + 64));
  // stage the pose through pinned memory so the copy is truly asynchronous
  double *stage = reinterpret_cast<double *>(c->pinned);
  for (int k = 0; k < 7; k++) stage[k] = pose7_host[k];
  double *d_stage = c->scratch[7].as<double>();
  MLOAM_CUDA_OK(c, cudaMemcpyAsync(d_stage, stage, 7 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  k_lm_init<<<1, 32, 0, c->stream>>>(c->lm_state.as<LMState>(), d_stage, max_inner, min_corr);
  c->launches++;
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

int linearize_device(Ctx *c, const FeatSet *sets, int n_sets, const SolveCfg &cfg, LinEval eval, const double *d_pose7,
                     double *d_out30, const PendingFit *fit, bool two_pass, bool *two_pass_done) {
  LinArgs a;
  int n_total = 0;
  for (int s = 0; s < 2; s++) {
    if (s < n_sets) {
      a.set[s].pts = sets[s].pts, a.set[s].valid = sets[s].valid, a.set[s].coeff = sets[s].coeff;
      a.set[s].n = sets[s].n, a.set[s].is_plane = sets[s].is_plane, a.set[s].d_n = sets[s].d_n;
      a.set[s].sinfo = sets[s].sinfo, a.set[s].mask = sets[s].mask;
      n_total = sets[s].n > n_total ? sets[s].n : n_total;
    } else {
      a.set[s].pts = nullptr, a.set[s].valid = nullptr, a.set[s].coeff = nullptr, a.set[s].n = 0, a.set[s].is_plane = 0, a.set[s].d_n = nullptr;
      a.set[s].sinfo = nullptr, a.set[s].mask = nullptr;
    }
  }
  LMState *st = c->lm_state.as<LMState>();
  a.n_sets = n_sets, a.sqrt_info = cfg.sqrt_info, a.huber_a = cfg.huber_a;
  a.pose = eval == kEvalBegin ? st->x : (eval == kEvalCandidate ? st->xc : d_pose7);
  a.done = eval == kEvalCandidate ? &st->done : nullptr;
  int nb = (n_total + LIN_THREADS - 1) / LIN_THREADS;
  if (nb < 1) nb = 1;
  // n_total is a launch upper bound (device-side counts are usually far smaller): 64 blocks x 256 threads cover a
  // typical frame's ~10^4 features one per thread, and the tail's fixed-order sum reads 64 partials in one round.
  const int max_nb = c->sm_count;
  if (nb > max_nb) nb = max_nb;
  if (nb > 64) nb = 64;
  MLOAM_CUDA_OK(c, c->partials.reserve(sizeof(double) * NE_PACK * (size_t)(max_nb + 3)));
  unsigned *ticket = reinterpret_cast<unsigned *>(c->partials.as<double>() + (size_t)NE_PACK * (max_nb + 2));
  if (c->ticket_zeroed_for != c->partials.p) {  // a fresh partials buffer: the last-block ticket starts at zero
    MLOAM_CUDA_OK(c, cudaMemsetAsync(ticket, 0, sizeof(double), c->stream));
    c->ticket_zeroed_for = c->partials.p;
  }
  const bool collective = c->nccl_comm && cfg.collective;  // sum over the ranks wanted for this solve
  const bool fused = eval != kEvalAtPose && (!collective || c->p2p_on) && !d_out30;
  // only the collective solves (scan2map on every rank in lock-step) exchange; per-rank solves on the same context — the tracker,
  // mloam_normal_equations — stay local
  a.p2p = (fused && c->p2p_on && cfg.collective) ? static_cast<const P2PView *>(c->p2p_view) : nullptr;
  a.lm_mode = fused ? eval : 0, a.eig_thre = cfg.eig_thre, a.ticket = ticket;
  a.state_rw = st;
  // both evaluations of an LM iteration in one launch: only with the fused tail (the barrier is released by the block that ran it)
  a.two_pass = (two_pass && fused && eval == kEvalBegin) ? 1 : 0;
  if (two_pass_done) *two_pass_done = a.two_pass != 0;
  // a fit the matcher deferred to this evaluation
  const int kfit = fit ? fit->K : 0;
  memset(a.fit, 0, sizeof(a.fit));
  a.fit_min_plane_dis = 0.f, a.fit_check_fov = 0;
  if (kfit) {
    a.fit[0] = fit->set[0], a.fit[1] = fit->set[1];
    a.fit_min_plane_dis = fit->min_plane_dis, a.fit_check_fov = fit->check_fov;
  }
  {
    ProfScope ps(c, "linearize");
    if (kfit == 5) k_linearize<5><<<nb, LIN_THREADS, 0, c->stream>>>(a, c->partials.as<double>());
    else if (kfit == 10) k_linearize<10><<<nb, LIN_THREADS, 0, c->stream>>>(a, c->partials.as<double>());
    else k_linearize<0><<<nb, LIN_THREADS, 0, c->stream>>>(a, c->partials.as<double>());
    c->launches++;
  }
  if (fused) {
    MLOAM_CUDA_OK(c, cudaGetLastError());
    return MLOAM_OK;
  }
  if (collective && eval != kEvalAtPose) {
    // multi-GPU: rank-local sum -> NCCL all-reduce of the 30 packed doubles -> identical LM step on every rank
    double *ne = c->partials.as<double>() + (size_t)NE_PACK * max_nb;
    {
      ProfScope ps(c, "lm");
      k_lm<<<1, LM_THREADS, 0, c->stream>>>(c->partials.as<double>(), nb, st, 0, 0.0, ne);
      c->launches++;
    }
    int rc = comm_allreduce_doubles(c, ne, NE_PACK);
    if (rc) return rc;
    ProfScope ps(c, "lm");
    k_lm<<<1, LM_THREADS, 0, c->stream>>>(ne, 1, st, eval, cfg.eig_thre, d_out30);
    c->launches++;
  } else {
    ProfScope ps(c, "lm");
    k_lm<<<1, LM_THREADS, 0, c->stream>>>(c->partials.as<double>(), nb, st, eval, cfg.eig_thre, d_out30);
    c->launches++;
  }
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

// ---------------------------------------------------------------------------------------- batched Evaluate
__global__ void k_factor_evaluate(int kind, int n, const double *__restrict__ points, const double *__restrict__ coeffs,
                                  const double *__restrict__ sqrt_info, const double *__restrict__ params,
                                  double *__restrict__ res, double *__restrict__ jac) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const D3 p{points[i * 3], points[i * 3 + 1], points[i * 3 + 2]};
  const double *cf = coeffs + (size_t)i * 6;
  const double s = sqrt_info ? sqrt_info[i] : 1.0;
  const D3 c0{cf[0], cf[1], cf[2]}, c1{cf[3], cf[4], cf[5]};
  if (kind <= 1) {
    const PoseR P = make_poser(params);
    double J[6];
    const double r = kind == 0 ? plane_factor(P, p, c0, cf[3], s, J, jac != nullptr) : edge_factor(P, p, c0, c1, s, J, jac != nullptr);
    res[i] = r;
    if (jac) {
      for (int k = 0; k < 6; k++) jac[(size_t)i * 7 + k] = J[k];
      jac[(size_t)i * 7 + 6] = 0.0;
    }
  } else if (kind == 2) {
    const PoseR P = make_poser(params);
    double r[3], J[18];
    edge_vector_factor(P, p, c0, c1, r, J, jac != nullptr);
    for (int k = 0; k < 3; k++) res[(size_t)i * 3 + k] = r[k];
    if (jac)
      for (int a = 0; a < 3; a++) {
        for (int k = 0; k < 6; k++) jac[(size_t)i * 21 + a * 7 + k] = J[a * 6 + k];
        jac[(size_t)i * 21 + a * 7 + 6] = 0.0;
      }
  } else {
    const Chain c = make_chain(params, params + 7, params + 14);
    double Jp[6], Ji[6], Je[6];
    const bool wj = jac != nullptr;
    const double r = kind == 3 ? odom_plane_factor(c, p, c0, cf[3], s, wj ? Jp : nullptr, wj ? Ji : nullptr, wj ? Je : nullptr)
                               : odom_edge_factor(c, p, c0, c1, s, wj ? Jp : nullptr, wj ? Ji : nullptr, wj ? Je : nullptr);
    res[i] = r;
    if (jac) {
      double *o = jac + (size_t)i * 21;
      for (int k = 0; k < 6; k++) o[k] = Jp[k], o[7 + k] = Ji[k], o[14 + k] = Je[k];
      o[6] = o[13] = o[20] = 0.0;
    }
  }
}

int factor_evaluate_device(Ctx *c, int kind, int n, const double *d_points, const double *d_coeffs, const double *d_sqrt_info,
                           const double *d_params, double *d_res, double *d_jac) {
  if (kind < 0 || kind > 4) {
    c->err = "factor_evaluate: kind must be 0..4";
    return MLOAM_E_INVALID;
  }
  if (n <= 0) return MLOAM_OK;
  k_factor_evaluate<<<(n + 127) / 128, 128, 0, c->stream>>>(kind, n, d_points, d_coeffs, d_sqrt_info, d_params, d_res, d_jac);
  c->launches++;
  MLOAM_CUDA_OK(c, cudaGetLastError());
  return MLOAM_OK;
}

}  // namespace mloam
