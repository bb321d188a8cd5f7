// common.cuh — shared device-side types and small math for the M-LOAM hot-path kernels (sm_100a).
//
// All translation units are compiled with -fmad=false: every float/double operation rounds once, in
// the order written, so the float gates of the reference (kNN distances, line/plane fits,
// feature_extract.hpp:667,693,830-836) are reproduced decision for decision.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#define MLOAM_FULL_MASK 0xffffffffu

namespace mloam {

// ------------------------------------------------------------------ double 3-vector / 3x3 (row-major)
struct D3 {
  double x, y, z;
};
__host__ __device__ inline D3 operator+(const D3 &a, const D3 &b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__host__ __device__ inline D3 operator-(const D3 &a, const D3 &b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__host__ __device__ inline D3 operator*(double s, const D3 &a) { return {s * a.x, s * a.y, s * a.z}; }
__host__ __device__ inline D3 neg(const D3 &a) { return {-a.x, -a.y, -a.z}; }
__host__ __device__ inline double dot(const D3 &a, const D3 &b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__host__ __device__ inline D3 cross(const D3 &a, const D3 &b) {
  return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
__host__ __device__ inline double norm(const D3 &a) { return sqrt(dot(a, a)); }

struct M33 {
  double m[9];
};
__host__ __device__ inline D3 matvec(const M33 &A, const D3 &v) {
  return {A.m[0] * v.x + A.m[1] * v.y + A.m[2] * v.z, A.m[3] * v.x + A.m[4] * v.y + A.m[5] * v.z,
          A.m[6] * v.x + A.m[7] * v.y + A.m[8] * v.z};
}
// v^T A
__host__ __device__ inline D3 vecmat(const D3 &v, const M33 &A) {
  return {v.x * A.m[0] + v.y * A.m[3] + v.z * A.m[6], v.x * A.m[1] + v.y * A.m[4] + v.z * A.m[7],
          v.x * A.m[2] + v.y * A.m[5] + v.z * A.m[8]};
}
// v^T A^T  ( = (A v)^T )
__host__ __device__ inline D3 vecmatT(const D3 &v, const M33 &A) { return matvec(A, v); }
// v^T [p]x  with [p]x the skew matrix of utility.h:187-195:  v^T [p]x = (v x p)^T ... written out
__host__ __device__ inline D3 vec_skew(const D3 &v, const D3 &p) {
  // [p]x = [0 -pz py; pz 0 -px; -py px 0]
  return {v.y * p.z - v.z * p.y, -v.x * p.z + v.z * p.x, v.x * p.y - v.y * p.x};
}

// ------------------------------------------------------------------ quaternion (x, y, z, w), Eigen conventions
struct Q4 {
  double x, y, z, w;
};
__host__ __device__ inline Q4 qmul(const Q4 &a, const Q4 &b) {
  return {a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y, a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z,
          a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x, a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
__host__ __device__ inline Q4 qconj(const Q4 &q) { return {-q.x, -q.y, -q.z, q.w}; }
__host__ __device__ inline Q4 qnormalized(const Q4 &q) {
  double n = sqrt(q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w);
  return {q.x / n, q.y / n, q.z / n, q.w / n};
}
// q * v as Eigen evaluates it: v + 2w (u x v) + 2 u x (u x v)
__host__ __device__ inline D3 qrot(const Q4 &q, const D3 &v) {
  D3 u{q.x, q.y, q.z};
  D3 uv = cross(u, v);
  uv = uv + uv;
  return v + q.w * uv + cross(u, uv);
}
__host__ __device__ inline M33 qmat(const Q4 &q) {
  const double tx = 2 * q.x, ty = 2 * q.y, tz = 2 * q.z;
  const double twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const double txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const double tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  return M33{{1 - (tyy + tzz), txy - twz, txz + twy, txy + twz, 1 - (txx + tzz), tyz - twx, txz - twy, tyz + twx,
              1 - (txx + tyy)}};
}

struct PoseD {
  Q4 q;
  D3 t;
};
__host__ __device__ inline PoseD pose_from_param(const double *x) {
  return PoseD{Q4{x[3], x[4], x[5], x[6]}, D3{x[0], x[1], x[2]}};
}
// pointAssociateToMap (utility.h:103-117): double math, float store
__host__ __device__ inline float3 associate(const PoseD &T, float px, float py, float pz) {
  D3 v = qrot(T.q, D3{(double)px, (double)py, (double)pz}) + T.t;
  return make_float3((float)v.x, (float)v.y, (float)v.z);
}

// PoseLocalParameterization::Plus (pose_local_parameterization.cpp:26-46)
__host__ __device__ inline void pose_plus(const double *x, const double *delta, const double *V, double *out) {
  double dx[6];
  for (int i = 0; i < 6; i++) {
    double s = 0;
    for (int j = 0; j < 6; j++) s += V[i * 6 + j] * delta[j];
    dx[i] = s;
  }
  out[0] = x[0] + dx[0], out[1] = x[1] + dx[1], out[2] = x[2] + dx[2];
  const Q4 dq{dx[3] / 2.0, dx[4] / 2.0, dx[5] / 2.0, 1.0};  // Utility::deltaQ, utility.h:173-185
  const Q4 qn = qnormalized(qmul(Q4{x[3], x[4], x[5], x[6]}, dq));
  out[3] = qn.x, out[4] = qn.y, out[5] = qn.z, out[6] = qn.w;
}


// ------------------------------------------------------------------ direct-indexed voxel grid map
// The submap lives in HBM as (a) `sorted`: the points grouped by cell, cells in x-fastest linear order, w = original
// index (int bits), and (b) `cell_start`: one exclusive prefix per cell of a DENSE grid over the map's bounding box
// (n_cells + 1 entries).  A cell lookup is one 4-byte load at a computed address — no keys, no probing, no chains —
// and because x is the fastest index the points of x-adjacent cells are contiguous: the 3x3x3 neighbourhood of a
// query is 9 contiguous point runs.  Grid origin / dimensions / cell edge are decided ON THE DEVICE by the build
// (bounding box of the finite points; the cell edge doubles until the grid fits the slot's capacity), so a rebuild
// needs no host round trip and stays capturable in a CUDA graph.
struct GridHdr {
  int ox, oy, oz;          // cell coordinates of the grid origin
  int nx, ny, nz;
  int n_cells;             // nx * ny * nz  (<= capacity)
  int level;               // cell = requested cell * 2^level
  float cell, inv_cell;
  int n_sorted;            // finite points placed in `sorted` (non-finite input points are dropped like PCL does)
  int n_occupied;          // cells holding at least one point (statistics)
  int bb_min[3], bb_max[3];  // bounding box accumulators (order-preserving int encoding of the float coordinates)
  int ticket;              // last-block ticket of the prefix-scan kernels
  int pad[1];
};

struct MapView {
  const float4 *sorted;    // cell-major points: xyz + original index (int bits) in w
  const float4 *orig;      // original order (ring walks of the scan-to-scan matcher); null unless the slot keeps it
  const unsigned *cell_start;
  const GridHdr *hdr;
  int m;                   // input points (original indices run over [0, m))
};

// The header fields a query needs, loaded once per kernel.
struct GridP {
  int ox, oy, oz, nx, ny, nz;
  float cell, inv_cell;
};
__device__ __forceinline__ GridP load_grid(const MapView &mv) {
  GridP g;
  if (!mv.hdr) {  // unused set of a two-set launch
    g.ox = g.oy = g.oz = 0, g.nx = g.ny = g.nz = 0, g.cell = 1.0f, g.inv_cell = 1.0f;
    return g;
  }
  const int4 a = __ldg(reinterpret_cast<const int4 *>(mv.hdr));           // ox oy oz nx
  const int4 b = __ldg(reinterpret_cast<const int4 *>(mv.hdr) + 1);       // ny nz n_cells level
  const float2 c = __ldg(reinterpret_cast<const float2 *>(mv.hdr) + 4);   // cell inv_cell
  g.ox = a.x, g.oy = a.y, g.oz = a.z, g.nx = a.w, g.ny = b.x, g.nz = b.y, g.cell = c.x, g.inv_cell = c.y;
  return g;
}
static_assert(sizeof(GridHdr) % 16 == 0, "GridHdr is read with vector loads");

// ------------------------------------------------------------------ peer-memory exchange (multi-GPU)
// Exchange buffer of one rank (cudaMalloc'ed, IPC-mapped into every peer):
//   [0]      u64 epoch        number of exchanges this rank has completed (local use)
//   [64]     u32 flags[2][8]  flags[parity][q] = epoch + 1 once rank q's contribution for that epoch has landed here
//   [256]    f64 slots[2][8][32]  rank q's packed normal equations
#define MLOAM_P2P_MAX_RANKS 8
#define MLOAM_P2P_BYTES 8192
struct P2PView {
  double *slots[MLOAM_P2P_MAX_RANKS];     // per rank: its buffer's slots[2][8][32]
  unsigned *flags[MLOAM_P2P_MAX_RANKS];   // per rank: its buffer's flags[2][8]
  unsigned long long *epoch;              // local
  int nranks, rank;
};

// ------------------------------------------------------------------ LM state (device resident)
// Everything ceres::Solve keeps between iterations for one 6-dof (or 12-dof) block, plus the packed
// normal equations the reduction writes.  NE_MAX covers 12x12 (78 upper + 12 + cost + rows).
#define MLOAM_NE_MAX 92

struct LMState {
  double x[7];             // accepted pose (parameter block)
  double xc[7];            // candidate pose being evaluated
  double H[36];            // loss-corrected J^T J at x
  double g[6];             // loss-corrected J^T r at x
  double cost;             // 1/2 sum rho at x
  double scale[6];         // Jacobi scaling, fixed at iteration 0
  double diag[6];          // LM diagonal (clamped, on the scaled system)
  double radius, decrease_factor;
  double model_cost_change;
  double x_norm;
  double V_update[36];     // PoseLocalParameterization::V_update_
  double eig[6];
  double H0[36];           // J^T J at the start of the Solve (evalHessian)
  double initial_cost;
  int is_degenerate;
  int reuse_diagonal;
  int iteration;           // LM iterations attempted in this Solve
  int num_invalid;
  int done;                // Solve finished
  int termination;
  int total_iterations;    // over outer iterations
  int rows;                // residual rows of the last evaluation
  int n_valid[2];          // matched corner / surf features
  int max_inner;
  int pad;
  int min_corr;            // a Solve with fewer matched features is skipped (lidar_tracker.cpp:64-68)
  int skipped;             // ... and this flag is raised
  long long dbg_cycles[4]; // SM cycles spent in lm_tail since k_lm_init: [0] stage-in + reduction, [1] state machine, [2] calls
};

}  // namespace mloam
