// lvo_solver.cuh — residual / Jacobian evaluation, J^T W J accumulation and the Levenberg-Marquardt loop, i.e. what
// `ceres::Solve` does for the reference's problems (src/laserOdometry.cpp:369-376,571-576; src/laserMapping.cpp:
// 565-572,712-720) with the residual semantics of src/lidarFactor.hpp:12-138.
//
//   * residuals and ANALYTIC local Jacobians of LidarEdgeFactor / LidarPlaneFactor / LidarPlaneNormFactor
//     (d r/d t = d r/d p ; d r/d delta = d r/d p * (-2 [R c]_x) for Ceres' EigenQuaternionParameterization, whose Plus
//     is q_delta * q with delta the half rotation vector — SURVEY §8a A14-A17);
//   * ceres::HuberLoss(0.1) + Corrector (rho'' <= 0 branch): rows scaled by sqrt(rho'), cost = sum rho / 2 (A18);
//   * block-reduced 6x6 J^T W J (21 unique), J^T r (6) and cost in double: fixed-shape tree (warp shuffles, then a
//     fixed-order sum over warps) => bitwise deterministic, no float atomics;
//   * the trust-region loop of Ceres 1.12 defaults (LEVENBERG_MARQUARDT, DENSE_QR, Jacobi scaling frozen at
//     iteration 0, radius 1e4, min_relative_decrease 1e-3, function / parameter / gradient tolerances, the candidate
//     discarded when a tolerance fires, rejected and invalid steps counted as iterations — A19) run by thread 0 in
//     double.  The damped 6x6 system is solved from the normal equations (Cholesky) instead of a QR of the stacked
//     Jacobian: same minimiser, difference O(cond * eps), far below the 1e-4 m / 1e-5 rad pose tolerance.
// One CTA of LVO_LM_THREADS threads per lane runs the WHOLE inner loop (<= max_iters evaluations of all factors) without returning to
// the host: the threads stride over the lane's factor slots, 28 doubles are reduced by warp shuffles and then across the warps in rank
// order through shared memory (bitwise deterministic), thread 0 takes the trust-region decision and publishes the next evaluation
// point.  (Round 1 spread a lane over a cluster of up to 8 CTAs with DSMEM reductions; two cluster barriers per evaluation cost more
// than the extra SMs gave once every SM had a lane of its own.)
// Each LM iteration costs one pass over the factors because cost, J^T W J and J^T r at the candidate are accumulated
// together (if the step is accepted they are the next iteration's system).
#pragma once
#include "lvo_internal.h"
#include <float.h>

#ifndef LVO_LM_THREADS
#define LVO_LM_THREADS 384     // one CTA per lane: 12 warps x <= 170 registers, no spills; block barriers instead of cluster barriers
#endif
#ifndef LVO_LM_MINB
#define LVO_LM_MINB 1
#endif
#define LVO_NACC 28  // 21 + 6 + 1

// ---- small dense routines (double) ---------------------------------------------------------------------------
// cyclic Jacobi for a symmetric 3x3; eigenvalues ascending in w, eigenvectors in the columns of V (row-major)
__device__ inline void sym_eigen3_dev(const double M[9], double w[3], double V[9]) {
  double a[3][3], v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) a[r][c] = M[r * 3 + c];
  for (int sweep = 0; sweep < 64; ++sweep) {
    const double off = a[0][1] * a[0][1] + a[0][2] * a[0][2] + a[1][2] * a[1][2];
    const double diag = a[0][0] * a[0][0] + a[1][1] * a[1][1] + a[2][2] * a[2][2];
    if (off <= 1e-32 * diag || off == 0.0) break;
#pragma unroll
    for (int p = 0; p < 2; ++p)
#pragma unroll
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
#pragma unroll
        for (int k = 0; k < 3; ++k) { const double akp = a[k][p], akq = a[k][q]; a[k][p] = c * akp - s * akq; a[k][q] = s * akp + c * akq; }
#pragma unroll
        for (int k = 0; k < 3; ++k) { const double apk = a[p][k], aqk = a[q][k]; a[p][k] = c * apk - s * aqk; a[q][k] = s * apk + c * aqk; }
#pragma unroll
        for (int k = 0; k < 3; ++k) { const double vkp = v[k][p], vkq = v[k][q]; v[k][p] = c * vkp - s * vkq; v[k][q] = s * vkp + c * vkq; }
      }
  }
  int o0 = 0, o1 = 1, o2 = 2;
  double e0 = a[0][0], e1 = a[1][1], e2 = a[2][2];
  // stable 3-element sort by eigenvalue
  if (e1 < e0) { double t = e0; e0 = e1; e1 = t; int ti = o0; o0 = o1; o1 = ti; }
  if (e2 < e1) { double t = e1; e1 = e2; e2 = t; int ti = o1; o1 = o2; o2 = ti; }
  if (e1 < e0) { double t = e0; e0 = e1; e1 = t; int ti = o0; o0 = o1; o1 = ti; }
  w[0] = e0; w[1] = e1; w[2] = e2;
  const int ord[3] = {o0, o1, o2};
  for (int c = 0; c < 3; ++c) for (int r = 0; r < 3; ++r) V[r * 3 + c] = v[r][ord[c]];
}

// least squares min ||A y - b|| for a 5x3 A by Householder QR (A, b destroyed)
__device__ inline bool lsq_qr_5x3(double A[15], double b[5], double y[3]) {
  const int m = 5, n = 3;
  for (int k = 0; k < n; ++k) {
    double norm = 0;
    for (int i = k; i < m; ++i) norm += A[i * n + k] * A[i * n + k];
    norm = sqrt(norm);
    if (norm == 0.0) return false;
    const double alpha = A[k * n + k] > 0 ? -norm : norm;
    const double v0 = A[k * n + k] - alpha;
    double vtv = v0 * v0;
    for (int i = k + 1; i < m; ++i) vtv += A[i * n + k] * A[i * n + k];
    if (vtv == 0.0) return false;
    for (int j = k + 1; j < n; ++j) {
      double dot = v0 * A[k * n + j];
      for (int i = k + 1; i < m; ++i) dot += A[i * n + k] * A[i * n + j];
      const double f = 2.0 * dot / vtv;
      A[k * n + j] -= f * v0;
      for (int i = k + 1; i < m; ++i) A[i * n + j] -= f * A[i * n + k];
    }
    {
      double dot = v0 * b[k];
      for (int i = k + 1; i < m; ++i) dot += A[i * n + k] * b[i];
      const double f = 2.0 * dot / vtv;
      b[k] -= f * v0;
      for (int i = k + 1; i < m; ++i) b[i] -= f * A[i * n + k];
    }
    A[k * n + k] = alpha;
  }
  for (int k = n - 1; k >= 0; --k) {
    double s = b[k];
    for (int j = k + 1; j < n; ++j) s -= A[k * n + j] * y[j];
    y[k] = s / A[k * n + k];
  }
  return true;
}

// Cholesky solve of a 6x6 SPD system (A full row-major, destroyed).  false if not positive definite.
// Fully unrolled and division-free apart from one reciprocal square root per pivot: this runs on ONE thread while the
// rest of the CTA waits, so its dependent-latency chain is the critical path of every LM iteration.
__device__ __forceinline__ bool chol6_solve(double A[36], const double b[6], double y[6]) {
  double inv[6];
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double d = A[j * 6 + j];
#pragma unroll
    for (int k = 0; k < j; ++k) d -= A[j * 6 + k] * A[j * 6 + k];
    if (!(d > 0.0)) return false;
    const double r = rsqrt(d);
    inv[j] = r;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double s = A[i * 6 + j];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= A[i * 6 + k] * A[j * 6 + k];
      A[i * 6 + j] = s * r;
    }
  }
  double z[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double s = b[i];
#pragma unroll
    for (int k = 0; k < i; ++k) s -= A[i * 6 + k] * z[k];
    z[i] = s * inv[i];
  }
#pragma unroll
  for (int i = 5; i >= 0; --i) {
    double s = z[i];
#pragma unroll
    for (int k = i + 1; k < 6; ++k) s -= A[k * 6 + i] * y[k];
    y[i] = s * inv[i];
  }
  return true;
}

// EigenQuaternionParameterization::Plus on the q block, plain addition on t
__device__ inline void plus7_dev(const double* x, const double* delta, double* xp) {
  const double nd = sqrt(delta[0] * delta[0] + delta[1] * delta[1] + delta[2] * delta[2]);
  if (nd > 0.0) {
    const double s = sin(nd) / nd;
    const double dq[4] = {s * delta[0], s * delta[1], s * delta[2], cos(nd)};
    quat_mul(dq, x, xp);
  } else {
    xp[0] = x[0]; xp[1] = x[1]; xp[2] = x[2]; xp[3] = x[3];
  }
  xp[4] = x[4] + delta[3]; xp[5] = x[5] + delta[4]; xp[6] = x[6] + delta[5];
}

// ---- one residual block: accumulate rho' * J^T J (upper triangle), rho' * J^T r, rho / 2 --------------------------
// DISTORT: the factor carries an interpolation ratio s (f.d) that may differ from 1 (DISTORTION 1, laserOdometry.cpp:455-459):
// lp = slerp(Identity, q; s) * c + s t, lidarFactor.hpp:27-33 / :79-85.  The 3x4 Jacobian d lp / d(qx,qy,qz,qw) is taken through the
// functor as written (the slerp weights depend on q.w; Eigen's v + w uv + u x uv, uv = 2 u x v, differentiated without assuming a
// unit quaternion) and multiplied by the 4x3 plus-Jacobian of EigenQuaternionParameterization (SURVEY A17).
__device__ __forceinline__ d3 interp_point_jacobian(const double* x, double s, const d3& c, double Jl[3][6]) {
  const SlerpW k = slerp_identity_weights(x[3], s, true);
  const double u[3] = {k.scale1 * x[0], k.scale1 * x[1], k.scale1 * x[2]};
  const double ws = k.scale0 + k.scale1 * x[3];
  const double qs[4] = {u[0], u[1], u[2], ws};
  const d3 rc = quat_rotate(qs, c);
  const double cv[3] = {c.x, c.y, c.z};
  const double uc = u[0] * cv[0] + u[1] * cv[1] + u[2] * cv[2];
  const double cx[3][3] = {{0, -c.z, c.y}, {c.z, 0, -c.x}, {-c.y, c.x, 0}};
  const d3 b2 = d3cross(d3{u[0], u[1], u[2]}, c);
  const double bw[3] = {2.0 * b2.x, 2.0 * b2.y, 2.0 * b2.z};
  const double dws_dw = k.ds0_dw + k.ds1_dw * x[3] + k.scale1;
  const double P[4][3] = {{x[3], x[2], -x[1]}, {-x[2], x[3], x[0]}, {x[1], -x[0], x[3]}, {-x[0], -x[1], -x[2]}};
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double A[3], G[4];
#pragma unroll
    for (int j = 0; j < 3; ++j) A[j] = -2.0 * ws * cx[i][j] + 2.0 * ((i == j ? uc : 0.0) + u[i] * cv[j] - 2.0 * cv[i] * u[j]);
#pragma unroll
    for (int j = 0; j < 3; ++j) G[j] = A[j] * k.scale1;
    G[3] = (A[0] * x[0] + A[1] * x[1] + A[2] * x[2]) * k.ds1_dw + bw[i] * dws_dw;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      Jl[i][j] = G[0] * P[0][j] + G[1] * P[1][j] + G[2] * P[2][j] + G[3] * P[3][j];
      Jl[i][3 + j] = i == j ? s : 0.0;
    }
  }
  return d3{rc.x + s * x[4], rc.y + s * x[5], rc.z + s * x[6]};
}

template <bool DISTORT>
__device__ __forceinline__ void accumulate_factor(const LvoFactor& f, const double* x, double huber, double* acc) {
  // Corrector weight of a block with squared norm s (A18); adds rho / 2 to the cost
  auto loss = [&](double s) -> double {
    const double b = huber * huber;
    double rho0, rho1;
    if (s > b) { const double rr = sqrt(s); rho0 = 2 * huber * rr - b; rho1 = fmax(DBL_MIN, huber / rr); }
    else { rho0 = s; rho1 = 1.0; }
    acc[27] += 0.5 * rho0;
    return rho1;
  };
  // one Jacobian row: every index below is a compile-time constant, so J rows and accumulators stay in registers (a row loop with
  // a run-time trip count puts them in local memory).  Explicit FMAs: the TU is compiled with -fmad=false for the float paths
  // that must match the x86 reference bit for bit; these double sums are ordered differently from Ceres anyway (DESIGN.md 2).
  auto add_row = [&](const double (&Jr)[6], double ri, double rho1) {
    int t = 0;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
      const double wa = rho1 * Jr[a];
#pragma unroll
      for (int c = a; c < 6; ++c) { acc[t] = fma(wa, Jr[c], acc[t]); ++t; }
      acc[21 + a] = fma(wa, ri, acc[21 + a]);
    }
  };
  if (DISTORT && f.type <= 1 && f.d != 1.0) {
    double Jl[3][6];
    const d3 lp = interp_point_jacobian(x, f.d, d3{f.c[0], f.c[1], f.c[2]}, Jl);
    if (f.type == 0) {
      // (lp - a) x (lp - b) / |a - b| = (lp - a) x e with e = (a - b) / |a - b| = f.b (lvo_internal.h); d r / d lp = -[e]x
      const d3 u{lp.x - f.a[0], lp.y - f.a[1], lp.z - f.a[2]}, e{f.b[0], f.b[1], f.b[2]};
      const d3 nu = d3cross(u, e);
      const double r[3] = {nu.x, nu.y, nu.z};
      const double rho1 = loss(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
      const double D[3][3] = {{0, e.z, -e.y}, {-e.z, 0, e.x}, {e.y, -e.x, 0}};
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        double Jr[6];
#pragma unroll
        for (int c = 0; c < 6; ++c) Jr[c] = D[i][0] * Jl[0][c] + D[i][1] * Jl[1][c] + D[i][2] * Jl[2][c];
        add_row(Jr, r[i], rho1);
      }
    } else {
      const double r0 = (lp.x - f.a[0]) * f.b[0] + (lp.y - f.a[1]) * f.b[1] + (lp.z - f.a[2]) * f.b[2];
      const double rho1 = loss(r0 * r0);
      double Jr[6];
#pragma unroll
      for (int c = 0; c < 6; ++c) Jr[c] = f.b[0] * Jl[0][c] + f.b[1] * Jl[1][c] + f.b[2] * Jl[2][c];
      add_row(Jr, r0, rho1);
    }
    return;
  }
  const d3 rc = quat_rotate(x, d3{f.c[0], f.c[1], f.c[2]});
  const d3 lp{rc.x + x[4], rc.y + x[5], rc.z + x[6]};
  if (f.type == 0) {
    const d3 u{lp.x - f.a[0], lp.y - f.a[1], lp.z - f.a[2]}, e{f.b[0], f.b[1], f.b[2]};
    const d3 nu = d3cross(u, e);
    const double r[3] = {nu.x, nu.y, nu.z};
    const double rho1 = loss(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
    const double D[3][3] = {{0, e.z, -e.y}, {-e.z, 0, e.x}, {e.y, -e.x, 0}};
    const double Jp[3][3] = {{0, 2 * rc.z, -2 * rc.y}, {-2 * rc.z, 0, 2 * rc.x}, {2 * rc.y, -2 * rc.x, 0}};
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      double Jr[6];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        Jr[c] = D[i][0] * Jp[0][c] + D[i][1] * Jp[1][c] + D[i][2] * Jp[2][c];
        Jr[3 + c] = D[i][c];
      }
      add_row(Jr, r[i], rho1);
    }
  } else {
    double n[3], r0;
    if (f.type == 1) {  // LidarPlaneFactor: b holds ljm_norm
      n[0] = f.b[0]; n[1] = f.b[1]; n[2] = f.b[2];
      r0 = (lp.x - f.a[0]) * n[0] + (lp.y - f.a[1]) * n[1] + (lp.z - f.a[2]) * n[2];
    } else {            // LidarPlaneNormFactor
      n[0] = f.a[0]; n[1] = f.a[1]; n[2] = f.a[2];
      r0 = (n[0] * lp.x + n[1] * lp.y + n[2] * lp.z) + f.d;
    }
    const double rho1 = loss(r0 * r0);
    // n^T * (-2 [rc]_x)
    const double Jr[6] = {-2 * (n[1] * rc.z - n[2] * rc.y), -2 * (n[2] * rc.x - n[0] * rc.z), -2 * (n[0] * rc.y - n[1] * rc.x), n[0], n[1], n[2]};
    add_row(Jr, r0, rho1);
  }
}

struct SolveArgs {
  LaneState* ls;
  const LvoFactor* factors;   // [lanes][factor_cap]
  int factor_cap;
  int which;                  // 0 = odometry (x = para_q,para_t), 1 = mapping (x = map_x)
  int outer;                  // outer iteration index (trace / stats slot)
  int max_iters;
  double huber;
  double* trace;              // [lanes][LVO_MAX_OUTER][LVO_MAX_LM + 1][LVO_TRACE_W] or null
  int distort;                // != 0: factors may carry an interpolation ratio s != 1 (scan-to-scan with DISTORTION 1)
  int n_outer;                // outer iterations of the frame (stats slots to fill when the loop is cut short)
  int fixpoint_skip;          // LVO_OPT_FIXPOINT_SKIP
  int* reset_cnt;             // [lanes] or null: per-lane counter the solve zeroes for the next outer iteration (the scan-to-scan slow-list length)
};

struct LmShared {
  double red[LVO_LM_THREADS / 32][LVO_NACC];
  double sum[LVO_NACC];      // reduced accumulators of the last evaluation
  double xeval[7];           // point to evaluate next
  int ctrl;                  // 0 = evaluate xeval, 1 = finished
};

// All threads of the CTA call this; afterwards sh.sum holds the sums over all factors of the lane (fixed summation tree:
// per-thread strided partial sums, warp shuffle tree, warps in rank order => bitwise deterministic).
template <bool DISTORT>
__device__ __forceinline__ void lm_evaluate(const SolveArgs& a, const LvoFactor* __restrict__ F, int nslots, const double* x, LmShared& sh) {
  double acc[LVO_NACC];
#pragma unroll
  for (int i = 0; i < LVO_NACC; ++i) acc[i] = 0.0;
  double xl[7];
#pragma unroll
  for (int i = 0; i < 7; ++i) xl[i] = x[i];
  for (int s = threadIdx.x; s < nslots; s += LVO_LM_THREADS) {
    const LvoFactor f = F[s];
    if (f.type >= 0) accumulate_factor<DISTORT>(f, xl, a.huber, acc);
  }
  const unsigned ln = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < LVO_NACC; ++i) {
    double v = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if (ln == 0) sh.red[w][i] = v;
  }
  __syncthreads();
  if (threadIdx.x < LVO_NACC) {
    double v = 0;
#pragma unroll
    for (int ww = 0; ww < LVO_LM_THREADS / 32; ++ww) v += sh.red[ww][threadIdx.x];
    sh.sum[threadIdx.x] = v;
  }
  __syncthreads();
}
// thread 0: publish the next evaluation point / the stop flag
__device__ __forceinline__ void lm_broadcast(LmShared& sh, const double* xc, bool go) {
  if (go) for (int i = 0; i < 7; ++i) sh.xeval[i] = xc[i];
  sh.ctrl = go ? 0 : 1;
}

// State of the trust-region loop, owned by thread 0.
struct LmCtl {
  double x[7], x0[7], H[21], g[6], cost, x_norm;
  double scale[6], diag[6], radius, decrease;
  double xc[7], model_cost_change;
  bool reuse_diag;
  int iter, invalid_run, nfactors;
};

__device__ __noinline__ double gradient_max_norm_dev(const double* x, const double* g) {
  // || x - Plus(x, -g) ||_inf.  The translation block of Plus is a plain addition, so its entries of the difference are
  // |g_t| exactly: if one of them already exceeds the tolerance the test "<= 1e-10" is decided without the quaternion
  // exponential (sin / cos in double on the one thread everybody waits for).
  const double gt = fmax(fabs(g[3]), fmax(fabs(g[4]), fabs(g[5])));
  if (gt > 1e-10) return gt;
  double ng[6], xp[7];
  for (int c = 0; c < 6; ++c) ng[c] = -g[c];
  plus7_dev(x, ng, xp);
  double m = 0;
  for (int i = 0; i < 7; ++i) m = fmax(m, fabs(x[i] - xp[i]));
  return m;
}
__device__ inline void lm_trace(const SolveArgs& a, int lane, int row, const double* x, double cost, double radius, int flags) {
  if (!a.trace || row > LVO_MAX_LM) return;
  double* t = a.trace + (((size_t)lane * LVO_MAX_OUTER + a.outer) * (LVO_MAX_LM + 1) + row) * LVO_TRACE_W;
  for (int i = 0; i < 7; ++i) t[i] = x[i];
  t[7] = cost; t[8] = radius; t[9] = (double)flags;
}
// Computes the next candidate (looping over invalid steps).  Returns true if a candidate must be evaluated.
__device__ __noinline__ bool lm_next_step(const SolveArgs& a, int lane, LmCtl& c) {
  const int idx[6][6] = {{0, 1, 2, 3, 4, 5}, {1, 6, 7, 8, 9, 10}, {2, 7, 11, 12, 13, 14}, {3, 8, 12, 15, 16, 17}, {4, 9, 13, 16, 18, 19}, {5, 10, 14, 17, 19, 20}};
  while (true) {
    if (c.iter >= a.max_iters) return false;  // NO_CONVERGENCE
    c.iter++;
    if (!c.reuse_diag)
      for (int i = 0; i < 6; ++i) c.diag[i] = fmin(fmax(c.scale[i] * c.scale[i] * c.H[idx[i][i]], 1e-6), 1e32);
    double A[36], SHS[36], b[6], y[6];
    for (int i = 0; i < 6; ++i) {
      for (int j = 0; j < 6; ++j) { SHS[i * 6 + j] = c.scale[i] * c.H[idx[i][j]] * c.scale[j]; A[i * 6 + j] = SHS[i * 6 + j]; }
      A[i * 6 + i] += c.diag[i] / c.radius;
      b[i] = c.scale[i] * c.g[i];
    }
    c.reuse_diag = true;
    bool valid = chol6_solve(A, b, y);
    double step[6];
    if (valid) for (int i = 0; i < 6; ++i) { step[i] = -y[i]; if (!isfinite(step[i])) valid = false; }
    if (valid) {
      double lin = 0, quad = 0;
      for (int i = 0; i < 6; ++i) {
        lin += step[i] * b[i];
        double t = 0;
        for (int j = 0; j < 6; ++j) t += SHS[i * 6 + j] * step[j];
        quad += step[i] * t;
      }
      c.model_cost_change = -lin - 0.5 * quad;
      if (!(c.model_cost_change > 0.0)) valid = false;
    }
    if (!valid) {
      const bool stop = ++c.invalid_run >= 5;
      if (!stop) { c.radius = c.radius / c.decrease; c.decrease *= 2.0; c.reuse_diag = true; }
      lm_trace(a, lane, c.iter, c.x, c.cost, c.radius, 0);
      if (stop || c.radius < 1e-32) return false;
      continue;
    }
    c.invalid_run = 0;
    double delta[6];
    for (int i = 0; i < 6; ++i) delta[i] = step[i] * c.scale[i];
    plus7_dev(c.x, delta, c.xc);
    return true;
  }
}

template <bool DISTORT>
__global__ void __launch_bounds__(LVO_LM_THREADS, LVO_LM_MINB) k_lm_solve(SolveArgs a) {
  __shared__ LmShared sh;
  __shared__ LmCtl ctl;  // only thread 0 touches it; shared to keep it out of its registers
  const bool lead = threadIdx.x == 0;
  const int lane = blockIdx.x;
  LaneState& s = a.ls[lane];
  if (a.reset_cnt && threadIdx.x == 0) a.reset_cnt[lane] = 0;   // the association kernels of this iteration are through with it
  if (a.which == 0 ? (s.odo_inited == 0 || s.odo_done != 0) : (s.map_too_small != 0 || s.map_done != 0)) return;
  const int nslots = a.which == 0 ? (s.n_sharp + s.n_flat) : (s.n_stack[0] + s.n_stack[1]);
  const LvoFactor* F = a.factors + (size_t)lane * a.factor_cap;
  double* xg = a.which == 0 ? s.para_q : s.map_x;  // para_q[4], para_t[3] are contiguous
  if (threadIdx.x < 7) sh.xeval[threadIdx.x] = xg[threadIdx.x];
  __syncthreads();
  lm_evaluate<DISTORT>(a, F, nslots, sh.xeval, sh);
  if (lead) {
    LmCtl& c = ctl;
    for (int i = 0; i < 7; ++i) c.x[i] = c.x0[i] = sh.xeval[i];
    for (int i = 0; i < 21; ++i) c.H[i] = sh.sum[i];
    for (int i = 0; i < 6; ++i) c.g[i] = sh.sum[21 + i];
    c.cost = sh.sum[27];
    c.iter = 0; c.invalid_run = 0; c.radius = 1e4; c.decrease = 2.0; c.reuse_diag = false;
    const int dg[6] = {0, 6, 11, 15, 18, 20};
    for (int i = 0; i < 6; ++i) c.scale[i] = 1.0 / (1.0 + sqrt(c.H[dg[i]]));
    double xn = 0; for (int i = 0; i < 7; ++i) xn += c.x[i] * c.x[i];
    c.x_norm = sqrt(xn);
    int nf = a.which == 0 ? (s.stats.odo_corner_corr[a.outer] + s.stats.odo_plane_corr[a.outer]) : (s.stats.map_corner_corr[a.outer] + s.stats.map_surf_corr[a.outer]);
    c.nfactors = nf;
    bool go = false;
    if (nf == 0) {
      lm_trace(a, lane, 0, c.x, 0.0, c.radius, 32);
    } else {
      const bool gconv = gradient_max_norm_dev(c.x, c.g) <= 1e-10;
      lm_trace(a, lane, 0, c.x, c.cost, c.radius, 32 | (gconv ? 16 : 0));
      if (!gconv) go = lm_next_step(a, lane, c);
    }
    lm_broadcast(sh, c.xc, go);
  }
  __syncthreads();
  while (sh.ctrl == 0) {
    lm_evaluate<DISTORT>(a, F, nslots, sh.xeval, sh);
    if (lead) {
      LmCtl& c = ctl;
      const double new_cost = sh.sum[27];
      bool go = false;
      double sn = 0; for (int i = 0; i < 7; ++i) sn += (c.x[i] - c.xc[i]) * (c.x[i] - c.xc[i]);
      const double step_norm = sqrt(sn);
      const double cost_change = c.cost - new_cost;
      if (step_norm <= 1e-8 * (c.x_norm + 1e-8)) {
        lm_trace(a, lane, c.iter, c.x, c.cost, c.radius, 1 | 4);     // parameter tolerance: candidate discarded
      } else if (fabs(cost_change) <= 1e-6 * c.cost) {
        lm_trace(a, lane, c.iter, c.x, c.cost, c.radius, 1 | 8);     // function tolerance: candidate discarded
      } else {
        const double rel = cost_change / c.model_cost_change;
        if (rel > 1e-3) {  // StepAccepted
          const double t = 2.0 * rel - 1.0;
          c.radius = fmin(1e16, c.radius / fmax(1.0 / 3.0, 1.0 - t * t * t));
          c.decrease = 2.0; c.reuse_diag = false;
          for (int i = 0; i < 7; ++i) c.x[i] = c.xc[i];
          for (int i = 0; i < 21; ++i) c.H[i] = sh.sum[i];
          for (int i = 0; i < 6; ++i) c.g[i] = sh.sum[21 + i];
          c.cost = new_cost;
          double xn = 0; for (int i = 0; i < 7; ++i) xn += c.x[i] * c.x[i];
          c.x_norm = sqrt(xn);
          const bool gconv = gradient_max_norm_dev(c.x, c.g) <= 1e-10;
          lm_trace(a, lane, c.iter, c.x, c.cost, c.radius, 1 | 2 | (gconv ? 16 : 0));
          go = !gconv;
        } else {           // StepRejected
          c.radius = c.radius / c.decrease; c.decrease *= 2.0; c.reuse_diag = true;
          lm_trace(a, lane, c.iter, c.x, c.cost, c.radius, 1);
          go = true;
        }
        if (c.radius < 1e-32) go = false;
        if (go) go = lm_next_step(a, lane, c);
      }
      lm_broadcast(sh, c.xc, go);
    }
    __syncthreads();
  }
  if (lead) {
    LmCtl& c = ctl;
    for (int i = 0; i < 7; ++i) xg[i] = c.x[i];
    // Fixed point: no step was accepted, the pose is bit for bit the one this outer iteration started from.  The next outer
    // iteration would see the same pose and the same clouds, build the same correspondences and the same problem and stop the
    // same way (every kernel on the path is deterministic), and so would all the others: their results are this iteration's.
    bool fixed = a.fixpoint_skip != 0;
    for (int i = 0; i < 7; ++i) fixed = fixed && __double_as_longlong(c.x[i]) == __double_as_longlong(c.x0[i]);
    const double fc = c.nfactors ? c.cost : 0.0;
    if (a.which == 0) {
      s.stats.odo_lm_iters[a.outer] = c.iter; s.stats.odo_final_cost[a.outer] = fc;
      s.stats.odo_outer_executed = a.outer + 1;
      if (fixed) {
        s.odo_done = 1;
        for (int o = a.outer + 1; o < a.n_outer; ++o) {
          s.stats.odo_corner_corr[o] = s.stats.odo_corner_corr[a.outer]; s.stats.odo_plane_corr[o] = s.stats.odo_plane_corr[a.outer];
          s.stats.odo_lm_iters[o] = c.iter; s.stats.odo_final_cost[o] = fc;
        }
      }
    } else {
      s.stats.map_lm_iters[a.outer] = c.iter; s.stats.map_final_cost[a.outer] = fc;
      s.stats.map_outer_executed = a.outer + 1;
      if (fixed) {
        s.map_done = 1;
        for (int o = a.outer + 1; o < a.n_outer; ++o) {
          s.stats.map_corner_corr[o] = s.stats.map_corner_corr[a.outer]; s.stats.map_surf_corr[o] = s.stats.map_surf_corr[a.outer];
          s.stats.map_lm_iters[o] = c.iter; s.stats.map_final_cost[o] = fc;
        }
      }
    }
  }
}

// one CTA per lane (max_slots is kept for the call sites; the factor loop is strided over the CTA whatever the count)
static inline void lvo_launch_lm(cudaStream_t st, const SolveArgs& sa, int lanes, int max_slots) {
  (void)max_slots;
  if (sa.distort) k_lm_solve<true><<<lanes, LVO_LM_THREADS, 0, st>>>(sa);
  else k_lm_solve<false><<<lanes, LVO_LM_THREADS, 0, st>>>(sa);
}
