// tests/uncertainty_oracle.cpp — TEST INFRASTRUCTURE ONLY.  The pose-uncertainty record (include/lvo.h lvo_pose_uncertainty) on the
// CPU oracle, which is used as it is (oracle/*.hpp are included, not changed).  Built by tests/uncertainty_oracle.py with the oracle's
// flags (-O3 -ffp-contract=off: no FMA contraction, as the device TU's -fmad=false).
//
//   * the information of a solve: J^T J of the Huber-corrected rows at the solve's final x, in the solver tangent u = (delta, dt),
//     from the oracle's own evaluation (ceres_lm.hpp evaluate), rows summed in row order;
//   * the pipeline's record of each stage: LaserOdometry::process / LaserMapping::process call `solve(factors, x, lm, trace)`
//     unqualified from non-const members with non-const arguments.  The overload below, declared before those headers, takes the
//     arguments as non-const references and is therefore the better match there; it calls the oracle's solve and keeps the factors'
//     count, the final cost and the information at the final pose.  The last outer iteration of a frame overwrites the others;
//   * the derived fields, operation for operation what lidar-visual-odometry_b200/csrc/lvo_solver.cuh computes (sym_eigen_dev<N>,
//     pose_uncertainty_derive), so that the same information matrix gives the same bits on both sides.
#include "common.hpp"
#include "knn.hpp"
#include "voxel_grid.hpp"
#include "scan_registration.hpp"
#include "ceres_lm.hpp"

#include <algorithm>
#include <utility>

namespace lvo_oracle {

struct UncRecord {
  int solved = 0, n_factors = 0;
  double cost = 0;
  double H[21] = {0};
};

// J^T J of the corrected rows at x (upper triangle, row-major), rows in order
inline void information_at(const std::vector<Factor>& F, const double* x, double huber, double* H21) {
  Evaluation e;
  evaluate(F, x, huber, true, e);
  for (int t = 0; t < 21; ++t) H21[t] = 0.0;
  for (size_t i = 0; i < e.r.size(); ++i) {
    const double* J = &e.J[i * 6];
    int t = 0;
    for (int a = 0; a < 6; ++a)
      for (int c = a; c < 6; ++c) H21[t++] += J[a] * J[c];
  }
}

// the record the overload below writes (set by the caller around odometry / mapping)
inline UncRecord*& current_record() { static UncRecord* r = nullptr; return r; }

inline LmSummary solve(std::vector<Factor>& F, double* x, LmOptions& opt, std::vector<LmTraceRow>* trace) {
  const LmSummary s = solve(static_cast<const std::vector<Factor>&>(F), x, static_cast<const LmOptions&>(opt), trace);
  if (UncRecord* r = current_record()) {
    r->solved = 1;
    r->n_factors = (int)F.size();
    r->cost = s.final_cost;
    if (F.empty()) std::fill(r->H, r->H + 21, 0.0);
    else information_at(F, x, opt.huber, r->H);
  }
  return s;
}

}  // namespace lvo_oracle

#include "laser_odometry.hpp"
#include "laser_mapping.hpp"

using namespace lvo_oracle;

namespace {

// cyclic Jacobi, as sym_eigen_dev<N>: eigenvalues ascending (stable insertion sort), eigenvectors in the columns of V (row-major)
template <int N>
void sym_eigen(const double* M, double* w, double* V) {
  double a[N][N], v[N][N];
  for (int r = 0; r < N; ++r) for (int c = 0; c < N; ++c) { a[r][c] = M[r * N + c]; v[r][c] = r == c ? 1.0 : 0.0; }
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int p = 0; p < N - 1; ++p)
      for (int q = p + 1; q < N; ++q) off += a[p][q] * a[p][q];
    for (int p = 0; p < N; ++p) diag += a[p][p] * a[p][p];
    if (off <= 1e-32 * diag || off == 0.0) break;
    for (int p = 0; p < N - 1; ++p)
      for (int q = p + 1; q < N; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < N; ++k) { const double akp = a[k][p], akq = a[k][q]; a[k][p] = c * akp - s * akq; a[k][q] = s * akp + c * akq; }
        for (int k = 0; k < N; ++k) { const double apk = a[p][k], aqk = a[q][k]; a[p][k] = c * apk - s * aqk; a[q][k] = s * apk + c * aqk; }
        for (int k = 0; k < N; ++k) { const double vkp = v[k][p], vkq = v[k][q]; v[k][p] = c * vkp - s * vkq; v[k][q] = s * vkp + c * vkq; }
      }
  }
  double e[N]; int ord[N];
  for (int i = 0; i < N; ++i) { e[i] = a[i][i]; ord[i] = i; }
  for (int i = 1; i < N; ++i)
    for (int j = i; j > 0 && e[j] < e[j - 1]; --j) { std::swap(e[j], e[j - 1]); std::swap(ord[j], ord[j - 1]); }
  for (int c = 0; c < N; ++c) { w[c] = e[c]; for (int r = 0; r < N; ++r) V[r * N + c] = v[r][ord[c]]; }
}

// from an information matrix in p = (t, theta): eigenvectors with their largest-magnitude entry positive (first on ties), covariance
// V diag(1 / lambda) V^T when lambda_min > 0 and lambda_min >= 1e-14 lambda_max, else zero
void derive_p(const double* info, double* cov, double* w, double* V, int* pd) {
  sym_eigen<6>(info, w, V);
  for (int c = 0; c < 6; ++c) {
    int m = 0;
    for (int r = 1; r < 6; ++r) if (fabs(V[r * 6 + c]) > fabs(V[m * 6 + c])) m = r;
    if (V[m * 6 + c] < 0.0) for (int r = 0; r < 6; ++r) V[r * 6 + c] = -V[r * 6 + c];
  }
  *pd = (w[0] > 0.0 && w[0] >= 1e-14 * w[5]) ? 1 : 0;
  double inv[6];
  for (int k = 0; k < 6; ++k) inv[k] = *pd ? 1.0 / w[k] : 0.0;
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) {
      double s = 0.0;
      for (int k = 0; k < 6; ++k) s += (V[i * 6 + k] * inv[k]) * V[j * 6 + k];
      cov[i * 6 + j] = s; cov[j * 6 + i] = s;
    }
}
// from H_u in the tangent (delta, dt): p = M u, theta = 2 delta, so H_p = M^-T H_u M^-1 (blocks H_tt, H_t,delta / 2, H_delta,delta / 4)
void derive_u(const double* Hu21, double* info, double* cov, double* w, double* V, int* pd) {
  double Hu[6][6];
  int t = 0;
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) { Hu[i][j] = Hu21[t]; Hu[j][i] = Hu21[t]; ++t; }
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 6; ++j) info[i * 6 + j] = Hu[i < 3 ? i + 3 : i - 3][j < 3 ? j + 3 : j - 3] * ((i < 3 ? 1.0 : 0.5) * (j < 3 ? 1.0 : 0.5));
  derive_p(info, cov, w, V, pd);
}

Factor factor_of(const double* p, double s) {
  Factor f;
  f.type = (int)p[0];
  f.c = Vec3{p[1], p[2], p[3]}; f.a = Vec3{p[4], p[5], p[6]}; f.b = Vec3{p[7], p[8], p[9]}; f.m = Vec3{p[10], p[11], p[12]};
  f.d = p[13]; f.s = s;
  return f;
}

// extract -> odometry -> mapping every skip_frame-th frame, as lvo_oracle_step (oracle/capi.cpp) chains them, with the two records
struct Pipeline {
  int n_scans = 64, skip_frame = 1, frame_count = 0;
  double min_range = 5.0;
  ScanRegOut reg;
  LaserOdometry odo;
  LaserMapping map;
  Cloud registered;
  UncRecord rec[2];
};

}  // namespace

extern "C" {

// derived fields from an information matrix in p (info36), or from H_u (Hu21; info36 is then an output)
void unc_from_info(const double* info36, double* cov36, double* w6, double* V36, int* pd) { derive_p(info36, cov36, w6, V36, pd); }
void unc_from_hu(const double* Hu21, double* info36, double* cov36, double* w6, double* V36, int* pd) { derive_u(Hu21, info36, cov36, w6, V36, pd); }

// the oracle's LM solve of nf factors (14 doubles each as lvo_oracle_solve; s[nf] interpolation ratios or null = 1), x[7] in / out;
// Hu21 gets the information at the final x and *cost the final cost
void unc_solve(const double* f, const double* s, long nf, double* x, int max_iters, double huber, double* Hu21, double* cost) {
  std::vector<Factor> F;
  for (long i = 0; i < nf; ++i) F.push_back(factor_of(f + i * 14, s ? s[i] : 1.0));
  LmOptions o; o.max_num_iterations = max_iters; o.huber = huber;
  UncRecord r;
  current_record() = &r;
  solve(F, x, o, nullptr);
  current_record() = nullptr;
  for (int k = 0; k < 21; ++k) Hu21[k] = r.H[k];
  *cost = r.cost;
}

void* unc_pipeline_create(int n_scans, double min_range, double line_res, double plane_res, int outer, int lm_iters, double huber, int distortion,
                          int skip_frame) {
  Pipeline* p = new Pipeline();
  p->n_scans = n_scans; p->min_range = min_range; p->skip_frame = skip_frame < 1 ? 1 : skip_frame;
  p->odo.outer_iters = outer; p->odo.lm.max_num_iterations = lm_iters; p->odo.lm.huber = huber; p->odo.distortion = distortion;
  p->map.outer_iters = outer; p->map.lm.max_num_iterations = lm_iters; p->map.lm.huber = huber;
  p->map.lineRes = (float)line_res; p->map.planeRes = (float)plane_res;
  return p;
}
void unc_pipeline_destroy(void* h) { delete (Pipeline*)h; }

// one frame; returns 1 if the frame was mapped.  A stage that does not solve on its frame (first odometry frame, map too small) leaves
// solved = 0; a frame that does not map leaves the mapping record as it was.
int unc_pipeline_step(void* h, const Pt* in, long n) {
  Pipeline* p = (Pipeline*)h;
  scan_registration(in, (size_t)n, p->n_scans, p->min_range, p->reg);
  p->rec[0] = UncRecord();
  current_record() = &p->rec[0];
  p->odo.process(p->reg.sharp, p->reg.lessSharp, p->reg.flat, p->reg.lessFlat, false, &p->reg.full);
  const bool do_map = (p->frame_count % p->skip_frame) == 0;   // laserOdometry.cpp:643
  if (do_map) {
    p->frame_count = 0;
    p->rec[1] = UncRecord();
    current_record() = &p->rec[1];
    p->map.process(p->odo.laserCloudCornerLast, p->odo.laserCloudSurfLast, p->odo.distortion == 2 ? &p->odo.fullOut : &p->reg.full, p->odo.q_w_curr,
                   p->odo.t_w_curr, &p->registered, false);
  }
  current_record() = nullptr;
  p->frame_count++;
  return do_map ? 1 : 0;
}

// the record of stage 0 (odometry) or 1 (mapping): ints3 = [solved, positive_definite, n_factors]; zero information when not solved
void unc_pipeline_record(void* h, int stage, int* ints3, double* cost, double* Hu21, double* info36, double* cov36, double* w6, double* V36) {
  const UncRecord& u = ((Pipeline*)h)->rec[stage ? 1 : 0];
  ints3[0] = u.solved; ints3[2] = u.solved ? u.n_factors : 0;
  *cost = u.solved ? u.cost : 0.0;
  for (int k = 0; k < 21; ++k) Hu21[k] = u.solved ? u.H[k] : 0.0;
  derive_u(Hu21, info36, cov36, w6, V36, &ints3[1]);
}

}  // extern "C"
