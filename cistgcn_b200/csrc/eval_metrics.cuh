// Per-(sample, frame) warp work of the fused evaluation metrics, shared by eval_metrics_kernel (eval_metrics.cu) and
// eval_metrics_grouped_kernel (eval_grouped.cu).  References: environment/test.py:65-94 Metrics.compute and :125-129 the
// scatter of the used joints back into the full skeleton; losses/losses.py:50-61 mpjpe, :64-77 weighted_mpjpe, :79-144
// pa_mpjpe, :147-161 n_mpjpe, :164-179 mean_velocity_error, :200-239 bone_length_error.
#pragma once
#include <math.h>

#include "../../include/cistgcn_b200.h"
#include "simt.h"

namespace cgm {

constexpr int NT = 256, NW = NT / 32;
constexpr int MAXJ = 64;          // joints of the full skeleton (H36M 32, AMASS 18, ExPI 36)

struct Args {
  const float* pred;      // (B, To, Vu, 3) model output on the used joints
  const float* target;    // (B, To, Vf, 3) full skeleton
  const int* src_map;     // [Vf]: index into pred's joints, or -1 = keep the target's joint (environment/test.py:125-129)
  const int* bones;       // [NB][2] joint pairs of the full skeleton, or NULL
  const float* wt[2];     // optional per-joint weights (B, To, Vf) for two weighted_mpjpe variants
  float* assembled;       // optional (B, To, Vf, 3): pred scattered into the full skeleton
  double* sums;           // [CISTGCN_METRIC_COUNT][To], accumulated
  long long B;
  int To, Vu, Vf, NB;
};

// Jacobi eigen-decomposition of a symmetric 3x3 matrix (fp64): A = Q diag(w) Q^T
__device__ inline void jacobi3(double A[3][3], double Q[3][3], double w[3]) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) Q[i][j] = i == j ? 1.0 : 0.0;
  for (int sweep = 0; sweep < 12; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    if (off < 1e-300) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (fabs(A[p][q]) < 1e-300) continue;
        const double theta = (A[q][q] - A[p][p]) / (2.0 * A[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) {                  // A <- A J
          const double akp = A[k][p], akq = A[k][q];
          A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {                  // A <- J^T A
          const double apk = A[p][k], aqk = A[q][k];
          A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {
          const double qkp = Q[k][p], qkq = Q[k][q];
          Q[k][p] = c * qkp - s * qkq; Q[k][q] = s * qkp + c * qkq;
        }
      }
  }
  for (int i = 0; i < 3; ++i) w[i] = A[i][i];
}

// Procrustes pieces of losses.pa_mpjpe (:98-127) from H = X0^T Y0: rotation R (with the reference's reflection fix: the
// LAST ROW of V and the last singular value are multiplied by sign(det(V U^T)), :112-114) and trace = sum of the fixed
// singular values.  H = U S V^T  =>  H^T H = V S^2 V^T,  U = H V S^-1.
__device__ inline void procrustes3(const double H[3][3], double R[3][3], double* trace) {
  double A[3][3], V[3][3], w[3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { double s = 0; for (int k = 0; k < 3; ++k) s += H[k][i] * H[k][j]; A[i][j] = s; }
  jacobi3(A, V, w);
  int ord[3] = {0, 1, 2};                               // singular values in descending order, like torch.linalg.svd
  for (int i = 0; i < 2; ++i)
    for (int j = i + 1; j < 3; ++j)
      if (w[ord[j]] > w[ord[i]]) { const int t = ord[i]; ord[i] = ord[j]; ord[j] = t; }
  double Vs[3][3], U[3][3], s[3];
  for (int k = 0; k < 3; ++k) {
    s[k] = sqrt(fmax(w[ord[k]], 0.0));
    for (int i = 0; i < 3; ++i) Vs[i][k] = V[i][ord[k]];
  }
  for (int k = 0; k < 3; ++k) {                         // U[:, k] = H V[:, k] / s_k
    double u[3];
    for (int i = 0; i < 3; ++i) { u[i] = 0; for (int j = 0; j < 3; ++j) u[i] += H[i][j] * Vs[j][k]; }
    double n = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
    if (k == 2 && (s[2] < 1e-12 * s[0] || n < 1e-300)) {  // rank-deficient: complete U to an orthonormal basis (either sign:
      u[0] = U[1][0] * U[2][1] - U[2][0] * U[1][1];       // the reflection fix below removes the ambiguity from R)
      u[1] = U[2][0] * U[0][1] - U[0][0] * U[2][1];
      u[2] = U[0][0] * U[1][1] - U[1][0] * U[0][1];
      n = sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
    }
    for (int i = 0; i < 3; ++i) U[i][k] = n > 0 ? u[i] / n : 0.0;
  }
  double R0[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { double r = 0; for (int k = 0; k < 3; ++k) r += Vs[i][k] * U[j][k]; R0[i][j] = r; }
  const double det = R0[0][0] * (R0[1][1] * R0[2][2] - R0[1][2] * R0[2][1]) - R0[0][1] * (R0[1][0] * R0[2][2] - R0[1][2] * R0[2][0]) +
                     R0[0][2] * (R0[1][0] * R0[2][1] - R0[1][1] * R0[2][0]);
  const double sg = det > 0 ? 1.0 : (det < 0 ? -1.0 : 0.0);
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R[i][j] = (i == 2 ? sg : 1.0) * R0[i][j];      // V[:, :, -1] *= sign: the last ROW of V
  *trace = s[0] + s[1] + sg * s[2];
}

// One warp's item (sample b, frame t): stages the assembled and target poses at t (and t + 1) in the warp's slices sp /
// st, writes `assembled`, and returns in m[CISTGCN_METRIC_*] the warp sums of every metric over the joints (all lanes
// hold them; the velocity term is 0 at the last frame).
CG_DEV void metrics_item(const Args& a, float (&sp)[2][MAXJ * 3], float (&st)[2][MAXJ * 3], long long b, int t, int lane,
                         float (&m)[CISTGCN_METRIC_COUNT]) {
  const int To = a.To, Vf = a.Vf, Vu = a.Vu;
  const bool has_next = t + 1 < To;
  for (int f = 0; f < (has_next ? 2 : 1); ++f) {
    const float* tg = a.target + ((b * To + t + f) * Vf) * 3;
    const float* pr = a.pred + ((b * To + t + f) * Vu) * 3;
    for (int j = lane; j < Vf; j += 32) {
      const int mj = a.src_map[j];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float tv = __ldg(tg + j * 3 + k);
        st[f][j * 3 + k] = tv;
        sp[f][j * 3 + k] = mj >= 0 ? __ldg(pr + mj * 3 + k) : tv;
      }
    }
  }
  __syncwarp();
  const float* P = sp[0];
  const float* T0 = st[0];
  if (a.assembled) {
    float* o = a.assembled + ((b * To + t) * Vf) * 3;
    for (int i = lane; i < Vf * 3; i += 32) o[i] = P[i];
  }
  // ---- per-joint quantities
  float e = 0.f, ew0 = 0.f, ew1 = 0.f, ve = 0.f, dot = 0.f, pp = 0.f;
  float mx[3] = {0.f, 0.f, 0.f}, my[3] = {0.f, 0.f, 0.f};
  for (int j = lane; j < Vf; j += 32) {
    const float dx = P[j * 3] - T0[j * 3], dy = P[j * 3 + 1] - T0[j * 3 + 1], dz = P[j * 3 + 2] - T0[j * 3 + 2];
    const float ej = sqrtf(dx * dx + dy * dy + dz * dz);
    e += ej;
    if (a.wt[0]) ew0 += __ldg(a.wt[0] + (b * To + t) * Vf + j) * ej;
    if (a.wt[1]) ew1 += __ldg(a.wt[1] + (b * To + t) * Vf + j) * ej;
#pragma unroll
    for (int k = 0; k < 3; ++k) { dot += T0[j * 3 + k] * P[j * 3 + k]; pp += P[j * 3 + k] * P[j * 3 + k]; mx[k] += T0[j * 3 + k]; my[k] += P[j * 3 + k]; }
    if (has_next) {
      const float* P1 = sp[1];
      const float* T1 = st[1];
      float q = 0.f;
#pragma unroll
      for (int k = 0; k < 3; ++k) { const float dv = (P1[j * 3 + k] - P[j * 3 + k]) - (T1[j * 3 + k] - T0[j * 3 + k]); q += dv * dv; }
      ve += sqrtf(q);
    }
  }
  e = cg::warp_sum(e); ew0 = cg::warp_sum(ew0); ew1 = cg::warp_sum(ew1); ve = cg::warp_sum(ve);
  dot = cg::warp_sum(dot); pp = cg::warp_sum(pp);
#pragma unroll
  for (int k = 0; k < 3; ++k) { mx[k] = cg::warp_sum(mx[k]) / Vf; my[k] = cg::warp_sum(my[k]) / Vf; }
  // ---- N-MPJPE (:147-161): scale = mean_j(t . p) / mean_j(p . p)
  const float scale = dot / pp;
  float en = 0.f;
  for (int j = lane; j < Vf; j += 32) {
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) { const float dv = scale * P[j * 3 + k] - T0[j * 3 + k]; q += dv * dv; }
    en += sqrtf(q);
  }
  en = cg::warp_sum(en);
  // ---- bone lengths (:200-215)
  float eb = 0.f;
  for (int k = lane; k < a.NB; k += 32) {
    const int j0 = a.bones[2 * k], j1 = a.bones[2 * k + 1];
    float lp = 0.f, lt = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float d0 = P[j0 * 3 + c] - P[j1 * 3 + c], d1 = T0[j0 * 3 + c] - T0[j1 * 3 + c];
      lp += d0 * d0; lt += d1 * d1;
    }
    eb += fabsf(sqrtf(lp) - sqrtf(lt));
  }
  eb = cg::warp_sum(eb);
  // ---- PA-MPJPE (:79-144), following the reference step by step (its quirks included)
  float hx[9], nx = 0.f, ny = 0.f;
#pragma unroll
  for (int i = 0; i < 9; ++i) hx[i] = 0.f;
  for (int j = lane; j < Vf; j += 32) {
    float x0[3], y0[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      x0[k] = T0[j * 3 + k] - mx[k];
      y0[k] = P[j * 3 + k] - my[k];
      if (x0[k] * x0[k] < 1e-6f) x0[k] = 1e-3f;          // X0[X0 ** 2 < 1e-6] = 1e-3  (:95)
      nx += x0[k] * x0[k]; ny += y0[k] * y0[k];
    }
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) hx[r * 3 + c] += x0[r] * y0[c];
  }
  nx = cg::warp_sum(nx); ny = cg::warp_sum(ny);
#pragma unroll
  for (int i = 0; i < 9; ++i) hx[i] = cg::warp_sum(hx[i]);
  float normX = sqrtf(nx), normY = sqrtf(ny);
  if (normX < 1e-3f) normX = 1e-3f;                        // :100
  double H[3][3], R[3][3], tr = 0.0;
  for (int i = 0; i < 9; ++i) H[i / 3][i % 3] = (double)hx[i] / ((double)normX * (double)normY);
  procrustes3(H, R, &tr);                                  // every lane redundantly: no divergence, no broadcast
  float sa = (float)(tr * (double)normX / (double)normY);
  float Rf[9];
  for (int i = 0; i < 9; ++i) Rf[i] = (float)R[i / 3][i % 3];
  float tv[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) tv[c] = mx[c] - sa * (my[0] * Rf[0 * 3 + c] + my[1] * Rf[1 * 3 + c] + my[2] * Rf[2 * 3 + c]);
  if (sa != sa) sa = 1.f;                                  // :129-131 NaN guards
#pragma unroll
  for (int i = 0; i < 9; ++i) if (Rf[i] != Rf[i]) Rf[i] = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) if (tv[c] != tv[c]) tv[c] = 0.f;
  float epa = 0.f;
  for (int j = lane; j < Vf; j += 32) {
    float q = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float al = sa * (P[j * 3] * Rf[0 * 3 + c] + P[j * 3 + 1] * Rf[1 * 3 + c] + P[j * 3 + 2] * Rf[2 * 3 + c]) + tv[c];
      const float dv = al - T0[j * 3 + c];
      q += dv * dv;
    }
    epa += sqrtf(q);
  }
  epa = cg::warp_sum(epa);
  m[CISTGCN_METRIC_MPJPE] = e;
  m[CISTGCN_METRIC_PA_MPJPE] = epa;
  m[CISTGCN_METRIC_N_MPJPE] = en;
  m[CISTGCN_METRIC_VELOCITY] = ve;
  m[CISTGCN_METRIC_BONE_LENGTH] = eb;
  m[CISTGCN_METRIC_WEIGHTED0] = ew0;
  m[CISTGCN_METRIC_WEIGHTED1] = ew1;
}

}  // namespace cgm
