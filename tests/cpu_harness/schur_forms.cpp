// tests/cpu_harness/schur_forms.cpp — TEST INFRASTRUCTURE.
// Compares, on the CPU, the per-track Schur terms the assembly kernels build from the camera-frame helpers of
// lifcal_b200/csrc/lfba_math.cuh (point eliminated inside the 3 x 3 block, then projected onto the pose) with the
// same terms written out through the pose-point coupling V = M^T A R and W = V Hi. Built only by the tests.
#include <cmath>
#include <cstring>

#include "../../include/lfba.h"
#include "../../lifcal_b200/csrc/lfba_math.cuh"

using namespace lfba;

namespace {

// M (3 x 6) of a track, row-major: columns dR_a X, then I3
void full_m(const double* fe, const double* X, double M[18]) {
  for (int a = 0; a < 3; ++a)
    for (int i = 0; i < 3; ++i) {
      double v = 0.0;
      for (int k = 0; k < 3; ++k) v += fe[9 * (a + 1) + 3 * i + k] * X[k];
      M[6 * i + a] = v;
    }
  for (int i = 0; i < 3; ++i)
    for (int a = 0; a < 3; ++a) M[6 * i + 3 + a] = i == a ? 1.0 : 0.0;
}
double sym_at(const double* S, int i, int j) {
  if (i > j) { const int t = i; i = j; j = t; }
  return S[3 * i - i * (i + 1) / 2 + j];
}
// V = M^T A R (6 x 3)
void full_v(const double* A, const double* fe, const double* M, double V[18]) {
  double AR[9];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      double v = 0.0;
      for (int k = 0; k < 3; ++k) v += sym_at(A, i, k) * fe[3 * k + j];
      AR[3 * i + j] = v;
    }
  for (int a = 0; a < 6; ++a)
    for (int j = 0; j < 3; ++j) {
      double v = 0.0;
      for (int i = 0; i < 3; ++i) v += M[6 * i + a] * AR[3 * i + j];
      V[3 * a + j] = v;
    }
}

}  // namespace

// One point with two tracks (frames fe1, fe2). Inputs: track records A (6), b (3), C (3 x NC row-major) of track 1,
// A of track 2, the point X, Hi = (Hpp + D)^-1 (upper 6), g_p (3), Hcp (NC x 3), pose steps y1, y2 (6), camera step
// yc (NC). Outputs, for the reference form (ref) and the camera-frame form (fac), concatenated:
//   S_ff of track 1 (lower 21) | g_f (6) | S_cf (NC x 6) | pair block W1 V2^T (36) | y_p (3)
extern "C" void schur_forms(int NC, const double* A1, const double* b1, const double* C1, const double* fe1,
                            const double* A2, const double* fe2, const double* X, const double* Hi, const double* gp,
                            const double* Hcp, const double* y1, const double* y2, const double* yc, double* ref,
                            double* fac) {
  const int n = 21 + 6 + 6 * NC + 36 + 3;
  std::memset(ref, 0, sizeof(double) * n);
  std::memset(fac, 0, sizeof(double) * n);
  double* rS = ref;
  double* rg = ref + 21;
  double* rc = ref + 27;
  double* rp = ref + 27 + 6 * NC;
  double* ry = rp + 36;
  double* fS = fac;
  double* fg = fac + 21;
  double* fc = fac + 27;
  double* fp = fac + 27 + 6 * NC;
  double* fy = fp + 36;

  // ---- reference: V, W ----
  double M1[18], M2[18], V1[18], V2[18], W1[18];
  full_m(fe1, X, M1);
  full_m(fe2, X, M2);
  full_v(A1, fe1, M1, V1);
  full_v(A2, fe2, M2, V2);
  for (int a = 0; a < 6; ++a)
    for (int j = 0; j < 3; ++j) {
      double v = 0.0;
      for (int k = 0; k < 3; ++k) v += V1[3 * a + k] * sym_at(Hi, k, j);
      W1[3 * a + j] = v;
    }
  for (int a = 0, h = 0; a < 6; ++a)
    for (int c = 0; c <= a; ++c, ++h) {
      double v = 0.0;
      for (int i = 0; i < 3; ++i)
        for (int k = 0; k < 3; ++k) v += M1[6 * i + a] * sym_at(A1, i, k) * M1[6 * k + c];
      for (int j = 0; j < 3; ++j) v -= W1[3 * a + j] * V1[3 * c + j];
      rS[h] = v;
    }
  for (int a = 0; a < 6; ++a) {
    double v = 0.0;
    for (int i = 0; i < 3; ++i) v += M1[6 * i + a] * b1[i];
    for (int j = 0; j < 3; ++j) v -= W1[3 * a + j] * gp[j];
    rg[a] = v;
  }
  for (int c = 0; c < NC; ++c)
    for (int a = 0; a < 6; ++a) {
      double v = 0.0;
      for (int i = 0; i < 3; ++i) v += C1[i * NC + c] * M1[6 * i + a];
      for (int j = 0; j < 3; ++j) v -= Hcp[3 * c + j] * W1[3 * a + j];
      rc[6 * c + a] = v;
    }
  for (int a = 0; a < 6; ++a)
    for (int b = 0; b < 6; ++b) {
      double v = 0.0;
      for (int j = 0; j < 3; ++j) v += W1[3 * a + j] * V2[3 * b + j];
      rp[6 * a + b] = v;
    }
  {
    double r[3];
    for (int j = 0; j < 3; ++j) {
      double v = gp[j];
      for (int c = 0; c < NC; ++c) v -= Hcp[3 * c + j] * yc[c];
      for (int a = 0; a < 6; ++a) v -= V1[3 * a + j] * y1[a] + V2[3 * a + j] * y2[a];
      r[j] = v;
    }
    for (int i = 0; i < 3; ++i) ry[i] = sym_at(Hi, i, 0) * r[0] + sym_at(Hi, i, 1) * r[1] + sym_at(Hi, i, 2) * r[2];
  }

  // ---- camera-frame form, as k_points / k_frame_all / k_pairs / k_point_step compose the helpers ----
  double T[27];  // T_p = Hi Hcp^T, stored [3 c + j]
  for (int c = 0; c < NC; ++c) sym3_vec(Hi, Hcp + 3 * c, T + 3 * c);
  double m1[9], m2[9], B1[9], B2[9], K1[9], At[6];
  track_m(fe1, X, m1);
  track_m(fe2, X, m2);
  track_b(A1, fe1, B1);
  track_b(A2, fe2, B2);
  mat3_sym3(B1, Hi, K1);
  track_atilde(A1, B1, K1, At);
  mt_sym_m_acc(m1, At, fS);
  {
    double bt[3];
    mat3_vec(K1, gp, bt);
    for (int i = 0; i < 3; ++i) bt[i] = b1[i] - bt[i];
    mt_vec_acc(m1, bt, 1.0, fg);
  }
  for (int c = 0; c < NC; ++c) {
    const double col[3] = {C1[c], C1[NC + c], C1[2 * NC + c]};
    mt_vec_acc(m1, col, 1.0, fc + 6 * c);
    double bt[3];
    mat3_vec(B1, T + 3 * c, bt);
    mt_vec_acc(m1, bt, -1.0, fc + 6 * c);
  }
  {
    double G[9];
    mat3_mat3t(K1, B2, G);
    mt_mat_m_acc(m1, G, m2, fp);
  }
  {
    double h[3] = {0, 0, 0};
    track_vt_y_acc(A1, fe1, m1, y1, h);
    track_vt_y_acc(A2, fe2, m2, y2, h);
    const double r[3] = {gp[0] - h[0], gp[1] - h[1], gp[2] - h[2]};
    sym3_vec(Hi, r, fy);
    for (int c = 0; c < NC; ++c)
      for (int j = 0; j < 3; ++j) fy[j] -= T[3 * c + j] * yc[c];
  }
}

// W = V Hi from mt_mat (the form k_cov_points uses) against the reference
extern "C" void track_w_forms(const double* A, const double* fe, const double* X, const double* Hi, double* ref,
                              double* fac) {
  double M[18], V[18];
  full_m(fe, X, M);
  full_v(A, fe, M, V);
  for (int a = 0; a < 6; ++a)
    for (int j = 0; j < 3; ++j) {
      double v = 0.0;
      for (int k = 0; k < 3; ++k) v += V[3 * a + k] * sym_at(Hi, k, j);
      ref[3 * a + j] = v;
    }
  double m[9], B[9], K[9];
  track_m(fe, X, m);
  track_b(A, fe, B);
  mat3_sym3(B, Hi, K);
  mt_mat(m, K, fac);
}
