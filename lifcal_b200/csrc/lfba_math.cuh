// lfba_math.cuh — per-item arithmetic of the LF-BA hot path, written as __host__ __device__ functions so
// that the CUDA kernels (lfba_kernels.cu) and the CPU test harness (tests/cpu_harness) run the SAME code.
//
// What is computed (reference file:line it replaces):
//   cam_model_init   camera-block decode of OurCostFunctionBundle::operator_function
//                    (src/BundleAdjustment/BundleAdjustment.h:123-146) + per-evaluation scalars
//   lens_entry       the 10-step fixed-point undistortion of a micro-lens centre (src/CameraModel.h:93-125)
//                    AND its exact forward-mode derivative recurrence (what Ceres' Jets carry through the
//                    loop), once per distinct lens instead of once per observation (SURVEY.md E.1/E.2)
//   frame_entry      R = Rx Ry Rz and dR/da_k of RigidBody::getTransformationMatrix (src/CameraModel.h:246-264),
//                    once per frame instead of once per observation
//   track_setup      everything that depends only on (camera, pose, point): P_c = R X + t and the
//                    per-track scalars of the analytic Jacobian
//   obs_eval         residual (2) + analytic Jacobian of CameraModel::projectPoint (src/CameraModel.h:127-195)
//                    w.r.t. the camera-frame point (G, 2x3) and the live camera parameters (Jc, 2xNC)
//   robust_scale     ceres::CauchyLoss(a) + Corrector (rho'' < 0 branch): sqrt(rho') and rho
// The reference differentiates with ceres::Jet<double,26>; here the derivative is analytic. The chain rule
// through pose and point is applied per TRACK (point, frame), not per observation:
//   J_i = [ Jc_i | G_i M | G_i R ],  M = [dR/da0 X, dR/da1 X, dR/da2 X, I3]  (SURVEY.md E.3)
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define LFBA_HD __host__ __device__ __forceinline__
#else
#define LFBA_HD inline
#endif

namespace lfba {

constexpr int kMaxNC = 9;         // live camera parameters: 5 + nRadial(<=2) + 2*tangential
constexpr int kLensStride = 16;   // doubles per lens-table entry (one 128-byte line)
constexpr int kFrameStride = 40;  // doubles per frame-table entry: R(9) dR0(9) dR1(9) dR2(9) t(3) pad(1)

// lens-table entry layout
//  [0] mx [1] my                      lens centre (raw px)
//  [2] ux [3] uy                      u10: undistorted centre on the MLA plane (mm), before the mlAdj scaling
//  [4] dux/dc3 [5] duy/dc3            derivative w.r.t. camera[3] (cx)
//  [6] dux/dc4 [7] duy/dc4            derivative w.r.t. camera[4] (cy)
//  [8..9] d/dk0  [10..11] d/dk1  [12..13] d/dt0  [14..15] d/dt1

struct CamModel {
  int n_radial, tangential, ml_adjust, robust, any_dist, nc;
  double fL, bL0, B;    // |camera[0..2]|
  double sg[3];         // sign of camera[0..2]: d|x|/dx with Jet semantics (x < 0 ? -1 : +1)
  double crx, cry;      // c_raw = |(c + 0.5) * scale - 0.5|
  double dcrx, dcry;    // d c_raw / d camera[3], camera[4]
  double sx, sy, isx, isy;  // raw pixel size (mm) and reciprocal
  double k0, k1, t0, t1;
  double k0x2, k1x4, t0x2, t1x2, t0x6, t1x6;  // multiples used by dist_shift_jac
  double invD, alpha, zC0, gB, inv_fL, gamma;
  double dalpha_dfL, dalpha_dbL0, dz_dfL, dz_dbL0, dgB_dfL, dgB_dbL0, dgB_dB, dgamma_dbL0, dgamma_dB;
  double loss_b, loss_c;  // Cauchy: b = a^2, c = 1/b
};

LFBA_HD void cam_model_init(CamModel& m, const double* c, uint32_t config, double spx, double spy, double scale,
                            double loss_a) {
  m.n_radial = (int)(config & 3u);
  m.tangential = (config & 0x4u) ? 1 : 0;
  m.ml_adjust = (config & 0x800u) ? 1 : 0;
  m.robust = (config & 0x200u) ? 1 : 0;
  m.any_dist = (m.n_radial > 0 || m.tangential) ? 1 : 0;
  m.nc = 5 + m.n_radial + 2 * m.tangential;
  m.fL = fabs(c[0]);
  m.bL0 = fabs(c[1]);
  m.B = fabs(c[2]);
  for (int i = 0; i < 3; ++i) m.sg[i] = c[i] < 0.0 ? -1.0 : 1.0;
  const double cx_in = (c[3] + 0.5) * scale - 0.5, cy_in = (c[4] + 0.5) * scale - 0.5;
  m.crx = fabs(cx_in);
  m.cry = fabs(cy_in);
  m.dcrx = (cx_in < 0.0 ? -1.0 : 1.0) * scale;
  m.dcry = (cy_in < 0.0 ? -1.0 : 1.0) * scale;
  m.sx = spx / scale;
  m.sy = spy / scale;
  m.isx = 1.0 / m.sx;
  m.isy = 1.0 / m.sy;
  m.k0 = m.n_radial > 0 ? c[5] : 0.0;
  m.k1 = m.n_radial > 1 ? c[6] : 0.0;
  m.t0 = m.tangential ? c[5 + m.n_radial] : 0.0;
  m.t1 = m.tangential ? c[6 + m.n_radial] : 0.0;
  m.k0x2 = 2.0 * m.k0;
  m.k1x4 = 4.0 * m.k1;
  m.t0x2 = 2.0 * m.t0;
  m.t1x2 = 2.0 * m.t1;
  m.t0x6 = 6.0 * m.t0;
  m.t1x6 = 6.0 * m.t1;
  const double D = m.fL - m.bL0;
  m.invD = 1.0 / D;
  m.alpha = m.fL * m.invD;
  m.zC0 = m.fL * m.bL0 * m.invD;
  m.gB = m.fL * m.B * m.invD;
  m.inv_fL = 1.0 / m.fL;
  const double id2 = m.invD * m.invD;
  m.dalpha_dfL = -m.bL0 * id2;
  m.dalpha_dbL0 = m.fL * id2;
  m.dz_dfL = -m.bL0 * m.bL0 * id2;
  m.dz_dbL0 = m.fL * m.fL * id2;
  m.dgB_dfL = m.B * m.dalpha_dfL;
  m.dgB_dbL0 = m.B * m.dalpha_dbL0;
  m.dgB_dB = m.alpha;
  if (m.ml_adjust) {
    const double s = m.bL0 + m.B, is2 = 1.0 / (s * s);
    m.gamma = m.bL0 / s;
    m.dgamma_dbL0 = m.B * is2;
    m.dgamma_dB = -m.bL0 * is2;
  } else {
    m.gamma = 1.0;
    m.dgamma_dbL0 = 0.0;
    m.dgamma_dB = 0.0;
  }
  m.loss_b = loss_a * loss_a;
  m.loss_c = 1.0 / m.loss_b;
}

// radial + tangential shift (src/CameraModel.h:205-241), value only
LFBA_HD void dist_shift(const CamModel& m, double x, double y, double& dx, double& dy) {
  // same expression tree as dist_shift_jac so both paths round identically
  const double xx = x * x, yy = y * y, xy = x * y;
  const double r2 = xx + yy;
  const double dr = r2 * fma(m.k1, r2, m.k0);
  const double ax = fma(2.0, xx, r2), ay = fma(2.0, yy, r2), xy2 = xy + xy;
  dx = fma(x, dr, fma(m.t0, ax, m.t1 * xy2));
  dy = fma(y, dr, fma(m.t1, ay, m.t0 * xy2));
}

// shift, its 2x2 Jacobian A = d(shift)/d(x,y) and d(shift)/d(k0,k1,t0,t1) (each a 2-vector). A is symmetric:
// A[0] = d dx/dx, A[1] = d dx/dy = d dy/dx, A[2] = d dy/dy. 30 FP64 instructions (multiples of the coefficients are
// model constants): this runs once per observation inside the fused evaluation kernel.
//   dr = k0 r2 + k1 r2^2,  dr' = k0 + 2 k1 r2
//   dx = x dr + t0 (r2 + 2 x^2) + 2 t1 x y,   dy = y dr + t1 (r2 + 2 y^2) + 2 t0 x y
LFBA_HD void dist_shift_jac(const CamModel& m, double x, double y, double& dx, double& dy, double A[3],
                            double dk0[2], double dk1[2], double dt0[2], double dt1[2]) {
  const double xx = x * x, yy = y * y, xy = x * y;
  const double r2 = xx + yy, r4 = r2 * r2;
  const double dr = r2 * fma(m.k1, r2, m.k0);
  const double ddr2 = fma(m.k1x4, r2, m.k0x2);  // 2 dr'
  const double ax = fma(2.0, xx, r2), ay = fma(2.0, yy, r2), xy2 = xy + xy;
  dx = fma(x, dr, fma(m.t0, ax, m.t1 * xy2));
  dy = fma(y, dr, fma(m.t1, ay, m.t0 * xy2));
  A[0] = fma(m.t1x2, y, fma(m.t0x6, x, fma(xx, ddr2, dr)));
  A[1] = fma(xy, ddr2, fma(m.t0x2, y, m.t1x2 * x));
  A[2] = fma(m.t0x2, x, fma(m.t1x6, y, fma(yy, ddr2, dr)));
  dk0[0] = x * r2;
  dk0[1] = y * r2;
  dk1[0] = x * r4;
  dk1[1] = y * r4;
  dt0[0] = ax;
  dt0[1] = xy2;
  dt1[0] = xy2;
  dt1[1] = ay;
}

// One lens-table entry: u_0 = cd, u_i = cd - shift(u_{i-1}), i = 1..10 (exactly ten steps, src/CameraModel.h:109),
// carrying U_i = du_i/dcd (2x2) and E_i = du_i/d(k0,k1,t0,t1) (2x4) through the same ten steps:
//   U_i = I - A(u_{i-1}) U_{i-1},   E_i = -A(u_{i-1}) E_{i-1} - dshift/dtheta(u_{i-1}).
LFBA_HD void lens_entry(const CamModel& m, double mx, double my, double* e) {
  const double cdx = (mx - m.crx) * m.sx, cdy = (my - m.cry) * m.sy;
  double ux = cdx, uy = cdy;
  double U[4] = {1.0, 0.0, 0.0, 1.0};
  double E[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // E[2*k + row], k = k0,k1,t0,t1
  if (m.any_dist) {
    for (int it = 0; it < 10; ++it) {
      double dx, dy, A[3], d[8];
      dist_shift_jac(m, ux, uy, dx, dy, A, d + 0, d + 2, d + 4, d + 6);
      const double n0 = 1.0 - (A[0] * U[0] + A[1] * U[2]), n1 = -(A[0] * U[1] + A[1] * U[3]);
      const double n2 = -(A[1] * U[0] + A[2] * U[2]), n3 = 1.0 - (A[1] * U[1] + A[2] * U[3]);
      U[0] = n0;
      U[1] = n1;
      U[2] = n2;
      U[3] = n3;
      for (int k = 0; k < 4; ++k) {
        const double ex = E[2 * k], ey = E[2 * k + 1];
        E[2 * k] = -(A[0] * ex + A[1] * ey) - d[2 * k];
        E[2 * k + 1] = -(A[1] * ex + A[2] * ey) - d[2 * k + 1];
      }
      ux = (cdx - dx);
      uy = (cdy - dy);
    }
  }
  e[0] = mx;
  e[1] = my;
  e[2] = ux;
  e[3] = uy;
  // d cd / d camera[3] = (-dcrx * sx, 0);  d cd / d camera[4] = (0, -dcry * sy)
  const double fx = -m.dcrx * m.sx, fy = -m.dcry * m.sy;
  e[4] = U[0] * fx;
  e[5] = U[2] * fx;
  e[6] = U[1] * fy;
  e[7] = U[3] * fy;
  for (int k = 0; k < 8; ++k) e[8 + k] = E[k];
}

// R = Rx(a0) Ry(a1) Rz(a2) (row-major) and dR/da_k; f[36..38] = translation.
LFBA_HD void frame_entry(const double* v, double* f) {
  const double c0 = cos(v[0]), s0 = sin(v[0]);
  const double c1 = cos(v[1]), s1 = sin(v[1]);
  const double c2 = cos(v[2]), s2 = sin(v[2]);
  double* R = f;
  R[0] = c1 * c2;
  R[1] = -c1 * s2;
  R[2] = s1;
  R[3] = s0 * s1 * c2 + c0 * s2;
  R[4] = -s0 * s1 * s2 + c0 * c2;
  R[5] = -s0 * c1;
  R[6] = -c0 * s1 * c2 + s0 * s2;
  R[7] = c0 * s1 * s2 + s0 * c2;
  R[8] = c0 * c1;
  double* d0 = f + 9;  // d/da0: derivative of (s0, c0) -> (c0, -s0)
  d0[0] = 0.0;
  d0[1] = 0.0;
  d0[2] = 0.0;
  d0[3] = c0 * s1 * c2 - s0 * s2;
  d0[4] = -c0 * s1 * s2 - s0 * c2;
  d0[5] = -c0 * c1;
  d0[6] = s0 * s1 * c2 + c0 * s2;
  d0[7] = -s0 * s1 * s2 + c0 * c2;
  d0[8] = -s0 * c1;
  double* d1 = f + 18;  // d/da1
  d1[0] = -s1 * c2;
  d1[1] = s1 * s2;
  d1[2] = c1;
  d1[3] = s0 * c1 * c2;
  d1[4] = -s0 * c1 * s2;
  d1[5] = s0 * s1;
  d1[6] = -c0 * c1 * c2;
  d1[7] = c0 * c1 * s2;
  d1[8] = -c0 * s1;
  double* d2 = f + 27;  // d/da2
  d2[0] = -c1 * s2;
  d2[1] = -c1 * c2;
  d2[2] = 0.0;
  d2[3] = -s0 * s1 * s2 + c0 * c2;
  d2[4] = -s0 * s1 * c2 - c0 * s2;
  d2[5] = 0.0;
  d2[6] = c0 * s1 * s2 + s0 * c2;
  d2[7] = c0 * s1 * c2 - s0 * s2;
  d2[8] = 0.0;
  f[36] = v[3];
  f[37] = v[4];
  f[38] = v[5];
  f[39] = 0.0;
}

LFBA_HD void mat3_vec(const double* R, const double* x, double* y) {
  y[0] = R[0] * x[0] + R[1] * x[1] + R[2] * x[2];
  y[1] = R[3] * x[0] + R[4] * x[1] + R[5] * x[2];
  y[2] = R[6] * x[0] + R[7] * x[1] + R[8] * x[2];
}

// camera-frame point of a track
LFBA_HD void track_point(const double* fe, const double* X, double Pc[3]) {
  mat3_vec(fe, X, Pc);
  Pc[0] += fe[36];
  Pc[1] += fe[37];
  Pc[2] += fe[38];
}

struct TrackCtx {
  double wpx, wpy; // gB * P_c.xy / q_z: the part of the projected point that does not depend on the micro lens
  double Px, Py;   // P_c.xy / q_z
  double a1;       // alpha / q_z
  double g1;       // gB / q_z
  double kl;       // d w0 / d u   (scalar): mlAdj ? (kappa + 1) * gamma : kappa
  double af, bf, ab, bb, aB, bB;  // d w0 / d(fL,bL0,B) = u * a + q * b  (signs of the |.| folded in)
};

LFBA_HD void track_setup(const CamModel& m, const double Pc[3], TrackCtx& t) {
  const double iq = 1.0 / (Pc[2] + m.zC0);
  t.Px = Pc[0] * iq;
  t.Py = Pc[1] * iq;
  t.a1 = m.alpha * iq;
  t.g1 = m.gB * iq;
  t.wpx = t.g1 * Pc[0];
  t.wpy = t.g1 * Pc[1];
  const double kappa = m.gB * (t.a1 - m.inv_fL);  // d pm / d cu
  const double k1 = m.ml_adjust ? kappa + 1.0 : kappa;
  t.kl = k1 * m.gamma;
  // d pm / d theta at fixed cu = cu * a' + q * b'
  const double af = m.gB * (m.dalpha_dfL * iq + m.inv_fL * m.inv_fL) - m.inv_fL * m.dgB_dfL;
  const double bf = m.dgB_dfL - t.g1 * m.dz_dfL;
  const double ab = m.gB * m.dalpha_dbL0 * iq - m.inv_fL * m.dgB_dbL0;
  const double bb = m.dgB_dbL0 - t.g1 * m.dz_dbL0;
  const double aB = -m.alpha * m.inv_fL;
  const double bB = m.alpha;
  // in terms of u (cu = gamma * u), plus the path through gamma(bL0, B) when mlAdj
  t.af = m.sg[0] * (m.gamma * af);
  t.bf = m.sg[0] * bf;
  t.ab = m.sg[1] * (m.gamma * ab + k1 * m.dgamma_dbL0);
  t.bb = m.sg[1] * bb;
  t.aB = m.sg[2] * (m.gamma * aB + k1 * m.dgamma_dB);
  t.bB = m.sg[2] * bB;
}

// ---- one observation ------------------------------------------------------------------------------------------
// Projection of src/CameraModel.h:127-195 at fixed (camera, pose, point), as a function of the micro lens:
//   q  = P + a1 gamma u,   pm = gB (q - gamma u / fL) = gB P + kappa gamma u,   w0 = pm + gamma u  (mlAdj)
// i.e. w0 = wp + kl u with the per-TRACK wp = gB P and kl (track_setup): two FMAs per observation.
//   mlAdj:  w = w0 + shift(w0)                r = w / s + c_raw - o      M = d r / d w0 = diag(1/s) (I + A(w0))
//   else :  w = w0 + (m - c_raw) s            (no forward distortion)   M = diag(1/s)
// dk = d shift / d(k0,k1,t0,t1) at w0 (the direct term of the forward distortion), zero unless mlAdj with distortion.
// Every form below (value only, Jacobian, features) goes through this one function: they agree bit for bit.
// ml_adjust / any_dist are passed beside the model so that a caller that knows them at compile time (the fused kernel)
// gets straight-line code.
template <class LensEntry>
LFBA_HD void obs_core(const CamModel& m, const TrackCtx& t, const LensEntry& e, double ox, double oy, double r[2],
                      double M[4], double dk[8], const bool ml_adjust, const bool any_dist) {
  double wx = fma(t.kl, e[2], t.wpx), wy = fma(t.kl, e[3], t.wpy);
  M[0] = m.isx;
  M[1] = 0.0;
  M[2] = 0.0;
  M[3] = m.isy;
#pragma unroll
  for (int k = 0; k < 8; ++k) dk[k] = 0.0;
  if (ml_adjust) {
    if (any_dist) {
      double dx, dy, A[3];
      dist_shift_jac(m, wx, wy, dx, dy, A, dk + 0, dk + 2, dk + 4, dk + 6);
      wx += dx;
      wy += dy;
      M[0] = fma(m.isx, A[0], m.isx);
      M[1] = m.isx * A[1];
      M[2] = m.isy * A[1];
      M[3] = fma(m.isy, A[2], m.isy);
    }
  } else {
    wx = fma(e[0] - m.crx, m.sx, wx);
    wy = fma(e[1] - m.cry, m.sy, wy);
  }
  r[0] = fma(wx, m.isx, m.crx) - ox;
  r[1] = fma(wy, m.isy, m.cry) - oy;
}

// residual only. Not called by a kernel: the CPU harness (tests/cpu_harness) uses it as the value-only form the analytic
// Jacobian path must agree with bit for bit
LFBA_HD void obs_residual(const CamModel& m, const TrackCtx& t, const double* e, double ox, double oy,
                          double r[2]) {
  double wx = fma(t.kl, e[2], t.wpx), wy = fma(t.kl, e[3], t.wpy);
  if (m.ml_adjust) {
    if (m.any_dist) {
      double dx, dy;
      dist_shift(m, wx, wy, dx, dy);
      wx += dx;
      wy += dy;
    }
  } else {
    wx = fma(e[0] - m.crx, m.sx, wx);
    wy = fma(e[1] - m.cry, m.sy, wy);
  }
  r[0] = fma(wx, m.isx, m.crx) - ox;
  r[1] = fma(wy, m.isy, m.cry) - oy;
}

// Columns of d r / d(cx, cy, k0.., t0, t1) — what every form shares: through u (lens table, scaled by the per-track
// kl: Mk = kl M), through (m - c_raw) when !mlAdj, the additive + c_raw of the output, and the direct term of the
// forward distortion. out_x[c], out_y[c] for c = 0 .. NC-4 (cx, cy, then the live distortion parameters).
template <int NC, int NRAD, class LensEntry>
LFBA_HD void obs_lens_columns(const CamModel& m, const TrackCtx& t, const LensEntry& e, const double M[4],
                              const double dk[8], double* out_x, double* out_y, const bool ml_adjust,
                              const bool any_dist) {
  constexpr int TAN = (NC - 5 - NRAD) / 2;
  const double K00 = t.kl * M[0], K01 = t.kl * M[1], K10 = t.kl * M[2], K11 = t.kl * M[3];
  double c3x = m.dcrx, c3y = 0.0, c4x = 0.0, c4y = m.dcry;
  if (!ml_adjust) {
    const double d3 = -m.dcrx * m.sx, d4 = -m.dcry * m.sy;
    c3x = fma(M[0], d3, c3x);
    c3y = M[2] * d3;
    c4x = M[1] * d4;
    c4y = fma(M[3], d4, c4y);
  }
  out_x[0] = fma(K00, e[4], fma(K01, e[5], c3x));
  out_y[0] = fma(K10, e[4], fma(K11, e[5], c3y));
  out_x[1] = fma(K00, e[6], fma(K01, e[7], c4x));
  out_y[1] = fma(K10, e[6], fma(K11, e[7], c4y));
  const bool fwd = ml_adjust && any_dist;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const bool live = (k == 0 && NRAD > 0) || (k == 1 && NRAD > 1) || (k >= 2 && TAN);
    if (!live) continue;
    const int col = 2 + (k < 2 ? k : NRAD + (k - 2));  // compile-time after unrolling
    double jx = K01 * e[9 + 2 * k], jy = K11 * e[9 + 2 * k];
    if (fwd) {
      jx = fma(dk[2 * k], m.isx, jx);
      jy = fma(dk[2 * k + 1], m.isy, jy);
    }
    out_x[col] = fma(K00, e[8 + 2 * k], jx);
    out_y[col] = fma(K10, e[8 + 2 * k], jy);
  }
}

// residual + analytic Jacobian. G: 2x3 row-major d r / d P_c.  Jc: 2 x NC row-major, columns in camera-block
// order [fL, bL0, B, cx, cy, k0.., t0, t1].
// NRAD (number of radial parameters) is a template parameter so that every column index below is a compile-time
// constant: with run-time column placement the Jacobian array ends up in local memory (measured: 70 LDL/STL per
// observation). Tangential distortion is implied: TAN = (NC - 5 - NRAD) / 2.
template <int NC, int NRAD, class LensEntry>
LFBA_HD void obs_eval(const CamModel& m, const TrackCtx& t, const LensEntry& e, double ox, double oy, double r[2],
                      double G[6], double* Jc) {
  constexpr int TAN = (NC - 5 - NRAD) / 2;
  static_assert(5 + NRAD + 2 * TAN == NC && NRAD >= 0 && NRAD <= 2 && (TAN == 0 || TAN == 1), "NC / NRAD mismatch");
  double M[4], dk[8];
  obs_core(m, t, e, ox, oy, r, M, dk, m.ml_adjust != 0, m.any_dist != 0);
  const double ux = e[2], uy = e[3];
  const double ca = t.a1 * m.gamma;
  const double qx = fma(ca, ux, t.Px), qy = fma(ca, uy, t.Py);

  // d r / d P_c = M * g1 * [I | -q]
  G[0] = M[0] * t.g1;
  G[1] = M[1] * t.g1;
  G[2] = -(G[0] * qx + G[1] * qy);
  G[3] = M[2] * t.g1;
  G[4] = M[3] * t.g1;
  G[5] = -(G[3] * qx + G[4] * qy);

  // fL, bL0, B
  {
    const double dfx = ux * t.af + qx * t.bf, dfy = uy * t.af + qy * t.bf;
    const double dbx = ux * t.ab + qx * t.bb, dby = uy * t.ab + qy * t.bb;
    const double dBx = ux * t.aB + qx * t.bB, dBy = uy * t.aB + qy * t.bB;
    Jc[0] = M[0] * dfx + M[1] * dfy;
    Jc[NC + 0] = M[2] * dfx + M[3] * dfy;
    Jc[1] = M[0] * dbx + M[1] * dby;
    Jc[NC + 1] = M[2] * dbx + M[3] * dby;
    Jc[2] = M[0] * dBx + M[1] * dBy;
    Jc[NC + 2] = M[2] * dBx + M[3] * dBy;
  }
  obs_lens_columns<NC, NRAD>(m, t, e, M, dk, Jc + 3, Jc + NC + 3, m.ml_adjust != 0, m.any_dist != 0);
}

// ---- feature form of the per-observation Jacobian ---------------------------------------------------------
// Inside one track every Jacobian column of an observation is a combination, with per-TRACK coefficients, of a few
// per-observation 2-vectors ("features"). With M (2x2), q and u as above:
//     f0 = M[:,0]   f1 = M[:,1]   f2 = M q   f3 = M u   f(4+j) = d r / d camera[3+j]   (j = 0 .. NC-4)
//     d r/d P_c   = g1 [ f0 | f1 | -f2 ]
//     d r/d fL    = af f3 + bf f2,   d r/d bL0 = ab f3 + bb f2,   d r/d B = aB f3 + bB f2
// so the normal-equation blocks of a track follow from the Gram matrix of NF = NC + 1 features (+ their products with
// r): 65 running sums for NC = 9 instead of 36 (track) + 55 (camera) = 91, and 2 NF (NF + 3) / 2 FMAs per observation
// instead of 180. The exact same sums result (this is algebra, not an approximation); only the rounding order differs.
template <int NC>
struct FeatDims {
  static constexpr int NF = NC + 1;
  static constexpr int NQ = NF * (NF + 1) / 2;  // Gram, lower triangle, row-major: Q(a,b), a >= b at a(a+1)/2 + b
  static constexpr int NG = NQ + NF;            // + h(a) = sum f_a . r
};

// residual and features; F[a] = x component, F[NF + a] = y component of feature a. The fused kernel uses the reduced set
// (obs_features9 + gram9_expand); this full set is the form the CPU harness checks the expansion against.
template <int NC, int NRAD, class LensEntry>
LFBA_HD void obs_features(const CamModel& m, const TrackCtx& t, const LensEntry& e, double ox, double oy, double r[2],
                          double* F) {
  constexpr int NF = NC + 1;
  constexpr int TAN = (NC - 5 - NRAD) / 2;
  static_assert(5 + NRAD + 2 * TAN == NC && NRAD >= 0 && NRAD <= 2 && (TAN == 0 || TAN == 1), "NC / NRAD mismatch");
  double M[4], dk[8];
  obs_core(m, t, e, ox, oy, r, M, dk, m.ml_adjust != 0, m.any_dist != 0);
  const double ux = e[2], uy = e[3];
  const double ca = t.a1 * m.gamma;
  const double qx = fma(ca, ux, t.Px), qy = fma(ca, uy, t.Py);
  F[0] = M[0];
  F[NF + 0] = M[2];
  F[1] = M[1];
  F[NF + 1] = M[3];
  F[2] = M[0] * qx + M[1] * qy;
  F[NF + 2] = M[2] * qx + M[3] * qy;
  F[3] = M[0] * ux + M[1] * uy;
  F[NF + 3] = M[2] * ux + M[3] * uy;
  obs_lens_columns<NC, NRAD>(m, t, e, M, dk, F + 4, F + NF + 4, m.ml_adjust != 0, m.any_dist != 0);
}

// ---- reduced feature set (NC + 0 features) --------------------------------------------------------------------
// f2 = M q is not independent: q = P + (a1 gamma) u with per-TRACK P and a1, so f2 = Px f0 + Py f1 + (a1 gamma) f3.
// Dropping it leaves NF9 = NC features [f0, f1, f3, f4, ...] and 54 instead of 65 running sums for NC = 9; the
// sums that involve f2 are rebuilt once per track (gram9_expand) — the same algebra, 22 fewer DFMA per observation.
template <int NC>
struct Feat9Dims {
  static constexpr int NF = NC;
  static constexpr int NQ = NF * (NF + 1) / 2;
  static constexpr int NG = NQ + NF;
};

// residual and the NC features; F[a] = x component, F[NC + a] = y component.
// New index -> old index (obs_features): 0 -> 0, 1 -> 1, a >= 2 -> a + 1.
// For NC = 9 with mlAdj and distortion: 42 (obs_core) + 4 + 36 FP64 instructions; only wp, kl of the track are read.
template <int NC, int NRAD, class LensEntry>
LFBA_HD void obs_features9(const CamModel& m, const TrackCtx& t, const LensEntry& e, double ox, double oy, double r[2],
                           double* F, const bool ml_adjust, const bool any_dist) {
  constexpr int NF = NC;
  constexpr int TAN = (NC - 5 - NRAD) / 2;
  static_assert(5 + NRAD + 2 * TAN == NC && NRAD >= 0 && NRAD <= 2 && (TAN == 0 || TAN == 1), "NC / NRAD mismatch");
  double M[4], dk[8];
  obs_core(m, t, e, ox, oy, r, M, dk, ml_adjust, any_dist);
  F[0] = M[0];
  F[NF + 0] = M[2];
  F[1] = M[1];
  F[NF + 1] = M[3];
  F[2] = fma(M[0], e[2], M[1] * e[3]);
  F[NF + 2] = fma(M[2], e[2], M[3] * e[3]);
  obs_lens_columns<NC, NRAD>(m, t, e, M, dk, F + 3, F + NF + 3, ml_adjust, any_dist);
}

// Rebuild the NC+1-feature Gram sums (layout of FeatDims<NC>: Q lower triangle row-major, then h) from the NC-feature
// sums gn (layout of Feat9Dims<NC>), using f2 = Px f0 + Py f1 + c f3, c = a1 * gamma.
template <int NC>
LFBA_HD void gram9_expand(const TrackCtx& t, double c, const double* gn, double* go) {
  constexpr int NF9 = NC, NQ9 = NF9 * (NF9 + 1) / 2;
  constexpr int NF = NC + 1, NQ = NF * (NF + 1) / 2;
  auto Qn = [&](int a, int b) -> double { return a >= b ? gn[a * (a + 1) / 2 + b] : gn[b * (b + 1) / 2 + a]; };
#pragma unroll
  for (int a = 0; a < NF; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) {
      double v;
      if (a == 2 && b == 2) {
        v = t.Px * (t.Px * Qn(0, 0) + 2.0 * (t.Py * Qn(1, 0) + c * Qn(2, 0))) +
            t.Py * (t.Py * Qn(1, 1) + 2.0 * c * Qn(2, 1)) + c * c * Qn(2, 2);
      } else if (a == 2 || b == 2) {
        const int o = a == 2 ? b : a;            // the other (old) index, != 2
        const int n = o < 2 ? o : o - 1;         // its new index
        v = t.Px * Qn(0, n) + t.Py * Qn(1, n) + c * Qn(2, n);
      } else {
        v = Qn(a < 2 ? a : a - 1, b < 2 ? b : b - 1);
      }
      go[a * (a + 1) / 2 + b] = v;
    }
  const double* hn = gn + NQ9;
#pragma unroll
  for (int a = 0; a < NF; ++a)
    go[NQ + a] = a == 2 ? t.Px * hn[0] + t.Py * hn[1] + c * hn[2] : hn[a < 2 ? a : a - 1];
}

// Track blocks from the Gram sums. Q, h as in FeatDims; outputs: rec = [A(6) b(3) C(3 x NC)], hcc (lower, NC(NC+1)/2), gc.
// Every output entry is independent; `stride`/`first` let L lanes split the entries (entry index % stride == first).
template <int NC>
struct GramMap {
  static constexpr int NF = NC + 1;
  LFBA_HD static double Q(const double* g, int a, int b) { return a >= b ? g[a * (a + 1) / 2 + b] : g[b * (b + 1) / 2 + a]; }
  // coefficient pair (on f3, on f2) of camera column c < 3, and the feature index of a lens column c >= 3
  LFBA_HD static void geo(const TrackCtx& t, int c, double& a, double& b) {
    a = c == 0 ? t.af : (c == 1 ? t.ab : t.aB);
    b = c == 0 ? t.bf : (c == 1 ? t.bb : t.bB);
  }
  // <column c1, column c2> of the camera Jacobian
  LFBA_HD static double cc(const TrackCtx& t, const double* g, int c1, int c2) {
    if (c1 < 3 && c2 < 3) {
      double a1, b1, a2, b2;
      geo(t, c1, a1, b1);
      geo(t, c2, a2, b2);
      return a1 * a2 * Q(g, 3, 3) + (a1 * b2 + b1 * a2) * Q(g, 3, 2) + b1 * b2 * Q(g, 2, 2);
    }
    if (c1 >= 3 && c2 >= 3) return Q(g, c1 + 1, c2 + 1);
    const int cl = c1 >= 3 ? c1 : c2, cg = c1 >= 3 ? c2 : c1;
    double a, b;
    geo(t, cg, a, b);
    return a * Q(g, cl + 1, 3) + b * Q(g, cl + 1, 2);
  }
  // <G column i, camera column c>;  G = g1 [f0 | f1 | -f2]
  LFBA_HD static double gcam(const TrackCtx& t, const double* g, int i, int c) {
    const double gi = i == 2 ? -t.g1 : t.g1;
    if (c < 3) {
      double a, b;
      geo(t, c, a, b);
      return gi * (a * Q(g, 3, i) + b * Q(g, 2, i));
    }
    return gi * Q(g, c + 1, i);
  }
  LFBA_HD static double gg(const TrackCtx& t, const double* g, int i, int j) {
    const double s = ((i == 2) != (j == 2)) ? -1.0 : 1.0;
    return s * t.g1 * t.g1 * Q(g, i, j);
  }
};

// CauchyLoss(a) + Corrector for rho'' < 0: returns sqrt(rho') (the factor applied to r and J) and rho(s).
// Non-robust: factor 1, rho = s.
LFBA_HD double robust_scale(const CamModel& m, double s, double& rho) {
  if (!m.robust) {
    rho = s;
    return 1.0;
  }
  const double sum = 1.0 + s * m.loss_c;
  rho = m.loss_b * log(sum);
  return sqrt(1.0 / sum);
}

// ---- 3x3 symmetric helpers (storage: [a00,a01,a02,a11,a12,a22]) ----
// inverse of an SPD 3x3 through its Cholesky factor (what Ceres' InvertPSDMatrix<3> does); false if not PD
LFBA_HD bool spd3_inverse(const double a[6], double inv[6]) {
  const double l00s = a[0];
  if (!(l00s > 0.0)) return false;
  const double l00 = sqrt(l00s), i00 = 1.0 / l00;
  const double l10 = a[1] * i00, l20 = a[2] * i00;
  const double l11s = a[3] - l10 * l10;
  if (!(l11s > 0.0)) return false;
  const double l11 = sqrt(l11s), i11 = 1.0 / l11;
  const double l21 = (a[4] - l20 * l10) * i11;
  const double l22s = a[5] - l20 * l20 - l21 * l21;
  if (!(l22s > 0.0)) return false;
  const double l22 = sqrt(l22s), i22 = 1.0 / l22;
  // inverse of L (lower): m
  const double m10 = -l10 * i00 * i11;
  const double m21 = -l21 * i11 * i22;
  const double m20 = -(l20 * i00 + l21 * m10) * i22;
  // inv = L^-T L^-1
  inv[0] = i00 * i00 + m10 * m10 + m20 * m20;
  inv[1] = m10 * i11 + m20 * m21;
  inv[2] = m20 * i22;
  inv[3] = i11 * i11 + m21 * m21;
  inv[4] = m21 * i22;
  inv[5] = i22 * i22;
  return true;
}
LFBA_HD void sym3_vec(const double a[6], const double x[3], double y[3]) {
  y[0] = a[0] * x[0] + a[1] * x[1] + a[2] * x[2];
  y[1] = a[1] * x[0] + a[3] * x[1] + a[4] * x[2];
  y[2] = a[2] * x[0] + a[4] * x[1] + a[5] * x[2];
}

// a0 b0 + a1 b1 + a2 b2 with the roundings nvcc --fmad=true gives that expression (the middle product rounded, the
// other two fused), written out so that every kernel inlining the helpers below computes the same bits
LFBA_HD double dot3_fma(double a0, double b0, double a1, double b1, double a2, double b2) {
  return fma(a2, b2, fma(a0, b0, a1 * b1));
}

// ---- Pose-point coupling of one track, in the camera frame ----
// The pose x point block of J^T W J of track t = (p, f) is V = M^T B, with B = A R (A the track's 3 x 3 block, R the
// frame's rotation) and M = [dR0 X, dR1 X, dR2 X, I3] (3 x 6, d P_c / d pose). Every Schur term of a track has the form
// M^T (3 x 3) M or (3 x NC)^T M, so the point is eliminated inside the 3 x 3 camera-frame block and the result is
// projected onto the pose once; V and W = V Hpp^-1 are never formed. With Hi = (Hpp + D)^-1, K = B Hi and
// T_p = Hi Hcp^T (3 x NC, stored per point by k_points):
//     S_ff   += M^T (A - K B^T) M          g_f  += M^T (b - K g_p)          S_cf += (C - B T_p)^T M
//     S_f1f2 -= M1^T (K1 B2^T) M2           y_p   = Hi (g_p - sum_t B^T M y_f) - T_p y_c
// Every kernel builds these quantities with the helpers below, so all of them compute the same bits.
// Storage: 3 x 3 symmetric as upper [00 01 02 11 12 22], general 3 x 3 row-major, m[3 a + i] = (dR_a X)_i.

// m, the 3 x 3 part of M, from the frame-table entry fe (R, dR/da0..2) and the point X
LFBA_HD void track_m(const double* fe, const double* X, double m[9]) {
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const double* dR = fe + 9 * (a + 1);
#pragma unroll
    for (int i = 0; i < 3; ++i) m[3 * a + i] = dot3_fma(dR[3 * i], X[0], dR[3 * i + 1], X[1], dR[3 * i + 2], X[2]);
  }
}
// B = A R (A symmetric)
LFBA_HD void track_b(const double A[6], const double* R, double B[9]) {
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    B[j] = dot3_fma(A[0], R[j], A[1], R[3 + j], A[2], R[6 + j]);
    B[3 + j] = dot3_fma(A[1], R[j], A[3], R[3 + j], A[4], R[6 + j]);
    B[6 + j] = dot3_fma(A[2], R[j], A[4], R[3 + j], A[5], R[6 + j]);
  }
}
// K = B Hi (Hi symmetric)
LFBA_HD void mat3_sym3(const double B[9], const double Hi[6], double K[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double* b = B + 3 * i;
    K[3 * i] = dot3_fma(b[0], Hi[0], b[1], Hi[1], b[2], Hi[2]);
    K[3 * i + 1] = dot3_fma(b[0], Hi[1], b[1], Hi[3], b[2], Hi[4]);
    K[3 * i + 2] = dot3_fma(b[0], Hi[2], b[1], Hi[4], b[2], Hi[5]);
  }
}
// G = K B2^T (general 3 x 3)
LFBA_HD void mat3_mat3t(const double K[9], const double B2[9], double G[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)
      G[3 * i + j] = dot3_fma(K[3 * i], B2[3 * j], K[3 * i + 1], B2[3 * j + 1], K[3 * i + 2], B2[3 * j + 2]);
}
// A~ = A - K B^T, the track's camera-frame block with its point eliminated (symmetric: K B^T = B Hi B^T)
LFBA_HD void track_atilde(const double A[6], const double B[9], const double K[9], double At[6]) {
  int h = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = i; j < 3; ++j, ++h)
      At[h] = A[h] - dot3_fma(K[3 * i], B[3 * j], K[3 * i + 1], B[3 * j + 1], K[3 * i + 2], B[3 * j + 2]);
}
// acc += M^T S M for a symmetric 3 x 3 S: the lower triangle of the 6 x 6 pose block, row-major ((a, c <= a) at
// a (a + 1) / 2 + c)
LFBA_HD void mt_sym_m_acc(const double m[9], const double S[6], double acc[21]) {
  double Sm[9];
#pragma unroll
  for (int c = 0; c < 3; ++c) sym3_vec(S, m + 3 * c, Sm + 3 * c);
  int h = 0;
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int c = 0; c <= a; ++c, ++h) {
      if (a < 3) acc[h] += dot3_fma(m[3 * a], Sm[3 * c], m[3 * a + 1], Sm[3 * c + 1], m[3 * a + 2], Sm[3 * c + 2]);
      else if (c < 3) acc[h] += Sm[3 * c + a - 3];
      else acc[h] += S[3 * (c - 3) - (c - 3) * (c - 2) / 2 + (a - 3)];  // upper (c - 3, a - 3)
    }
}
// acc += s M^T v (6), s = +-1
LFBA_HD void mt_vec_acc(const double m[9], const double v[3], double s, double acc[6]) {
#pragma unroll
  for (int a = 0; a < 3; ++a) acc[a] += s * dot3_fma(m[3 * a], v[0], m[3 * a + 1], v[1], m[3 * a + 2], v[2]);
#pragma unroll
  for (int i = 0; i < 3; ++i) acc[3 + i] += s * v[i];
}
// acc += M1^T G M2 (6 x 6 row-major) for a general 3 x 3 G
LFBA_HD void mt_mat_m_acc(const double m1[9], const double G[9], const double m2[9], double acc[36]) {
  double GM[18];  // G M2, 3 x 6 row-major
#pragma unroll
  for (int i = 0; i < 3; ++i) {
#pragma unroll
    for (int b = 0; b < 3; ++b)
      GM[6 * i + b] = dot3_fma(G[3 * i], m2[3 * b], G[3 * i + 1], m2[3 * b + 1], G[3 * i + 2], m2[3 * b + 2]);
#pragma unroll
    for (int b = 0; b < 3; ++b) GM[6 * i + 3 + b] = G[3 * i + b];
  }
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int b = 0; b < 6; ++b)
      acc[6 * a + b] += a < 3 ? dot3_fma(m1[3 * a], GM[b], m1[3 * a + 1], GM[6 + b], m1[3 * a + 2], GM[12 + b])
                              : GM[6 * (a - 3) + b];
}
// W = M^T K (6 x 3 row-major): V Hi for K = B Hi
LFBA_HD void mt_mat(const double m[9], const double K[9], double W[18]) {
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int j = 0; j < 3; ++j) W[3 * a + j] = dot3_fma(m[3 * a], K[j], m[3 * a + 1], K[3 + j], m[3 * a + 2], K[6 + j]);
#pragma unroll
  for (int k = 0; k < 9; ++k) W[9 + k] = K[k];
}
// h += V^T y_f = R^T (A (M y_f)) for the pose step y_f (6) of the track's frame
LFBA_HD void track_vt_y_acc(const double A[6], const double* R, const double m[9], const double* yf, double h[3]) {
  double u[3], w[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) u[i] = yf[3 + i] + dot3_fma(m[i], yf[0], m[3 + i], yf[1], m[6 + i], yf[2]);
  sym3_vec(A, u, w);
#pragma unroll
  for (int j = 0; j < 3; ++j) h[j] += dot3_fma(R[j], w[0], R[3 + j], w[1], R[6 + j], w[2]);
}

// distance constraint (src/BundleAdjustment/BundleAdjustment.h:262-267): r = (|p1 - p2| - d) / (sigma + 1e-6),
// j = d r / d p1 = -(d r / d p2)
LFBA_HD void distance_eval(const double* p1, const double* p2, double dist, double sigma, double& r, double j[3]) {
  const double dx = p1[0] - p2[0], dy = p1[1] - p2[1], dz = p1[2] - p2[2];
  const double n = sqrt(dx * dx + dy * dy + dz * dz);
  const double w = 1.0 / (sigma + 0.000001);
  r = (n - dist) * w;
  const double f = w / n;
  j[0] = dx * f;
  j[1] = dy * f;
  j[2] = dz * f;
}

}  // namespace lfba
