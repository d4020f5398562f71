// lfba_kernels.cu — hand-written sm_100a FP64 kernels of the LF-BA Levenberg-Marquardt iteration.
//
// Reference being replaced: one ceres::Solve iteration over the problem built at
// src/CameraCalibration.cpp:858-953 (Ceres 2.1.0: ProgramEvaluator + AutoDiff of OurCostFunctionBundle,
// CauchyLoss/Corrector, SchurEliminator<2,3,Dynamic>, TrustRegionMinimizer; SURVEY.md Appendix B).
//
// Round structure (all on one stream, no host decisions; the host only polls LmState::done):
//   E  k_tables            per-lens undistortion table + per-frame rotation table at the CANDIDATE parameters
//      k_eval_rows         (lfba_rows.cu) fused residual + analytic Jacobian + robust weighting + per-track
//                          normal-equation blocks in the camera frame (A = G^T G, b = G^T r, C = G^T Jc) + camera
//                          block (Hcc, gc) + cost.  The Jacobian never leaves registers.
//      k_reduce_eval       deterministic reduction of the per-CTA partials; candidate scalars
//   C1 k_control_accept    step tests, rho, accept/reject (buffer flip), radius update   [device-resident LM]
//   B  k_points            per point: Hpp, g_p, Hcp; damping; 3x3 inverse; T_p = Hpp^-1 Hcp^T; camera-camera Schur term
//      k_frame_all         per frame: pose diagonal block, pose gradient, camera-pose block, Schur-corrected in the
//                          camera frame (+ k_frame_finish when a frame's tracks are split over several CTAs)
//      k_pairs             per co-visible frame pair: -sum_p M1^T (B1 Hpp^-1 B2^T) M2
//      k_coupled, k_constraints, k_add_camera
//   C2 k_finalize          Jacobi scaling (iteration 0), gradient norms, iteration row, termination tests,
//                          LM damping of the reduced system
//   S  (lfba_chol.cu)      Cholesky + solves of the reduced system
//   P  k_point_step        per-point back substitution, candidate point, model-cost/step-norm partials
//      k_reduced_step      candidate camera/poses/coupled points (manifold + bounds), reduced-part scalars
// Scatter into the reduced system is gather-by-destination (per frame, per frame pair): no atomics on the hot
// blocks and a fixed summation order.
#include <stdlib.h>
#include <cstdlib>
#include <float.h>
#include <cstdio>

#include "lfba_device.cuh"
#include "lfba_kernels.h"

namespace lfba {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ unsigned long long gtimer() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// entry (r, c), c <= r, of the skyline: closed form (SkyMap), no index loads
__device__ __forceinline__ double* S_at(const Dev& d, int r, int c) {
  const SkyMap m{d.band, d.np6};
  if (r < d.np6) {
    const int f = r / 6;
    return d.S + m.row(f, r - 6 * f) + (c - m.c0(f));
  }
  return d.S + m.border_row(r - d.np6) + c;
}

// Sum NV per-thread values over the CTA (fixed order: lanes by butterfly, warps ascending), result to out[0..NV).
template <int NV>
__device__ __forceinline__ void block_reduce_store(double* vals, double* out, double* smem /*[nwarps*NV]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const double s = warp_sum(vals[v]);
    if (lane == 0) smem[warp * NV + v] = s;
  }
  __syncthreads();
  for (int v = threadIdx.x; v < NV; v += blockDim.x) {
    double s = 0.0;
    for (int w = 0; w < nw; ++w) s += smem[w * NV + v];
    out[v] = s;
  }
  __syncthreads();
}

// ================================================================================================
// E. candidate evaluation
// ================================================================================================
__global__ void k_tables(Dev d) {
  const LmState* st = d.st;
  if (st->done || st->eval_skip) return;
  const int cand = 1 - st->cur;
  __shared__ CamModel cm;
  if (threadIdx.x == 0) {
    cam_model_init(cm, d.camera[cand], d.config, d.spx, d.spy, d.scale, d.opt.loss_a);
    if (blockIdx.x == 0 && d.cm_buf) *d.cm_buf = cm;  // -> __constant__ memory of the evaluation kernel (launch_eval)
  }
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < d.NL) {
    double e[kLensStride];
    lens_entry(cm, d.lens_xy[2 * i], d.lens_xy[2 * i + 1], e);
    double2* dst = reinterpret_cast<double2*>(d.lens + (size_t)i * kLensStride);
#pragma unroll
    for (int k = 0; k < kLensStride / 2; ++k) dst[k] = make_double2(e[2 * k], e[2 * k + 1]);
  }
  if (i < d.F) {
    double f[kFrameStride];
    frame_entry(d.views[cand] + 6 * i, f);
    double* dst = d.frames[cand] + (size_t)i * kFrameStride;
#pragma unroll
    for (int k = 0; k < kFrameStride; ++k) dst[k] = f[k];
  }
}

// The fused evaluation kernel itself is k_eval_rows (lfba_rows.cu).

// Sum the CTA partials of k_eval_rows (fixed order) -> camsum[cand]; sum the step partials of
// k_point_step (previous round); candidate cost of the distance constraints; assemble eval_scalars.
__global__ void __launch_bounds__(1024) k_reduce_eval(Dev d) {
  LmState* st = d.st;
  if (st->done) return;
  const int cand = 1 - st->cur;
  const int NH = d.NC * (d.NC + 1) / 2, NV = NH + d.NC + 1;
  __shared__ double sh[64];
  __shared__ double shs[8];
  __shared__ double sls[2];
  const int v = threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;  // 32 warps; a warp sums one value over the CTAs
  {  // lane = value (coalesced rows of the CTA partials), warps stride over the CTAs, warp partials added in warp order
    __shared__ double wp[32][64];
    for (int h2 = 0; h2 < 2; ++h2) {
      const int q = lane + 32 * h2;
      double s_ = 0.0;
      if (q < NV && !st->eval_skip)
        for (int b = warp; b < d.grid_eval; b += 32) s_ += d.part_eval[(size_t)b * 64 + q];
      wp[warp][q] = s_;
    }
    __syncthreads();
    if (v < 64) {
      double s_ = 0.0;
      for (int w = 0; w < 32; ++w) s_ += wp[w][v];
      sh[v] = s_;
      if (v < NV) d.camsum[cand][v] = s_;
    }
  }
  if (warp < 8) {
    const int k = warp;
    double s_ = 0.0;
    if (d.refine_points && (st->iter == 0 || st->solve_ok)) {
      if (k == 5) {  // slot 5 is a maximum: max |delta| over this rank's eliminated points
        for (int b = lane; b < d.grid_pts; b += 32) s_ = fmax(s_, d.part_step[(size_t)b * 8 + k]);
      } else {
        for (int b = lane; b < d.grid_pts; b += 32) s_ += d.part_step[(size_t)b * 8 + k];
      }
    }
    s_ = k == 5 ? warp_max(s_) : warp_sum(s_);
    if (lane == 0) shs[k] = s_;
  } else if (warp == 8) {  // recalib: gradient(candidate) . delta over this rank's tracks (k_ls_gdot)
    double s_ = 0.0;
    if (d.recalib && !st->eval_skip && st->iter > 0)
      for (int b = lane; b < d.grid_pts; b += 32) s_ += d.part_ls[b];
    s_ = warp_sum(s_);
    if (lane == 0) sls[0] = s_;
  }
  __syncthreads();
  if (v == 0) {
    double cost = sh[NV - 1];
    if (d.rank == 0 && !st->eval_skip) {
      const double* pts = d.points[cand];
      for (int k = 0; k < d.K; ++k) {
        double r, j[3];
        distance_eval(pts + 3 * d.c_p1[k], pts + 3 * d.c_p2[k], d.c_dist[k], d.c_sigma[k], r, j);
        cost += 0.5 * r * r;
      }
    }
    double* es = d.eval_scalars;
    es[ES_COST] = cost;
    const double own = d.rank == 0 ? 1.0 : 0.0;
    es[ES_MCC] = shs[0] + own * st->mcc_red;
    es[ES_STEP2] = shs[1] + own * st->step2_red;
    es[ES_NORM2] = shs[2] + own * st->norm2_red;
    es[ES_GDELTA] = shs[3] + own * st->gdelta_red;
    es[ES_BAD] = shs[4];
    double lsgd = 0.0;
    if (d.recalib && !st->eval_skip && st->iter > 0) {
      // camera part of gradient(candidate) . delta: this rank's share of g_c (camsum) times delta_c = -y_c
      lsgd = sls[0];
      for (int c = 0; c < d.NC; ++c) {
        const int r = d.cam_red[c];
        if (r >= 0) lsgd += sh[NH + c] * (-d.y[r]);
      }
    }
    es[ES_LSGD] = lsgd;
    es[7] = 0.0;
    for (int r = 0; r < d.nranks; ++r) es[ES_COUNT + r] = r == d.rank ? fmax(shs[5], own * st->dmax_red) : 0.0;
  }
}

// ---- projected Armijo line search (Ceres ArmijoLineSearch with CUBIC interpolation; line_search.cc, polynomial.cc) ----
struct LsSample {
  double x, value, gradient;
  int value_valid, gradient_valid;
};
__device__ double ls_ipow(double x, int e) {
  double r = 1.0;
  for (int i = 0; i < e; ++i) r *= x;
  return r;
}
// Polynomial through the samples' values and (where valid) gradients, minimised on [lo, hi]: end points and the
// stationary points inside (sign changes of p' on a 4096-point grid, bisected).
__device__ double ls_minimize_interpolant(const LsSample* smp, int ns, double lo, double hi) {
  int ncon = 0;
  for (int i = 0; i < ns; ++i) ncon += (smp[i].value_valid ? 1 : 0) + (smp[i].gradient_valid ? 1 : 0);
  const int deg = ncon - 1;
  double A[36], b[6], coef[6];
  for (int i = 0; i < 36; ++i) A[i] = 0.0;
  int row = 0;
  for (int i = 0; i < ns; ++i) {
    if (smp[i].value_valid) {
      for (int j = 0; j <= deg; ++j) A[row * ncon + j] = ls_ipow(smp[i].x, deg - j);
      b[row++] = smp[i].value;
    }
    if (smp[i].gradient_valid) {
      for (int j = 0; j < deg; ++j) A[row * ncon + j] = (deg - j) * ls_ipow(smp[i].x, deg - j - 1);
      b[row++] = smp[i].gradient;
    }
  }
  for (int c = 0; c < ncon; ++c) {  // Gaussian elimination, partial pivoting
    int piv = c;
    for (int i = c + 1; i < ncon; ++i)
      if (fabs(A[i * ncon + c]) > fabs(A[piv * ncon + c])) piv = i;
    for (int j = 0; j < ncon; ++j) {
      const double t = A[c * ncon + j];
      A[c * ncon + j] = A[piv * ncon + j];
      A[piv * ncon + j] = t;
    }
    const double tb = b[c];
    b[c] = b[piv];
    b[piv] = tb;
    const double dd = A[c * ncon + c];
    if (dd == 0.0) continue;
    for (int i = c + 1; i < ncon; ++i) {
      const double f = A[i * ncon + c] / dd;
      for (int j = c; j < ncon; ++j) A[i * ncon + j] -= f * A[c * ncon + j];
      b[i] -= f * b[c];
    }
  }
  for (int i = ncon - 1; i >= 0; --i) {  // coefficients, highest degree first
    double s_ = b[i];
    for (int j = i + 1; j < ncon; ++j) s_ -= A[i * ncon + j] * coef[j];
    coef[i] = A[i * ncon + i] != 0.0 ? s_ / A[i * ncon + i] : 0.0;
  }
  auto poly = [&](double x) {
    double v = 0.0;
    for (int j = 0; j <= deg; ++j) v = v * x + coef[j];
    return v;
  };
  auto dpoly = [&](double x) {
    double v = 0.0;
    for (int j = 0; j < deg; ++j) v = v * x + (deg - j) * coef[j];
    return v;
  };
  double best_x = lo, best_v = poly(lo);
  if (poly(hi) < best_v) {
    best_v = poly(hi);
    best_x = hi;
  }
  const int G = 4096;
  double xa = lo, da = dpoly(lo);
  for (int i = 1; i <= G; ++i) {
    const double xb = lo + (hi - lo) * i / G, db = dpoly(xb);
    if ((da <= 0 && db >= 0) || (da >= 0 && db <= 0)) {
      double l = xa, h = xb, dl = da;
      for (int it = 0; it < 100; ++it) {
        const double m = 0.5 * (l + h), dm = dpoly(m);
        if ((dl <= 0 && dm <= 0) || (dl >= 0 && dm >= 0)) {
          l = m;
          dl = dm;
        } else {
          h = m;
        }
      }
      const double xm = 0.5 * (l + h), vm = poly(xm);
      if (vm < best_v) {
        best_v = vm;
        best_x = xm;
      }
    }
    xa = xb;
    da = db;
  }
  return best_x;
}

// ================================================================================================
// C1. accept / reject — ceres::internal::TrustRegionMinimizer::Minimize loop body after the candidate
// evaluation (DoLineSearch for bounds-constrained problems, ParameterToleranceReached, FunctionToleranceReached,
// IsStepSuccessful, HandleSuccessfulStep / StepRejected / HandleInvalidStep) and
// LevenbergMarquardtStrategy::StepAccepted/StepRejected.
// ================================================================================================
__global__ void k_control_accept(Dev d) {
  LmState* st = d.st;
  if (st->done) return;
  const double* es = d.eval_scalars;
  const Options& o = d.opt;
  lfba_iteration& row = st->row;
  if (st->iter == 0) {  // IterationZero
    st->t_start = st->t_iter = gtimer();
    st->cur ^= 1;
    st->x_cost = es[ES_COST];
    st->x_norm2 = es[ES_NORM2];
    st->min_cost = DBL_MAX;
    st->first = 1;
    st->n_jac_evals = 1;
    row.iteration = 0;
    row.step_is_valid = 1;
    row.step_is_successful = 1;
    row.line_search_iterations = 0;
    row.cost = st->x_cost;
    row.cost_change = 0.0;
    row.step_norm = 0.0;
    row.relative_decrease = 0.0;
    st->pending_row = 1;
    return;
  }
  row.iteration = st->iter;
  row.line_search_iterations = 0;
  const double mcc = es[ES_MCC];
  const bool valid = !st->eval_skip && st->solve_ok && es[ES_BAD] == 0.0 && mcc > 0.0;
  if (!valid) {  // HandleInvalidStep
    st->ls_active = st->ls_failed = st->ls_iters = 0;
    if (++st->num_invalid >= o.max_invalid) {
      st->done = 1;
      st->termination = LFBA_TERM_FAILURE;
      st->stop_reason = LFBA_STOP_INVALID_STEPS;
      st->status = LFBA_FAILURE;
      return;
    }
    st->radius = st->radius / st->decrease_factor;
    st->decrease_factor *= 2.0;
    row.step_is_valid = 0;
    row.step_is_successful = 0;
    row.cost = st->x_cost;
    row.cost_change = 0.0;
    row.step_norm = 0.0;
    row.relative_decrease = 0.0;
    st->pending_row = 1;
    return;
  }
  st->num_invalid = 0;
  st->n_jac_evals += 1;
  double cand_cost = es[ES_COST];
  const bool cost_finite = isfinite(cand_cost);
  if (!cost_finite) cand_cost = DBL_MAX;
  row.step_is_valid = 1;
  if (d.recalib) {
    // Bounds make Ceres search along delta from step size 1 on phi(a) = cost(Plus(x, a delta)) (projected: Plus clamps
    // to the box) until phi(a) <= phi(0) + 1e-4 a phi'(0); contraction by minimising the polynomial through phi(0),
    // phi'(0) and value + gradient of the last two trials, inside [1e-3, 0.6] a; at most 20 trials, a |delta|_inf >= 1e-9.
    // The candidate just evaluated IS the current trial (a = 1 for the first one): its cost and phi'(a) = g(x_a).delta
    // came with the fused evaluation pass, no extra evaluation is needed when a = 1 is accepted.
    if (st->ls_failed) {  // search gave up earlier: this is the full step again, taken as Ceres does (delta unchanged)
      st->ls_failed = 0;
      st->ls_active = 0;
      row.line_search_iterations = st->ls_iters;
    } else {
      LsSample cur;
      cur.x = st->ls_active ? st->ls_alpha : 1.0;
      cur.value = cand_cost;
      cur.value_valid = cost_finite ? 1 : 0;
      cur.gradient = es[ES_LSGD];
      cur.gradient_valid = (cost_finite && isfinite(cur.gradient)) ? 1 : 0;
      if (!st->ls_active) {
        st->ls_phi0 = st->x_cost;
        st->ls_dphi0 = es[ES_GDELTA];
        st->ls_iters = 0;
        st->ls_prev_valid = st->ls_prev_gvalid = 0;
      }
      const bool armijo = cur.value_valid && cur.value <= st->ls_phi0 + 1e-4 * st->ls_dphi0 * cur.x;
      if (d.debug)
        printf("[lfba dbg] iter %d line search: a=%.17g phi=%.17g dphi=%.17g | phi0=%.17g dphi0=%.17g armijo=%d trials=%d\n",
               st->iter, cur.x, cur.value, cur.gradient, st->ls_phi0, st->ls_dphi0, (int)armijo, st->ls_iters);
      if (!armijo) {
        bool fail = ++st->ls_iters >= 20;
        double a_new = 1.0;
        if (!fail) {
          const double lo = 1e-3 * cur.x, hi = 0.6 * cur.x;
          if (!cur.value_valid) {
            a_new = fmin(fmax(cur.x * 0.5, lo), hi);
          } else {
            LsSample smp[3];
            int ns = 0;
            smp[ns].x = 0.0;
            smp[ns].value = st->ls_phi0;
            smp[ns].gradient = st->ls_dphi0;
            smp[ns].value_valid = smp[ns].gradient_valid = 1;
            ++ns;
            smp[ns++] = cur;
            if (st->ls_prev_valid) {
              smp[ns].x = st->ls_prev_x;
              smp[ns].value = st->ls_prev_v;
              smp[ns].gradient = st->ls_prev_g;
              smp[ns].value_valid = 1;
              smp[ns].gradient_valid = st->ls_prev_gvalid;
              ++ns;
            }
            a_new = ls_minimize_interpolant(smp, ns, lo, hi);
          }
          double dmax = 0.0;
          for (int r = 0; r < d.nranks; ++r) dmax = fmax(dmax, es[ES_COUNT + r]);
          if (a_new * dmax < 1e-9) fail = true;
        }
        if (fail) {
          if (st->ls_active) {  // back to the full step: one more evaluation at a = 1
            st->ls_failed = 1;
            st->ls_alpha = 1.0;
            st->ls_trial = 1;
            return;
          }
          // the failed trial was a = 1 itself: its evaluation is the candidate
          row.line_search_iterations = st->ls_iters;
        } else {
          st->ls_prev_x = cur.x;
          st->ls_prev_v = cur.value;
          st->ls_prev_g = cur.gradient;
          st->ls_prev_valid = cur.value_valid;
          st->ls_prev_gvalid = cur.gradient_valid;
          st->ls_active = 1;
          st->ls_alpha = a_new;
          st->ls_trial = 1;
          return;
        }
      } else {
        row.line_search_iterations = st->ls_iters;  // delta <- a delta: the candidate already is Plus(x, a delta)
      }
      st->ls_active = 0;
    }
  }
  row.step_norm = sqrt(es[ES_STEP2]);
  if (row.step_norm <= o.ptol * (sqrt(st->x_norm2) + o.ptol)) {
    st->done = 1;
    st->termination = LFBA_CONVERGENCE;
    st->stop_reason = LFBA_STOP_PARAMETER_TOLERANCE;
    return;
  }
  row.cost_change = st->x_cost - cand_cost;
  if (fabs(row.cost_change) <= o.ftol * st->x_cost) {
    st->done = 1;
    st->termination = LFBA_CONVERGENCE;
    st->stop_reason = LFBA_STOP_FUNCTION_TOLERANCE;
    return;
  }
  row.relative_decrease = cand_cost >= DBL_MAX ? -DBL_MAX : (st->x_cost - cand_cost) / mcc;
  if (row.relative_decrease > o.min_rel_dec) {
    st->cur ^= 1;
    st->x_cost = cand_cost;
    st->x_norm2 = es[ES_NORM2];
    row.cost = cand_cost;
    row.step_is_successful = 1;
    const double q = 2.0 * row.relative_decrease - 1.0;
    st->radius = st->radius / fmax(1.0 / 3.0, 1.0 - q * q * q);
    st->radius = fmin(o.rmax, st->radius);
    st->decrease_factor = 2.0;
  } else {
    row.step_is_successful = 0;
    row.cost = cand_cost;
    st->radius = st->radius / st->decrease_factor;
    st->decrease_factor *= 2.0;
  }
  st->pending_row = 1;
}

// ---- line-search support kernels (recalib only) ----
// phi'(a) = gradient(x_a) . delta at the candidate x_a just evaluated: per track, b_t = G^T r (camera frame, from the
// fused pass) against the motion of the camera-frame point along delta, R delta_p + M delta_f. Fixed-order partials.
__global__ void __launch_bounds__(128) k_ls_gdot(Dev d) {
  LmState* st = d.st;
  if (st->done || st->eval_skip || st->iter == 0) return;
  const int cand = 1 - st->cur;
  const int RS = rec_stride(d.NC);
  __shared__ double red[4];
  double acc = 0.0;
  const double* __restrict__ recs = d.rec[cand];
  const double* __restrict__ frames = d.frames[cand];
  const double* __restrict__ points = d.points[cand];
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < d.T; t += gridDim.x * blockDim.x) {
    const int p = d.trk_point[t], f = d.trk_frame[t];
    const double* fe = frames + (size_t)f * kFrameStride;
    const double* b = recs + (size_t)t * RS + 6;
    double mv[3] = {0.0, 0.0, 0.0};
    if (d.refine_points) {
      const double* dp = d.pstep + 3 * (size_t)p;
      mat3_vec(fe, dp, mv);
    }
    if (d.refine_poses) {
      const double* X = points + 3 * (size_t)p;
      const double* yf = d.y + 6 * f;
      double m[9];
      mat3_vec(fe + 9, X, m + 0);
      mat3_vec(fe + 18, X, m + 3);
      mat3_vec(fe + 27, X, m + 6);
#pragma unroll
      for (int i = 0; i < 3; ++i) mv[i] += -(m[i] * yf[0] + m[3 + i] * yf[1] + m[6 + i] * yf[2]) - yf[3 + i];
    }
    acc += b[0] * mv[0] + b[1] * mv[1] + b[2] * mv[2];
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) d.part_ls[blockIdx.x] = (red[0] + red[1]) + (red[2] + red[3]);
}

// A pending contraction trial: candidate := Plus(x, a delta) for the eliminated points, with their share of |x - x+|^2
// and |x+|^2 (the slots of k_point_step's partials that depend on the candidate).
__global__ void __launch_bounds__(128) k_ls_apply(Dev d) {
  LmState* st = d.st;
  if (st->done || !st->ls_trial || !d.refine_points) return;
  const int cur = st->cur, cand = 1 - cur;
  const double a = st->ls_alpha;
  __shared__ double red[4 * 2];
  double acc[2] = {0.0, 0.0};
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < d.P; p += gridDim.x * blockDim.x) {
    if (!d.pt_active[p] || d.pt_coupled[p] >= 0) continue;
    const double* X = d.points[cur] + 3 * (size_t)p;
    double* Xc = d.points[cand] + 3 * (size_t)p;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double xn = X[j] + a * d.pstep[3 * (size_t)p + j];
      Xc[j] = xn;
      const double dl = xn - X[j];
      acc[0] += dl * dl;
      acc[1] += xn * xn;
    }
  }
  double out[2];
  {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int v = 0; v < 2; ++v) {
      const double s_ = warp_sum(acc[v]);
      if (lane == 0) red[warp * 2 + v] = s_;
    }
    __syncthreads();
    for (int v = 0; v < 2; ++v) out[v] = (red[v] + red[2 + v]) + (red[4 + v] + red[6 + v]);
  }
  if (threadIdx.x == 0) {
    d.part_step[(size_t)blockIdx.x * 8 + 1] = out[0];
    d.part_step[(size_t)blockIdx.x * 8 + 2] = out[1];
  }
}

// ... and for the reduced parameters (camera with manifold + bounds, poses, coupled points). Last kernel of a trial
// round: clears the flag.
__global__ void __launch_bounds__(256) k_ls_apply_reduced(Dev d) {
  LmState* st = d.st;
  if (st->done || !st->ls_trial) return;
  const int cur = st->cur, cand = 1 - cur;
  const double a = st->ls_alpha;
  __shared__ double red[8 * 8];
  __shared__ double out[8];
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const double* y = d.y;
  for (int j = threadIdx.x; j < d.np6; j += blockDim.x) {
    const double x = d.views[cur][j];
    const double xn = x + a * (-y[j]);
    d.views[cand][j] = xn;
    if (d.frm_active[j / 6]) {
      const double dl = xn - x;
      acc[1] += dl * dl;
      acc[2] += xn * xn;
    }
  }
  for (int j = threadIdx.x; j < 3 * d.Pc; j += blockDim.x) {
    const int r = d.np6 + j;
    const int p = d.coupled_pts[j / 3];
    const double x = d.points[cur][3 * (size_t)p + j % 3];
    const double xn = x + a * (-y[r]);
    d.points[cand][3 * (size_t)p + j % 3] = xn;
    const double dl = xn - x;
    acc[1] += dl * dl;
    acc[2] += xn * xn;
  }
  for (int c = threadIdx.x; c < 17; c += blockDim.x) {
    const double x = d.camera[cur][c];
    double xn = x;
    const int r = c < d.NC ? d.cam_red[c] : -1;
    if (r >= 0) xn = x + a * (-y[r]);
    xn = fmin(fmax(xn, d.cam_lo[c]), d.cam_hi[c]);
    d.camera[cand][c] = xn;
    const double dl = xn - x;
    acc[1] += dl * dl;
    acc[2] += xn * xn;
  }
  block_reduce_store<8>(acc, out, red);
  if (threadIdx.x == 0) {
    st->step2_red = out[1];
    st->norm2_red = out[2];
    st->ls_trial = 0;
  }
}

// ================================================================================================
// B. system assembly at the accepted state
// ================================================================================================
// Per point: Hpp = sum_t R^T A_t R, g_p = sum_t R^T b_t, Hcp = sum_t C_t^T R  (E-block of SchurEliminator),
// Jacobi scale (iteration 0), LM damping, inverse Hi of the damped block, T_p = Hi Hcp^T, camera-camera Schur term.
template <int NC>
__global__ void __launch_bounds__(128) k_points(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  const int cur = st->cur;
  constexpr int NH = NC * (NC + 1) / 2;
  constexpr int NV = NH + NC + 3;  // Schur cam-cam (NH), Schur cam gradient (NC), |g|^2, fail count, (max separately)
  constexpr int RS = rec_stride(NC);
  __shared__ double red[4 * NV];
  __shared__ double redmax[4];
  double acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = 0.0;
  double gmax = 0.0;
  const double mu = st->radius;
  const bool first = st->first != 0;
  const double* __restrict__ frames = d.frames[cur];
  const double* __restrict__ recs = d.rec[cur];

  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < d.P; p += gridDim.x * blockDim.x) {
    if (!d.pt_active[p]) continue;
    double* pd = d.pdata + (size_t)p * kPointStride;
    if (d.pt_coupled[p] >= 0) {  // stays in the reduced system (k_coupled); no elimination
      for (int k = 0; k < kPointStride; ++k) pd[k] = 0.0;
      continue;
    }
    double H[6] = {0, 0, 0, 0, 0, 0}, gp[3] = {0, 0, 0}, Hcp[3 * NC];
#pragma unroll
    for (int k = 0; k < 3 * NC; ++k) Hcp[k] = 0.0;
    for (int t = d.pt_trk_begin[p]; t < d.pt_trk_begin[p + 1]; ++t) {
      // a lane reads ITS track record (288 B for NC = 9): wide loads cut the L1 wavefronts of this strided access
      double rc[RS + 3];
      load_record<RS, RS % 4 == 0>(recs + (size_t)t * RS, rc);
      const double* R = frames + (size_t)d.trk_frame[t] * kFrameStride;
      const double A[6] = {rc[0], rc[1], rc[2], rc[3], rc[4], rc[5]};
      double AR[9];
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        AR[0 + j] = A[0] * R[j] + A[1] * R[3 + j] + A[2] * R[6 + j];
        AR[3 + j] = A[1] * R[j] + A[3] * R[3 + j] + A[4] * R[6 + j];
        AR[6 + j] = A[2] * R[j] + A[4] * R[3 + j] + A[5] * R[6 + j];
      }
      H[0] += R[0] * AR[0] + R[3] * AR[3] + R[6] * AR[6];
      H[1] += R[0] * AR[1] + R[3] * AR[4] + R[6] * AR[7];
      H[2] += R[0] * AR[2] + R[3] * AR[5] + R[6] * AR[8];
      H[3] += R[1] * AR[1] + R[4] * AR[4] + R[7] * AR[7];
      H[4] += R[1] * AR[2] + R[4] * AR[5] + R[7] * AR[8];
      H[5] += R[2] * AR[2] + R[5] * AR[5] + R[8] * AR[8];
#pragma unroll
      for (int j = 0; j < 3; ++j) gp[j] += R[j] * rc[6] + R[3 + j] * rc[7] + R[6 + j] * rc[8];
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const double c0 = rc[9 + c], c1 = rc[9 + NC + c], c2 = rc[9 + 2 * NC + c];
#pragma unroll
        for (int j = 0; j < 3; ++j) Hcp[3 * c + j] += c0 * R[j] + c1 * R[3 + j] + c2 * R[6 + j];
      }
    }
    const double hd[3] = {H[0], H[3], H[5]};
    double* ps = d.pscale + 3 * (size_t)p;
    if (first)
      for (int j = 0; j < 3; ++j) ps[j] = 1.0 / (1.0 + sqrt(hd[j]));
    double dmp[3];
    for (int j = 0; j < 3; ++j) {
      const double s2 = ps[j] * ps[j];
      dmp[j] = d.undamped ? 0.0 : fmin(fmax(s2 * hd[j], d.opt.min_diag), d.opt.max_diag) / (mu * s2);
    }
    const double Hd[6] = {H[0] + dmp[0], H[1], H[2], H[3] + dmp[1], H[4], H[5] + dmp[2]};
    double Hi[6];
    if (!spd3_inverse(Hd, Hi)) {
      acc[NH + NC + 1] += 1.0;
      for (int k = 0; k < 6; ++k) Hi[k] = 0.0;
    }
    // T_p = Hi Hcp^T (NC x 3 here: Tm[3 c + j]): the point record's camera coupling and the camera-camera Schur term
    double Tm[3 * NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) sym3_vec(Hi, Hcp + 3 * c, Tm + 3 * c);
    // camera-camera Schur term: -(Hcp Hi) Hcp^T, -(Hcp Hi) g_p
    int h = 0;
#pragma unroll
    for (int c1 = 0; c1 < NC; ++c1)
#pragma unroll
      for (int c2 = 0; c2 <= c1; ++c2) {
        acc[h] -= Tm[3 * c1] * Hcp[3 * c2] + Tm[3 * c1 + 1] * Hcp[3 * c2 + 1] + Tm[3 * c1 + 2] * Hcp[3 * c2 + 2];
        ++h;
      }
#pragma unroll
    for (int c = 0; c < NC; ++c) acc[NH + c] -= Tm[3 * c] * gp[0] + Tm[3 * c + 1] * gp[1] + Tm[3 * c + 2] * gp[2];
    acc[NH + NC] += gp[0] * gp[0] + gp[1] * gp[1] + gp[2] * gp[2];
    {  // 320-byte record, 32-byte aligned: ten 256-bit stores (forty 8-byte stores cost forty times 32 L1 wavefronts per warp)
      double pv[kPointStride];
#pragma unroll
      for (int k = 0; k < 6; ++k) pv[k] = Hi[k];
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        pv[6 + k] = gp[k];
        pv[9 + k] = dmp[k];
      }
#pragma unroll
      for (int k = 0; k < kPointStride - 12; ++k) pv[12 + k] = k < 3 * NC ? Tm[k] : 0.0;
#pragma unroll
      for (int k = 0; k < kPointStride / 4; ++k) stg256(pd + 4 * k, pv[4 * k], pv[4 * k + 1], pv[4 * k + 2], pv[4 * k + 3]);
    }
    gmax = fmax(gmax, fmax(fabs(gp[0]), fmax(fabs(gp[1]), fabs(gp[2]))));
  }
  block_reduce_store<NV>(acc, d.part_pts + (size_t)blockIdx.x * 64, red);
  gmax = warp_max(gmax);
  if ((threadIdx.x & 31) == 0) redmax[threadIdx.x >> 5] = gmax;
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    for (int w = 0; w < (int)((blockDim.x + 31) >> 5); ++w) m = fmax(m, redmax[w]);
    d.part_pts[(size_t)blockIdx.x * 64 + 63] = m;
  }
}

// M = [dR0 X, dR1 X, dR2 X, I3] (3x6, d P_c / d pose) of a track
__device__ __forceinline__ void track_M(const double* fe, const double* X, double m[9]) {
  mat3_vec(fe + 9, X, m + 0);
  mat3_vec(fe + 18, X, m + 3);
  mat3_vec(fe + 27, X, m + 6);
}

// entry v of k_frame_all's per-frame sums -> its place in the reduced system
template <int NC>
__device__ __forceinline__ void frame_all_scatter(const Dev& d, int f, int v, double sv) {
  constexpr int NP = 21 + 6 + 6 + 6;
  double* dst = nullptr;
  if (v < 21) {
    int a = 0, h = v;
    while (h > a) { h -= a + 1; ++a; }
    dst = S_at(d, 6 * f + a, 6 * f + h);
  } else if (v < 27) {
    dst = d.g + 6 * f + (v - 21);
  } else if (v < 33) {
    dst = d.gfull + 6 * f + (v - 27);
  } else if (v < NP) {
    dst = d.hdiag + 6 * f + (v - 33);
  } else {
    const int c = (v - NP) / 6, a = (v - NP) % 6;
    const int r = d.cam_red[c];
    if (r >= 0) dst = S_at(d, r, 6 * f + a);
  }
  if (dst) *dst += sv;
}

template <int NC>
__global__ void __launch_bounds__(128) k_frame_all(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  const int cur = st->cur;
  // split index fastest: the CTAs in flight at any time cover FEW frames, whose points' records (each point is seen by a
  // handful of neighbouring frames) are then still in L2 when the next frame asks for them
  const int split = blockIdx.x, nsplit = gridDim.x;
  constexpr int RS = rec_stride(NC);
  constexpr int NP = 21 + 6 + 6 + 6;  // S_ff (lower 21), reduced gradient, full gradient, diag(F^T F)
  constexpr int NV = NP + 6 * NC;     // + camera-pose block
  __shared__ double fe[kFrameStride];
  __shared__ double red[4 * NV];
  __shared__ double out[NV];
  // The NP pose-side sums (each updated once per track) are kept per thread in shared memory, [v][thread]: the
  // registers then hold only the 6 NC camera-pose sums, and the loop-carried accumulators no longer spill.
  __shared__ double sacc[NP * 128];  // launched with 128 threads
  double* const my = sacc + threadIdx.x;
  for (int f = blockIdx.y; f < d.F; f += gridDim.y) {  // (one frame per CTA unless F exceeds the grid limit)
  __syncthreads();
  if (threadIdx.x < kFrameStride) fe[threadIdx.x] = d.frames[cur][(size_t)f * kFrameStride + threadIdx.x];
  __syncthreads();
  double acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = 0.0;
#pragma unroll
  for (int v = 0; v < NP; ++v) my[128 * v] = 0.0;
  const double* __restrict__ recs = d.rec[cur];
  const double* __restrict__ points = d.points[cur];
  for (int idx = d.frm_begin[f] + split * blockDim.x + threadIdx.x; idx < d.frm_begin[f + 1];
       idx += nsplit * blockDim.x) {
    const int t = d.frm_trk[idx];
    const int p = d.trk_point[t];
    // first the 3x3 part of the record and of the point data (A, b | Hpp^-1, g_p); the camera parts are loaded after
    // the pose block is done, so that they are not live across it
    const double* rcp = recs + (size_t)t * RS;
    const double2* pd2 = reinterpret_cast<const double2*>(d.pdata + (size_t)p * kPointStride);
    double rc[12], pd[12];
    if (RS % 4 == 0) {  // records are 32-byte aligned: 256-bit loads (one sector per instruction and lane)
#pragma unroll
      for (int k = 0; k < 3; ++k) ldg256(rcp + 4 * k, rc + 4 * k);
    } else if (RS % 2 == 0) {
#pragma unroll
      for (int k = 0; k < 5; ++k) {
        const double2 v2 = __ldg(reinterpret_cast<const double2*>(rcp) + k);
        rc[2 * k] = v2.x;
        rc[2 * k + 1] = v2.y;
      }
    } else {
#pragma unroll
      for (int k = 0; k < 10; ++k) rc[k] = __ldg(rcp + k);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) ldg256(d.pdata + (size_t)p * kPointStride + 4 * k, pd + 4 * k);  // 320-byte records
    const double A[6] = {rc[0], rc[1], rc[2], rc[3], rc[4], rc[5]};
    const double b[3] = {rc[6], rc[7], rc[8]};
    double m[9], B[9];
    track_m(fe, points + 3 * (size_t)p, m);
    track_b(A, fe, B);
    {  // pose block and gradients, the point eliminated in the camera frame: A~ = A - K B^T, b~ = b - K g_p (K = B Hi)
      double lp[NP];
#pragma unroll
      for (int v = 0; v < NP; ++v) lp[v] = 0.0;
      double K[9];
      {
        const double Hi[6] = {pd[0], pd[1], pd[2], pd[3], pd[4], pd[5]};
        mat3_sym3(B, Hi, K);
      }
      double At[6];
      track_atilde(A, B, K, At);
      mt_sym_m_acc(m, At, lp);
      double bt[3];
      {
        const double gp[3] = {pd[6], pd[7], pd[8]};
        mat3_vec(K, gp, bt);
      }
#pragma unroll
      for (int i = 0; i < 3; ++i) bt[i] = b[i] - bt[i];
      mt_vec_acc(m, bt, 1.0, lp + 21);
      mt_vec_acc(m, b, 1.0, lp + 27);
      // diag(M^T A M), un-complemented
#pragma unroll
      for (int a = 0; a < 3; ++a) {
        double y[3];
        sym3_vec(A, m + 3 * a, y);
        lp[33 + a] = dot3_fma(m[3 * a], y[0], m[3 * a + 1], y[1], m[3 * a + 2], y[2]);
      }
      lp[36] = A[0];
      lp[37] = A[3];
      lp[38] = A[5];
#pragma unroll
      for (int v = 0; v < NP; ++v) my[128 * v] += lp[v];
    }
    // camera-pose block: (C - B T_p)^T M, streamed in memory order in 256-bit pieces — no register copy of the two
    // 3 x NC blocks (they were 104 registers beside the 93 accumulators, most of the spill traffic). C is 3 x NC row-major
    // at doubles 9 .. of the track record: value (i, c) adds C_ic m[3a + i] to entry (c, a < 3) and itself to entry
    // (c, 3 + i). T_p is NC x 3 at doubles 12 .. of the point record: the three values of camera c give (B T_p)_c, whose
    // projection M^T (B T_p)_c is subtracted from entries (c, 0..5).
    {
      static_assert(RS % 4 == 0, "records are whole 32-byte sectors");
      auto add_c = [&](int k, double v) {  // k: index into C, compile-time after unrolling
        const int i = k / NC, c = k - i * NC;
#pragma unroll
        for (int a = 0; a < 3; ++a) acc[NP + 6 * c + a] = fma(v, m[3 * a + i], acc[NP + 6 * c + a]);
        acc[NP + 6 * c + 3 + i] += v;
      };
      double bt[3];
      auto sub_t = [&](int k, double v) {  // k: index into T_p
        const int c = k / 3, jj = k - 3 * c;
#pragma unroll
        for (int i = 0; i < 3; ++i) bt[i] = jj == 0 ? B[3 * i] * v : fma(B[3 * i + jj], v, bt[i]);
        if (jj == 2) mt_vec_acc(m, bt, -1.0, acc + NP + 6 * c);
      };
      add_c(0, rc[9]);
      add_c(1, rc[10]);
      add_c(2, rc[11]);
#pragma unroll
      for (int q = 3; q < RS / 4; ++q) {
        double t4[4];
        ldg256(rcp + 4 * q, t4);
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * q + e - 9 < 3 * NC) add_c(4 * q + e - 9, t4[e]);
      }
#pragma unroll
      for (int q = 3; q < kPointStride / 4; ++q) {
        double t4[4];
        ldg256(d.pdata + (size_t)p * kPointStride + 4 * q, t4);
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (4 * q + e - 12 < 3 * NC) sub_t(4 * q + e - 12, t4[e]);
      }
    }
  }
#pragma unroll
  for (int v = 0; v < NP; ++v) acc[v] = my[128 * v];
  block_reduce_store<NV>(acc, out, red);
  if (threadIdx.x < NV) {
    if (nsplit == 1) frame_all_scatter<NC>(d, f, threadIdx.x, out[threadIdx.x]);
    else d.frame_part[((size_t)f * nsplit + split) * NV + threadIdx.x] = out[threadIdx.x];  // summed by k_frame_finish
  }
  }
}

// Second stage when a frame is split over several CTAs (few active frames per rank: multi-GPU shards): the partial sums
// are added in split order — no atomics, the same bits every run.
template <int NC>
__global__ void __launch_bounds__(128) k_frame_finish(Dev d, int nsplit) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  constexpr int NV = 21 + 6 + 6 + 6 + 6 * NC;
  const int f = blockIdx.x, v = threadIdx.x;
  if (v >= NV) return;
  double sv = 0.0;
  for (int sp = 0; sp < nsplit; ++sp) sv += d.frame_part[((size_t)f * nsplit + sp) * NV + v];
  frame_all_scatter<NC>(d, f, v, sv);
}

// Per co-visible frame pair (f1 > f2): S[f1, f2] = -sum_p W_{p,f1} V_{p,f2}^T = -sum_p M1^T (B1 Hi B2^T) M2, factored
// through the 3 x 3 camera-frame product (the helpers k_frame_all uses), from the track records, the two frame-table
// entries and the point.
template <int NC>
__global__ void __launch_bounds__(256) k_pairs(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  const int cur = st->cur;
  // one CTA per pair, 1..8 warps (the launcher picks the width so that a rank with few pairs still fills the machine)
  const int pair = blockIdx.x, lane = threadIdx.x & 31, wrp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const int f1 = d.pair_f1[pair], f2 = d.pair_f2[pair];
  __shared__ double sred[8][36];
  __shared__ double fe[2][kFrameStride];
  for (int k = threadIdx.x; k < 2 * kFrameStride; k += blockDim.x)  // the CTA may be a single warp
    fe[k / kFrameStride][k % kFrameStride] = d.frames[cur][(size_t)(k < kFrameStride ? f1 : f2) * kFrameStride + k % kFrameStride];
  __syncthreads();
  const double* __restrict__ recs = d.rec[cur];
  const double* __restrict__ points = d.points[cur];
  double acc[36];
#pragma unroll
  for (int v = 0; v < 36; ++v) acc[v] = 0.0;
  for (int i = d.pair_begin[pair] + threadIdx.x; i < d.pair_begin[pair + 1]; i += blockDim.x) {
    const int t1 = d.pair_t1[i], t2 = d.pair_t2[i];
    const int p = d.trk_point[t1];
    const double* X = points + 3 * (size_t)p;
    double G[9];
    {
      double A[6], B[9], K[9];
      load_record<6, false>(recs + (size_t)t1 * rec_stride(NC), A);
      track_b(A, fe[0], B);
      {
        double Hi[6];
        load_record<6, false>(d.pdata + (size_t)p * kPointStride, Hi);  // Hpp^-1 leads the point record
        mat3_sym3(B, Hi, K);
      }
      load_record<6, false>(recs + (size_t)t2 * rec_stride(NC), A);
      track_b(A, fe[1], B);
      mat3_mat3t(K, B, G);
    }
    double m1[9], m2[9];
    track_m(fe[0], X, m1);
    track_m(fe[1], X, m2);
    mt_mat_m_acc(m1, G, m2, acc);
  }
#pragma unroll
  for (int v = 0; v < 36; ++v) {
    const double s = warp_sum(acc[v]);
    if (lane == 0) sred[wrp][v] = s;
  }
  __syncthreads();
  if (threadIdx.x < 36) {
    double s = 0.0;
    for (int w = 0; w < nw; ++w) s += sred[w][threadIdx.x];  // fixed order
    *S_at(d, 6 * f1 + threadIdx.x / 6, 6 * f2 + threadIdx.x % 6) -= s;
  }
}

// Points touched by a distance constraint stay in the reduced system (SURVEY.md H3): their blocks are added
// to S directly. A handful of points: one thread each.
template <int NC>
__global__ void k_coupled(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  const int cur = st->cur;
  constexpr int RS = rec_stride(NC);
  const int ci = blockIdx.x * blockDim.x + threadIdx.x;
  if (ci >= d.Pc) return;
  const int p = d.coupled_pts[ci];
  const int ro = d.np6 + 3 * ci;
  const double* X = d.points[cur] + 3 * (size_t)p;
  double H[6] = {0, 0, 0, 0, 0, 0}, gp[3] = {0, 0, 0}, Hcp[3 * NC];
  for (int k = 0; k < 3 * NC; ++k) Hcp[k] = 0.0;
  for (int t = d.pt_trk_begin[p]; t < d.pt_trk_begin[p + 1]; ++t) {
    const double* rc = d.rec[cur] + (size_t)t * RS;
    const int f = d.trk_frame[t];
    const double* fe = d.frames[cur] + (size_t)f * kFrameStride;
    const double* R = fe;
    const double A[6] = {rc[0], rc[1], rc[2], rc[3], rc[4], rc[5]};
    double AR[9];
    for (int j = 0; j < 3; ++j) {
      AR[0 + j] = A[0] * R[j] + A[1] * R[3 + j] + A[2] * R[6 + j];
      AR[3 + j] = A[1] * R[j] + A[3] * R[3 + j] + A[4] * R[6 + j];
      AR[6 + j] = A[2] * R[j] + A[4] * R[3 + j] + A[5] * R[6 + j];
    }
    H[0] += R[0] * AR[0] + R[3] * AR[3] + R[6] * AR[6];
    H[1] += R[0] * AR[1] + R[3] * AR[4] + R[6] * AR[7];
    H[2] += R[0] * AR[2] + R[3] * AR[5] + R[6] * AR[8];
    H[3] += R[1] * AR[1] + R[4] * AR[4] + R[7] * AR[7];
    H[4] += R[1] * AR[2] + R[4] * AR[5] + R[7] * AR[8];
    H[5] += R[2] * AR[2] + R[5] * AR[5] + R[8] * AR[8];
    for (int j = 0; j < 3; ++j) gp[j] += R[j] * rc[6] + R[3 + j] * rc[7] + R[6 + j] * rc[8];
    for (int c = 0; c < NC; ++c)
      for (int j = 0; j < 3; ++j)
        Hcp[3 * c + j] += rc[9 + c] * R[j] + rc[9 + NC + c] * R[3 + j] + rc[9 + 2 * NC + c] * R[6 + j];
    if (d.refine_poses) {  // S[point, pose f] += V^T
      double m[9];
      track_M(fe, X, m);
      for (int a = 0; a < 6; ++a)
        for (int j = 0; j < 3; ++j) {
          double v;
          if (a < 3) v = m[3 * a] * AR[j] + m[3 * a + 1] * AR[3 + j] + m[3 * a + 2] * AR[6 + j];
          else v = AR[3 * (a - 3) + j];
          *S_at(d, ro + j, 6 * f + a) += v;
        }
    }
  }
  *S_at(d, ro + 0, ro + 0) += H[0];
  *S_at(d, ro + 1, ro + 0) += H[1];
  *S_at(d, ro + 2, ro + 0) += H[2];
  *S_at(d, ro + 1, ro + 1) += H[3];
  *S_at(d, ro + 2, ro + 1) += H[4];
  *S_at(d, ro + 2, ro + 2) += H[5];
  d.hdiag[ro + 0] += H[0];
  d.hdiag[ro + 1] += H[3];
  d.hdiag[ro + 2] += H[5];
  for (int j = 0; j < 3; ++j) {
    d.g[ro + j] += gp[j];
    d.gfull[ro + j] += gp[j];
  }
  for (int c = 0; c < NC; ++c) {
    const int r = d.cam_red[c];
    if (r < 0) continue;
    for (int j = 0; j < 3; ++j) *S_at(d, r, ro + j) += Hcp[3 * c + j];
  }
}

// Distance constraints (OurConstraintFunctionBundle, no loss) between coupled points; rank 0 only, one thread.
__global__ void k_constraints(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st) || d.rank != 0) return;
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  const double* pts = d.points[st->cur];
  for (int k = 0; k < d.K; ++k) {
    const int p1 = d.c_p1[k], p2 = d.c_p2[k];
    double r, j[3];
    distance_eval(pts + 3 * p1, pts + 3 * p2, d.c_dist[k], d.c_sigma[k], r, j);
    const int o1 = d.np6 + 3 * d.pt_coupled[p1], o2 = d.np6 + 3 * d.pt_coupled[p2];
    for (int a = 0; a < 3; ++a) {
      for (int b = 0; b <= a; ++b) {
        *S_at(d, o1 + a, o1 + b) += j[a] * j[b];
        *S_at(d, o2 + a, o2 + b) += j[a] * j[b];
      }
      for (int b = 0; b < 3; ++b) {
        if (o1 > o2) *S_at(d, o1 + a, o2 + b) -= j[a] * j[b];
        else if (o2 > o1) *S_at(d, o2 + a, o1 + b) -= j[a] * j[b];
      }
      d.g[o1 + a] += j[a] * r;
      d.g[o2 + a] -= j[a] * r;
      d.gfull[o1 + a] += j[a] * r;
      d.gfull[o2 + a] -= j[a] * r;
      d.hdiag[o1 + a] += j[a] * j[a];
      d.hdiag[o2 + a] += j[a] * j[a];
    }
  }
}

// Camera block: Hcc, gc of the accepted state (from k_eval_rows) + the Schur terms of k_points; point
// gradient statistics into the system scalars.
__global__ void __launch_bounds__(1024) k_add_camera(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  const int NC = d.NC, NH = NC * (NC + 1) / 2;
  const double* cs = d.camsum[st->cur];
  __shared__ double sp[64];
  const int v = threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // 64 values per CTA of k_points, summed over the CTAs: lane = value (coalesced 256-byte rows), warps stride over the
  // CTAs, then the 32 warp partials are added in warp order (fixed order: deterministic)
  {
    __shared__ double wp[32][64];
    for (int h2 = 0; h2 < 2; ++h2) {
      const int q = lane + 32 * h2;
      double s_ = 0.0;
      if (d.refine_points) {
        if (q == 63) {
          for (int b = warp; b < d.grid_pts; b += 32) s_ = fmax(s_, d.part_pts[(size_t)b * 64 + q]);
        } else {
          for (int b = warp; b < d.grid_pts; b += 32) s_ += d.part_pts[(size_t)b * 64 + q];
        }
      }
      wp[warp][q] = s_;
    }
    __syncthreads();
    if (v < 64) {
      double s_ = 0.0;
      for (int w = 0; w < 32; ++w) s_ = v == 63 ? fmax(s_, wp[w][v]) : s_ + wp[w][v];
      sp[v] = s_;
    }
  }
  __syncthreads();
  if (v < NH) {
    int c1 = 0, h = v;
    while (h > c1) { h -= c1 + 1; ++c1; }
    const int r1 = d.cam_red[c1], r2 = d.cam_red[h];
    if (r1 >= 0 && r2 >= 0) *S_at(d, r1, r2) += cs[v] + sp[v];
    if (c1 == h && r1 >= 0) d.hdiag[r1] += cs[v];
  } else if (v < NH + NC) {
    const int r = d.cam_red[v - NH];
    if (r >= 0) {
      d.g[r] += cs[v] + sp[v];
      d.gfull[r] += cs[v];
    }
  } else if (v == NH + NC) {
    d.sys_scalars[SS_GNORM2] = sp[NH + NC];
    d.sys_scalars[SS_PTFAIL] = sp[NH + NC + 1];
    for (int r = 0; r < d.nranks; ++r) d.sys_scalars[SS_COUNT + r] = (r == d.rank) ? sp[63] : 0.0;
  }
}

// ================================================================================================
// C2. finalize the iteration row, termination tests, Jacobi scaling and LM damping of the reduced system
// (EvaluateGradientAndJacobian's scaling + gradient norms, FinalizeIterationAndCheckIfMinimizerCanContinue,
//  LevenbergMarquardtStrategy::ComputeStep's diagonal). One CTA.
// ================================================================================================
__global__ void __launch_bounds__(1024) k_finalize(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  if (d.undamped) {
    // covariance: S stays the Gauss-Newton matrix (the min_lm_diagonal clamp would damp even an infinite radius); the
    // pose rows and columns of the gauge frame and of frames without observations become identity
    if (threadIdx.x == 0) st->solve_ok = d.sys_scalars[SS_PTFAIL] > 0.0 ? 0 : 1;
    auto fixed = [&](int r) { return r < d.np6 && (r / 6 == d.gauge_frame || !d.frm_active[r / 6]); };
    const int lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int r = threadIdx.x >> 5; r < d.n; r += nw) {
      const bool fr = fixed(r);
      for (int c = d.row_c0[r] + lane; c <= r; c += 32)
        if (fr || fixed(c)) *S_at(d, r, c) = r == c ? 1.0 : 0.0;
    }
    return;
  }
  const Options& o = d.opt;
  __shared__ double sg2[32], sgm[32];
  const bool first = st->first != 0;
  const bool refresh = st->pending_row && st->row.step_is_successful;
  double g2 = 0.0, gm = 0.0;
  for (int j = threadIdx.x; j < d.n; j += blockDim.x) {
    if (first) d.rscale[j] = 1.0 / (1.0 + sqrt(d.hdiag[j]));
    if (refresh) {
      // |x - Plus(x, -g)|: identical to |g| except where a box bound of the camera block clips it
      double gj = d.gfull[j];
      if (d.recalib) {
        for (int c = 0; c < d.NC; ++c)
          if (d.cam_red[c] == j) {
            const double x = d.camera[st->cur][c];
            const double xn = fmin(fmax(x - gj, d.cam_lo[c]), d.cam_hi[c]);
            gj = x - xn;
          }
      }
      g2 += gj * gj;
      gm = fmax(gm, fabs(gj));
    }
  }
  g2 = warp_sum(g2);
  gm = warp_max(gm);
  if ((threadIdx.x & 31) == 0) {
    sg2[threadIdx.x >> 5] = g2;
    sgm[threadIdx.x >> 5] = gm;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (st->pending_row) {
      lfba_iteration& row = st->row;
      if (refresh) {
        double t2 = d.sys_scalars[SS_GNORM2], tm = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) {
          t2 += sg2[w];
          tm = fmax(tm, sgm[w]);
        }
        for (int r = 0; r < d.nranks; ++r) tm = fmax(tm, d.sys_scalars[SS_COUNT + r]);
        st->gnorm = sqrt(t2);
        st->gmax = tm;
      }
      row.gradient_norm = st->gnorm;
      row.gradient_max_norm = st->gmax;
      if (row.step_is_successful) {
        st->n_success++;
        if (st->x_cost < st->min_cost) st->min_cost = st->x_cost;
      } else {
        st->n_fail++;
      }
      row.trust_region_radius = st->radius;
      const unsigned long long now = gtimer();
      row.iteration_time_s = 1e-9 * (double)(now - st->t_iter);
      row.cumulative_time_s = 1e-9 * (double)(now - st->t_start);
      st->t_iter = now;
      if (st->n_rows < kMaxLog) d.log[st->n_rows] = row;
      st->n_rows++;
      st->pending_row = 0;
      if (row.iteration >= o.max_iter) {
        st->done = 1;
        st->termination = LFBA_NO_CONVERGENCE;
        st->stop_reason = LFBA_STOP_MAX_ITERATIONS;
      } else if (row.step_is_successful && row.gradient_max_norm <= o.gtol) {
        st->done = 1;
        st->termination = LFBA_CONVERGENCE;
        st->stop_reason = LFBA_STOP_GRADIENT_TOLERANCE;
      } else if (row.trust_region_radius <= o.rmin) {
        st->done = 1;
        st->termination = LFBA_CONVERGENCE;
        st->stop_reason = LFBA_STOP_MIN_RADIUS;
      }
      st->iter = row.iteration + 1;
    }
    st->first = 0;
    st->eval_skip = 0;
    // a point block that is not positive definite makes the linear solve fail (LINEAR_SOLVER_FAILURE)
    st->solve_ok = d.sys_scalars[SS_PTFAIL] > 0.0 ? 0 : 1;
  }
  __syncthreads();
  if (st->done) return;
  const double mu = st->radius;
  for (int j = threadIdx.x; j < d.n; j += blockDim.x) {
    const double s2 = d.rscale[j] * d.rscale[j];
    const double dm = fmin(fmax(s2 * d.hdiag[j], o.min_diag), o.max_diag) / (mu * s2);
    d.rdamp[j] = dm;
    *S_at(d, j, j) += dm;
    // augmented row: the reduced right-hand side, forward-substituted for free by the factorisation
    *S_at(d, d.n, j) = d.g[j];
  }
}

// ================================================================================================
// P. steps and candidate
// ================================================================================================
// Per point back substitution y_p = Hpp^-1 (g_p - sum_t V_t^T y_f) - T_p y_c (T_p = Hpp^-1 Hcp^T from k_points),
// candidate X+ = X - y_p, and the point's share of: model cost change 1/2 y.(g + D y), |step|^2, |x+|^2, g.delta.
template <int NC>
__global__ void __launch_bounds__(128) k_point_step(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st) || !st->solve_ok) return;
  const int cur = st->cur, cand = 1 - cur;
  __shared__ double red[4 * 8];
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  double dmax = 0.0;
  const double* __restrict__ y = d.y;
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < d.P; p += gridDim.x * blockDim.x) {
    if (!d.pt_active[p] || d.pt_coupled[p] >= 0) continue;
    double pd[kPointStride];
    load_record<kPointStride, true>(d.pdata + (size_t)p * kPointStride, pd);  // 320-byte records, 32-byte aligned
    double tc[3] = {0, 0, 0};  // T_p y_c
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const int r = d.cam_red[c];
      const double yc = r >= 0 ? y[r] : 0.0;
      tc[0] += pd[12 + 3 * c] * yc;
      tc[1] += pd[13 + 3 * c] * yc;
      tc[2] += pd[14 + 3 * c] * yc;
    }
    double h[3] = {0, 0, 0};
    if (d.refine_poses) {  // sum_t V_t^T y_f, from the track's A block, its frame entry and X
      const double* __restrict__ frames = d.frames[cur];
      const double* X = d.points[cur] + 3 * (size_t)p;
      const double Xp[3] = {X[0], X[1], X[2]};
      for (int t = d.pt_trk_begin[p]; t < d.pt_trk_begin[p + 1]; ++t) {
        const int f = d.trk_frame[t];
        const double* fe = frames + (size_t)f * kFrameStride;
        double m[9], A[6];
        load_record<6, false>(d.rec[cur] + (size_t)t * rec_stride(NC), A);
        track_m(fe, Xp, m);
        track_vt_y_acc(A, fe, m, y + 6 * f, h);
      }
    }
    const double gp[3] = {pd[6], pd[7], pd[8]};
    const double rhs[3] = {gp[0] - h[0], gp[1] - h[1], gp[2] - h[2]};
    double yp[3];
    sym3_vec(pd, rhs, yp);
#pragma unroll
    for (int j = 0; j < 3; ++j) yp[j] -= tc[j];
    const double* X = d.points[cur] + 3 * (size_t)p;
    double* Xc = d.points[cand] + 3 * (size_t)p;
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      const double xn = X[j] - yp[j];
      Xc[j] = xn;
      const double dl = xn - X[j];
      acc[0] += 0.5 * yp[j] * (gp[j] + pd[9 + j] * yp[j]);
      acc[1] += dl * dl;
      acc[2] += xn * xn;
      acc[3] += gp[j] * dl;
      if (!isfinite(yp[j])) acc[4] += 1.0;
      if (d.recalib) {  // the projected line search re-applies delta at other step sizes
        d.pstep[3 * (size_t)p + j] = -yp[j];
        dmax = fmax(dmax, fabs(yp[j]));
      }
    }
  }
  block_reduce_store<8>(acc, d.part_step + (size_t)blockIdx.x * 8, red);
  if (d.recalib) {  // slot 5: max |delta| (a maximum, not a sum)
    dmax = warp_max(dmax);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dmax;
    __syncthreads();
    if (threadIdx.x == 0) d.part_step[(size_t)blockIdx.x * 8 + 5] = fmax(fmax(red[0], red[1]), fmax(red[2], red[3]));
  }
}

// Back substitution output y (reduced) -> candidate camera (SubsetManifold + box bounds), poses, coupled points;
// reduced-part scalars. One CTA.
__global__ void __launch_bounds__(1024) k_reduced_step(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st)) return;
  const int cur = st->cur, cand = 1 - cur;
  __shared__ double red[32 * 8];
  __shared__ double out[8];
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (st->solve_ok) {
    const double* y = d.y;
    // poses
    for (int j = threadIdx.x; j < d.np6; j += blockDim.x) {
      const double x = d.views[cur][j];
      const double xn = x - y[j];
      d.views[cand][j] = xn;
      if (d.frm_active[j / 6]) {
        const double dl = xn - x;
        acc[0] += 0.5 * y[j] * (d.gfull[j] + d.rdamp[j] * y[j]);
        acc[1] += dl * dl;
        acc[2] += xn * xn;
        acc[3] += d.gfull[j] * (-y[j]);
      }
      if (!isfinite(y[j])) acc[4] += 1.0;
    }
    if (!d.refine_poses)
      for (int j = threadIdx.x; j < 6 * d.F; j += blockDim.x) d.views[cand][j] = d.views[cur][j];
    // coupled points
    for (int j = threadIdx.x; j < 3 * d.Pc; j += blockDim.x) {
      const int r = d.np6 + j;
      const int p = d.coupled_pts[j / 3];
      const double x = d.points[cur][3 * (size_t)p + j % 3];
      const double xn = x - y[r];
      d.points[cand][3 * (size_t)p + j % 3] = xn;
      const double dl = xn - x;
      acc[0] += 0.5 * y[r] * (d.gfull[r] + d.rdamp[r] * y[r]);
      acc[1] += dl * dl;
      acc[2] += xn * xn;
      acc[3] += d.gfull[r] * (-y[r]);
      if (!isfinite(y[r])) acc[4] += 1.0;
    }
    // camera block: all 17 entries count in |x|; held-constant and inactive entries do not move
    for (int c = threadIdx.x; c < 17; c += blockDim.x) {
      const double x = d.camera[cur][c];
      double xn = x;
      const int r = c < d.NC ? d.cam_red[c] : -1;
      if (r >= 0) {
        xn = x - y[r];
        acc[0] += 0.5 * y[r] * (d.gfull[r] + d.rdamp[r] * y[r]);
        acc[3] += d.gfull[r] * (-y[r]);
        if (!isfinite(y[r])) acc[4] += 1.0;
      }
      xn = fmin(fmax(xn, d.cam_lo[c]), d.cam_hi[c]);
      d.camera[cand][c] = xn;
      const double dl = xn - x;
      acc[1] += dl * dl;
      acc[2] += xn * xn;
    }
  }
  block_reduce_store<8>(acc, out, red);
  if (d.recalib) {  // max |delta| over the reduced parameters (line-search step-size floor)
    double m = 0.0;
    if (st->solve_ok)
      for (int j = threadIdx.x; j < d.n; j += blockDim.x) m = fmax(m, fabs(d.y[j]));
    m = warp_max(m);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
      double mm = 0.0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) mm = fmax(mm, red[w]);
      st->dmax_red = mm;
    }
  }
  if (threadIdx.x == 0) {
    st->mcc_red = out[0];
    st->step2_red = out[1];
    st->norm2_red = out[2];
    st->gdelta_red = out[3];
    if (out[4] > 0.0) st->solve_ok = 0;
    st->eval_skip = st->solve_ok ? 0 : 1;
  }
}

// Start of a solve: candidate := initial parameters, |x0|^2 partials (k_reduce_eval reads them in round 0).
__global__ void __launch_bounds__(128) k_init_norms(Dev d) {
  __shared__ double red[4 * 8];
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const int cand = 1 - d.st->cur;
  if (d.refine_points)
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < d.P; p += gridDim.x * blockDim.x) {
      if (!d.pt_active[p] || d.pt_coupled[p] >= 0) continue;
      const double* X = d.points[cand] + 3 * (size_t)p;
      acc[2] += X[0] * X[0] + X[1] * X[1] + X[2] * X[2];
    }
  block_reduce_store<8>(acc, d.part_step + (size_t)blockIdx.x * 8, red);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double s = 0.0;
    if (d.recalib)  // IterationZero of a bounds-constrained problem projects the start point into the box
      for (int c = 0; c < 17; ++c) d.camera[cand][c] = fmin(fmax(d.camera[cand][c], d.cam_lo[c]), d.cam_hi[c]);
    for (int c = 0; c < 17; ++c) s += d.camera[cand][c] * d.camera[cand][c];
    if (d.refine_poses)
      for (int f = 0; f < d.F; ++f)
        if (d.frm_active[f])
          for (int j = 0; j < 6; ++j) s += d.views[cand][6 * f + j] * d.views[cand][6 * f + j];
    for (int c = 0; c < d.Pc; ++c) {
      const double* X = d.points[cand] + 3 * (size_t)d.coupled_pts[c];
      s += X[0] * X[0] + X[1] * X[1] + X[2] * X[2];
    }
    d.st->norm2_red = s;
    d.st->mcc_red = d.st->step2_red = d.st->gdelta_red = d.st->dmax_red = 0.0;
  }
}

// ================================================================================================
// launchers
// ================================================================================================
void prepare_eval_kernels() {
  prepare_rows_kernels();
  prepare_eval_only_kernels();
}
void launch_tables(const Dev& d, cudaStream_t s) {
  const int n = d.NL > d.F ? d.NL : d.F;
  k_tables<<<(n + 127) / 128, 128, 0, s>>>(d);
}
int launch_eval(const Dev& d, int L, cudaStream_t s) {
  launch_eval_rows(d, L, s);
  return 1;
}
void launch_reduce_eval(const Dev& d, cudaStream_t s) { k_reduce_eval<<<1, 1024, 0, s>>>(d); }
int launch_ls_gdot(const Dev& d, cudaStream_t s) {  // recalib: phi'(a) of the projected line search, before k_reduce_eval
  if (!d.recalib) return 0;
  k_ls_gdot<<<d.grid_pts, 128, 0, s>>>(d);
  return 1;
}
int launch_ls_apply(const Dev& d, cudaStream_t s) {  // recalib: moves the candidate when a contraction trial is pending
  if (!d.recalib) return 0;
  k_ls_apply<<<d.grid_pts, 128, 0, s>>>(d);
  k_ls_apply_reduced<<<1, 256, 0, s>>>(d);
  return 2;
}
void launch_control_accept(const Dev& d, cudaStream_t s) { k_control_accept<<<1, 1, 0, s>>>(d); }
int launch_assembly(const Dev& d, int frame_splits, cudaStream_t s) {
  int launches = 0;
  if (d.refine_points) {
    LFBA_DISPATCH_NC(d.NC, (k_points<NC><<<d.grid_pts, 128, 0, s>>>(d)));
    ++launches;
  }
  if (d.refine_poses) {
    dim3 grid(frame_splits, std::min(d.F, 65535));
    LFBA_DISPATCH_NC(d.NC, (k_frame_all<NC><<<grid, 128, 0, s>>>(d)));
    launches += 1;
    if (frame_splits > 1) {
      LFBA_DISPATCH_NC(d.NC, (k_frame_finish<NC><<<d.F, 128, 0, s>>>(d, frame_splits)));
      launches += 1;
    }
    if (d.refine_points && d.npairs > 0) {
      int wpp = 1;  // warps per pair: enough CTAs x warps to cover the SMs a few times
      while (wpp < 8 && (long long)d.npairs * wpp < 4096) wpp *= 2;
      LFBA_DISPATCH_NC(d.NC, (k_pairs<NC><<<d.npairs, 32 * wpp, 0, s>>>(d)));
      ++launches;
    }
  }
  if (d.Pc > 0) {
    LFBA_DISPATCH_NC(d.NC, (k_coupled<NC><<<(d.Pc + 31) / 32, 32, 0, s>>>(d)));
    ++launches;
  }
  if (d.K > 0) {
    k_constraints<<<1, 32, 0, s>>>(d);
    ++launches;
  }
  k_add_camera<<<1, 1024, 0, s>>>(d);
  return launches + 1;
}
void launch_finalize(const Dev& d, cudaStream_t s) { k_finalize<<<1, 1024, 0, s>>>(d); }
int launch_steps(const Dev& d, cudaStream_t s) {
  int launches = 1;
  if (d.refine_points) {
    LFBA_DISPATCH_NC(d.NC, (k_point_step<NC><<<d.grid_pts, 128, 0, s>>>(d)));
    ++launches;
  }
  k_reduced_step<<<1, 1024, 0, s>>>(d);
  return launches;
}
void launch_init_norms(const Dev& d, cudaStream_t s) { k_init_norms<<<d.grid_pts, 128, 0, s>>>(d); }

}  // namespace lfba
