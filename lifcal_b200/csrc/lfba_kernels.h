// lfba_kernels.h — launchers of the LF-BA kernels (lfba_kernels.cu, lfba_chol.cu, lfba_setup.cu).
#pragma once
#include <cuda_runtime.h>

#include "lfba_device.cuh"

namespace lfba {

// CALL with `NC` a compile-time constant equal to the live camera parameter count NCV (5 .. 9)
#define LFBA_DISPATCH_NC(NCV, CALL)   \
  switch (NCV) {                      \
    case 5: { constexpr int NC = 5; CALL; } break; \
    case 6: { constexpr int NC = 6; CALL; } break; \
    case 7: { constexpr int NC = 7; CALL; } break; \
    case 8: { constexpr int NC = 8; CALL; } break; \
    default: { constexpr int NC = 9; CALL; } break; \
  }

// ---- lfba_kernels.cu: one LM round ----
void launch_init_norms(const Dev& d, cudaStream_t s);
void launch_tables(const Dev& d, cudaStream_t s);
int launch_eval(const Dev& d, int lanes_per_track, cudaStream_t s);  // returns the number of kernels launched
void launch_reduce_eval(const Dev& d, cudaStream_t s);
int launch_ls_gdot(const Dev& d, cudaStream_t s);   // recalib only (else no launch); returns kernels launched
int launch_ls_apply(const Dev& d, cudaStream_t s);  // recalib only
void launch_control_accept(const Dev& d, cudaStream_t s);
int launch_assembly(const Dev& d, int frame_splits, cudaStream_t s);  // returns the number of kernels launched
void launch_finalize(const Dev& d, cudaStream_t s);
int launch_steps(const Dev& d, cudaStream_t s);

// ---- lfba_chol.cu: reduced system ----
// In-place tiled Cholesky of the skyline matrix (n + 1 rows: the last row is the rhs, which comes out
// forward-substituted), then the backward substitution into d.y. Returns the number of kernels launched.
void prepare_device_kernels();
void prepare_eval_kernels();
// lfba_rows.cu: fused evaluation over the packed stream, cooperative cp.async lens gather
void prepare_rows_kernels();
void launch_eval_rows(const Dev& d, int lanes_per_track, cudaStream_t s);
// lfba_chol_part.cu: partitioned factorisation of the banded-arrowhead system (P CTAs instead of one chain of F pivots)
struct PartPlan;
PartPlan* part_plan_create(const Dev& d, int bandwidth_frames, cudaStream_t s);  // never null; may be inactive
void part_plan_destroy(PartPlan* p);
bool part_plan_active(const PartPlan* p);
int launch_part_solve(const Dev& d, PartPlan* p, cudaStream_t s);
int launch_reduced_solve(const Dev& d, int n_tiles, const int* d_tile_first /*[n_tiles] first nonzero tile col*/,
                         int bandwidth_frames, cudaStream_t s, PartPlan* plan);
// The in-place factorisations only (banded one-CTA kernel when it fits, else the tiled one): L is left in d.S, in the
// skyline layout, unpermuted. Returns the number of kernels launched.
int launch_chol_inplace(const Dev& d, int n_tiles, const int* d_tile_first, int bandwidth_frames, cudaStream_t s);

// ---- lfba_cov.cu: covariance from the factorised reduced system ----
void prepare_cov_kernels();
// Selected inversion of L L^T (L in d.S) over the skyline envelope into Z (same layout, S_len doubles), then the
// 17 x 17 camera block and the F x 6 x 6 pose blocks into out[289 + 36 F]. Returns the number of kernels launched.
int launch_covariance(const Dev& d, double* Z, double* out, cudaStream_t s);
// After launch_covariance on the same stream: the 3 x 3 block of every point into out[9 P] (row-major, exactly
// symmetric; zero for inactive points and when points are not refined). Returns the number of kernels launched.
int launch_cov_points(const Dev& d, const double* Z, double* out, cudaStream_t s);

// ---- lfba_eval.cu: eval-only kernel (residuals + Jacobians materialised in Ceres' block layout) ----
struct EvalOut {
  double* residuals;   // [2N]
  double* jac_camera;  // [2N*17] or null
  double* jac_view;    // [2N*6] or null
  double* jac_point;   // [2N*3] or null
  double* stats;       // [8]: sum ex^2, sum ey^2, max|ex|, max|ey|, inliers, cost
  double inlier_thr2;
  int compact_camera;  // 0: jac_camera is 2 x 17 per observation (Ceres' block, zero columns written); 1: 2 x NC (live columns)
};
struct EvalIn {
  const double2* obs;      // input order
  const int32_t* lens_id;  // input order
  const int32_t* point_idx;
  const int32_t* frame_idx;
};
void launch_eval_only(const Dev& d, const EvalIn& in, const EvalOut& out, int which, cudaStream_t s);
void prepare_eval_only_kernels();  // per device
void launch_tables_for(const Dev& d, int which, cudaStream_t s);  // tables at parameter buffer `which`

// ---- FP64 peak micro-benchmark ----
double measure_fp64_tflops(cudaStream_t s);

}  // namespace lfba
