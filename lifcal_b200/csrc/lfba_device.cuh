// lfba_device.cuh — device-side data layout of one rank's share of an LF-BA problem, and the LM state that
// lives in HBM for the whole solve (the host only polls `done`).
//
// Layout in HBM (per rank; N observations, T tracks = (point, frame) pairs, P points, F frames, NL lenses):
//   obs      double2[N]   observed micro-image point, sorted by (point, frame)          16 B/obs  \  the streamed
//   lens_id  int32[N]     index into the lens table                                      4 B/obs  /  20 B/obs
//   lens     double[NL*16] per-lens undistortion table (rebuilt per evaluation, L2-resident)
//   frames   double[2][F*40] per-frame rotation table for the accepted / candidate poses
//   trk_*    int32[T]     point, frame, first observation of each track (+ begin[T])
//   rec      double[2][T*REC] per-track normal-equation blocks in the camera frame (A 6, b 3, C 3xNC),
//                          double-buffered: accepted state / candidate
//   pdata    double[P*40] per-point Schur data (inverse of the damped 3x3, gradient, damping, inverse x camera coupling)
//   S        skyline lower-triangular reduced system [poses 6F | coupled points 3Pc | camera | rhs row]
// Parameters are double-buffered (accepted x / candidate x+) so that accept/reject is an index flip on device.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/lfba.h"
#include "lfba_math.cuh"

namespace lfba {

#if defined(__CUDACC__)
// 256-bit global accesses (sm_100: LDG.E.256 / STG.E.256). A lane that reads or writes ITS OWN record (track record,
// point data) touches one 32-byte sector per instruction instead of half or a quarter of it: fewer L1 wavefronts on the
// read side, no partially filled sectors towards L2 on the write side. The address must be 32-byte aligned.
__device__ __forceinline__ void ldg256(const double* p, double* out) {
  asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(out[0]), "=d"(out[1]), "=d"(out[2]), "=d"(out[3]) : "l"(p));
}
__device__ __forceinline__ void stg256(double* p, double a, double b, double c, double d) {
  asm volatile("st.global.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(p), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}
// N doubles of a record at p: 256-bit loads when the caller guarantees 32-byte alignment of p and N % 4 == 0 (ALIGN32),
// else 128-bit (N even, 16-byte aligned), else scalar
template <int N, bool ALIGN32>
__device__ __forceinline__ void load_record(const double* __restrict__ p, double* out) {
  if (ALIGN32 && N % 4 == 0) {
#pragma unroll
    for (int k = 0; k < N / 4; ++k) ldg256(p + 4 * k, out + 4 * k);
  } else if (N % 2 == 0) {
#pragma unroll
    for (int k = 0; k < N / 2; ++k) {
      const double2 v2 = __ldg(reinterpret_cast<const double2*>(p) + k);
      out[2 * k] = v2.x;
      out[2 * k + 1] = v2.y;
    }
  } else {
#pragma unroll
    for (int k = 0; k < N; ++k) out[k] = __ldg(p + k);
  }
}
#endif

constexpr int kPointStride = 40;  // pdata: Hinv(6) gp(3) dmp(3) T_p = Hinv Hcp^T (3*NC<=27, [3 c + j]) pad
constexpr int kMaxLog = 1024;
constexpr int kTile = 64;         // Cholesky tile

// doubles per track record: A (6) b (3) C (3 NC), padded to a multiple of 4 so that a record is a whole number of 32-byte
// sectors for every model variant (NC = 8: 33 -> 36) and the 256-bit per-lane loads / stores always apply
__host__ __device__ constexpr int rec_stride(int nc) { return (9 + 3 * nc + 3) & ~3; }

// Skyline offsets in closed form (no dependent index loads on the latency chain). The solver lays the reduced system out
// as: pose row r = 6 f + i starts at column 6 max(0, f - bw); border rows (coupled points, camera, rhs) start at column 0.
// So frame f's six rows hold 36 min(f, bw) + 21 entries, and everything before frame f is a polynomial in f.
struct SkyMap {
  int bw, np6;
  __host__ __device__ long long frame_off(int f) const {
    return f <= bw ? 18ll * f * (f - 1) + 21ll * f
                   : 18ll * bw * (bw - 1) + 21ll * bw + (long long)(f - bw) * (36 * bw + 21);
  }
  __host__ __device__ int c0(int f) const { return 6 * (f > bw ? f - bw : 0); }
  __host__ __device__ long long row(int f, int i) const {  // offset of entry (6 f + i, c0(f))
    const int len0 = 6 * f - c0(f) + 1;
    return frame_off(f) + (long long)i * len0 + (i * (i - 1)) / 2;
  }
  __host__ __device__ long long border_row(int b) const {  // offset of entry (np6 + b, 0)
    return frame_off(np6 / 6) + (long long)b * (np6 + 1) + ((long long)b * (b - 1)) / 2;
  }
};

// scalars exchanged between kernels / ranks through small device arrays
enum EvalScalar {  // tiny buffer reduced (sum) across ranks after the candidate evaluation
  ES_COST = 0,     // candidate cost (observations of this rank + constraints on rank 0)
  ES_MCC,          // model cost change partial (points of this rank; reduced part added on rank 0)
  ES_STEP2,        // |x - x+|^2 partial
  ES_NORM2,        // |x+|^2 partial
  ES_GDELTA,       // gradient . delta partial
  ES_BAD,          // non-finite step flag (count)
  ES_LSGD,         // recalib: gradient(candidate) . delta partial = phi'(alpha) of the projected line search
  ES_COUNT = 8     // followed by nranks slots: max |delta| over the parameters of each rank (line-search step-size floor)
};
enum SysScalar {   // trailer of the big buffer reduced (sum) across ranks with S and g
  SS_GNORM2 = 0,   // sum of squared gradient over the points of this rank
  SS_PTFAIL,       // number of points whose damped 3x3 block was not positive definite
  SS_COUNT = 4     // followed by nranks slots for max |g| over points (one slot per rank)
};

struct LmState {
  int iter;         // index of the iteration row being produced (0 = IterationZero)
  int cur;          // buffer index of the accepted state
  int done;
  int eval_skip;    // candidate evaluation skipped: the step was known to be invalid
  int solve_ok;     // Cholesky succeeded and the step is finite
  int num_invalid;  // consecutive invalid steps
  int termination, stop_reason, status;
  int n_success, n_fail, n_rows;
  int first;        // Jacobi scaling still to be computed (iteration 0)
  int pending_row;  // a row is waiting for its gradient norms (k_finalize)
  int n_jac_evals;
  // projected Armijo line search of bounds-constrained problems (recalib; Ceres TrustRegionMinimizer::DoLineSearch)
  int ls_active;    // a search is in progress: the candidate just evaluated was the trial at step size ls_alpha
  int ls_trial;     // a contraction trial is pending: this round skips assembly / solve / step, k_ls_apply moves the candidate
  int ls_iters;     // contractions so far (the row's line_search_iterations)
  int ls_failed;    // the search gave up: the full step is re-evaluated and taken without the Armijo test
  int ls_prev_valid, ls_prev_gvalid;
  double ls_alpha, ls_phi0, ls_dphi0;
  double ls_prev_x, ls_prev_v, ls_prev_g;
  double dmax_red;  // max |delta| over the reduced parameters (camera, poses, coupled points)
  double radius, decrease_factor;
  double x_cost, x_norm2, min_cost;
  double gmax, gnorm;
  double mcc_red, step2_red, norm2_red, gdelta_red;  // reduced-part contributions to the candidate scalars
  lfba_iteration row;
  unsigned long long t_start, t_iter;
};

// post-control kernels (assembly, reduced solve, step) do nothing in a round whose only job is a line-search trial
__host__ __device__ inline bool linear_phase_idle(const LmState* st) { return st->done || st->ls_trial; }

struct Options {
  int max_iter;
  double ftol, ptol, gtol, r0, rmax, rmin, min_rel_dec, min_diag, max_diag;
  int max_invalid;
  double loss_a;
};

// Everything a kernel needs, passed by value.
struct Dev {
  // sizes
  int64_t N;
  int T, P, F, NL, K;       // tracks, points, frames, lenses, constraints
  int NC;                   // live camera parameters
  int n;                    // reduced system size (without the rhs row)
  int np6;                  // 6F if poses are refined else 0
  int band;                 // co-visibility bandwidth in frames: pose row 6f+i of S starts at column 6 max(0, f - band)
  int Pc;                   // coupled points
  int n_cam_red;            // free camera parameters in the reduced system
  int rank, nranks;
  uint32_t config;
  int recalib, refine_poses, refine_points;
  int debug;                // LFBA_DEBUG set: the control kernel prints its line-search decisions
  int undamped;             // covariance: assemble J^T W J itself (no LM damping; k_finalize keeps no iteration row)
  int gauge_frame;          // covariance: frame whose pose is held fixed (identity rows in S), -1 = none
  double spx, spy, scale;
  Options opt;
  // observations (sorted by point, frame)
  const double2* obs;
  const int32_t* lens_id;
  const int32_t* trk_point;
  const int32_t* trk_frame;
  const int32_t* trk_begin;   // [T+1]
  const int32_t* pt_trk_begin;  // [P+1]
  const int32_t* frm_begin;   // [F+1] into frm_trk
  const int32_t* frm_trk;     // track ids grouped by frame
  const int32_t* pair_begin;  // [npairs+1] into pair_t1/pair_t2
  const int32_t* pair_f1;     // [npairs]
  const int32_t* pair_f2;
  const int32_t* pair_t1;
  const int32_t* pair_t2;
  int npairs;
  const int32_t* eval_order;  // track processing order of the evaluation kernel (length-sorted)
  int round_cost;             // fixed part of a round's cost in rows (split of the rounds over the warps)
  const int2* eval_pf;        // [T] (point, frame) of track eval_order[pos]: one coalesced load per round and lane
  // packed evaluation stream (lfba_setup.cuh, build_stream): rows of 32 entries in the order k_eval_rows consumes them
  const double2* s_obs;       // [n_rows * 32]
  const int32_t* s_lid;       // [n_rows * 32], -1 = padding
  const int32_t* step_base;   // [n_rounds + 1]
  int n_rounds, n_rows, stream_L;
  // point / frame flags
  const int32_t* pt_coupled;  // [P] index among coupled points or -1
  const int32_t* coupled_pts; // [Pc]
  const int32_t* pt_active;   // [P] 1 if the point is in the problem on this rank
  const int32_t* frm_active;  // [F] 1 if the frame has observations on any rank
  const int32_t* c_p1;
  const int32_t* c_p2;
  const double* c_dist;
  const double* c_sigma;
  int cam_red[kMaxNC];        // camera column -> reduced index (absolute) or -1 when held constant
  double cam_lo[17], cam_hi[17];  // box bounds on the camera block (recalib), +-DBL_MAX otherwise
  // parameters, double-buffered
  double* camera[2];   // [17]
  double* views[2];    // [6F]
  double* points[2];   // [3P]
  // tables
  double* lens;        // [NL*16]
  CamModel* cm_buf;    // camera model of the candidate parameters, written by k_tables (copied into constant memory)
  const double* lens_xy;  // [NL*2] lens centres
  double* frames[2];   // [F*40]
  // per-track / per-point work arrays
  double* rec[2];
  double* camsum[2];   // [64]: Hcc (lower, NC*(NC+1)/2), gc (NC), cost
  double* pdata;
  double* pscale;      // [3P] Jacobi scale of the point columns
  double* frame_part;  // [F * frame_splits * (39 + 6 NC)] partial sums of k_frame_all when frames are split over CTAs
  // reduced system
  double* S;           // skyline storage
  const int64_t* row_off;  // [n+2]
  const int32_t* row_c0;   // [n+1] first stored column of each row
  double* g;           // [n]   reduced rhs  (lives right after S in the reduce buffer)
  double* gfull;       // [n]   gradient J^T r of the reduced parameters (before the Schur correction)
  double* hdiag;       // [n]   diagonal of F^T F (undamped, before Schur)
  double* sys_scalars; // [SS_COUNT + nranks]
  double* rscale;      // [n] Jacobi scale of the reduced columns
  double* rdamp;       // [n] LM damping added to the reduced diagonal
  double* y;           // [n] reduced solution
  double* eval_scalars;  // [ES_COUNT]
  // partial sums of the block reductions
  double* part_eval;   // [grid_eval * 64]
  double* part_pts;    // [grid_pts * 64]
  double* part_step;   // [grid_pts * 8]
  double* pstep;       // [3P] recalib: delta of the eliminated points (the line search re-applies it at step size alpha)
  double* part_ls;     // [grid_pts] recalib: per-CTA partial sums of gradient(candidate) . delta
  int grid_eval, grid_pts;
  LmState* st;
  lfba_iteration* log;
};

}  // namespace lfba
