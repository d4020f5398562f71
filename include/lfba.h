/*
 * lfba.h — C ABI of the B200-native light-field bundle adjustment (LF-BA) hot path.
 *
 * This library replaces the body of LiFCal's
 *     bool CameraCalibration::performBundleAdjustment()
 *         (reference: src/CameraCalibration.cpp:774-992, declared src/CameraCalibration.h:43)
 * i.e. the Ceres problem construction (:858-953), the solver options (:955-962) and
 * ceres::Solve (:965), together with the cost functors it evaluates
 *     OurCostFunctionBundle / OurConstraintFunctionBundle (src/BundleAdjustment/BundleAdjustment.h:25-279)
 *     CameraModel::projectPoint / radialDistortion / tangentialDistortion (src/CameraModel.h:87-241)
 *     RigidBody::getTransformationMatrix (src/CameraModel.h:246-264).
 * The reference has no FFI of its own; the seam a maintainer binds is this header (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C, no torch / CUDA types in any signature; every buffer is caller-owned HOST memory
 *     unless a function says otherwise; nothing is retained after a call returns
 *     (lfba_solver objects keep device copies only).
 *   - all floating point is IEEE double (the reference solves in double).
 *   - the CUDA kernels are the only compute path: there is no CPU fallback. Without a usable
 *     sm_100 device every compute entry point returns LFBA_NO_DEVICE.
 */
#ifndef LFBA_H_
#define LFBA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LFBA_VERSION 100 /* 0.1.0 */

/* Width of the Ceres camera parameter block — MAX_NUMBER_OF_CAMERA_PARAMETERS,
 * src/CalibrationData/CalibrationData.h:19.  Layout (src/CameraCalibration.cpp:832-853):
 * [fL, bL0, B, cx, cy, radial k0..k(nRad-1), tangential t0, t1, 0 ...]. */
#define LFBA_MAX_CAMERA_PARAMETERS 17

/* `config` bit mask, exactly as built at src/CameraCalibration.cpp:778-814 and decoded at
 * src/BundleAdjustment/BundleAdjustment.h:35-79. */
#define LFBA_CFG_NRADIAL_MASK 0x000003u  /* number of radial distortion parameters, 0..2 */
#define LFBA_CFG_TANGENTIAL 0x000004u    /* tangential distortion (2 parameters) */
#define LFBA_CFG_REFINE_POSES 0x000100u  /* Model.refineExtrinsicOrientations */
#define LFBA_CFG_ROBUST 0x000200u        /* Model.robustCostFunction -> CauchyLoss(0.5) */
#define LFBA_CFG_REFINE_POINTS 0x000400u /* Model.refineCoordinatesPoints */
#define LFBA_CFG_MLADJ 0x000800u         /* Model.adjustMicroLensCenters */

/* calibData->calib_type, src/CalibrationData/CalibrationData.h:52-56. */
#define LFBA_CALIBRATION_ARUCO 0
#define LFBA_RECALIBRATION 1 /* camera[0], camera[2] constant; +-30% bounds on camera[1,3,4] (:927-953) */

typedef enum lfba_status {
  LFBA_OK = 0,
  LFBA_INVALID_ARGUMENT = 1, /* includes refinePoses=0 && refinePoints=1, which null-derefs in the reference */
  LFBA_NO_DEVICE = 2,        /* CUDA path unavailable: there is no fallback */
  LFBA_CUDA_ERROR = 3,
  LFBA_NCCL_ERROR = 4,
  LFBA_OUT_OF_MEMORY = 5,
  LFBA_FAILURE = 6 /* solver failed (too many consecutive invalid steps) */
} lfba_status;

/* Mirrors ceres::TerminationType as far as this path can produce it. */
typedef enum lfba_termination {
  LFBA_CONVERGENCE = 0,
  LFBA_NO_CONVERGENCE = 1, /* max_num_iterations reached */
  LFBA_TERM_FAILURE = 2
} lfba_termination;

/* Which test ended the solve (extra detail Ceres only gives in summary.message). */
typedef enum lfba_stop_reason {
  LFBA_STOP_NONE = 0,
  LFBA_STOP_PARAMETER_TOLERANCE = 1,
  LFBA_STOP_FUNCTION_TOLERANCE = 2,
  LFBA_STOP_GRADIENT_TOLERANCE = 3,
  LFBA_STOP_MAX_ITERATIONS = 4,
  LFBA_STOP_MIN_RADIUS = 5,
  LFBA_STOP_INVALID_STEPS = 6
} lfba_stop_reason;

/* The inputs of performBundleAdjustment(), flattened (SURVEY.md 8(b)).
 * Observations are one per micro-image point, in the reference's frame-major order
 * (src/CameraCalibration.cpp:859-871), but any order is accepted. */
typedef struct lfba_problem {
  uint32_t config;    /* LFBA_CFG_* */
  int32_t calib_type; /* LFBA_CALIBRATION_ARUCO | LFBA_RECALIBRATION */
  double spx, spy;    /* pixelSize_totFoc (mm), passed twice at :882 */
  double scale;       /* (double)depth_to_raw_im_scale, :882 */
  int64_t n_obs;
  int32_t n_frames;
  int32_t n_points;
  const double* obs_x; /* frame.rawImageCoordinates[i][0]  (raw image px) */
  const double* obs_y;
  const double* ml_x; /* frame.microLensCenter[i][0]  (raw image px) */
  const double* ml_y;
  const int32_t* point_idx; /* index into p3d_w of frame.objectCoordinatesByRawID[i] */
  const int32_t* frame_idx; /* index into frames[] */
  /* distance constraints (constraintList, :916-925); used only if
   * LFBA_CFG_REFINE_POINTS && calib_type != LFBA_RECALIBRATION, as in the reference */
  int32_t n_constraints;
  const int32_t* c_p1;
  const int32_t* c_p2;
  const double* c_dist;
  const double* c_sigma;
} lfba_problem;

/* Solver options.  lfba_options_init() fills in what the reference sets (:955-962) on top of the
 * Ceres 2.1.0 defaults (SURVEY.md Appendix B.0). */
typedef struct lfba_options {
  int32_t max_num_iterations;  /* 200 */
  double function_tolerance;   /* 1e-6 */
  double parameter_tolerance;  /* 1e-8 */
  double gradient_tolerance;   /* 1e-10 */
  double initial_trust_region_radius; /* 1e4 */
  double max_trust_region_radius;     /* 1e16 */
  double min_trust_region_radius;     /* 1e-32 */
  double min_relative_decrease;       /* 1e-3 */
  double min_lm_diagonal;             /* 1e-6 */
  double max_lm_diagonal;             /* 1e32 */
  int32_t max_num_consecutive_invalid_steps; /* 5 */
  double loss_scale;                  /* CauchyLoss(a): a = 0.5 (:892) */
  int32_t minimizer_progress_to_stdout; /* 1 in the reference; prints the Ceres iteration table */
  int32_t device;                     /* CUDA device ordinal for a single-GPU solve; -1 = current */
  int32_t num_gpus;                   /* lfba_solve only: shard over this many visible GPUs (single process) */
  int32_t profile;                    /* 1: record per-kernel CUDA-event times into the summary */
  int32_t emulate_shards;             /* > 1: run the multi-GPU code path on ONE device — the problem is sharded this many
                                         ways exactly like num_gpus would, the shards run in lock-step on one stream and a
                                         device kernel sums their partial systems where the NCCL all-reduce would be
                                         (SURVEY.md section 4, item 4). lfba_solve and lfba_solver_create honour it. */
  int32_t reserved[7];
} lfba_options;

/* One row of the Ceres progress table (SURVEY.md Appendix B.7) = the per-iteration parity record. */
typedef struct lfba_iteration {
  int32_t iteration;
  int32_t step_is_valid;
  int32_t step_is_successful;
  int32_t line_search_iterations;
  double cost;
  double cost_change;
  double gradient_max_norm;
  double gradient_norm;
  double step_norm;
  double relative_decrease; /* tr_ratio */
  double trust_region_radius;
  double iteration_time_s;
  double cumulative_time_s;
} lfba_iteration;

#define LFBA_NUM_KERNEL_TIMERS 12
typedef struct lfba_summary {
  int32_t termination_type; /* lfba_termination */
  int32_t stop_reason;      /* lfba_stop_reason */
  int32_t num_iterations;   /* rows logged == ceres summary.iterations.size() */
  int32_t num_successful_steps;
  int32_t num_unsuccessful_steps;
  int32_t reduced_system_size; /* n of the reduced camera system */
  double initial_cost;
  double final_cost;
  int64_t num_jacobian_evals;    /* fused residual+Jacobian passes over all observations */
  int64_t num_observations;      /* N (global, all ranks) */
  int64_t num_tracks;            /* (point, frame) pairs */
  int64_t num_lenses;            /* distinct micro-lens centres */
  int64_t gpu_launches;          /* kernels launched by this library during the call */
  double setup_time_s;           /* H2D + sort + track/lens tables */
  double solve_time_s;           /* LM loop, host wall clock */
  double solve_gpu_ms;           /* LM loop, CUDA events */
  double kernel_ms[LFBA_NUM_KERNEL_TIMERS]; /* when opt.profile: accumulated per-kernel event times */
  int64_t kernel_calls[LFBA_NUM_KERNEL_TIMERS];
  /* caller-provided iteration log (may be NULL): filled with min(num_iterations, capacity) rows */
  lfba_iteration* iterations;
  int32_t iterations_capacity;
  int32_t reserved_i;
  /* set-up: the six observation arrays (40 B per observation) go up on their own copy stream, overlapped with the
   * device-side indexing; bytes and device time of that upload (CUDA events on the copy stream) */
  int64_t h2d_bytes;
  double h2d_ms;
} lfba_summary;

/* indices into lfba_summary.kernel_ms */
#define LFBA_T_LENS 0      /* per-lens undistortion table + per-frame rotation table */
#define LFBA_T_EVAL 1      /* fused residual + analytic Jacobian + track normal-equation blocks */
#define LFBA_T_SCHUR 2     /* per-point block assembly + 3x3 Schur elimination into S, g */
#define LFBA_T_ALLREDUCE 3 /* NCCL */
#define LFBA_T_DAMP 4      /* Jacobi scaling + LM diagonal on the reduced system */
#define LFBA_T_CHOL 5      /* tiled FP64 Cholesky + forward substitution */
#define LFBA_T_BACKSOLVE 6 /* reduced back substitution */
#define LFBA_T_POINTSTEP 7 /* per-point back substitution + candidate + model cost */
#define LFBA_T_CONTROL 8   /* LM accept/reject/radius/termination */
#define LFBA_T_MISC 9

/* Reprojection statistics of CameraCalibration::calcReprojectionError (:1026-1103). */
typedef struct lfba_reproj_stats {
  double std_x, std_y; /* sqrt(sum e^2 / n) */
  double mae_x, mae_y; /* max |e| (the reference's name) */
  int64_t num_points;
  int64_t num_inliers; /* e.x^2+e.y^2 <= thr^2 */
} lfba_reproj_stats;

/* Multi-process sharding (one process per GPU, e.g. under torchrun): every rank passes its shard
 * of the observations (global point/frame indices, all observations of a point on ONE rank) and
 * the same full camera/views/points arrays.  `nccl_unique_id` is the 128-byte ncclUniqueId made by
 * lfba_comm_unique_id() on rank 0 and distributed by the host's own plumbing (torch.distributed,
 * MPI, a file ...). */
typedef struct lfba_comm {
  int32_t rank;
  int32_t nranks;
  char nccl_unique_id[128];
  void* handle; /* optional: a communicator made by lfba_comm_create() (reused across solves); NULL = create one */
} lfba_comm;

typedef struct lfba_solver lfba_solver; /* opaque, device-resident problem */

int lfba_version(void);
const char* lfba_last_error(void); /* thread-local message of the last failing call */
const char* lfba_status_string(int status);
void lfba_options_init(lfba_options* opt);
/* number of usable sm_100 devices (0 => every compute call returns LFBA_NO_DEVICE) */
int lfba_device_count(void);
/* The library keeps the large device blocks of a finished solve (by size, per device) for the next one: repeated drop-in
 * calls on the same problem shape then pay no allocation. This returns them to the CUDA memory pool. */
void lfba_trim_cache(void);

/* Drop-in for src/CameraCalibration.cpp:858-965: camera[17], views[6F], points[3P] are in/out, updated
 * in place to the last accepted LM iterate exactly like Ceres does (SURVEY.md B.2). */
int lfba_solve(const lfba_problem* problem, const lfba_options* options, double* camera17, double* views6F,
               double* points3P, lfba_summary* summary);

/* Residuals and (optionally) Jacobians of every reprojection block at the given parameters, in the
 * input observation order; the arithmetic of OurCostFunctionBundle::operator_function<double/Jet>
 * (src/BundleAdjustment/BundleAdjustment.h:120-195), without the robust-loss correction.
 *   residuals   [2N]     (r_x, r_y) interleaved
 *   jac_camera  [2N*17]  row-major 2x17 per observation (Ceres block layout), or NULL
 *   jac_view    [2N*6]   row-major 2x6, or NULL
 *   jac_point   [2N*3]   row-major 2x3, or NULL
 *   cost        0.5*sum rho(|r|^2) with the loss selected by `config` (constraints included), or NULL
 *   stats       calcReprojectionError statistics (:1026-1103) at inlier threshold `inlier_threshold`, or NULL */
int lfba_eval(const lfba_problem* problem, const lfba_options* options, const double* camera17,
              const double* views6F, const double* points3P, double* residuals, double* jac_camera,
              double* jac_view, double* jac_point, double* cost, lfba_reproj_stats* stats,
              double inlier_threshold);

/* ---- the step before the solve: observation generation (SURVEY.md 8(f) N2) ----
 * What CameraCalibration::projectPointsToRawImage (src/CameraCalibration.cpp:640-769) reads from the MicroLensGrid
 * (src/MicroLensGrid/MicroLensGrid.h:48-73, maps built by defineMlMaps :338-421), flattened. Host memory. */
typedef struct lfba_lens_grid {
  int32_t raw_width, raw_height;   /* rawWidth, rawHeight */
  int32_t scale;                   /* depth_to_raw_im_scale */
  float lens_diameter;             /* mlGrid->lensDiameter (px) */
  float lens_validity_radius_2;    /* mlGrid->lensValidityRadius_2 */
  float rotation;                  /* mlGrid->rotation (rad), used for the epipolar web when rotation_on_grid */
  int32_t rotation_on_grid;        /* mlGrid->isRotationOnGrid() */
  int32_t n_lenses;
  const float* lens_cx;            /* MicroLens::centerX of mlLensList[i] */
  const float* lens_cy;
  const int32_t* map_next;         /* [raw_width * raw_height] index of mapNextMl[pixel] in mlLensList, -1 = NULL */
  const int32_t* map_ml;           /* [raw_width * raw_height] index of mapMlPointer[pixel], -1 = NULL */
} lfba_lens_grid;

/* Drop-in for the loops of projectPointsToRawImage: features are given frame-major like the reference walks them
 * (frames[i].imageCoordinates[p] -> feat_x/y, virtualDepthValues[i][p] -> vdepth, i -> frame_idx,
 * index of frames[i].objectCoordinatesByID[p] in p3d_w -> point_idx); the outputs are the concatenation over frames of
 * rawImageCoordinates / microLensCenter / objectCoordinatesByRawID in the reference's order — exactly the observation
 * arrays of lfba_problem. float32 arithmetic as in the reference: lens selection bit-exact, coordinates float32-exact.
 * Two-call pattern: capacity = 0 only counts (*n_obs); features must lie inside the total-focus image. */
int lfba_project_to_raw(const lfba_lens_grid* grid, int64_t n_features, const double* feat_x, const double* feat_y,
                        const double* vdepth, const int32_t* frame_idx, const int32_t* point_idx, int64_t capacity,
                        double* obs_x, double* obs_y, double* ml_x, double* ml_y, int32_t* out_point_idx,
                        int32_t* out_frame_idx, int64_t* n_obs, int32_t device);
/* Drop-in for CameraCalibration::initPlenopticParameters (src/CameraCalibration.cpp:456-498): fL_init = fph_init *
 * pixel_size_totfoc, then the least-squares fit of bL = v B + bL0 over all (frame, feature) pairs k: v = vdepth[k]
 * (virtualDepthValues), bL = fL Z / (Z - fL) with Z the camera-frame depth of point point_idx[k] in frame frame_idx[k]
 * (views = Euler angles + translation of worldToCam as in lfba_solve); rows with v < 2 or bL < 0 do not count (:483-488).
 * LFBA_FAILURE when fewer than two distinct valid virtual depths are left. */
int lfba_init_plenoptic(double fph_init, double pixel_size_totfoc, int64_t n_pairs, const double* vdepth,
                        const int32_t* frame_idx, const int32_t* point_idx, int32_t n_frames, const double* views6F,
                        int32_t n_points, const double* points3P, double* fL_init, double* B_init, double* bL0_init,
                        int32_t device);
/* The web of epipolar lines of CameraCalibration::defineEpiPolarLines (:521-634), host-side: lines3 [n][3] = (ex, ey,
 * base-line length) grouped by float-equal length in ascending order, group_begin [n_groups + 1]. NULL arrays: count only. */
int lfba_epipolar_web(float lens_diameter, float rotation, int32_t rotation_on_grid, int32_t* n_lines, int32_t* n_groups,
                      double* lines3, int32_t* group_begin);

/* ---- device-resident session API (what lfba_solve / lfba_eval are built from) ---- */
int lfba_comm_unique_id(char out[128]);
/* Persistent NCCL communicator for this rank (collective: every rank calls it). Pass it in lfba_comm.handle so that
 * repeated lfba_solver_create() calls do not pay ncclCommInitRank each time. The device must be current. */
int lfba_comm_create(const lfba_comm* comm, void** handle);
void lfba_comm_destroy(void* handle);
/* comm == NULL: single GPU (options->device). Uploads and indexes the problem (sort by point/frame,
 * track table, lens table). */
int lfba_solver_create(const lfba_problem* problem, const lfba_options* options, const lfba_comm* comm,
                       lfba_solver** out);
int lfba_solver_set_parameters(lfba_solver* s, const double* camera17, const double* views6F,
                               const double* points3P);
int lfba_solver_get_parameters(lfba_solver* s, double* camera17, double* views6F, double* points3P);
/* Runs the LM loop on the device-resident state. */
int lfba_solver_run(lfba_solver* s, lfba_summary* summary);
/* Times `reps` launches of the fused evaluation pass (materialize = 0) or of the eval-only kernel that writes residuals +
 * Jacobians to HBM at the current parameters: materialize = 1 in Ceres' block layout (camera block 2 x 17, what lfba_eval
 * returns), materialize = 2 with the camera block's live columns only (2 x NC). Returns mean ms per launch. */
int lfba_solver_time_eval(lfba_solver* s, int reps, int materialize, double* mean_ms);
/* Diagnostics for parity tests: one fused evaluation pass (the LM loop's own kernel) at the parameters last given by
 * lfba_solver_set_parameters, and its raw outputs — per (point, frame) track the normal-equation blocks in the CAMERA
 * frame, rec = [A (6: upper triangle of sum w G^T G, row-major) | b (3: sum w G^T r) | C (3 x NC row-major: sum w G^T Jc)],
 * G = d r / d P_c (2x3), w = rho' of CauchyLoss (1 without the robust flag); and camsum = [Hcc (lower triangle, row-major,
 * NC (NC+1)/2) | gc (NC) | cost]. Arrays may be NULL. *n_tracks and *rec_stride are outputs; rec needs
 * n_tracks * rec_stride doubles (query with rec == NULL first), trk_point / trk_frame n_tracks ints, camsum 64 doubles.
 * Single-shard sessions only. */
int lfba_solver_track_blocks(lfba_solver* s, int64_t* n_tracks, int32_t* rec_stride, double* rec, double* camsum64,
                             int32_t* trk_point, int32_t* trk_frame);
/* ---- parameter covariance (ceres::Covariance of the camera and pose blocks) ----
 * Sigma = (J^T W J)^-1 of the free parameters at the given / accepted parameters, W = rho' of CauchyLoss per observation
 * under LFBA_CFG_ROBUST (the Corrector's scaling of J, rho'' < 0), else 1; distance-constraint rows included. Not
 * multiplied by sigma2. Rows and columns that are exactly 0: camera entries beyond the live NC, camera[0] and camera[2] in
 * recalibration (SubsetManifold), the gauge frame, frames without observations, all poses without REFINE_POSES.
 * Gauge: with points refined, rigid motion of the scene (and without a distance constraint its scale) is free; the
 * first frame with observations is held fixed. Without constraints the scale trades against bL0 and B and the call
 * returns LFBA_INVALID_ARGUMENT, except in recalibration, where the constant fL and B fix the scale (DESIGN.md 10).
 * LFBA_FAILURE when an undamped point block Hpp or a pivot of the undamped reduced system is not positive. */
#define LFBA_GAUGE_NONE 0        /* points not refined: the reduced system is regular as it stands */
#define LFBA_GAUGE_FIRST_FRAME 1 /* points refined (+ constraints or recalibration): pose of gauge_frame held fixed */
typedef struct lfba_covariance_info {
  int32_t gauge, gauge_frame;  /* gauge_frame = first frame with observations, -1 for LFBA_GAUGE_NONE */
  int32_t n_reduced;           /* size of the system that was inverted */
  int32_t reserved_i;
  int64_t num_residuals;       /* 2N + K */
  int64_t num_free_parameters; /* live camera + poses of observed frames + active points, minus the gauge */
  double cost;                 /* 0.5 sum rho at the parameters */
  double sigma2;               /* 2 cost / (num_residuals - num_free_parameters); 0 when that is not positive */
  double gpu_ms;               /* device time of the call (CUDA events): evaluation, assembly, factorisation, inversion */
  double selinv_ms;            /* of which the selected inversion and the read-out of the blocks */
  double points_ms;            /* device time of the per-point blocks (not part of gpu_ms); 0 when they were not asked for */
  double reserved[1];
} lfba_covariance_info;

/* Covariance blocks at the parameters lfba_solver_get_parameters returns. cov_camera17: 17x17 row-major; cov_poses:
 * F x 6 x 6. Either may be NULL. Single-shard sessions only. The session is left as it was: a following
 * lfba_solver_run produces the same iterations. */
int lfba_solver_covariance(lfba_solver* s, double* cov_camera17, double* cov_poses, lfba_covariance_info* info);
/* One-shot form for the drop-in caller of lfba_solve (it has no session), built like lfba_eval. */
int lfba_covariance(const lfba_problem* pb, const lfba_options* opt, const double* camera17, const double* views6F,
                    const double* points3P, double* cov_camera17, double* cov_poses, lfba_covariance_info* info);
/* The same, plus the 3 x 3 covariance block of every point: cov_points is P x 3 x 3 row-major (must not be NULL), each
 * block exactly symmetric (ceres::Covariance::GetCovarianceBlock(point, point)). Camera, poses and info other than
 * points_ms are those lfba_solver_covariance / lfba_covariance return, bit for bit. Blocks that are exactly 0: points
 * without observations and constraints, and every point without REFINE_POINTS (constant blocks, status LFBA_OK). With
 * points refined, the blocks are relative to the gauge: the first frame with observations held fixed, so a point's
 * uncertainty is the uncertainty of its position in that frame's pose, not in an absolute world frame. Points coupled
 * by a distance constraint get their block of the reduced system's inverse. On a non-OK status cov_points may have been
 * overwritten (with zeros). */
int lfba_solver_covariance_points(lfba_solver* s, double* cov_camera17, double* cov_poses, double* cov_points,
                                  lfba_covariance_info* info);
int lfba_covariance_points(const lfba_problem* pb, const lfba_options* opt, const double* camera17, const double* views6F,
                           const double* points3P, double* cov_camera17, double* cov_poses, double* cov_points,
                           lfba_covariance_info* info);

/* Measures the device's FP64 FMA throughput (TFLOP/s) with a dependent-chain-free DFMA kernel. */
int lfba_measure_fp64_peak(int device, double* tflops);
void lfba_solver_destroy(lfba_solver* s);

#ifdef __cplusplus
}
#endif
#endif /* LFBA_H_ */
