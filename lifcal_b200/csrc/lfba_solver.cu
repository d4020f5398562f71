// lfba_solver.cu — host side of the C ABI (include/lfba.h): problem set-up, the round loop that enqueues the
// LM kernels, NCCL plumbing, result read-back.
//
// Drop-in boundary: lfba_solve() replaces src/CameraCalibration.cpp:858-965 (ceres::Problem construction,
// Solver::Options, ceres::Solve); the parameter arrays camera[17], views[6F], p3d_w are updated in place to
// the last accepted iterate like Ceres does. All LM decisions are taken by device kernels; the host enqueues
// rounds and polls one flag.
//
// Structure: a Solver is ONE SHARD of a problem on one device (its observations, its partial reduced system). A Group
// is what a caller's handle owns: one shard (single GPU, or this process's rank of an NCCL job), or — test hook
// lfba_options.emulate_shards — several shards on one device and one stream, run in lock-step. A round has three
// phases separated by the two points where the partial sums of the shards meet:
//   phase_eval      tables, fused evaluation at the candidate, (recalib: phi'(a) of the line search), CTA-partial sums
//   [sum over shards: 8 + nranks scalars]          NCCL all-reduce, or k_shard_allreduce over the emulated shards
//   phase_assemble  accept/reject (+ projected Armijo line search), Schur assembly at the accepted state
//   [sum over shards: S | g | gfull | hdiag | scalars]
//   phase_solve     damping, reduced solve, back-substitution + candidate, (recalib: line-search trial point)
#include <dlfcn.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "lfba_device.cuh"
#include "lfba_kernels.h"
#include "lfba_setup.cuh"

namespace lfba {

static thread_local std::string g_last_error;
static void set_error(const std::string& m) { g_last_error = m; }
static double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ------------------------------------------------------------------------------------------------
// NCCL, bound at run time (dlopen): inside a PyTorch process this resolves to the libnccl torch already
// loaded, so torch.distributed and this library share one NCCL; a plain C++ host gets the system one.
// ------------------------------------------------------------------------------------------------
struct Nccl {
  typedef struct ncclComm* comm_t;
  typedef struct { char internal[128]; } UniqueId;
  int (*GetUniqueId)(UniqueId*) = nullptr;
  int (*CommInitRank)(comm_t*, int, UniqueId, int) = nullptr;
  int (*CommDestroy)(comm_t) = nullptr;
  int (*CommAbort)(comm_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, comm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  void* handle = nullptr;
  bool ok = false;
  static Nccl& get() {
    static Nccl n;
    static std::once_flag once;
    std::call_once(once, [] {
      const char* names[] = {"libnccl.so.2", "libnccl.so"};
      for (const char* nm : names) {
        n.handle = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (n.handle) break;
      }
      if (!n.handle) return;
      n.GetUniqueId = (int (*)(UniqueId*))dlsym(n.handle, "ncclGetUniqueId");
      n.CommInitRank = (int (*)(comm_t*, int, UniqueId, int))dlsym(n.handle, "ncclCommInitRank");
      n.CommDestroy = (int (*)(comm_t))dlsym(n.handle, "ncclCommDestroy");
      n.CommAbort = (int (*)(comm_t))dlsym(n.handle, "ncclCommAbort");
      n.AllReduce =
          (int (*)(const void*, void*, size_t, int, int, comm_t, cudaStream_t))dlsym(n.handle, "ncclAllReduce");
      n.GetErrorString = (const char* (*)(int))dlsym(n.handle, "ncclGetErrorString");
      n.ok = n.GetUniqueId && n.CommInitRank && n.CommDestroy && n.AllReduce;
    });
    return n;
  }
};
constexpr int kNcclFloat64 = 8;  // ncclDouble
constexpr int kNcclInt32 = 2;    // ncclInt32
constexpr int kNcclSum = 0, kNcclMax = 2;
constexpr int kMaxEmulatedShards = 16;

__global__ void k_point_flags(const int32_t* pt_trk_begin, const int32_t* pt_coupled, int32_t* pt_active, int P) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p < P) pt_active[p] = (pt_trk_begin[p + 1] > pt_trk_begin[p] || pt_coupled[p] >= 0) ? 1 : 0;
}

// Emulated shards: what the NCCL all-reduce (sum) does for real ranks — every shard's buffer becomes the sum over all
// shards, added in shard order (fixed: deterministic).
struct ShardBufs {
  double* p[kMaxEmulatedShards];
  int n;
};
__global__ void k_shard_allreduce(ShardBufs b, size_t count) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int r = 0; r < b.n; ++r) s += b.p[r][i];
    for (int r = 0; r < b.n; ++r) b.p[r][i] = s;
  }
}

// ------------------------------------------------------------------------------------------------
struct StreamHolder {  // declared first in Solver => destroyed last, after every stream-ordered free has been queued
  cudaStream_t s = nullptr;
  int device = 0;
  bool owned = true;
  ~StreamHolder() {
    if (s && owned) {
      cudaSetDevice(device);
      cudaStreamSynchronize(s);
      cudaStreamDestroy(s);
    }
  }
};

struct Solver {
  StreamHolder sh;
  lfba_options opt;
  uint32_t config = 0;
  int calib_type = 0;
  int device = 0;
  int sms = 148;
  cudaStream_t stream = nullptr;
  int rank = 0, nranks = 1;
  ProblemIndex ix;
  Dev d;
  int lanes = 4;
  int frame_splits = 1;
  int n_tiles = 0;
  int band_frames = 0;
  PartPlan* part_plan = nullptr;
  int64_t launches = 0;
  double setup_time = 0, t_create0 = 0;
  int64_t n_obs_global = 0;
  int K = 0, Pc = 0;
  double spx = 0, spy = 0, scale = 1;
  std::vector<int32_t> h_fa;  // [F] frame has observations on this shard, [F] = co-visibility bandwidth of this shard

  DevBuf<int32_t> pt_coupled, coupled_pts, pt_active, frm_active, c_p1, c_p2, tile_first, row_c0;
  DevBuf<int64_t> row_off;
  DevBuf<double> c_dist, c_sigma;
  DevBuf<double> camera0, views0, points0;  // parameters given by the caller: every run() starts from them
  DevBuf<double> camera[2], views[2], points[2], lens, frames[2], rec[2], camsum[2], pdata, pscale, pstep;
  DevBuf<double> redbuf;  // S | g | gfull | hdiag | sys_scalars   (one all-reduce)
  DevBuf<double> rscale, rdamp, y, eval_scalars, part_eval, part_pts, part_step, part_ls, frame_part;
  DevBuf<CamModel> cm_buf;
  DevBuf<LmState> st;
  DevBuf<lfba_iteration> log;
  size_t S_len = 0, red_len = 0, es_len = ES_COUNT;
  std::vector<int> h_coupled;
  cudaEvent_t ev[LFBA_NUM_KERNEL_TIMERS + 1];
  bool ev_made = false;
  bool prof = false;
  LmState h_state{};
  double t_dbg = 0;
  void dbg_phase(const char* name) {  // LFBA_DEBUG: host wall time of the set-up phases (with a stream drain each)
    if (!std::getenv("LFBA_DEBUG")) return;
    cudaStreamSynchronize(stream);
    const double t = now_s();
    cudaMemPool_t pool;
    unsigned long long res = 0, used = 0, thr = 0;
    cudaDeviceGetDefaultMemPool(&pool, device);
    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &res);
    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
    cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    std::fprintf(stderr, "[lfba dbg] setup %-28s %8.2f ms   pool reserved %.2f GB used %.2f GB threshold %.3g\n", name,
                 1e3 * (t - (t_dbg > 0 ? t_dbg : t_create0)), res / 1e9, used / 1e9, (double)thr);
    t_dbg = t;
  }

  ~Solver() {
    cudaSetDevice(device);
    if (ev_made)
      for (auto& e : ev) cudaEventDestroy(e);
    part_plan_destroy(part_plan);
    alloc_stream() = stream;  // member buffers are freed (stream-ordered) right after this body
  }

  // ---- set-up, step 1: device, stream, index of this shard's observations (no communication) ----
  void create_local(const lfba_problem& pb, const lfba_options& o, int rank_, int nranks_, cudaStream_t shared_stream) {
    t_create0 = now_s();
    opt = o;
    config = pb.config;
    calib_type = pb.calib_type;
    rank = rank_;
    nranks = nranks_;
    spx = pb.spx;
    spy = pb.spy;
    scale = pb.scale;
    const bool rposes = (config & LFBA_CFG_REFINE_POSES) != 0, rpoints = (config & LFBA_CFG_REFINE_POINTS) != 0;
    if (!rposes && rpoints)
      throw CudaError("refinePoses=0 with refine3Dpoints=1 is invalid (null dereference in the reference, "
                      "src/BundleAdjustment/BundleAdjustment.h:149-152)", LFBA_INVALID_ARGUMENT);
    if (pb.n_obs < 0 || pb.n_frames <= 0 || pb.n_points <= 0)
      throw CudaError("empty problem: need n_frames > 0 and n_points > 0", LFBA_INVALID_ARGUMENT);
    if (pb.n_obs > 0 && (!pb.obs_x || !pb.obs_y || !pb.ml_x || !pb.ml_y || !pb.point_idx || !pb.frame_idx))
      throw CudaError("null observation array", LFBA_INVALID_ARGUMENT);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
      throw CudaError("no CUDA device: the LF-BA path has no CPU fallback", LFBA_NO_DEVICE);
    if (o.device >= 0) device = o.device; else LFBA_CUDA(cudaGetDevice(&device));
    LFBA_CUDA(cudaSetDevice(device));
    int cc_major = 0;  // attribute queries: cudaGetDeviceProperties costs milliseconds per call
    LFBA_CUDA(cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, device));
    if (cc_major < 10) throw CudaError("device is not sm_100-class: kernels are built for sm_100a only", LFBA_NO_DEVICE);
    LFBA_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    if (shared_stream) {
      stream = shared_stream;
      sh.owned = false;
    } else {
      LFBA_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    }
    sh.s = stream;
    sh.device = device;
    alloc_stream() = stream;
    {
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thr = ~0ull;  // keep freed memory in the pool for the next solve
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
      }
    }
    dbg_phase("device+stream");
    build_index(pb, ix, stream, &launches);
    dbg_phase("build_index");
    const int P = ix.P, F = ix.F;
    const bool recalib = calib_type == LFBA_RECALIBRATION;
    const bool use_constraints = rpoints && !recalib && pb.n_constraints > 0;  // :916
    K = use_constraints ? pb.n_constraints : 0;
    if (K > 0 && (!pb.c_p1 || !pb.c_p2 || !pb.c_dist || !pb.c_sigma))
      throw CudaError("null constraint array", LFBA_INVALID_ARGUMENT);

    // ---- coupled points (touched by a distance constraint): kept in the reduced system ----
    std::vector<int32_t> h_ptc((size_t)P, -1);
    h_coupled.clear();
    for (int k = 0; k < K; ++k) {
      const int a = pb.c_p1[k], b = pb.c_p2[k];
      if (a < 0 || a >= P || b < 0 || b >= P) throw CudaError("constraint point id out of range", LFBA_INVALID_ARGUMENT);
      h_ptc[a] = 0;
      h_ptc[b] = 0;
    }
    for (int p = 0; p < P; ++p)
      if (h_ptc[p] == 0) {
        h_ptc[p] = (int)h_coupled.size();
        h_coupled.push_back(p);
      }
    Pc = (int)h_coupled.size();
    pt_coupled.alloc(P);
    pt_coupled.upload(h_ptc.data(), P, stream);
    coupled_pts.alloc(std::max(1, Pc));
    coupled_pts.upload(h_coupled.data(), Pc, stream);
    pt_active.alloc(P);
    k_point_flags<<<(P + 255) / 256, 256, 0, stream>>>(ix.pt_trk_begin.p, pt_coupled.p, pt_active.p, P);
    ++launches;
    c_p1.alloc(std::max(1, K));
    c_p2.alloc(std::max(1, K));
    c_dist.alloc(std::max(1, K));
    c_sigma.alloc(std::max(1, K));
    if (K) {
      c_p1.upload(pb.c_p1, K, stream);
      c_p2.upload(pb.c_p2, K, stream);
      c_dist.upload(pb.c_dist, K, stream);
      c_sigma.upload(pb.c_sigma, K, stream);
    }
    h_fa.assign((size_t)F + 1, 0);
    for (int f = 0; f < F; ++f) h_fa[f] = ix.h_frame_count[f] > 0 ? 1 : 0;
    h_fa[F] = ix.bandwidth;
    LFBA_CUDA(cudaStreamSynchronize(stream));  // the host vectors above go out of scope
    dbg_phase("coupled points + flags");
  }

  // ---- set-up, step 2: with the frame flags / bandwidth / observation count of ALL shards known ----
  void create_finish(const std::vector<int32_t>& fa_global, int64_t n_obs_all) {
    LFBA_CUDA(cudaSetDevice(device));
    alloc_stream() = stream;
    const lfba_options& o = opt;
    const bool rposes = (config & LFBA_CFG_REFINE_POSES) != 0, rpoints = (config & LFBA_CFG_REFINE_POINTS) != 0;
    const int P = ix.P, F = ix.F, T = ix.T;
    const int nrad = (int)(config & 3u), tang = (config & LFBA_CFG_TANGENTIAL) ? 1 : 0;
    const int NC = 5 + nrad + 2 * tang;
    const bool recalib = calib_type == LFBA_RECALIBRATION;
    n_obs_global = n_obs_all;
    frm_active.alloc((size_t)F + 2);
    frm_active.upload(fa_global.data(), (size_t)F + 1, stream);
    const int bw = fa_global[F];
    band_frames = bw;

    // ---- reduced system layout [poses | coupled points | camera | rhs] and its skyline profile ----
    std::memset(&d, 0, sizeof(d));
    d.np6 = rposes ? 6 * F : 0;
    d.band = bw;
    d.Pc = Pc;
    int ncr = 0;
    for (int c = 0; c < kMaxNC; ++c) d.cam_red[c] = -1;
    for (int c = 0; c < NC; ++c) {
      if (recalib && (c == 0 || c == 2)) continue;  // SubsetManifold(17, {0, 2}) (:930-940)
      d.cam_red[c] = d.np6 + 3 * Pc + ncr;
      ++ncr;
    }
    d.n_cam_red = ncr;
    d.n = d.np6 + 3 * Pc + ncr;
    const int n = d.n, n_aug = n + 1;
    std::vector<int32_t> h_c0((size_t)n_aug);
    std::vector<int64_t> h_off((size_t)n_aug + 1);
    for (int r = 0; r < n_aug; ++r) {
      int c0 = 0;
      if (r < d.np6) c0 = 6 * std::max(0, r / 6 - bw);
      h_c0[r] = c0;
    }
    h_off[0] = 0;
    for (int r = 0; r < n_aug; ++r) h_off[r + 1] = h_off[r] + (int64_t)(r - h_c0[r] + 1);
    S_len = (size_t)h_off[n_aug];
    n_tiles = (n_aug + kTile - 1) / kTile;
    std::vector<int32_t> h_tf((size_t)n_tiles);
    for (int t = 0; t < n_tiles; ++t) {
      int m = std::numeric_limits<int>::max();
      for (int r = t * kTile; r < std::min(n_aug, (t + 1) * kTile); ++r) m = std::min(m, h_c0[r] / kTile);
      h_tf[t] = m;
    }
    row_c0.alloc(n_aug);
    row_c0.upload(h_c0.data(), n_aug, stream);
    row_off.alloc((size_t)n_aug + 1);
    row_off.upload(h_off.data(), (size_t)n_aug + 1, stream);
    tile_first.alloc(n_tiles);
    tile_first.upload(h_tf.data(), n_tiles, stream);

    dbg_phase("layout");
    // ---- buffers ----
    red_len = S_len + 3 * (size_t)n + SS_COUNT + (size_t)nranks;
    es_len = ES_COUNT + (size_t)nranks;
    redbuf.alloc(red_len);
    rscale.alloc(std::max(1, n));
    rdamp.alloc(std::max(1, n));
    y.alloc(std::max(1, n));
    y.zero(stream);
    eval_scalars.alloc(es_len);
    eval_scalars.zero(stream);
    for (int b = 0; b < 2; ++b) {
      camera[b].alloc(17);
      views[b].alloc((size_t)6 * F);
      points[b].alloc((size_t)3 * P);
      frames[b].alloc((size_t)F * kFrameStride);
      rec[b].alloc((size_t)std::max(1, T) * rec_stride(NC));
      camsum[b].alloc(64);
      camsum[b].zero(stream);
    }
    lens.alloc((size_t)std::max(1, ix.NL) * kLensStride);
    pdata.alloc((size_t)P * kPointStride);
    pdata.zero(stream);
    pscale.alloc((size_t)3 * P);
    if (recalib) {
      pstep.alloc((size_t)3 * P);
      pstep.zero(stream);
    }
    st.alloc(1);
    log.alloc(kMaxLog);
    cm_buf.alloc(1);
    cm_buf.zero(stream);

    // ---- launch geometry ----
    d.grid_pts = std::max(1, std::min(4 * sms, (P + 127) / 128));
    part_pts.alloc((size_t)d.grid_pts * 64);
    part_step.alloc((size_t)d.grid_pts * 8);
    part_ls.alloc((size_t)d.grid_pts);
    part_pts.zero(stream);
    part_step.zero(stream);
    part_ls.zero(stream);
    // lanes per track (L): the fused evaluation walks ROUNDS of 32 / L length-adjacent tracks per warp. L = 1 has no
    // cross-lane reduction and no predicated per-track work (measured at cfg4: 4.9 ms vs 7.3 ms for L = 4), so L grows
    // only while there are too few rounds to give every warp of the grid a few of them.
    {
      const double mean_len = T > 0 ? (double)ix.N / T : 1.0;
      d.grid_eval = std::max(1, 2 * sms);
      const int64_t warps = (int64_t)d.grid_eval * 4;
      int L = 1;
      while (L < 16 && ((int64_t)T * L + 31) / 32 < 2 * warps && L * 2 <= mean_len) L *= 2;
      if (const char* e = std::getenv("LFBA_LANES")) L = std::max(1, std::min(16, std::atoi(e)));  // experiment
      lanes = L;
      const int64_t rounds = ((int64_t)T * L + 31) / 32;
      d.grid_eval = std::max(1, (int)std::min<int64_t>(2 * sms, (rounds + 3) / 4));
    }
    part_eval.alloc((size_t)d.grid_eval * 64);
    dbg_phase("buffers");
    build_stream(ix, lanes, stream, &launches);
    dbg_phase("packed stream");
    {
      // frames that have tracks ON THIS SHARD: a shard of a multi-GPU solve touches F / nranks of them, and one CTA per
      // frame would leave most SMs idle — split the frames' track lists over several CTAs then
      int f_local = 0;
      for (int f = 0; f < F; ++f) f_local += ix.h_frame_count[f] > 0 ? 1 : 0;
      f_local = std::max(1, f_local);
      const int per_frame = (T + f_local - 1) / f_local;
      frame_splits = std::max(1, std::min(16, std::min((4 * sms) / f_local, (per_frame + 255) / 256)));
      // long track lists are split even when there are frames enough: the CTAs in flight then cover few frames, whose
      // points' data is still in L2 when the neighbouring frames ask for it (measured at cfg4: 1.88 -> 1.75 ms)
      frame_splits = std::max(frame_splits, std::min(8, per_frame / 512));
      if (const char* e = std::getenv("LFBA_FRAME_SPLITS")) frame_splits = std::max(1, std::min(16, std::atoi(e)));  // test hook
      frame_part.alloc((size_t)std::max(1, F) * frame_splits * (39 + 6 * kMaxNC));
    }

    // ---- Dev ----
    d.N = ix.N; d.T = T; d.P = P; d.F = F; d.NL = ix.NL; d.K = K; d.NC = NC;
    d.rank = rank; d.nranks = nranks; d.config = config; d.recalib = recalib ? 1 : 0;
    d.refine_poses = rposes ? 1 : 0; d.refine_points = rpoints ? 1 : 0;
    d.debug = std::getenv("LFBA_DEBUG") != nullptr ? 1 : 0;
    d.spx = spx; d.spy = spy; d.scale = scale;
    d.opt.max_iter = o.max_num_iterations; d.opt.ftol = o.function_tolerance; d.opt.ptol = o.parameter_tolerance;
    d.opt.gtol = o.gradient_tolerance; d.opt.r0 = o.initial_trust_region_radius; d.opt.rmax = o.max_trust_region_radius;
    d.opt.rmin = o.min_trust_region_radius; d.opt.min_rel_dec = o.min_relative_decrease;
    d.opt.min_diag = o.min_lm_diagonal; d.opt.max_diag = o.max_lm_diagonal;
    d.opt.max_invalid = o.max_num_consecutive_invalid_steps; d.opt.loss_a = o.loss_scale;
    d.obs = ix.obs_sorted; d.lens_id = ix.lens_id_sorted; d.trk_point = ix.trk_point.p; d.trk_frame = ix.trk_frame.p;
    d.trk_begin = ix.trk_begin.p; d.pt_trk_begin = ix.pt_trk_begin.p; d.frm_begin = ix.frm_begin.p;
    d.frm_trk = ix.frm_trk.p; d.pair_begin = ix.pair_begin.p; d.pair_f1 = ix.pair_f1.p; d.pair_f2 = ix.pair_f2.p;
    d.pair_t1 = ix.pair_t1.p; d.pair_t2 = ix.pair_t2.p; d.npairs = ix.npairs; d.eval_order = ix.eval_order.p; d.eval_pf = ix.eval_pf.p;
    d.round_cost = 6;
    if (const char* e = std::getenv("LFBA_ROUND_COST")) d.round_cost = std::max(0, std::min(64, std::atoi(e)));  // experiment
    d.s_obs = ix.s_obs.p; d.s_lid = ix.s_lid.p; d.step_base = ix.step_base.p;
    d.n_rounds = ix.n_rounds; d.n_rows = ix.n_rows; d.stream_L = ix.stream_L;
    d.pt_coupled = pt_coupled.p; d.coupled_pts = coupled_pts.p; d.pt_active = pt_active.p; d.frm_active = frm_active.p;
    d.c_p1 = c_p1.p; d.c_p2 = c_p2.p; d.c_dist = c_dist.p; d.c_sigma = c_sigma.p;
    for (int c = 0; c < 17; ++c) {
      d.cam_lo[c] = -std::numeric_limits<double>::max();
      d.cam_hi[c] = std::numeric_limits<double>::max();
    }
    for (int b = 0; b < 2; ++b) {
      d.camera[b] = camera[b].p; d.views[b] = views[b].p; d.points[b] = points[b].p;
      d.frames[b] = frames[b].p; d.rec[b] = rec[b].p; d.camsum[b] = camsum[b].p;
    }
    d.lens = lens.p; d.lens_xy = ix.lens_xy.p; d.cm_buf = cm_buf.p;
    d.pdata = pdata.p; d.pscale = pscale.p; d.pstep = pstep.p;
    d.S = redbuf.p; d.row_off = row_off.p; d.row_c0 = row_c0.p;
    d.g = redbuf.p + S_len; d.gfull = d.g + n; d.hdiag = d.gfull + n; d.sys_scalars = d.hdiag + n;
    d.rscale = rscale.p; d.rdamp = rdamp.p; d.y = y.p; d.eval_scalars = eval_scalars.p;
    d.part_eval = part_eval.p; d.part_pts = part_pts.p; d.part_step = part_step.p; d.part_ls = part_ls.p;
    d.frame_part = frame_part.p;
    d.st = st.p; d.log = log.p;
    for (auto& e : ev) LFBA_CUDA(cudaEventCreate(&e));
    ev_made = true;
    prepare_device_kernels();
    prepare_eval_kernels();
    prepare_cov_kernels();
    dbg_phase("events + kernel attributes");
    part_plan = part_plan_create(d, band_frames, stream);
    LFBA_CUDA(cudaStreamSynchronize(stream));
    LFBA_CUDA(cudaGetLastError());
    dbg_phase("partition plan");
    setup_time = now_s() - t_create0;
  }

  void set_parameters(const double* cam, const double* vw_, const double* pts) {
    LFBA_CUDA(cudaSetDevice(device));
    alloc_stream() = stream;
    // the accepted-state slot is 0 until the first accept flips it; the initial point enters as candidate (slot 1)
    camera0.alloc(17);
    views0.alloc((size_t)6 * ix.F);
    points0.alloc((size_t)3 * ix.P);
    camera0.upload(cam, 17, stream);
    views0.upload(vw_, (size_t)6 * ix.F, stream);
    points0.upload(pts, (size_t)3 * ix.P, stream);
    reset_parameters();
    if (calib_type == LFBA_RECALIBRATION) {  // bounds from the INITIAL values (:943-951)
      const int bj[3] = {1, 3, 4};
      for (int k = 0; k < 3; ++k) {
        const double a = 0.7 * cam[bj[k]], b = 1.3 * cam[bj[k]];
        d.cam_lo[bj[k]] = std::min(a, b);
        d.cam_hi[bj[k]] = std::max(a, b);
      }
    }
    LFBA_CUDA(cudaStreamSynchronize(stream));
  }

  void reset_parameters() {
    for (int b = 0; b < 2; ++b) {
      LFBA_CUDA(cudaMemcpyAsync(camera[b].p, camera0.p, 17 * sizeof(double), cudaMemcpyDeviceToDevice, stream));
      LFBA_CUDA(cudaMemcpyAsync(views[b].p, views0.p, (size_t)6 * ix.F * sizeof(double), cudaMemcpyDeviceToDevice, stream));
      LFBA_CUDA(cudaMemcpyAsync(points[b].p, points0.p, (size_t)3 * ix.P * sizeof(double), cudaMemcpyDeviceToDevice, stream));
    }
  }

  void get_parameters(int which, double* cam, double* vw_, double* pts) {
    LFBA_CUDA(cudaSetDevice(device));
    if (cam) camera[which].download(cam, 17, stream);
    if (vw_) views[which].download(vw_, (size_t)6 * ix.F, stream);
    if (pts) points[which].download(pts, (size_t)3 * ix.P, stream);
    LFBA_CUDA(cudaStreamSynchronize(stream));
  }

  // ---- one LM solve, phase by phase (driven by Group::run) ----
  void begin_run() {
    LFBA_CUDA(cudaSetDevice(device));
    if (!camera0.p) throw CudaError("lfba_solver_run before lfba_solver_set_parameters", LFBA_INVALID_ARGUMENT);
    LmState init;
    std::memset(&init, 0, sizeof(init));
    init.cur = 0;
    init.solve_ok = 1;
    init.radius = opt.initial_trust_region_radius;
    init.decrease_factor = 2.0;
    reset_parameters();  // every run starts from the parameters last given by the caller
    LFBA_CUDA(cudaMemcpyAsync(st.p, &init, sizeof(LmState), cudaMemcpyHostToDevice, stream));
    launch_init_norms(d, stream);  // also projects the start point into the box (recalib)
    ++launches;
  }
  void mark(int slot) {
    if (prof) LFBA_CUDA(cudaEventRecord(ev[slot], stream));
  }
  void phase_eval() {
    if (prof) LFBA_CUDA(cudaEventRecord(ev[LFBA_NUM_KERNEL_TIMERS], stream));
    launch_tables(d, stream);
    mark(LFBA_T_LENS);
    launches += launch_eval(d, lanes, stream);
    launches += launch_ls_gdot(d, stream);
    mark(LFBA_T_EVAL);
    launch_reduce_eval(d, stream);
    launches += 2;
  }
  void phase_assemble() {
    launch_control_accept(d, stream);
    mark(LFBA_T_CONTROL);
    LFBA_CUDA(cudaMemsetAsync(redbuf.p, 0, red_len * sizeof(double), stream));
    launches += 2;
    launches += launch_assembly(d, frame_splits, stream);
    mark(LFBA_T_SCHUR);
  }
  void phase_solve() {
    mark(LFBA_T_ALLREDUCE);
    launch_finalize(d, stream);
    mark(LFBA_T_DAMP);
    launches += 1 + launch_reduced_solve(d, n_tiles, tile_first.p, band_frames, stream, part_plan);
    mark(LFBA_T_CHOL);
    launches += launch_steps(d, stream);
    launches += launch_ls_apply(d, stream);
    mark(LFBA_T_POINTSTEP);
  }

  // ---- covariance of camera and poses at the accepted parameters (lfba_solver_covariance) ----
  // One evaluation pass and the Schur assembly of the undamped J^T W J there, the in-place Cholesky, the selected
  // inversion. It runs on the round's work buffers with a fresh device LmState; the host's h_state and the caller's
  // parameters (camera0 ...) are not touched, and run() rebuilds everything else from them. With cov_points, the
  // per-point blocks follow from the selected inverse and the point data of the same assembly (k_cov_points).
  void covariance(double* cov_cam, double* cov_poses, double* cov_points, lfba_covariance_info* info) {
    LFBA_CUDA(cudaSetDevice(device));
    alloc_stream() = stream;
    if (!camera0.p) throw CudaError("lfba_solver_covariance before lfba_solver_set_parameters", LFBA_INVALID_ARGUMENT);
    const bool recalib = calib_type == LFBA_RECALIBRATION;
    // with points refined, rigid motion + scale are free; a distance constraint (or recalibration's constant fL and B)
    // fixes the scale, and holding one frame's pose then removes the rest (DESIGN.md section 10)
    if (d.refine_points && K == 0 && !recalib)
      throw CudaError("covariance: points are refined without a distance constraint, so the scale gauge (scene scale "
                      "against bL0 and B) leaves the covariance undefined", LFBA_INVALID_ARGUMENT);
    int gf = -1;
    if (d.refine_points)
      for (int f = 0; f < ix.F && gf < 0; ++f)
        if (h_fa[f]) gf = f;
    Dev dc = d;
    dc.undamped = 1;
    dc.gauge_frame = gf;
    const int F = ix.F;
    cudaEvent_t e0, e1, e2, e3 = nullptr;
    LFBA_CUDA(cudaEventCreate(&e0));
    LFBA_CUDA(cudaEventCreate(&e1));
    LFBA_CUDA(cudaEventCreate(&e2));
    if (cov_points) LFBA_CUDA(cudaEventCreate(&e3));
    LFBA_CUDA(cudaEventRecord(e0, stream));
    LmState init;
    std::memset(&init, 0, sizeof(init));
    init.cur = 1 - h_state.cur;  // the accepted parameters enter as the candidate of iteration zero
    init.solve_ok = 1;
    LFBA_CUDA(cudaMemcpyAsync(st.p, &init, sizeof(LmState), cudaMemcpyHostToDevice, stream));
    launch_tables(dc, stream);
    launches += launch_eval(dc, lanes, stream);
    launch_reduce_eval(dc, stream);
    launch_control_accept(dc, stream);  // iteration zero: the candidate becomes the accepted state, its cost x_cost
    LFBA_CUDA(cudaMemsetAsync(redbuf.p, 0, red_len * sizeof(double), stream));
    launches += 3 + launch_assembly(dc, frame_splits, stream);
    launch_finalize(dc, stream);
    launches += 1 + launch_chol_inplace(dc, n_tiles, tile_first.p, band_frames, stream);
    LFBA_CUDA(cudaEventRecord(e1, stream));
    DevBuf<double> Z(S_len), out((size_t)289 + 36 * (size_t)F);
    launches += launch_covariance(dc, Z.p, out.p, stream);
    LFBA_CUDA(cudaEventRecord(e2, stream));
    DevBuf<double> outp(cov_points ? (size_t)9 * ix.P : 0);
    if (cov_points) {
      launches += launch_cov_points(dc, Z.p, outp.p, stream);
      LFBA_CUDA(cudaEventRecord(e3, stream));
    }
    std::vector<double> h_out((size_t)289 + 36 * (size_t)F);
    out.download(h_out.data(), h_out.size(), stream);
    if (cov_points && ix.P > 0)
      LFBA_CUDA(cudaMemcpyAsync(cov_points, outp.p, (size_t)9 * ix.P * sizeof(double), cudaMemcpyDeviceToHost, stream));
    LmState hs;
    double ptfail = 0.0;
    LFBA_CUDA(cudaMemcpyAsync(&hs, st.p, sizeof(LmState), cudaMemcpyDeviceToHost, stream));
    LFBA_CUDA(cudaMemcpyAsync(&ptfail, d.sys_scalars + SS_PTFAIL, sizeof(double), cudaMemcpyDeviceToHost, stream));
    std::vector<int32_t> h_pa;
    if (d.refine_points) {
      h_pa.resize((size_t)ix.P);
      pt_active.download(h_pa.data(), (size_t)ix.P, stream);
    }
    LFBA_CUDA(cudaStreamSynchronize(stream));
    LFBA_CUDA(cudaGetLastError());
    float ms_all = 0.f, ms_inv = 0.f, ms_pts = 0.f;
    cudaEventElapsedTime(&ms_all, e0, e2);
    cudaEventElapsedTime(&ms_inv, e1, e2);
    if (e3) {
      cudaEventElapsedTime(&ms_pts, e2, e3);
      cudaEventDestroy(e3);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaEventDestroy(e2);
    if (ptfail > 0.0)
      throw CudaError("covariance: an undamped point block Hpp is not positive definite (a point is not determined by "
                      "its observations)", LFBA_FAILURE);
    if (!hs.solve_ok)
      throw CudaError("covariance: a pivot of the undamped reduced system is not positive (J^T W J is singular at "
                      "these parameters)", LFBA_FAILURE);
    if (cov_cam) std::memcpy(cov_cam, h_out.data(), 289 * sizeof(double));
    if (cov_poses) std::memcpy(cov_poses, h_out.data() + 289, (size_t)36 * F * sizeof(double));
    if (info) {
      std::memset(info, 0, sizeof(*info));
      info->gauge = gf >= 0 ? LFBA_GAUGE_FIRST_FRAME : LFBA_GAUGE_NONE;
      info->gauge_frame = gf;
      info->n_reduced = d.n;
      info->num_residuals = 2 * n_obs_global + K;
      int64_t np = d.n_cam_red;
      if (d.refine_poses)
        for (int f = 0; f < F; ++f) np += h_fa[f] ? 6 : 0;
      for (int32_t a : h_pa) np += a ? 3 : 0;
      if (gf >= 0) np -= 6;
      info->num_free_parameters = np;
      info->cost = hs.x_cost;
      const int64_t dof = info->num_residuals - np;
      info->sigma2 = dof > 0 ? 2.0 * hs.x_cost / (double)dof : 0.0;
      info->gpu_ms = ms_all;
      info->selinv_ms = ms_inv;
      info->points_ms = ms_pts;
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Sharding by point: contiguous point ranges balanced by observation count; every observation of a point goes to the
// point's owner (the per-point 3x3 elimination needs them together); constraint-coupled points live on shard 0.
// ------------------------------------------------------------------------------------------------
struct HostShards {
  std::vector<int> owner;
  struct Arrays {
    std::vector<double> ox, oy, mx, my;
    std::vector<int32_t> pi, fi;
  };
  std::vector<Arrays> sh;
  void split(const lfba_problem& pb, int G) {
    const int P = pb.n_points;
    const int64_t N = pb.n_obs;
    if (P <= 0 || pb.n_frames <= 0 || N < 0) throw CudaError("empty problem: need n_frames > 0 and n_points > 0", LFBA_INVALID_ARGUMENT);
    if (N > 0 && (!pb.obs_x || !pb.obs_y || !pb.ml_x || !pb.ml_y || !pb.point_idx || !pb.frame_idx))
      throw CudaError("null observation array", LFBA_INVALID_ARGUMENT);
    for (int64_t i = 0; i < N; ++i)
      if (pb.point_idx[i] < 0 || pb.point_idx[i] >= P || pb.frame_idx[i] < 0 || pb.frame_idx[i] >= pb.n_frames)
        throw CudaError("observation index out of range", LFBA_INVALID_ARGUMENT);
    const bool use_c = (pb.config & LFBA_CFG_REFINE_POINTS) && pb.calib_type != LFBA_RECALIBRATION && pb.n_constraints > 0;
    if (use_c) {
      if (!pb.c_p1 || !pb.c_p2 || !pb.c_dist || !pb.c_sigma) throw CudaError("null constraint array", LFBA_INVALID_ARGUMENT);
      for (int k = 0; k < pb.n_constraints; ++k)
        if (pb.c_p1[k] < 0 || pb.c_p1[k] >= P || pb.c_p2[k] < 0 || pb.c_p2[k] >= P)
          throw CudaError("constraint point id out of range", LFBA_INVALID_ARGUMENT);
    }
    std::vector<int64_t> cnt((size_t)P + 1, 0);
    for (int64_t i = 0; i < N; ++i) cnt[pb.point_idx[i] + 1]++;
    for (int p = 0; p < P; ++p) cnt[p + 1] += cnt[p];
    owner.assign((size_t)P, 0);
    for (int p = 0; p < P; ++p) owner[p] = (int)std::min<int64_t>(G - 1, (cnt[p] * G) / std::max<int64_t>(1, N));
    if (use_c)
      for (int k = 0; k < pb.n_constraints; ++k) owner[pb.c_p1[k]] = owner[pb.c_p2[k]] = 0;
    sh.assign((size_t)G, Arrays());
    for (int64_t i = 0; i < N; ++i) {
      Arrays& s = sh[(size_t)owner[pb.point_idx[i]]];
      s.ox.push_back(pb.obs_x[i]);
      s.oy.push_back(pb.obs_y[i]);
      s.mx.push_back(pb.ml_x[i]);
      s.my.push_back(pb.ml_y[i]);
      s.pi.push_back(pb.point_idx[i]);
      s.fi.push_back(pb.frame_idx[i]);
    }
  }
  lfba_problem view(const lfba_problem& pb, int r) const {
    lfba_problem lp = pb;
    lp.n_obs = (int64_t)sh[r].ox.size();
    lp.obs_x = sh[r].ox.data();
    lp.obs_y = sh[r].oy.data();
    lp.ml_x = sh[r].mx.data();
    lp.ml_y = sh[r].my.data();
    lp.point_idx = sh[r].pi.data();
    lp.frame_idx = sh[r].fi.data();
    return lp;
  }
};

// ------------------------------------------------------------------------------------------------
struct Group {
  std::vector<std::unique_ptr<Solver>> sh;
  std::vector<int> owner;  // emulated shards: owner of each point
  Nccl::comm_t comm = nullptr;
  bool own_comm = false;
  int rank = 0, nranks = 1;  // of this process in the NCCL job (1 when single-GPU or emulated)
  int* h_done = nullptr;     // pinned
  cudaEvent_t ev_round[4];
  bool ev_made = false;
  lfba_options opt;
  const std::atomic<int>* comm_aborted = nullptr;  // lfba_solve(num_gpus): set when a peer aborted the communicators

  ~Group() {
    if (!sh.empty()) cudaSetDevice(sh[0]->device);
    if (ev_made)
      for (auto& e : ev_round) cudaEventDestroy(e);
    while (!sh.empty()) sh.pop_back();  // reverse order: shard 0 owns the stream the emulated shards share
    if (comm && own_comm && !(comm_aborted && comm_aborted->load())) Nccl::get().CommDestroy(comm);
  }
  Solver& s0() { return *sh[0]; }
  bool emulated() const { return sh.size() > 1; }

  void nccl_allreduce(void* buf, size_t count, int dtype, int op) {
    if (nranks <= 1 || count == 0) return;
    const int rc = Nccl::get().AllReduce(buf, buf, count, dtype, op, comm, s0().stream);
    if (rc != 0) throw CudaError(std::string("ncclAllReduce: ") + Nccl::get().GetErrorString(rc), LFBA_NCCL_ERROR);
  }
  // where the partial sums of the shards meet; which: 0 = evaluation scalars, 1 = reduced system
  void reduce(int which) {
    if (emulated()) {
      ShardBufs b;
      b.n = (int)sh.size();
      for (int r = 0; r < b.n; ++r) b.p[r] = which == 0 ? sh[r]->eval_scalars.p : sh[r]->redbuf.p;
      const size_t count = which == 0 ? s0().es_len : s0().red_len;
      const int grid = (int)std::min<size_t>(4 * (size_t)s0().sms, (count + 255) / 256);
      k_shard_allreduce<<<std::max(1, grid), 256, 0, s0().stream>>>(b, count);
      s0().launches += 1;
    } else if (nranks > 1) {
      if (which == 0) nccl_allreduce(s0().eval_scalars.p, s0().es_len, kNcclFloat64, kNcclSum);
      else nccl_allreduce(s0().redbuf.p, s0().red_len, kNcclFloat64, kNcclSum);
    }
  }

  void create(const lfba_problem& pb, const lfba_options& o, const lfba_comm* cm) {
    opt = o;
    const int E = o.emulate_shards > 1 ? o.emulate_shards : 1;
    if (E > 1 && cm && cm->nranks > 1)
      throw CudaError("emulate_shards cannot be combined with an NCCL communicator", LFBA_INVALID_ARGUMENT);
    if (E > kMaxEmulatedShards) throw CudaError("emulate_shards > 16", LFBA_INVALID_ARGUMENT);
    if (E > 1) {
      HostShards hs;
      hs.split(pb, E);
      owner = hs.owner;
      for (int r = 0; r < E; ++r) {
        sh.emplace_back(new Solver());
        const lfba_problem lp = hs.view(pb, r);
        sh[r]->create_local(lp, o, r, E, r == 0 ? nullptr : sh[0]->stream);
      }
    } else {
      sh.emplace_back(new Solver());
      if (cm && cm->nranks > 1) {
        rank = cm->rank;
        nranks = cm->nranks;
      }
      sh[0]->create_local(pb, o, rank, nranks, nullptr);
      if (nranks > 1) {
        Nccl& n = Nccl::get();
        if (!n.ok) throw CudaError("libnccl.so.2 not found", LFBA_NCCL_ERROR);
        if (cm->handle) {
          comm = (Nccl::comm_t)cm->handle;
        } else {
          Nccl::UniqueId id;
          std::memcpy(id.internal, cm->nccl_unique_id, 128);
          const int rc = n.CommInitRank(&comm, nranks, id, rank);
          if (rc != 0) throw CudaError(std::string("ncclCommInitRank: ") + n.GetErrorString(rc), LFBA_NCCL_ERROR);
          own_comm = true;
        }
      }
    }
    // ---- frames with observations anywhere, co-visibility bandwidth, observation count: over all shards ----
    const int F = s0().ix.F;
    std::vector<int32_t> fa((size_t)F + 1, 0);
    int64_t n_all = 0;
    for (auto& s : sh) {
      for (int f = 0; f <= F; ++f) fa[f] = std::max(fa[f], s->h_fa[f]);
      n_all += s->ix.N;
    }
    if (nranks > 1) {
      Solver& s = s0();
      alloc_stream() = s.stream;
      DevBuf<int32_t> dfa((size_t)F + 1);
      DevBuf<double> dn(1);
      double h_n = (double)n_all;
      dfa.upload(fa.data(), (size_t)F + 1, s.stream);
      dn.upload(&h_n, 1, s.stream);
      nccl_allreduce(dfa.p, (size_t)F + 1, kNcclInt32, kNcclMax);
      nccl_allreduce(dn.p, 1, kNcclFloat64, kNcclSum);
      dfa.download(fa.data(), (size_t)F + 1, s.stream);
      dn.download(&h_n, 1, s.stream);
      LFBA_CUDA(cudaStreamSynchronize(s.stream));
      n_all = (int64_t)(h_n + 0.5);
    }
    for (auto& s : sh) s->create_finish(fa, n_all);
    h_done = pinned_flags();
    for (auto& e : ev_round) LFBA_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ev_made = true;
  }
  // four pinned ints per host thread for the `done` polling, allocated once (cudaMallocHost costs about a millisecond);
  // a Group only uses them inside run(), which blocks its thread
  static int* pinned_flags() {
    static thread_local int* p = nullptr;
    if (!p) LFBA_CUDA(cudaMallocHost(&p, 4 * sizeof(int)));
    return p;
  }

  void set_parameters(const double* c, const double* v, const double* p) {
    for (auto& s : sh) s->set_parameters(c, v, p);
  }
  void get_parameters(double* c, double* v, double* p) {
    Solver& a = s0();
    a.get_parameters(a.h_state.cur, c, v, p);
    if (p && emulated()) {  // every shard moved only its own points
      std::vector<double> tmp((size_t)3 * a.ix.P);
      for (size_t r = 1; r < sh.size(); ++r) {
        sh[r]->get_parameters(sh[r]->h_state.cur, nullptr, nullptr, tmp.data());
        for (int q = 0; q < a.ix.P; ++q)
          if (owner[q] == (int)r)
            for (int j = 0; j < 3; ++j) p[3 * (size_t)q + j] = tmp[3 * (size_t)q + j];
      }
    }
  }

  int run(lfba_summary* sum) {
    Solver& a = s0();
    LFBA_CUDA(cudaSetDevice(a.device));
    cudaStream_t stream = a.stream;
    const double t0 = now_s();
    std::vector<int64_t> launches0;
    for (auto& s : sh) launches0.push_back(s->launches);
    const bool prof = opt.profile != 0 && !emulated();
    a.prof = prof;
    double kms[LFBA_NUM_KERNEL_TIMERS] = {0};
    int64_t kcalls[LFBA_NUM_KERNEL_TIMERS] = {0};
    cudaEvent_t e_run0, e_run1;
    LFBA_CUDA(cudaEventCreate(&e_run0));
    LFBA_CUDA(cudaEventCreate(&e_run1));
    LFBA_CUDA(cudaEventRecord(e_run0, stream));
    for (auto& s : sh) s->begin_run();
    // recalib: a round may be a line-search trial (no LM row); each iteration has at most 20 contractions + 1
    const int max_rounds = (opt.max_num_iterations + 8) * (a.d.recalib ? 22 : 1);
    int rounds = 0;
    for (; rounds < max_rounds; ++rounds) {
      for (auto& s : sh) s->phase_eval();
      reduce(0);
      for (auto& s : sh) s->phase_assemble();
      reduce(1);
      for (auto& s : sh) s->phase_solve();
      // The host runs ONE round ahead of the device: round r + 1 is enqueued before the `done` flag of round r is read,
      // so the stream never drains between rounds (every kernel early-outs on the device flag once the solve is over;
      // all ranks see the same flags, so they enqueue the same rounds and the NCCL calls stay matched).
      const int slot = rounds & 3;
      LFBA_CUDA(cudaMemcpyAsync(h_done + slot, &a.st.p->done, sizeof(int), cudaMemcpyDeviceToHost, stream));
      LFBA_CUDA(cudaEventRecord(ev_round[slot], stream));
      LFBA_CUDA(cudaGetLastError());  // launch-configuration errors do not surface in later memcpy / sync calls
      if (prof) {
        LFBA_CUDA(cudaStreamSynchronize(stream));
        const int order[] = {LFBA_T_LENS, LFBA_T_EVAL, LFBA_T_CONTROL, LFBA_T_SCHUR, LFBA_T_ALLREDUCE, LFBA_T_DAMP,
                             LFBA_T_CHOL, LFBA_T_POINTSTEP};
        cudaEvent_t prev = a.ev[LFBA_NUM_KERNEL_TIMERS];
        for (int k : order) {
          float ms = 0.f;
          cudaEventElapsedTime(&ms, prev, a.ev[k]);
          kms[k] += ms;
          kcalls[k] += 1;
          prev = a.ev[k];
        }
        if (h_done[slot]) {
          ++rounds;
          break;
        }
      } else if (rounds >= 1) {
        LFBA_CUDA(cudaEventSynchronize(ev_round[(rounds - 1) & 3]));
        if (h_done[(rounds - 1) & 3]) {
          ++rounds;
          break;
        }
      }
    }
    LFBA_CUDA(cudaEventRecord(e_run1, stream));
    for (auto& s : sh) LFBA_CUDA(cudaMemcpyAsync(&s->h_state, s->st.p, sizeof(LmState), cudaMemcpyDeviceToHost, s->stream));
    LFBA_CUDA(cudaStreamSynchronize(stream));
    LFBA_CUDA(cudaGetLastError());
    float run_ms = 0.f;
    cudaEventElapsedTime(&run_ms, e_run0, e_run1);
    cudaEventDestroy(e_run0);
    cudaEventDestroy(e_run1);
    LmState& hs = a.h_state;
    int status = hs.status;
    if (!hs.done) {  // safety net: the round budget ran out (cannot happen: max_iter is tested on device)
      hs.termination = LFBA_NO_CONVERGENCE;
      hs.stop_reason = LFBA_STOP_MAX_ITERATIONS;
    }
    if (sum) {
      lfba_iteration* rows = sum->iterations;
      const int cap = sum->iterations_capacity;
      std::memset(sum, 0, sizeof(*sum));
      sum->iterations = rows;
      sum->iterations_capacity = cap;
      sum->termination_type = hs.termination;
      sum->stop_reason = hs.stop_reason;
      sum->num_iterations = hs.n_rows;
      sum->num_successful_steps = hs.n_success;
      sum->num_unsuccessful_steps = hs.n_fail;
      sum->reduced_system_size = a.d.n;
      sum->final_cost = hs.x_cost;
      sum->num_jacobian_evals = hs.n_jac_evals;
      sum->num_observations = a.n_obs_global;
      sum->num_tracks = a.ix.T;
      sum->num_lenses = a.ix.NL;
      for (size_t r = 0; r < sh.size(); ++r) sum->gpu_launches += sh[r]->launches - launches0[r];
      sum->setup_time_s = a.setup_time;
      for (auto& q : sh) {
        sum->h2d_bytes += q->ix.h2d_bytes;
        sum->h2d_ms = std::max(sum->h2d_ms, q->ix.h2d_ms);
      }
      sum->solve_time_s = now_s() - t0;
      sum->solve_gpu_ms = run_ms;
      for (int k = 0; k < LFBA_NUM_KERNEL_TIMERS; ++k) {
        sum->kernel_ms[k] = kms[k];
        sum->kernel_calls[k] = kcalls[k];
      }
      const int nrows = std::min(hs.n_rows, kMaxLog);
      std::vector<lfba_iteration> hl((size_t)std::max(1, nrows));
      if (nrows > 0) a.log.download(hl.data(), nrows, stream);
      LFBA_CUDA(cudaStreamSynchronize(stream));
      if (nrows > 0) sum->initial_cost = hl[0].cost;
      if (rows)
        for (int i = 0; i < std::min(nrows, cap); ++i) rows[i] = hl[i];
      if (opt.minimizer_progress_to_stdout && rank == 0) {  // Ceres' progress table (SURVEY.md B.7)
        std::printf("iter      cost      cost_change  |gradient|   |step|    tr_ratio  tr_radius  ls_iter  iter_time  total_time\n");
        for (int i = 0; i < nrows; ++i)
          std::printf("% 4d % 8e   % 3.2e   % 3.2e  % 3.2e  % 3.2e % 3.2e     % 4d   % 3.2e   % 3.2e\n", hl[i].iteration,
                      hl[i].cost, hl[i].cost_change, hl[i].gradient_max_norm, hl[i].step_norm, hl[i].relative_decrease,
                      hl[i].trust_region_radius, 1, hl[i].iteration_time_s, hl[i].cumulative_time_s);
      }
    }
    return status;
  }
};

}  // namespace lfba

using namespace lfba;

struct lfba_solver {
  Group g;
};

template <class F>
static int guarded(F&& f) {
  try {
    return f();
  } catch (const CudaError& e) {
    set_error(e.what());
    return e.code;
  } catch (const std::exception& e) {
    set_error(e.what());
    return LFBA_CUDA_ERROR;
  }
}

extern "C" {

int lfba_version(void) { return LFBA_VERSION; }
const char* lfba_last_error(void) { return g_last_error.c_str(); }
const char* lfba_status_string(int s) {
  switch (s) {
    case LFBA_OK: return "ok";
    case LFBA_INVALID_ARGUMENT: return "invalid argument";
    case LFBA_NO_DEVICE: return "no usable CUDA device (no CPU fallback)";
    case LFBA_CUDA_ERROR: return "CUDA error";
    case LFBA_NCCL_ERROR: return "NCCL error";
    case LFBA_OUT_OF_MEMORY: return "out of device memory";
    case LFBA_FAILURE: return "solver failure";
    default: return "unknown";
  }
}
void lfba_options_init(lfba_options* o) {
  std::memset(o, 0, sizeof(*o));
  o->max_num_iterations = 200;    // src/CameraCalibration.cpp:960
  o->function_tolerance = 1e-6;   // :958
  o->parameter_tolerance = 1e-8;  // :959
  o->gradient_tolerance = 1e-10;  // Ceres default
  o->initial_trust_region_radius = 1e4;
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
  o->max_num_consecutive_invalid_steps = 5;
  o->loss_scale = 0.5;                   // ceres::CauchyLoss(0.5), :892
  o->minimizer_progress_to_stdout = 1;   // :957
  o->device = -1;
  o->num_gpus = 1;
  o->profile = 0;
  o->emulate_shards = 0;
}
int lfba_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major >= 10) ++ok;
  }
  return ok;
}
void lfba_trim_cache(void) { BlockCache::get().trim(); }
int lfba_comm_unique_id(char out[128]) {
  Nccl& n = Nccl::get();
  if (!n.ok) {
    set_error("libnccl.so.2 not found");
    return LFBA_NCCL_ERROR;
  }
  Nccl::UniqueId id;
  if (n.GetUniqueId(&id) != 0) return LFBA_NCCL_ERROR;
  std::memcpy(out, id.internal, 128);
  return LFBA_OK;
}

int lfba_comm_create(const lfba_comm* cm, void** handle) {
  if (!cm || !handle || cm->nranks < 1) return LFBA_INVALID_ARGUMENT;
  Nccl& n = Nccl::get();
  if (!n.ok) {
    set_error("libnccl.so.2 not found");
    return LFBA_NCCL_ERROR;
  }
  Nccl::UniqueId id;
  std::memcpy(id.internal, cm->nccl_unique_id, 128);
  Nccl::comm_t c = nullptr;
  const int rc = n.CommInitRank(&c, cm->nranks, id, cm->rank);
  if (rc != 0) {
    set_error(std::string("ncclCommInitRank: ") + n.GetErrorString(rc));
    return LFBA_NCCL_ERROR;
  }
  *handle = (void*)c;
  return LFBA_OK;
}
void lfba_comm_destroy(void* handle) {
  if (handle) Nccl::get().CommDestroy((Nccl::comm_t)handle);
}

int lfba_solver_create(const lfba_problem* pb, const lfba_options* opt, const lfba_comm* comm, lfba_solver** out) {
  if (!pb || !opt || !out) return LFBA_INVALID_ARGUMENT;
  *out = nullptr;
  lfba_solver* h = new lfba_solver();
  const int rc = guarded([&] {
    h->g.create(*pb, *opt, comm);
    return (int)LFBA_OK;
  });
  if (rc != LFBA_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return LFBA_OK;
}
int lfba_solver_set_parameters(lfba_solver* h, const double* c, const double* v, const double* p) {
  if (!h || !c || !v || !p) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    h->g.set_parameters(c, v, p);
    return (int)LFBA_OK;
  });
}
int lfba_solver_get_parameters(lfba_solver* h, double* c, double* v, double* p) {
  if (!h) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    h->g.get_parameters(c, v, p);
    return (int)LFBA_OK;
  });
}
int lfba_solver_run(lfba_solver* h, lfba_summary* sum) {
  if (!h) return LFBA_INVALID_ARGUMENT;
  return guarded([&] { return h->g.run(sum); });
}
void lfba_solver_destroy(lfba_solver* h) { delete h; }

int lfba_solver_time_eval(lfba_solver* h, int reps, int materialize, double* mean_ms) {
  if (!h || reps <= 0 || !mean_ms) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    Solver& s = h->g.s0();
    LFBA_CUDA(cudaSetDevice(s.device));
    alloc_stream() = s.stream;
    // evaluate at the accepted parameters: present them as the candidate of a fresh state
    LmState init;
    std::memset(&init, 0, sizeof(init));
    init.cur = 1 - s.h_state.cur;
    init.solve_ok = 1;
    LFBA_CUDA(cudaMemcpyAsync(s.st.p, &init, sizeof(LmState), cudaMemcpyHostToDevice, s.stream));
    cudaEvent_t e0, e1;
    LFBA_CUDA(cudaEventCreate(&e0));
    LFBA_CUDA(cudaEventCreate(&e1));
    DevBuf<double> res, jc, jv, jp, stats;
    EvalIn in{s.ix.obs_in.p, s.ix.lens_id_in.p, s.ix.point_in.p, s.ix.frame_in.p};
    EvalOut out{nullptr, nullptr, nullptr, nullptr, nullptr, 1.0, 0};
    if (materialize) {
      const int compact = materialize == 2 ? 1 : 0;  // 2: camera block as 2 x NC live columns (SURVEY.md 8(d) layout)
      res.alloc((size_t)2 * s.ix.N);
      jc.alloc((size_t)2 * (compact ? s.d.NC : 17) * s.ix.N);
      jv.alloc((size_t)12 * s.ix.N);
      jp.alloc((size_t)6 * s.ix.N);
      stats.alloc(8);
      stats.zero(s.stream);
      out = EvalOut{res.p, jc.p, jv.p, jp.p, stats.p, 1.0, compact};
    }
    const int which = s.h_state.cur;
    launch_tables(s.d, s.stream);
    if (materialize) launch_tables_for(s.d, which, s.stream);
    if (materialize) launch_eval_only(s.d, in, out, which, s.stream); else launch_eval(s.d, s.lanes, s.stream);
    LFBA_CUDA(cudaEventRecord(e0, s.stream));
    for (int r = 0; r < reps; ++r) {
      if (materialize) launch_eval_only(s.d, in, out, which, s.stream); else launch_eval(s.d, s.lanes, s.stream);
    }
    LFBA_CUDA(cudaEventRecord(e1, s.stream));
    LFBA_CUDA(cudaEventSynchronize(e1));
    LFBA_CUDA(cudaGetLastError());
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    s.launches += reps + 2;
    *mean_ms = ms / reps;
    return (int)LFBA_OK;
  });
}

int lfba_solver_track_blocks(lfba_solver* h, int64_t* n_tracks, int32_t* rec_stride_out, double* rec, double* camsum64,
                             int32_t* trk_point, int32_t* trk_frame) {
  if (!h) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    if (h->g.emulated()) throw CudaError("lfba_solver_track_blocks: single-shard sessions only", LFBA_INVALID_ARGUMENT);
    Solver& s = h->g.s0();
    LFBA_CUDA(cudaSetDevice(s.device));
    const int RS = rec_stride(s.d.NC);
    if (n_tracks) *n_tracks = s.ix.T;
    if (rec_stride_out) *rec_stride_out = RS;
    if (!rec && !camsum64 && !trk_point && !trk_frame) return (int)LFBA_OK;
    s.begin_run();  // fresh state: the caller's parameters are the candidate (buffer 1)
    launch_tables(s.d, s.stream);
    launch_eval(s.d, s.lanes, s.stream);
    launch_reduce_eval(s.d, s.stream);
    s.launches += 3;
    if (rec) s.rec[1].download(rec, (size_t)s.ix.T * RS, s.stream);
    if (camsum64) s.camsum[1].download(camsum64, 64, s.stream);
    if (trk_point) s.ix.trk_point.download(trk_point, s.ix.T, s.stream);
    if (trk_frame) s.ix.trk_frame.download(trk_frame, s.ix.T, s.stream);
    LFBA_CUDA(cudaStreamSynchronize(s.stream));
    LFBA_CUDA(cudaGetLastError());
    return (int)LFBA_OK;
  });
}

int lfba_solver_covariance(lfba_solver* h, double* cov_camera17, double* cov_poses, lfba_covariance_info* info) {
  if (!h) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    if (h->g.emulated() || h->g.nranks > 1)
      throw CudaError("lfba_solver_covariance: single-shard sessions only (the reduced system of a sharded session is "
                      "summed over its shards)", LFBA_INVALID_ARGUMENT);
    h->g.s0().covariance(cov_camera17, cov_poses, nullptr, info);
    return (int)LFBA_OK;
  });
}

int lfba_solver_covariance_points(lfba_solver* h, double* cov_camera17, double* cov_poses, double* cov_points,
                                  lfba_covariance_info* info) {
  if (!h || !cov_points) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    if (h->g.emulated() || h->g.nranks > 1)
      throw CudaError("lfba_solver_covariance_points: single-shard sessions only (the reduced system of a sharded "
                      "session is summed over its shards)", LFBA_INVALID_ARGUMENT);
    h->g.s0().covariance(cov_camera17, cov_poses, cov_points, info);
    return (int)LFBA_OK;
  });
}

int lfba_measure_fp64_peak(int device, double* tflops) {
  if (!tflops) return LFBA_INVALID_ARGUMENT;
  return guarded([&] {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) throw CudaError("no CUDA device", LFBA_NO_DEVICE);
    if (device >= 0) LFBA_CUDA(cudaSetDevice(device));
    *tflops = measure_fp64_tflops(0);
    return (int)LFBA_OK;
  });
}

int lfba_eval(const lfba_problem* pb, const lfba_options* opt_in, const double* cam, const double* views,
              const double* points, double* residuals, double* jac_camera, double* jac_view, double* jac_point,
              double* cost, lfba_reproj_stats* stats, double inlier_threshold) {
  if (!pb || !cam || !views || !points) return LFBA_INVALID_ARGUMENT;
  lfba_options o;
  if (opt_in) o = *opt_in; else lfba_options_init(&o);
  o.emulate_shards = 0;
  return guarded([&] {
    Group g;
    g.create(*pb, o, nullptr);
    g.set_parameters(cam, views, points);
    Solver& s = g.s0();
    alloc_stream() = s.stream;
    const int64_t N = s.ix.N;
    DevBuf<double> res((size_t)2 * N), jc, jv, jp, st(8);
    if (jac_camera) jc.alloc((size_t)34 * N);
    if (jac_view) jv.alloc((size_t)12 * N);
    if (jac_point) jp.alloc((size_t)6 * N);
    st.zero(s.stream);
    EvalIn in{s.ix.obs_in.p, s.ix.lens_id_in.p, s.ix.point_in.p, s.ix.frame_in.p};
    EvalOut out{res.p, jc.p, jv.p, jp.p, st.p, inlier_threshold * inlier_threshold, 0};
    launch_tables_for(s.d, 0, s.stream);
    launch_eval_only(s.d, in, out, 0, s.stream);
    LFBA_CUDA(cudaGetLastError());
    if (residuals) res.download(residuals, (size_t)2 * N, s.stream);
    if (jac_camera) jc.download(jac_camera, (size_t)34 * N, s.stream);
    if (jac_view) jv.download(jac_view, (size_t)12 * N, s.stream);
    if (jac_point) jp.download(jac_point, (size_t)6 * N, s.stream);
    double hs[8];
    st.download(hs, 8, s.stream);
    LFBA_CUDA(cudaStreamSynchronize(s.stream));
    if (cost) {
      double c = hs[5];
      for (int k = 0; k < s.d.K; ++k) {
        double r, j[3];
        distance_eval(points + 3 * pb->c_p1[k], points + 3 * pb->c_p2[k], pb->c_dist[k], pb->c_sigma[k], r, j);
        c += 0.5 * r * r;
      }
      *cost = c;
    }
    if (stats) {
      stats->std_x = N > 0 ? std::sqrt(hs[0] / (double)N) : 0.0;
      stats->std_y = N > 0 ? std::sqrt(hs[1] / (double)N) : 0.0;
      stats->mae_x = hs[2];
      stats->mae_y = hs[3];
      stats->num_points = N;
      stats->num_inliers = (int64_t)(hs[4] + 0.5);
    }
    return (int)LFBA_OK;
  });
}

int lfba_covariance(const lfba_problem* pb, const lfba_options* opt_in, const double* cam, const double* views,
                    const double* points, double* cov_camera17, double* cov_poses, lfba_covariance_info* info) {
  if (!pb || !cam || !views || !points) return LFBA_INVALID_ARGUMENT;
  lfba_options o;
  if (opt_in) o = *opt_in; else lfba_options_init(&o);
  o.emulate_shards = 0;
  return guarded([&] {
    Group g;
    g.create(*pb, o, nullptr);
    g.set_parameters(cam, views, points);
    g.s0().covariance(cov_camera17, cov_poses, nullptr, info);
    return (int)LFBA_OK;
  });
}

int lfba_covariance_points(const lfba_problem* pb, const lfba_options* opt_in, const double* cam, const double* views,
                           const double* points, double* cov_camera17, double* cov_poses, double* cov_points,
                           lfba_covariance_info* info) {
  if (!pb || !cam || !views || !points || !cov_points) return LFBA_INVALID_ARGUMENT;
  lfba_options o;
  if (opt_in) o = *opt_in; else lfba_options_init(&o);
  o.emulate_shards = 0;
  return guarded([&] {
    Group g;
    g.create(*pb, o, nullptr);
    g.set_parameters(cam, views, points);
    g.s0().covariance(cov_camera17, cov_poses, cov_points, info);
    return (int)LFBA_OK;
  });
}

// Single-process entry: one GPU, `emulate_shards` shards on one GPU, or `num_gpus` GPUs with one host thread per GPU.
int lfba_solve(const lfba_problem* pb, const lfba_options* opt_in, double* cam, double* views, double* points,
               lfba_summary* sum) {
  if (!pb || !cam || !views || !points) return LFBA_INVALID_ARGUMENT;
  lfba_options o;
  if (opt_in) o = *opt_in; else lfba_options_init(&o);
  const int G = std::max(1, o.num_gpus);
  if (G == 1) {
    return guarded([&] {
      Group g;
      g.create(*pb, o, nullptr);
      g.set_parameters(cam, views, points);
      const int rc = g.run(sum);
      if (rc == LFBA_OK || g.s0().h_state.n_rows > 0) g.get_parameters(cam, views, points);
      return rc;
    });
  }
  // ---- multi-GPU in one process: validate and shard first, then one host thread per GPU ----
  if (o.emulate_shards > 1) {
    set_error("emulate_shards cannot be combined with num_gpus > 1");
    return LFBA_INVALID_ARGUMENT;
  }
  const int avail = lfba_device_count();
  if (avail < G) {
    set_error("num_gpus exceeds the number of usable devices");
    return LFBA_NO_DEVICE;
  }
  HostShards hs;
  {
    const int rc = guarded([&] {
      hs.split(*pb, G);
      return (int)LFBA_OK;
    });
    if (rc != LFBA_OK) return rc;
  }
  const int P = pb->n_points;
  lfba_comm base;
  std::memset(&base, 0, sizeof(base));
  base.nranks = G;
  const int rc0 = lfba_comm_unique_id(base.nccl_unique_id);
  if (rc0 != LFBA_OK) return rc0;
  Nccl& nccl = Nccl::get();
  std::vector<int> rcs((size_t)G, LFBA_OK);
  std::vector<std::string> errs((size_t)G);
  std::vector<std::vector<double>> pts_out((size_t)G);
  std::vector<double> c17(17), v6((size_t)6 * pb->n_frames);
  std::vector<Nccl::comm_t> comms((size_t)G, nullptr);
  // pre-flight rendezvous: every rank finishes its non-collective set-up (device, memory, index) before ANY rank
  // enters NCCL; if one fails, nobody does (a rank stuck alone in ncclCommInitRank would never return)
  std::mutex mu;
  std::condition_variable cv;
  int arrived = 0, preflight_failed = 0;
  std::atomic<int> late_failure{0};
  std::vector<std::thread> th;
  for (int r = 0; r < G; ++r)
    th.emplace_back([&, r] {
      bool past_rendezvous = false;
      rcs[r] = guarded([&] {
        const lfba_problem lp = hs.view(*pb, r);
        lfba_options lo = o;
        lo.device = r;
        lo.emulate_shards = 0;
        Group g;
        g.opt = lo;
        g.rank = r;
        g.nranks = G;
        g.comm_aborted = &late_failure;
        g.sh.emplace_back(new Solver());
        int pre_rc = LFBA_OK;
        std::string pre_err;
        try {
          g.sh[0]->create_local(lp, lo, r, G, nullptr);
        } catch (const CudaError& e) {
          pre_rc = e.code;
          pre_err = e.what();
        } catch (const std::exception& e) {
          pre_rc = LFBA_CUDA_ERROR;
          pre_err = e.what();
        }
        bool any_failed;
        {
          std::unique_lock<std::mutex> lk(mu);
          if (pre_rc != LFBA_OK) ++preflight_failed;
          ++arrived;
          cv.notify_all();
          cv.wait(lk, [&] { return arrived == G; });
          any_failed = preflight_failed > 0;
        }
        past_rendezvous = true;
        if (pre_rc != LFBA_OK) throw CudaError(pre_err, pre_rc);
        if (any_failed) throw CudaError("another rank failed during set-up", LFBA_FAILURE);
        Nccl::UniqueId id;
        std::memcpy(id.internal, base.nccl_unique_id, 128);
        const int nrc = nccl.CommInitRank(&g.comm, G, id, r);
        if (nrc != 0) throw CudaError(std::string("ncclCommInitRank: ") + nccl.GetErrorString(nrc), LFBA_NCCL_ERROR);
        g.own_comm = true;
        comms[r] = g.comm;
        // the rest of Group::create for an already-indexed shard
        Solver& s = g.s0();
        const int F = s.ix.F;
        std::vector<int32_t> fa = s.h_fa;
        {
          alloc_stream() = s.stream;
          DevBuf<int32_t> dfa((size_t)F + 1);
          DevBuf<double> dn(1);
          double h_n = (double)s.ix.N;
          dfa.upload(fa.data(), (size_t)F + 1, s.stream);
          dn.upload(&h_n, 1, s.stream);
          g.nccl_allreduce(dfa.p, (size_t)F + 1, kNcclInt32, kNcclMax);
          g.nccl_allreduce(dn.p, 1, kNcclFloat64, kNcclSum);
          dfa.download(fa.data(), (size_t)F + 1, s.stream);
          dn.download(&h_n, 1, s.stream);
          LFBA_CUDA(cudaStreamSynchronize(s.stream));
          s.create_finish(fa, (int64_t)(h_n + 0.5));
        }
        g.h_done = Group::pinned_flags();
        for (auto& e : g.ev_round) LFBA_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        g.ev_made = true;
        g.set_parameters(cam, views, points);
        lfba_summary local;
        std::memset(&local, 0, sizeof(local));
        lfba_summary* ps = (r == 0) ? sum : &local;
        const int rc = g.run(ps);
        pts_out[r].resize((size_t)3 * P);
        if (r == 0) g.get_parameters(c17.data(), v6.data(), pts_out[r].data());
        else g.get_parameters(nullptr, nullptr, pts_out[r].data());
        comms[r] = nullptr;
        return rc;
      });
      errs[r] = g_last_error;
      if (rcs[r] != LFBA_OK) {
        if (!past_rendezvous) {  // failed before the rendezvous (e.g. while sharding views): still let the others pass it
          std::unique_lock<std::mutex> lk(mu);
          ++preflight_failed;
          ++arrived;
          cv.notify_all();
        } else if (late_failure.exchange(1) == 0 && nccl.CommAbort) {
          // a rank died after NCCL was up: abort the peers' communicators so that they do not wait in a collective forever
          for (int q = 0; q < G; ++q)
            if (q != r && comms[q]) nccl.CommAbort(comms[q]);
        }
      }
    });
  for (auto& t : th) t.join();
  for (int r = 0; r < G; ++r)
    if (rcs[r] != LFBA_OK) {
      set_error("rank " + std::to_string(r) + ": " + errs[r]);
      return rcs[r];
    }
  // all ranks succeeded: only now touch the caller's arrays
  std::memcpy(cam, c17.data(), 17 * sizeof(double));
  std::memcpy(views, v6.data(), v6.size() * sizeof(double));
  for (int p = 0; p < P; ++p)
    for (int j = 0; j < 3; ++j) points[3 * (size_t)p + j] = pts_out[(size_t)hs.owner[p]][3 * (size_t)p + j];
  return LFBA_OK;
}

}  // extern "C"
