// lfba_chol.cu — FP64 Cholesky of the reduced camera system on its skyline (envelope) storage.
//
// Replaces Ceres' DenseSchurComplementSolver::SolveReducedLinearSystem (Eigen LLT of the dense
// (17+6F)^2 matrix, SURVEY.md B.4). The reduced system is ordered [poses | coupled points | camera | rhs],
// so with windowed visibility it is block-banded with a dense border (an arrowhead): Cholesky fills only
// inside the envelope, which is exactly what is stored. The right-hand side is kept as one extra matrix row:
// the factorisation leaves L^-1 g in it (forward substitution for free).
//
// Tiled left-looking factorisation, 64x64 tiles, one launch per tile column, one CTA per structurally
// non-zero tile of the column: A_ik -= sum_j L_ij L_kj^T (FP64 FMA, 4x4 register micro-tiles), POTRF of the
// diagonal tile (recomputed by every CTA of the column: no inter-CTA dependency inside a launch), TRSM.
// tcgen05 has no FP64 kind and the tiles are tiny, so this is plain DFMA work; the chain of n pivots is the
// latency that matters, not the flops.
#include <cstdio>

#include "lfba_band.cuh"
#include "lfba_device.cuh"
#include "lfba_kernels.h"

namespace lfba {

constexpr int TS = kTile;      // 64
constexpr int LD = TS + 1;     // padded leading dimension in shared memory
constexpr int kBandedSmemMax = 220 * 1024;

__device__ __forceinline__ double sky_load(const Dev& d, int r, int c, int n_aug) {
  if (r >= n_aug || c > r) return 0.0;
  if (r == d.n && c == d.n) return 0.0;
  const int c0 = d.row_c0[r];
  if (c < c0) return 0.0;
  return d.S[d.row_off[r] + (c - c0)];
}
__device__ __forceinline__ void sky_store(const Dev& d, int r, int c, int n_aug, double v) {
  if (r >= n_aug || c > r) return;
  if (r == d.n && c == d.n) return;
  const int c0 = d.row_c0[r];
  if (c < c0) return;
  d.S[d.row_off[r] + (c - c0)] = v;
}

// load tile (ti, tj) into smem [TS][LD]
__device__ __forceinline__ void load_tile(const Dev& d, int ti, int tj, int n_aug, double* sm) {
  for (int e = threadIdx.x; e < TS * TS; e += blockDim.x) {
    const int r = e / TS, c = e % TS;
    sm[r * LD + c] = sky_load(d, ti * TS + r, tj * TS + c, n_aug);
  }
}

// One tile column k. grid.x = number of tile rows i >= k; blockIdx.x = i - k.
__global__ void __launch_bounds__(256) k_chol_column(Dev d, int k, const int* __restrict__ tile_first) {
  LmState* st = d.st;
  if (linear_phase_idle(st) || !st->solve_ok) return;
  const int i = k + blockIdx.x;
  const int n_aug = d.n + 1;
  if (tile_first[i] > k) return;  // structurally zero tile
  extern __shared__ double sm[];
  double* sA = sm;                 // L_ij  / later A_ik
  double* sB = sm + TS * LD;       // L_kj
  double* sD = sm + 2 * TS * LD;   // diagonal tile
  __shared__ int s_fail;
  if (threadIdx.x == 0) s_fail = 0;

  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;  // 16x16 threads, 4x4 micro-tile each
  double acc[16], accd[16];
#pragma unroll
  for (int e = 0; e < 16; ++e) acc[e] = accd[e] = 0.0;

  const int jk = tile_first[k];
  const int ji = tile_first[i] > jk ? tile_first[i] : jk;
  for (int j = jk; j < k; ++j) {
    __syncthreads();
    load_tile(d, k, j, n_aug, sB);
    const bool both = (j >= ji) && (i != k);
    if (both) load_tile(d, i, j, n_aug, sA);
    __syncthreads();
#pragma unroll 4
    for (int t = 0; t < TS; ++t) {
      double b[4], bk[4], a[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        b[q] = sB[(tx * 4 + q) * LD + t];   // column index of the output (row of L_kj)
        bk[q] = sB[(ty * 4 + q) * LD + t];  // row index of the diagonal output
      }
#pragma unroll
      for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = 0; q < 4; ++q) accd[p * 4 + q] += bk[p] * b[q];
      if (both) {
#pragma unroll
        for (int p = 0; p < 4; ++p) a[p] = sA[(ty * 4 + p) * LD + t];
#pragma unroll
        for (int p = 0; p < 4; ++p)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[p * 4 + q] += a[p] * b[q];
      }
    }
  }
  __syncthreads();
  // D = A_kk - accd ; A = A_ik - acc
  load_tile(d, k, k, n_aug, sD);
  if (i != k) load_tile(d, i, k, n_aug, sA);
  __syncthreads();
#pragma unroll
  for (int p = 0; p < 4; ++p)
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int r = ty * 4 + p, c = tx * 4 + q;
      sD[r * LD + c] -= accd[p * 4 + q];
      if (i != k) sA[r * LD + c] -= acc[p * 4 + q];
    }
  __syncthreads();

  // POTRF of the diagonal tile (lower). Columns >= n (the rhs row and padding) are not pivots.
  const int nreal = min(TS, d.n - k * TS);
  for (int c = 0; c < nreal; ++c) {
    __syncthreads();  // trailing update of the previous column is complete
    const double piv = sD[c * LD + c];
    if (!(piv > 0.0)) {
      if (threadIdx.x == 0) s_fail = 1;
    }
    const double dinv = piv > 0.0 ? rsqrt(piv) : 0.0;
    __syncthreads();
    if (threadIdx.x < TS) {
      const int r = threadIdx.x;
      if (r == c) sD[c * LD + c] = piv > 0.0 ? sqrt(piv) : 1.0;
      else if (r > c) sD[r * LD + c] *= dinv;
    }
    __syncthreads();
    // trailing update of the lower triangle: (r, c2), c < c2 <= r
    const int m = TS - 1 - c;  // rows c+1..TS-1
    for (int e = threadIdx.x; e < m * m; e += blockDim.x) {
      const int r = c + 1 + e / m, c2 = c + 1 + e % m;
      if (c2 <= r) sD[r * LD + c2] -= sD[r * LD + c] * sD[c2 * LD + c];
    }
  }
  __syncthreads();
  if (i == k) {
    for (int e = threadIdx.x; e < TS * TS; e += blockDim.x) {
      const int r = e / TS, c = e % TS;
      if (c <= r && c < nreal) sky_store(d, k * TS + r, k * TS + c, n_aug, sD[r * LD + c]);
    }
    if (threadIdx.x == 0 && s_fail) st->solve_ok = 0;
    return;
  }
  // TRSM: X L_kk^T = A  (column by column)
  for (int c = 0; c < nreal; ++c) {
    const double dinv = 1.0 / sD[c * LD + c];
    if (threadIdx.x < TS) sA[threadIdx.x * LD + c] *= dinv;
    __syncthreads();
    const int m = TS - 1 - c;
    for (int e = threadIdx.x; e < TS * m; e += blockDim.x) {
      const int r = e / m, c2 = c + 1 + e % m;
      sA[r * LD + c2] -= sA[r * LD + c] * sD[c2 * LD + c];
    }
    __syncthreads();
  }
  for (int e = threadIdx.x; e < TS * TS; e += blockDim.x) {
    const int r = e / TS, c = e % TS;
    if (c < nreal) sky_store(d, i * TS + r, k * TS + c, n_aug, sA[r * LD + c]);
  }
}

// Backward substitution L^T y = z with z = the factorised rhs row. One CTA; right-looking over the rows of L
// so that every access is a contiguous skyline row.
__global__ void __launch_bounds__(256) k_backsolve(Dev d) {
  LmState* st = d.st;
  if (linear_phase_idle(st) || !st->solve_ok) return;
  const int n = d.n;
  double* y = d.y;
  const double* zrow = d.S + d.row_off[n];
  for (int j = threadIdx.x; j < n; j += blockDim.x) y[j] = zrow[j];
  __shared__ double yc;
  __syncthreads();
  for (int c = n - 1; c >= 0; --c) {
    const int c0 = d.row_c0[c];
    const double* Lr = d.S + d.row_off[c];
    if (threadIdx.x == 0) {
      const double v = y[c] / Lr[c - c0];
      y[c] = v;
      yc = v;
    }
    __syncthreads();
    const double v = yc;
    for (int j = c0 + threadIdx.x; j < c; j += blockDim.x) y[j] -= Lr[j - c0] * v;
    __syncthreads();
  }
}


// ------------------------------------------------------------------------------------------------
// Banded-arrowhead Cholesky, one CTA, everything on chip.
//
// With windowed visibility the reduced system is [block-banded pose part | dense border], border =
// coupled points + camera + the rhs row. A right-looking factorisation by 6x6 pose blocks only ever touches the
// (bw+1) frames of the current window plus the border: that window (6(bw+1)+nb)^2 lives in shared memory as a
// circular buffer of frame slots, finished columns of L stream back to HBM once, and the chain of F block pivots
// runs without a single kernel launch or global synchronisation. The rhs row rides along as a border row
// (forward substitution for free); the backward substitution is done by the same CTA, block by block.
// Cost: O(F * (6 bw + nb)^2 * 6) flops instead of n^3/3; latency ~1 us per frame instead of ~150 us per 64-tile.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int bslot(int f, int bw1) { return 6 * (f % bw1); }

__global__ void __launch_bounds__(kBandThreads) k_chol_banded(Dev d, int bw, int nb) {
  LmState* st = d.st;
  if (linear_phase_idle(st) || !st->solve_ok) return;
  extern __shared__ __align__(16) double sm[];
  const int F = d.np6 / 6;
  const int bw1 = bw + 1;
  const int NBAND = 6 * bw1;
  const BandGeom geo(bw, nb);
  const int LDW = geo.LDW;
  double* A = sm;                                                   // window + X + L_kk (band_sweep's layout)
  double* ys = sm + geo.doubles();                                  // n
  double* dinv_all = ys + d.n;                                      // n: 1 / L_cc of the pose pivots
  __shared__ double tvec[6];
  __shared__ double Lkk[21];
  __shared__ int s_fail;
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int npiv = nb - 1;  // border unknowns (the last border row is the rhs)

  if (tid == 0) s_fail = 0;
  const SkyMap sky{bw, d.np6};  // closed-form skyline offsets: no index loads on the chain
  BandArgs g{d.S, d.row_off, d.np6, bw, 0, F, F - 1, 0, 0, nb, nullptr, dinv_all, d.debug};
  band_load_initial(g, A);  // zeroes the window, loads the first bw + 1 frames; ends with a barrier
  for (int e = tid; e < nb * nb; e += nt) {
    const int b1 = e / nb, b2 = e % nb;
    if (b2 <= b1 && !(b1 == npiv && b2 == npiv)) A[(NBAND + b1) * LDW + NBAND + b2] = d.S[sky.border_row(b1) + d.np6 + b2];
  }
  __syncthreads();
#define CHOL_TICK(i)
  band_sweep(g, A, &s_fail);
  CHOL_TICK(5)
  // ---- dense Cholesky of the border block (coupled points + camera); the rhs row is not a pivot ----
  for (int c = 0; c < npiv; ++c) {
    __syncthreads();
    const double piv = A[(NBAND + c) * LDW + NBAND + c];
    const bool okp = piv > 0.0;
    const double r = okp ? rsqrt(piv) : 0.0;
    __syncthreads();
    if (tid == 0) {
      if (!okp) s_fail = 1;
      A[(NBAND + c) * LDW + NBAND + c] = okp ? piv * r : 1.0;
    } else if (tid < nb - c) {
      A[(NBAND + c + tid) * LDW + NBAND + c] *= r;
    }
    __syncthreads();
    const int m = nb - 1 - c;
    for (int e = tid; e < m * m; e += nt) {
      const int i = c + 1 + e / m, j = c + 1 + e % m;
      if (j <= i) A[(NBAND + i) * LDW + NBAND + j] -= A[(NBAND + i) * LDW + NBAND + c] * A[(NBAND + j) * LDW + NBAND + c];
    }
  }
  __syncthreads();
  for (int e = tid; e < nb * nb; e += nt) {
    const int b1 = e / nb, b2 = e % nb;
    if (b2 <= b1 && !(b1 == npiv && b2 == npiv)) d.S[sky.border_row(b1) + d.np6 + b2] = A[(NBAND + b1) * LDW + NBAND + b2];
  }
  if (tid == 0 && s_fail) st->solve_ok = 0;
  if (s_fail) return;
  CHOL_TICK(6)
  // ---- backward substitution L^T y = z, z = the factorised rhs row ----
  if (tid == 0) {
    for (int b = npiv - 1; b >= 0; --b) {
      double v = A[(NBAND + npiv) * LDW + NBAND + b];
      for (int b2 = b + 1; b2 < npiv; ++b2) v -= A[(NBAND + b2) * LDW + NBAND + b] * ys[d.np6 + b2];
      ys[d.np6 + b] = v / A[(NBAND + b) * LDW + NBAND + b];
    }
  }
  __syncthreads();
  const double* zrow = d.S + sky.border_row(npiv);
  // software pipeline: the L entries of block column k-1 are loaded while block k is being solved
  const int per = 8;  // entries per lane per output column: mrows <= 32 * per is checked on the host
  double lv[per];
  double lkk = 0.0, zk = 0.0;
  auto fetch_col = [&](int k) {
    const int nbf = min(bw, F - 1 - k);
    const int mrows = 6 * nbf + npiv;
    if (warp < 6) {
#pragma unroll
      for (int q = 0; q < per; ++q) {
        const int i = lane + 32 * q;
        lv[q] = 0.0;
        if (i < mrows) {
          const long long off = i < 6 * nbf ? sky.row(k + 1 + i / 6, i % 6) + (6 * k + warp - sky.c0(k + 1 + i / 6))
                                            : sky.border_row(i - 6 * nbf) + 6 * k + warp;
          lv[q] = d.S[off];
        }
      }
      if (lane == 0) zk = zrow[6 * k + warp];
    } else if (warp == 6 && lane < 21) {
      int i = 0, j = lane;
      while (j > i) { j -= i + 1; ++i; }
      lkk = d.S[sky.row(k, i) + (6 * k + j - sky.c0(k))];
    }
  };
  if (F > 0) fetch_col(F - 1);
  for (int k = F - 1; k >= 0; --k) {
    const int nbf = min(bw, F - 1 - k);
    const int mrows = 6 * nbf + npiv;
    if (warp < 6) {
      double acc = 0.0;
#pragma unroll
      for (int q = 0; q < per; ++q) {
        const int i = lane + 32 * q;
        if (i < mrows) acc += lv[q] * ys[i < 6 * nbf ? 6 * (k + 1) + i : d.np6 + (i - 6 * nbf)];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) tvec[warp] = zk - acc;
    } else if (warp == 6 && lane < 21) {
      Lkk[lane] = lkk;
    }
    if (k > 0) fetch_col(k - 1);
    __syncthreads();
    if (tid == 0) {
      double yk[6];
#pragma unroll
      for (int c = 5; c >= 0; --c) {
        double v = tvec[c];
#pragma unroll
        for (int c2 = 5; c2 > c; --c2) v -= Lkk[c2 * (c2 + 1) / 2 + c] * yk[c2];
        yk[c] = v * dinv_all[6 * k + c];
        ys[6 * k + c] = yk[c];
      }
    }
    __syncthreads();
  }
  CHOL_TICK(7)
  for (int j = tid; j < d.n; j += nt) d.y[j] = ys[j];
}

// per-device opt-in to > 48 KB of dynamic shared memory (call once per device with that device current)
void prepare_device_kernels() {
  cudaFuncSetAttribute(k_chol_column, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(3 * TS * LD * sizeof(double)));
  cudaFuncSetAttribute(k_chol_banded, cudaFuncAttributeMaxDynamicSharedMemorySize, kBandedSmemMax);
}

// shared memory needed by k_chol_banded, or 0 when the banded path does not apply / does not fit
size_t banded_smem_bytes(const Dev& d, int bw, int nb) {
  if (d.np6 == 0) return 0;
  const BandGeom geo(bw, nb);
  if (6 * geo.W > kBandPref * 480 || geo.W > 160) return 0;   // prefetch registers / panel rows of band_sweep
  if (6 * (size_t)bw + nb > 32 * 8) return 0;                 // backward-substitution lanes
  const size_t bytes = (geo.doubles() + 2 * (size_t)d.n + 8) * sizeof(double);
  return bytes <= (size_t)kBandedSmemMax ? bytes : 0;
}

void launch_chol_banded(const Dev& d, int bw, int nb, size_t smem, cudaStream_t s) {
  k_chol_banded<<<1, kBandThreads, smem, s>>>(d, bw, nb);
}

int launch_reduced_solve(const Dev& d, int n_tiles, const int* d_tile_first, int bw, cudaStream_t s, PartPlan* plan) {
  if (part_plan_active(plan)) return launch_part_solve(d, plan, s);
  return launch_chol_inplace(d, n_tiles, d_tile_first, bw, s);
}

int launch_chol_inplace(const Dev& d, int n_tiles, const int* d_tile_first, int bw, cudaStream_t s) {
  const int nb = d.n - d.np6 + 1;
  const size_t bsm = banded_smem_bytes(d, bw, nb);
  if (bsm > 0) {
    launch_chol_banded(d, bw, nb, bsm, s);
    return 1;
  }
  const size_t smem = 3 * TS * LD * sizeof(double);
  for (int k = 0; k < n_tiles; ++k) k_chol_column<<<n_tiles - k, 256, smem, s>>>(d, k, d_tile_first);
  k_backsolve<<<1, 256, 0, s>>>(d);
  return n_tiles + 1;
}

// ------------------------------------------------------------------------------------------------
// FP64 FMA throughput micro-benchmark (the roofline denominator for the FP64-pipe-bound fused kernel;
// MEASURED_PEAKS.json has no FP64 figure).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_dfma_peak(double* out, int iters) {
  double a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
  const double b = 1.0000001, c = 1e-9;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) a[i] = fma(a[i], b, c);
  }
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += a[i];
  if (s == 123.456) out[0] = s;
}

double measure_fp64_tflops(cudaStream_t s) {
  int dev = 0, sms = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  double* out = nullptr;
  cudaMalloc(&out, 8);
  const int iters = 4096, grid = sms * 8, block = 256;
  k_dfma_peak<<<grid, block, 0, s>>>(out, 64);
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0, s);
    k_dfma_peak<<<grid, block, 0, s>>>(out, iters);
    cudaEventRecord(e1, s);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 64.0 * (double)iters * (double)grid * (double)block;
    const double tf = flops / (ms * 1e-3) / 1e12;
    if (tf > best) best = tf;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(out);
  return best;
}

}  // namespace lfba
