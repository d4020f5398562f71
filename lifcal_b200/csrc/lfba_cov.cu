// lfba_cov.cu — covariance of camera and poses from the factorised reduced system (lfba_solver_covariance).
//
// With S = L L^T the undamped, Schur-reduced Gauss-Newton matrix [poses | coupled points | camera], Sigma = S^-1 is the
// marginal covariance of those parameters (ceres::Covariance semantics: not multiplied by sigma^2). Only blocks inside
// the envelope of L are wanted, and those are exactly what the selected inversion (Takahashi / Erisman-Tinney) computes
// from L alone, block column by block column from the last one: with J a block column of L and R the rows below J in
// its envelope,
//     Y        = L_RJ L_JJ^-1
//     Sigma_RJ = -Sigma_RR Y
//     Sigma_JJ = L_JJ^-T L_JJ^-1 - Sigma_RJ^T Y
// Sigma_RR lies inside the envelope (a row of R starts at or before J) and was finished by the later block columns.
// Blocks are the dense border one column at a time, then the 6 x 6 pose blocks; the chain is F + border steps, each
// O(|R|^2 * 6) with |R| <= 6 bw + border. One CTA, Y in shared memory, Sigma written to a second skyline buffer.
#include "lfba_device.cuh"
#include "lfba_kernels.h"
#include "lfba_setup.cuh"

namespace lfba {

constexpr int kSelinvThreads = 512;
constexpr int kSelinvSmemMax = 200 * 1024;

__device__ __forceinline__ long long sky_off(const SkyMap& m, int r, int c) {  // entry (r, c), c <= r, of the envelope
  if (r < m.np6) {
    const int f = r / 6;
    return m.row(f, r - 6 * f) + (c - m.c0(f));
  }
  return m.border_row(r - m.np6) + c;
}
__device__ __forceinline__ double sym_at(const double* Z, const SkyMap& m, int r, int c) {
  return r >= c ? Z[sky_off(m, r, c)] : Z[sky_off(m, c, r)];
}
__device__ __forceinline__ double warp_sum_cov(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One block column [j0, j0 + B) with npr pose rows [j0 + B, j0 + B + npr) and the border rows [bstart, n) below it.
template <int B>
__device__ void selinv_block(const double* __restrict__ L, double* __restrict__ Z, const SkyMap& sky, int n, int j0,
                             int npr, int bstart, double* Y, double* Li) {
  const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
  const int m = npr + (n - bstart);
  auto ridx = [&](int q) { return q < npr ? j0 + B + q : bstart + (q - npr); };
  // Y = L_RJ L_JJ^-1, row by row (y L_JJ = l, L_JJ lower); L_JJ^-1 by one thread
  for (int q = tid; q < m; q += nt) {
    const int r = ridx(q);
    double y[B];
#pragma unroll
    for (int c = B - 1; c >= 0; --c) {
      double v = L[sky_off(sky, r, j0 + c)];
#pragma unroll
      for (int c2 = c + 1; c2 < B; ++c2) v -= y[c2] * L[sky_off(sky, j0 + c2, j0 + c)];
      y[c] = v / L[sky_off(sky, j0 + c, j0 + c)];
    }
#pragma unroll
    for (int c = 0; c < B; ++c) Y[q * B + c] = y[c];
  }
  if (tid == nt - 1) {
    for (int c = 0; c < B; ++c) {
      Li[c * B + c] = 1.0 / L[sky_off(sky, j0 + c, j0 + c)];
      for (int i = c + 1; i < B; ++i) {
        double v = 0.0;
        for (int k = c; k < i; ++k) v += L[sky_off(sky, j0 + i, j0 + k)] * Li[k * B + c];
        Li[i * B + c] = -v / L[sky_off(sky, j0 + i, j0 + i)];
      }
    }
  }
  __syncthreads();
  // Sigma_RJ = -Sigma_RR Y: a warp per row of R, lanes over the columns of Sigma_RR
  for (int q = warp; q < m; q += nw) {
    const int r = ridx(q);
    double acc[B];
#pragma unroll
    for (int c = 0; c < B; ++c) acc[c] = 0.0;
    for (int q2 = lane; q2 < m; q2 += 32) {
      const double s = sym_at(Z, sky, r, ridx(q2));
#pragma unroll
      for (int c = 0; c < B; ++c) acc[c] += s * Y[q2 * B + c];
    }
#pragma unroll
    for (int c = 0; c < B; ++c) acc[c] = warp_sum_cov(acc[c]);
    if (lane == 0)
#pragma unroll
      for (int c = 0; c < B; ++c) Z[sky_off(sky, r, j0 + c)] = -acc[c];
  }
  __syncthreads();
  // Sigma_JJ = L_JJ^-T L_JJ^-1 - Sigma_RJ^T Y: a warp per entry of the lower triangle
  for (int e = warp; e < B * (B + 1) / 2; e += nw) {
    int c1 = 0, c2 = e;
    while (c2 > c1) { c2 -= c1 + 1; ++c1; }
    double acc = 0.0;
    for (int q = lane; q < m; q += 32) acc += Z[sky_off(sky, ridx(q), j0 + c1)] * Y[q * B + c2];
    acc = warp_sum_cov(acc);
    if (lane == 0) {
      double v = 0.0;
      for (int k = c1; k < B; ++k) v += Li[k * B + c1] * Li[k * B + c2];
      Z[sky_off(sky, j0 + c1, j0 + c2)] = v - acc;
    }
  }
  __syncthreads();
}

// Y: dynamic shared memory when it fits (use_smem), else the global scratch Yg; both [6 (6 bw + border)] doubles.
__global__ void __launch_bounds__(kSelinvThreads) k_selinv(Dev d, double* __restrict__ Z, double* Yg, int use_smem) {
  if (!d.st->solve_ok) return;
  extern __shared__ double sm_y[];
  __shared__ double Li[36];
  double* Y = use_smem ? sm_y : Yg;
  const SkyMap sky{d.band, d.np6};
  const int n = d.n, np6 = d.np6, F = np6 / 6;
  for (int j = n - 1; j >= np6; --j) selinv_block<1>(d.S, Z, sky, n, j, 0, j + 1, Y, Li);
  for (int f = F - 1; f >= 0; --f) {
    const int pend = 6 * min(F, f + d.band + 1);
    selinv_block<6>(d.S, Z, sky, n, 6 * f, pend - 6 * (f + 1), np6, Y, Li);
  }
}

// out[0, 289): camera block in the 17 x 17 layout (zero where a parameter is not in the reduced system);
// out[289, 289 + 36 F): 6 x 6 pose blocks (zero for held or unobserved frames, and when poses are not refined).
__global__ void k_cov_gather(Dev d, const double* __restrict__ Z, double* __restrict__ out) {
  const SkyMap sky{d.band, d.np6};
  const int total = 289 + 36 * d.F;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    double v = 0.0;
    if (!d.st->solve_ok) {
    } else if (e < 289) {
      const int c1 = e / 17, c2 = e % 17;
      if (c1 < d.NC && c2 < d.NC && d.cam_red[c1] >= 0 && d.cam_red[c2] >= 0) v = sym_at(Z, sky, d.cam_red[c1], d.cam_red[c2]);
    } else {
      const int f = (e - 289) / 36, i = (e - 289) % 36 / 6, j = (e - 289) % 6;
      if (d.np6 > 0 && d.frm_active[f] && f != d.gauge_frame) v = sym_at(Z, sky, 6 * f + i, 6 * f + j);
    }
    out[e] = v;
  }
}

static size_t selinv_y_doubles(const Dev& d) { return 6 * (size_t)(6 * d.band + (d.n - d.np6) + 1); }

void prepare_cov_kernels() {
  cudaFuncSetAttribute(k_selinv, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelinvSmemMax);
}

int launch_covariance(const Dev& d, double* Z, double* out, cudaStream_t s) {
  const size_t ny = selinv_y_doubles(d);
  const bool use_smem = ny * sizeof(double) <= (size_t)kSelinvSmemMax;
  alloc_stream() = s;
  DevBuf<double> Yg(use_smem ? 0 : ny);
  k_selinv<<<1, kSelinvThreads, use_smem ? ny * sizeof(double) : 0, s>>>(d, Z, Yg.p, use_smem ? 1 : 0);
  const int total = 289 + 36 * d.F;
  k_cov_gather<<<(total + 255) / 256, 256, 0, s>>>(d, Z, out);
  return 2;
}

}  // namespace lfba
