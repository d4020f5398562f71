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

// Per-point 3 x 3 blocks. An eliminated point p (pdata written by the undamped k_points) has, with Hi = Hpp^-1 and u the
// point's n x 3 coupling column of J^T W J (V_t^T of its tracks in pose rows, Hcp in camera rows),
//     Sigma_pp = Hi + Hi Q Hi,   Q = u^T Z u
// (block inverse of [[S, u], [u^T, Hpp]]). With w = u Hi (W_t = V_t Hi = M_t^T (B_t Hi) in pose rows, T_p^T = Hcp Hi in
// camera rows: the point record holds T_p), Hi Q Hi = w^T Z w =: Q~, and
//     Q~ = sum_{a,b} W_a^T Z[f_a, f_b] W_b + (N + N^T) + T_p Z[cam, cam] T_p^T,   N = sum_a W_a^T Z[f_a, cam] T_p^T.
// Q~ is symmetric, so it is its own symmetric part sym(X) = (X + X^T) / 2, and sym(W_a^T Z_ab W_b) = sym(W_b^T Z_ba W_a):
// with one track per (point, frame),
//     Q~ = sym( sum_a W_a^T y_a ) + T_p Z[cam, cam] T_p^T,   y_a = Z[f_a, f_a] W_a + 2 (sum_{f_b < f_a} Z[f_a, f_b] W_b + Z[f_a, cam] T_p^T)
// and Sigma_pp = Hi + sym(Q~). This reads only lower blocks of Z (row f_a, columns 6 f_b .. contiguous) and does half the
// pairs, 108 FMA each. Tracks in the gauge frame are skipped: that pose is not a parameter, and Z holds identity on its
// rows. Frames of one point are at most `band` apart, so every Z[f_a, f_b] lies in the envelope. A coupled point's block is its diagonal block of Z. One
// thread per point.
template <int NC>
__global__ void __launch_bounds__(128) k_cov_points(Dev d, const double* __restrict__ Z, double* __restrict__ out) {
  const SkyMap sky{d.band, d.np6};
  const int cur = d.st->cur;
  const double* __restrict__ recs = d.rec[cur];
  const double* __restrict__ frames = d.frames[cur];
  for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < d.P; p += gridDim.x * blockDim.x) {
    double Sg[6] = {0, 0, 0, 0, 0, 0};  // lower triangle: 00 10 11 20 21 22
    const int cp = d.refine_points && d.st->solve_ok && d.pt_active[p] ? d.pt_coupled[p] : -2;
    if (cp >= 0) {
      const int r0 = d.np6 + 3 * cp;
#pragma unroll
      for (int i = 0, h = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j, ++h) Sg[h] = Z[sky_off(sky, r0 + i, r0 + j)];
    } else if (cp == -1) {
      const double* __restrict__ pd = d.pdata + (size_t)p * kPointStride;
      const double* __restrict__ Tp = pd + 12;  // T_p[j][c] at 3 c + j; columns with cam_red[c] < 0 are skipped
      double Q[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
      if (d.refine_poses) {
        const int t0 = d.pt_trk_begin[p], t1 = d.pt_trk_begin[p + 1];
        // W of track t (frame f) = M^T (B Hi), from the helpers the assembly uses
        const double* X = d.points[cur] + 3 * (size_t)p;
        const double Xp[3] = {X[0], X[1], X[2]};
        auto track_W = [&](int t, int f, double W[18]) {
          double A[6], m[9], B[9], K[9], Hi[6];
          const double* fe = frames + (size_t)f * kFrameStride;
          load_record<6, false>(recs + (size_t)t * rec_stride(NC), A);
          track_m(fe, Xp, m);
          track_b(A, fe, B);
          load_record<6, false>(pd, Hi);
          mat3_sym3(B, Hi, K);
          mt_mat(m, K, W);
        };
        for (int a = t0; a < t1; ++a) {
          const int fa = d.trk_frame[a];
          if (fa == d.gauge_frame) continue;
          const long long za = sky.row(fa, 0) - sky.c0(fa);  // + offset of row i + column: entry (6 fa + i, column)
          const int len0 = 6 * fa - sky.c0(fa) + 1;
          auto zrow = [&](int i) { return za + (long long)i * len0 + (i * (i - 1)) / 2; };
          double y[18];
#pragma unroll
          for (int k = 0; k < 18; ++k) y[k] = 0.0;
          // pose-camera (camera rows are border rows: Z[r, 6 fa + i] is contiguous in i)
#pragma unroll
          for (int c = 0; c < NC; ++c) {
            const int r = d.cam_red[c];
            if (r < 0) continue;
            const double* zr = Z + sky.border_row(r - d.np6) + 6 * fa;
            const double h0 = Tp[3 * c], h1 = Tp[3 * c + 1], h2 = Tp[3 * c + 2];
#pragma unroll
            for (int i = 0; i < 6; ++i) {
              const double z = zr[i];
              y[3 * i] += z * h0;
              y[3 * i + 1] += z * h1;
              y[3 * i + 2] += z * h2;
            }
          }
          // pose-pose, frames before fa
          for (int b = t0; b < t1; ++b) {
            const int fb = d.trk_frame[b];
            if (fb >= fa || fb == d.gauge_frame) continue;
            double Wb[18];
            track_W(b, fb, Wb);
#pragma unroll
            for (int i = 0; i < 6; ++i) {
              const double* zr = Z + zrow(i) + 6 * fb;
#pragma unroll
              for (int j = 0; j < 6; ++j) {
                const double z = zr[j];
#pragma unroll
                for (int k = 0; k < 3; ++k) y[3 * i + k] += z * Wb[3 * j + k];
              }
            }
          }
          double Wa[18];
          track_W(a, fa, Wa);
#pragma unroll
          for (int k = 0; k < 18; ++k) y[k] *= 2.0;
          // diagonal block Z[fa, fa], read from its lower triangle
#pragma unroll
          for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = 0; j < 6; ++j) {
              const double z = i >= j ? Z[zrow(i) + 6 * fa + j] : Z[zrow(j) + 6 * fa + i];
#pragma unroll
              for (int k = 0; k < 3; ++k) y[3 * i + k] += z * Wa[3 * j + k];
            }
#pragma unroll
          for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 3; ++j) {
              double m = 0.0;
#pragma unroll
              for (int k = 0; k < 6; ++k) m += Wa[3 * k + i] * y[3 * k + j];
              Q[3 * i + j] += m;
            }
        }
      }
      // camera-camera (the outer loop unrolled as well gives 255 registers and spills; rolled: at most 166, none)
#pragma unroll 1
      for (int c1 = 0; c1 < NC; ++c1) {
        const int r1 = d.cam_red[c1];
        if (r1 < 0) continue;
        double y[3] = {0, 0, 0};
#pragma unroll
        for (int c2 = 0; c2 < NC; ++c2) {
          const int r2 = d.cam_red[c2];
          if (r2 < 0) continue;
          const double z = sym_at(Z, sky, r1, r2);
#pragma unroll
          for (int j = 0; j < 3; ++j) y[j] += z * Tp[3 * c2 + j];
        }
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
          for (int j = 0; j < 3; ++j) Q[3 * i + j] += Tp[3 * c1 + i] * y[j];
      }
      // Sigma = Hi + sym(Q~)
      const double Hi[6] = {pd[0], pd[1], pd[2], pd[3], pd[4], pd[5]};
#pragma unroll
      for (int i = 0, h = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j, ++h) Sg[h] = Hi[j * 3 - j * (j + 1) / 2 + i] + 0.5 * (Q[3 * i + j] + Q[3 * j + i]);
    }
    double* o = out + 9 * (size_t)p;
    o[0] = Sg[0]; o[1] = Sg[1]; o[2] = Sg[3];
    o[3] = Sg[1]; o[4] = Sg[2]; o[5] = Sg[4];
    o[6] = Sg[3]; o[7] = Sg[4]; o[8] = Sg[5];
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

int launch_cov_points(const Dev& d, const double* Z, double* out, cudaStream_t s) {
  if (d.P == 0) return 0;
  LFBA_DISPATCH_NC(d.NC, (k_cov_points<NC><<<d.grid_pts, 128, 0, s>>>(d, Z, out)));
  return 1;
}

}  // namespace lfba
