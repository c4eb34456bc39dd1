// tscm_covariance.cuh — parameter covariance Sigma = H^-1, H = J^T J (undamped, loss-corrected),
// from the Jacobi-scaled reduced camera system that the Schur kernels assemble at radius +inf
// (DESIGN.md 5e).  With D = diag(D_e, D_c) the Jacobi scales of k_jacobi_scale,
//   camera block   Sigma_cc = D_c S~^-1 D_c,               S~ = U~ - W~^T V~^-1 W~
//   board block f  Sigma_ff = D_e,f (V~_f^-1 + Y~_f S~^-1 Y~_f^T) D_e,f,   Y~_f = V~_f^-1 W~_f
// Three kernels:
//   k_cov_factor   ONE CTA: the packed lower triangle of S~ (at most 202 live columns: 164 KB)
//                  in shared memory (k_cov_factor_global: the same code on a triangle in global
//                  memory, for the wider systems of allow_large_rigs, up to 416 columns: 678 KB,
//                  L2-resident; it runs once per covariance call, so simplicity beats speed),
//                  right-looking LDL^T with one barrier per column and the
//                  rank test of ceres::Covariance (pivot <= 1e-14 x largest diagonal entry);
//                  the unit-lower factor goes to global memory mirrored into both triangles
//                  (row i holds L[i][k<i] and L[k>i][i]) with 1/d on the diagonal, so that the
//                  forward and the backward substitution both read contiguous rows.
//   k_cov_inverse  one warp per identity column c: L y = e_c, x = L^-T D^-1 y against the factor
//                  (it stays in L2); writes S~^-1 (scaled, the frames read it) and Sigma_cc.
//   k_cov_frames   one warp per frame: V~_f from the frame record of the Schur kernels, its own
//                  6x6 LDL^T with the same rank test, W~_f rebuilt from the view records in G
//                  (independent of the Schur form), M = W~_f S~^-1 W~_f^T over the frame's
//                  columns only, Sigma_ff = D_e (V~^-1 + V~^-1 M V~^-1) D_e.
// k_solve is not reused: its factor lives in the registers and shared memory of one CTA and
// dies with it, and it carries one right-hand side where the inverse needs NL.
#pragma once

#include "tscm_kernels.cuh"

namespace tscm {

// The largest reduced system a solver accepts by default (create_shard checks it with k_solve's
// shared memory, solve_dims(), which is the tighter bound on a B200: 16 cameras with one fixed),
// and the largest that k_cov_factor holds in shared memory.
constexpr int kCovMaxNL = 202;
constexpr int kCovFactorThreads = 512;
constexpr int kCovInvWarps = 4;             // identity columns per CTA of k_cov_inverse
constexpr int kCovFrameWarps = 4;           // frames per CTA of k_cov_frames
constexpr double kCovMinRcond = 1e-14;      // ceres::Covariance::Options::min_reciprocal_condition_number

__host__ __device__ inline size_t cov_factor_smem(int NL) { return (size_t)NL * (NL + 1) / 2 * sizeof(double); }
// dynamic shared memory of k_cov_inverse (x per warp) and k_cov_frames (W~_f and its columns per warp)
inline size_t cov_inverse_smem(int NL) { return (size_t)kCovInvWarps * NL * sizeof(double); }
inline size_t cov_frames_smem(int NL) { return (size_t)kCovFrameWarps * NL * (6 * sizeof(double) + sizeof(short)); }

// flag bits: 1 = S~ is rank deficient, 2 = some V~_f is
// a: the packed lower triangle, row i at i (i + 1) / 2, in shared or global memory of this CTA.
__device__ __forceinline__ void cov_ldlt(double* a, int NL, int nbk, const double* __restrict__ Sr,
                                         double* __restrict__ fac, int* __restrict__ flag) {
  __shared__ double s_thr;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  for (int i = warp; i < NL; i += nw)
    for (int k = lane; k <= i; k += 32)
      a[i * (i + 1) / 2 + k] = Sr[solve_tile_id(i >> 2, k >> 2, nbk) * 16 + (i & 3) * 4 + (k & 3)];
  __syncthreads();
  if (tid == 0) {
    double m = 0.0;
    for (int i = 0; i < NL; ++i) m = fmax(m, a[i * (i + 1) / 2 + i]);
    s_thr = kCovMinRcond * m;
  }
  bool ok = true;
  for (int j = 0; j < NL; ++j) {
    __syncthreads();                          // the updates of step j - 1 (and s_thr) are visible
    const double d = a[j * (j + 1) / 2 + j];
    if (!(d > s_thr)) { ok = false; break; }  // same d and threshold in every thread: uniform exit
    const double inv = 1.0 / d;
    // trailing update a[i][k] -= a[i][j] a[k][j] / d, j < k <= i; column j itself is only read
    for (int i = j + 1 + warp; i < NL; i += nw) {
      const int ri = i * (i + 1) / 2;
      const double lij = a[ri + j] * inv;
      for (int k = j + 1 + lane; k <= i; k += 32) a[ri + k] -= lij * a[k * (k + 1) / 2 + j];
    }
  }
  if (!ok) {
    if (tid == 0) atomicOr(flag, 1);
    return;
  }
  __syncthreads();
  for (int i = warp; i < NL; i += nw) {
    const int ri = i * (i + 1) / 2;
    for (int k = lane; k <= i; k += 32) {
      const double dk = a[k * (k + 1) / 2 + k];
      if (k == i) {
        fac[(size_t)i * NL + i] = 1.0 / dk;
      } else {
        const double l = a[ri + k] / dk;
        fac[(size_t)i * NL + k] = l;
        fac[(size_t)k * NL + i] = l;
      }
    }
  }
}

__global__ void __launch_bounds__(kCovFactorThreads)
k_cov_factor(int NL, int nbk, const double* __restrict__ Sr, double* __restrict__ fac, int* __restrict__ flag) {
  extern __shared__ double a[];
  cov_ldlt(a, NL, nbk, Sr, fac, flag);
}

// tri: [NL (NL + 1) / 2] scratch
__global__ void __launch_bounds__(kCovFactorThreads)
k_cov_factor_global(int NL, int nbk, const double* __restrict__ Sr, double* __restrict__ fac, int* __restrict__ flag,
                    double* tri) {
  cov_ldlt(tri, NL, nbk, Sr, fac, flag);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sinv: S~^-1 (column c at c * NL); cam_out: D_c S~^-1 D_c, both NL x NL and symmetric.
__global__ void __launch_bounds__(32 * kCovInvWarps)
k_cov_inverse(DeviceProblem P, const double* __restrict__ scale_c, const double* __restrict__ fac,
              const int* __restrict__ flag, double* __restrict__ Sinv, double* __restrict__ cam_out) {
  extern __shared__ double s_x[];             // [kCovInvWarps][NL]
  if (*flag) return;
  const int NL = P.NL, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int c = blockIdx.x * kCovInvWarps + warp;
  if (c >= NL) return;
  double* x = s_x + warp * NL;
  for (int i = lane; i < NL; i += 32) x[i] = 0.0;
  __syncwarp();
  // forward: y_c = 1, y_i = -sum_{c <= k < i} L[i][k] y_k; then z = D^-1 y
  if (lane == 0) x[c] = 1.0;
  __syncwarp();
  for (int i = c + 1; i < NL; ++i) {
    const double* row = fac + (size_t)i * NL;
    double s = 0.0;
    for (int k = c + lane; k < i; k += 32) s += row[k] * x[k];
    s = warp_sum(s);
    if (lane == 0) x[i] = -s;
    __syncwarp();
  }
  for (int i = c + lane; i < NL; i += 32) x[i] *= fac[(size_t)i * NL + i];
  __syncwarp();
  // backward: x_i = z_i - sum_{k > i} L[k][i] x_k (row i of the mirrored factor)
  for (int i = NL - 2; i >= 0; --i) {
    const double* row = fac + (size_t)i * NL;
    double s = 0.0;
    for (int k = i + 1 + lane; k < NL; k += 32) s += row[k] * x[k];
    s = warp_sum(s);
    if (lane == 0) x[i] -= s;
    __syncwarp();
  }
  const double sc = scale_c[P.live_cam[c] * 13 + P.live_kk[c]];
  for (int i = lane; i < NL; i += 32) {
    Sinv[(size_t)c * NL + i] = x[i];
    cam_out[(size_t)c * NL + i] = scale_c[P.live_cam[i] * 13 + P.live_kk[i]] * x[i] * sc;
  }
}

// LDL^T of a symmetric 6x6 (full, row-major) into unit-lower L (strict part) and pivots d;
// false when a pivot fails the rank test against the largest diagonal entry.
__device__ __forceinline__ bool ldlt6(double M[36], double d[6]) {
  double mx = 0.0;
#pragma unroll
  for (int i = 0; i < 6; ++i) mx = fmax(mx, M[i * 6 + i]);
  const double thr = kCovMinRcond * mx;
  bool ok = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) {
    double dj = M[j * 6 + j];
#pragma unroll
    for (int k = 0; k < j; ++k) dj -= M[j * 6 + k] * M[j * 6 + k] * d[k];
    ok = ok && (dj > thr);
    d[j] = dj;
    const double inv = 1.0 / dj;
#pragma unroll
    for (int i = j + 1; i < 6; ++i) {
      double s = M[i * 6 + j];
#pragma unroll
      for (int k = 0; k < j; ++k) s -= M[i * 6 + k] * M[j * 6 + k] * d[k];
      M[i * 6 + j] = s * inv;
    }
  }
  return ok;
}

// out: [F][6][6] board blocks of this shard.
__global__ void __launch_bounds__(32 * kCovFrameWarps)
k_cov_frames(DeviceProblem P, ParamSet ps, const double* __restrict__ scale_e, const double* __restrict__ scale_c,
             const double* __restrict__ frame_rec, int Fpad, const double* __restrict__ Sinv,
             int* __restrict__ flag, double* __restrict__ out) {
  extern __shared__ double s_w[];             // [kCovFrameWarps][NL][6] W~_f, one row per live column of
                                              // the frame | [kCovFrameWarps][NL] its live column in S~
  if (*flag & 1) return;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int f = blockIdx.x * kCovFrameWarps + warp;
  if (f >= P.F) return;
  const int NL = P.NL;
  double se[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) se[i] = scale_e[f * 6 + i];
  // V~_f^-1 (undamped, scaled: entries [27, 48) of the frame record)
  double Vi[36];
  bool v_ok;
  {
    double M[36], d[6];
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
      for (int j = i; j < 6; ++j) {
        const double v = frame_rec[(size_t)(27 + tri6(i, j)) * Fpad + f];
        M[i * 6 + j] = v;
        M[j * 6 + i] = v;
      }
    v_ok = ldlt6(M, d);
#pragma unroll
    for (int c = 0; c < 6; ++c) {
      double e[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        double s = i == c ? 1.0 : 0.0;
#pragma unroll
        for (int k = 0; k < i; ++k) s -= M[i * 6 + k] * e[k];
        e[i] = s;
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) e[i] /= d[i];
#pragma unroll
      for (int i = 5; i >= 0; --i) {
        double s = e[i];
#pragma unroll
        for (int k = i + 1; k < 6; ++k) s -= M[k * 6 + i] * e[k];
        e[i] = s;
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) Vi[i * 6 + c] = e[i];
    }
  }
  if (!v_ok) {
    if (lane == 0) atomicOr(flag, 2);
    return;
  }
  // W~_f = D_e W D_c over the live columns of the cameras that see the frame
  double (*W)[6] = reinterpret_cast<double (*)[6]>(s_w + (size_t)warp * NL * 6);
  short* g = reinterpret_cast<short*>(s_w + (size_t)kCovFrameWarps * NL * 6) + warp * NL;
  int nf = 0;
  for (int q = P.frame_ptr[f]; q < P.frame_ptr[f + 1]; ++q) {
    const int v = P.frame_views[q], m = P.view_camera[v];
    const int n = P.live_off[m + 1] - P.live_off[m];
    const double* Gv = ps.G + (size_t)v * kViewStride;
    for (int k = lane; k < n; k += 32) {
      const int kk = n == 13 ? k : k + 6;
      const double sc = scale_c[m * 13 + kk];
#pragma unroll
      for (int p = 0; p < 6; ++p)
        W[nf + k][p] = se[p] * (kk < 6 ? Gv[kOffBC + p * 6 + kk] : Gv[kOffBI + p * 8 + (kk - 6)]) * sc;
      g[nf + k] = (short)(P.live_off[m] + k);
    }
    nf += n;
  }
  __syncwarp();
  // M = W~ S~^-1 W~^T: lane a owns columns a, a + 32, ...; t_a = S~^-1[a][:] W~^T
  double acc[21];
#pragma unroll
  for (int e = 0; e < 21; ++e) acc[e] = 0.0;
  for (int a0 = 0; a0 < nf; a0 += 32) {
    const int a = a0 + lane;
    const bool on = a < nf;
    const int ga = on ? g[a] : 0;
    double t[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
    for (int b = 0; b < nf; ++b) {
      const double sab = on ? Sinv[(size_t)g[b] * NL + ga] : 0.0;   // column g_b, coalesced over a
#pragma unroll
      for (int q = 0; q < 6; ++q) t[q] += sab * W[b][q];
    }
    if (on) {
#pragma unroll
      for (int p = 0; p < 6; ++p)
#pragma unroll
        for (int q = p; q < 6; ++q) acc[tri6(p, q)] += W[a][p] * t[q];
    }
  }
#pragma unroll
  for (int e = 0; e < 21; ++e) acc[e] = warp_sum(acc[e]);
  // Sigma_ff = D_e (V~^-1 + V~^-1 M V~^-1) D_e, every lane redundantly; lane e < 21 stores upper
  // entry e and its mirror
  double T[36];                                          // V~^-1 M
#pragma unroll
  for (int p = 0; p < 6; ++p)
#pragma unroll
    for (int q = 0; q < 6; ++q) {
      double s = 0.0;
#pragma unroll
      for (int r = 0; r < 6; ++r) s += Vi[p * 6 + r] * acc[r <= q ? tri6(r, q) : tri6(q, r)];
      T[p * 6 + q] = s;
    }
  double mine = 0.0;
  int pq = 0;
#pragma unroll
  for (int p = 0; p < 6; ++p)
#pragma unroll
    for (int q = p; q < 6; ++q) {
      double s = Vi[p * 6 + q];
#pragma unroll
      for (int r = 0; r < 6; ++r) s += T[p * 6 + r] * Vi[r * 6 + q];
      const bool me = lane == tri6(p, q);
      mine = me ? s * se[p] * se[q] : mine;
      pq = me ? p * 8 + q : pq;
    }
  if (lane < 21) {
    const int p = pq >> 3, q = pq & 7;
    out[(size_t)f * 36 + p * 6 + q] = mine;
    out[(size_t)f * 36 + q * 6 + p] = mine;
  }
}

}  // namespace tscm
