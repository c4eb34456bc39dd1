// tscm_monoinit.cu — mono cold start of TripleSphereCamera::calibrate on the GPU
// (SURVEY.md §8f #3), batched over the frames of one camera.
//
// Replaces, for every frame with a detection,
//   estimate_focal      /root/reference/TS.cpp:110-168   per board row: 4-column design matrix of
//                       the circle through the row's corners, cv::SVD::solveZ, focal estimate
//   estimate_extrinsic  /root/reference/TS.cpp:170-203   corners lifted to the unit sphere
//                       (TS.h:39-57), turned so that a corner near the board centre looks down +z,
//                       cv::solvePnPRansac on the normalised plane, result kept as [r1 r2 t]
// The two OpenCV calls are third-party code (absent C++ library): they are restated after their
// published algorithms — one-sided Jacobi SVD for solveZ; for solvePnPRansac(SOLVEPNP_ITERATIVE)
// on a planar target: Hartley-normalised DLT homography, pose from H, Levenberg-Marquardt on the
// reprojection error run to convergence, inliers re-fitted until the set is stable (the 8.0
// threshold in normalised units only removes corners whose back-projection is NaN or blew up) —
// and pinned, like the CPU oracle, against golden vectors of the real OpenCV 4.13.
//
// Mapping: one thread per (frame, board row) for the focal fits; one WARP per frame for the pose
// (k_mi_extrinsic_warp: the lanes split the rows of the Jacobi sweeps and the points of the
// Gauss-Newton sums, the frame's DLT matrix lives in the warp's shared memory; 2.7 ms for 5,000
// frames).  A thread-per-frame form (k_mi_extrinsic) keeps every sum in the oracle's statement
// order — it is the fallback for boards too large for shared memory and the A/B reference
// (TSCM_MI_FORM=thread; 32 ms: a single dependent chain per frame).  This translation unit is
// compiled with -fmad=false, so each double operation is one IEEE instruction as in the oracle
// (oracle/mono_init_oracle.cpp, -ffp-contract=off); what remains is the rounding of
// sin/cos/atan2/asin in CUDA's libm against glibc's and, in the warp form, the association of
// the lane-parallel sums.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../include/tscm.h"
#include "tscm_internal.h"

namespace tscm {
namespace mi {

struct Intr { double fx, fy, cx, cy, xi, lamda, alpha, b, c; };

constexpr int kMaxRow = 64;          // corners per board row (focal kernel, registers/local)
constexpr int kThreads = 64;

// cv::SVD::solveZ on an m x n matrix reached through W(i, j) (n <= 9): one-sided Jacobi, the
// right singular vector of the smallest singular value, unit length.
template <int N, typename Acc>
__device__ void solve_z(Acc W, int m, double* z) {
  double V[N * N];
#pragma unroll
  for (int k = 0; k < N * N; ++k) V[k] = 0.0;
#pragma unroll
  for (int j = 0; j < N; ++j) V[j * N + j] = 1.0;
  for (int sweep = 0; sweep < 60; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < N - 1; ++p)
      for (int q = p + 1; q < N; ++q) {
        double a = 0, b = 0, g = 0;
        for (int i = 0; i < m; ++i) {
          const double wp = W(i, p), wq = W(i, q);
          a += wp * wp; b += wq * wq; g += wp * wq;
        }
        if (fabs(g) <= 1e-300 || fabs(g) <= 2.220446049250313e-16 * sqrt(a * b)) continue;
        rotated = true;
        const double zeta = (b - a) / (2.0 * g);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
        for (int i = 0; i < m; ++i) {
          const double x = W(i, p), y = W(i, q);
          W(i, p) = c * x - sn * y; W(i, q) = sn * x + c * y;
        }
        for (int i = 0; i < N; ++i) {
          const double x = V[i * N + p], y = V[i * N + q];
          V[i * N + p] = c * x - sn * y; V[i * N + q] = sn * x + c * y;
        }
      }
    if (!rotated) break;
  }
  int best = 0;
  double best_norm = -1.0;
  for (int j = 0; j < N; ++j) {
    double s = 0;
    for (int i = 0; i < m; ++i) s += W(i, j) * W(i, j);
    if (best_norm < 0 || s < best_norm) { best_norm = s; best = j; }
  }
  double nz = 0;
  for (int i = 0; i < N; ++i) nz += V[i * N + best] * V[i * N + best];
  nz = sqrt(nz);
  for (int i = 0; i < N; ++i) z[i] = V[i * N + best] / nz;
}

// thread = (frame, board row): TS.cpp:127-158.  focal[frame * H + row] = estimate (NaN included, as
// the reference would add it), -1 = row skipped.
__global__ void __launch_bounds__(kThreads)
k_mi_focal_rows(const double* __restrict__ pixels, const uint8_t* __restrict__ has, int F, int W, int H,
                double cx, double cy, double* __restrict__ focal) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= F * H) return;
  const int k = t / H, r = t - k * H;
  const double skipped = -1.0;
  if (!has[k]) { focal[t] = skipped; return; }
  double D[kMaxRow * 4];
  const double* row = pixels + ((size_t)k * W * H + (size_t)r * W) * 2;
  for (int j = 0; j < W; ++j) {
    const double x = row[2 * j] - cx, y = row[2 * j + 1] - cy;
    D[4 * j] = x; D[4 * j + 1] = y; D[4 * j + 2] = 0.5; D[4 * j + 3] = -0.5 * (x * x + y * y);
  }
  double c[4];
  solve_z<4>([&](int i, int j) -> double& { return D[4 * i + j]; }, W, c);
  const double s = c[0] * c[0] + c[1] * c[1] + c[2] * c[3];
  if (s < 0) { focal[t] = skipped; return; }
  const double d = sqrt(1 / s);
  const double nx = c[0] * d, ny = c[1] * d;
  const double ob = nx * nx + ny * ny;
  if (ob > 0.95) { focal[t] = skipped; return; }
  focal[t] = fabs(c[2] * d / sqrt(1 - ob));
}

// TS.h:39-57
__device__ void unit_sphere(const Intr& I, double px, double py, const double* T, double* o) {
  const double x0 = px - I.cx, y0 = py - I.cy;
  const double det = I.fx * I.fy - I.b * I.c;
  const double mx = (I.fy * x0 - I.b * y0) / det, my = (-I.c * x0 + I.fx * y0) / det;
  const double k = I.alpha / (1 - I.alpha);
  const double r2 = mx * mx + my * my;
  const double gamma = (k + sqrt(1 + (1 - k * k) * r2)) / (r2 + 1);
  const double gk = gamma - k;
  const double eta = I.lamda * gk + sqrt((gk * gk - 1) * I.lamda * I.lamda + 1);
  const double mz = eta * gk;
  const double ml = mz - I.lamda;
  const double mu = I.xi * ml + sqrt(I.xi * I.xi * (ml * ml - 1) + 1);
  const double v[3] = {mu * eta * gamma * mx, mu * eta * gamma * my, mu * ml - I.xi};
  for (int r = 0; r < 3; ++r) o[r] = T[3 * r] * v[0] + T[3 * r + 1] * v[1] + T[3 * r + 2] * v[2];
}

// cv::Rodrigues, vector -> matrix
__device__ void rodrigues_v2m(const double* r, double* R) {
  const double theta = sqrt(r[0] * r[0] + r[1] * r[1] + r[2] * r[2]);
  for (int k = 0; k < 9; ++k) R[k] = (k % 4 == 0) ? 1.0 : 0.0;
  if (theta < 2.220446049250313e-16) return;
  const double c = cos(theta), s = sin(theta), c1 = 1.0 - c, it = 1.0 / theta;
  const double x = r[0] * it, y = r[1] * it, z = r[2] * it;
  R[0] = c + c1 * x * x;     R[1] = c1 * x * y - s * z; R[2] = c1 * x * z + s * y;
  R[3] = c1 * x * y + s * z; R[4] = c + c1 * y * y;     R[5] = c1 * y * z - s * x;
  R[6] = c1 * x * z - s * y; R[7] = c1 * y * z + s * x; R[8] = c + c1 * z * z;
}
// cv::Rodrigues, matrix -> vector: nearest rotation first (OpenCV: SVD, U V^T; here the same
// polar factor by Newton's iteration), then through the quaternion.
__device__ void rodrigues_m2v(const double* src, double* out) {
  double M[9];
  for (int i = 0; i < 9; ++i) M[i] = src[i];
  for (int it = 0; it < 12; ++it) {
    const double c00 = M[4] * M[8] - M[5] * M[7], c01 = M[5] * M[6] - M[3] * M[8], c02 = M[3] * M[7] - M[4] * M[6];
    const double det = M[0] * c00 + M[1] * c01 + M[2] * c02;
    if (!(fabs(det) > 1e-300)) break;
    const double T[9] = {c00, c01, c02,
                         M[2] * M[7] - M[1] * M[8], M[0] * M[8] - M[2] * M[6], M[1] * M[6] - M[0] * M[7],
                         M[1] * M[5] - M[2] * M[4], M[2] * M[3] - M[0] * M[5], M[0] * M[4] - M[1] * M[3]};
    double change = 0.0;
    for (int i = 0; i < 9; ++i) {
      const double v = 0.5 * (M[i] + T[i] / det);
      change = fmax(change, fabs(v - M[i]));
      M[i] = v;
    }
    if (change < 1e-16) break;
  }
  double q[4];
  const double tr = M[0] + M[4] + M[8];
  if (tr > 0) {
    const double s = sqrt(tr + 1.0) * 2;
    q[0] = 0.25 * s; q[1] = (M[7] - M[5]) / s; q[2] = (M[2] - M[6]) / s; q[3] = (M[3] - M[1]) / s;
  } else {
    int i = 0;
    if (M[4] > M[0]) i = 1;
    if (M[8] > M[4 * i]) i = 2;
    const int j = (i + 1) % 3, k = (i + 2) % 3;
    const double s = sqrt(1.0 + M[4 * i] - M[4 * j] - M[4 * k]) * 2;
    q[0] = (M[3 * k + j] - M[3 * j + k]) / s;
    q[1 + i] = 0.25 * s;
    q[1 + j] = (M[3 * j + i] + M[3 * i + j]) / s;
    q[1 + k] = (M[3 * k + i] + M[3 * i + k]) / s;
  }
  if (q[0] < 0) for (int e = 0; e < 4; ++e) q[e] = -q[e];
  const double vn = sqrt(q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  out[0] = out[1] = out[2] = 0.0;
  if (vn > 0) {
    const double ang = 2.0 * atan2(vn, q[0]);
    for (int i = 0; i < 3; ++i) out[i] = q[1 + i] / vn * ang;
  }
}

__device__ bool chol_solve6(double* A, double* b) {
  const int n = 6;
  for (int j = 0; j < n; ++j) {
    double d = A[j * n + j];
    for (int k = 0; k < j; ++k) d -= A[j * n + k] * A[j * n + k];
    if (!(d > 0)) return false;
    d = sqrt(d);
    A[j * n + j] = d;
    for (int i = j + 1; i < n; ++i) {
      double v = A[i * n + j];
      for (int k = 0; k < j; ++k) v -= A[i * n + k] * A[j * n + k];
      A[i * n + j] = v / d;
    }
  }
  for (int i = 0; i < n; ++i) { double v = b[i]; for (int k = 0; k < i; ++k) v -= A[i * n + k] * b[k]; b[i] = v / A[i * n + i]; }
  for (int i = n - 1; i >= 0; --i) { double v = b[i]; for (int k = i + 1; k < n; ++k) v -= A[k * n + i] * b[k]; b[i] = v / A[i * n + i]; }
  return true;
}

// Per-frame scratch in frame-minor layout: element e of frame f at base[e * F + f].  The DLT
// matrix, which the Jacobi sweeps walk ~10^5 times per frame, lives in SHARED memory when all
// frames fit one wave of blocks (16 frames x 12.4 KB per block at K = 88; lane-minor, so the
// lanes of an access hit distinct banks) and in the global scratch otherwise.
struct Scratch {
  double* xy;      // [2K][F] normalised-plane points
  double* A;       // [2K * 9][F] DLT matrix (global fallback)
  uint8_t* use;    // [K][F] inlier flags
  int F;
  int a_in_smem;   // 1: the DLT matrix of thread t is at smem[e * blockDim.x + t]
};

// solvePnP(SOLVEPNP_ITERATIVE) on the flagged points of a planar target with an identity camera
// matrix: R (row-major), t.  false = fewer than 4 points or a degenerate homography.
__device__ bool pnp_planar(const Scratch& S, int f, int K, const double* __restrict__ worlds, double* R, double* t,
                           double* Abase, size_t Astride) {
  const int F = S.F;
  auto X = [&](int i) { return worlds[3 * i]; };
  auto Y = [&](int i) { return worlds[3 * i + 1]; };
  auto Z = [&](int i) { return worlds[3 * i + 2]; };
  auto x = [&](int i) { return S.xy[(size_t)(2 * i) * F + f]; };
  auto y = [&](int i) { return S.xy[(size_t)(2 * i + 1) * F + f]; };
  auto used = [&](int i) { return S.use[(size_t)i * F + f] != 0; };
  int n = 0, first = -1;
  double mx = 0, my = 0, mX = 0, mY = 0;
  for (int i = 0; i < K; ++i) {
    if (!used(i)) continue;
    if (first < 0) first = i;
    mx += x(i); my += y(i); mX += X(i); mY += Y(i);
    ++n;
  }
  if (n < 4) return false;
  mx /= n; my /= n; mX /= n; mY /= n;
  double sx = 0, sX = 0;
  for (int i = 0; i < K; ++i) {
    if (!used(i)) continue;
    sx += sqrt((x(i) - mx) * (x(i) - mx) + (y(i) - my) * (y(i) - my));
    sX += sqrt((X(i) - mX) * (X(i) - mX) + (Y(i) - mY) * (Y(i) - mY));
  }
  if (!(sx > 0) || !(sX > 0)) return false;
  sx = sqrt(2.0) * n / sx; sX = sqrt(2.0) * n / sX;      // Hartley normalisation
  {
    int row = 0;
    for (int i = 0; i < K; ++i) {
      if (!used(i)) continue;
      const double u = (x(i) - mx) * sx, v = (y(i) - my) * sx, a = (X(i) - mX) * sX, b = (Y(i) - mY) * sX;
      const double r0[9] = {a, b, 1, 0, 0, 0, -u * a, -u * b, -u};
      const double r1[9] = {0, 0, 0, a, b, 1, -v * a, -v * b, -v};
      for (int k = 0; k < 9; ++k) {
        Abase[(size_t)(row * 9 + k) * Astride] = r0[k];
        Abase[(size_t)((row + 1) * 9 + k) * Astride] = r1[k];
      }
      row += 2;
    }
  }
  double Hn[9];
  solve_z<9>([&](int i, int j) -> double& { return Abase[(size_t)(i * 9 + j) * Astride]; }, 2 * n, Hn);
  // H = T_img^-1 * Hn * T_obj
  const double Ti[9] = {1 / sx, 0, mx, 0, 1 / sx, my, 0, 0, 1};
  const double To[9] = {sX, 0, -mX * sX, 0, sX, -mY * sX, 0, 0, 1};
  double T1[9], H[9];
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += Ti[3 * r + k] * Hn[3 * k + c]; T1[3 * r + c] = s; }
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += T1[3 * r + k] * To[3 * k + c]; H[3 * r + c] = s; }
  const double n1 = sqrt(H[0] * H[0] + H[3] * H[3] + H[6] * H[6]);
  const double n2 = sqrt(H[1] * H[1] + H[4] * H[4] + H[7] * H[7]);
  if (!(n1 > 0) || !(n2 > 0)) return false;
  double sc = 2.0 / (n1 + n2);
  const double z0 = Z(first);
  if ((H[6] * mX + H[7] * mY + H[8]) * sc < 0) sc = -sc;           // the board lies in front of the camera
  double r1[3] = {H[0] * sc, H[3] * sc, H[6] * sc}, r2[3] = {H[1] * sc, H[4] * sc, H[7] * sc};
  t[0] = H[2] * sc; t[1] = H[5] * sc; t[2] = H[8] * sc;
  {
    const double a1 = sqrt(r1[0] * r1[0] + r1[1] * r1[1] + r1[2] * r1[2]);
    const double a2 = sqrt(r2[0] * r2[0] + r2[1] * r2[1] + r2[2] * r2[2]);
    for (int k = 0; k < 3; ++k) { r1[k] /= a1; r2[k] /= a2; }
    double s[3], d[3];
    for (int k = 0; k < 3; ++k) { s[k] = r1[k] + r2[k]; d[k] = r1[k] - r2[k]; }
    const double ns = sqrt(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]);
    const double dd = (d[0] * s[0] + d[1] * s[1] + d[2] * s[2]) / (ns * ns);
    for (int k = 0; k < 3; ++k) d[k] -= dd * s[k];
    const double nd = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    const double h = sqrt(0.5);
    for (int k = 0; k < 3; ++k) { r1[k] = h * (s[k] / ns + d[k] / nd); r2[k] = h * (s[k] / ns - d[k] / nd); }
  }
  R[0] = r1[0]; R[1] = r2[0]; R[2] = r1[1] * r2[2] - r1[2] * r2[1];
  R[3] = r1[1]; R[4] = r2[1]; R[5] = r1[2] * r2[0] - r1[0] * r2[2];
  R[6] = r1[2]; R[7] = r2[2]; R[8] = r1[0] * r2[1] - r1[1] * r2[0];
  for (int k = 0; k < 3; ++k) t[k] -= R[3 * k + 2] * z0;
  // damped Gauss-Newton on sum |(Px/Pz, Py/Pz) - (x, y)|^2, left-multiplicative rotation update
  auto cost_at = [&](const double* Rm, const double* tm) {
    double c = 0;
    for (int i = 0; i < K; ++i) {
      if (!used(i)) continue;
      const double p[3] = {X(i), Y(i), Z(i)};
      double P[3];
      for (int r = 0; r < 3; ++r) P[r] = Rm[3 * r] * p[0] + Rm[3 * r + 1] * p[1] + Rm[3 * r + 2] * p[2] + tm[r];
      const double eu = P[0] / P[2] - x(i), ev = P[1] / P[2] - y(i);
      c += eu * eu + ev * ev;
    }
    return c;
  };
  double lambda = 1e-6, cost = cost_at(R, t);
  for (int it = 0; it < 200; ++it) {
    double JtJ[36], Jtr[6];
    for (int k = 0; k < 36; ++k) JtJ[k] = 0;
    for (int k = 0; k < 6; ++k) Jtr[k] = 0;
    for (int i = 0; i < K; ++i) {
      if (!used(i)) continue;
      const double p[3] = {X(i), Y(i), Z(i)};
      double q[3], P[3];
      for (int r = 0; r < 3; ++r) { q[r] = R[3 * r] * p[0] + R[3 * r + 1] * p[1] + R[3 * r + 2] * p[2]; P[r] = q[r] + t[r]; }
      const double iz = 1.0 / P[2], u = P[0] * iz, v = P[1] * iz;
      const double dP[3][6] = {{0, q[2], -q[1], 1, 0, 0}, {-q[2], 0, q[0], 0, 1, 0}, {q[1], -q[0], 0, 0, 0, 1}};
      double Ju[6], Jv[6];
      for (int k = 0; k < 6; ++k) { Ju[k] = iz * (dP[0][k] - u * dP[2][k]); Jv[k] = iz * (dP[1][k] - v * dP[2][k]); }
      const double eu = u - x(i), ev = v - y(i);
      for (int a = 0; a < 6; ++a) {
        Jtr[a] += Ju[a] * eu + Jv[a] * ev;
        for (int b = 0; b <= a; ++b) JtJ[a * 6 + b] += Ju[a] * Ju[b] + Jv[a] * Jv[b];
      }
    }
    for (int a = 0; a < 6; ++a) for (int b = a + 1; b < 6; ++b) JtJ[a * 6 + b] = JtJ[b * 6 + a];
    bool improved = false;
    double step_norm = 0;
    for (int tries = 0; tries < 30 && !improved; ++tries) {
      double Am[36], d[6];
      for (int k = 0; k < 36; ++k) Am[k] = JtJ[k];
      for (int k = 0; k < 6; ++k) { Am[k * 6 + k] *= 1.0 + lambda; d[k] = -Jtr[k]; }
      if (!chol_solve6(Am, d)) { lambda *= 10; continue; }
      double dR[9], Rn[9], tn[3];
      rodrigues_v2m(d, dR);
      for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += dR[3 * r + k] * R[3 * k + c]; Rn[3 * r + c] = s; }
      for (int k = 0; k < 3; ++k) tn[k] = t[k] + d[3 + k];
      const double cn = cost_at(Rn, tn);
      if (cn <= cost) {
        step_norm = 0;
        for (int k = 0; k < 3; ++k) step_norm += d[k] * d[k] + d[3 + k] * d[3 + k] / (1.0 + t[k] * t[k]);
        for (int k = 0; k < 9; ++k) R[k] = Rn[k];
        for (int k = 0; k < 3; ++k) t[k] = tn[k];
        improved = true; cost = cn; lambda = fmax(lambda * 0.1, 1e-12);
      } else {
        lambda *= 10;
      }
    }
    if (!improved || step_norm < 1e-28) break;
  }
  return true;
}

// thread = frame: TS.cpp:172-202
__global__ void __launch_bounds__(kThreads)
k_mi_extrinsic(const double* __restrict__ pixels, const uint8_t* __restrict__ has, const double* __restrict__ worlds,
               int F, int W, int H, Intr I, Scratch S, double* __restrict__ mono_rt, uint8_t* __restrict__ ok) {
  extern __shared__ __align__(16) double mi_smem[];
  const int f = blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const int K = W * H;
  double* Abase = S.a_in_smem ? mi_smem + threadIdx.x : S.A + f;
  const size_t Astride = S.a_in_smem ? blockDim.x : (size_t)F;
  double* M = mono_rt + 9 * (size_t)f;
  for (int k = 0; k < 9; ++k) M[k] = 0.0;
  ok[f] = 0;
  if (!has[f]) return;
  const double* px = pixels + (size_t)f * K * 2;
  const double eye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  const int centre = K / 2 - W / 2 - 1;                                    // TS.cpp:177
  double p[3];
  unit_sphere(I, px[2 * centre], px[2 * centre + 1], eye, p);
  const double az = atan2(p[0], p[2]), el = asin(p[1]);
  const double R1[9] = {cos(az), 0, -sin(az), 0, 1, 0, sin(az), 0, cos(az)};
  const double R2[9] = {1, 0, 0, 0, cos(el), -sin(el), 0, sin(el), cos(el)};
  double T[9];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      double s = 0.0;
      for (int q = 0; q < 3; ++q) s += R2[3 * r + q] * R1[3 * q + c];
      T[3 * r + c] = s;
    }
  for (int i = 0; i < K; ++i) {
    double ray[3];
    unit_sphere(I, px[2 * i], px[2 * i + 1], T, ray);
    const double u = ray[0] / ray[2], v = ray[1] / ray[2];
    S.xy[(size_t)(2 * i) * F + f] = u;
    S.xy[(size_t)(2 * i + 1) * F + f] = v;
    S.use[(size_t)i * F + f] = (isfinite(u) && isfinite(v)) ? 1 : 0;
  }
  // solvePnPRansac: fit, drop the points beyond the 8.0 threshold, re-fit until the set is stable
  double R[9], t[3], rvec[3];
  for (int round = 0; round < 8; ++round) {
    if (!pnp_planar(S, f, K, worlds, R, t, Abase, Astride)) return;
    // the pose leaves solvePnP as (rvec, tvec) and is turned back into a matrix for the test
    rodrigues_m2v(R, rvec);
    double Rr[9];
    rodrigues_v2m(rvec, Rr);
    bool changed = false;
    for (int i = 0; i < K; ++i) {
      if (!S.use[(size_t)i * F + f]) continue;
      double P[3];
      for (int r = 0; r < 3; ++r)
        P[r] = Rr[3 * r] * worlds[3 * i] + Rr[3 * r + 1] * worlds[3 * i + 1] + Rr[3 * r + 2] * worlds[3 * i + 2] + t[r];
      const double eu = 1.0 * P[0] / P[2] + 0.0 - S.xy[(size_t)(2 * i) * F + f];
      const double ev = 1.0 * P[1] / P[2] + 0.0 - S.xy[(size_t)(2 * i + 1) * F + f];
      if (!(eu * eu + ev * ev <= 8.0 * 8.0)) { S.use[(size_t)i * F + f] = 0; changed = true; }
    }
    if (!changed) break;
  }
  double pose[9];
  rodrigues_v2m(rvec, pose);
  // Rt = transform.t() * Rt; tvec = transform.t() * tvec; third column <- tvec (TS.cpp:195-200)
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 2; ++c) {
      double s = 0.0;
      for (int q = 0; q < 3; ++q) s += T[3 * q + r] * pose[3 * q + c];
      M[3 * r + c] = s;
    }
    double s = 0.0;
    for (int q = 0; q < 3; ++q) s += T[3 * q + r] * t[q];
    M[3 * r + 2] = s;
  }
  ok[f] = 1;
}


// ---------------------------------------------------------------------------------------------
// Warp-cooperative form of k_mi_extrinsic: ONE WARP per frame.  The thread-per-frame kernel above
// keeps every sum in the scalar statement order but is a single dependent chain per frame (32 ms
// for 5,000 frames, each thread walking its DLT matrix ~10^5 times).  Here the lanes split the
// rows of the Jacobi sweeps and the points of the Gauss-Newton sums; partial sums meet in a
// butterfly (every lane ends with the same bits, so control flow stays uniform), the DLT matrix,
// the points and the flags live in the warp's shared memory.  Same algorithm, same stopping
// rules; what changes is the association of the sums (1e-16 per sum, far inside the 1e-8 flat
// bottom of the least-squares minimum both forms stop in).
// ---------------------------------------------------------------------------------------------
constexpr int kMiWarps = 4;          // frames per CTA

__device__ __forceinline__ double wsum(double x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

struct WarpScratch {
  double* A;         // [9][ld] DLT matrix, column-major
  double* V;         // [9][9] accumulated rotations
  double* xy;        // [2][K] normalised-plane points (x row, y row)
  uint8_t* use;      // [K]
  int ld;
};
__host__ __device__ inline size_t mi_warp_smem_bytes(int K) {
  const size_t ld = 2 * (size_t)K;
  return (9 * ld + 81 + 2 * (size_t)K) * sizeof(double) + (((size_t)K + 15) & ~(size_t)15);
}

// solveZ of the m x 9 matrix in S.A: one-sided Jacobi, rows split over the lanes
__device__ void solve_z9_warp(const WarpScratch& S, int m, int lane, double* z) {
  const int ld = S.ld;
  for (int k = lane; k < 81; k += 32) S.V[k] = (k % 10 == 0) ? 1.0 : 0.0;
  __syncwarp();
  for (int sweep = 0; sweep < 60; ++sweep) {
    bool rotated = false;
    for (int p = 0; p < 8; ++p)
      for (int q = p + 1; q < 9; ++q) {
        double* Ap = S.A + p * ld;
        double* Aq = S.A + q * ld;
        double a = 0, b = 0, g = 0;
        for (int i = lane; i < m; i += 32) {
          const double wp = Ap[i], wq = Aq[i];
          a += wp * wp; b += wq * wq; g += wp * wq;
        }
        a = wsum(a); b = wsum(b); g = wsum(g);
        if (fabs(g) <= 1e-300 || fabs(g) <= 2.220446049250313e-16 * sqrt(a * b)) continue;
        rotated = true;
        const double zeta = (b - a) / (2.0 * g);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
        for (int i = lane; i < m; i += 32) {
          const double x = Ap[i], y = Aq[i];
          Ap[i] = c * x - sn * y; Aq[i] = sn * x + c * y;
        }
        if (lane < 9) {
          const double x = S.V[lane * 9 + p], y = S.V[lane * 9 + q];
          S.V[lane * 9 + p] = c * x - sn * y; S.V[lane * 9 + q] = sn * x + c * y;
        }
        __syncwarp();
      }
    if (!rotated) break;
  }
  int best = 0;
  double best_norm = -1.0;
  for (int j = 0; j < 9; ++j) {
    double sacc = 0;
    for (int i = lane; i < m; i += 32) sacc += S.A[j * ld + i] * S.A[j * ld + i];
    sacc = wsum(sacc);
    if (best_norm < 0 || sacc < best_norm) { best_norm = sacc; best = j; }
  }
  double nz = 0;
  for (int i = 0; i < 9; ++i) nz += S.V[i * 9 + best] * S.V[i * 9 + best];
  nz = sqrt(nz);
  for (int i = 0; i < 9; ++i) z[i] = S.V[i * 9 + best] / nz;
  __syncwarp();
}

__device__ bool pnp_planar_warp(const WarpScratch& S, int K, const double* __restrict__ worlds, int lane, double* R,
                                double* t) {
  const double* xs = S.xy;
  const double* ys = S.xy + K;
  // number of flagged points, the first of them, the four means
  int n = 0, first = K;
  double mx = 0, my = 0, mX = 0, mY = 0;
  for (int i = lane; i < K; i += 32) {
    if (!S.use[i]) continue;
    ++n; first = min(first, i);
    mx += xs[i]; my += ys[i]; mX += worlds[3 * i]; mY += worlds[3 * i + 1];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    n += __shfl_xor_sync(0xffffffffu, n, o);
    first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
  }
  if (n < 4) return false;
  mx = wsum(mx) / n; my = wsum(my) / n; mX = wsum(mX) / n; mY = wsum(mY) / n;
  double sx = 0, sX = 0;
  for (int i = lane; i < K; i += 32) {
    if (!S.use[i]) continue;
    sx += sqrt((xs[i] - mx) * (xs[i] - mx) + (ys[i] - my) * (ys[i] - my));
    sX += sqrt((worlds[3 * i] - mX) * (worlds[3 * i] - mX) + (worlds[3 * i + 1] - mY) * (worlds[3 * i + 1] - mY));
  }
  sx = wsum(sx); sX = wsum(sX);
  if (!(sx > 0) || !(sX > 0)) return false;
  sx = sqrt(2.0) * n / sx; sX = sqrt(2.0) * n / sX;      // Hartley normalisation
  // DLT rows of the flagged points, in point order: rows 2 r, 2 r + 1 for the r-th flagged point
  {
    int base = 0;
    for (int i0 = 0; i0 < K; i0 += 32) {
      const int i = i0 + lane;
      const bool u_ = i < K && S.use[i];
      const unsigned mask = __ballot_sync(0xffffffffu, u_);
      if (u_) {
        const int row = 2 * (base + __popc(mask & ((1u << lane) - 1u)));
        const double u = (xs[i] - mx) * sx, v = (ys[i] - my) * sx;
        const double a = (worlds[3 * i] - mX) * sX, b = (worlds[3 * i + 1] - mY) * sX;
        const double r0[9] = {a, b, 1, 0, 0, 0, -u * a, -u * b, -u};
        const double r1[9] = {0, 0, 0, a, b, 1, -v * a, -v * b, -v};
#pragma unroll
        for (int k = 0; k < 9; ++k) { S.A[k * S.ld + row] = r0[k]; S.A[k * S.ld + row + 1] = r1[k]; }
      }
      base += __popc(mask);
    }
  }
  __syncwarp();
  double Hn[9];
  solve_z9_warp(S, 2 * n, lane, Hn);
  // from here to the Gauss-Newton loop every lane computes the same few hundred flops
  const double Ti[9] = {1 / sx, 0, mx, 0, 1 / sx, my, 0, 0, 1};
  const double To[9] = {sX, 0, -mX * sX, 0, sX, -mY * sX, 0, 0, 1};
  double T1[9], H[9];
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += Ti[3 * r + k] * Hn[3 * k + c]; T1[3 * r + c] = s; }
  for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += T1[3 * r + k] * To[3 * k + c]; H[3 * r + c] = s; }
  const double n1 = sqrt(H[0] * H[0] + H[3] * H[3] + H[6] * H[6]);
  const double n2 = sqrt(H[1] * H[1] + H[4] * H[4] + H[7] * H[7]);
  if (!(n1 > 0) || !(n2 > 0)) return false;
  double sc = 2.0 / (n1 + n2);
  const double z0 = worlds[3 * first + 2];
  if ((H[6] * mX + H[7] * mY + H[8]) * sc < 0) sc = -sc;
  double r1[3] = {H[0] * sc, H[3] * sc, H[6] * sc}, r2[3] = {H[1] * sc, H[4] * sc, H[7] * sc};
  t[0] = H[2] * sc; t[1] = H[5] * sc; t[2] = H[8] * sc;
  {
    const double a1 = sqrt(r1[0] * r1[0] + r1[1] * r1[1] + r1[2] * r1[2]);
    const double a2 = sqrt(r2[0] * r2[0] + r2[1] * r2[1] + r2[2] * r2[2]);
    for (int k = 0; k < 3; ++k) { r1[k] /= a1; r2[k] /= a2; }
    double s[3], d[3];
    for (int k = 0; k < 3; ++k) { s[k] = r1[k] + r2[k]; d[k] = r1[k] - r2[k]; }
    const double ns = sqrt(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]);
    const double dd = (d[0] * s[0] + d[1] * s[1] + d[2] * s[2]) / (ns * ns);
    for (int k = 0; k < 3; ++k) d[k] -= dd * s[k];
    const double nd = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
    const double h = sqrt(0.5);
    for (int k = 0; k < 3; ++k) { r1[k] = h * (s[k] / ns + d[k] / nd); r2[k] = h * (s[k] / ns - d[k] / nd); }
  }
  R[0] = r1[0]; R[1] = r2[0]; R[2] = r1[1] * r2[2] - r1[2] * r2[1];
  R[3] = r1[1]; R[4] = r2[1]; R[5] = r1[2] * r2[0] - r1[0] * r2[2];
  R[6] = r1[2]; R[7] = r2[2]; R[8] = r1[0] * r2[1] - r1[1] * r2[0];
  for (int k = 0; k < 3; ++k) t[k] -= R[3 * k + 2] * z0;
  auto cost_at = [&](const double* Rm, const double* tm) {
    double c = 0;
    for (int i = lane; i < K; i += 32) {
      if (!S.use[i]) continue;
      const double p[3] = {worlds[3 * i], worlds[3 * i + 1], worlds[3 * i + 2]};
      double P[3];
      for (int r = 0; r < 3; ++r) P[r] = Rm[3 * r] * p[0] + Rm[3 * r + 1] * p[1] + Rm[3 * r + 2] * p[2] + tm[r];
      const double eu = P[0] / P[2] - xs[i], ev = P[1] / P[2] - ys[i];
      c += eu * eu + ev * ev;
    }
    return wsum(c);
  };
  double lambda = 1e-6, cost = cost_at(R, t);
  for (int it = 0; it < 200; ++it) {
    double L[21], Jtr[6];                       // lower triangle of J^T J, row-major packed
#pragma unroll
    for (int k = 0; k < 21; ++k) L[k] = 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) Jtr[k] = 0;
    for (int i = lane; i < K; i += 32) {
      if (!S.use[i]) continue;
      const double p[3] = {worlds[3 * i], worlds[3 * i + 1], worlds[3 * i + 2]};
      double q[3], P[3];
      for (int r = 0; r < 3; ++r) { q[r] = R[3 * r] * p[0] + R[3 * r + 1] * p[1] + R[3 * r + 2] * p[2]; P[r] = q[r] + t[r]; }
      const double iz = 1.0 / P[2], u = P[0] * iz, v = P[1] * iz;
      const double dP[3][6] = {{0, q[2], -q[1], 1, 0, 0}, {-q[2], 0, q[0], 0, 1, 0}, {q[1], -q[0], 0, 0, 0, 1}};
      double Ju[6], Jv[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) { Ju[k] = iz * (dP[0][k] - u * dP[2][k]); Jv[k] = iz * (dP[1][k] - v * dP[2][k]); }
      const double eu = u - xs[i], ev = v - ys[i];
#pragma unroll
      for (int a = 0; a < 6; ++a) {
        Jtr[a] += Ju[a] * eu + Jv[a] * ev;
#pragma unroll
        for (int b = 0; b <= a; ++b) L[a * (a + 1) / 2 + b] += Ju[a] * Ju[b] + Jv[a] * Jv[b];
      }
    }
#pragma unroll
    for (int k = 0; k < 21; ++k) L[k] = wsum(L[k]);
#pragma unroll
    for (int k = 0; k < 6; ++k) Jtr[k] = wsum(Jtr[k]);
    double JtJ[36];
#pragma unroll
    for (int a = 0; a < 6; ++a)
#pragma unroll
      for (int b = 0; b <= a; ++b) { JtJ[a * 6 + b] = L[a * (a + 1) / 2 + b]; JtJ[b * 6 + a] = L[a * (a + 1) / 2 + b]; }
    bool improved = false;
    double step_norm = 0;
    for (int tries = 0; tries < 30 && !improved; ++tries) {
      double Am[36], d[6];
      for (int k = 0; k < 36; ++k) Am[k] = JtJ[k];
      for (int k = 0; k < 6; ++k) { Am[k * 6 + k] *= 1.0 + lambda; d[k] = -Jtr[k]; }
      if (!chol_solve6(Am, d)) { lambda *= 10; continue; }
      double dR[9], Rn[9], tn[3];
      rodrigues_v2m(d, dR);
      for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) { double s = 0; for (int k = 0; k < 3; ++k) s += dR[3 * r + k] * R[3 * k + c]; Rn[3 * r + c] = s; }
      for (int k = 0; k < 3; ++k) tn[k] = t[k] + d[3 + k];
      const double cn = cost_at(Rn, tn);
      if (cn <= cost) {
        step_norm = 0;
        for (int k = 0; k < 3; ++k) step_norm += d[k] * d[k] + d[3 + k] * d[3 + k] / (1.0 + t[k] * t[k]);
        for (int k = 0; k < 9; ++k) R[k] = Rn[k];
        for (int k = 0; k < 3; ++k) t[k] = tn[k];
        improved = true; cost = cn; lambda = fmax(lambda * 0.1, 1e-12);
      } else {
        lambda *= 10;
      }
    }
    if (!improved || step_norm < 1e-28) break;
  }
  return true;
}

// warp = frame: TS.cpp:172-202
__global__ void __launch_bounds__(32 * kMiWarps)
k_mi_extrinsic_warp(const double* __restrict__ pixels, const uint8_t* __restrict__ has,
                    const double* __restrict__ worlds, int F, int W, int H, Intr I, size_t warp_bytes,
                    double* __restrict__ mono_rt, uint8_t* __restrict__ ok) {
  extern __shared__ __align__(16) unsigned char mi_wsmem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int f = blockIdx.x * kMiWarps + warp;
  if (f >= F) return;
  const int K = W * H;
  WarpScratch S;
  S.ld = 2 * K;
  S.A = reinterpret_cast<double*>(mi_wsmem + (size_t)warp * warp_bytes);
  S.V = S.A + 9 * (size_t)S.ld;
  S.xy = S.V + 81;
  S.use = reinterpret_cast<uint8_t*>(S.xy + 2 * (size_t)K);
  double* M = mono_rt + 9 * (size_t)f;
  if (lane == 0) {                       // lane 0 owns the frame's outputs
    for (int k = 0; k < 9; ++k) M[k] = 0.0;
    ok[f] = 0;
  }
  if (!has[f]) return;
  const double* px = pixels + (size_t)f * K * 2;
  const double eye[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  const int centre = K / 2 - W / 2 - 1;                                    // TS.cpp:177
  double p[3];
  unit_sphere(I, px[2 * centre], px[2 * centre + 1], eye, p);
  const double az = atan2(p[0], p[2]), el = asin(p[1]);
  const double R1[9] = {cos(az), 0, -sin(az), 0, 1, 0, sin(az), 0, cos(az)};
  const double R2[9] = {1, 0, 0, 0, cos(el), -sin(el), 0, sin(el), cos(el)};
  double T[9];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      double s = 0.0;
      for (int q = 0; q < 3; ++q) s += R2[3 * r + q] * R1[3 * q + c];
      T[3 * r + c] = s;
    }
  for (int i = lane; i < K; i += 32) {
    double ray[3];
    unit_sphere(I, px[2 * i], px[2 * i + 1], T, ray);
    const double u = ray[0] / ray[2], v = ray[1] / ray[2];
    S.xy[i] = u;
    S.xy[K + i] = v;
    S.use[i] = (isfinite(u) && isfinite(v)) ? 1 : 0;
  }
  __syncwarp();
  double R[9], t[3], rvec[3];
  for (int round = 0; round < 8; ++round) {
    if (!pnp_planar_warp(S, K, worlds, lane, R, t)) return;
    rodrigues_m2v(R, rvec);
    double Rr[9];
    rodrigues_v2m(rvec, Rr);
    bool changed = false;
    for (int i = lane; i < K; i += 32) {
      if (!S.use[i]) continue;
      double P[3];
      for (int r = 0; r < 3; ++r)
        P[r] = Rr[3 * r] * worlds[3 * i] + Rr[3 * r + 1] * worlds[3 * i + 1] + Rr[3 * r + 2] * worlds[3 * i + 2] + t[r];
      const double eu = 1.0 * P[0] / P[2] + 0.0 - S.xy[i];
      const double ev = 1.0 * P[1] / P[2] + 0.0 - S.xy[K + i];
      if (!(eu * eu + ev * ev <= 8.0 * 8.0)) { S.use[i] = 0; changed = true; }
    }
    changed = __any_sync(0xffffffffu, changed);
    __syncwarp();
    if (!changed) break;
  }
  double pose[9];
  rodrigues_v2m(rvec, pose);
  if (lane == 0) {
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 2; ++c) {
        double s = 0.0;
        for (int q = 0; q < 3; ++q) s += T[3 * q + r] * pose[3 * q + c];
        M[3 * r + c] = s;
      }
      double s = 0.0;
      for (int q = 0; q < 3; ++q) s += T[3 * q + r] * t[q];
      M[3 * r + 2] = s;
    }
    ok[f] = 1;
  }
}

}  // namespace mi
}  // namespace tscm

using namespace tscm;

extern "C" int tscm_mono_init(const tscm_mono_init_problem* P, int device, tscm_mono_init_result* R) {
  internal::DeviceScope scope;
  if (!P || !R || !P->worlds || !P->has_board || !P->pixels || !R->mono_rt || !R->frame_ok) {
    internal::set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT;
  }
  const int F = P->num_frames, W = P->board_width, H = P->board_height, K = W * H;
  if (F <= 0 || W <= 0 || H <= 0 || W > mi::kMaxRow || K / 2 - W / 2 - 1 < 0) {
    internal::set_error("bad mono-init sizes: %d frames, board %d x %d (rows of at most %d corners)", F, W, H, mi::kMaxRow);
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  internal::SelectedDevice dev;
  RC_TRY(internal::select_device(device, "the mono cold start", &dev));
  R->kernel_ms = 0.0;
  R->focal_rows_used = 0;
  internal::Scratch scratch;
  double *d_px = nullptr, *d_worlds = nullptr, *d_focal = nullptr, *d_rt = nullptr;
  uint8_t *d_has = nullptr, *d_ok = nullptr;
  mi::Scratch S;
  S.F = F;
  CUDA_TRY(scratch.alloc(&d_px, (size_t)F * K * 2));
  CUDA_TRY(scratch.alloc(&d_worlds, (size_t)K * 3));
  CUDA_TRY(scratch.alloc(&d_has, (size_t)F));
  CUDA_TRY(scratch.alloc(&d_ok, (size_t)F));
  CUDA_TRY(scratch.alloc(&d_rt, (size_t)F * 9));
  CUDA_TRY(cudaMemcpy(d_px, P->pixels, (size_t)F * K * 2 * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_worlds, P->worlds, (size_t)K * 3 * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_has, P->has_board, (size_t)F, cudaMemcpyHostToDevice));
  CUDA_TRY(scratch.create_events());
  mi::Intr I;
  if (P->has_init_guess) {                                              // TS.cpp:41
    const double* g = R->intrinsics;
    I = mi::Intr{g[0], g[1], g[2], g[3], g[4], g[5], g[6], g[7], g[8]};
  } else {
    // TS.cpp:43-47: integer halves of the image size, xi = lamda = 0, alpha = 0.5
    I = mi::Intr{0, 0, P->image_width / 2 - 0.5, P->image_height / 2 - 0.5, 0.0, 0.0, 0.5, 0.0, 0.0};
    CUDA_TRY(scratch.alloc(&d_focal, (size_t)F * H));
    CUDA_TRY(cudaEventRecord(scratch.e0, 0));
    mi::k_mi_focal_rows<<<(F * H + mi::kThreads - 1) / mi::kThreads, mi::kThreads>>>(d_px, d_has, F, W, H, I.cx, I.cy, d_focal);
    CUDA_TRY(cudaEventRecord(scratch.e1, 0));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(scratch.add_ms(&R->kernel_ms));
    std::vector<double> focal((size_t)F * H);
    CUDA_TRY(cudaMemcpy(focal.data(), d_focal, focal.size() * sizeof(double), cudaMemcpyDeviceToHost));
    double sum = 0;                                                     // TS.cpp:155-163, frame-major order
    int used = 0;
    for (double v : focal) if (!(v < 0)) { sum += v; ++used; }
    R->focal_rows_used = used;
    I.fx = I.fy = used > 0 ? sum / used : 0.0;
  }
  const double out[9] = {I.fx, I.fy, I.cx, I.cy, I.xi, I.lamda, I.alpha, I.b, I.c};
  std::memcpy(R->intrinsics, out, sizeof(out));
  std::memset(R->mono_rt, 0, sizeof(double) * 9 * (size_t)F);
  std::memset(R->frame_ok, 0, (size_t)F);
  if (!P->has_init_guess && I.fx == 0) return TSCM_OK;  // the caller returns false (TS.cpp:50)
  // warp-per-frame form whenever a frame's scratch fits shared memory (K <= ~350); TSCM_MI_FORM=thread
  // selects the thread-per-frame kernel, which keeps the oracle's statement order (A/B, tests)
  {
    const size_t wb = (mi::mi_warp_smem_bytes(K) + 15) & ~(size_t)15;
    const char* form = std::getenv("TSCM_MI_FORM");
    if (wb * mi::kMiWarps <= 200 * 1024 && !(form && form[0] == 't')) {
      CUDA_TRY(cudaFuncSetAttribute(mi::k_mi_extrinsic_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(wb * mi::kMiWarps)));
      CUDA_TRY(cudaEventRecord(scratch.e0, 0));
      mi::k_mi_extrinsic_warp<<<(F + mi::kMiWarps - 1) / mi::kMiWarps, 32 * mi::kMiWarps, wb * mi::kMiWarps>>>(
          d_px, d_has, d_worlds, F, W, H, I, wb, d_rt, d_ok);
      CUDA_TRY(cudaEventRecord(scratch.e1, 0));
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(scratch.add_ms(&R->kernel_ms));
      CUDA_TRY(cudaMemcpy(R->mono_rt, d_rt, (size_t)F * 9 * sizeof(double), cudaMemcpyDeviceToHost));
      CUDA_TRY(cudaMemcpy(R->frame_ok, d_ok, (size_t)F, cudaMemcpyDeviceToHost));
      return TSCM_OK;
    }
  }
  CUDA_TRY(scratch.alloc(&S.xy, (size_t)2 * K * F));
  CUDA_TRY(scratch.alloc(&S.use, (size_t)K * F));
  // frames per block: as many DLT matrices as fit 200 KB of shared memory (16 at K = 88)
  const size_t a_bytes = (size_t)2 * K * 9 * sizeof(double);
  int fpb = (int)std::min<size_t>(32, (200 * 1024) / a_bytes);
  S.A = nullptr;
  // Shared memory makes a thread 1.45x faster (22 vs 32 ms for its serial chain at K = 88) but caps
  // an SM at `fpb` frames: it pays while all frames fit one wave (5,000 frames: 46 ms in 2.1 waves
  // against 32 ms with every frame resident at once on the global scratch).  TSCM_MI_SMEM=0/1 forces.
  const char* mode = std::getenv("TSCM_MI_SMEM");
  const bool one_wave = fpb >= 4 && (F + fpb - 1) / fpb <= dev.sm_count;
  S.a_in_smem = mode ? (mode[0] == '1' && fpb >= 4) : one_wave;
  size_t smem = 0;
  if (S.a_in_smem) {
    smem = a_bytes * fpb;
    CUDA_TRY(cudaFuncSetAttribute(mi::k_mi_extrinsic, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  } else {
    fpb = mi::kThreads;
    CUDA_TRY(scratch.alloc(&S.A, (size_t)2 * K * 9 * F));
  }
  CUDA_TRY(cudaEventRecord(scratch.e0, 0));
  mi::k_mi_extrinsic<<<(F + fpb - 1) / fpb, fpb, smem>>>(d_px, d_has, d_worlds, F, W, H, I, S, d_rt, d_ok);
  CUDA_TRY(cudaEventRecord(scratch.e1, 0));
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(scratch.add_ms(&R->kernel_ms));
  CUDA_TRY(cudaMemcpy(R->mono_rt, d_rt, (size_t)F * 9 * sizeof(double), cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(R->frame_ok, d_ok, (size_t)F, cudaMemcpyDeviceToHost));
  return TSCM_OK;
}
