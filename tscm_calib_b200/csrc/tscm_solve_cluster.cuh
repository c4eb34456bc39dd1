// tscm_solve_cluster.cuh — K4 for reduced systems wider than one CTA holds: the blocked LDL^T of
// k_solve (tscm_solve.cuh) spread over a thread-block cluster of 2-8 CTAs (opt-in,
// tscm_options.allow_large_rigs; DESIGN.md 5f).
//
// k_solve keeps the augmented, padded lower block triangle in the registers of one CTA and the
// panels of the whole factor in its shared memory: 202 live parameters fill a B200's 232,448 bytes.
// Here the tiles are cut into ncta contiguous ranges of the column-major tile order, one per CTA
// (352 tile threads x 4 tiles: 1,408 tiles, so 4 CTAs hold NL = 416, 5,565 tiles), and
//   * step s: the owners of tiles (i, s) eliminate their panel rows exactly as in k_solve and
//     STORE them into the panel buffer of every CTA of the cluster (DSMEM, double-buffered by the
//     parity of s) and into a global copy of the factor (L2-resident, k_solve's panel layout);
//     the owner of tile (s+1, s+1) broadcasts that tile the same way; ONE cluster barrier;
//   * every CTA's pivot warp then factors block s + 1 from its local copies (the look-ahead of
//     k_solve, done redundantly per CTA on identical bits), while the tile owners apply
//     A -= P(i, s) D^-1 P(j, s)^T from the local panel buffer; one __syncthreads makes the new
//     pivot record visible to the CTA before the next panel step.
// No DSMEM access precedes the first cluster barrier (which guarantees that every CTA has
// started): each CTA's pivot warp reads pivot block 0 from M itself.
// The double buffer needs no second cluster barrier: a CTA that writes panel s + 1 has passed
// barrier s, which every CTA reached only after its last read of the buffer of parity s + 1
// (update s - 1).  After the last step CTA 0 alone runs the back-substitution (k_solve's warp,
// reading the factor from global memory) and the tail; the other CTAs exit, no DSMEM access
// follows the last barrier.
// The arithmetic is k_solve's, operation for operation: same ldlt4 / rcp_cubic, same update order
// per tile, same back-substitution; with tail_nt = k_solve's block size also the same per-thread
// partial sums of the tail.  The result is bit-identical to k_solve wherever both run.
#pragma once

#include <cooperative_groups.h>

#include "tscm_solve.cuh"

namespace tscm {

constexpr int kClusterThreads = 384;                       // 11 tile warps + the pivot warp
constexpr int kClusterT = 4;                               // tiles per tile thread
constexpr int kClusterTilesPerCta = kClusterT * (kClusterThreads - 32);
constexpr int kClusterMaxCtas = 8;                         // portable cluster size
constexpr int kLargeRigMaxNL = 416;                        // 32 cameras, none fixed

struct ClusterDims {
  int nbk;        // 4x4 block rows of the augmented, padded matrix
  int ntile;      // nbk (nbk + 1) / 2
  int ncta;       // CTAs of the cluster (2..8)
  int tpc;        // tiles per CTA (the last CTA may hold fewer)
  int tail_nt;    // threads of the tail sums (k_solve's block size where it fits: same partials)
  size_t smem;    // dynamic shared memory per CTA
};

inline ClusterDims cluster_dims(int NL, int C) {
  ClusterDims d;
  d.nbk = (NL + 1 + 3) / 4;
  d.ntile = d.nbk * (d.nbk + 1) / 2;
  d.ncta = std::max(2, (d.ntile + kClusterTilesPerCta - 1) / kClusterTilesPerCta);
  d.tpc = (d.ntile + d.ncta - 1) / d.ncta;
  d.tail_nt = std::min(kClusterThreads, solve_dims(NL, C).NT);
  const size_t doubles = (size_t)2 * 16 * std::max(1, d.nbk - 1)   // panels s, s + 1
                         + (size_t)d.nbk * 10                        // published pivot tiles
                         + (size_t)d.nbk * kPivRec                   // pivot records
                         + (size_t)3 * (NL + 4)                      // x, gsv, sc
                         + (size_t)C * kCamRec                       // camera records
                         + (size_t)C * 169                           // scaled camera blocks U_s
                         + (size_t)4 * 32 + 4;                       // reduction scratch
  d.smem = doubles * sizeof(double) + (size_t)2 * (NL + 4) * sizeof(short) + 16;
  return d;
}

// Lg: [solve_pan_off(nbk, nbk)] the panels of the factor, k_solve's layout (written by every CTA,
// read by CTA 0's back-substitution).  tpc, tail_nt: ClusterDims.
template <int RMAX>   // rows per lane of the back-substitution warp
__global__ void __launch_bounds__(kClusterThreads, 1)
k_solve_cluster(DeviceProblem P, ParamSet ps0, ParamSet ps1, LmState* st, const double* __restrict__ M /*tiles*/,
                const double* __restrict__ scale_c, double* __restrict__ y_c /*[NL]*/, double* Lg, int tpc,
                int tail_nt) {
  pdl_entry();
  if (st->done) return;
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int rank = (int)cluster.block_rank(), ncta = (int)cluster.num_blocks();
  const int sel = st->cur;
  const ParamSet& ps = sel ? ps1 : ps0;     // current x
  const ParamSet& pc = sel ? ps0 : ps1;     // candidate
  extern __shared__ __align__(16) double s_mem[];
  const int NL = P.NL, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, NT = blockDim.x;
  const int nbk = (NL + 1 + 3) >> 2, ntile = (nbk * (nbk + 1)) >> 1;
  const int pbuf = 16 * max(1, nbk - 1);             // one panel buffer (panel 0 is the longest)
  double* Pb = s_mem;                                // [2][pbuf] panels of the current and the next step
  double* Pt = Pb + 2 * pbuf;                        // [nbk][10] published pivot tiles
  double* piv = Pt + nbk * 10;                       // [nbk][kPivRec]
  double* x = piv + nbk * kPivRec;                   // [NL + 4] solution y
  double* gsv = x + NL + 4;                          // [NL + 4] scaled gradient
  double* sc = gsv + NL + 4;                         // [NL + 4] Jacobi scale
  double* s_comm = sc + NL + 4;                      // [C][kCamRec] camera records of the current point
  double* s_U = s_comm + P.C * kCamRec;              // [C][13][13] scaled camera blocks sc_i sc_j U_ij
  double* s_red = s_U + P.C * 169;                   // [32][4] + 4
  short* s_cam = reinterpret_cast<short*>(s_red + 4 * 32 + 4);   // [NL + 4]
  short* s_kk = s_cam + NL + 4;                                  // [NL + 4]
  __shared__ int s_ok;

  // ---- tile ownership and load: tiles [rank tpc, min(ntile, (rank + 1) tpc)) -------------------
  const int NTt = NT - 32;
  const int c0 = rank * tpc, c1 = min(ntile, c0 + tpc);
  constexpr int T = kClusterT;
  int bi[T], bj[T];
  bool valid[T];
  double acc[T][16];
#pragma unroll
  for (int k = 0; k < T; ++k) {
    const int id = c0 + tid + k * NTt;
    valid[k] = id < c1 && tid < NTt;
    bi[k] = bj[k] = -1;
    if (valid[k]) {
      const double2* src = reinterpret_cast<const double2*>(M + (size_t)id * 16);
#pragma unroll
      for (int q = 0; q < 8; ++q) { const double2 v = src[q]; acc[k][2 * q] = v.x; acc[k][2 * q + 1] = v.y; }
      const float D = 2.0f * nbk + 1.0f;
      int j = (int)((D - sqrtf(D * D - 8.0f * (float)id)) * 0.5f);
      j = max(0, min(j, nbk - 1));
      while (j + 1 < nbk && (j + 1) * nbk - ((j + 1) * j) / 2 <= id) ++j;
      while (j * nbk - (j * (j - 1)) / 2 > id) --j;
      bj[k] = j;
      bi[k] = j + (id - (j * nbk - (j * (j - 1)) / 2));
    } else {
#pragma unroll
      for (int e = 0; e < 16; ++e) acc[k][e] = 0.0;
    }
  }
#pragma unroll
  for (int k = 0; k < T; ++k) {
    if (!valid[k] || 4 * bi[k] + 3 < NL) continue;
#pragma unroll
    for (int e = 0; e < 16; ++e) {
      const int r = 4 * bi[k] + (e >> 2), c = 4 * bj[k] + (e & 3);
      if (c >= NL) acc[k][e] = r == c ? 1.0 : 0.0;
      else if (r > NL) acc[k][e] = 0.0;
    }
  }
  const bool pivot_warp = tid >= NTt;
  // a pivot tile as it is before update s - 1, to every CTA (DSMEM: only after the first cluster
  // barrier, which guarantees that every CTA of the cluster has started)
  auto publish_pivot = [&](int b, const double* a) {
    for (int r = 0; r < ncta; ++r) {
      double* t = cluster.map_shared_rank(Pt + 10 * b, r);
      t[0] = a[0];
      t[1] = a[4]; t[2] = a[5];
      t[3] = a[8]; t[4] = a[9]; t[5] = a[10];
      t[6] = a[12]; t[7] = a[13]; t[8] = a[14]; t[9] = a[15];
    }
  };
  auto factor_block = [&](int s, const double* t10) {
    Piv4 f;
    ldlt4(t10, f);
    if (lane == 0) {
      double* pr = piv + kPivRec * s;
      pr[0] = f.i0; pr[1] = f.i1; pr[2] = f.i2; pr[3] = f.i3;
      pr[4] = t10[1]; pr[5] = t10[3]; pr[6] = f.w21; pr[7] = t10[6]; pr[8] = f.w31; pr[9] = f.w32;
      pr[20] = f.l10; pr[21] = f.l20; pr[22] = f.l21; pr[23] = f.l30; pr[24] = f.l31; pr[25] = f.l32;
      const int j0 = 4 * s;
      const bool ok = (j0 >= NL || f.d0 > 0.0) && (j0 + 1 >= NL || f.d1 > 0.0) &&
                      (j0 + 2 >= NL || f.d2 > 0.0) && (j0 + 3 >= NL || f.d3 > 0.0);
      if (!ok) s_ok = 0;
    }
  };
  // pivot block 0: every CTA's pivot warp reads tile 0 from M itself (with the identity padding of
  // the load above), so nothing crosses CTAs before the first cluster barrier.  Its lane 0 owns
  // s_ok: set and cleared by the same thread, published by that barrier.
  if (pivot_warp) {
    constexpr int kLower[10] = {0, 4, 5, 8, 9, 10, 12, 13, 14, 15};
    double t10[10];
#pragma unroll
    for (int e = 0; e < 10; ++e) {
      const int r = kLower[e] >> 2, c = kLower[e] & 3;
      double v = M[kLower[e]];
      if (3 >= NL) {
        if (c >= NL) v = r == c ? 1.0 : 0.0;
        else if (r > NL) v = 0.0;
      }
      t10[e] = v;
    }
    if (lane == 0) s_ok = 1;
    factor_block(0, t10);
  }
  // every CTA has started (DSMEM may be used from here on) and piv[0] is visible to the CTA
  cluster.sync();
  // ---- blocked LDL^T: one cluster barrier and one CTA barrier per block column -----------------
  // (k_solve's last step, P(nbk - 1), has no panel rows and no next pivot: it is left out)
  for (int s = 0; s + 1 < nbk; ++s) {
    const int nrows = 4 * (nbk - 1 - s);
    double* pan = Pb + (s & 1) * pbuf;
    double* pan_g = Lg + solve_pan_off(s, nbk);
    // -- P(s): panel rows to every CTA and to the global factor ---------------------------------------
#pragma unroll
    for (int k = 0; k < T; ++k) {
      if (!valid[k]) continue;
      if (bj[k] == s && bi[k] > s) {
        const double* pr = piv + kPivRec * s + 20;
        const double l10 = pr[0], l20 = pr[1], l21 = pr[2], l30 = pr[3], l31 = pr[4], l32 = pr[5];
        const int b2 = 2 * (bi[k] - s - 1);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          double p[2][4];
#pragma unroll
          for (int a = 0; a < 2; ++a) {
            const double* row = &acc[k][(2 * h + a) * 4];
            const double p0 = row[0];
            const double p1 = fma(-p0, l10, row[1]);
            const double p2 = fma(-p1, l21, fma(-p0, l20, row[2]));
            const double p3 = fma(-p2, l32, fma(-p1, l31, fma(-p0, l30, row[3])));
            p[a][0] = p0; p[a][1] = p1; p[a][2] = p2; p[a][3] = p3;
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int off = c * nrows + h * (nrows >> 1) + b2;
            const double2 v = make_double2(p[0][c], p[1][c]);
            *reinterpret_cast<double2*>(pan_g + off) = v;
            for (int r = 0; r < ncta; ++r) *reinterpret_cast<double2*>(cluster.map_shared_rank(pan + off, r)) = v;
          }
        }
      } else if (bj[k] == s + 1 && bi[k] == s + 1) {
        publish_pivot(s + 1, acc[k]);
      }
    }
    cluster.sync();
    // -- U(s) --------------------------------------------------------------------------------------
    const double g0 = piv[kPivRec * s], g1 = piv[kPivRec * s + 1], g2 = piv[kPivRec * s + 2],
                 g3 = piv[kPivRec * s + 3];
    if (pivot_warp) {
      double t10[10];
#pragma unroll
      for (int e = 0; e < 10; ++e) t10[e] = Pt[10 * (s + 1) + e];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const double2 b01 = *reinterpret_cast<const double2*>(pan + c * nrows);
        const double2 b23 = *reinterpret_cast<const double2*>(pan + c * nrows + (nrows >> 1));
        const double g = c == 0 ? g0 : (c == 1 ? g1 : (c == 2 ? g2 : g3));
        const double fb[4] = {b01.x, b01.y, b23.x, b23.y};
        const double q[4] = {fb[0] * g, fb[1] * g, fb[2] * g, fb[3] * g};
        t10[0] = fma(-fb[0], q[0], t10[0]);
        t10[1] = fma(-fb[1], q[0], t10[1]); t10[2] = fma(-fb[1], q[1], t10[2]);
        t10[3] = fma(-fb[2], q[0], t10[3]); t10[4] = fma(-fb[2], q[1], t10[4]); t10[5] = fma(-fb[2], q[2], t10[5]);
        t10[6] = fma(-fb[3], q[0], t10[6]); t10[7] = fma(-fb[3], q[1], t10[7]); t10[8] = fma(-fb[3], q[2], t10[8]);
        t10[9] = fma(-fb[3], q[3], t10[9]);
      }
      factor_block(s + 1, t10);
    } else {
#pragma unroll
      for (int k = 0; k < T; ++k) {
        if (!valid[k] || bj[k] <= s) continue;
        const double* pi = pan + 2 * (bi[k] - s - 1);
        const double* pj = pan + 2 * (bj[k] - s - 1);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const double2 a01 = *reinterpret_cast<const double2*>(pi + c * nrows);
          const double2 a23 = *reinterpret_cast<const double2*>(pi + c * nrows + (nrows >> 1));
          const double2 b01 = *reinterpret_cast<const double2*>(pj + c * nrows);
          const double2 b23 = *reinterpret_cast<const double2*>(pj + c * nrows + (nrows >> 1));
          const double g = c == 0 ? g0 : (c == 1 ? g1 : (c == 2 ? g2 : g3));
          const double fa[4] = {a01.x, a01.y, a23.x, a23.y};
          const double q[4] = {b01.x * g, b01.y * g, b23.x * g, b23.y * g};
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[k][a * 4 + b] = fma(-fa[a], q[b], acc[k][a * 4 + b]);
        }
      }
    }
    __syncthreads();
  }
  if (rank != 0) return;
  // ---- CTA 0: explicit block inverses, back-substitution, tail (k_solve's code) -----------------
  for (int s = tid; s < nbk; s += NT) {
    double* pr = piv + kPivRec * s;
    const double i0 = pr[0], i1 = pr[1], i2 = pr[2], i3 = pr[3];
    const double w10 = pr[4], w20 = pr[5], w21 = pr[6], w30 = pr[7], w31 = pr[8], w32 = pr[9];
    const int nbc = NL - 4 * s;
    double n[10];
    n[9] = i3;
    n[7] = i2; n[8] = -i2 * (w32 * n[9]);
    n[4] = i1; n[5] = -i1 * (w21 * n[7]); n[6] = -i1 * fma(w21, n[8], w31 * n[9]);
    n[0] = i0; n[1] = -i0 * (w10 * n[4]); n[2] = -i0 * fma(w10, n[5], w20 * n[7]);
    n[3] = -i0 * fma(w10, n[6], fma(w20, n[8], w30 * n[9]));
    if (nbc < 4) { n[3] = n[6] = n[8] = n[9] = 0.0; }
    if (nbc < 3) { n[2] = n[5] = n[7] = 0.0; }
    if (nbc < 2) { n[1] = n[4] = 0.0; }
#pragma unroll
    for (int e = 0; e < 10; ++e) pr[10 + e] = n[e];
  }
  __syncthreads();
  if (warp == 0) {
    // x_k = (y_k - sum_{j > k} P[j][k] x_j) / d_k, lane = row; the factor is read from L2 (.cg: the
    // other CTAs wrote it, ordered by the cluster barriers)
    const int bl = nbk - 1;
    double r[RMAX];
    const double* colb[RMAX];
    int half[RMAX];
#pragma unroll
    for (int m = 0; m < RMAX; ++m) {
      const int k = lane + 32 * m;
      r[m] = 0.0;
      colb[m] = Lg;
      half[m] = 0;
      if (k < NL) {
        const int s = k >> 2;
        const int nr = 4 * (nbk - 1 - s);
        colb[m] = Lg + solve_pan_off(s, nbk) + (k & 3) * nr - 2 * (s + 1);
        half[m] = nr >> 1;
        if (s < bl) {
          const int rr = NL - 4 * (s + 1);
          r[m] = __ldcg(Lg + solve_pan_off(s, nbk) + (k & 3) * nr + ((rr >> 1) & 1) * (nr >> 1) + 2 * (rr >> 2) + (rr & 1));
        }
        else r[m] = piv[kPivRec * bl + piv_widx(NL & 3, k & 3)];
      }
    }
    for (int jb = bl; jb >= 0; --jb) {
      const int j0 = 4 * jb;
      if (j0 >= NL) continue;
      double2 p01[RMAX], p23[RMAX];
#pragma unroll
      for (int m = 0; m < RMAX; ++m) {
        const int k = lane + 32 * m;
        p01[m] = p23[m] = make_double2(0.0, 0.0);
        if (k < j0) {
          const double* col = colb[m] + 2 * jb;
          p01[m] = __ldcg(reinterpret_cast<const double2*>(col));
          p23[m] = __ldcg(reinterpret_cast<const double2*>(col + half[m]));
        }
      }
      const double* nn = piv + kPivRec * jb + 10;
      const double n0 = nn[0], n1 = nn[1], n2 = nn[2], n3 = nn[3], n4 = nn[4], n5 = nn[5], n6 = nn[6],
                   n7 = nn[7], n8 = nn[8], n9 = nn[9];
      const int msel = j0 >> 5, l0 = j0 & 31;
      double rv = r[0];
#pragma unroll
      for (int m = 1; m < RMAX; ++m) rv = msel == m ? r[m] : rv;
      const double r0 = __shfl_sync(0xffffffffu, rv, l0), r1 = __shfl_sync(0xffffffffu, rv, l0 + 1),
                   r2 = __shfl_sync(0xffffffffu, rv, l0 + 2), r3 = __shfl_sync(0xffffffffu, rv, l0 + 3);
      const double x0 = fma(n0, r0, n1 * r1) + fma(n2, r2, n3 * r3);
      const double x1 = fma(n4, r1, n5 * r2) + n6 * r3;
      const double x2 = fma(n7, r2, n8 * r3);
      const double x3 = n9 * r3;
      if (lane == 0) {
        const int nbc = min(4, NL - j0);
        x[j0] = x0;
        if (nbc > 1) x[j0 + 1] = x1;
        if (nbc > 2) x[j0 + 2] = x2;
        if (nbc > 3) x[j0 + 3] = x3;
      }
#pragma unroll
      for (int m = 0; m < RMAX; ++m)
        r[m] -= fma(p01[m].x, x0, p01[m].y * x1) + fma(p23[m].x, x2, p23[m].y * x3);
    }
  } else {
    const int t1 = tid - 32, n1 = NT - 32;
    for (int i = t1; i < NL; i += n1) {
      const int c = P.live_cam[i], kk = P.live_kk[i];
      s_cam[i] = (short)c; s_kk[i] = (short)kk;
      sc[i] = scale_c[c * 13 + kk];
    }
    for (int i = t1; i < P.C * kCamRec; i += n1) s_comm[i] = ps.comm[i];
    __syncwarp();
    asm volatile("bar.sync 1, %0;" ::"r"(n1) : "memory");
    for (int k = t1; k < NL; k += n1) gsv[k] = sc[k] * cam_grad(s_comm + s_cam[k] * kCamRec, s_kk[k]);
    for (int q = t1; q < P.C * 169; q += n1) {
      const int c = q / 169, a = (q % 169) / 13, b = q % 13;
      const int o0 = P.live_off[c], n = P.live_off[c + 1] - o0, sh = 13 - n;
      double v = 0.0;
      if (a >= sh && b >= sh)
        v = sc[o0 + a - sh] * sc[o0 + b - sh] * (a <= b ? cam_block(s_comm + c * kCamRec, a, b)
                                                         : cam_block(s_comm + c * kCamRec, b, a));
      s_U[q] = v;
    }
  }
  __syncthreads();
  // ---- y_c, candidate camera parameters, camera-side partial sums (threads [0, tail_nt)) ----------
  double lin = 0.0, dn2 = 0.0, quad = 0.0, xn2 = 0.0;
  if (tid < tail_nt) {
    for (int i = tid; i < NL; i += tail_nt) {
      const double y = x[i];
      y_c[i] = y;
      lin += y * gsv[i];
      const double delta = -y * sc[i];
      dn2 += delta * delta;
      const int ci = s_cam[i];
      const int o0 = P.live_off[ci], n = P.live_off[ci + 1] - o0;
      const double* Urow = s_U + ci * 169 + s_kk[i] * 13 + (13 - n);
      double row = 0.0;
      for (int t = 0; t < n; ++t) row += Urow[t] * x[o0 + t];
      quad += y * row;
    }
    for (int idx = tid; idx < P.C * 15; idx += tail_nt) {
      const int c = idx / 15, k = idx % 15;
      const bool free_rt = (c != P.fixed_camera);
      const double xv = k < 6 ? ps.cam_rt[c * 6 + k] : ps.intr[c * 9 + (k - 6)];
      double xn = xv;
      if (k < 6) {
        if (free_rt) xn = xv + (-x[P.live_off[c] + k] * sc[P.live_off[c] + k]);
      } else if (k - 6 < 7) {
        const int li = P.live_off[c] + (free_rt ? 6 : 0) + (k - 6);
        xn = xv + (-x[li] * sc[li]);
      }
      if (k < 6) pc.cam_rt[c * 6 + k] = xn; else pc.intr[c * 9 + (k - 6)] = xn;
      if (k >= 6 || free_rt) xn2 += xn * xn;
    }
  }
  double v4[4] = {lin, quad, dn2, xn2};
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v4[q] += __shfl_xor_sync(0xffffffffu, v4[q], o);
  if (lane == 0) {
#pragma unroll
    for (int q = 0; q < 4; ++q) s_red[warp * 4 + q] = v4[q];
  }
  __syncthreads();
  if (tid == 0) {
    double t4[4] = {0.0, 0.0, 0.0, 0.0};
    const int nw = tail_nt >> 5;
    for (int w = 0; w < nw; ++w)
#pragma unroll
      for (int q = 0; q < 4; ++q) t4[q] += s_red[w * 4 + q];
    st->cam_lin = t4[0]; st->cam_quad = t4[1]; st->cam_dn2 = t4[2]; st->cam_xn2 = t4[3];
    st->solve_ok = s_ok;
  }
}

}  // namespace tscm
