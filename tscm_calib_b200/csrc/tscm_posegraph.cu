// tscm_posegraph.cu — tscm_pose_graph_init(): pose-graph initialisation (SURVEY 8f #2),
// multi_calib.cpp:6-153 with both candidate-scoring loops on the GPU (tscm_posegraph.cuh); the O(n)
// pose algebra around them stays on the host.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/tscm.h"
#include "tscm_internal.h"
#include "tscm_posegraph.cuh"

using namespace tscm;
using internal::set_error;

extern "C" int tscm_pose_graph_init(const tscm_pose_graph_problem* P, int device, tscm_pose_graph_result* R) {
  internal::DeviceScope device_scope;
  if (!P || !R || !P->worlds || !P->intrinsics || !P->has_board || !P->mono_rt || !P->pixels ||
      !R->camera_pose || !R->board_pose || !R->board_initialised) {
    set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT;
  }
  const int C = P->num_cameras, B = P->num_boards, K = P->corners_per_board;
  if (C <= 0 || B <= 0 || K <= 0) { set_error("bad pose-graph sizes C=%d B=%d K=%d", C, B, K); return TSCM_ERR_INVALID_ARGUMENT; }
  internal::SelectedDevice dev;
  RC_TRY(internal::select_device(device, "the pose-graph scoring", &dev));
  R->kernel_ms = 0.0;
  R->projections = 0;
  const double nan = std::nan("");
  if (R->camera_candidate_error) std::fill(R->camera_candidate_error, R->camera_candidate_error + (size_t)C * B, nan);
  if (R->board_candidate_error) std::fill(R->board_candidate_error, R->board_candidate_error + (size_t)C * B, nan);
  if (R->camera_choice) std::fill(R->camera_choice, R->camera_choice + C, -1);
  if (R->board_choice) std::fill(R->board_choice, R->board_choice + B, -1);
  std::fill(R->board_initialised, R->board_initialised + B, (uint8_t)0);

  internal::Scratch scratch;
  const size_t px_doubles = (size_t)C * B * K * 2;
  double *d_px = nullptr, *d_worlds = nullptr, *d_base = nullptr, *d_T = nullptr, *d_E = nullptr, *d_err = nullptr;
  int32_t* d_shared = nullptr;
  CUDA_TRY(scratch.alloc(&d_px, px_doubles));
  CUDA_TRY(scratch.alloc(&d_worlds, (size_t)K * 3));
  CUDA_TRY(cudaMemcpy(d_px, P->pixels, px_doubles * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(d_worlds, P->worlds, (size_t)K * 3 * sizeof(double), cudaMemcpyHostToDevice));
  CUDA_TRY(scratch.alloc(&d_base, (size_t)B * 24));
  CUDA_TRY(scratch.alloc(&d_T, (size_t)B * 24));
  CUDA_TRY(scratch.alloc(&d_err, (size_t)B));
  CUDA_TRY(scratch.alloc(&d_shared, (size_t)B));
  CUDA_TRY(scratch.create_events());

  // ---------------- camera chain: multi_calib.cpp:14-93 ----------------
  // candidates per pass: the (board, side) x candidate error matrix is kept below 1 GiB
  size_t E_doubles = 0;
  std::vector<double> cam_pose((size_t)C * 12, 0.0), base, cand, T, err;
  std::vector<int32_t> shared;
  for (int i = 0; i < C; ++i) {
    double* out = cam_pose.data() + 12 * (size_t)i;
    if (i == 0) { out[0] = out[4] = out[8] = 1.0; continue; }      // multi_calib.cpp:18-23
    const double* camk = cam_pose.data() + 12 * (size_t)(i - 1);
    const uint8_t *ha = P->has_board + (size_t)(i - 1) * B, *hb = P->has_board + (size_t)i * B;
    shared.clear();
    for (int j = 0; j < B; ++j) if (ha[j] && hb[j]) shared.push_back(j);
    const int n = (int)shared.size();
    if (n == 0) {
      set_error("cameras %d and %d share no board (give the cameras in adjacent order)", i - 1, i);
      return TSCM_ERR_NO_CANDIDATE;
    }
    base.resize((size_t)n * 24); cand.resize((size_t)n * 12); T.resize((size_t)n * 24); err.resize(n);
    for (int f = 0; f < n; ++f) {
      double* b = base.data() + (size_t)f * 24;
      pg_host::split(P->mono_rt + ((size_t)i * B + shared[f]) * 9, b);             // (Ri | ti)
      pg_host::split(P->mono_rt + ((size_t)(i - 1) * B + shared[f]) * 9, b + 12);  // (Rp | tp)
      pg_host::chain_candidate(b, b + 12, camk, cand.data() + (size_t)f * 12);
      pg_host::chain_transforms(camk, cand.data() + (size_t)f * 12, T.data() + (size_t)f * 24);
    }
    CUDA_TRY(cudaMemcpy(d_base, base.data(), base.size() * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_T, T.data(), T.size() * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_shared, shared.data(), (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice));
    const size_t row = (size_t)2 * n;
    int chunk = (int)std::min<size_t>((size_t)n, std::max<size_t>(kPgThreads, ((size_t)1 << 27) / row / kPgThreads * kPgThreads));
    if (row * chunk > E_doubles) {
      E_doubles = row * chunk;
      CUDA_TRY(scratch.alloc(&d_E, E_doubles));
    }
    // shared boards per CTA: as many as fit 48 KB, fewer while the grid is below 8 CTAs per SM
    int tile = 8;
    while (tile > 1 && pg_pair_smem_bytes(K, tile) > 48 * 1024) --tile;
    const size_t smem1 = pg_pair_smem_bytes(K, 1);
    if (smem1 > 200 * 1024) {
      set_error("K = %d corners per board exceed the shared-memory staging of the scoring kernel", K);
      return TSCM_ERR_UNSUPPORTED;
    }
    if (smem1 > 48 * 1024)
      CUDA_TRY(cudaFuncSetAttribute(k_pg_pair_score, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    for (int c0 = 0; c0 < n; c0 += chunk) {
      const int nc = std::min(chunk, n - c0);
      const int gx = (nc + kPgThreads - 1) / kPgThreads;
      int t = tile;
      while (t > 1 && (int64_t)gx * ((n + t - 1) / t) < (int64_t)dev.sm_count * 8) --t;
      if ((n + t - 1) / t > 65535) {
        set_error("%d shared boards exceed the scoring grid (%d boards per CTA)", n, t);
        return TSCM_ERR_UNSUPPORTED;
      }
      PgPairArgs A;
      A.pixels = d_px; A.shared = d_shared; A.base = d_base; A.cand = d_T + (size_t)c0 * 24;
      A.worlds = d_worlds; A.E = d_E;
      A.intr[0] = pg_intr(P->intrinsics + 9 * (size_t)(i - 1));
      A.intr[1] = pg_intr(P->intrinsics + 9 * (size_t)i);
      A.cam_stride = (int64_t)B * K * 2;
      A.cam[0] = i - 1; A.cam[1] = i;
      A.n = n; A.nc = nc; A.K = K; A.tile = t;
      CUDA_TRY(cudaEventRecord(scratch.e0, 0));
      k_pg_pair_score<<<dim3(gx, (n + t - 1) / t), kPgThreads, pg_pair_smem_bytes(K, t)>>>(A);
      k_pg_sum<<<gx, kPgThreads>>>(d_E, 2 * n, nc, d_err + c0);
      CUDA_TRY(cudaEventRecord(scratch.e1, 0));
      CUDA_TRY(cudaGetLastError());
      CUDA_TRY(scratch.add_ms(&R->kernel_ms));
      R->projections += (int64_t)nc * n * 2 * K;
    }
    CUDA_TRY(cudaMemcpy(err.data(), d_err, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost));
    double min_error = 1e10;                       // multi_calib.cpp:51-52, 82-86
    int min_id = -1;
    for (int c = 0; c < n; ++c) {
      if (R->camera_candidate_error) R->camera_candidate_error[(size_t)i * B + shared[c]] = err[c];
      if (err[c] < min_error) { min_error = err[c]; min_id = c; }
    }
    if (min_id < 0) {
      set_error("camera %d: none of the %d candidate poses scores below 1e10", i, n);
      return TSCM_ERR_NO_CANDIDATE;
    }
    std::memcpy(out, cand.data() + (size_t)min_id * 12, 12 * sizeof(double));
    if (R->camera_choice) R->camera_choice[i] = shared[min_id];
  }
  std::memcpy(R->camera_pose, cam_pose.data(), cam_pose.size() * sizeof(double));

  // ---------------- board poses: multi_calib.cpp:95-152 ----------------
  {
    std::vector<double> bc((size_t)B * C * 12, 0.0), E2((size_t)B * C * C, 0.0);
    for (int i = 0; i < B; ++i)
      for (int j = 0; j < C; ++j) {
        if (!P->has_board[(size_t)j * B + i]) continue;
        double Pb[12];
        pg_host::split(P->mono_rt + ((size_t)j * B + i) * 9, Pb);
        pg_host::board_candidate(cam_pose.data() + 12 * (size_t)j, Pb, bc.data() + ((size_t)i * C + j) * 12);
      }
    double *d_bc = nullptr, *d_cam = nullptr, *d_intr = nullptr, *d_E2 = nullptr;
    uint8_t* d_has = nullptr;
    CUDA_TRY(scratch.alloc(&d_bc, bc.size()));
    CUDA_TRY(scratch.alloc(&d_cam, cam_pose.size()));
    CUDA_TRY(scratch.alloc(&d_intr, (size_t)C * 9));
    CUDA_TRY(scratch.alloc(&d_E2, E2.size()));
    CUDA_TRY(scratch.alloc(&d_has, (size_t)C * B));
    CUDA_TRY(cudaMemcpy(d_bc, bc.data(), bc.size() * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_cam, cam_pose.data(), cam_pose.size() * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_intr, P->intrinsics, (size_t)C * 9 * sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(d_has, P->has_board, (size_t)C * B, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemset(d_E2, 0, E2.size() * sizeof(double)));      // (board, candidate, camera) triples without a view stay 0
    PgBoardArgs A;
    A.pixels = d_px; A.has = d_has; A.cam_pose = d_cam; A.cand = d_bc; A.worlds = d_worlds; A.intr = d_intr;
    A.E = d_E2; A.C = C; A.B = B; A.K = K;
    const int64_t total = (int64_t)B * C * C;
    CUDA_TRY(cudaEventRecord(scratch.e0, 0));
    k_pg_board_score<<<(unsigned)((total + kPgThreads - 1) / kPgThreads), kPgThreads>>>(A);
    CUDA_TRY(cudaEventRecord(scratch.e1, 0));
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(scratch.add_ms(&R->kernel_ms));
    CUDA_TRY(cudaMemcpy(E2.data(), d_E2, E2.size() * sizeof(double), cudaMemcpyDeviceToHost));
    std::vector<int> id;
    for (int i = 0; i < B; ++i) {
      id.clear();
      for (int j = 0; j < C; ++j) if (P->has_board[(size_t)j * B + i]) id.push_back(j);
      const int m = (int)id.size();
      if (m == 0) continue;                          // multi_calib.cpp:102
      int min_id = 0;
      if (m > 1) {                                   // multi_calib.cpp:128-149
        double min_error = 1e10;
        min_id = -1;
        for (int c = 0; c < m; ++c) {
          double error = 0;
          for (int k = 0; k < m; ++k) error += E2[((size_t)i * C + id[c]) * C + id[k]];
          if (R->board_candidate_error) R->board_candidate_error[(size_t)i * C + id[c]] = error;
          if (error < min_error) { min_error = error; min_id = c; }
        }
        R->projections += (int64_t)m * m * K;
        if (min_id < 0) {
          set_error("board %d: none of the %d candidate poses scores below 1e10", i, m);
          return TSCM_ERR_NO_CANDIDATE;
        }
      }
      std::memcpy(R->board_pose + 12 * (size_t)i, bc.data() + ((size_t)i * C + id[min_id]) * 12, 12 * sizeof(double));
      R->board_initialised[i] = 1;
      if (R->board_choice) R->board_choice[i] = id[min_id];
    }
  }
  return TSCM_OK;
}

