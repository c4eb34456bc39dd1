// Test-only C wrapper around MultiCalib::compute_covariance() (tscm_calib_b200/host/), so that
// pytest can drive the C++ adapter's covariance through ctypes.  Built by
// tests/test_covariance_gpu.py; not part of the product library.
#include <cstring>
#include <vector>

#include "../../tscm_calib_b200/host/multi_calib_b200.h"

extern "C" {

// An initialised rig from flat arrays (C-ABI problem layout: views camera-major, every frame
// initialised), MultiCalib::calibrate() and then MultiCalib::compute_covariance(): parameters are
// refined in place, standard deviations out (cam_sd C x 15, board_sd F x 6).  Returns 1 on success.
int multicalib_covariance(int C, int F, int K, int V, const double* board_xy, const int* view_camera,
                          const int* view_frame, const double* obs, double* intr, double* cam_rt,
                          double* board_rt, double* cam_sd, double* board_sd) {
  std::vector<cv::Point3d> worlds(K);
  for (int j = 0; j < K; ++j) worlds[j] = cv::Point3d(board_xy[2 * j], board_xy[2 * j + 1], 0.0);
  std::vector<MultiCalib_camera> cams;
  for (int m = 0; m < C; ++m) {
    std::vector<bool> has(F, false);
    std::vector<std::vector<cv::Point2d>> px(F);
    for (int v = 0; v < V; ++v) {
      if (view_camera[v] != m) continue;
      const int i = view_frame[v];
      has[i] = true;
      px[i].resize(K);
      std::memcpy((void*)px[i].data(), obs + (size_t)v * K * 2, sizeof(double) * 2 * K);
    }
    const double* a = intr + 9 * (size_t)m;
    MultiCalib_camera cam(a[2], a[3], a[0], a[1], a[4], a[5], a[6], a[7], a[8], cv::Mat::eye(3, 3),
                          cv::Mat::zeros(3, 1), has, px);
    std::memcpy(cam.rt_.data(), cam_rt + 6 * (size_t)m, sizeof(double) * 6);
    cams.push_back(cam);
  }
  std::vector<MultiCalib_chessboard> boards;
  for (int i = 0; i < F; ++i) {
    MultiCalib_chessboard b(cv::Mat::eye(3, 3), cv::Mat::zeros(3, 1));
    std::memcpy(b.rt_.data(), board_rt + 6 * (size_t)i, sizeof(double) * 6);
    boards.push_back(b);
  }
  MultiCalib calib(cams, boards, worlds);
  calib.quiet = true;
  calib.calibrate();
  if (!calib.compute_covariance()) return 0;
  for (int m = 0; m < C; ++m) {
    std::memcpy(intr + 9 * (size_t)m, calib.cameras_[m].intrinsic_.data(), sizeof(double) * 9);
    std::memcpy(cam_rt + 6 * (size_t)m, calib.cameras_[m].rt_.data(), sizeof(double) * 6);
    for (int k = 0; k < 15; ++k) cam_sd[15 * (size_t)m + k] = calib.camera_std_dev[m][k];
  }
  for (int i = 0; i < F; ++i) {
    std::memcpy(board_rt + 6 * (size_t)i, calib.chessboards_[i].rt_.data(), sizeof(double) * 6);
    for (int k = 0; k < 6; ++k) board_sd[6 * (size_t)i + k] = calib.board_std_dev[i][k];
  }
  return 1;
}

}  // extern "C"
