// multi_calib_b200.h — drop-in `MultiCalib` whose joint refinement runs on the B200.
//
// Mirrors /root/reference/multi_calib.h:9-129 (MultiCalib_camera, MultiCalib_chessboard,
// MultiCalib: same public members and method names).  MultiCalib::calibrate()
// (multi_calib.cpp:155-284) keeps its contract — parameters refined in place in
// cameras_[m].intrinsic_/rt_ and chessboards_[i].rt_, update_param(), BriefReport line and
// the per-camera mean reprojection error printed — but the ceres::Problem / ceres::Solve
// body is replaced by one tscm_solve() call.  write_yaml() reproduces the calibration file
// of main.cpp:293-319 (cam%d 1x9, Twc%d 3x4 [R|t]) in cv::FileStorage's YAML dialect.
#pragma once

#include <string>
#include <vector>

#include "../../include/tscm.h"
#include "cv_compat.h"
#include "ts_camera.h"

class MultiCalib_camera {
 public:
  MultiCalib_camera() {}
  MultiCalib_camera(double cx, double cy, double fx, double fy, double xi, double lamda, double alpha,
                    double b, double c, cv::Mat R, cv::Mat t, std::vector<bool> has_chessboard,
                    std::vector<std::vector<cv::Point2d>> pixel_coordinates);
  bool is_initial() { return is_initial_; }
  bool has_chessboard(int id) { return has_chessboard_[id]; }
  std::vector<std::vector<cv::Point2d>> pixels() { return pixel_coordinates_; }
  const std::vector<std::vector<cv::Point2d>>& pixels_ref() const { return pixel_coordinates_; }
  void update_Rt(cv::Mat R, cv::Mat t) { R_ = R; t_ = t; }
  void update_param();
  cv::Mat R() { return R_; }
  cv::Mat t() { return t_; }
  double cx() { return intrinsic_[2]; }
  double cy() { return intrinsic_[3]; }
  double fx() { return intrinsic_[0]; }
  double fy() { return intrinsic_[1]; }
  double xi() { return intrinsic_[4]; }
  double lamda() { return intrinsic_[5]; }
  double alpha() { return intrinsic_[6]; }
  double b() { return intrinsic_[7]; }
  double c() { return intrinsic_[8]; }
  std::vector<double> intrinsic_;   // fx fy cx cy xi lambda alpha b c   (multi_calib.h:22)
  std::vector<double> rt_;          // angle-axis, t                     (multi_calib.h:18)
  cv::Mat intrinsic_matrix_;        // 1x9, what the YAML writer stores  (multi_calib.h:32)
 private:
  std::vector<bool> has_chessboard_;
  std::vector<std::vector<cv::Point2d>> pixel_coordinates_;
  cv::Mat R_, t_;
  bool is_initial_ = false;
};

class MultiCalib_chessboard {
 public:
  MultiCalib_chessboard() {}
  MultiCalib_chessboard(cv::Mat R, cv::Mat t);
  bool is_initial() { return is_initial_; }
  void update_param();
  cv::Mat R() { return R_; }
  cv::Mat t() { return t_; }
  std::vector<double> rt_;
 private:
  cv::Mat R_, t_;
  bool is_initial_ = false;
};

class MultiCalib {
 public:
  // Pose-graph initialisation of multi_calib.cpp:6-153 from per-camera mono calibrations; the
  // candidate scoring runs on CUDA device `device` (-1 = current), tscm_pose_graph_init().
  MultiCalib(std::vector<TripleSphereCamera> cameras, const std::vector<cv::Point3d>& worlds, int device = -1);
  // Already-initialised rig (the members are public in the reference as well).
  MultiCalib(std::vector<MultiCalib_camera> cameras, std::vector<MultiCalib_chessboard> chessboards,
             const std::vector<cv::Point3d>& worlds)
      : cameras_(cameras), chessboards_(chessboards), worlds_(worlds) { init_options(); }
  ~MultiCalib() {}
  void calibrate();
  // main.cpp:293-319.  Returns false when the file cannot be written.
  bool write_yaml(const std::string& filename);
  // Parameter uncertainties at the current parameters (call it after calibrate()), through
  // tscm_compute_covariance() with options() (so num_gpus applies): fills camera_std_dev and
  // board_std_dev with sqrt(residual_variance * diag(Sigma)), OpenCV's stdDeviations.  Returns
  // false (and leaves them untouched) when there is nothing to compute or the covariance fails,
  // e.g. TSCM_ERR_RANK_DEFICIENT.
  bool compute_covariance();
  // C x 15: [rt 6 | fx fy cx cy xi lambda alpha b c]; 0 where not free (camera 0's rt, b, c)
  std::vector<std::vector<double>> camera_std_dev;
  // B x 6: board pose [angle-axis 3 | t 3]; 0 for boards that are not part of the problem
  std::vector<std::vector<double>> board_std_dev;
  double residual_variance = 0.0;
  std::vector<MultiCalib_camera> cameras_;
  std::vector<MultiCalib_chessboard> chessboards_;
  std::vector<cv::Point3d> worlds_;

  tscm_options& options() { return options_; }
  const tscm_summary& last_summary() const { return summary_; }
  // read-out of the last calibrate(): multi_calib.cpp:235-283
  std::vector<double> camera_reprojection_error;
  double average_reprojection_error = 0.0;
  int device = -1;
  bool quiet = false;
  double pose_graph_kernel_ms = 0.0;   // device time of the constructor's scoring kernels

 private:
  void init_options();
  tscm_options options_;
  tscm_summary summary_;
};
