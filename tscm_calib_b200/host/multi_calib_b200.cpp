// multi_calib_b200.cpp — see multi_calib_b200.h.
#include "multi_calib_b200.h"

#include <cmath>
#include <cstdio>
#include <cstring>
#include <iostream>
#include <utility>

namespace {

cv::Mat vec3(double a, double b, double c) {
  cv::Mat m(3, 1);
  m.at<double>(0, 0) = a; m.at<double>(1, 0) = b; m.at<double>(2, 0) = c;
  return m;
}

std::vector<double> pack_rt(const cv::Mat& R, const cv::Mat& t) {
  cv::Mat r;
  cv::Rodrigues(R, r);
  return {r.at<double>(0, 0), r.at<double>(1, 0), r.at<double>(2, 0),
          t.at<double>(0, 0), t.at<double>(1, 0), t.at<double>(2, 0)};
}

}  // namespace

MultiCalib_camera::MultiCalib_camera(double cx, double cy, double fx, double fy, double xi, double lamda,
                                     double alpha, double b, double c, cv::Mat R, cv::Mat t,
                                     std::vector<bool> has_chessboard,
                                     std::vector<std::vector<cv::Point2d>> pixel_coordinates) {
  rt_ = pack_rt(R, t);
  R_ = R; t_ = t;
  intrinsic_ = {fx, fy, cx, cy, xi, lamda, alpha, b, c};
  has_chessboard_ = std::move(has_chessboard);
  pixel_coordinates_ = std::move(pixel_coordinates);
  is_initial_ = true;
  // R_, t_ stay the matrices that were handed in (multi_calib.h:20-21): the pose-graph chain
  // composes them as they are, not their re-orthogonalised Rodrigues round trip
  intrinsic_matrix_ = cv::Mat(1, 9);
  for (int k = 0; k < 9; ++k) intrinsic_matrix_.at<double>(0, k) = intrinsic_[k];
}

void MultiCalib_camera::update_param() {
  cv::Rodrigues(vec3(rt_[0], rt_[1], rt_[2]), R_);
  t_ = vec3(rt_[3], rt_[4], rt_[5]);
  intrinsic_matrix_ = cv::Mat(1, 9);
  for (int k = 0; k < 9; ++k) intrinsic_matrix_.at<double>(0, k) = intrinsic_[k];
}

MultiCalib_chessboard::MultiCalib_chessboard(cv::Mat R, cv::Mat t) {
  rt_ = pack_rt(R, t);
  R_ = R; t_ = t;
  is_initial_ = true;
}

void MultiCalib_chessboard::update_param() {
  cv::Rodrigues(vec3(rt_[0], rt_[1], rt_[2]), R_);
  t_ = vec3(rt_[3], rt_[4], rt_[5]);
}

void MultiCalib::init_options() {
  tscm_options_init(&options_);          // Ceres defaults: 50 iterations (multi_calib.cpp:209-212)
  options_.verbose = 1;                  // summary.BriefReport() (multi_calib.cpp:218)
  std::memset(&summary_, 0, sizeof(summary_));
}

// Pose-graph initialisation (multi_calib.cpp:6-153): camera i is chained to camera i-1 through
// every board both see, the candidate with the smallest summed reprojection error wins; board
// poses likewise over the cameras that see them.  The exhaustive candidate scoring
// (multi_calib.cpp:50-88, 128-149: n^2 x 2 x K projections per camera pair) runs on the GPU
// through tscm_pose_graph_init(); there is no CPU path.
MultiCalib::MultiCalib(std::vector<TripleSphereCamera> cameras, const std::vector<cv::Point3d>& worlds, int device_) {
  init_options();
  device = device_;
  worlds_ = worlds;
  const int camera_num = (int)cameras.size();
  const int board_num = camera_num ? (int)cameras[0].has_chessboard().size() : 0;
  const int K = (int)worlds.size();
  cameras_.resize(camera_num);
  chessboards_.resize(board_num);
  if (camera_num == 0 || board_num == 0 || K == 0) return;
  std::vector<double> w(3 * (size_t)K), intr(9 * (size_t)camera_num), rt(9 * (size_t)camera_num * board_num, 0.0),
      px(2 * (size_t)camera_num * board_num * K, 0.0);
  std::vector<uint8_t> has((size_t)camera_num * board_num, 0), board_ok(board_num, 0);
  for (int j = 0; j < K; ++j) { w[3 * j] = worlds[j].x; w[3 * j + 1] = worlds[j].y; w[3 * j + 2] = worlds[j].z; }
  for (int m = 0; m < camera_num; ++m) {
    TripleSphereCamera& cam = cameras[m];
    const double in[9] = {cam.fx(), cam.fy(), cam.cx(), cam.cy(), cam.xi(), cam.lamda(), cam.alpha(), cam.b(), cam.c()};
    std::memcpy(intr.data() + 9 * (size_t)m, in, sizeof(in));
    const auto& pixels = cam.pixels_ref();
    for (int i = 0; i < board_num; ++i) {
      const size_t v = (size_t)m * board_num + i;
      if (!cam.has_chessboard(i)) continue;
      if ((int)pixels[i].size() != K) {
        std::cout << "[tscm] camera " << m << ", board " << i << ": " << pixels[i].size() << " corners, expected " << K << std::endl;
        return;
      }
      has[v] = 1;
      const cv::Mat Rt = cam.Rt(i);
      for (int k = 0; k < 9; ++k) rt[9 * v + k] = Rt.at<double>(k / 3, k % 3);
      for (int j = 0; j < K; ++j) { px[(v * K + j) * 2] = pixels[i][j].x; px[(v * K + j) * 2 + 1] = pixels[i][j].y; }
    }
  }
  std::vector<double> cam_pose(12 * (size_t)camera_num), board_pose(12 * (size_t)board_num, 0.0);
  tscm_pose_graph_problem prob;
  prob.num_cameras = camera_num; prob.num_boards = board_num; prob.corners_per_board = K;
  prob.worlds = w.data(); prob.intrinsics = intr.data(); prob.has_board = has.data();
  prob.mono_rt = rt.data(); prob.pixels = px.data();
  tscm_pose_graph_result res;
  std::memset(&res, 0, sizeof(res));
  res.camera_pose = cam_pose.data(); res.board_pose = board_pose.data(); res.board_initialised = board_ok.data();
  const int rc = tscm_pose_graph_init(&prob, device, &res);
  if (rc != TSCM_OK) {
    // the reference prints and returns (multi_calib.cpp:31-35) or indexes Rs[-1] (multi_calib.cpp:51,86)
    std::cout << "[tscm] pose-graph initialisation failed: " << tscm_last_error() << std::endl;
    return;
  }
  pose_graph_kernel_ms = res.kernel_ms;
  auto mat = [](const double* p, int rows, int cols) {
    cv::Mat M(rows, cols);
    for (int r = 0; r < rows; ++r) for (int c = 0; c < cols; ++c) M.at<double>(r, c) = p[r * cols + c];
    return M;
  };
  for (int m = 0; m < camera_num; ++m) {
    TripleSphereCamera& cam = cameras[m];
    const double* p = cam_pose.data() + 12 * (size_t)m;
    cameras_[m] = MultiCalib_camera(cam.cx(), cam.cy(), cam.fx(), cam.fy(), cam.xi(), cam.lamda(), cam.alpha(), cam.b(),
                                    cam.c(), mat(p, 3, 3), mat(p + 9, 3, 1), cam.has_chessboard(), cam.pixels());
  }
  for (int i = 0; i < board_num; ++i) {
    if (!board_ok[i]) continue;                       // multi_calib.cpp:102
    const double* p = board_pose.data() + 12 * (size_t)i;
    chessboards_[i] = MultiCalib_chessboard(mat(p, 3, 3), mat(p + 9, 3, 1));
  }
}

// Replaces multi_calib.cpp:155-284.
bool MultiCalib::compute_covariance() {
  const int C = (int)cameras_.size(), B = (int)chessboards_.size(), K = (int)worlds_.size();
  std::vector<double> board_xy(2 * (size_t)K);
  for (int j = 0; j < K; ++j) { board_xy[2 * j] = worlds_[j].x; board_xy[2 * j + 1] = worlds_[j].y; }
  // the problem calibrate() solves: views (m, i) with an initialised board detected by camera m
  std::vector<int> frame_id(B, -1);
  std::vector<char> used(B, 0);
  for (int m = 0; m < C; ++m) {
    const auto& px = cameras_[m].pixels_ref();
    for (int i = 0; i < B; ++i)
      if (chessboards_[i].is_initial() && (int)px[i].size() == K) used[i] = 1;
  }
  int F = 0;
  for (int i = 0; i < B; ++i) if (used[i]) frame_id[i] = F++;
  std::vector<int32_t> view_camera, view_frame;
  std::vector<double> obs;
  for (int m = 0; m < C; ++m) {
    const auto& px = cameras_[m].pixels_ref();
    for (int i = 0; i < B; ++i) {
      if (frame_id[i] < 0 || (int)px[i].size() != K) continue;
      view_camera.push_back(m);
      view_frame.push_back(frame_id[i]);
      const double* d = reinterpret_cast<const double*>(px[i].data());   // cv::Point2d = {x, y}
      obs.insert(obs.end(), d, d + 2 * (size_t)K);
    }
  }
  if (F == 0 || view_camera.empty()) return false;
  std::vector<double> intr(9 * (size_t)C), cam_rt(6 * (size_t)C), board_rt(6 * (size_t)F);
  for (int m = 0; m < C; ++m) {
    std::memcpy(&intr[9 * m], cameras_[m].intrinsic_.data(), sizeof(double) * 9);
    std::memcpy(&cam_rt[6 * m], cameras_[m].rt_.data(), sizeof(double) * 6);
  }
  for (int i = 0; i < B; ++i)
    if (frame_id[i] >= 0) std::memcpy(&board_rt[6 * frame_id[i]], chessboards_[i].rt_.data(), sizeof(double) * 6);
  tscm_problem p;
  p.num_cameras = C; p.num_frames = F; p.corners_per_board = K; p.num_views = (int)view_camera.size();
  p.board_xy = board_xy.data(); p.view_camera = view_camera.data(); p.view_frame = view_frame.data();
  p.obs_xy = obs.data();
  p.fixed_camera = 0;
  const int n = 6 * (C - 1) + 7 * C;
  std::vector<double> cam_cov((size_t)n * n), board_cov(36 * (size_t)F);
  tscm_covariance cov;
  cov.camera = cam_cov.data(); cov.board = board_cov.data();
  cov.residual_variance = 0.0; cov.kernel_ms = 0.0;
  tscm_options opt = options_;
  opt.verbose = 0;
  const int rc = tscm_compute_covariance(&p, &opt, intr.data(), cam_rt.data(), board_rt.data(), &cov, device);
  if (rc != TSCM_OK) {
    if (!quiet) std::cout << "[tscm] covariance failed: " << tscm_last_error() << std::endl;
    return false;
  }
  const double s2 = cov.residual_variance;
  residual_variance = s2;
  camera_std_dev.assign(C, std::vector<double>(15, 0.0));
  int o = 0;
  for (int m = 0; m < C; ++m) {
    for (int k = (m == 0 ? 6 : 0); k < 13; ++k, ++o) camera_std_dev[m][k] = std::sqrt(s2 * cam_cov[(size_t)o * n + o]);
  }
  board_std_dev.assign(B, std::vector<double>(6, 0.0));
  for (int i = 0; i < B; ++i)
    if (frame_id[i] >= 0)
      for (int k = 0; k < 6; ++k) board_std_dev[i][k] = std::sqrt(s2 * board_cov[36 * (size_t)frame_id[i] + 7 * k]);
  return true;
}

void MultiCalib::calibrate() {
  const int C = (int)cameras_.size(), B = (int)chessboards_.size(), K = (int)worlds_.size();
  std::vector<double> board_xy(2 * (size_t)K);
  for (int j = 0; j < K; ++j) { board_xy[2 * j] = worlds_[j].x; board_xy[2 * j + 1] = worlds_[j].y; }
  // Residual blocks exist for (camera m, board i) iff the board is initialised and the
  // camera detected it (pixels[i] non-empty): multi_calib.cpp:162-169.  Boards that end up
  // with no view are not part of the problem.
  std::vector<int> frame_id(B, -1);
  std::vector<int32_t> view_camera, view_frame;
  std::vector<char> used(B, 0);
  for (int m = 0; m < C; ++m) {
    const auto& px = cameras_[m].pixels_ref();
    for (int i = 0; i < B; ++i)
      if (chessboards_[i].is_initial() && (int)px[i].size() == K) used[i] = 1;
  }
  int F = 0;
  for (int i = 0; i < B; ++i) if (used[i]) frame_id[i] = F++;
  for (int m = 0; m < C; ++m) {
    const auto& px = cameras_[m].pixels_ref();
    for (int i = 0; i < B; ++i) {
      if (!chessboards_[i].is_initial() || (int)px[i].size() != K) continue;
      view_camera.push_back(m);
      view_frame.push_back(frame_id[i]);
    }
  }
  if (F == 0 || view_camera.empty()) { std::cout << "[tscm] nothing to calibrate" << std::endl; return; }
  // the detections are packed into page-locked staging memory (tscm_host_alloc), so that the
  // upload inside tscm_solve() runs at the full PCIe rate; pageable memory if that fails
  const size_t obs_doubles = view_camera.size() * 2 * (size_t)K;
  double* pinned = static_cast<double*>(tscm_host_alloc(obs_doubles * sizeof(double)));
  std::vector<double> pageable;
  if (!pinned) pageable.resize(obs_doubles);
  double* obs = pinned ? pinned : pageable.data();
  {
    size_t o = 0;
    for (int m = 0; m < C; ++m) {
      const auto& px = cameras_[m].pixels_ref();
      for (int i = 0; i < B; ++i) {
        if (!chessboards_[i].is_initial() || (int)px[i].size() != K) continue;
        std::memcpy(obs + o, px[i].data(), sizeof(double) * 2 * K);   // cv::Point2d = {x, y}
        o += 2 * (size_t)K;
      }
    }
  }
  std::vector<double> intr(9 * (size_t)C), cam_rt(6 * (size_t)C), board_rt(6 * (size_t)F);
  for (int m = 0; m < C; ++m) {
    std::memcpy(&intr[9 * m], cameras_[m].intrinsic_.data(), sizeof(double) * 9);
    std::memcpy(&cam_rt[6 * m], cameras_[m].rt_.data(), sizeof(double) * 6);
  }
  for (int i = 0; i < B; ++i)
    if (frame_id[i] >= 0) std::memcpy(&board_rt[6 * frame_id[i]], chessboards_[i].rt_.data(), sizeof(double) * 6);

  tscm_problem p;
  p.num_cameras = C; p.num_frames = F; p.corners_per_board = K; p.num_views = (int)view_camera.size();
  p.board_xy = board_xy.data(); p.view_camera = view_camera.data(); p.view_frame = view_frame.data();
  p.obs_xy = obs;
  p.fixed_camera = 0;                     // SetParameterBlockConstant(cameras_[0].rt_), multi_calib.cpp:186
  std::memset(&summary_, 0, sizeof(summary_));
  tscm_options opt = options_;
  if (quiet) opt.verbose = 0;
  const int rc = tscm_solve(&p, &opt, intr.data(), cam_rt.data(), board_rt.data(), &summary_, device);
  tscm_host_free(pinned);
  if (rc != TSCM_OK) { std::cout << "[tscm] calibrate failed: " << tscm_last_error() << std::endl; return; }
  for (int m = 0; m < C; ++m) {
    std::memcpy(cameras_[m].intrinsic_.data(), &intr[9 * m], sizeof(double) * 9);
    std::memcpy(cameras_[m].rt_.data(), &cam_rt[6 * m], sizeof(double) * 6);
    if (cameras_[m].is_initial()) cameras_[m].update_param();
  }
  for (int i = 0; i < B; ++i) {
    if (frame_id[i] >= 0) std::memcpy(chessboards_[i].rt_.data(), &board_rt[6 * frame_id[i]], sizeof(double) * 6);
    if (chessboards_[i].is_initial()) chessboards_[i].update_param();
  }
  // mean Euclidean reprojection error per camera and overall (multi_calib.cpp:235-283)
  camera_reprojection_error.assign(C, 0.0);
  double error_sum = 0; long total = 0;
  for (int m = 0; m < C; ++m) {
    const auto& px = cameras_[m].pixels_ref();
    cv::Mat Rc = cameras_[m].R(), tc = cameras_[m].t();
    double error = 0; long cnt = 0;
    for (int i = 0; i < B; ++i) {
      if (!chessboards_[i].is_initial()) continue;
      cv::Mat Rb = chessboards_[i].R(), tb = chessboards_[i].t();
      for (size_t j = 0; j < px[i].size(); ++j) {
        double w[3], q[3];
        for (int r = 0; r < 3; ++r)
          w[r] = Rb.at<double>(r, 0) * worlds_[j].x + Rb.at<double>(r, 1) * worlds_[j].y +
                 Rb.at<double>(r, 2) * worlds_[j].z + tb.at<double>(r, 0);
        for (int r = 0; r < 3; ++r)
          q[r] = Rc.at<double>(r, 0) * w[0] + Rc.at<double>(r, 1) * w[1] + Rc.at<double>(r, 2) * w[2] + tc.at<double>(r, 0);
        const double r2 = q[0] * q[0] + q[1] * q[1];
        const double d1 = std::sqrt(r2 + q[2] * q[2]);
        const double z1 = q[2] + cameras_[m].xi() * d1;
        const double d2 = std::sqrt(r2 + z1 * z1);
        const double z2 = z1 + cameras_[m].lamda() * d2;
        const double d3 = std::sqrt(r2 + z2 * z2);
        const double den = z2 + cameras_[m].alpha() / (1 - cameras_[m].alpha()) * d3;
        const double u = cameras_[m].fx() * q[0] / den + cameras_[m].b() * q[1] / den + cameras_[m].cx();
        const double v = cameras_[m].c() * q[0] / den + cameras_[m].fy() * q[1] / den + cameras_[m].cy();
        error += std::sqrt((px[i][j].x - u) * (px[i][j].x - u) + (px[i][j].y - v) * (px[i][j].y - v));
        ++cnt; ++total;
      }
    }
    error_sum += error;
    camera_reprojection_error[m] = cnt ? error / cnt : 0.0;
    if (!quiet) std::cout << "camera_" << m << " reprojection error: " << camera_reprojection_error[m] << std::endl;
  }
  average_reprojection_error = total ? error_sum / total : 0.0;
  if (!quiet) std::cout << "average reproject error: " << average_reprojection_error << std::endl;
}

// cv::FileStorage(YAML) dialect of main.cpp:305-319: "%YAML:1.0", one !!opencv-matrix per key.
bool MultiCalib::write_yaml(const std::string& filename) {
  FILE* f = std::fopen(filename.c_str(), "w");
  if (!f) return false;
  auto emit = [&](const char* name, int rows, int cols, const double* v) {
    std::fprintf(f, "%s: !!opencv-matrix\n   rows: %d\n   cols: %d\n   dt: d\n   data: [ ", name, rows, cols);
    for (int k = 0; k < rows * cols; ++k) {
      char buf[40];
      if (v[k] == std::floor(v[k]) && std::fabs(v[k]) < 1e15) std::snprintf(buf, sizeof(buf), "%.0f.", v[k]);
      else std::snprintf(buf, sizeof(buf), "%.16e", v[k]);
      std::fprintf(f, "%s%s", buf, k + 1 < rows * cols ? ((k % 2 == 1) ? ",\n       " : ", ") : " ]\n");
    }
  };
  std::fprintf(f, "%%YAML:1.0\n---\n");
  for (size_t i = 0; i < cameras_.size(); ++i) {
    char key[16];
    std::snprintf(key, sizeof(key), "cam%d", (int)i);
    emit(key, 1, 9, cameras_[i].intrinsic_.data());
    std::snprintf(key, sizeof(key), "Twc%d", (int)i);
    cv::Mat R = cameras_[i].R(), t = cameras_[i].t();
    double T[12];
    for (int r = 0; r < 3; ++r) {
      for (int c = 0; c < 3; ++c) T[4 * r + c] = R.at<double>(r, c);
      T[4 * r + 3] = t.at<double>(r, 0);
    }
    emit(key, 3, 4, T);
  }
  std::fclose(f);
  return true;
}
