/*
 * tscm.h — C-ABI of the B200-native TSCM-Calib calibration solve.
 *
 * This is the drop-in boundary for the ONE path this repo replaces: the two
 * `ceres::Solve` call sites of the reference,
 *
 *   TripleSphereCamera::refinement   /root/reference/TS.cpp:247-282   (mono)
 *   MultiCalib::calibrate            /root/reference/multi_calib.cpp:155-218 (rig)
 *
 * together with the residual functors Ceres differentiates for them
 * (TS.h:100-131, multi_calib.h:146-195).  Everything crosses the boundary as
 * plain pointers and sizes; no C++/torch/OpenCV types, no exceptions.
 *
 * Data conventions (all taken from the reference, units mm / pixels):
 *   intrinsics  C x 9 doubles  {fx, fy, cx, cy, xi, lambda, alpha, b, c}
 *               packing of TS.cpp:53-61 / multi_calib.h:22.  b, c are carried but
 *               never read by the functors (TS.h:122-125, multi_calib.h:175-178).
 *   cam_rt      C x 6 doubles  {angle-axis(3), t(3)}  reference->camera
 *               (MultiCalib_camera::rt_, multi_calib.h:18,70)
 *   board_rt    F x 6 doubles  {angle-axis(3), t(3)}  board->reference
 *               (MultiCalib_chessboard::rt_, multi_calib.h:96,111;
 *                TripleSphereCamera::rt_[i], TS.cpp:72)
 *   A "view" is one (camera m, frame i) pair in which camera m detected the
 *   board.  Views are ordered camera-major, frame-minor — the loop order of
 *   multi_calib.cpp:162-169 — and every view carries exactly K corners
 *   (all-or-nothing detection, main.cpp:33-37).
 *   obs_xy is the concatenation of cameras_[m].pixels()[i] (cv::Point2d =
 *   {double x, y}) over views in that order: num_views x K x 2 doubles.
 *
 * The mono problem (TS.cpp) is the rig problem with C = 1, fixed_camera = 0 and
 * cam_rt = 0: AngleAxisRotatePoint with a zero vector takes its Taylor branch
 * and returns the point bit-exactly, so both functors produce identical
 * residuals.
 */
#ifndef TSCM_H_
#define TSCM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSCM_INTRINSIC_SIZE 9  /* AutoDiffCostFunction<...,9> block, TS.cpp:264 */
#define TSCM_POSE_SIZE 6       /* AutoDiffCostFunction<...,6,6,...>, multi_calib.cpp:180 */

/* ceres::TerminationType values the reference tests against (TS.cpp:281). */
enum {
  TSCM_CONVERGENCE = 0,
  TSCM_NO_CONVERGENCE = 1,
  TSCM_FAILURE = 2
};

/* loss_type: the reference passes NULL (TS.cpp:265, multi_calib.cpp:181,198). */
enum {
  TSCM_LOSS_NONE = 0,
  TSCM_LOSS_HUBER = 1,   /* ceres::HuberLoss(a)  */
  TSCM_LOSS_CAUCHY = 2   /* ceres::CauchyLoss(a) */
};

/* Return codes of every entry point (0 = ok). */
enum {
  TSCM_OK = 0,
  TSCM_ERR_INVALID_ARGUMENT = 1,
  TSCM_ERR_CUDA = 2,          /* CUDA runtime error; tscm_last_error() has the text */
  TSCM_ERR_NO_DEVICE = 3,     /* no sm_100 device: there is NO CPU fallback */
  TSCM_ERR_COMM = 4,          /* NCCL failure */
  TSCM_ERR_UNSUPPORTED = 5,
  TSCM_ERR_NO_CANDIDATE = 6,  /* pose graph: no usable candidate (tscm_pose_graph_init) */
  TSCM_ERR_RANK_DEFICIENT = 7 /* covariance: H is singular (gauge freedom, degenerate board) */
};

/* Size limit: the reduced camera system has NL = 13 C - 6 live parameters (13 C with
 * fixed_camera = -1), and by default it is factored in the shared memory of one thread block.  A
 * solver accepts NL <= 202: at most 16 cameras with one fixed, or 15 with none (16 cameras with none
 * fixed, NL 208, need 233,984 bytes per block, over the 232,448 of a B200).  Larger problems
 * fail with TSCM_ERR_UNSUPPORTED at creation (tscm_solver_create, tscm_solve,
 * tscm_compute_covariance).
 * With tscm_options.allow_large_rigs = 1 the limit is NL <= 416 (32 cameras, with or without a
 * fixed one): systems above 202 are factored by a thread-block cluster of 2-8 CTAs, and their
 * covariance by a factor in global memory.  Sharded solves (num_gpus > 1, tscm_solver_attach_comm,
 * tscm_solver_p2p_attach) stay limited to NL <= 202 and return TSCM_ERR_UNSUPPORTED above. */
typedef struct tscm_problem {
  int32_t num_cameras;        /* C  (cameras_.size(), multi_calib.cpp:157) */
  int32_t num_frames;         /* F  (chessboards_.size(), multi_calib.cpp:158); every frame
                                 must be seen by >= 1 camera (multi_calib.cpp:102,167) */
  int32_t corners_per_board;  /* K  (worlds_.size()) */
  int32_t num_views;          /* number of (camera, frame) pairs with a detection */
  const double* board_xy;     /* K x 2: worlds_[j].x, worlds_[j].y; z is ignored
                                 exactly as in TS.h:107-109 / multi_calib.h:154-156 */
  const int32_t* view_camera; /* num_views: camera index m, non-decreasing */
  const int32_t* view_frame;  /* num_views: frame index i, increasing within a camera */
  const double* obs_xy;       /* num_views x K x 2 observed pixels */
  int32_t fixed_camera;       /* camera whose cam_rt is held constant
                                 (SetParameterBlockConstant, multi_calib.cpp:186): 0 for
                                 the rig and for mono; -1 = none */
} tscm_problem;

/* Solver options.  tscm_options_init() fills the ceres::Solver::Options
 * defaults that are in effect at TS.cpp:271-274 / multi_calib.cpp:209-212. */
typedef struct tscm_options {
  int32_t max_num_iterations;               /* 50 (rig, Ceres default) / 100 (mono, TS.cpp:274) */
  double function_tolerance;                /* 1e-6  */
  double gradient_tolerance;                /* 1e-10 */
  double parameter_tolerance;               /* 1e-8  */
  double initial_trust_region_radius;       /* 1e4   */
  double max_trust_region_radius;           /* 1e16  */
  double min_trust_region_radius;           /* 1e-32 */
  double min_relative_decrease;             /* 1e-3  */
  double min_lm_diagonal;                   /* 1e-6  */
  double max_lm_diagonal;                   /* 1e32  */
  int32_t max_num_consecutive_invalid_steps;/* 5     */
  int32_t jacobi_scaling;                   /* 1     */
  int32_t loss_type;                        /* TSCM_LOSS_NONE */
  double loss_scale;                        /* `a` of HuberLoss(a)/CauchyLoss(a) */
  int32_t parameter_tolerance_needs_successful_step;
                                            /* 0: Ceres <= 2.0 (parameter and function tolerance are
                                               tested on every valid step);
                                               1: Ceres >= 2.1 (both tests only after at least one
                                               successful step) */
  int32_t disable_tolerances;               /* 1: fixed-iteration timing mode — run exactly
                                               max_num_iterations LM iterations */
  int32_t verbose;                          /* 1: print BriefReport() line (TS.cpp:280) */
  int32_t num_gpus;                         /* 0 or 1: one GPU.  N > 1: the frames are sharded over the
                                               N devices [device, device + N) of this process
                                               (SURVEY.md 8b/8e; peer access between them is required).
                                               The reference is single-process, so this is how
                                               MultiCalib::calibrate() reaches more than one GPU. */
  int32_t allow_large_rigs;                 /* 0 (default): NL <= 202 (see "Size limit").  1: NL <= 416,
                                               up to 32 cameras, one GPU above 202.  Fixed when the
                                               solver is created: tscm_solver_set_options refuses a
                                               change with TSCM_ERR_INVALID_ARGUMENT. */
} tscm_options;

typedef struct tscm_summary {
  int32_t termination_type;        /* TSCM_CONVERGENCE / NO_CONVERGENCE / FAILURE */
  int32_t num_iterations;          /* summary.iterations.size(): iteration 0 included */
  int32_t num_successful_steps;    /* iteration 0 counts, as in Ceres */
  int32_t num_unsuccessful_steps;
  double initial_cost;             /* 1/2 sum r^2 (after loss) at the start */
  double final_cost;               /* min over recorded iterations */
  double final_radius;
  /* Optional per-iteration trace, caller-owned, `trace_capacity` entries each
   * (may be NULL).  Entry k describes recorded iteration k. */
  int32_t trace_capacity;
  double* trace_cost;              /* IterationSummary::cost */
  double* trace_radius;            /* IterationSummary::trust_region_radius */
  double* trace_gradient_max_norm; /* IterationSummary::gradient_max_norm */
  double* trace_step_norm;         /* IterationSummary::step_norm */
  int32_t* trace_step_flags;       /* bit0 step_is_valid, bit1 step_is_successful */
} tscm_summary;

void tscm_options_init(tscm_options* options);

/* One-shot solve: the call a reference adapter makes instead of ceres::Solve.
 * Host pointers in, parameters updated in place (as Ceres does through the raw
 * double* it was handed: TS.cpp:266-267, multi_calib.cpp:182-184).  Uses CUDA
 * device `device` (-1 = current device); options->num_gpus > 1 shards the frames over
 * the devices [device, device + num_gpus).
 *
 * The solver built for a problem STRUCTURE (device, C, F, K, the view lists, the board and
 * fixed_camera) is kept after the call, so that the next tscm_solve() on the same structure
 * — a re-calibration with new detections, another LM run from a different start — only
 * uploads observations and parameters: no allocation, no index tables, no graph capture.
 * tscm_cache_configure(0) disables this, tscm_cache_release() frees what is held.  Observations
 * staged in memory from tscm_host_alloc() (page-locked) upload at full PCIe rate. */
int tscm_solve(const tscm_problem* problem, const tscm_options* options,
               double* intrinsics, double* cam_rt, double* board_rt,
               tscm_summary* summary, int device);
void tscm_cache_configure(int32_t max_solvers);   /* default 1; 0 = no caching */
void tscm_cache_release(void);
/* Page-locked host memory for observation staging (cudaHostAlloc / cudaFreeHost).  The last block
 * freed is kept for the next request of at most its size (page-locking 56 MB costs more than a warm
 * solve); tscm_cache_configure(0) disables that, tscm_cache_release() frees it. */
void* tscm_host_alloc(size_t bytes);
void tscm_host_free(void* p);

/* Resident solver: observations stay in HBM between solves. */
typedef struct tscm_solver tscm_solver;

int tscm_solver_create(const tscm_problem* problem, const tscm_options* options,
                       int device, tscm_solver** out);
void tscm_solver_destroy(tscm_solver* solver);
int tscm_solver_set_options(tscm_solver* solver, const tscm_options* options);
/* Host -> device parameter upload / device -> host download. */
int tscm_solver_set_parameters(tscm_solver* solver, const double* intrinsics,
                               const double* cam_rt, const double* board_rt);
int tscm_solver_get_parameters(tscm_solver* solver, double* intrinsics,
                               double* cam_rt, double* board_rt);
/* Replace the observations (host pointer, num_views x K x 2). */
int tscm_solver_set_observations(tscm_solver* solver, const double* obs_xy);
/* Run the LM loop on the parameters currently on the device. */
int tscm_solver_run(tscm_solver* solver, tscm_summary* summary);

/* Multi-GPU: frames are sharded across ranks (each rank's tscm_problem holds
 * only its own frames/views; cameras are replicated).  `unique_id` is the
 * 128-byte ncclUniqueId produced by tscm_comm_unique_id() on rank 0 and
 * broadcast by the host (torch.distributed / MPI / a file). */
int tscm_comm_unique_id(void* unique_id_128);
int tscm_solver_attach_comm(tscm_solver* solver, int rank, int num_ranks,
                            const void* unique_id_128);

/* Multi-GPU on one NVLink/NVSwitch node, one PROCESS per GPU (preferred over NCCL): the two
 * exchange steps of an LM iteration run inside this library's own kernels over peer memory.
 * Every rank exports the 64-byte CUDA-IPC handle of its mailbox, the host gathers the handles
 * of all ranks (rank order, 64 bytes each) and hands them to every rank.  At most 8 ranks.
 * Either attach call makes the solver a rank of a sharded solve; with both, peer memory is
 * used.  The host must put a barrier between the attach calls of all ranks and the first
 * tscm_solver_run(), and every rank must make the same sequence of calls: an exchange waits
 * for its peers on the device and gives up after `tscm_solver_set_exchange_timeout` seconds
 * (default 10 s), which ends the solve with TSCM_FAILURE and returns TSCM_ERR_COMM.
 * (Inside ONE process use tscm_options.num_gpus instead: no IPC, same kernels.) */
int tscm_solver_p2p_export(tscm_solver* solver, void* handle_64);
int tscm_solver_p2p_attach(tscm_solver* solver, int rank, int num_ranks, const void* handles);
int tscm_solver_set_exchange_timeout(tscm_solver* solver, double seconds);

/* ---- parameter covariance ---------------------------------------------------------------
 * The covariance of the estimate at the current parameters x, as ceres::Covariance reports it:
 *   Sigma = H^-1,  H = J^T J,
 * J the Jacobian of all residuals at x with the configured robust loss applied through Ceres'
 * corrector (the J of the LM step), no LM diagonal.  Only LIVE parameters enter: per camera
 * [rt(6) unless it is the fixed camera][fx fy cx cy xi lambda alpha] (the layout of
 * tscm_solver_reduced_system), plus 6 per frame.  Unlike ceres::Covariance on the reference's
 * 9-wide intrinsic block, b and c are excluded: their Jacobian columns are identically zero
 * (TS.h:122-125), so that block would be rank deficient.  The fixed camera's rt has no entries.
 * Returned are the camera block (n x n, n = tscm_solver_reduced_size()) and the 6 x 6 diagonal
 * block of every board pose; camera x board and board x board cross blocks are not computed.
 * It is evaluated as Sigma = D (D H D)^-1 D with the Jacobi scales D of the LM solve:
 *   camera block  D_c S~^-1 D_c,   S~ the undamped scaled reduced camera system,
 *   board f       D_e,f (V~_f^-1 + Y~_f S~^-1 Y~_f^T) D_e,f,   Y~_f = V~_f^-1 W~_f.
 * Sigma is raw, as in Ceres; standard deviations in OpenCV's sense (calibrateCameraExtended) are
 * sqrt(residual_variance * diag(Sigma)) with
 *   residual_variance = sum |r|^2 / (2N - (n + 6F)),
 * r the plain (loss-free) residuals, N observations and F frames over all shards and ranks (NaN
 * when 2N <= n + 6F).
 * TSCM_ERR_RANK_DEFICIENT (nothing written): a pivot of the LDL^T of S~ or of some V~_f is
 * <= 1e-14 x the largest diagonal entry of that matrix (the default
 * min_reciprocal_condition_number of ceres::Covariance) — e.g. fixed_camera = -1 leaves a
 * 6-dimensional gauge freedom, or a board pose is not determined by its views.
 * Host pointers.  The solver's state is unaffected: a later tscm_solver_run() behaves as if this
 * call had not been made. */
typedef struct tscm_covariance {
  double* camera;            /* optional, n x n row-major, n = tscm_solver_reduced_size(), live order */
  double* board;             /* optional, F x 6 x 6 row-major: covariance of board_rt[f] */
  double residual_variance;  /* out: sum |r|^2 / (2N - n_free), plain residuals */
  double kernel_ms;          /* out: device time of the covariance kernels (CUDA events) */
} tscm_covariance;

/* At the parameters on the device (after tscm_solver_run(): the solution).  On a num_gpus group
 * `board` holds all F frames in problem order.  Multi-process ranks: collective like run(); the
 * camera block is identical on every rank, `board` holds the rank's own frames, indexed as in
 * tscm_solver_get_parameters(). */
int tscm_solver_covariance(tscm_solver* solver, tscm_covariance* cov);
/* One-shot form at the given parameters (host pointers, not modified), through the solver cache
 * of tscm_solve(): after a tscm_solve() of the same structure it only uploads observations and
 * parameters — no new solver, no graph capture.  (Named apart from the struct: in C a function
 * and a typedef cannot share the name tscm_covariance.) */
int tscm_compute_covariance(const tscm_problem* problem, const tscm_options* options, const double* intrinsics,
                            const double* cam_rt, const double* board_rt, tscm_covariance* cov,
                            int device);

/* ---- inspection entry points (used by the parity tests and the bench) ---- */

/* One residual + analytic-Jacobian pass at the current device parameters.
 * residuals: N x 2 (N = num_views*K), jacobian: N x 2 x 21 with the column
 * order of AutoDiffCostFunction<...,2,6,6,9> (multi_calib.cpp:177-180):
 * camera_rt(6), chessboard_rt(6), intrinsic(9).  Either may be NULL. Host
 * pointers.  The fixed camera's rt columns are reported as zeros. */
int tscm_solver_eval_jacobian(tscm_solver* solver, double* residuals, double* jacobian,
                              double* cost);
/* Reduced camera system of the next LM step at the current point and radius:
 * lhs n x n (row-major, symmetric, both triangles), rhs n, n = tscm_solver_reduced_size();
 * per camera: [rt(6) unless fixed][fx fy cx cy xi lambda alpha]. */
int tscm_solver_reduced_size(const tscm_solver* solver);
int tscm_solver_reduced_system(tscm_solver* solver, double radius, double* lhs, double* rhs);
/* Mean Euclidean reprojection error per camera and overall, the reference's
 * accuracy read-out (multi_calib.cpp:235-283): per_camera has C entries. */
int tscm_solver_reprojection_error(tscm_solver* solver, double* per_camera, double* overall,
                                   double* rms);
/* Time `repeats` back-to-back launches of one stage on the solver's stream with
 * CUDA events; returns the average milliseconds per launch.
 * stage: 0 = residual+Jacobian+normal-equation kernel, 1 = Schur elimination,
 *        2 = reduced solve, 3 = back-substitution, 4 = whole LM iterations (iteration
 *        zero, then `repeats` replays of the iteration graph; fails if the loop
 *        terminates early), 5 = whole evaluation pass (kernels + reductions),
 *        6 / 7 = the two kernels of stage 0 on their own (k_eval5: moments of every view;
 *        k_view_blocks: per-view blocks from the moments). */
int tscm_solver_time_stage(tscm_solver* solver, int stage, int repeats, double* ms_per_launch);
/* Schur-elimination form (test hook: the default, 0 = chosen from the visibility pattern, is
 * what every production call uses): 1 = dense rows (k_schur_frames + k_schur_update), 2 = fused
 * producer/consumer CTA (k_schur2), 3 = per-camera-pair (k_pair_* + k_schur_pairs2).  Returns
 * TSCM_ERR_UNSUPPORTED when the form cannot hold this problem. */
int tscm_solver_set_schur_form(tscm_solver* solver, int form);
/* Test hook: the kernel of the reduced solve.  0 = chosen from NL (what every production call
 * uses: one CTA up to 202 live parameters, a thread-block cluster above), 1 = one CTA (k_solve;
 * TSCM_ERR_UNSUPPORTED above 202), 2 = cluster (k_solve_cluster, at any size). */
int tscm_solver_set_reduced_solve(tscm_solver* solver, int form);
/* bit 0: creation / solve phase timings on stderr; bit 1: in-kernel cycle counts of k_solve;
 * bit 2: solvers created from now on chain their kernels WITHOUT programmatic dependent launch
 * (A/B timing). */
void tscm_set_debug(int32_t flags);
/* Number of kernels launched by this solver since creation. */
int64_t tscm_solver_launch_count(const tscm_solver* solver);
/* Measured FP64 FMA throughput of the device (TFLOP/s, FMA = 2 flops): the
 * denominator of the FP64 roofline this FP64-bound path is judged against. */
int tscm_device_fp64_peak(int device, double* tflops);

/* ---- remap tables (SURVEY.md 8f #4) --------------------------------------------------
 * The per-pixel loops that fill CV_32FC1 lookup tables through the TS projection:
 *   TripleSphereCamera::undistort             /root/reference/TS.cpp:284-306
 *   TripleSphereCamera::undistort_chessboard  /root/reference/TS.cpp:308-330 (mapx/mapy part)
 *   Remap::init_remap                         /root/reference/EpipolarRectify/rectify.cpp:86-199
 * One job = one rectangular block of the output maps: for block pixel (i, j)
 *   ray  = ((j - ray_cx)/ray_fx, (i - ray_cy)/ray_fy, 1)        TS.cpp:293-295, rectify.cpp:98
 *   P    = matrix * ray                                         rectify.cpp:99, TS.cpp:321-322
 *   (u,v)= TS projection of P with skew b, c                    TS.cpp:332-344
 *          or (-1,-1) when cutoff_w2 > 0 and Z <= -cutoff_w2*|P| rectify.cpp:7,28
 *   mapx[row0+i][col0+j] = (float)(u + offset_x), mapy likewise rectify.cpp:113-114
 * Results are bit-identical to those loops evaluated in IEEE double without FMA
 * contraction.  Host pointers; mapx/mapy are map_height x map_width floats, pixels not
 * covered by any job are left untouched.  At most 64 jobs per call. */
typedef struct tscm_remap_job {
  double intrinsics[TSCM_INTRINSIC_SIZE]; /* source camera {fx,fy,cx,cy,xi,lambda,alpha,b,c} */
  double matrix[9];                       /* row-major 3x3 */
  double ray_fx, ray_fy, ray_cx, ray_cy;
  double offset_x, offset_y;
  double cutoff_w2;                       /* 0 = none (TS.cpp); 0.42399 in rectify.cpp:7 */
  int32_t width, height;                  /* block size */
  int32_t row0, col0;                     /* block origin in the maps */
} tscm_remap_job;

/* kernel_ms (may be NULL): device time of the table kernel, CUDA events. */
int tscm_remap_tables(const tscm_remap_job* jobs, int32_t num_jobs, int32_t map_width,
                      int32_t map_height, float* mapx, float* mapy, int device,
                      double* kernel_ms);

/* ---- pose-graph initialisation (SURVEY.md 8f #2) -------------------------------------
 * MultiCalib's constructor, /root/reference/multi_calib.cpp:6-153, from the per-camera mono
 * results: camera i is chained to camera i-1 through every board both detected
 * (multi_calib.cpp:26-48); each of those n candidate poses is scored by the summed
 * reprojection error (TS.h:58-69) of BOTH cameras over ALL n shared boards
 * (multi_calib.cpp:50-88: n^2 x 2 x K TS projections — the hot loop, on the GPU here) and the
 * smallest sum wins; board poses likewise over the cameras that see them
 * (multi_calib.cpp:95-152).  The candidate errors are bit-identical to those loops evaluated
 * in IEEE double without FMA contraction, so the same candidates win.
 *   intrinsics  C x 9          {fx,fy,cx,cy,xi,lambda,alpha,b,c} of the mono calibrations
 *   has_board   C x B bytes    TripleSphereCamera::has_chessboard(j)
 *   mono_rt     C x B x 9      TripleSphereCamera::Rt(j), row-major 3x3 [r1 r2 t] (TS.cpp:195-201);
 *                              r1, r2 are narrowed to float and r3 = r1 x r2 is a float product,
 *                              as Rt_to_R_t does with cv::Vec3f (multi_calib.h:130-137)
 *   pixels      C x B x K x 2  TripleSphereCamera::pixels()[j]; ignored where has_board = 0
 *   worlds      K x 3
 * Poses come back as 12 doubles: R row-major (9) | t (3) — MultiCalib_camera::R()/t(),
 * MultiCalib_chessboard::R()/t().  Host pointers. */
typedef struct tscm_pose_graph_problem {
  int32_t num_cameras;        /* C */
  int32_t num_boards;         /* B */
  int32_t corners_per_board;  /* K */
  const double* worlds;
  const double* intrinsics;
  const uint8_t* has_board;
  const double* mono_rt;
  const double* pixels;
} tscm_pose_graph_problem;

typedef struct tscm_pose_graph_result {
  double* camera_pose;             /* C x 12, camera 0 = identity (multi_calib.cpp:18-23) */
  double* board_pose;              /* B x 12, untouched where board_initialised = 0 */
  uint8_t* board_initialised;      /* B: 0 for a board no camera saw (multi_calib.cpp:102) */
  int32_t* camera_choice;          /* optional, C: board whose candidate won; -1 for camera 0 */
  int32_t* board_choice;           /* optional, B: camera whose candidate won; -1 = uninitialised */
  double* camera_candidate_error;  /* optional, C x B: summed error of the candidate built from
                                      board j, NaN where the pair (i-1, i) does not share it */
  double* board_candidate_error;   /* optional, B x C: NaN where camera j did not see board i or
                                      the board has one candidate only (multi_calib.cpp:105-113) */
  double kernel_ms;                /* out: device time of the scoring kernels (CUDA events) */
  int64_t projections;             /* out: TS projections evaluated */
} tscm_pose_graph_result;

/* TSCM_ERR_NO_CANDIDATE: two adjacent cameras share no board (the reference indexes Rs[-1]
 * there, multi_calib.cpp:51,86) or no candidate scored below the 1e10 start value. */
int tscm_pose_graph_init(const tscm_pose_graph_problem* problem, int device,
                         tscm_pose_graph_result* result);

/* ---- mono cold start (SURVEY.md 8f #3) ------------------------------------------------
 * TripleSphereCamera::calibrate up to the refinement, /root/reference/TS.cpp:36-52, batched over
 * the frames of one camera:
 *   estimate_focal      TS.cpp:110-168  per board row a circle fit (cv::SVD::solveZ of the 4-column
 *                       design matrix), mean of the accepted rows -> fx = fy
 *   estimate_extrinsic  TS.cpp:170-203  corners lifted to the unit sphere (TS.h:39-57), turned so
 *                       that a corner near the board centre looks down +z, cv::solvePnPRansac
 *                       (defaults, identity camera matrix) on the normalised plane, turned back,
 *                       kept as the 3x3 [r1 r2 t]
 * One GPU thread per (frame, row) for the focal fits, one warp per frame for the pose; no FMA
 * contraction.  The two OpenCV calls are restated (one-sided Jacobi SVD; homography + LM to
 * convergence + inlier re-fitting) and pinned against golden vectors of the real OpenCV.
 *   has_board  F bytes       has_chessboard[k] (a frame without corners: pixels[k].size() == 0)
 *   pixels     F x K x 2     K = board_width * board_height corners, row-major board order
 *   worlds     K x 3
 * has_init_guess = 0: cx, cy = integer halves of the image size - 0.5, xi = lamda = 0, alpha = 0.5
 * (TS.cpp:43-47) and the focal length is estimated; result->intrinsics[0] == 0 means the estimate
 * failed (the reference returns false, TS.cpp:50) and no pose is computed.
 * has_init_guess = 1: result->intrinsics is INPUT (the 7-argument constructor path, TS.cpp:41). */
typedef struct tscm_mono_init_problem {
  int32_t num_frames;                 /* F = pixels.size() */
  int32_t board_width, board_height;  /* chessboard_num */
  int32_t image_width, image_height;  /* img_size */
  const double* worlds;
  const uint8_t* has_board;
  const double* pixels;
  int32_t has_init_guess;
} tscm_mono_init_problem;

typedef struct tscm_mono_init_result {
  double intrinsics[TSCM_INTRINSIC_SIZE]; /* {fx,fy,cx,cy,xi,lambda,alpha,b,c}: in/out, see above */
  double* mono_rt;                    /* F x 9: Rt_[k] row-major, zero where frame_ok = 0 */
  uint8_t* frame_ok;                  /* F: 1 where a pose was found (0: no board, or PnP failed —
                                         NaN rays under the current guess; OpenCV would raise) */
  int32_t focal_rows_used;            /* out: total_num of TS.cpp:156 */
  double kernel_ms;                   /* out: device time of the two kernels (CUDA events) */
} tscm_mono_init_result;

int tscm_mono_init(const tscm_mono_init_problem* problem, int device, tscm_mono_init_result* result);

const char* tscm_last_error(void);
const char* tscm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* TSCM_H_ */
