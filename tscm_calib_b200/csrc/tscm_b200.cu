// tscm_b200.cu — C-ABI implementation (include/tscm.h) of the solver and host orchestration
// of the device-side Levenberg-Marquardt loop.  The host never touches a
// residual: it uploads the problem, captures one LM iteration as a CUDA graph,
// replays it, and reads back the summary.  There is no CPU fallback.
//
// Replaces: ceres::Solve at /root/reference/TS.cpp:278 and multi_calib.cpp:216.
//
// Besides the solver this file holds the error text, the device check and the device scope that
// every translation unit shares (tscm_internal.h).  The remap tables (tscm_remap.cu), the pose
// graph (tscm_posegraph.cu) and the mono cold start (tscm_monoinit.cu) have their own files.
//
// Host-side structure:
//   * one tscm_solver per device ("shard"): every buffer lives in ONE arena allocation, every
//     static index table in ONE uploaded blob, so that creating a solver is a handful of CUDA
//     calls;
//   * a group solver (tscm_options.num_gpus > 1) owns one shard per device of this process and
//     drives them from the calling thread; the shards exchange through the peer-memory kernels
//     of tscm_p2p.cuh over directly mapped peer pointers;
//   * tscm_solve() keeps the solver of the last problem structure (tscm_cache_configure).

#include <cuda_runtime.h>
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/tscm.h"
#include "tscm_kernels.cuh"
#include "tscm_eval5.cuh"
#include "tscm_solve.cuh"
#include "tscm_solve_cluster.cuh"
#include "tscm_p2p.cuh"
#include "tscm_schur_pairs.cuh"
#include "tscm_pair_lists.h"
#include "tscm_covariance.cuh"
#include "tscm_internal.h"

using tscm::internal::set_error;

namespace {

thread_local std::string g_last_error;
int g_debug = 0;     // tscm_set_debug(): bit 0 phase timings on stderr, bit 1 k_solve cycle counts

using Clock = std::chrono::steady_clock;
double ms_since(Clock::time_point t0) {
  return std::chrono::duration<double, std::milli>(Clock::now() - t0).count();
}

// ---------------------------------------------------------------------------
// NCCL through dlopen: the process that hosts us (PyTorch) already carries an
// NCCL; binding at run time avoids a second copy with clashing symbols.
// ---------------------------------------------------------------------------
struct NcclApi {
  typedef struct { char internal[128]; } UniqueId;
  typedef void* Comm;
  int (*GetUniqueId)(UniqueId*) = nullptr;
  int (*CommInitRank)(Comm*, int, UniqueId, int) = nullptr;
  int (*CommDestroy)(Comm) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, Comm, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
};
constexpr int kNcclFloat64 = 8;  // ncclDouble
constexpr int kNcclSum = 0, kNcclMax = 2;

NcclApi& nccl() {
  static NcclApi api;
  static std::once_flag once;
  std::call_once(once, []() {
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return;
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(h, "ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(h, "ncclCommDestroy");
    api.AllReduce = (decltype(api.AllReduce))dlsym(h, "ncclAllReduce");
    api.GroupStart = (decltype(api.GroupStart))dlsym(h, "ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))dlsym(h, "ncclGroupEnd");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(h, "ncclGetErrorString");
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce &&
             api.GroupStart && api.GroupEnd;
  });
  return api;
}

// Device properties are queried once per device (cudaGetDeviceProperties costs ~2 ms).
struct DeviceInfo {
  bool queried = false;
  int major = 0, minor = 0, sm_count = 0;
  size_t smem_optin = 0;
};
int device_info(int device, DeviceInfo* out) {
  static std::mutex mu;
  static DeviceInfo table[64];
  std::lock_guard<std::mutex> lock(mu);
  if (device < 0 || device >= 64) { set_error("device %d out of range", device); return TSCM_ERR_INVALID_ARGUMENT; }
  DeviceInfo& d = table[device];
  if (!d.queried) {
    CUDA_TRY(cudaDeviceGetAttribute(&d.major, cudaDevAttrComputeCapabilityMajor, device));
    CUDA_TRY(cudaDeviceGetAttribute(&d.minor, cudaDevAttrComputeCapabilityMinor, device));
    CUDA_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, device));
    int optin = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    d.smem_optin = (size_t)optin;
    d.queried = true;
  }
  *out = d;
  return TSCM_OK;
}

// All device buffers of a solver: requests are collected, then served by one cudaMalloc and
// zeroed by one memset.
struct Arena {
  struct Req { void** slot; size_t bytes, off; };
  std::vector<Req> reqs;
  size_t total = 0;
  char* base = nullptr;
  template <typename T>
  void want(T** slot, size_t n) {
    size_t b = std::max<size_t>(1, n) * sizeof(T);
    b = (b + 255) & ~(size_t)255;
    reqs.push_back(Req{reinterpret_cast<void**>(slot), b, total});
    total += b;
  }
  int commit(cudaStream_t st) {
    CUDA_TRY(cudaMalloc((void**)&base, std::max<size_t>(256, total)));
    CUDA_TRY(cudaMemsetAsync(base, 0, std::max<size_t>(256, total), st));
    for (const Req& r : reqs) *r.slot = base + r.off;
    return TSCM_OK;
  }
};
// Static index tables: appended on the host, uploaded with one copy.
struct Blob {
  struct Fix { const void** slot; size_t off; };
  std::vector<char> bytes;
  std::vector<Fix> fixes;
  char* d_base = nullptr;
  template <typename T>
  void add(const T** slot, const T* data, size_t n) {
    const size_t off = (bytes.size() + 15) & ~(size_t)15;
    bytes.resize(off + std::max<size_t>(1, n) * sizeof(T));
    if (n) std::memcpy(bytes.data() + off, data, n * sizeof(T));
    fixes.push_back(Fix{reinterpret_cast<const void**>(slot), off});
  }
  template <typename T>
  void add(const T** slot, const std::vector<T>& v) { add(slot, v.data(), v.size()); }
  int upload(cudaStream_t st) {
    CUDA_TRY(cudaMemcpyAsync(d_base, bytes.data(), bytes.size(), cudaMemcpyHostToDevice, st));
    for (const Fix& f : fixes) *f.slot = d_base + f.off;
    CUDA_TRY(cudaStreamSynchronize(st));      // `bytes` is pageable and about to go away
    return TSCM_OK;
  }
};

}  // namespace

using namespace tscm;

enum { kSchurAuto = 0, kSchurRows = 1, kSchurFused = 2, kSchurPairs = 3 };

// A run of consecutive views of one camera: where a shard's observations sit in the caller's array.
struct ObsSegment { int dst_view, src_view, count; };

struct tscm_solver {
  int device = 0;
  int sm_count = 148;
  size_t smem_optin = 0;
  cudaStream_t stream = nullptr;
  tscm_options options{};
  LmOptions lm{};
  DeviceProblem P{};
  ParamSet ps[2]{};
  LmState* d_state = nullptr;
  LmState* h_state = nullptr;       // pinned: [0] final state, [1], [2] pipelined polls
  int* h_err = nullptr;             // pinned: exchange error flag
  char* h_trace = nullptr;          // pinned staging of the trace block
  Trace trace{};
  char* d_trace = nullptr;          // [4][capacity] doubles | [capacity] ints
  int trace_capacity = 0;
  bool x_in_set1 = false;           // host-side knowledge of LmState::cur after the last run
  // device memory
  Arena arena;
  std::vector<void*> extra;         // later allocations (forced Schur form, bigger trace)
  double2* d_obs_in = nullptr;      // staging: reference layout [V][K]
  double2* d_obsT = nullptr;
  double* d_scale_e = nullptr;
  double* d_scale_c = nullptr;
  double* d_Spart = nullptr;
  double* d_rpart = nullptr;
  double* d_Sr = nullptr;
  double* d_yc = nullptr;
  double* d_mom = nullptr;          // [ntiles][188][32] moments of the evaluation in flight (k_eval5 -> k_view_blocks)
  double* d_fcg = nullptr;          // [ntiles][27][32] frame constants of the evaluation in flight
  double* d_bs_part = nullptr;
  double* d_gmax_part = nullptr;
  double* d_xn2_part = nullptr;
  unsigned int* d_ticket = nullptr;
  double* d_comm_stage = nullptr;   // NCCL fallback: staged evaluation record (+ gmax)
  char* d_blob = nullptr;
  // Schur elimination
  SchurArgs schur{};
  Schur2Args schur2{};
  SchurSplitArgs split{};
  PairArgs pairs{};
  int schur_form = kSchurAuto;      // the form in use (never kSchurAuto after creation)
  size_t split_smem = 0, schur2_smem = 0;
  int schur2_nt = 0;
  int schur_nblk = 0, schur_nt = 256, schur_ept = 1;
  SolveDims solve{};
  // reduced solve (tscm_solve_cluster.cuh): single CTA up to kCovMaxNL live parameters, cluster above
  bool use_cluster = false;         // the form in use (tscm_solver_set_reduced_solve forces one)
  ClusterDims cluster{};
  double* d_cluster_L = nullptr;    // [solve_pan_off(nbk, nbk)] factor panels of k_solve_cluster
  size_t eval5_smem = 0;
  E5Items e5items{};
  int want_err = 0;                 // accumulate sum sqrt(s) (reprojection read-out only)
  int bs_nblk = 0, fg_nblk = 0, post_lpf = 8;
  double* d_cam_sum_part = nullptr;
  // graph of one LM iteration (and of kGroupIters iterations, group shards only)
  cudaGraphExec_t graph_exec = nullptr, graph_exec_n = nullptr;
  bool graph_dirty = true;
  int launches_per_iter = 0;
  bool use_pdl = true;              // tscm_set_debug bit 2 turns it off (A/B timing)
  bool pdl = false;                 // launches carry the programmatic-dependent-launch attribute (graph capture)
  cudaEvent_t poll_ev[2] = {nullptr, nullptr};
  // comm
  NcclApi::Comm comm = nullptr;
  int rank = 0, num_ranks = 1;
  // NVLink peer-memory exchange (tscm_p2p.cuh): mailbox of this rank, mappings of the peers
  bool p2p_on = false;
  double* d_mailbox = nullptr;      // own cudaMalloc: its IPC handle is exported
  unsigned long long* d_p2p_seq = nullptr;
  unsigned int* d_p2p_ticket = nullptr;
  int* d_p2p_err = nullptr;
  void* p2p_ipc[kP2PMaxRanks] = {};
  P2PArgs p2p{};
  int64_t launches = 0;
  // host copies
  int C = 0, F = 0, K = 0, V = 0;
  std::vector<int> h_view_camera, h_view_frame, h_frame_ptr, h_frame_views, h_live_off;
  std::vector<double> h_board;
  int fixed_camera = 0;
  std::vector<double> obs_count;    // [C] observations per camera: local (ranks) or global (group shards)
  // group (num_gpus > 1): this object is a facade, the shards do the work
  std::vector<tscm_solver*> kids;
  std::vector<int> kid_frame;       // [n + 1] frame range of every shard
  std::vector<std::vector<ObsSegment>> kid_seg;
  bool is_kid = false;
  // covariance (tscm_solver_covariance), allocated on first use
  double* d_cov_fac = nullptr;      // [NL][NL] LDL^T factor of S~, mirrored
  double* d_cov_sinv = nullptr;     // [NL][NL] S~^-1 (scaled)
  double* d_cov_cam = nullptr;      // [NL][NL] camera block, unscaled
  double* d_cov_board = nullptr;    // [F][36] board blocks, unscaled
  double* d_cov_tri = nullptr;      // packed lower triangle of S~ for the factor above kCovMaxNL
  int* d_cov_flag = nullptr;
  cudaEvent_t cov_ev[2] = {nullptr, nullptr};
};

namespace {

constexpr int kGroupIters = 4;      // LM iterations per graph launch of a group shard

void fill_lm_options(const tscm_options& o, LmOptions& lm) {
  lm.max_num_iterations = o.max_num_iterations;
  lm.function_tolerance = o.function_tolerance;
  lm.gradient_tolerance = o.gradient_tolerance;
  lm.parameter_tolerance = o.parameter_tolerance;
  lm.initial_radius = o.initial_trust_region_radius;
  lm.max_radius = o.max_trust_region_radius;
  lm.min_radius = o.min_trust_region_radius;
  lm.min_relative_decrease = o.min_relative_decrease;
  lm.min_lm_diagonal = o.min_lm_diagonal;
  lm.max_lm_diagonal = o.max_lm_diagonal;
  lm.max_num_consecutive_invalid_steps = o.max_num_consecutive_invalid_steps;
  lm.jacobi_scaling = o.jacobi_scaling;
  lm.loss_type = o.loss_type;
  lm.loss_scale = o.loss_scale;
  lm.ptol_needs_success = o.parameter_tolerance_needs_successful_step;
  lm.disable_tolerances = o.disable_tolerances;
}
bool lm_equal(const LmOptions& a, const LmOptions& b) {
  return a.max_num_iterations == b.max_num_iterations && a.function_tolerance == b.function_tolerance &&
         a.gradient_tolerance == b.gradient_tolerance && a.parameter_tolerance == b.parameter_tolerance &&
         a.initial_radius == b.initial_radius && a.max_radius == b.max_radius && a.min_radius == b.min_radius &&
         a.min_relative_decrease == b.min_relative_decrease && a.min_lm_diagonal == b.min_lm_diagonal &&
         a.max_lm_diagonal == b.max_lm_diagonal &&
         a.max_num_consecutive_invalid_steps == b.max_num_consecutive_invalid_steps &&
         a.jacobi_scaling == b.jacobi_scaling && a.loss_type == b.loss_type && a.loss_scale == b.loss_scale &&
         a.ptol_needs_success == b.ptol_needs_success && a.disable_tolerances == b.disable_tolerances;
}

int validate_options(const tscm_options* o) {
  if (o->max_num_iterations < 0 || !(o->initial_trust_region_radius > 0.0) ||
      (o->loss_type != TSCM_LOSS_NONE && !(o->loss_scale > 0.0)) || o->loss_type < 0 ||
      o->loss_type > TSCM_LOSS_CAUCHY || o->num_gpus < 0 || o->num_gpus > kP2PMaxRanks ||
      (o->allow_large_rigs != 0 && o->allow_large_rigs != 1)) {
    set_error("invalid options");
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  return TSCM_OK;
}

// The limits of the opt-in to reduced systems wider than one CTA holds, from the host tables alone
// (before any device is touched).  Without the opt-in create_shard applies the default limit.
int validate_large_rig(const tscm_problem* p, const tscm_options* o) {
  if (!o->allow_large_rigs) return TSCM_OK;
  const int NL = 13 * p->num_cameras - (p->fixed_camera >= 0 ? 6 : 0);
  if (NL > kLargeRigMaxNL) {
    set_error("reduced system of %d live parameters (%d cameras) exceeds the limit of %d of allow_large_rigs "
              "(32 cameras with none fixed)", NL, p->num_cameras, kLargeRigMaxNL);
    return TSCM_ERR_UNSUPPORTED;
  }
  if (NL > kCovMaxNL && o->num_gpus > 1) {
    set_error("reduced system of %d live parameters: sharded solves (num_gpus > 1) support at most %d", NL,
              kCovMaxNL);
    return TSCM_ERR_UNSUPPORTED;
  }
  return TSCM_OK;
}

int validate_problem(const tscm_problem* p, bool need_obs) {
  if (!p) { set_error("problem is NULL"); return TSCM_ERR_INVALID_ARGUMENT; }
  if (p->num_cameras <= 0 || p->num_frames <= 0 || p->corners_per_board <= 0 || p->num_views <= 0) {
    set_error("empty problem: C=%d F=%d K=%d views=%d", p->num_cameras, p->num_frames,
              p->corners_per_board, p->num_views);
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  if (!p->board_xy || !p->view_camera || !p->view_frame || (need_obs && !p->obs_xy)) {
    set_error("problem has NULL arrays");
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  if (p->fixed_camera < -1 || p->fixed_camera >= p->num_cameras) {
    set_error("fixed_camera %d out of range", p->fixed_camera);
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  std::vector<char> seen(p->num_frames, 0);
  for (int v = 0; v < p->num_views; ++v) {
    const int m = p->view_camera[v], i = p->view_frame[v];
    if (m < 0 || m >= p->num_cameras || i < 0 || i >= p->num_frames) {
      set_error("view %d references camera %d / frame %d out of range", v, m, i);
      return TSCM_ERR_INVALID_ARGUMENT;
    }
    if (v > 0) {
      const int pm = p->view_camera[v - 1], pi = p->view_frame[v - 1];
      if (m < pm || (m == pm && i <= pi)) {
        set_error("views must be ordered camera-major with increasing frames (view %d)", v);
        return TSCM_ERR_INVALID_ARGUMENT;
      }
    }
    seen[i] = 1;
  }
  for (int i = 0; i < p->num_frames; ++i)
    if (!seen[i]) {
      set_error("frame %d is seen by no camera (drop it: multi_calib.cpp:102,167)", i);
      return TSCM_ERR_INVALID_ARGUMENT;
    }
  return TSCM_OK;
}

// ---------------------------------------------------------------------------
// kernel launches of one shard
// ---------------------------------------------------------------------------
// Every launch goes through here.  While the iteration graph is captured (s->pdl) the kernels
// are chained with programmatic dependent launch: see pdl_entry() in tscm_kernels.cuh.
template <typename... KArgs, typename... Args>
void launch_k(tscm_solver* s, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = s->pdl ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
  s->launches += 1;
}

// The residual + Jacobian + normal-equation pass: k_eval5 (moments of every view) followed by
// k_view_blocks (per-view blocks from the moments).
// part: 0 = the whole pass, 1 = k_eval5 only, 2 = k_view_blocks only (stage timing).
void launch_eval_kernel(tscm_solver* s, int which, int part = 0) {
  const DeviceProblem& P = s->P;
  const int ntiles = (P.V + 31) / 32;
  if (part != 2) {
    launch_k(s, k_eval5, dim3(std::min(ntiles, s->sm_count)), dim3(kE5Threads), (size_t)(s->eval5_smem), 
        P, s->ps[0], s->ps[1], s->d_state, which, s->lm, s->want_err, s->d_mom, s->d_fcg, s->e5items);
  }
  if (part != 1) {
    launch_k(s, k_view_blocks, dim3(ntiles), dim3(kVbThreads), (size_t)(vb_smem_bytes()), P, s->ps[0], s->ps[1], s->d_state, which,
                                                                      s->d_mom, s->d_fcg, s->e5items);
  }
}

// which: 0 = current, 1 = candidate (relative to st->cur); 2/3 = absolute set 0/1.
// prep: run k_prep_cams first (the iteration graph does not: k_backsub's extra block already
// wrote the candidate's constants).  decide: fold the accept/reject decision into the tail block
// (single GPU; with several GPUs the records are exchanged first and the decision follows).
void launch_evaluation(tscm_solver* s, int which, int initial, bool prep = true, bool decide = false) {
  const DeviceProblem& P = s->P;
  cudaStream_t st = s->stream;
  if (prep) {
    launch_k(s, k_prep_cams, dim3((P.C + 31) / 32), dim3(32), (size_t)(0), P, s->ps[0], s->ps[1], s->d_state, which);
  }
  launch_eval_kernel(s, which);
  PostArgs a;
  a.gmax_part = s->d_gmax_part; a.xn2_part = s->d_xn2_part;
  a.bs_part = s->d_bs_part; a.bs_nblk = s->bs_nblk; a.fg_nblk = s->fg_nblk;
  a.cam_sum_part = s->d_cam_sum_part; a.lanes_per_frame = s->post_lpf;
  a.ticket = s->d_ticket; a.initial = initial; a.decide = decide ? 1 : 0;
  launch_k(s, k_post_eval, dim3(P.C * kPostSplit + s->fg_nblk), dim3(kPostThreads), (size_t)(0), P, s->ps[0], s->ps[1], s->d_state, which,
                                                            s->lm, s->trace, a);
}

// Global sums of the evaluation record.  The record lives in ps[sel].comm; the selection is
// only known on the device.
int launch_eval_allreduce(tscm_solver* s, int which, bool decide = false) {
  if (s->num_ranks <= 1) return TSCM_OK;
  if (s->p2p_on) {
    launch_k(s, k_xchg_eval, dim3(1), dim3(kXchgThreads), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, which, s->lm,
                                                    s->trace, s->p2p, decide ? 1 : 0);
    return TSCM_OK;
  }
  // The record of the set the device selects is staged through a fixed buffer: only that
  // record may be summed (the current point's is already global).
  NcclApi& n = nccl();
  const int cnt = s->P.C * kCamRec + kCommExtra;
  const int blocks = (cnt + 1 + 255) / 256;
  launch_k(s, k_comm_stage, dim3(blocks), dim3(256), (size_t)(0), s->ps[0], s->ps[1], s->d_state, which, cnt, s->d_comm_stage, 0);
  n.GroupStart();
  int rc = n.AllReduce(s->d_comm_stage, s->d_comm_stage, (size_t)cnt, kNcclFloat64, kNcclSum, s->comm, s->stream);
  if (rc) { set_error("ncclAllReduce(sum) failed: %d", rc); n.GroupEnd(); return TSCM_ERR_COMM; }
  rc = n.AllReduce(s->d_comm_stage + cnt, s->d_comm_stage + cnt, 1, kNcclFloat64, kNcclMax, s->comm, s->stream);
  if (rc) { set_error("ncclAllReduce(max) failed: %d", rc); n.GroupEnd(); return TSCM_ERR_COMM; }
  rc = n.GroupEnd();
  if (rc) { set_error("ncclGroupEnd failed: %d", rc); return TSCM_ERR_COMM; }
  launch_k(s, k_comm_stage, dim3(blocks), dim3(256), (size_t)(0), s->ps[0], s->ps[1], s->d_state, which, cnt, s->d_comm_stage, 1);
  return TSCM_OK;
}

void launch_schur(tscm_solver* s, double radius_override) {
  SchurArgs a = s->schur;
  a.radius_override = radius_override;
  if (s->schur_form == kSchurRows) {
    SchurSplitArgs b = s->split;
    b.a = a;
    launch_k(s, k_schur_frames, dim3((s->F + kSfWarps - 1) / kSfWarps), dim3(32 * kSfWarps), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, s->lm, b);
    if (s->schur_ept == 1)
      launch_k(s, k_schur_update<1>, dim3(s->schur_nblk), dim3(s->schur_nt), (size_t)(s->split_smem), s->P, s->d_state, b);
    else
      launch_k(s, k_schur_update<2>, dim3(s->schur_nblk), dim3(s->schur_nt), (size_t)(s->split_smem), s->P, s->d_state, b);
  } else if (s->schur_form == kSchurPairs) {
    SchurSplitArgs b = s->split;
    b.a = a;
    launch_k(s, k_pair_frames, dim3((s->F + 31) / 32), dim3(256), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, s->lm, b);
    launch_k(s, k_pair_blocks, dim3((s->V * 16 + 255) / 256), dim3(256), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, b);
    launch_k(s, k_schur_pairs2, dim3(s->sm_count), dim3(kPairWarps * 32), (size_t)(kPair2Smem), s->d_state, s->pairs);
    launch_k(s, k_reduce_pairs, dim3(s->pairs.npairs), dim3(kPairReduceGroups * kPairPart), (size_t)(0), s->P, s->d_state, s->pairs);
  } else {
    Schur2Args b = s->schur2;
    b.a = a;
    launch_k(s, k_schur2, dim3(s->schur_nblk), dim3(s->schur2_nt), (size_t)(s->schur2_smem), s->P, s->ps[0], s->ps[1],
                                                                        s->d_state, s->lm, b);
  }
  const int n = s->P.Q + s->P.NL;
  const int nparts = s->schur_form == kSchurPairs ? 1 : s->schur_nblk;   // k_reduce_pairs leaves one complete partial
  AssembleArgs g;
  g.scale_c = s->d_scale_c; g.radius_override = radius_override; g.nbk = s->solve.nbk;
  g.add_cam = (s->num_ranks > 1 && !s->p2p_on) ? 0 : 1;                  // NCCL: after the all-reduce
  if (s->p2p_on && s->num_ranks > 1)
    launch_k(s, k_reduce_s_p2p, dim3((n + 31) / 32), dim3(kReduceThreads), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, s->lm,
                                                                    s->d_Spart, s->d_rpart, nparts, s->d_Sr, g, s->p2p);
  else
    launch_k(s, k_reduce_s, dim3((n + 31) / 32), dim3(kReduceThreads), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, s->lm,
                                                                s->d_Spart, s->d_rpart, nparts, s->d_Sr, g);
}

int launch_schur_allreduce(tscm_solver* s, double radius_override) {
  if (s->num_ranks <= 1 || s->p2p_on) return TSCM_OK;   // P2P: exchanged inside k_reduce_s_p2p
  NcclApi& n = nccl();
  int rc = n.AllReduce(s->d_Sr, s->d_Sr, (size_t)s->solve.ntile * 16, kNcclFloat64, kNcclSum, s->comm, s->stream);
  if (rc) { set_error("ncclAllReduce(S) failed: %d", rc); return TSCM_ERR_COMM; }
  AssembleArgs g;
  g.scale_c = s->d_scale_c; g.radius_override = radius_override; g.nbk = s->solve.nbk; g.add_cam = 1;
  const int cnt = s->P.Q + s->P.NL;
  launch_k(s, k_add_cam_terms, dim3((cnt + 255) / 256), dim3(256), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, s->lm, s->d_Sr, g);
  return TSCM_OK;
}

// k_solve_cluster: a cluster of ncta CTAs, with programmatic dependent launch like every kernel
void launch_solve_cluster(tscm_solver* s) {
  const ClusterDims& d = s->cluster;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(d.ncta); cfg.blockDim = dim3(kClusterThreads); cfg.dynamicSmemBytes = d.smem;
  cfg.stream = s->stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = d.ncta; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = s->pdl ? 2 : 1;
  auto kernel = s->P.NL <= 32 * 7 ? k_solve_cluster<7> : k_solve_cluster<13>;
  cudaLaunchKernelEx(&cfg, kernel, s->P, s->ps[0], s->ps[1], s->d_state, (const double*)s->d_Sr,
                     (const double*)s->d_scale_c, s->d_yc, s->d_cluster_L, d.tpc, d.tail_nt);
  s->launches += 1;
}

void launch_solve(tscm_solver* s) {
  if (s->use_cluster) { launch_solve_cluster(s); return; }
  const SolveDims& d = s->solve;
  const int prof = (g_debug & 2) ? 1 : 0;
  if (d.T == 1)
    launch_k(s, k_solve<1, 4>, dim3(1), dim3(d.NT), (size_t)(d.smem), s->P, s->ps[0], s->ps[1], s->d_state, s->d_Sr, s->d_scale_c,
                                                   s->d_yc, prof);
  else
    launch_k(s, k_solve<4, 7>, dim3(1), dim3(d.NT), (size_t)(d.smem), s->P, s->ps[0], s->ps[1], s->d_state, s->d_Sr, s->d_scale_c,
                                                   s->d_yc, prof);
}

void launch_backsub(tscm_solver* s) {
  // one extra block prepares the derived constants of the candidate cameras
  launch_k(s, k_backsub, dim3(s->bs_nblk + 1), dim3(kBacksubThreads), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state,
                                                              s->schur, s->d_yc, s->d_bs_part, s->bs_nblk,
                                                              s->schur_form == kSchurRows ? s->split.Wg : nullptr);
}

int launch_iteration(tscm_solver* s) {
  launch_schur(s, 0.0);
  RC_TRY(launch_schur_allreduce(s, 0.0));
  launch_solve(s);
  launch_backsub(s);
  const bool single = s->num_ranks <= 1;
  launch_evaluation(s, 1, 0, /*prep=*/false, /*decide=*/single);
  if (!single) {
    RC_TRY(launch_eval_allreduce(s, 1, /*decide=*/true));
    if (!s->p2p_on) {
      launch_k(s, k_decide, dim3(1), dim3(kDecideThreads), (size_t)(0), s->P, s->ps[0], s->ps[1], s->d_state, s->lm, s->trace);
    }
  }
  return TSCM_OK;
}

int capture_iterations(tscm_solver* s, int iters, cudaGraphExec_t* out) {
  cudaGraph_t graph = nullptr;
  const int64_t before = s->launches;
  CUDA_TRY(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
  int rc = TSCM_OK;
  s->pdl = s->use_pdl;
  for (int k = 0; k < iters && !rc; ++k) rc = launch_iteration(s);
  s->pdl = false;
  const cudaError_t e = cudaStreamEndCapture(s->stream, &graph);
  s->launches_per_iter = (int)((s->launches - before) / std::max(1, iters));
  s->launches = before;
  if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
  if (e != cudaSuccess) { set_error("graph capture failed: %s", cudaGetErrorString(e)); return TSCM_ERR_CUDA; }
  const cudaError_t ei = cudaGraphInstantiate(out, graph, 0);
  cudaGraphDestroy(graph);
  if (ei != cudaSuccess) { set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(ei)); return TSCM_ERR_CUDA; }
  return TSCM_OK;
}

int ensure_graph(tscm_solver* s) {
  if (!s->graph_dirty && s->graph_exec) return TSCM_OK;
  if (s->graph_exec) { cudaGraphExecDestroy(s->graph_exec); s->graph_exec = nullptr; }
  if (s->graph_exec_n) { cudaGraphExecDestroy(s->graph_exec_n); s->graph_exec_n = nullptr; }
  RC_TRY(capture_iterations(s, 1, &s->graph_exec));
  if (s->is_kid) RC_TRY(capture_iterations(s, kGroupIters, &s->graph_exec_n));
  s->graph_dirty = false;
  return TSCM_OK;
}

// Iteration zero: evaluate the initial point held in parameter set 0.  Asynchronous.
int run_initial(tscm_solver* s) {
  CUDA_TRY(cudaMemsetAsync(s->d_state, 0, sizeof(LmState), s->stream));
  CUDA_TRY(cudaMemsetAsync(s->d_p2p_err, 0, sizeof(int), s->stream));
  launch_evaluation(s, 2, 1);
  RC_TRY(launch_eval_allreduce(s, 2));
  const int n = s->P.F * 6 + s->P.C * 13;
  k_jacobi_scale<<<(n + 255) / 256, 256, 0, s->stream>>>(s->P, s->ps[0], s->ps[1], s->d_state, s->lm,
                                                        s->d_scale_e, s->d_scale_c);
  k_init<<<1, kDecideThreads, 0, s->stream>>>(s->P, s->ps[0], s->ps[1], s->d_state, s->lm, s->trace);
  s->launches += 2;
  CUDA_TRY(cudaGetLastError());
  return TSCM_OK;
}

// Evaluate the point in set `cur` with the configured loss, compute the Jacobi scaling there (as
// iteration 0 does) and assemble the reduced camera system at `radius` into d_Sr (radius = +inf:
// the undamped system).  Asynchronous; on a sharded solve every shard must make the same call.
int assemble_at(tscm_solver* s, double radius) {
  const int cur = s->x_in_set1 ? 1 : 0;
  LmState* tmp = s->h_state + 1;
  std::memset(tmp, 0, sizeof(LmState));
  tmp->cur = cur;
  CUDA_TRY(cudaMemcpyAsync(s->d_state, tmp, sizeof(LmState), cudaMemcpyHostToDevice, s->stream));
  launch_evaluation(s, 2 + cur, 1);
  RC_TRY(launch_eval_allreduce(s, 2 + cur));
  const int n = s->P.F * 6 + s->P.C * 13;
  k_jacobi_scale<<<(n + 255) / 256, 256, 0, s->stream>>>(s->P, s->ps[0], s->ps[1], s->d_state, s->lm,
                                                        s->d_scale_e, s->d_scale_c);
  s->launches += 1;
  launch_schur(s, radius);
  RC_TRY(launch_schur_allreduce(s, radius));
  return TSCM_OK;
}

int fetch_state(tscm_solver* s) {
  CUDA_TRY(cudaMemcpyAsync(s->h_state, s->d_state, sizeof(LmState), cudaMemcpyDeviceToHost, s->stream));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  return TSCM_OK;
}

// x always starts a run / a timed stage in parameter set 0
int move_x_to_set0(tscm_solver* k) {
  if (!k->x_in_set1) return TSCM_OK;
  CUDA_TRY(cudaMemcpyAsync(k->ps[0].intr, k->ps[1].intr, (size_t)k->C * 9 * sizeof(double), cudaMemcpyDeviceToDevice, k->stream));
  CUDA_TRY(cudaMemcpyAsync(k->ps[0].cam_rt, k->ps[1].cam_rt, (size_t)k->C * 6 * sizeof(double), cudaMemcpyDeviceToDevice, k->stream));
  CUDA_TRY(cudaMemcpyAsync(k->ps[0].board_rt, k->ps[1].board_rt, (size_t)k->F * 6 * sizeof(double), cudaMemcpyDeviceToDevice, k->stream));
  k->x_in_set1 = false;
  return TSCM_OK;
}

size_t trace_bytes(int capacity) { return (size_t)capacity * (4 * sizeof(double) + sizeof(int)); }
void wire_trace(tscm_solver* s, int capacity) {
  double* d = reinterpret_cast<double*>(s->d_trace);
  s->trace.cost = d; s->trace.radius = d + capacity; s->trace.gmax = d + 2 * (size_t)capacity;
  s->trace.step_norm = d + 3 * (size_t)capacity;
  s->trace.flags = reinterpret_cast<int*>(d + 4 * (size_t)capacity);
  s->trace.capacity = capacity;
  s->trace_capacity = capacity;
}
int ensure_trace(tscm_solver* s, int capacity) {
  if (capacity <= s->trace_capacity) return TSCM_OK;
  capacity = std::max(capacity, 128);
  char* d = nullptr;
  CUDA_TRY(cudaMalloc((void**)&d, trace_bytes(capacity)));
  CUDA_TRY(cudaMemsetAsync(d, 0, trace_bytes(capacity), s->stream));
  s->extra.push_back(d);
  s->d_trace = d;
  if (s->h_trace) cudaFreeHost(s->h_trace);
  s->h_trace = nullptr;
  CUDA_TRY(cudaMallocHost((void**)&s->h_trace, trace_bytes(capacity)));
  wire_trace(s, capacity);
  s->graph_dirty = true;
  return TSCM_OK;
}

const char* termination_name(int t) {
  return t == TSCM_CONVERGENCE ? "CONVERGENCE" : t == TSCM_NO_CONVERGENCE ? "NO_CONVERGENCE" : "FAILURE";
}

// ---------------------------------------------------------------------------
// Schur-elimination form: tables and buffers
// ---------------------------------------------------------------------------
double visibility_fill(const tscm_solver* s) {
  // live columns of the views over F x NL
  double cols = 0.0;
  for (int v = 0; v < s->V; ++v) {
    const int m = s->h_view_camera[v];
    cols += s->h_live_off[m + 1] - s->h_live_off[m];
  }
  return cols / ((double)s->F * s->P.NL);
}

int choose_schur_form(const tscm_solver* s) {
  const int NLp = s->schur.NLp, ntiles = s->schur.ntiles;
  const size_t split_smem = (size_t)(2 * (2 * kSchurFB * 6 * NLp + kSchurFB * 6)) * sizeof(double);
  // dense rows whenever they fit shared memory and the reduced system is wide enough to amortise
  // the second kernel (measured, tools/form_ab.py: 8-camera ring at fill 0.39, 150-5,000 frames: rows
  // 3-10 % ahead of the fused form; 4-camera rig at fill 0.39: fused 0-5 % ahead)
  if (split_smem <= s->smem_optin && (visibility_fill(s) >= 0.4 || s->P.NL >= 64)) return kSchurRows;
  const int schur2_nt = kSchurFB * 32 + (ntiles + 31) / 32 * 32;
  const size_t schur2_smem = (size_t)(2 * (2 * kSchurFB * 6 * NLp + kSchurFB * 6) + kSchurFB * 64) * sizeof(double);
  if (schur2_nt <= 640 && schur2_smem <= s->smem_optin) return kSchurFused;
  return kSchurPairs;
}

// Registers the tables (blob) and buffers (arena) of `form`; pointers are valid after
// arena.commit() + blob.upload().
int plan_schur(tscm_solver* s, int form, Arena& arena, Blob& blob) {
  const int F = s->F, V = s->V, C = s->C, NL = s->P.NL, NLp = s->schur.NLp, ntiles = s->schur.ntiles;
  if (V >= (1 << 27)) { set_error("too many views"); return TSCM_ERR_UNSUPPORTED; }
  if (form == kSchurRows || form == kSchurFused) {
    // per-frame column descriptors: live columns of the frame's views, camera order
    std::vector<int> col_ptr(F + 1, 0);
    for (int f = 0; f < F; ++f) {
      int n = 0;
      for (int q = s->h_frame_ptr[f]; q < s->h_frame_ptr[f + 1]; ++q) {
        const int m = s->h_view_camera[s->h_frame_views[q]];
        n += s->h_live_off[m + 1] - s->h_live_off[m];
      }
      col_ptr[f + 1] = col_ptr[f] + n;
    }
    const size_t ncol = (size_t)col_ptr[F];
    std::vector<int> col_src(ncol);
    std::vector<short> col_g(ncol), col_sidx(ncol);
    for (int f = 0; f < F; ++f) {
      size_t o = (size_t)col_ptr[f];
      for (int q = s->h_frame_ptr[f]; q < s->h_frame_ptr[f + 1]; ++q) {
        const int v = s->h_frame_views[q], m = s->h_view_camera[v];
        const int n = s->h_live_off[m + 1] - s->h_live_off[m];
        for (int k = 0; k < n; ++k, ++o) {
          const int kk = n == 13 ? k : k + 6;
          col_src[o] = v * 16 + kk;
          col_g[o] = (short)(s->h_live_off[m] + k);
          col_sidx[o] = (short)(m * 13 + kk);
        }
      }
    }
    blob.add(&s->schur2.col_ptr, col_ptr);
    blob.add(&s->schur2.col_src, col_src);
    blob.add(&s->schur2.col_g, col_g);
    blob.add(&s->split.col_sidx, col_sidx);
  }
  if (form == kSchurRows) {
    s->split_smem = (size_t)(2 * (2 * kSchurFB * 6 * NLp + kSchurFB * 6)) * sizeof(double);
    if (s->split_smem > s->smem_optin) { set_error("dense-row Schur form needs %zu bytes of shared memory", s->split_smem); return TSCM_ERR_UNSUPPORTED; }
    arena.want(&s->split.Wg, (size_t)F * 6 * NLp);
    arena.want(&s->split.Yg, (size_t)F * 6 * NLp);
    arena.want(&s->split.zg, ((size_t)F + 8) * 6);
    arena.want(&s->split.fact, (size_t)F * 32);
  } else if (form == kSchurFused) {
    s->schur2_nt = kSchurFB * 32 + (ntiles + 31) / 32 * 32;
    s->schur2_smem = (size_t)(2 * (2 * kSchurFB * 6 * NLp + kSchurFB * 6) + kSchurFB * 64) * sizeof(double);
    if (s->schur2_nt > 640 || s->schur2_smem > s->smem_optin) {
      set_error("fused Schur form cannot hold a reduced system of %d live parameters", NL);
      return TSCM_ERR_UNSUPPORTED;
    }
  } else if (form == kSchurPairs) {
    static_assert(sizeof(PairEntry) == sizeof(int2) && sizeof(PairRange) == sizeof(int2), "int2 layout");
    if (kPair2Smem > s->smem_optin) { set_error("pair Schur form needs %zu bytes of shared memory", (size_t)kPair2Smem); return TSCM_ERR_UNSUPPORTED; }
    const PairLists lists = build_pair_lists(C, F, V, s->h_view_camera.data(), s->h_view_frame.data(), kPairChunk);
    std::vector<short> loff(C + 1);
    for (int m = 0; m <= C; ++m) loff[m] = (short)s->h_live_off[m];
    s->pairs.nitems = (int)lists.item_range.size();
    s->pairs.npairs = (int)lists.pair_a.size();
    blob.add(reinterpret_cast<const PairEntry**>(&s->pairs.ent), lists.ent);
    blob.add(reinterpret_cast<const PairRange**>(&s->pairs.item_range), lists.item_range);
    blob.add(&s->pairs.pair_item, lists.pair_item);
    blob.add(&s->pairs.pair_items, lists.pair_items);
    blob.add(&s->pairs.pair_a, lists.pair_a);
    blob.add(&s->pairs.pair_b, lists.pair_b);
    blob.add(&s->pairs.live_off, loff);
    arena.want(&s->pairs.part, (size_t)std::max(1, s->pairs.nitems) * kPairPart);
    arena.want(&s->split.Wv, (size_t)V * 96);
    arena.want(&s->split.Yv, (size_t)V * 96);
    arena.want(&s->split.fact, (size_t)F * 32);
  } else {
    set_error("unknown Schur form %d", form);
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  return TSCM_OK;
}

int set_smem_attr(const void* fn, size_t bytes) {
  if (bytes > 48 * 1024)
    CUDA_TRY(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
  return TSCM_OK;
}

// Whether the single-CTA k_solve (and the shared-memory k_cov_factor) hold this solver's reduced
// system: the default limit, and the choice between k_solve and k_solve_cluster.  Needs s->solve.
bool single_cta_fits(const tscm_solver* s) {
  const int NL = s->P.NL;
  return NL <= kCovMaxNL && s->solve.smem <= s->smem_optin && cov_factor_smem(NL) <= s->smem_optin;
}

// Prepares k_solve_cluster for this solver: cluster size, the global copy of the factor, and a
// check that the device can schedule the cluster with its shared memory (so that no launch inside
// the iteration graph can fail for it).
int ensure_cluster(tscm_solver* s) {
  if (s->d_cluster_L) return TSCM_OK;
  const int NL = s->P.NL;
  const ClusterDims d = cluster_dims(NL, s->C);
  if (NL > kLargeRigMaxNL || d.ncta > kClusterMaxCtas) {
    set_error("reduced system of %d live parameters exceeds the limit of %d of the cluster solve", NL, kLargeRigMaxNL);
    return TSCM_ERR_UNSUPPORTED;
  }
  // the attribute is per kernel and process-wide: set it once to the largest system accepted
  // (32 cameras, 416 live parameters), so that a solver never lowers it under another's launch
  const size_t smem_max = cluster_dims(kLargeRigMaxNL, 32).smem;
  if (d.smem > smem_max || smem_max > s->smem_optin) {
    set_error("cluster solve needs %zu bytes of shared memory per block, the device allows %zu", smem_max, s->smem_optin);
    return TSCM_ERR_UNSUPPORTED;
  }
  const void* fns[2] = {(const void*)k_solve_cluster<7>, (const void*)k_solve_cluster<13>};
  const void* fn = NL <= 32 * 7 ? fns[0] : fns[1];
  for (const void* f : fns) CUDA_TRY(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(d.ncta); cfg.blockDim = dim3(kClusterThreads); cfg.dynamicSmemBytes = d.smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = d.ncta; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  int nclusters = 0;
  const cudaError_t e = cudaOccupancyMaxActiveClusters(&nclusters, fn, &cfg);
  if (e != cudaSuccess || nclusters < 1) {
    cudaGetLastError();
    set_error("the device cannot schedule a cluster of %d CTAs with %zu bytes of shared memory each (%s)", d.ncta,
              d.smem, e != cudaSuccess ? cudaGetErrorString(e) : "no active cluster");
    return TSCM_ERR_UNSUPPORTED;
  }
  double* L = nullptr;
  CUDA_TRY(cudaMalloc((void**)&L, (size_t)solve_pan_off(d.nbk, d.nbk) * sizeof(double)));
  s->extra.push_back(L);
  s->d_cluster_L = L;
  s->cluster = d;
  return TSCM_OK;
}

// after commit + upload
int wire_schur(tscm_solver* s, int form) {
  s->split.col_ptr = s->schur2.col_ptr; s->split.col_src = s->schur2.col_src; s->split.col_g = s->schur2.col_g;
  if (form == kSchurRows) {
    s->split.Wv = nullptr; s->split.Yv = nullptr;
    RC_TRY(set_smem_attr((const void*)k_schur_update<1>, s->split_smem));
    RC_TRY(set_smem_attr((const void*)k_schur_update<2>, s->split_smem));
  } else if (form == kSchurFused) {
    RC_TRY(set_smem_attr((const void*)k_schur2, s->schur2_smem));
  } else {
    s->pairs.Wv = s->split.Wv; s->pairs.Yv = s->split.Yv;
    s->pairs.Sout = s->d_Spart; s->pairs.rout = s->d_rpart;
    RC_TRY(set_smem_attr((const void*)k_schur_pairs2, kPair2Smem));
  }
  s->schur_form = form;
  s->graph_dirty = true;
  return TSCM_OK;
}

void free_shard(tscm_solver* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  if (s->graph_exec) cudaGraphExecDestroy(s->graph_exec);
  if (s->graph_exec_n) cudaGraphExecDestroy(s->graph_exec_n);
  if (s->comm && nccl().ok) nccl().CommDestroy(s->comm);
  for (int r = 0; r < kP2PMaxRanks; ++r)
    if (s->p2p_ipc[r]) cudaIpcCloseMemHandle(s->p2p_ipc[r]);
  for (int k = 0; k < 2; ++k) {
    if (s->poll_ev[k]) cudaEventDestroy(s->poll_ev[k]);
    if (s->cov_ev[k]) cudaEventDestroy(s->cov_ev[k]);
  }
  if (s->arena.base) cudaFree(s->arena.base);
  for (void* p : s->extra) cudaFree(p);
  if (s->d_mailbox) cudaFree(s->d_mailbox);
  if (s->h_state) cudaFreeHost(s->h_state);
  if (s->h_err) cudaFreeHost(s->h_err);
  if (s->h_trace) cudaFreeHost(s->h_trace);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

int upload_observations(tscm_solver* s, const double* obs_xy, const std::vector<ObsSegment>* segs) {
  CUDA_TRY(cudaSetDevice(s->device));
  const size_t view_bytes = (size_t)s->K * sizeof(double2);
  if (!segs) {
    CUDA_TRY(cudaMemcpyAsync(s->d_obs_in, obs_xy, (size_t)s->V * view_bytes, cudaMemcpyHostToDevice, s->stream));
  } else {
    for (const ObsSegment& g : *segs)
      CUDA_TRY(cudaMemcpyAsync(reinterpret_cast<char*>(s->d_obs_in) + (size_t)g.dst_view * view_bytes,
                               reinterpret_cast<const char*>(obs_xy) + (size_t)g.src_view * view_bytes,
                               (size_t)g.count * view_bytes, cudaMemcpyHostToDevice, s->stream));
  }
  dim3 grid((s->V + 31) / 32, (s->K + 31) / 32), block(32, 8);
  k_transpose_obs<<<grid, block, 0, s->stream>>>(s->d_obs_in, s->d_obsT, s->V, s->K, s->P.Vpad);
  s->launches += 1;
  CUDA_TRY(cudaGetLastError());
  return TSCM_OK;
}

// One shard on the device select_device() made current.  p->obs_xy may be NULL (uploaded later).
int create_shard(const tscm_problem* p, const tscm_options* o, const internal::SelectedDevice& dev, bool is_kid,
                 tscm_solver** out) {
  *out = nullptr;
  const auto t0 = Clock::now();
  auto lap = [&](const char* what) {
    if (g_debug & 1) std::fprintf(stderr, "[tscm create] %-28s %8.2f ms\n", what, ms_since(t0));
  };
  std::unique_ptr<tscm_solver, void (*)(tscm_solver*)> owner(new tscm_solver(), free_shard);
  tscm_solver* s = owner.get();
  s->device = dev.index;
  s->sm_count = dev.sm_count;
  s->smem_optin = dev.smem_optin;
  s->is_kid = is_kid;
  s->use_pdl = (g_debug & 4) == 0;
  s->options = *o;
  fill_lm_options(*o, s->lm);
  CUDA_TRY(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking));
  const int C = p->num_cameras, F = p->num_frames, K = p->corners_per_board, V = p->num_views;
  s->C = C; s->F = F; s->K = K; s->V = V; s->fixed_camera = p->fixed_camera;
  DeviceProblem& P = s->P;
  P.C = C; P.F = F; P.K = K; P.V = V; P.fixed_camera = p->fixed_camera;
  P.Vpad = (V + 31) / 32 * 32;

  // ---- index tables (host) -------------------------------------------------------------
  s->h_view_camera.assign(p->view_camera, p->view_camera + V);
  s->h_view_frame.assign(p->view_frame, p->view_frame + V);
  s->h_board.assign(p->board_xy, p->board_xy + 2 * (size_t)K);
  std::vector<int>& live_off = s->h_live_off;
  live_off.assign(C + 1, 0);
  for (int c = 0; c < C; ++c) live_off[c + 1] = live_off[c] + (c == p->fixed_camera ? 7 : 13);
  const int NL = live_off[C];
  P.NL = NL; P.Q = NL * (NL + 1) / 2;
  // The reduced system is factored by ONE CTA of k_solve, and the covariance kernels size their
  // shared arrays by kCovMaxNL: a system is accepted when both fit.  On a B200 (232,448 bytes of
  // opt-in shared memory per block) k_solve is the tighter bound: 16 cameras with one fixed
  // (NL 202) need 220,056 bytes, 16 with none fixed (NL 208) 233,984.  With allow_large_rigs a
  // wider system (up to kLargeRigMaxNL, validate_large_rig) goes to k_solve_cluster instead.
  s->solve = solve_dims(NL, C);
  const bool single_fits = single_cta_fits(s);
  if (!single_fits && o->allow_large_rigs && !is_kid) {
    s->use_cluster = true;
  } else if (!single_fits) {
    set_error("reduced system of %d live parameters (%d cameras) exceeds the limit of %d (16 cameras with one "
              "fixed): the solve needs %zu bytes of shared memory per block, the device allows %zu",
              NL, C, kCovMaxNL, s->solve.smem, s->smem_optin);
    return TSCM_ERR_UNSUPPORTED;
  }
  std::vector<short> live_cam(NL), live_kk(NL);
  for (int c = 0; c < C; ++c)
    for (int k = 0; k < live_off[c + 1] - live_off[c]; ++k) {
      live_cam[live_off[c] + k] = (short)c;
      live_kk[live_off[c] + k] = (short)(c == p->fixed_camera ? k + 6 : k);
    }
  std::vector<int>& frame_ptr = s->h_frame_ptr;
  std::vector<int>& frame_views = s->h_frame_views;
  frame_ptr.assign(F + 1, 0);
  frame_views.assign(V, 0);
  std::vector<int> cam_view_begin(C + 1, 0);
  for (int v = 0; v < V; ++v) { frame_ptr[p->view_frame[v] + 1]++; cam_view_begin[p->view_camera[v] + 1]++; }
  for (int i = 0; i < F; ++i) frame_ptr[i + 1] += frame_ptr[i];
  for (int c = 0; c < C; ++c) cam_view_begin[c + 1] += cam_view_begin[c];
  {
    std::vector<int> fill(frame_ptr.begin(), frame_ptr.end() - 1);
    for (int v = 0; v < V; ++v) frame_views[fill[p->view_frame[v]]++] = v;   // camera order kept
  }
  s->obs_count.assign(C, 0.0);
  for (int c = 0; c < C; ++c) s->obs_count[c] = (double)(cam_view_begin[c + 1] - cam_view_begin[c]) * K;
  // camera-partial slots: one per (evaluation tile of 32 views, distinct camera in it)
  const int nblk_eval = (V + 31) / 32;
  std::vector<int> blk_slot(nblk_eval + 1, 0), cam_slot_begin(C + 1, 0);
  {
    int nslot = 0, prev_cam = -1;
    for (int b = 0; b < nblk_eval; ++b) {
      blk_slot[b] = nslot;
      int last = -1;
      for (int v = 32 * b; v < std::min(V, 32 * b + 32); ++v)
        if (p->view_camera[v] != last) {
          last = p->view_camera[v];
          if (last < prev_cam) { set_error("internal: slot table"); return TSCM_ERR_INVALID_ARGUMENT; }
          prev_cam = last;
          cam_slot_begin[last + 1]++;
          ++nslot;
        }
    }
    blk_slot[nblk_eval] = nslot;
    P.nslot = nslot;
    for (int c = 0; c < C; ++c) cam_slot_begin[c + 1] += cam_slot_begin[c];
  }
  // 4x4 tiles of the upper block triangle, row-major (k_schur_update / k_schur2)
  const int nb = (NL + 3) / 4;
  std::vector<short> tile_bi, tile_bj;
  for (int bi = 0; bi < nb; ++bi) for (int bj = bi; bj < nb; ++bj) { tile_bi.push_back((short)bi); tile_bj.push_back((short)bj); }
  const int ntiles = (int)tile_bi.size();
  s->schur.ntiles = ntiles;
  s->schur.NLp = nb * 4;
  s->schur_ept = ntiles <= 512 ? 1 : 2;
  s->schur_nt = std::max(256, ((ntiles + s->schur_ept - 1) / s->schur_ept + 31) / 32 * 32);
  s->schur_nblk = std::max(1, std::min(s->sm_count, (F + kSchurFB - 1) / kSchurFB));
  int fpb = (F + s->schur_nblk - 1) / s->schur_nblk;
  {
    // frames per CTA: the even split over the SMs (5,000 frames: 148 CTAs x 34 frames; a shard of
    // 625 frames: 70 x 9).  Round 1 rounded up to a multiple of the staging batch (125 x 40, 40 x 16):
    // iteration 304.3 -> 300.7 us on config 3.  TSCM_SCHUR_EVEN=0 restores the rounding (A/B).
    const char* ev = std::getenv("TSCM_SCHUR_EVEN");
    if (ev && ev[0] == '0') fpb = (fpb + kSchurFB - 1) / kSchurFB * kSchurFB;
  }
  s->schur_nblk = (F + fpb - 1) / fpb;
  s->schur.frames_per_block = fpb;
  s->schur.Fpad = (F + 31) / 32 * 32;
  s->eval5_smem = e5_smem_bytes(K, C);
  if (s->eval5_smem > s->smem_optin) {
    set_error("problem (%d corners, %d cameras) needs %zu bytes of shared memory per CTA in k_eval5 (limit %zu)", K, C,
              s->eval5_smem, s->smem_optin);
    return TSCM_ERR_UNSUPPORTED;
  }
  lap("index tables (host)");

  Blob blob;
  Arena& A = s->arena;
  blob.add(&P.board_xy, s->h_board);
  blob.add(&P.view_camera, s->h_view_camera);
  blob.add(&P.view_frame, s->h_view_frame);
  blob.add(&P.frame_ptr, frame_ptr);
  blob.add(&P.frame_views, frame_views);
  blob.add(&P.cam_view_begin, cam_view_begin);
  blob.add(&P.live_off, live_off);
  blob.add(&P.live_cam, live_cam);
  blob.add(&P.live_kk, live_kk);
  {
    std::vector<short> q_i(P.Q), q_j(P.Q);
    int q = 0;
    for (int i = 0; i < NL; ++i) for (int j = i; j < NL; ++j) { q_i[q] = (short)i; q_j[q] = (short)j; ++q; }
    blob.add(&P.q_i, q_i);
    blob.add(&P.q_j, q_j);
  }
  blob.add(&P.blk_slot, blk_slot);
  blob.add(&P.cam_slot_begin, cam_slot_begin);
  blob.add(&s->schur.tile_bi, tile_bi);
  blob.add(&s->schur.tile_bj, tile_bj);
  const int form = choose_schur_form(s);
  RC_TRY(plan_schur(s, form, A, blob));
  lap("Schur tables (host)");

  // ---- buffers ----------------------------------------------------------------------------
  A.want(&s->d_obs_in, (size_t)V * K);
  A.want(&s->d_obsT, (size_t)P.Vpad * K);
  for (int k = 0; k < 2; ++k) {
    A.want(&s->ps[k].intr, (size_t)C * 9);
    A.want(&s->ps[k].cam_rt, (size_t)C * 6);
    A.want(&s->ps[k].board_rt, (size_t)F * 6);
    A.want(&s->ps[k].cam, (size_t)C);
    A.want(&s->ps[k].G, (size_t)V * kViewStride);
    A.want(&s->ps[k].cam_part, (size_t)P.nslot * kCamRec);
    A.want(&s->ps[k].comm, (size_t)C * kCamRec + kCommExtra);
    A.want(&s->ps[k].gmax, 1);
  }
  A.want(&s->d_state, 1);
  A.want(&s->d_scale_e, (size_t)F * 6);
  A.want(&s->d_scale_c, (size_t)C * 13);
  A.want(&s->schur.frame_rec, (size_t)kFrameRec * s->schur.Fpad);
  A.want(&s->d_Spart, (size_t)s->schur_nblk * P.Q);
  A.want(&s->d_rpart, (size_t)s->schur_nblk * NL);
  A.want(&s->d_Sr, (size_t)s->solve.ntile * 16);
  A.want(&s->d_yc, (size_t)NL);
  s->bs_nblk = (F + kBacksubFrames - 1) / kBacksubFrames;
  {
    int maxv = 1;
    for (int f = 0; f < F; ++f) maxv = std::max(maxv, frame_ptr[f + 1] - frame_ptr[f]);
    // a frame has at most one view per camera: 16 cameras by default, 32 with allow_large_rigs
    s->post_lpf = maxv <= 8 ? 8 : (maxv <= 16 ? 16 : 32);
    const int fpc = kPostThreads / s->post_lpf;
    s->fg_nblk = (F + fpc - 1) / fpc;
  }
  A.want(&s->d_cam_sum_part, (size_t)C * kPostSplit * kCamRec);
  A.want(&s->d_ticket, 1);
  A.want(&s->d_p2p_seq, 2);
  A.want(&s->d_p2p_ticket, 1);
  A.want(&s->d_p2p_err, 1);
  A.want(&s->d_comm_stage, (size_t)C * kCamRec + kCommExtra + 8);
  A.want(&s->d_bs_part, (size_t)4 * s->bs_nblk);
  A.want(&s->d_gmax_part, (size_t)s->fg_nblk);
  A.want(&s->d_xn2_part, (size_t)s->fg_nblk);
  {
    const size_t ntile_e = ((size_t)V + 31) / 32;
    s->e5items = e5_items((int)ntile_e, std::min((int)ntile_e, s->sm_count), (K + kE5Producers - 1) / kE5Producers);
    A.want(&s->d_mom, (size_t)s->e5items.nitems * kE5MomEntries * 32);
    A.want(&s->d_fcg, ntile_e * kFcElems * 32);
    if (g_debug & 1) {
      // solveT / solve_smem: tiles per thread and shared memory per CTA of the kernel that runs;
      // cluster: its CTAs (0: the single-CTA k_solve)
      const ClusterDims cd = cluster_dims(NL, C);
      std::fprintf(stderr,
                   "[tscm create] paths: form=%s ept=%d solveT=%d lpf=%d e5grid=%d e5tiles=%d e5whole=%d e5split=%d "
                   "NL=%d solve_smem=%zu smem_optin=%zu cluster=%d\n",
                   form == kSchurRows ? "rows" : (form == kSchurFused ? "fused" : "pairs"), s->schur_ept,
                   s->use_cluster ? kClusterT : s->solve.T, s->post_lpf, std::min((int)ntile_e, s->sm_count),
                   (int)ntile_e, s->e5items.n_whole, s->e5items.split, NL, s->use_cluster ? cd.smem : s->solve.smem,
                   s->smem_optin, s->use_cluster ? cd.ncta : 0);
    }
  }
  const int cap = std::max(128, std::min(s->options.max_num_iterations, 1 << 16) + 2);
  A.want(&s->d_trace, trace_bytes(cap));
  A.want(&s->d_blob, blob.bytes.size());
  RC_TRY(A.commit(s->stream));
  blob.d_base = s->d_blob;
  RC_TRY(blob.upload(s->stream));
  lap("arena + table upload");
  P.obsT = s->d_obsT;
  s->schur.Spart = s->d_Spart; s->schur.rpart = s->d_rpart;
  s->schur.scale_e = s->d_scale_e; s->schur.scale_c = s->d_scale_c;
  wire_trace(s, cap);
  CUDA_TRY(cudaMallocHost((void**)&s->h_state, 3 * sizeof(LmState)));
  CUDA_TRY(cudaMallocHost((void**)&s->h_err, sizeof(int)));
  *s->h_err = 0;
  CUDA_TRY(cudaMallocHost((void**)&s->h_trace, trace_bytes(cap)));
  CUDA_TRY(cudaEventCreateWithFlags(&s->poll_ev[0], cudaEventDisableTiming));
  CUDA_TRY(cudaEventCreateWithFlags(&s->poll_ev[1], cudaEventDisableTiming));
  {
    // mailbox of the peer-memory exchange (tiny; its own allocation so that its IPC handle can
    // be exported right after creation)
    const int nwords = P.Q + NL;
    s->p2p.nA = (nwords + 31) / 32 * 32;
    s->p2p.nctaA = (nwords + 31) / 32;
    s->p2p.nB = (C * kCamRec + kCommExtra + 1 + 31) / 32 * 32;
    const size_t words = p2p_mailbox_words(s->p2p.nA, s->p2p.nctaA, s->p2p.nB);
    CUDA_TRY(cudaMalloc((void**)&s->d_mailbox, words * sizeof(double)));
    CUDA_TRY(cudaMemsetAsync(s->d_mailbox, 0, words * sizeof(double), s->stream));
    s->p2p.seq = s->d_p2p_seq; s->p2p.ticket = s->d_p2p_ticket; s->p2p.err = s->d_p2p_err;
    s->p2p.timeout_ns = 10ull * 1000000000ull;
  }
  RC_TRY(wire_schur(s, form));
  if (s->use_cluster) {
    RC_TRY(ensure_cluster(s));
  } else {
    RC_TRY(set_smem_attr((const void*)k_solve<1, 4>, s->solve.smem));
    RC_TRY(set_smem_attr((const void*)k_solve<4, 7>, s->solve.smem));
  }
  RC_TRY(set_smem_attr((const void*)k_eval5, s->eval5_smem));
  RC_TRY(set_smem_attr((const void*)k_view_blocks, vb_smem_bytes()));
  lap("kernel attributes");
  if (p->obs_xy) {
    RC_TRY(upload_observations(s, p->obs_xy, nullptr));
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    lap("observations H2D + transpose");
  }
  *out = owner.release();
  return TSCM_OK;
}

// ---------------------------------------------------------------------------
// group = one shard per device of this process
// ---------------------------------------------------------------------------
struct ShardPlan {
  std::vector<int> frame;                         // [n + 1]
  std::vector<std::vector<int>> vcam, vfrm;       // per shard
  std::vector<std::vector<ObsSegment>> seg;       // per shard
};

// Contiguous frame ranges balanced by view count; a shard's views keep the camera-major order.
ShardPlan plan_shards(const tscm_problem* p, int n) {
  ShardPlan sp;
  const int F = p->num_frames, V = p->num_views, C = p->num_cameras;
  std::vector<int> per_frame(F, 0), cvb(C + 1, 0);
  for (int v = 0; v < V; ++v) { per_frame[p->view_frame[v]]++; cvb[p->view_camera[v] + 1]++; }
  for (int c = 0; c < C; ++c) cvb[c + 1] += cvb[c];
  sp.frame.assign(n + 1, 0);
  {
    long long acc = 0;
    int r = 1;
    for (int f = 0; f < F && r < n; ++f) {
      acc += per_frame[f];
      // close shard r - 1 once it holds its share, or when every later shard needs the frames left
      if (acc * n >= (long long)V * r || F - (f + 1) <= n - r) sp.frame[r++] = f + 1;
    }
    for (; r <= n; ++r) sp.frame[r] = F;
  }
  sp.vcam.resize(n); sp.vfrm.resize(n); sp.seg.resize(n);
  for (int r = 0; r < n; ++r) {
    const int f0 = sp.frame[r], f1 = sp.frame[r + 1];
    for (int m = 0; m < C; ++m) {
      const int* fb = p->view_frame + cvb[m];
      const int* fe = p->view_frame + cvb[m + 1];
      const int a = (int)(std::lower_bound(fb, fe, f0) - p->view_frame);
      const int b = (int)(std::lower_bound(fb, fe, f1) - p->view_frame);
      if (b > a) sp.seg[r].push_back(ObsSegment{(int)sp.vcam[r].size(), a, b - a});
      for (int v = a; v < b; ++v) { sp.vcam[r].push_back(m); sp.vfrm[r].push_back(p->view_frame[v] - f0); }
    }
  }
  return sp;
}

void destroy_solver(tscm_solver* s) {
  if (!s) return;
  if (!s->kids.empty() || (!s->stream && !s->arena.base)) {   // group facade (owns no device state itself)
    for (tscm_solver* k : s->kids) free_shard(k);
    delete s;
    return;
  }
  free_shard(s);
}

// `dev`: select_device() of the first device of the group
int create_group(const tscm_problem* p, const tscm_options* o, const internal::SelectedDevice& dev, int n,
                 tscm_solver** out) {
  const int device = dev.index;
  if (device + n > dev.visible) {
    set_error("num_gpus = %d from device %d, but only %d device(s) are visible", n, device, dev.visible);
    return TSCM_ERR_NO_DEVICE;
  }
  if (p->num_frames < n) { set_error("%d frames cannot be sharded over %d GPUs", p->num_frames, n); return TSCM_ERR_INVALID_ARGUMENT; }
  std::unique_ptr<tscm_solver, void (*)(tscm_solver*)> owner(new tscm_solver(), destroy_solver);
  tscm_solver* g = owner.get();
  g->device = device;
  g->options = *o;
  g->C = p->num_cameras; g->F = p->num_frames; g->K = p->corners_per_board; g->V = p->num_views;
  g->fixed_camera = p->fixed_camera;
  g->h_view_camera.assign(p->view_camera, p->view_camera + p->num_views);
  g->h_view_frame.assign(p->view_frame, p->view_frame + p->num_views);
  g->h_board.assign(p->board_xy, p->board_xy + 2 * (size_t)p->corners_per_board);
  g->obs_count.assign(g->C, 0.0);
  for (int v = 0; v < g->V; ++v) g->obs_count[p->view_camera[v]] += g->K;
  ShardPlan sp = plan_shards(p, n);
  g->kid_frame = sp.frame;
  g->kid_seg = sp.seg;
  for (int r = 0; r < n; ++r) {
    tscm_problem q = *p;
    q.num_frames = sp.frame[r + 1] - sp.frame[r];
    q.num_views = (int)sp.vcam[r].size();
    q.view_camera = sp.vcam[r].data();
    q.view_frame = sp.vfrm[r].data();
    q.obs_xy = nullptr;
    internal::SelectedDevice kd;
    RC_TRY(internal::select_device(device + r, "the calibration solve", &kd));
    tscm_solver* k = nullptr;
    RC_TRY(create_shard(&q, o, kd, true, &k));
    k->obs_count = g->obs_count;      // global counts: the read-out divides global sums
    g->kids.push_back(k);
  }
  // peer access + direct mailbox pointers
  for (int i = 0; i < n; ++i) {
    cudaSetDevice(device + i);
    for (int j = 0; j < n; ++j) {
      if (i == j) continue;
      int can = 0;
      cudaDeviceCanAccessPeer(&can, device + i, device + j);
      if (!can) { set_error("device %d cannot access device %d: num_gpus needs peer access", device + i, device + j); return TSCM_ERR_UNSUPPORTED; }
      const cudaError_t e = cudaDeviceEnablePeerAccess(device + j, 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) { set_error("cudaDeviceEnablePeerAccess(%d -> %d): %s", device + i, device + j, cudaGetErrorString(e)); return TSCM_ERR_CUDA; }
    }
  }
  for (int i = 0; i < n; ++i) {
    tscm_solver* k = g->kids[i];
    cudaSetDevice(k->device);
    cudaStreamSynchronize(k->stream);     // mailbox zeroed before any peer writes to it
  }
  for (int i = 0; i < n; ++i) {
    tscm_solver* k = g->kids[i];
    for (int j = 0; j < n; ++j) k->p2p.mb[j] = g->kids[j]->d_mailbox;
    k->p2p.rank = i; k->p2p.world = n;
    k->rank = i; k->num_ranks = n;
    k->p2p_on = true;
    k->graph_dirty = true;
  }
  if (p->obs_xy) {
    for (int i = 0; i < n; ++i) RC_TRY(upload_observations(g->kids[i], p->obs_xy, &g->kid_seg[i]));
    for (tscm_solver* k : g->kids) { cudaSetDevice(k->device); cudaStreamSynchronize(k->stream); }
  }
  *out = owner.release();
  return TSCM_OK;
}

// every shard (or the solver itself)
template <typename Fn>
int for_shards(tscm_solver* s, Fn fn) {
  if (s->kids.empty()) return fn(s, 0);
  for (size_t i = 0; i < s->kids.size(); ++i) {
    const int rc = fn(s->kids[i], (int)i);
    if (rc) return rc;
  }
  return TSCM_OK;
}
int sync_shards(tscm_solver* s) {
  return for_shards(s, [](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    CUDA_TRY(cudaStreamSynchronize(k->stream));
    return TSCM_OK;
  });
}
tscm_solver* lead(tscm_solver* s) { return s->kids.empty() ? s : s->kids[0]; }

// The evaluation records of the read-outs: every shard evaluates its current point, under the
// plain (loss-free) residuals with the sum of sqrt(s) if `want_err`, or under the configured loss
// (plain = false: the records a later run() starts from), and the records are summed over the
// shards or ranks.  Waits for every shard.
int evaluate_shards(tscm_solver* s, bool plain, bool want_err) {
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    const int cur = k->x_in_set1 ? 1 : 0;
    const LmOptions saved = k->lm;
    if (plain) k->lm.loss_type = 0;
    k->want_err = want_err ? 1 : 0;
    launch_evaluation(k, 2 + cur, 1);
    const int rc = launch_eval_allreduce(k, 2 + cur);
    k->lm = saved;
    k->want_err = 0;
    return rc;
  }));
  return sync_shards(s);
}

// Sums a host record of C * kCamRec + kCommExtra doubles over the ranks of a multi-process solve,
// in place, through the exchange of the evaluation record (which it overwrites).
int allreduce_record(tscm_solver* L, std::vector<double>& rec) {
  const int cur = L->x_in_set1 ? 1 : 0;
  CUDA_TRY(cudaSetDevice(L->device));
  CUDA_TRY(cudaMemcpyAsync(L->ps[cur].comm, rec.data(), rec.size() * sizeof(double), cudaMemcpyHostToDevice, L->stream));
  RC_TRY(launch_eval_allreduce(L, 2 + cur));
  CUDA_TRY(cudaStreamSynchronize(L->stream));
  CUDA_TRY(cudaMemcpy(rec.data(), L->ps[cur].comm, rec.size() * sizeof(double), cudaMemcpyDeviceToHost));
  return TSCM_OK;
}

// ---------------------------------------------------------------------------
// solver cache of tscm_solve()
// ---------------------------------------------------------------------------
struct CacheEntry {
  tscm_solver* solver = nullptr;
  int device = 0, num_gpus = 1;
  uint64_t stamp = 0;
};
std::mutex g_cache_mu;
std::vector<CacheEntry> g_cache;
int g_cache_max = 1;
uint64_t g_cache_clock = 0;
void* g_host_block = nullptr;       // tscm_host_alloc: the one page-locked block kept for reuse
size_t g_host_bytes = 0;
bool g_host_busy = false;

bool same_structure(const tscm_solver* s, const tscm_problem* p) {
  if (s->C != p->num_cameras || s->F != p->num_frames || s->K != p->corners_per_board || s->V != p->num_views ||
      s->fixed_camera != p->fixed_camera)
    return false;
  return std::memcmp(s->h_view_camera.data(), p->view_camera, (size_t)s->V * sizeof(int)) == 0 &&
         std::memcmp(s->h_view_frame.data(), p->view_frame, (size_t)s->V * sizeof(int)) == 0 &&
         std::memcmp(s->h_board.data(), p->board_xy, (size_t)s->K * 2 * sizeof(double)) == 0;
}

void cache_evict_oldest_locked() {
  size_t old = 0;
  for (size_t i = 1; i < g_cache.size(); ++i) if (g_cache[i].stamp < g_cache[old].stamp) old = i;
  destroy_solver(g_cache[old].solver);
  g_cache.erase(g_cache.begin() + old);
}

int upload_all_observations(tscm_solver* s, const double* obs_xy) {
  return for_shards(s, [&](tscm_solver* k, int i) -> int {
    return upload_observations(k, obs_xy, s->kids.empty() ? nullptr : &s->kid_seg[i]);
  });
}

// The cached solver of this structure, taken out of the cache (nobody else may use it meanwhile),
// or nullptr.
tscm_solver* cache_checkout(const tscm_problem* p, int device, int ngpu, int allow_large_rigs) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  for (size_t i = 0; i < g_cache.size(); ++i) {
    CacheEntry& e = g_cache[i];
    if (e.device == device && e.num_gpus == ngpu && e.solver->options.allow_large_rigs == allow_large_rigs &&
        same_structure(e.solver, p)) {
      tscm_solver* s = e.solver;
      g_cache.erase(g_cache.begin() + i);
      return s;
    }
  }
  return nullptr;
}
// Back into the cache (keep = the solver is in a usable state), or destroyed.
void cache_checkin(tscm_solver* s, int device, int ngpu, bool keep) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  if (keep && g_cache_max > 0) {
    while ((int)g_cache.size() >= g_cache_max) cache_evict_oldest_locked();
    CacheEntry e;
    e.solver = s; e.device = device; e.num_gpus = ngpu; e.stamp = ++g_cache_clock;
    g_cache.push_back(e);
  } else {
    destroy_solver(s);
  }
}

// The solver of a one-shot call (tscm_solve, tscm_compute_covariance) on a validated problem:
// validates the options, selects the device, takes the cached solver of this structure (with the
// options set) or creates one, and uploads the observations.  Hand it back with cache_checkin().
struct Checkout {
  tscm_solver* s = nullptr;
  int device = 0, ngpu = 1;
  bool hit = false;
};
int checkout_solver(const tscm_problem* problem, const tscm_options* options, int device, const char* what,
                    Checkout* c) {
  tscm_options defaults;
  tscm_options_init(&defaults);
  if (!options) options = &defaults;
  RC_TRY(validate_options(options));
  RC_TRY(validate_large_rig(problem, options));
  internal::SelectedDevice dev;
  RC_TRY(internal::select_device(device, what, &dev));
  c->device = dev.index;
  c->ngpu = std::max(1, options->num_gpus);
  c->s = cache_checkout(problem, c->device, c->ngpu, options->allow_large_rigs);
  c->hit = c->s != nullptr;
  int rc = TSCM_OK;
  if (c->hit) {
    rc = tscm_solver_set_options(c->s, options);
  } else {
    tscm_problem q = *problem;
    q.obs_xy = nullptr;                        // uploaded below, without a sync of its own
    rc = tscm_solver_create(&q, options, c->device, &c->s);
  }
  if (!rc) rc = upload_all_observations(c->s, problem->obs_xy);
  if (rc && c->s) {
    destroy_solver(c->s);
    c->s = nullptr;
  }
  return rc;
}

// ---------------------------------------------------------------------------
// covariance (tscm_covariance.cuh)
// ---------------------------------------------------------------------------
int ensure_cov_buffers(tscm_solver* k) {
  if (k->d_cov_fac) return TSCM_OK;
  const size_t NL = (size_t)k->P.NL;
  // above kCovMaxNL (allow_large_rigs only) the factor works on a packed triangle in global memory
  const bool large = k->P.NL > kCovMaxNL;
  if (large && (!k->options.allow_large_rigs || k->P.NL > kLargeRigMaxNL)) { set_error("covariance: %d live parameters exceed %d", k->P.NL, kCovMaxNL); return TSCM_ERR_UNSUPPORTED; }
  if (!large && cov_factor_smem(k->P.NL) > k->smem_optin) { set_error("covariance needs %zu bytes of shared memory", cov_factor_smem(k->P.NL)); return TSCM_ERR_UNSUPPORTED; }
  Arena a;
  a.want(&k->d_cov_fac, NL * NL);
  a.want(&k->d_cov_sinv, NL * NL);
  a.want(&k->d_cov_cam, NL * NL);
  a.want(&k->d_cov_board, (size_t)k->F * 36);
  a.want(&k->d_cov_flag, 1);
  if (large) a.want(&k->d_cov_tri, NL * (NL + 1) / 2);
  RC_TRY(a.commit(k->stream));
  k->extra.push_back(a.base);
  if (!large) RC_TRY(set_smem_attr((const void*)k_cov_factor, cov_factor_smem(k->P.NL)));
  RC_TRY(set_smem_attr((const void*)k_cov_frames, cov_frames_smem(kLargeRigMaxNL)));
  for (int e = 0; e < 2; ++e) CUDA_TRY(cudaEventCreate(&k->cov_ev[e]));
  return TSCM_OK;
}

// The three covariance kernels on the system assemble_at(+inf) left in d_Sr.  Asynchronous.
int launch_covariance(tscm_solver* k) {
  const int NL = k->P.NL, cur = k->x_in_set1 ? 1 : 0;
  CUDA_TRY(cudaMemsetAsync(k->d_cov_flag, 0, sizeof(int), k->stream));
  CUDA_TRY(cudaEventRecord(k->cov_ev[0], k->stream));
  if (k->d_cov_tri)
    k_cov_factor_global<<<1, kCovFactorThreads, 0, k->stream>>>(NL, k->solve.nbk, k->d_Sr, k->d_cov_fac,
                                                                 k->d_cov_flag, k->d_cov_tri);
  else
    k_cov_factor<<<1, kCovFactorThreads, cov_factor_smem(NL), k->stream>>>(NL, k->solve.nbk, k->d_Sr, k->d_cov_fac,
                                                                            k->d_cov_flag);
  k_cov_inverse<<<(NL + kCovInvWarps - 1) / kCovInvWarps, 32 * kCovInvWarps, cov_inverse_smem(NL), k->stream>>>(
      k->P, k->d_scale_c, k->d_cov_fac, k->d_cov_flag, k->d_cov_sinv, k->d_cov_cam);
  k_cov_frames<<<(k->F + kCovFrameWarps - 1) / kCovFrameWarps, 32 * kCovFrameWarps, cov_frames_smem(NL), k->stream>>>(
      k->P, k->ps[cur], k->d_scale_e, k->d_scale_c, k->schur.frame_rec, k->schur.Fpad, k->d_cov_sinv, k->d_cov_flag,
      k->d_cov_board);
  CUDA_TRY(cudaEventRecord(k->cov_ev[1], k->stream));
  k->launches += 3;
  CUDA_TRY(cudaGetLastError());
  return TSCM_OK;
}

}  // namespace

// ---- helpers shared with the other translation units (tscm_internal.h) ----
namespace tscm {
namespace internal {
void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
}
int select_device(int device, const char* what, SelectedDevice* out) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    set_error("no CUDA device: %s has no CPU fallback", what);
    return TSCM_ERR_NO_DEVICE;
  }
  if (device < 0) CUDA_TRY(cudaGetDevice(&device));
  if (device >= ndev) { set_error("device %d does not exist (%d visible)", device, ndev); return TSCM_ERR_NO_DEVICE; }
  DeviceInfo prop;
  RC_TRY(device_info(device, &prop));
  if (prop.major < 10) {
    set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return TSCM_ERR_NO_DEVICE;
  }
  CUDA_TRY(cudaSetDevice(device));
  if (out) {
    out->index = device;
    out->visible = ndev;
    out->sm_count = prop.sm_count;
    out->smem_optin = prop.smem_optin;
  }
  return TSCM_OK;
}
DeviceScope::DeviceScope() { if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); } }
DeviceScope::~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
}  // namespace internal
}  // namespace tscm

extern "C" {


const char* tscm_last_error(void) { return g_last_error.c_str(); }
const char* tscm_version(void) { return "tscm-b200 0.2.0 (sm_100a, fp64)"; }
void tscm_set_debug(int32_t flags) { g_debug = flags; }

void tscm_options_init(tscm_options* o) {
  if (!o) return;
  std::memset(o, 0, sizeof(*o));
  o->max_num_iterations = 50;
  o->function_tolerance = 1e-6;
  o->gradient_tolerance = 1e-10;
  o->parameter_tolerance = 1e-8;
  o->initial_trust_region_radius = 1e4;
  o->max_trust_region_radius = 1e16;
  o->min_trust_region_radius = 1e-32;
  o->min_relative_decrease = 1e-3;
  o->min_lm_diagonal = 1e-6;
  o->max_lm_diagonal = 1e32;
  o->max_num_consecutive_invalid_steps = 5;
  o->jacobi_scaling = 1;
  o->loss_type = TSCM_LOSS_NONE;
  o->loss_scale = 1.0;
  o->num_gpus = 1;
}

// Page-locking 56 MB costs 15-30 ms and unlocking it as much again — more than the solve of a warm
// start.  The last block handed back is therefore kept (one slot, like the solver cache and under the
// same switch: tscm_cache_configure(0) turns it off, tscm_cache_release() frees it).
void* tscm_host_alloc(size_t bytes) {
  bytes = std::max<size_t>(1, bytes);
  {
    std::lock_guard<std::mutex> lock(g_cache_mu);
    if (g_host_block && !g_host_busy && g_host_bytes >= bytes) { g_host_busy = true; return g_host_block; }
  }
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) {
    set_error("cudaMallocHost(%zu) failed", bytes);
    cudaGetLastError();
    return nullptr;
  }
  std::lock_guard<std::mutex> lock(g_cache_mu);
  if (g_cache_max > 0 && !g_host_busy) {           // this block becomes the cached one
    if (g_host_block) cudaFreeHost(g_host_block);
    g_host_block = p; g_host_bytes = bytes; g_host_busy = true;
  }
  return p;
}
void tscm_host_free(void* p) {
  if (!p) return;
  {
    std::lock_guard<std::mutex> lock(g_cache_mu);
    if (p == g_host_block) {
      if (g_cache_max > 0) { g_host_busy = false; return; }
      g_host_block = nullptr; g_host_bytes = 0; g_host_busy = false;
    }
  }
  cudaFreeHost(p);
}

int tscm_solver_set_options(tscm_solver* s, const tscm_options* o) {
  if (!s || !o) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  RC_TRY(validate_options(o));
  if (o->allow_large_rigs != s->options.allow_large_rigs) {
    set_error("allow_large_rigs is fixed when the solver is created");
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  s->options = *o;
  return for_shards(s, [&](tscm_solver* k, int) -> int {
    LmOptions lm{};
    fill_lm_options(*o, lm);
    // the options are kernel arguments baked into the iteration graph
    if (!lm_equal(lm, k->lm)) k->graph_dirty = true;
    k->lm = lm;
    k->options = *o;
    return TSCM_OK;
  });
}

int tscm_solver_create(const tscm_problem* p, const tscm_options* o, int device, tscm_solver** out) {
  internal::DeviceScope device_scope;
  if (!out) { set_error("out is NULL"); return TSCM_ERR_INVALID_ARGUMENT; }
  *out = nullptr;
  const auto t0 = Clock::now();
  RC_TRY(validate_problem(p, false));
  tscm_options defaults;
  tscm_options_init(&defaults);
  if (!o) o = &defaults;
  RC_TRY(validate_options(o));
  RC_TRY(validate_large_rig(p, o));
  internal::SelectedDevice dev;
  RC_TRY(internal::select_device(device, "the calibration solve", &dev));
  if (g_debug & 1) std::fprintf(stderr, "[tscm create] %-28s %8.2f ms\n", "validate", ms_since(t0));
  const int n = std::max(1, o->num_gpus);
  if (n > 1) return create_group(p, o, dev, n, out);
  return create_shard(p, o, dev, false, out);
}

void tscm_solver_destroy(tscm_solver* s) {
  internal::DeviceScope device_scope;
  destroy_solver(s);
}

int tscm_solver_set_observations(tscm_solver* s, const double* obs_xy) {
  internal::DeviceScope device_scope;
  if (!s || !obs_xy) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  RC_TRY(upload_all_observations(s, obs_xy));
  return sync_shards(s);     // the caller may reuse obs_xy
}

int tscm_solver_set_parameters(tscm_solver* s, const double* intr, const double* cam_rt,
                               const double* board_rt) {
  internal::DeviceScope device_scope;
  if (!s || !intr || !cam_rt || !board_rt) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  RC_TRY(for_shards(s, [&](tscm_solver* k, int i) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    const double* brt = s->kids.empty() ? board_rt : board_rt + (size_t)s->kid_frame[i] * 6;
    // The initial point always goes to parameter set 0; run() starts with cur = 0.
    CUDA_TRY(cudaMemcpyAsync(k->ps[0].intr, intr, (size_t)k->C * 9 * sizeof(double), cudaMemcpyHostToDevice, k->stream));
    CUDA_TRY(cudaMemcpyAsync(k->ps[0].cam_rt, cam_rt, (size_t)k->C * 6 * sizeof(double), cudaMemcpyHostToDevice, k->stream));
    CUDA_TRY(cudaMemcpyAsync(k->ps[0].board_rt, brt, (size_t)k->F * 6 * sizeof(double), cudaMemcpyHostToDevice, k->stream));
    // the constant block and the b, c intrinsics must also exist in set 1
    CUDA_TRY(cudaMemcpyAsync(k->ps[1].intr, intr, (size_t)k->C * 9 * sizeof(double), cudaMemcpyHostToDevice, k->stream));
    CUDA_TRY(cudaMemcpyAsync(k->ps[1].cam_rt, cam_rt, (size_t)k->C * 6 * sizeof(double), cudaMemcpyHostToDevice, k->stream));
    CUDA_TRY(cudaMemsetAsync(k->d_state, 0, sizeof(LmState), k->stream));
    k->x_in_set1 = false;
    return TSCM_OK;
  }));
  return sync_shards(s);
}

int tscm_solver_get_parameters(tscm_solver* s, double* intr, double* cam_rt, double* board_rt) {
  internal::DeviceScope device_scope;
  if (!s) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  RC_TRY(for_shards(s, [&](tscm_solver* k, int i) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    const ParamSet& ps = k->ps[k->x_in_set1 ? 1 : 0];
    double* brt = board_rt ? (s->kids.empty() ? board_rt : board_rt + (size_t)s->kid_frame[i] * 6) : nullptr;
    if (i == 0 && intr) CUDA_TRY(cudaMemcpyAsync(intr, ps.intr, (size_t)k->C * 9 * sizeof(double), cudaMemcpyDeviceToHost, k->stream));
    if (i == 0 && cam_rt) CUDA_TRY(cudaMemcpyAsync(cam_rt, ps.cam_rt, (size_t)k->C * 6 * sizeof(double), cudaMemcpyDeviceToHost, k->stream));
    if (brt) CUDA_TRY(cudaMemcpyAsync(brt, ps.board_rt, (size_t)k->F * 6 * sizeof(double), cudaMemcpyDeviceToHost, k->stream));
    return TSCM_OK;
  }));
  return sync_shards(s);
}

int tscm_solver_run(tscm_solver* s, tscm_summary* summary) {
  internal::DeviceScope device_scope;
  if (!s) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  const int max_it = s->options.max_num_iterations;
  // ---- prepare every shard (no exchange kernels yet) -----------------------------------------
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    RC_TRY(ensure_trace(k, std::min(max_it, 1 << 16) + 2));
    RC_TRY(move_x_to_set0(k));
    return ensure_graph(k);
  }));
  // ---- iteration zero on every shard, then batches of iterations ------------------------------
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    return run_initial(k);
  }));
  // Replay the iteration graph in batches; the device-side `done` flag of the batch BEFORE the
  // one just enqueued is polled, so the GPU never waits for the host (kernels of a finished
  // solve are no-ops).
  tscm_solver* L = lead(s);
  const bool group = !s->kids.empty();
  const int batch = 8;
  int launched = 0, nbatch = 0;
  bool done = false;
  while (launched < max_it && !done) {
    const int n = std::min(batch, max_it - launched);
    RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
      CUDA_TRY(cudaSetDevice(k->device));
      int left = n;
      if (group)
        for (; left >= kGroupIters; left -= kGroupIters) CUDA_TRY(cudaGraphLaunch(k->graph_exec_n, k->stream));
      for (; left > 0; --left) CUDA_TRY(cudaGraphLaunch(k->graph_exec, k->stream));
      k->launches += (int64_t)n * k->launches_per_iter;
      return TSCM_OK;
    }));
    launched += n;
    CUDA_TRY(cudaSetDevice(L->device));
    CUDA_TRY(cudaMemcpyAsync(L->h_state + 1 + (nbatch & 1), L->d_state, sizeof(LmState), cudaMemcpyDeviceToHost, L->stream));
    CUDA_TRY(cudaEventRecord(L->poll_ev[nbatch & 1], L->stream));
    if (nbatch > 0) {
      CUDA_TRY(cudaEventSynchronize(L->poll_ev[(nbatch - 1) & 1]));
      done = L->h_state[1 + ((nbatch - 1) & 1)].done != 0;
    }
    ++nbatch;
  }
  // ---- results ----------------------------------------------------------------------------------
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    CUDA_TRY(cudaMemcpyAsync(k->h_state, k->d_state, sizeof(LmState), cudaMemcpyDeviceToHost, k->stream));
    if (k->p2p_on) CUDA_TRY(cudaMemcpyAsync(k->h_err, k->d_p2p_err, sizeof(int), cudaMemcpyDeviceToHost, k->stream));
    return TSCM_OK;
  }));
  const int want_trace = summary ? std::min(std::max(0, (int)summary->trace_capacity), L->trace.capacity) : 0;
  if (want_trace > 0) {
    CUDA_TRY(cudaSetDevice(L->device));
    CUDA_TRY(cudaMemcpyAsync(L->h_trace, L->d_trace, trace_bytes(L->trace.capacity), cudaMemcpyDeviceToHost, L->stream));
  }
  RC_TRY(sync_shards(s));
  int comm_err = 0;
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    CUDA_TRY(cudaGetLastError());
    k->x_in_set1 = (k->h_state->cur & 1) != 0;
    if (k->p2p_on && *k->h_err) comm_err = 1;
    return TSCM_OK;
  }));
  const LmState& st = *L->h_state;
  if (summary) {
    summary->termination_type = st.done ? st.termination : TSCM_NO_CONVERGENCE;
    summary->num_iterations = st.recorded;
    summary->num_successful_steps = st.num_successful;
    summary->num_unsuccessful_steps = st.num_unsuccessful;
    summary->initial_cost = st.initial_cost;
    summary->final_cost = st.final_cost;
    summary->final_radius = st.radius;
    const int n = std::min(st.recorded, want_trace);
    if (n > 0) {
      const size_t cap = (size_t)L->trace.capacity;
      const double* h = reinterpret_cast<const double*>(L->h_trace);
      if (summary->trace_cost) std::memcpy(summary->trace_cost, h, n * sizeof(double));
      if (summary->trace_radius) std::memcpy(summary->trace_radius, h + cap, n * sizeof(double));
      if (summary->trace_gradient_max_norm) std::memcpy(summary->trace_gradient_max_norm, h + 2 * cap, n * sizeof(double));
      if (summary->trace_step_norm) std::memcpy(summary->trace_step_norm, h + 3 * cap, n * sizeof(double));
      if (summary->trace_step_flags) std::memcpy(summary->trace_step_flags, h + 4 * cap, n * sizeof(int));
    }
  }
  if (comm_err) { set_error("peer-memory exchange timed out waiting for another rank"); return TSCM_ERR_COMM; }
  if (s->options.verbose && L->rank == 0) {
    // summary.BriefReport() of TS.cpp:280 / multi_calib.cpp:218
    std::printf("Ceres Solver Report: Iterations: %d, Initial cost: %e, Final cost: %e, Termination: %s\n",
                st.num_successful + st.num_unsuccessful, st.initial_cost, st.final_cost,
                termination_name(st.done ? st.termination : TSCM_NO_CONVERGENCE));
  }
  return TSCM_OK;
}

void tscm_cache_configure(int32_t max_solvers) {
  internal::DeviceScope device_scope;
  std::lock_guard<std::mutex> lock(g_cache_mu);
  g_cache_max = std::max(0, (int)max_solvers);
  while ((int)g_cache.size() > g_cache_max) cache_evict_oldest_locked();
  if (g_cache_max == 0 && g_host_block && !g_host_busy) { cudaFreeHost(g_host_block); g_host_block = nullptr; g_host_bytes = 0; }
}
void tscm_cache_release(void) {
  internal::DeviceScope device_scope;
  std::lock_guard<std::mutex> lock(g_cache_mu);
  for (CacheEntry& e : g_cache) destroy_solver(e.solver);
  g_cache.clear();
  if (g_host_block && !g_host_busy) { cudaFreeHost(g_host_block); g_host_block = nullptr; g_host_bytes = 0; }
}

int tscm_solve(const tscm_problem* problem, const tscm_options* options, double* intrinsics,
               double* cam_rt, double* board_rt, tscm_summary* summary, int device) {
  internal::DeviceScope device_scope;
  const auto t0 = Clock::now();
  RC_TRY(validate_problem(problem, true));
  if (!intrinsics || !cam_rt || !board_rt) { set_error("NULL parameter arrays"); return TSCM_ERR_INVALID_ARGUMENT; }
  // ---- solver: cached for this structure, or new ---------------------------------------------
  const double ms_lookup = ms_since(t0);
  Checkout c;
  RC_TRY(checkout_solver(problem, options, device, "the calibration solve", &c));
  tscm_solver* s = c.s;
  const double ms_create = ms_since(t0);
  // the parameters ride behind the observations on the same streams (one sync for both)
  int rc = tscm_solver_set_parameters(s, intrinsics, cam_rt, board_rt);
  const double ms_set = ms_since(t0);
  if (!rc) rc = tscm_solver_run(s, summary);
  const double ms_run = ms_since(t0);
  if (!rc) rc = tscm_solver_get_parameters(s, intrinsics, cam_rt, board_rt);
  const double ms_get = ms_since(t0);
  cache_checkin(s, c.device, c.ngpu, rc == TSCM_OK);
  if (g_debug & 1)
    std::fprintf(stderr, "[tscm_solve] %s: lookup %.2f  create/upload %.2f  set %.2f  run %.2f  get %.2f  total %.2f ms\n",
                 c.hit ? "cached solver" : "new solver", ms_lookup, ms_create - ms_lookup, ms_set - ms_create,
                 ms_run - ms_set, ms_get - ms_run, ms_since(t0));
  return rc;
}

int tscm_comm_unique_id(void* unique_id_128) {
  NcclApi& n = nccl();
  if (!n.ok) { set_error("libnccl.so.2 could not be loaded"); return TSCM_ERR_COMM; }
  NcclApi::UniqueId id;
  int rc = n.GetUniqueId(&id);
  if (rc) { set_error("ncclGetUniqueId failed: %d", rc); return TSCM_ERR_COMM; }
  std::memcpy(unique_id_128, &id, 128);
  return TSCM_OK;
}

#define NO_GROUP(s, what)                                                                           \
  do {                                                                                              \
    if (!(s)->kids.empty()) {                                                                       \
      set_error(what " works on single-device solvers (num_gpus <= 1)");                            \
      return TSCM_ERR_UNSUPPORTED;                                                                  \
    }                                                                                               \
  } while (0)

// Sharded solves exchange the reduced system at the default size limit only.
static int no_large_shards(const tscm_solver* s) {
  if (s->P.NL <= kCovMaxNL) return TSCM_OK;
  set_error("reduced system of %d live parameters: multi-process solves support at most %d", s->P.NL, kCovMaxNL);
  return TSCM_ERR_UNSUPPORTED;
}

int tscm_solver_attach_comm(tscm_solver* s, int rank, int num_ranks, const void* unique_id_128) {
  internal::DeviceScope device_scope;
  if (!s || !unique_id_128 || rank < 0 || rank >= num_ranks) { set_error("bad comm arguments"); return TSCM_ERR_INVALID_ARGUMENT; }
  NO_GROUP(s, "tscm_solver_attach_comm");
  RC_TRY(no_large_shards(s));
  NcclApi& n = nccl();
  if (!n.ok) { set_error("libnccl.so.2 could not be loaded"); return TSCM_ERR_COMM; }
  CUDA_TRY(cudaSetDevice(s->device));
  NcclApi::UniqueId id;
  std::memcpy(&id, unique_id_128, 128);
  int rc = n.CommInitRank(&s->comm, num_ranks, id, rank);
  if (rc) { set_error("ncclCommInitRank failed: %d", rc); return TSCM_ERR_COMM; }
  s->rank = rank; s->num_ranks = num_ranks;
  s->graph_dirty = true;
  return TSCM_OK;
}

int tscm_solver_p2p_export(tscm_solver* s, void* handle_64) {
  internal::DeviceScope device_scope;
  if (!s || !handle_64) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  NO_GROUP(s, "tscm_solver_p2p_export");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  CUDA_TRY(cudaSetDevice(s->device));
  CUDA_TRY(cudaStreamSynchronize(s->stream));      // the mailbox is zeroed before anyone maps it
  cudaIpcMemHandle_t h;
  CUDA_TRY(cudaIpcGetMemHandle(&h, s->d_mailbox));
  std::memcpy(handle_64, &h, 64);
  return TSCM_OK;
}

int tscm_solver_p2p_attach(tscm_solver* s, int rank, int num_ranks, const void* handles) {
  internal::DeviceScope device_scope;
  if (!s || !handles || rank < 0 || rank >= num_ranks) { set_error("bad p2p arguments"); return TSCM_ERR_INVALID_ARGUMENT; }
  NO_GROUP(s, "tscm_solver_p2p_attach");
  RC_TRY(no_large_shards(s));
  if (num_ranks > kP2PMaxRanks) { set_error("peer-memory exchange supports at most %d ranks", kP2PMaxRanks); return TSCM_ERR_INVALID_ARGUMENT; }
  CUDA_TRY(cudaSetDevice(s->device));
  for (int r = 0; r < num_ranks; ++r) {
    if (r == rank) { s->p2p.mb[r] = s->d_mailbox; continue; }
    cudaIpcMemHandle_t h;
    std::memcpy(&h, (const char*)handles + 64 * r, 64);
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      set_error("cudaIpcOpenMemHandle(rank %d) failed: %s", r, cudaGetErrorString(e));
      return TSCM_ERR_COMM;
    }
    s->p2p_ipc[r] = ptr;
    s->p2p.mb[r] = static_cast<double*>(ptr);
  }
  s->p2p.rank = rank; s->p2p.world = num_ranks;
  s->rank = rank; s->num_ranks = num_ranks;
  s->p2p_on = true;
  s->graph_dirty = true;
  return TSCM_OK;
}

int tscm_solver_set_exchange_timeout(tscm_solver* s, double seconds) {
  if (!s || !(seconds > 0.0)) { set_error("bad arguments"); return TSCM_ERR_INVALID_ARGUMENT; }
  return for_shards(s, [&](tscm_solver* k, int) -> int {
    k->p2p.timeout_ns = (unsigned long long)(seconds * 1e9);
    k->graph_dirty = true;
    return TSCM_OK;
  });
}

int tscm_solver_set_schur_form(tscm_solver* s, int form) {
  internal::DeviceScope device_scope;
  if (!s) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  return for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    const int f = form == kSchurAuto ? choose_schur_form(k) : form;
    if (f == k->schur_form) return TSCM_OK;
    CUDA_TRY(cudaStreamSynchronize(k->stream));
    Arena a;
    Blob b;
    RC_TRY(plan_schur(k, f, a, b));
    char* d_blob = nullptr;
    a.want(&d_blob, b.bytes.size());
    RC_TRY(a.commit(k->stream));
    k->extra.push_back(a.base);
    b.d_base = d_blob;
    RC_TRY(b.upload(k->stream));
    return wire_schur(k, f);
  });
}

int tscm_solver_set_reduced_solve(tscm_solver* s, int form) {
  internal::DeviceScope device_scope;
  if (!s || form < 0 || form > 2) { set_error("bad arguments"); return TSCM_ERR_INVALID_ARGUMENT; }
  return for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    const bool fits = single_cta_fits(k);
    const bool cluster = form == 2 || (form == 0 && !fits);
    if (!cluster && !fits) {
      set_error("the single-CTA solve cannot hold a reduced system of %d live parameters (limit %d)", k->P.NL,
                kCovMaxNL);
      return TSCM_ERR_UNSUPPORTED;
    }
    if (cluster) {
      CUDA_TRY(cudaStreamSynchronize(k->stream));
      RC_TRY(ensure_cluster(k));
    } else {
      RC_TRY(set_smem_attr((const void*)k_solve<1, 4>, k->solve.smem));
      RC_TRY(set_smem_attr((const void*)k_solve<4, 7>, k->solve.smem));
    }
    k->use_cluster = cluster;
    k->graph_dirty = true;
    return TSCM_OK;
  });
}

int tscm_solver_eval_jacobian(tscm_solver* s, double* residuals, double* jacobian, double* cost) {
  internal::DeviceScope device_scope;
  if (!s) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  NO_GROUP(s, "tscm_solver_eval_jacobian");
  CUDA_TRY(cudaSetDevice(s->device));
  const int cur = s->x_in_set1 ? 1 : 0;
  const size_t N = (size_t)s->V * s->K;
  internal::Scratch scratch;
  double *d_r = nullptr, *d_J = nullptr;
  if (residuals) CUDA_TRY(scratch.alloc(&d_r, N * 2));
  if (jacobian) CUDA_TRY(scratch.alloc(&d_J, N * 42));
  k_prep_cams<<<(s->C + 31) / 32, 32, 0, s->stream>>>(s->P, s->ps[0], s->ps[1], s->d_state, 2 + cur);
  k_eval_rows<<<(unsigned)((N + 127) / 128), 128, 0, s->stream>>>(s->P, s->ps[cur], s->lm, d_r, d_J);
  s->launches += 2;
  if (cost) {
    launch_evaluation(s, 2 + cur, 1);
    RC_TRY(launch_eval_allreduce(s, 2 + cur));
  }
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  CUDA_TRY(cudaGetLastError());
  if (residuals) CUDA_TRY(cudaMemcpy(residuals, d_r, N * 2 * sizeof(double), cudaMemcpyDeviceToHost));
  if (jacobian) CUDA_TRY(cudaMemcpy(jacobian, d_J, N * 42 * sizeof(double), cudaMemcpyDeviceToHost));
  if (cost) {
    std::vector<double> comm((size_t)s->C * kCamRec);
    CUDA_TRY(cudaMemcpy(comm.data(), s->ps[cur].comm, comm.size() * sizeof(double), cudaMemcpyDeviceToHost));
    double c = 0.0;
    for (int m = 0; m < s->C; ++m) c += comm[(size_t)m * kCamRec + kCamCost];
    *cost = c;
  }
  return TSCM_OK;
}

int tscm_solver_reduced_size(const tscm_solver* s) {
  if (!s) return -1;
  return s->kids.empty() ? s->P.NL : s->kids[0]->P.NL;
}

int tscm_solver_reduced_system(tscm_solver* s, double radius, double* lhs, double* rhs) {
  internal::DeviceScope device_scope;
  if (!s || !(radius > 0.0)) { set_error("bad arguments"); return TSCM_ERR_INVALID_ARGUMENT; }
  NO_GROUP(s, "tscm_solver_reduced_system");
  CUDA_TRY(cudaSetDevice(s->device));
  RC_TRY(assemble_at(s, radius));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  CUDA_TRY(cudaGetLastError());
  // the assembled system as k_solve receives it (4x4 tiles of the lower block triangle)
  const int NL = s->P.NL, nbk = s->solve.nbk;
  std::vector<double> tiles((size_t)s->solve.ntile * 16);
  CUDA_TRY(cudaMemcpy(tiles.data(), s->d_Sr, tiles.size() * sizeof(double), cudaMemcpyDeviceToHost));
  auto at = [&](int r, int c) { return tiles[(size_t)solve_tile_id(r >> 2, c >> 2, nbk) * 16 + (r & 3) * 4 + (c & 3)]; };
  for (int r = 0; r < NL; ++r)
    for (int c = 0; c <= r; ++c) {
      if (lhs) { lhs[(size_t)r * NL + c] = at(r, c); lhs[(size_t)c * NL + r] = at(r, c); }
    }
  if (rhs) for (int c = 0; c < NL; ++c) rhs[c] = at(NL, c);
  return TSCM_OK;
}

// Mean Euclidean reprojection error per camera and overall (multi_calib.cpp:235-283).  On a
// sharded solve (ranks or a num_gpus group) the sums are global, and so must the counts be: a
// group knows them; the ranks of a multi-process solve exchange them like an evaluation record.
int tscm_solver_reprojection_error(tscm_solver* s, double* per_camera, double* overall, double* rms) {
  internal::DeviceScope device_scope;
  if (!s) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  const int C = s->C;
  // Read-out uses the plain (loss-free) residuals, like multi_calib.cpp:235-283.
  RC_TRY(evaluate_shards(s, /*plain=*/true, /*want_err=*/true));
  tscm_solver* L = lead(s);
  const int cur = L->x_in_set1 ? 1 : 0;
  CUDA_TRY(cudaSetDevice(L->device));
  CUDA_TRY(cudaGetLastError());
  std::vector<double> comm((size_t)C * kCamRec);
  CUDA_TRY(cudaMemcpy(comm.data(), L->ps[cur].comm, comm.size() * sizeof(double), cudaMemcpyDeviceToHost));
  std::vector<double> count = L->obs_count;
  const bool multi_process = s->kids.empty() && s->num_ranks > 1;
  if (multi_process) {
    // exchange the local counts through the record's err slot
    std::vector<double> rec((size_t)C * kCamRec + kCommExtra, 0.0);
    for (int m = 0; m < C; ++m) rec[(size_t)m * kCamRec + kCamErr] = L->obs_count[m];
    RC_TRY(allreduce_record(L, rec));
    for (int m = 0; m < C; ++m) count[m] = rec[(size_t)m * kCamRec + kCamErr];
  }
  double sum = 0.0, cost = 0.0, total = 0.0;
  for (int m = 0; m < C; ++m) {
    const double e = comm[(size_t)m * kCamRec + kCamErr];
    const double n = count[m];
    if (per_camera) per_camera[m] = n > 0 ? e / n : 0.0;
    sum += e; total += n;
    cost += comm[(size_t)m * kCamRec + kCamCost];
  }
  if (overall) *overall = total > 0 ? sum / total : 0.0;
  if (rms) *rms = total > 0 ? std::sqrt(2.0 * cost / total) : 0.0;
  // restore the records of the configured loss for a subsequent run()
  if (L->lm.loss_type || multi_process) RC_TRY(evaluate_shards(s, /*plain=*/false, /*want_err=*/false));
  return TSCM_OK;
}

// Covariance of the live parameters at the current point (DESIGN.md 5e, tscm_covariance.cuh).
// Collective on a sharded solve, like run(): every shard assembles the undamped system over the
// usual exchange and inverts S~ redundantly; each shard computes the blocks of its own frames.
int tscm_solver_covariance(tscm_solver* s, tscm_covariance* out) {
  internal::DeviceScope device_scope;
  if (!s || !out) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  const int C = s->C;
  tscm_solver* L = lead(s);
  const int NL = L->P.NL;
  const bool multi_process = s->kids.empty() && s->num_ranks > 1;
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    return ensure_cov_buffers(k);
  }));
  // sum |r|^2 of the plain (loss-free) residuals
  RC_TRY(evaluate_shards(s, /*plain=*/true, /*want_err=*/false));
  const int cur = L->x_in_set1 ? 1 : 0;
  CUDA_TRY(cudaSetDevice(L->device));
  CUDA_TRY(cudaGetLastError());
  std::vector<double> rec((size_t)C * kCamRec + kCommExtra, 0.0);
  CUDA_TRY(cudaMemcpy(rec.data(), L->ps[cur].comm, (size_t)C * kCamRec * sizeof(double), cudaMemcpyDeviceToHost));
  double rr = 0.0;
  for (int m = 0; m < C; ++m) rr += 2.0 * rec[(size_t)m * kCamRec + kCamCost];
  // the undamped system under the configured loss (which also restores that loss's records for a
  // later run()), then the covariance kernels
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    return assemble_at(k, INFINITY);
  }));
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    return launch_covariance(k);
  }));
  RC_TRY(sync_shards(s));
  int flag = 0;
  double ms = 0.0;
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    CUDA_TRY(cudaGetLastError());
    int f = 0;
    CUDA_TRY(cudaMemcpy(&f, k->d_cov_flag, sizeof(int), cudaMemcpyDeviceToHost));
    flag |= f;
    float e = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&e, k->cov_ev[0], k->cov_ev[1]));
    ms = std::max(ms, (double)e);
    return TSCM_OK;
  }));
  // global counts: a group knows them; the ranks of a multi-process solve exchange them (and the
  // frame rank test) through an evaluation record, as tscm_solver_reprojection_error does
  std::vector<double> count = L->obs_count;
  double frames = s->F;
  if (multi_process) {
    std::fill(rec.begin(), rec.end(), 0.0);
    for (int m = 0; m < C; ++m) rec[(size_t)m * kCamRec + kCamErr] = L->obs_count[m];
    rec[kCamCost] = L->F;
    rec[(size_t)C * kCamRec] = (flag & 2) ? 1.0 : 0.0;
    RC_TRY(allreduce_record(L, rec));
    for (int m = 0; m < C; ++m) count[m] = rec[(size_t)m * kCamRec + kCamErr];
    frames = rec[kCamCost];
    if (rec[(size_t)C * kCamRec] > 0.0) flag |= 2;
    // restore the records of the configured loss
    RC_TRY(evaluate_shards(s, /*plain=*/false, /*want_err=*/false));
    CUDA_TRY(cudaGetLastError());
  }
  if (flag) {
    set_error((flag & 1) ? "covariance: J^T J is rank deficient in the camera parameters (a gauge freedom: "
                           "is no camera fixed?)"
                         : "covariance: J^T J is rank deficient in a board pose (a degenerate board)");
    return TSCM_ERR_RANK_DEFICIENT;
  }
  double N = 0.0;
  for (int m = 0; m < C; ++m) N += count[m];
  const double dof = 2.0 * N - (NL + 6.0 * frames);
  out->residual_variance = dof > 0.0 ? rr / dof : NAN;
  out->kernel_ms = ms;
  if (out->camera) {
    CUDA_TRY(cudaSetDevice(L->device));
    CUDA_TRY(cudaMemcpy(out->camera, L->d_cov_cam, (size_t)NL * NL * sizeof(double), cudaMemcpyDeviceToHost));
    for (int r = 0; r < NL; ++r)          // columns are solved independently: average the two triangles
      for (int c = 0; c < r; ++c) {
        const double v = 0.5 * (out->camera[(size_t)r * NL + c] + out->camera[(size_t)c * NL + r]);
        out->camera[(size_t)r * NL + c] = v;
        out->camera[(size_t)c * NL + r] = v;
      }
  }
  if (out->board) {
    RC_TRY(for_shards(s, [&](tscm_solver* k, int i) -> int {
      CUDA_TRY(cudaSetDevice(k->device));
      double* dst = out->board + (s->kids.empty() ? 0 : (size_t)s->kid_frame[i] * 36);
      CUDA_TRY(cudaMemcpy(dst, k->d_cov_board, (size_t)k->F * 36 * sizeof(double), cudaMemcpyDeviceToHost));
      return TSCM_OK;
    }));
  }
  return TSCM_OK;
}

int tscm_compute_covariance(const tscm_problem* problem, const tscm_options* options, const double* intrinsics,
                    const double* cam_rt, const double* board_rt, tscm_covariance* cov, int device) {
  internal::DeviceScope device_scope;
  RC_TRY(validate_problem(problem, true));
  if (!intrinsics || !cam_rt || !board_rt || !cov) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  // the solver cache of tscm_solve(): after a solve of this structure only data is uploaded
  Checkout c;
  RC_TRY(checkout_solver(problem, options, device, "the covariance", &c));
  int rc = tscm_solver_set_parameters(c.s, intrinsics, cam_rt, board_rt);
  if (!rc) rc = tscm_solver_covariance(c.s, cov);
  cache_checkin(c.s, c.device, c.ngpu, rc == TSCM_OK || rc == TSCM_ERR_RANK_DEFICIENT);
  return rc;
}

int tscm_solver_time_stage(tscm_solver* s, int stage, int repeats, double* ms_per_launch) {
  internal::DeviceScope device_scope;
  if (!s || repeats <= 0 || !ms_per_launch) { set_error("bad arguments"); return TSCM_ERR_INVALID_ARGUMENT; }
  if (stage != 4) NO_GROUP(s, "tscm_solver_time_stage (stages other than 4)");
  RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
    CUDA_TRY(cudaSetDevice(k->device));
    RC_TRY(move_x_to_set0(k));
    return ensure_graph(k);
  }));
  tscm_solver* L = lead(s);
  CUDA_TRY(cudaSetDevice(L->device));
  internal::Scratch timer;
  CUDA_TRY(timer.create_events());
  if (stage != 4) {
    // make the device state valid and not `done`
    LmOptions saved = s->lm;
    s->lm.disable_tolerances = 1; s->lm.max_num_iterations = 1 << 30;
    int rc = run_initial(s);
    if (!rc) { launch_schur(s, 0.0); rc = launch_schur_allreduce(s, 0.0); }
    if (!rc) { launch_solve(s); launch_backsub(s); launch_evaluation(s, 3, 0); }
    if (rc) { s->lm = saved; return rc; }
    CUDA_TRY(cudaStreamSynchronize(s->stream));
    CUDA_TRY(cudaEventRecord(timer.e0, s->stream));
    for (int r = 0; r < repeats; ++r) {
      switch (stage) {
        case 0: launch_eval_kernel(s, 3); break;
        case 1: launch_schur(s, 0.0); break;
        case 2: launch_solve(s); break;
        case 3: launch_backsub(s); break;
        case 5: launch_evaluation(s, 3, 0); break;
        case 6: launch_eval_kernel(s, 3, 1); break;
        case 7: launch_eval_kernel(s, 3, 2); break;
        default: s->lm = saved; set_error("unknown stage %d", stage); return TSCM_ERR_INVALID_ARGUMENT;
      }
    }
    CUDA_TRY(cudaEventRecord(timer.e1, s->stream));
    s->lm = saved;
  } else {
    // whole LM iterations: iteration zero, then replay the graph.  The options
    // baked into the graph are the solver's (use disable_tolerances = 1 and
    // max_num_iterations >= repeats for a fixed-iteration measurement).
    RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
      CUDA_TRY(cudaSetDevice(k->device));
      return run_initial(k);
    }));
    RC_TRY(sync_shards(s));
    CUDA_TRY(cudaSetDevice(L->device));
    CUDA_TRY(cudaEventRecord(timer.e0, L->stream));
    const bool group = !s->kids.empty();
    int left = repeats;
    while (left > 0) {
      const int n = group && left >= kGroupIters ? kGroupIters : 1;
      RC_TRY(for_shards(s, [&](tscm_solver* k, int) -> int {
        CUDA_TRY(cudaSetDevice(k->device));
        CUDA_TRY(cudaGraphLaunch(n == 1 ? k->graph_exec : k->graph_exec_n, k->stream));
        k->launches += (int64_t)n * k->launches_per_iter;
        return TSCM_OK;
      }));
      left -= n;
    }
    CUDA_TRY(cudaSetDevice(L->device));
    CUDA_TRY(cudaEventRecord(timer.e1, L->stream));
  }
  double ms = 0.0;
  CUDA_TRY(timer.add_ms(&ms));
  RC_TRY(sync_shards(s));
  CUDA_TRY(cudaSetDevice(L->device));
  CUDA_TRY(cudaGetLastError());
  *ms_per_launch = ms / repeats;
  // where x ended up (the timed stages evaluate set 1 explicitly and never flip `cur`)
  RC_TRY(fetch_state(L));
  const bool in1 = (L->h_state->cur & 1) != 0;
  for_shards(s, [&](tscm_solver* k, int) -> int { k->x_in_set1 = in1; return TSCM_OK; });
  if (stage == 4) {
    // a solve that terminated early turns the remaining launches into no-ops:
    // such a measurement is not a measurement
    if (L->h_state->done || L->h_state->iteration != repeats) {
      set_error("LM loop stopped after %d of %d timed iterations (termination %d)",
                L->h_state->iteration, repeats, L->h_state->termination);
      return TSCM_ERR_UNSUPPORTED;
    }
  }
  return TSCM_OK;
}

int64_t tscm_solver_launch_count(const tscm_solver* s) {
  if (!s) return 0;
  int64_t n = s->launches;
  for (const tscm_solver* k : s->kids) n += k->launches;
  return n;
}

int tscm_device_fp64_peak(int device, double* tflops) {
  internal::DeviceScope device_scope;
  if (!tflops) { set_error("NULL argument"); return TSCM_ERR_INVALID_ARGUMENT; }
  internal::SelectedDevice dev;
  RC_TRY(internal::select_device(device, "the FP64 peak measurement", &dev));
  internal::Scratch scratch;
  double* d_out = nullptr;
  const int blocks = dev.sm_count * 8, threads = 256, iters = 4096;
  CUDA_TRY(scratch.alloc(&d_out, (size_t)blocks * threads));
  CUDA_TRY(scratch.create_events());
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(scratch.e0));
    k_dfma_peak<<<blocks, threads>>>(d_out, iters, 1.0000001);
    CUDA_TRY(cudaEventRecord(scratch.e1));
    double ms = 0.0;
    CUDA_TRY(scratch.add_ms(&ms));
    const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
    if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  CUDA_TRY(cudaGetLastError());
  *tflops = best;
  return TSCM_OK;
}

}  // extern "C"
