// tscm_internal.h — the host helpers shared by the translation units of libtscm_b200.so (defined in
// tscm_b200.cu; not part of the C-ABI, hidden from the dynamic symbol table).  The translation units:
//   tscm_b200.cu       the solver: creation, run, read-outs, covariance, the tscm_solve() cache
//   tscm_remap.cu      tscm_remap_tables()    (kernel: tscm_remap.cuh)
//   tscm_posegraph.cu  tscm_pose_graph_init() (kernels: tscm_posegraph.cuh)
//   tscm_monoinit.cu   tscm_mono_init()       (kernels in the file; compiled with -fmad=false)
#pragma once

#include <cuda_runtime.h>

#include <cstddef>
#include <vector>

#include "../../include/tscm.h"

namespace tscm {
namespace internal {

// printf-style text behind tscm_last_error() of the calling thread
__attribute__((visibility("hidden"))) void set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                                          \
  do {                                                                                                          \
    cudaError_t e_ = (expr);                                                                                    \
    if (e_ != cudaSuccess) {                                                                                    \
      ::tscm::internal::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return TSCM_ERR_CUDA;                                                                                     \
    }                                                                                                           \
  } while (0)
#define RC_TRY(expr)            \
  do {                          \
    const int rc_ = (expr);     \
    if (rc_) return rc_;        \
  } while (0)

struct SelectedDevice {
  int index = 0;         // the device made current
  int visible = 0;       // devices visible to the process
  int sm_count = 0;
  size_t smem_optin = 0; // opt-in shared memory per block
};

// The device check of every entry point; there is no CPU fallback anywhere in the library.  In
// order: a CUDA device exists (`what` names the caller in the error text), a negative `device`
// means the current one, that device exists and is sm_100.  Then makes it current and fills *out
// (optional).  Returns a TSCM_* code: TSCM_ERR_NO_DEVICE for each failed check.
__attribute__((visibility("hidden"))) int select_device(int device, const char* what, SelectedDevice* out);

// restores the caller's current device on scope exit
struct __attribute__((visibility("hidden"))) DeviceScope {
  int prev = -1;
  DeviceScope();
  ~DeviceScope();
};

// The device memory and the start/stop event pair of one call, released on scope exit.
class __attribute__((visibility("hidden"))) Scratch {
 public:
  Scratch() = default;
  Scratch(const Scratch&) = delete;
  Scratch& operator=(const Scratch&) = delete;
  ~Scratch() {
    for (void* q : blocks_) cudaFree(q);
    if (e0) cudaEventDestroy(e0);
    if (e1) cudaEventDestroy(e1);
  }
  // cudaMalloc of n elements (an empty request still gets 8 bytes)
  template <typename T>
  cudaError_t alloc(T** p, size_t n) {
    void* q = nullptr;
    const cudaError_t e = cudaMalloc(&q, n ? n * sizeof(T) : 8);
    if (e != cudaSuccess) return e;
    blocks_.push_back(q);
    *p = static_cast<T*>(q);
    return cudaSuccess;
  }
  cudaError_t create_events() {
    cudaError_t e = cudaEventCreate(&e0);
    return e != cudaSuccess ? e : cudaEventCreate(&e1);
  }
  // waits for e1 and adds the milliseconds from e0 to e1 to *ms
  cudaError_t add_ms(double* ms) {
    cudaError_t e = cudaEventSynchronize(e1);
    if (e != cudaSuccess) return e;
    float t = 0.f;
    e = cudaEventElapsedTime(&t, e0, e1);
    *ms += t;
    return e;
  }
  cudaEvent_t e0 = nullptr, e1 = nullptr;

 private:
  std::vector<void*> blocks_;
};

}  // namespace internal
}  // namespace tscm
