// tscm_remap.cu — tscm_remap_tables(): the remap tables of TS.cpp:284-330 and rectify.cpp:86-199
// (SURVEY 8f #4) as one batched kernel, k_remap_tables (tscm_remap.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../include/tscm.h"
#include "tscm_internal.h"
#include "tscm_remap.cuh"

using namespace tscm;
using internal::set_error;

extern "C" int tscm_remap_tables(const tscm_remap_job* jobs, int32_t num_jobs, int32_t map_width,
                                 int32_t map_height, float* mapx, float* mapy, int device, double* kernel_ms) {
  internal::DeviceScope device_scope;
  if (!jobs || !mapx || !mapy || num_jobs <= 0 || map_width <= 0 || map_height <= 0) {
    set_error("bad remap arguments"); return TSCM_ERR_INVALID_ARGUMENT;
  }
  if (num_jobs > kRemapMaxJobs) {
    set_error("%d remap jobs exceed the per-call limit of %d", num_jobs, kRemapMaxJobs);
    return TSCM_ERR_INVALID_ARGUMENT;
  }
  std::vector<RemapBatch> hb(1);
  RemapBatch& B = hb[0];
  std::memset(&B, 0, sizeof(B));
  int64_t total = 0;
  for (int k = 0; k < num_jobs; ++k) {
    const tscm_remap_job& j = jobs[k];
    if (j.width <= 0 || j.height <= 0 || j.row0 < 0 || j.col0 < 0 ||
        (int64_t)j.row0 + j.height > map_height || (int64_t)j.col0 + j.width > map_width) {
      set_error("remap job %d: block %dx%d at (%d,%d) does not fit the %dx%d maps", k, j.width, j.height,
                j.col0, j.row0, map_width, map_height);
      return TSCM_ERR_INVALID_ARGUMENT;
    }
    if (j.ray_fx == 0.0 || j.ray_fy == 0.0) { set_error("remap job %d: zero ray focal length", k); return TSCM_ERR_INVALID_ARGUMENT; }
    RemapJobDev& d = B.job[k];
    std::memcpy(d.intr, j.intrinsics, sizeof(d.intr));
    std::memcpy(d.M, j.matrix, sizeof(d.M));
    d.ray_fx = j.ray_fx; d.ray_fy = j.ray_fy; d.ray_cx = j.ray_cx; d.ray_cy = j.ray_cy;
    d.offset_x = j.offset_x; d.offset_y = j.offset_y; d.cutoff_w2 = j.cutoff_w2;
    d.width = j.width; d.height = j.height; d.row0 = j.row0; d.col0 = j.col0;
    d.first_pixel = total;
    total += (int64_t)j.width * j.height;
  }
  B.num_jobs = num_jobs; B.map_width = map_width; B.total_pixels = total;
  internal::SelectedDevice dev;
  RC_TRY(internal::select_device(device, "remap tables", &dev));
  internal::Scratch scratch;
  RemapBatch* d_batch = nullptr;
  float *d_x = nullptr, *d_y = nullptr;
  const size_t map_pixels = (size_t)map_width * map_height;
  CUDA_TRY(scratch.alloc(&d_batch, 1));
  CUDA_TRY(scratch.alloc(&d_x, map_pixels));
  CUDA_TRY(scratch.alloc(&d_y, map_pixels));
  CUDA_TRY(cudaMemcpy(d_batch, &B, sizeof(RemapBatch), cudaMemcpyHostToDevice));
  CUDA_TRY(scratch.create_events());
  // one wave of resident CTAs (8 x 256 threads per SM), grid-stride over the pixels
  const int64_t want = (total + 255) / 256;
  const int grid = (int)std::min<int64_t>(want, (int64_t)dev.sm_count * 8);
  CUDA_TRY(cudaEventRecord(scratch.e0, 0));
  k_remap_tables<<<grid, 256>>>(d_batch, d_x, d_y);
  CUDA_TRY(cudaEventRecord(scratch.e1, 0));
  CUDA_TRY(cudaGetLastError());
  for (int k = 0; k < num_jobs; ++k) {   // only the blocks that were written
    const tscm_remap_job& j = jobs[k];
    const size_t o = (size_t)j.row0 * map_width + j.col0, pitch = (size_t)map_width * sizeof(float);
    CUDA_TRY(cudaMemcpy2D(mapx + o, pitch, d_x + o, pitch, (size_t)j.width * sizeof(float), j.height, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy2D(mapy + o, pitch, d_y + o, pitch, (size_t)j.width * sizeof(float), j.height, cudaMemcpyDeviceToHost));
  }
  double ms = 0.0;
  CUDA_TRY(scratch.add_ms(&ms));
  if (kernel_ms) *kernel_ms = ms;
  return TSCM_OK;
}
