// One specialised instance of the fused post-physics kernel.
//
// Compiled by genesis_forge_b200/spec.py with -DGFB_SPEC_HEADER="<generated header>".  The header
// defines, as compile-time constants, the STRUCTURE of one term table and its slab plan:
//     namespace gfb_spec { TILE, PHASES, kP (gfb_program_head, live values zeroed), kPlan (gfb::Plan) }
// post_kernel.cuh then reads structure from those constants (term loops unroll, switches fold,
// shared-memory offsets become immediates) and live values from the kernel parameters as usual.
// A table with lowered user-defined observation terms (GFB_SPEC_USER_OBS) also exports
// gfb_spec_user_observe, their reset path for gfb_observe.  gfb_spec_state_slots is the mask of the
// GFB_B_USER_STATE slots the lowered class-style terms read and write (GFB_SPEC_STATE_SLOTS, 0 without).
#include <cuda_runtime.h>

#include "../../include/gfb200.h"
#include "plan.h"

#include GFB_SPEC_HEADER

#define GFB_SPEC 1
#include "post_kernel.cuh"

namespace {
// host copies of the structure for the library's match test
const gfb_program_head h_canon = gfb_spec::kP_host;
const gfb::Plan h_plan = gfb_spec::kPlan_host;
int smem_attr = 0;
}  // namespace

extern "C" int gfb_spec_info(int* tile, unsigned* phases, const void** canon, const void** plan, int* head_bytes,
                             int* plan_bytes) {
  *tile = gfb_spec::TILE;
  *phases = gfb_spec::PHASES;
  *canon = &h_canon;
  *plan = &h_plan;
  *head_bytes = (int)sizeof(gfb_program_head);
  *plan_bytes = (int)sizeof(gfb::Plan);
  return 0;
}

#ifndef GFB_SPEC_STATE_SLOTS
#define GFB_SPEC_STATE_SLOTS 0u
#endif
extern "C" unsigned gfb_spec_state_slots(void) { return GFB_SPEC_STATE_SLOTS; }

extern "C" int gfb_spec_blocks_per_sm(unsigned smem) {
  if ((int)smem > 44 * 1024 && (int)smem > smem_attr) {
    if (cudaFuncSetAttribute(gfb::post_kernel<gfb_spec::TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess)
      return 0;
    smem_attr = (int)smem;
  }
  int n = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, gfb::post_kernel<gfb_spec::TILE>, gfb_spec::TILE, smem) != cudaSuccess)
    n = 0;
  return n;
}

#ifdef GFB_SPEC_USER_OBS
namespace {
// Reset path of the lowered user-defined observation terms: for the listed envs (all when idx is null),
// from global memory only -- post-reset engine state, this step's contact outputs and counters, and the
// cached (pre-reset) inverse base quaternion for body-frame vectors, as observe_kernel -- into the
// (N, GFB_SPEC_USER_OBS) rows of GFB_B_OBS_EXT1 that the observe-only plan's GFB_O_USER columns read.
__global__ void __launch_bounds__(128) user_observe_kernel(const __grid_constant__ gfb_buffers b, int num_envs,
                                                           const int64_t* idx, int n, int has_max_len) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t e = idx ? (size_t)idx[i] : (size_t)i;
  const float4 q = reinterpret_cast<const float4*>(b.buf[GFB_B_INV_BASE_QUAT])[e];
  const int ep_len = reinterpret_cast<const int32_t*>(b.buf[GFB_B_EPISODE_LENGTH])[e];
  const int max_len = has_max_len ? reinterpret_cast<const int32_t*>(b.buf[GFB_B_MAX_EPISODE_LENGTH])[e] : 0;
  const gfb::V3 zero = {0.f, 0.f, 0.f};
  gfb::user_observations_global(
      gfb::UserCtx{b, e, ep_len, max_len, false, false, q.x, gfb::V3{q.y, q.z, q.w}, zero, zero, zero, nullptr, 0,
                   nullptr, gfb_spec::kPlan, nullptr, num_envs, true},
      reinterpret_cast<float*>(b.buf[GFB_B_OBS_EXT1]) + e * GFB_SPEC_USER_OBS);
}
}  // namespace

extern "C" int gfb_spec_user_observe(const gfb_buffers* b, int num_envs, const int64_t* idx, int n, int has_max_len,
                                     void* stream) {
  if (n <= 0) return 0;
  user_observe_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(*b, num_envs, idx, n,
                                                                                     has_max_len);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
#endif

extern "C" int gfb_spec_launch(const gfb::KParams* kp, int grid, unsigned smem, void* stream) {
  if ((int)smem > 44 * 1024 && (int)smem > smem_attr) {
    if (cudaFuncSetAttribute(gfb::post_kernel<gfb_spec::TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess)
      return 1;
    smem_attr = (int)smem;
  }
  gfb::post_kernel<gfb_spec::TILE><<<grid, gfb_spec::TILE, smem, static_cast<cudaStream_t>(stream)>>>(*kp);
  return cudaGetLastError() == cudaSuccess ? 0 : 1;
}
