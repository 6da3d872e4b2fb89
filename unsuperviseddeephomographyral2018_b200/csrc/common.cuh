// Shared helpers of libudh (error reporting, launch checks, warp/block reductions).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <stdlib.h>

#include "../../include/udh.h"

namespace udh {

void set_error(const char* fmt, ...);

// ---- in-library instrumentation (bench.py reads it): kernel-launch counter and per-phase CUDA-event timers ----
enum ProfTag {
  PROF_CONV_FWD0 = 0,    // +layer (0..7)
  PROF_CONV_DGRAD0 = 8,  // +layer
  PROF_CONV_WGRAD0 = 16, // +layer
  PROF_POOL_FWD = 24, PROF_POOL_BWD, PROF_FC_FWD, PROF_FC_BWD, PROF_DLT, PROF_WARP_FWD, PROF_WARP_BWD, PROF_SSIM,
  PROF_H4P_LOSS, PROF_ADAM, PROF_ELTWISE, PROF_TC_PREP, PROF_NUM_TAGS
};
extern unsigned long long g_launches;
extern int g_sm_reserve;      // SMs the persistent tensor-core kernels leave free (set per layer by the backward loops)
extern int g_sm_reserve_top;  // SMs the conv4_x backward kernels leave free (udh_set_sm_reserve_top): these few launches run
                              // while the fc-gradient allreduce occupies SMs; they have <= 2 items per CTA either way
// CTAs a persistent one-CTA-per-SM kernel should launch on the current device
inline int persistent_ctas() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int n = sms - g_sm_reserve;
  return n > 0 ? n : 1;
}
extern int g_bwd_marker_layer;   // udh_set_bwd_marker
// SMs the persistent backward kernels of conv layer i leave free: conv4_x's reserve (udh_set_sm_reserve_top), none elsewhere
inline int bwd_sm_reserve(int i) { return i >= 6 ? g_sm_reserve_top : 0; }
int bwd_marker_record(int layer, cudaStream_t st);   // udh_set_bwd_marker: event before layer's backward kernels
void prof_begin(int tag, cudaStream_t st);
void prof_end(int tag, cudaStream_t st);
struct ProfScope {
  int tag; cudaStream_t st;
  ProfScope(int t, cudaStream_t s) : tag(t), st(s) { prof_begin(tag, st); }
  ~ProfScope() { prof_end(tag, st); }
};

inline int check_launch(const char* what) {
  ++g_launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return UDH_ECUDA;
  }
  return UDH_OK;
}

#define UDH_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      udh::set_error(__VA_ARGS__);    \
      return UDH_EINVAL;              \
    }                                 \
  } while (0)

#define UDH_CUDA(call)                                                      \
  do {                                                                      \
    cudaError_t e__ = (call);                                               \
    if (e__ != cudaSuccess) {                                               \
      udh::set_error("%s failed: %s", #call, cudaGetErrorString(e__));      \
      return UDH_ECUDA;                                                     \
    }                                                                       \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// ---- programmatic dependent launch (PDL) for the back-to-back kernels of the bf16 step ---------------------------------
// A kernel launched through launch_chain() may be scheduled while its predecessor in the stream is still draining: its CTAs
// take over SMs as the predecessor's CTAs exit and run their prologue (barrier init, TMEM allocation, tensor-map prefetch)
// early.  Every such kernel calls pdl_wait() before its first global-memory access (it returns once the predecessor grid
// has completed and its writes are visible) and pdl_trigger() right after, so completion is transitive along the chain.
// UDH_PDL=0 in the environment falls back to plain launches (griddepcontrol.wait is then a no-op).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
inline bool pdl_enabled() {
  static int on = -1;
  if (on < 0) { const char* e = getenv("UDH_PDL"); on = (e && e[0] == '0') ? 0 : 1; }
  return on != 0;
}
template <typename... KArgs, typename... Args>
inline void launch_chain(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);     // errors surface through check_launch()
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of NV values per thread; result valid in thread 0.  `scratch` holds NV * 32 elements of T.
template <typename T, int NV>
__device__ __forceinline__ void block_sum(T (&v)[NV], T* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = warp_sum(v[i]);
  if (lane == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) scratch[i * 32 + warp] = v[i];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      T x = lane < nwarp ? scratch[i * 32 + lane] : T(0);
      v[i] = warp_sum(x);
    }
  }
}

}  // namespace udh
