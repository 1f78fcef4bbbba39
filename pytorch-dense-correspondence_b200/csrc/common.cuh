// Shared helpers for libddn_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>

#include "../../include/ddn_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libddn_b200 is written for sm_100a (B200) only"
#endif

namespace ddn {

extern std::atomic<long long> g_launches;
void set_error(const char* fmt, ...);

#define DDN_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      ::ddn::set_error(__VA_ARGS__);             \
      return DDN_EINVAL;                         \
    }                                            \
  } while (0)

#define DDN_CUDA(call)                                                                  \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      ::ddn::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
      return (int)e__;                                                                  \
    }                                                                                   \
  } while (0)

#define DDN_TRY(call)          \
  do {                         \
    int r__ = (call);          \
    if (r__ != 0) return r__;  \
  } while (0)

// Programmatic dependent launch.  Every kernel of this library is launched with the programmatic-stream-serialization
// attribute and starts with pdl_prologue(): `launch_dependents` lets the NEXT kernel's CTAs become resident as soon as an
// SM has room for them (they park in `griddepcontrol.wait`, issuing nothing), and `wait` returns once the PREVIOUS kernel
// has completed and its memory is visible.  A step is ~230 dependent launches; this removes the drain + launch gap between
// them (and, in the persistent tcgen05 kernels, overlaps barrier init / TMEM allocation with the predecessor's tail).
// Rule: nothing written by an earlier kernel may be read before pdl_wait(), and EVERY thread of every kernel executes it
// (a kernel that skipped it could finish before its predecessor and break the chain for its successor).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() { pdl_trigger(); pdl_wait(); }

// cluster_x > 1 groups the grid's CTAs along x into clusters of that size (the CTA pairs of the tcgen05 cta_group::2 kernels).
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, unsigned cluster_x, dim3 block, size_t smem, cudaStream_t st,
                                        Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
    ++n;
  }
  attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
  cfg.attrs = attr; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

// Every kernel launch goes through one of these so gpu_launches is an honest count.
#define DDN_LAUNCH_CLUSTER(kernel, grid, cluster_x, block, smem, stream, ...)                                        \
  do {                                                                                                               \
    DDN_CUDA(::ddn::launch_kernel(kernel, dim3(grid), (unsigned)(cluster_x), dim3(block), (smem), (stream), __VA_ARGS__)); \
    ::ddn::g_launches.fetch_add(1, std::memory_order_relaxed);                                                       \
  } while (0)
#define DDN_LAUNCH(kernel, grid, block, smem, stream, ...) DDN_LAUNCH_CLUSTER(kernel, grid, 1, block, smem, stream, __VA_ARGS__)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

int num_sms();

// Optional per-kernel-class timing with CUDA events on the launching stream (off by default; bench.py turns it on).
enum ProfClass { PROF_CONV_FWD_SIMT = 0, PROF_CONV_DGRAD_SIMT, PROF_CONV_WGRAD_SIMT, PROF_CONV_FWD_TC, PROF_CONV_DGRAD_TC,
                 PROF_CONV_WGRAD_TC, PROF_LOSS_FWD, PROF_LOSS_BWD, PROF_NUM_CLASSES };
struct ProfScope {
  ProfScope(int cls, double work, cudaStream_t st);
  ~ProfScope();
  int slot; cudaStream_t st;
};

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
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

}  // namespace ddn
