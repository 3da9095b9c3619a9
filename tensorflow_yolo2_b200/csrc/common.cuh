// common.cuh -- error plumbing and small device helpers shared by all translation units.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <stdlib.h>

#include "../../include/yolo2_b200.h"

namespace y2 {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

// Switches (environment variables Y2_*) that select a reference path for tests and tools, or take PDL out of the
// picture.  Read ONCE per process (a launch used to pay ~10 getenv() calls); y2_reload_env() re-reads them (tests that
// flip a switch inside one process).
struct EnvSwitches {
  bool bn_bwd_generic, affine_generic, no_pdl, conv_no_streamk, conv_force_streamk, conv_force_tiled, conv_no_cta2,
      conv_no_is, conv_force_is, conv_no_tma_store_f32;
};
const EnvSwitches& env();

#define Y2_ARG(cond)                                                              \
  do {                                                                            \
    if (!(cond)) {                                                                \
      y2::set_error("%s: bad argument: %s", __func__, #cond);                     \
      return Y2_ERR_BAD_ARG;                                                      \
    }                                                                             \
  } while (0)

#define Y2_CUDA(expr)                                                             \
  do {                                                                            \
    cudaError_t e__ = (expr);                                                     \
    if (e__ != cudaSuccess) {                                                     \
      y2::set_error("%s: %s -> %s", __func__, #expr, cudaGetErrorString(e__));    \
      (void)cudaGetLastError(); /* non-sticky errors must not leak into the caller's next CUDA call */ \
      return (int)e__;                                                            \
    }                                                                             \
  } while (0)

// after a <<<>>> launch: count it and surface launch-configuration errors
#define Y2_LAUNCHED()                                                             \
  do {                                                                            \
    y2::count_launch();                                                           \
    Y2_CUDA(cudaPeekAtLastError());                                               \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t a, size_t b) { return (a + b - 1) / b * b; }

__device__ __forceinline__ float leaky(float v, float alpha) { return fmaxf(v, alpha * v); }

// Programmatic dependent launch (PDL).  A persistent kernel calls pdl_launch_dependents() on entry -- the NEXT kernel of
// the stream may then be scheduled onto SMs as this kernel's CTAs retire, instead of after the whole grid has drained plus
// a launch latency -- and a kernel launched with the attribute calls pdl_wait() before its first access to global memory
// (it returns once the preceding kernel has completed and its writes are visible).  Only the prologue (barrier init, TMEM
// allocation, descriptor prefetch) runs ahead.  Both are no-ops when the launch carries no programmatic dependency.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// launch attribute list: cluster dimension (always) + programmatic stream serialization (unless Y2_NO_PDL is set)
static inline int fill_launch_attrs(cudaLaunchAttribute* attr, unsigned cluster) {
  int n = 0;
  attr[n].id = cudaLaunchAttributeClusterDimension;
  attr[n].val.clusterDim.x = cluster;
  attr[n].val.clusterDim.y = 1;
  attr[n].val.clusterDim.z = 1;
  ++n;
  if (!env().no_pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  return n;
}

}  // namespace y2
