// Shared host-side helpers for the C-ABI library: error reporting and launch checks.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include "../../include/gecco_b200.h"

namespace gecco {

// Thread-local text for gecco_last_error(); every failing export sets it.
void set_error(const char* fmt, ...);

inline int fail_cuda(cudaError_t e, const char* what) {
  set_error("%s: %s", what, cudaGetErrorString(e));
  return GECCO_ERR_CUDA;
}

// Counts kernel launches issued through the library on this thread (gecco_launch_count).
extern thread_local long long g_launches;

#define GECCO_CHECK_LAUNCH(what)                              \
  do {                                                        \
    cudaError_t e__ = cudaGetLastError();                     \
    if (e__ != cudaSuccess) return gecco::fail_cuda(e__, what); \
    ++gecco::g_launches;                                      \
  } while (0)

#define GECCO_REQUIRE(cond, ...)        \
  do {                                  \
    if (!(cond)) {                      \
      gecco::set_error(__VA_ARGS__);    \
      return GECCO_ERR_INVALID;         \
    }                                   \
  } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Launch helper of the small kernels (folds, AdaGN apply, lookup, head, ...): a plain launch, without programmatic
// dependent launch.  Measured A/B on one B200, launching them with the attribute LOSES 2 % of the sampler step (595-599
// against 585-586 ms): the dependents that become resident early are the persistent one-CTA-per-SM GEMMs, which then sit
// on the SMs' shared memory while the small kernel is still running.  The tcgen05 kernels keep their own PDL launches,
// and the small kernels keep griddepcontrol.wait / launch_dependents (pdl_wait(), ptx.cuh): a tcgen05 kernel that
// follows one relies on the trigger, and without the attribute the wait is a no-op.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_small(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

int sm_count();

}  // namespace gecco
