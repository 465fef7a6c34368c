// Host-side helpers shared by all translation units of libvitk: error reporting (thread-local
// message behind vitk_last_error), launch checks, device properties.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/vitk.h"

namespace vitk {

int set_error(int code, const char* fmt, ...);   // stores the message, returns code
int cuda_error(cudaError_t e, const char* what); // returns (int)e after storing the message
int num_sms();                                   // SM count of the current device (cached)
void count_launch();                             // bumps the process-wide kernel launch counter

#define VITK_REQUIRE(cond, code, ...)                         \
  do {                                                        \
    if (!(cond)) return ::vitk::set_error((code), __VA_ARGS__); \
  } while (0)

#define VITK_CUDA(expr)                                             \
  do {                                                              \
    cudaError_t _e = (expr);                                        \
    if (_e != cudaSuccess) return ::vitk::cuda_error(_e, #expr);    \
  } while (0)

#define VITK_LAUNCH_CHECK(name)                                     \
  do {                                                              \
    ::vitk::count_launch();                                         \
    cudaError_t _e = cudaGetLastError();                            \
    if (_e != cudaSuccess) return ::vitk::cuda_error(_e, name);     \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ----------------------------------------------------------------------------- programmatic dependent launch
// Every hot kernel is launched with programmatic stream serialization: its CTAs may become resident (and
// run their prologue: barrier init, TMEM allocation, descriptor prefetch) while the previous kernel in the
// stream is still draining its last wave, and they block in pdl_wait() before touching global memory until
// that kernel has completed and flushed.  ~300 dependent launches per step, each with a 3–4 µs
// launch + prologue + tail bubble otherwise.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace vitk
