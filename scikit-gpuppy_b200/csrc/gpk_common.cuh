// Common definitions for the gpk (Gaussian-process kernels) library, sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cmath>

namespace gpk {

// Every dense matrix the library owns is padded to a multiple of TILE rows/cols;
// padding rows carry an identity diagonal so factor/inverse/log-det are unchanged.
constexpr int TILE = 128;

inline int round_up(int a, int b) { return (a + b - 1) / b * b; }
inline long round_up_l(long a, long b) { return (a + b - 1) / b * b; }
// Per-device slot for lazily initialised state (function attributes, constant tables, small device buffers): the
// design is one process per GPU, but a process that builds handles on several devices must not share these.
constexpr int GPK_MAX_DEVICES = 64;
inline int current_device_slot() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= GPK_MAX_DEVICES) d = 0;
  return d;
}

// last error text of the calling host thread, returned through gpk_last_error()
extern thread_local char g_err[512];

// measurement state (gpk_profile / gpk_profile_read): kernel-launch counter and, when profiling is on,
// one CUDA-event pair around every DMMA GEMM launch on its own stream.
struct ProfPair { cudaEvent_t a, b; };
extern thread_local long g_launch_count;
extern thread_local bool g_prof_on;
void prof_push(cudaEvent_t a, cudaEvent_t b);

// gpk_test_poison: while nonzero, every device buffer the library allocates is filled with this byte (test hook: a
// read of memory the library never wrote then shows in the results)
inline thread_local int g_poison = 0;
inline thread_local size_t g_poison_bytes = 0;   // bytes filled since the last gpk_test_poison call
inline cudaError_t poison_fill(void* p, size_t bytes) {
  if (!g_poison || !p || !bytes) return cudaSuccess;
  g_poison_bytes += bytes;
  const cudaError_t e = cudaMemset(p, g_poison, bytes);
  return e == cudaSuccess ? cudaDeviceSynchronize() : e;
}

#define GPK_CUDA_OK(expr)                                                         \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) {                                                      \
      snprintf(gpk::g_err, sizeof(gpk::g_err), "%s:%d: %s -> %s", __FILE__,       \
               __LINE__, #expr, cudaGetErrorString(_e));                          \
      return -1;                                                                  \
    }                                                                             \
  } while (0)

#define GPK_LAUNCH_OK()                                                           \
  do {                                                                            \
    ++gpk::g_launch_count;                                                        \
    cudaError_t _e = cudaGetLastError();                                          \
    if (_e != cudaSuccess) {                                                      \
      snprintf(gpk::g_err, sizeof(gpk::g_err), "%s:%d: launch -> %s", __FILE__,   \
               __LINE__, cudaGetErrorString(_e));                                 \
      return -1;                                                                  \
    }                                                                             \
  } while (0)

#define GPK_TRY(expr)                                                             \
  do {                                                                            \
    int _r = (expr);                                                              \
    if (_r < 0) return _r;                                                        \
  } while (0)

// Programmatic dependent launch for the latency-bound chain of the sub-2048 recursion (a leaf or a small GEMM per
// 128-block step, each depending on the one before): the next kernel's CTAs are scheduled while this one drains and
// wait at pdl_wait() for its results, so launch latency and the tail of the grid overlap. Kernels launched without
// the attribute see both calls as no-ops.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deterministic block-wide sum for blockDim.x == 256; result valid on thread 0.
__device__ __forceinline__ double block_sum_256(double v, double* red /*>=8 doubles*/) {
  v = warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) r += red[i];
  }
  return r;
}

}  // namespace gpk
