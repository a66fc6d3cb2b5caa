// Shared helpers for the dcb200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <cstring>
#include <map>
#include <mutex>

#include "../../include/dcb200.h"

namespace dcb {

// thread-local last-error text returned by dcb_last_error()
char* last_error_buf();
int fail(int code, const char* fmt, ...);

#define DCB_CHECK_ARG(cond, ...)                                   \
  do { if (!(cond)) return ::dcb::fail(DCB_ERR_INVALID_ARGUMENT, __VA_ARGS__); } while (0)

#define DCB_CUDA_OK(expr)                                                              \
  do { cudaError_t _e = (expr);                                                        \
       if (_e != cudaSuccess)                                                          \
         return ::dcb::fail(DCB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,              \
                            cudaGetErrorString(_e), __FILE__, __LINE__); } while (0)

// Launch check that does not synchronise (graph-capturable).
#define DCB_LAUNCH_OK(name)                                                            \
  do { cudaError_t _e = cudaPeekAtLastError();                                         \
       if (_e != cudaSuccess)                                                          \
         return ::dcb::fail(DCB_ERR_CUDA, "launch of %s failed: %s", name,             \
                            cudaGetErrorString(_e)); } while (0)

static inline int cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

int sm_count();   // cached multiprocessor count of the current device
int policy(int key);               // current value of a dcb_policy_key (dcb_set_policy)
void note_kernel(const char* name); // records the contraction kernel a call dispatched to (dcb_last_kernel)

extern unsigned long long g_launches;   // kernels launched by the library (dcb_launch_count)

// Sets a kernel's function attributes once, before its first launch that needs them: the maximum dynamic shared memory
// (smem_max > 0: above the default 48 KB) and, for clusters of more than the portable 8 CTAs, the non-portable size.
inline cudaError_t prepare_kernel(const void* kernel, int smem_max, int cluster) {
  static std::mutex mu;
  static std::map<const void*, int> applied;     // per kernel: 1 = shared-memory limit set, 2 = non-portable clusters allowed
  const int want = (smem_max > 0 ? 1 : 0) | (cluster > 8 ? 2 : 0);
  std::lock_guard<std::mutex> lock(mu);
  int& have = applied[kernel];
  cudaError_t e = cudaSuccess;
  if (want & ~have & 1) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max);
  if (e == cudaSuccess && (want & ~have & 2)) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
  if (e == cudaSuccess) have |= want;
  return e;
}

// Kernel launch with optional PROGRAMMATIC DEPENDENT LAUNCH (policy DCB_POLICY_PDL): the kernel may be scheduled while
// its predecessor in the stream is still running, executes its prologue (barrier / TMEM set-up, tensor-map prefetch,
// loads of STATIC data such as weights) and blocks in pdl_wait() until the predecessor has completed and its writes
// are visible.  Only kernels that call pdl_wait() before touching anything an earlier kernel of the stream produces
// may be launched with pdl = true.  Captured into CUDA graphs as programmatic dependency edges.
// cluster > 0: the kernel runs as thread-block clusters of `cluster` CTAs (grid must be a multiple of it).
// Counts the launch in g_launches; a failure is reported through fail(DCB_ERR_CUDA) with the kernel's name.
template <typename... ExpTypes, typename... ActTypes>
static inline int launch(void (*kernel)(ExpTypes...), const char* name, int grid, int block, size_t smem, int smem_max,
                         cudaStream_t st, bool pdl, int cluster, ActTypes&&... args) {
  cudaError_t e = prepare_kernel(reinterpret_cast<const void*>(kernel), smem_max, cluster);
  if (e == cudaSuccess) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid, 1, 1); cfg.blockDim = dim3((unsigned)block, 1, 1);
    cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    unsigned n = 0;
    if (cluster > 0) {
      at[n].id = cudaLaunchAttributeClusterDimension;
      at[n].val.clusterDim.x = (unsigned)cluster; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
      ++n;
    }
    if (pdl) {
      at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      at[n].val.programmaticStreamSerializationAllowed = 1;
      ++n;
    }
    cfg.attrs = at; cfg.numAttrs = n;
    e = cudaLaunchKernelEx(&cfg, kernel, static_cast<ExpTypes>(args)...);
  }
  if (e != cudaSuccess) return fail(DCB_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e));
  g_launches += 1;
  return DCB_OK;
}

// ---- device helpers ----
// programmatic dependent launch (see launch): let the next kernel of the stream start its prologue / wait for the
// previous kernel's completion.  Both are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

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

}  // namespace dcb
