// Peer-mapped memory between the ranks of one NVSwitch box (one process per GPU) and the small device-side
// synchronisation primitives built on it.  New functionality - the reference is single-device - specified in
// SURVEY.md section 8e: the sharded 8x-TTA prediction writes its probability maps straight into rank 0's buffer from
// the fused head epilogue (NVLink stores), and data-parallel training exchanges the BatchNorm / loss sums inside the
// kernels (csrc/bn_fused.cu) instead of running one NCCL all-reduce per layer.
//   * dcb_peer_alloc / _open: cudaMalloc'ed, zero-filled buffer + its CUDA IPC handle; the other ranks open the handle
//     (the host passes the 64-byte handles around with torch.distributed, which is plumbing only);
//   * dcb_counter_advance: device-resident epoch counter (so captured CUDA graphs stay valid across calls);
//   * dcb_flag_signal: release-store of the epoch into flags that live in peers' memory;
//   * dcb_flag_wait: spin until n local flags carry the epoch (bounded: traps instead of hanging);
//   * dcb_peer_allreduce_f64: one-shot all-reduce (sum) of a small double vector: every rank stores its vector into
//     every peer's slot, publishes a flag, waits for all flags and adds the slots in rank order (bit-identical on
//     every rank).
#include "common.cuh"

namespace dcb {

__device__ __forceinline__ unsigned long long peer_ld_acquire(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void peer_st_release(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

__global__ void counter_advance_kernel(unsigned long long* c) { *c = *c + 1ULL; }

struct FlagList { unsigned long long* p[8]; int n; };

__global__ void flag_signal_kernel(const FlagList fl, const unsigned long long* epoch, long long offset) {
  __threadfence_system();
  if ((int)threadIdx.x < fl.n) peer_st_release(fl.p[threadIdx.x], (unsigned long long)((long long)*epoch + offset));
}

__global__ void flag_wait_kernel(const unsigned long long* flags, int n, const unsigned long long* epoch, long long offset, int at_least) {
  if ((int)threadIdx.x < n) {
    const unsigned long long want = (unsigned long long)((long long)*epoch + offset);
    const long long t0 = clock64();
    for (;;) {
      const unsigned long long v = peer_ld_acquire(flags + threadIdx.x);
      if (at_least ? (v >= want) : (v == want)) break;
      __nanosleep(100);
      if (clock64() - t0 > 20000000000LL) __trap();     // ~10 s: a rank died or the protocol is broken
    }
  }
  __syncthreads();
  __threadfence_system();
}

struct PeerPtrs { double* xchg[8]; unsigned long long* flags[8]; };

__global__ void __launch_bounds__(256)
peer_allreduce_f64_kernel(double* vals, int n, const PeerPtrs pp, int world, int rank, long long slot_doubles, int slot_flag,
                          const unsigned long long* epoch_ptr) {
  const unsigned long long epoch = *epoch_ptr;
  for (int p = 0; p < world; ++p) {
    double* dst = pp.xchg[p] + slot_doubles + (long long)rank * n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = vals[i];
  }
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < world) peer_st_release(pp.flags[threadIdx.x] + slot_flag * 8 + rank, epoch);
  if ((int)threadIdx.x < world) {
    const unsigned long long* f = pp.flags[rank] + slot_flag * 8 + threadIdx.x;
    const long long t0 = clock64();
    while (peer_ld_acquire(f) != epoch) {
      __nanosleep(100);
      if (clock64() - t0 > 20000000000LL) __trap();
    }
  }
  __syncthreads();
  const double* src = pp.xchg[rank] + slot_doubles;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    double acc = 0;
    for (int r = 0; r < world; ++r) acc += __ldcv(src + (long long)r * n + i);
    vals[i] = acc;
  }
}

}  // namespace dcb

using namespace dcb;

extern "C" int dcb_peer_alloc(size_t bytes, void** ptr, unsigned char* handle_out) {
  DCB_CHECK_ARG(ptr && handle_out && bytes > 0, "dcb_peer_alloc: bad arguments");
  void* p = nullptr;
  DCB_CUDA_OK(cudaMalloc(&p, bytes));
  DCB_CUDA_OK(cudaMemset(p, 0, bytes));
  DCB_CUDA_OK(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  cudaError_t e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) { cudaFree(p); return fail(DCB_ERR_CUDA, "cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e)); }
  static_assert(sizeof(h) == 64, "CUDA IPC handles are 64 bytes");
  memcpy(handle_out, &h, 64);
  *ptr = p;
  return DCB_OK;
}

extern "C" int dcb_peer_open(const unsigned char* handle, void** ptr) {
  DCB_CHECK_ARG(handle && ptr, "dcb_peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  void* p = nullptr;
  cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) return fail(DCB_ERR_CUDA, "cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
  *ptr = p;
  return DCB_OK;
}

extern "C" int dcb_peer_close(void* ptr) {
  if (ptr) DCB_CUDA_OK(cudaIpcCloseMemHandle(ptr));
  return DCB_OK;
}

extern "C" int dcb_peer_free(void* ptr) {
  if (ptr) DCB_CUDA_OK(cudaFree(ptr));
  return DCB_OK;
}

extern "C" int dcb_counter_advance(unsigned long long* counter, dcb_stream_t stream) {
  DCB_CHECK_ARG(counter, "dcb_counter_advance: null pointer");
  counter_advance_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(counter);
  g_launches += 1;
  DCB_LAUNCH_OK("counter_advance_kernel");
  return DCB_OK;
}

extern "C" int dcb_flag_signal(unsigned long long* const* flag_ptrs, int n, const unsigned long long* epoch_dev, long long offset,
                               dcb_stream_t stream) {
  DCB_CHECK_ARG(flag_ptrs && n > 0 && n <= 8 && epoch_dev, "dcb_flag_signal: bad arguments");
  FlagList fl;
  fl.n = n;
  for (int i = 0; i < 8; ++i) fl.p[i] = i < n ? flag_ptrs[i] : nullptr;
  flag_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(fl, epoch_dev, offset);
  g_launches += 1;
  DCB_LAUNCH_OK("flag_signal_kernel");
  return DCB_OK;
}

extern "C" int dcb_flag_wait(const unsigned long long* flags, int n, const unsigned long long* epoch_dev, long long offset,
                             int at_least, dcb_stream_t stream) {
  DCB_CHECK_ARG(flags && n > 0 && n <= 32 && epoch_dev, "dcb_flag_wait: bad arguments");
  flag_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, n, epoch_dev, offset, at_least);
  g_launches += 1;
  DCB_LAUNCH_OK("flag_wait_kernel");
  return DCB_OK;
}

extern "C" int dcb_peer_allreduce_f64(double* vals, int n, const dcb_peer_exchange_t* px, dcb_stream_t stream) {
  DCB_CHECK_ARG(vals && n > 0 && px && px->world >= 1 && px->world <= 8 && px->rank >= 0 && px->rank < px->world && px->epoch_dev,
                "dcb_peer_allreduce_f64: bad arguments");
  if (px->world == 1) return DCB_OK;
  DCB_CHECK_ARG((long long)px->world * n <= px->slot_doubles, "dcb_peer_allreduce_f64: %d values x %d ranks exceed the slot (%lld doubles)",
                n, px->world, px->slot_doubles);
  PeerPtrs pp;
  for (int i = 0; i < 8; ++i) {
    pp.xchg[i] = i < px->world ? reinterpret_cast<double*>(px->xchg[i]) : nullptr;
    pp.flags[i] = i < px->world ? reinterpret_cast<unsigned long long*>(px->flags[i]) : nullptr;
    if (i < px->world && (!pp.xchg[i] || !pp.flags[i])) return fail(DCB_ERR_INVALID_ARGUMENT, "dcb_peer_allreduce_f64: missing pointer for rank %d", i);
  }
  peer_allreduce_f64_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(vals, n, pp, px->world, px->rank, (long long)px->slot * px->slot_doubles,
                                                                  px->slot, px->epoch_dev);
  g_launches += 1;
  DCB_LAUNCH_OK("peer_allreduce_f64_kernel");
  return DCB_OK;
}
