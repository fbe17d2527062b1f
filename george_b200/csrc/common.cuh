// common.cuh — shared plumbing of libbgp_b200: status/error handling, launch accounting, stream-ordered
// device memory, and small device-side helpers (warp/block reductions, cluster barriers, 1-D TMA bulk loads).
#pragma once

#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <atomic>
#include <string>

#include "../../include/bgp.h"

namespace bgp {

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
struct Status {
  int code;
};

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define BGP_CUDA(expr)                                                                            \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      ::bgp::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return (_e == cudaErrorMemoryAllocation) ? BGP_ERR_NOMEM : BGP_ERR_CUDA;                    \
    }                                                                                             \
  } while (0)

#define BGP_TRY(expr)            \
  do {                           \
    int _s = (expr);             \
    if (_s != BGP_OK) return _s; \
  } while (0)

// every kernel launch of the library goes through this so bench.py can report "gpu_launches"
#define BGP_LAUNCH_CHECK()                                                                       \
  do {                                                                                           \
    ::bgp::g_launches.fetch_add(1, std::memory_order_relaxed);                                   \
    cudaError_t _e = cudaGetLastError();                                                         \
    if (_e != cudaSuccess) {                                                                     \
      ::bgp::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, __LINE__); \
      return BGP_ERR_CUDA;                                                                       \
    }                                                                                            \
  } while (0)

int require_device();  // BGP_ERR_NO_DEVICE unless an sm_100 GPU is current
int num_sms();

// stream-ordered allocation from the device's default pool with an unlimited release threshold: after the
// first compute() of a given size, re-allocation is a free-list hit (no cudaMalloc on the hot path).
int dev_alloc(void** p, size_t bytes, cudaStream_t s);
void dev_free(void* p, cudaStream_t s);

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  cudaStream_t s = 0;
  int alloc(size_t count, cudaStream_t stream) {
    release();
    s = stream;
    n = count;
    if (count == 0) return BGP_OK;
    return dev_alloc((void**)&p, count * sizeof(T), stream);
  }
  // grow-only: keep the old block when it is large enough
  int reserve(size_t count, cudaStream_t stream) {
    if (count <= n && p) { s = stream; return BGP_OK; }
    return alloc(count, stream);
  }
  void release() {
    if (p) dev_free(p, s);
    p = nullptr;
    n = 0;
  }
  ~DevBuf() { release(); }
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
};

// Owned stream / event, created on first use.  The destructor synchronises, then destroys.  A DevBuf is freed on its
// stream, so an owner declares its Streams before its DevBufs (members are destroyed in reverse order).
struct Stream {
  cudaStream_t s = nullptr;
  int create() {
    if (!s) BGP_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    return BGP_OK;
  }
  void sync() const { if (s) cudaStreamSynchronize(s); }
  operator cudaStream_t() const { return s; }
  ~Stream() { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } }
  Stream() {}
  Stream(const Stream&) = delete;
  Stream& operator=(const Stream&) = delete;
};

struct Event {
  cudaEvent_t e = nullptr;
  int create() {
    if (!e) BGP_CUDA(cudaEventCreate(&e));
    return BGP_OK;
  }
  operator cudaEvent_t() const { return e; }
  ~Event() { if (e) { cudaEventSynchronize(e); cudaEventDestroy(e); } }
  Event() {}
  Event(Event&& o) noexcept : e(o.e) { o.e = nullptr; }  // (kept in a growing std::vector)
  Event(const Event&) = delete;
  Event& operator=(const Event&) = delete;
};

// ---------------------------------------------------------------------------------------------------------------
// device side
// ---------------------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// (|value| max, lowest index on ties): the order Eigen's maxCoeff(&idx) visits a vector (hodlr.h:189)
__device__ __forceinline__ void argmax_combine(double& v, int& i, double ov, int oi) {
  if (ov > v || (ov == v && oi < i)) { v = ov; i = oi; }
}
__device__ __forceinline__ void warp_argmax(double& v, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    double ov = __shfl_xor_sync(0xffffffffu, v, o);
    int oi = __shfl_xor_sync(0xffffffffu, i, o);
    argmax_combine(v, i, ov, oi);
  }
}

// block-wide sum; `scratch` holds >= 32 doubles of shared memory; result valid in every thread
__device__ __forceinline__ double block_sum(double v, double* scratch) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) scratch[w] = v;
  __syncthreads();
  double t = (lane < nw) ? scratch[lane] : 0.0;
  t = warp_sum(t);
  return t;
}

// ---- mbarrier + 1-D bulk async copy (TMA engine without a tensor map; SASS: UBLKCP) -------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(phase)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// cooperative tile load of `count` doubles; TMA bulk when 16-byte aligned & sized, plain loads otherwise.
// `bar` is a CTA-shared mbarrier already initialised with count 1; `*phase` flips on every TMA use.
__device__ __forceinline__ void load_coords(double* dst, const double* __restrict__ src, int count, uint64_t* bar,
                                            uint32_t& phase) {
  const uint32_t bytes = (uint32_t)count * 8u;
  const bool bulk = ((bytes & 15u) == 0) && ((reinterpret_cast<uintptr_t>(src) & 15u) == 0) && bytes > 0;
  if (bulk) {
    if (threadIdx.x == 0) {
      mbar_expect_tx(bar, bytes);
      tma_load_1d(dst, src, bytes, bar);
    }
    mbar_wait(bar, phase);
    phase ^= 1u;
  } else {
    for (int i = threadIdx.x; i < count; i += blockDim.x) dst[i] = src[i];
    __syncthreads();
  }
}

#endif  // __CUDACC__

}  // namespace bgp
