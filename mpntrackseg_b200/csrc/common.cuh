// Shared helpers for libmpntrack_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mpntrack_b200.h"

namespace mpn {

void set_error(const char* fmt, ...);

#define MPN_CHECK_ARG(cond, ...)            \
  do {                                      \
    if (!(cond)) {                          \
      ::mpn::set_error(__VA_ARGS__);        \
      return MPN_EINVAL;                    \
    }                                       \
  } while (0)

#define MPN_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t err__ = (call);                                                     \
    if (err__ != cudaSuccess) {                                                     \
      ::mpn::set_error("%s:%d %s: %s", __FILE__, __LINE__, #call,                   \
                       cudaGetErrorString(err__));                                  \
      return MPN_ECUDA;                                                             \
    }                                                                               \
  } while (0)

#define MPN_LAUNCH_CHECK() MPN_CUDA(cudaGetLastError())

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t align_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

int sm_count();

// Monotonic count of kernel launches issued by this library (bench.py reports the delta).
void count_launch(int n = 1);

// Optional per-kernel timing (mpn_profile_begin/end): brackets a launch with CUDA events on
// its own stream.  kind: 0 = mp_edge_kernel, 1 = mp_node_kernel.
bool profiling();
void profile_mark(int kind, bool begin, cudaStream_t s);

// Exclusive scan of n int64 values (in may alias out); out has n+1 entries, out[n]=total.
// Runs on `stream`; no host sync.
int exclusive_scan_i64(const int64_t* in, int64_t* out, int64_t n, cudaStream_t stream);
int exclusive_scan_i32(const int32_t* in, int32_t* out, int64_t n, cudaStream_t stream);

// Block-wide exclusive scan of one value per thread (blockDim.x a multiple of 32, at most 1024); *total gets the
// block total.  Every thread of the block must call it; it ends with a barrier, so smem can be reused.
template <typename T>
__device__ __forceinline__ T block_exclusive_scan(T v, T* smem /*[32]*/, T* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  T incl = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    T o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) smem[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    T w = lane < (blockDim.x >> 5) ? smem[lane] : T(0);
    T wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      T o = __shfl_up_sync(0xffffffffu, wi, d);
      if (lane >= d) wi += o;
    }
    smem[lane] = wi - w;                            // exclusive warp offsets
    if (lane == 31) *total = wi;
  }
  __syncthreads();
  T res = smem[warp] + incl - v;
  __syncthreads();
  return res;
}

// Bump allocator over a caller-provided workspace (256-byte aligned pieces).
struct Carver {
  char* base;
  int64_t off = 0;
  explicit Carver(void* p) : base(static_cast<char*>(p)) {}
  template <typename T>
  T* take(int64_t count) {
    T* p = reinterpret_cast<T*>(base + off);
    off += align_up(count * (int64_t)sizeof(T), 256);
    return p;
  }
};

}  // namespace mpn
