// Device helpers shared by the KNN kernels (graph_build.cu, knn_graph.cu, knn_graph_tc.cu): the float order key, the
// window of a batch-global row, the time-valid test and the block-level select of a row's k-th smallest (key, index).
#pragma once
#include <stdint.h>

namespace mpn {

constexpr unsigned kFullMask = 0xffffffffu;

// Monotone map float -> uint32 (ascending); a positive NaN sorts last, like torch.sort.
__device__ __forceinline__ uint32_t order_key(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float key_value(uint32_t key) {
  return __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
}

// Window g of batch-global row i: gptr[g] <= i < gptr[g + 1].
__device__ __forceinline__ int64_t window_of(const int64_t* __restrict__ gptr, int64_t num_graphs, int64_t i) {
  int64_t lo = 0, hi = num_graphs;
  while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if (gptr[mid] <= i) lo = mid; else hi = mid; }
  return lo;
}

// Two detections may be joined: different frames, at most max_dist apart (max_dist < 0: any distance).
__device__ __forceinline__ bool frames_connect(int64_t fi, int64_t fj, int64_t max_dist) {
  const int64_t d = fi > fj ? fi - fj : fj - fi;
  return d > 0 && (max_dist < 0 || d <= max_dist);
}

// ------------------------------------------------------------------ block-level k-th (key, index) select
// A row of n floats is ranked by (order_key, index).  Thread t of the SEL_THREADS-thread block owns the entries
// j = q * SEL_THREADS + t; RowKeys<PER> hands out their keys chunk by chunk.
constexpr int SEL_THREADS = 256;

// PER > 0: the keys are read once into registers (n <= PER * SEL_THREADS).
template <int PER>
struct RowKeys {
  uint32_t key[PER];
  __device__ __forceinline__ RowKeys(const float* __restrict__ rowp, int64_t n) {
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      const int64_t j = threadIdx.x + q * SEL_THREADS;
      key[q] = j < n ? order_key(rowp[j]) : 0xffffffffu;
    }
  }
  __device__ __forceinline__ int chunks(int64_t) const { return PER; }
  __device__ __forceinline__ uint32_t operator[](int q) const { return key[q]; }
};

// PER == 0 (streamed): the keys are re-read from the row on every pass, for any n.
template <>
struct RowKeys<0> {
  const float* __restrict__ rowp;
  int64_t n;
  __device__ __forceinline__ RowKeys(const float* __restrict__ r, int64_t len) : rowp(r), n(len) {}
  __device__ __forceinline__ int chunks(int64_t len) const { return (int)((len + SEL_THREADS - 1) / SEL_THREADS); }
  __device__ __forceinline__ uint32_t operator[](int q) const {
    const int64_t j = threadIdx.x + (int64_t)q * SEL_THREADS;
    return j < n ? order_key(rowp[j]) : 0xffffffffu;
  }
};

struct SelectSmem {
  int hist[256];
  uint32_t prefix;
  int remaining, count;
  int32_t found;
};

// Entry j of the row is among its k smallest (ties by ascending index) iff
//   key_j < tau || (key_j == tau && j <= found);
// k >= n: tau = 0xffffffff, found = n (every entry is in).  Called by the whole block; tau and found come back
// block-uniform.  Radix select over the 4 key bytes; the tie walk at the end re-reads the row.
template <int PER>
__device__ __forceinline__ void select_kth(const RowKeys<PER>& keys, const float* __restrict__ rowp, int64_t n, int64_t k,
                                           SelectSmem& sm, uint32_t& tau, int32_t& found) {
  tau = 0xffffffffu;
  found = (int32_t)n;
  if (k >= n) return;
  const int tid = threadIdx.x, lane = tid & 31;
  const int nq = keys.chunks(n);
  if (tid == 0) { sm.prefix = 0u; sm.remaining = (int)k; sm.found = -1; }
  uint32_t mask = 0u;
  for (int shift = 24; shift >= 0; shift -= 8) {
    sm.hist[tid] = 0;
    __syncthreads();
    const uint32_t prefix = sm.prefix;
#pragma unroll
    for (int q = 0; q < nq; ++q) {
      const uint32_t key = keys[q];
      if (tid + (int64_t)q * SEL_THREADS < n && (key & mask) == prefix) atomicAdd(&sm.hist[(key >> shift) & 255u], 1);
    }
    __syncthreads();
    if (tid < 32) {
      // bin holding the `remaining`-th element: lane l owns bins 8l..8l+7, warp scan over the lane totals
      int h[8], tot = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { h[q] = sm.hist[8 * lane + q]; tot += h[q]; }
      int incl = tot;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(kFullMask, incl, d); if (lane >= d) incl += v; }
      const int rem0 = sm.remaining;
      if (incl >= rem0 && incl - tot < rem0) {                              // exactly one lane
        int rem = rem0 - (incl - tot), b = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) { if (h[q] >= rem) { b = q; break; } rem -= h[q]; }
        sm.remaining = rem;
        sm.prefix = prefix | ((uint32_t)(8 * lane + b) << shift);
        sm.count = h[b];
      }
    }
    mask |= 255u << shift;
    __syncthreads();
  }
  tau = sm.prefix;
  const int need = sm.remaining;
  if (sm.count == need) {                                                   // no tie straddles the boundary: last equal element
    int32_t mine = -1;
#pragma unroll
    for (int q = 0; q < nq; ++q) {
      const int64_t j = tid + (int64_t)q * SEL_THREADS;
      if (j < n && keys[q] == tau) mine = (int32_t)j;
    }
    if (mine >= 0) atomicMax(&sm.found, mine);
  } else if (tid < 32) {                                                    // first `need` equal elements in index order
    int seen = 0;
    int32_t f = (int32_t)(n - 1);
    for (int64_t j0 = 0; j0 < n; j0 += 32) {
      const int64_t j = j0 + lane;
      const bool eq = j < n && order_key(rowp[j]) == tau;
      const unsigned m = __ballot_sync(kFullMask, eq);
      const int c = __popc(m);
      if (seen + c >= need) {
        unsigned mm = m;
        for (int q = 1; q < need - seen; ++q) mm &= mm - 1;
        f = (int32_t)(j0 + __ffs(mm) - 1);
        break;
      }
      seen += c;
    }
    if (lane == 0) sm.found = f;
  }
  __syncthreads();
  found = sm.found;
}

}  // namespace mpn
