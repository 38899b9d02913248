// Fused, batched construction of KNN-pruned window graphs (training-mode semantics of
// MOTGraph._get_edge_ixs, data/mot_graph.py:195-221): for G independent windows at once
//   1. dense ReID distance blocks  D_g[i][j] = || reid_i - reid_j + 1e-6 ||_2  (i < j, mirrored;
//      pairs of the same frame or farther apart than max_frame_dist = +inf),
//   2. per-row k-th smallest (distance, index) threshold                         (utils/graph.py:65-70),
//   3. keep (i<j) iff in_k(i,j) AND/OR in_k(j,i); pairs are emitted sorted by (i, j) (utils/graph.py:73-85),
// with a single host synchronisation (the pair count).  Node ids are batch-global.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "knn_select.cuh"

namespace mpn {

constexpr int DT = 64;        // distance tile (rows x cols per CTA)
constexpr int DK = 32;        // feature slab

// blockIdx.y = window, blockIdx.x = upper-triangular tile id inside the window.
__global__ void __launch_bounds__(256) dist_blocks_kernel(const float* __restrict__ reid, int64_t dim,
                                                          const int64_t* __restrict__ frame,
                                                          const int64_t* __restrict__ gptr,
                                                          const int64_t* __restrict__ doff, int64_t max_dist,
                                                          float* __restrict__ dense) {
  const int g = blockIdx.y;
  const int64_t n0 = gptr[g], n = gptr[g + 1] - n0;
  const int nt = (int)((n + DT - 1) / DT);
  // tile id -> (ti <= tj) over the upper triangle, row-major
  int t = blockIdx.x;
  if (t >= nt * (nt + 1) / 2) return;
  int ti = 0;
  while (t >= nt - ti) { t -= nt - ti; ++ti; }
  const int tj = ti + t;
  float* D = dense + doff[g];
  __shared__ float sa[DK][DT + 1];
  __shared__ float sb[DK][DT + 1];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // 16 x 16 threads, 4 x 4 outputs each
  float acc[4][4] = {};
  const float eps = 1e-6f;
  for (int64_t k0 = 0; k0 < dim; k0 += DK) {
    for (int idx = threadIdx.x; idx < DT * DK; idx += 256) {
      const int r = idx / DK, kk = idx % DK;
      const int64_t ia = (int64_t)ti * DT + r, ib = (int64_t)tj * DT + r, k = k0 + kk;
      sa[kk][r] = (ia < n && k < dim) ? reid[(n0 + ia) * dim + k] : 0.f;
      sb[kk][r] = (ib < n && k < dim) ? reid[(n0 + ib) * dim + k] : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < DK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[q] = sa[kk][ty * 4 + q]; b[q] = sb[kk][tx * 4 + q]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float d = (a[i] - b[j]) + eps;                      // F.pairwise_distance: x1 - x2 + eps
          acc[i][j] = fmaf(d, d, acc[i][j]);
        }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t li = (int64_t)ti * DT + ty * 4 + i;
    if (li >= n) continue;
    const int64_t fi = frame[n0 + li];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t lj = (int64_t)tj * DT + tx * 4 + j;
      if (lj >= n || lj <= li) continue;                            // strictly upper triangle; mirrored below
      const float v = frames_connect(fi, frame[n0 + lj], max_dist) ? sqrtf(acc[i][j]) : INFINITY;
      D[li * n + lj] = v;
      D[lj * n + li] = v;                                           // utils/graph.py:58-60 (symmetric fill)
    }
  }
  // diagonal entries (no self edges)
  if (ti == tj && threadIdx.x < DT) {
    const int64_t li = (int64_t)ti * DT + threadIdx.x;
    if (li < n) D[li * n + li] = INFINITY;
  }
}

// Exact row of each flagged node (amb[i] != 0) of the tensor-core builds, same arithmetic as dist_blocks_kernel
// (sequential over the feature dimension).  scratch_ld > 0: `dense` is a scratch area of rows and amb[i] - 1 is this
// row's slot (the thresholded build writes no dense blocks).
__global__ void __launch_bounds__(256) exact_rows_kernel(const float* __restrict__ reid, int64_t dim,
                                                         const int64_t* __restrict__ frame, const int64_t* __restrict__ gptr,
                                                         int64_t num_graphs, const int64_t* __restrict__ doff, int64_t max_dist,
                                                         const int32_t* __restrict__ amb, float* __restrict__ dense,
                                                         int64_t scratch_ld, int64_t scratch_rows) {
  const int64_t i = blockIdx.x;
  if (!amb[i]) return;
  const int64_t g = window_of(gptr, num_graphs, i);
  const int64_t n0 = gptr[g], n = gptr[g + 1] - n0, li = i - n0;
  if (scratch_ld > 0 && amb[i] > scratch_rows) return;
  float* rowp = scratch_ld > 0 ? dense + (int64_t)(amb[i] - 1) * scratch_ld : dense + doff[g] + li * n;
  const int64_t fi = frame[i];
  const float eps = 1e-6f;
  for (int64_t lj = threadIdx.x; lj < n; lj += blockDim.x) {
    float v = INFINITY;
    if (lj != li && frames_connect(fi, frame[n0 + lj], max_dist)) {
      // the reference evaluates pairs as (row = smaller index, col = larger index)
      const float* pa = reid + (n0 + (li < lj ? li : lj)) * dim;
      const float* pb = reid + (n0 + (li < lj ? lj : li)) * dim;
      float acc = 0.f;
      for (int64_t k = 0; k < dim; ++k) { const float d = (pa[k] - pb[k]) + eps; acc = fmaf(d, d, acc); }
      v = sqrtf(acc);
    }
    rowp[lj] = v;
  }
}

// warp per node i: every time-valid pair (i, j>i) of its window with its distance (no KNN pruning);
// kFill=false counts, true writes at row_start.
template <bool kFill>
__global__ void time_valid_pairs_kernel(const float* __restrict__ dense, const int64_t* __restrict__ gptr,
                                        int64_t num_graphs, const int64_t* __restrict__ doff,
                                        const int64_t* __restrict__ frame, int64_t num_nodes, int64_t max_dist,
                                        int64_t* __restrict__ row_cnt_or_start, int64_t* __restrict__ out_row,
                                        int64_t* __restrict__ out_col, float* __restrict__ out_dist) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < num_nodes; i += nwarps) {
    const int64_t g = window_of(gptr, num_graphs, i);
    const int64_t n0 = gptr[g], n = gptr[g + 1] - n0, li = i - n0;
    const float* D = dense + doff[g];
    const int64_t fi = frame[i];
    int64_t cursor = kFill ? row_cnt_or_start[i] : 0;
    for (int64_t j0 = li + 1; j0 < n; j0 += 32) {
      const int64_t lj = j0 + lane;
      const bool ok = lj < n && frames_connect(fi, frame[n0 + lj], max_dist);
      const float d = ok ? D[li * n + lj] : 0.f;
      const unsigned m = __ballot_sync(kFullMask, ok);
      if (kFill && ok) {
        const int64_t pos = cursor + __popc(m & ((1u << lane) - 1u));
        out_row[pos] = i;
        out_col[pos] = n0 + lj;
        out_dist[pos] = d;
      }
      cursor += __popc(m);
    }
    if (!kFill && lane == 0) row_cnt_or_start[i] = cursor;
  }
}


// ------------------------------------------------------------------ row select
// One CTA per node: select_kth ranks the row, then the row of the "is among my k nearest" bit matrix M and
// (tensor-core path) the ambiguity test of the approximate distances.  Windows of up to SEL_MAX_N nodes keep the row's
// keys in registers (SEL_PER per thread); larger windows re-read the row (SEL_PER = 0).  Every row is ranked on ITS OWN
// entries, so nothing downstream assumes that the distance matrix is symmetric (repaired rows are exact, their mirror
// entries stay approximate).
constexpr int SEL_MAX_N = 20 * SEL_THREADS;

template <bool kAmb, int SEL_PER>
__global__ void __launch_bounds__(SEL_THREADS) row_select_kernel(
    const float* __restrict__ dense, const int64_t* __restrict__ gptr, int64_t num_graphs, const int64_t* __restrict__ doff,
    const int64_t* __restrict__ moff, int64_t k, const int32_t* __restrict__ row_mask, uint32_t* __restrict__ thr_key,
    int32_t* __restrict__ thr_idx, uint32_t* __restrict__ M, const float* __restrict__ norm2,
    const float* __restrict__ win_nmax, float beta, float keps, int32_t* __restrict__ amb, int32_t* __restrict__ amb_count,
    int64_t scratch_ld, int64_t scratch_rows) {
  __shared__ SelectSmem sm;
  __shared__ float s_min[SEL_THREADS / 32];
  const int64_t i = blockIdx.x;
  if (row_mask != nullptr && row_mask[i] == 0) return;
  const int64_t g = window_of(gptr, num_graphs, i);
  const int64_t n0 = gptr[g], n = gptr[g + 1] - n0, li = i - n0;
  // scratch_ld > 0: `dense` holds exact rows of the flagged nodes only, row_mask[i] - 1 is the row's slot
  if (scratch_ld > 0 && row_mask[i] > scratch_rows) return;
  const float* rowp = scratch_ld > 0 ? dense + (int64_t)(row_mask[i] - 1) * scratch_ld : dense + doff[g] + li * n;
  const int words = (int)((n + 31) >> 5);
  uint32_t* mrow = M + moff[g] + li * words;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const RowKeys<SEL_PER> keys(rowp, n);
  uint32_t tau;
  int32_t found;
  select_kth(keys, rowp, n, k, sm, tau, found);
  if (tid == 0) { thr_key[i] = tau; thr_idx[i] = found; }
  // row of M and the smallest value left outside the top-k
  float mn = INFINITY;
  const int nq = keys.chunks(n);
#pragma unroll
  for (int q = 0; q < nq; ++q) {
    const int64_t j = tid + (int64_t)q * SEL_THREADS;
    if ((int64_t)q * SEL_THREADS < n) {                                   // uniform per warp group
      const uint32_t key = keys[q];
      const bool in = j < n && (key < tau || (key == tau && j <= found));
      const unsigned m = __ballot_sync(kFullMask, in);
      const int w = q * (SEL_THREADS / 32) + warp;
      if (lane == 0 && w < words) mrow[w] = m;
      if (kAmb && j < n && !in) mn = fminf(mn, key_value(key));
    }
  }
  if (kAmb) {
    for (int d = 16; d > 0; d >>= 1) mn = fminf(mn, __shfl_xor_sync(kFullMask, mn, d));
    if (lane == 0) s_min[warp] = mn;
    __syncthreads();
    if (tid == 0) {
      for (int q = 1; q < SEL_THREADS / 32; ++q) mn = fminf(mn, s_min[q]);
      int flag = 0;
      if (tau != 0xffffffffu) {
        const float vk = key_value(tau);
        if (isfinite(vk) && isfinite(mn)) {
          const float band = beta * (norm2[i] + win_nmax[g] + keps);      // absolute error bound on d^2
          flag = (mn - vk) <= 2.f * band ? 1 : 0;                         // the approximate rows hold d^2
        }
      }
      amb[i] = flag;
      if (flag) atomicAdd(amb_count, 1);
    }
  }
}

template <bool kAmb>
static void launch_row_select(int64_t max_n, int64_t n, cudaStream_t s, const float* dense, const int64_t* gptr, int64_t num_graphs,
                              const int64_t* doff, const int64_t* moff, int64_t k, const int32_t* row_mask, uint32_t* thr_key,
                              int32_t* thr_idx, uint32_t* M, const float* norm2, const float* win_nmax, float beta, float keps,
                              int32_t* amb, int32_t* amb_count, int64_t scratch_ld = 0, int64_t scratch_rows = 0) {
  const unsigned g = (unsigned)n;
#define MPN_SEL(PER)                                                                                                     \
  row_select_kernel<kAmb, PER><<<g, SEL_THREADS, 0, s>>>(dense, gptr, num_graphs, doff, moff, k, row_mask, thr_key, thr_idx, M, \
                                                         norm2, win_nmax, beta, keps, amb, amb_count, scratch_ld, scratch_rows)
  if (max_n <= 5 * SEL_THREADS) MPN_SEL(5);
  else if (max_n <= 9 * SEL_THREADS) MPN_SEL(9);
  else if (max_n <= 12 * SEL_THREADS) MPN_SEL(12);
  else if (max_n <= SEL_MAX_N) MPN_SEL(20);
  else MPN_SEL(0);
#undef MPN_SEL
  count_launch();
}

__global__ void window_max_kernel(const float* __restrict__ v, const int64_t* __restrict__ gptr, float* __restrict__ out) {
  __shared__ float s[8];
  const int64_t a = gptr[blockIdx.x], b = gptr[blockIdx.x + 1];
  float m = 0.f;
  for (int64_t j = a + threadIdx.x; j < b; j += blockDim.x) m = fmaxf(m, v[j]);
  for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(kFullMask, m, d));
  if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) { for (int q = 1; q < (int)(blockDim.x >> 5); ++q) m = fmaxf(m, s[q]); out[blockIdx.x] = m; }
}

// MT[j][i] = M[i][j] per window: one warp per 32 x 32 bit tile.
__global__ void bit_transpose_kernel(const uint32_t* __restrict__ M, uint32_t* __restrict__ MT, const int64_t* __restrict__ gptr,
                                     const int64_t* __restrict__ moff) {
  const int64_t w = blockIdx.y;
  const int64_t n = gptr[w + 1] - gptr[w];
  const int words = (int)((n + 31) >> 5);
  const uint32_t* m = M + moff[w];
  uint32_t* mt = MT + moff[w];
  const int lane = threadIdx.x & 31;
  const int64_t tiles = (int64_t)words * words;
  for (int64_t t = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; t < tiles; t += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int rb = (int)(t / words), cb = (int)(t - (int64_t)rb * words);   // rows 32rb.., bit columns 32cb..
    const int64_t r = (int64_t)rb * 32 + lane;
    const uint32_t word = r < n ? m[r * words + cb] : 0u;
    uint32_t mine = 0u;
#pragma unroll
    for (int b = 0; b < 32; ++b) {
      const unsigned col = __ballot_sync(kFullMask, (word >> b) & 1u);   // column 32cb + b over rows 32rb..32rb+31
      if (lane == b) mine = col;
    }
    const int64_t c = (int64_t)cb * 32 + lane;
    if (c < n) mt[c * words + rb] = mine;
  }
}

// warp per node i: kept pairs (i, j > i) from the bit matrices, ascending j; kFill=false counts.
template <bool kFill>
__global__ void mask_pairs_kernel(const uint32_t* __restrict__ M, const uint32_t* __restrict__ MT, const float* __restrict__ dense,
                                  const int64_t* __restrict__ gptr, int64_t num_graphs, const int64_t* __restrict__ doff,
                                  const int64_t* __restrict__ moff, const int64_t* __restrict__ frame, int64_t num_nodes,
                                  int64_t max_dist, int reciprocal, int64_t* __restrict__ row_cnt_or_start,
                                  int64_t* __restrict__ out_row, int64_t* __restrict__ out_col, float* __restrict__ out_dist) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < num_nodes; i += nwarps) {
    const int64_t g = window_of(gptr, num_graphs, i);
    const int64_t n0 = gptr[g], n = gptr[g + 1] - n0, li = i - n0;
    const int words = (int)((n + 31) >> 5);
    const uint32_t* mi = M + moff[g] + li * words;
    const uint32_t* mti = MT + moff[g] + li * words;
    const int64_t fi = frame[i];
    int64_t cursor = kFill ? row_cnt_or_start[i] : 0;
    for (int c0 = (int)((li + 1) >> 5); c0 < words; c0 += 32) {
      const int c = c0 + lane;
      uint32_t bits = 0u;
      if (c < words) {
        bits = reciprocal ? (mi[c] & mti[c]) : (mi[c] | mti[c]);
        const int64_t jbase = (int64_t)c * 32;
        if (jbase <= li) bits &= (li - jbase >= 31) ? 0u : (0xffffffffu << (li - jbase + 1));   // j > i only
        uint32_t rest = bits;
        while (rest) {                                                  // few bits: drop pairs that are not time-valid
          const int b = __ffs(rest) - 1;
          rest &= rest - 1;
          const int64_t lj = jbase + b;
          if (lj >= n || !frames_connect(fi, frame[n0 + lj], max_dist)) bits &= ~(1u << b);
        }
      }
      int cnt = __popc(bits), incl = cnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(kFullMask, incl, d); if (lane >= d) incl += v; }
      if (kFill) {
        int64_t pos = cursor + incl - cnt;
        while (bits) {
          const int b = __ffs(bits) - 1;
          bits &= bits - 1;
          const int64_t lj = (int64_t)c * 32 + b;
          out_row[pos] = i;
          out_col[pos] = n0 + lj;
          out_dist[pos] = dense != nullptr ? dense[doff[g] + li * n + lj] : 0.f;   // (recomputed exactly by the caller)
          ++pos;
        }
      }
      cursor += __shfl_sync(kFullMask, incl, 31);
    }
    if (!kFill && lane == 0) row_cnt_or_start[i] = cursor;
  }
}

__global__ void graph_offsets_kernel(const int64_t* __restrict__ gptr, int64_t num_graphs, int64_t* __restrict__ doff,
                                     int64_t* __restrict__ moff) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int64_t acc = 0, macc = 0;
    for (int64_t g = 0; g < num_graphs; ++g) {
      const int64_t n = gptr[g + 1] - gptr[g];
      doff[g] = acc; acc += n * n;
      moff[g] = macc; macc += n * ((n + 31) >> 5);                      // words of the window's bit matrices
    }
    doff[num_graphs] = acc;
    moff[num_graphs] = macc;
  }
}

__global__ void graph_pair_ptr_kernel(const int64_t* __restrict__ gptr, int64_t num_graphs, int64_t num_nodes,
                                      const int64_t* __restrict__ row_start, int64_t* __restrict__ out) {
  for (int64_t g = blockIdx.x * blockDim.x + threadIdx.x; g <= num_graphs; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t node = g < num_graphs ? gptr[g] : num_nodes;
    out[g] = row_start[node];
  }
}

int64_t gram_workspace_bytes(int64_t num_nodes, int64_t total_tiles, int64_t num_graphs, int64_t dim);
float gram_band_keps(int64_t dim);
int gram_dist_blocks(const float* reid, int64_t dim, const int64_t* frame, const int64_t* gptr, const int64_t* h_gptr,
                     int64_t num_graphs, const int64_t* doff, int64_t max_dist, void* ws, float* dense,
                     int32_t* status, float** norm2_out, int32_t** amb_out, int32_t** amb_count_out, cudaStream_t s);
bool gram_thresholded_applies(const int64_t* h_gptr, int64_t num_graphs, int64_t top_k);
int gram_thresholded_select(const float* reid, int64_t dim, const int64_t* frame, const int64_t* gptr, const int64_t* h_gptr,
                            int64_t num_graphs, const int64_t* moff, int64_t max_dist, int64_t top_k, void* ws,
                            const float* win_nmax_buf, float beta, uint32_t* M, int32_t* status, float** norm2_out,
                            int32_t** amb_out, int32_t** amb_count_out,
                            void (*window_max)(const float*, const int64_t*, int64_t, float*, cudaStream_t), cudaStream_t s);

static void launch_window_max(const float* v, const int64_t* gptr, int64_t num_graphs, float* out, cudaStream_t s) {
  window_max_kernel<<<(unsigned)num_graphs, 256, 0, s>>>(v, gptr, out);
  count_launch();
}

}  // namespace mpn

using namespace mpn;

extern "C" {

int64_t mpn_knn_graph_workspace(int64_t num_nodes, int64_t sum_sq_nodes, int64_t num_graphs) {
  const int64_t mask_words = sum_sq_nodes / 32 + num_nodes + 32;       // >= sum_g n_g * ceil(n_g / 32)
  const int64_t base = align_up(sum_sq_nodes * 4, 256) + 2 * align_up((num_graphs + 1) * 8, 256) +
                       2 * align_up(num_nodes * 4, 256) + align_up((num_nodes + 1) * 8, 256) +
                       2 * align_up(mask_words * 4, 256) + align_up(num_graphs * 4, 256) + 2048;
  // tensor-core path: packed fp16 hi/lo image of the embeddings (dim <= 512 covered) + per-node scalars
  return base + gram_workspace_bytes(num_nodes, num_nodes / 128 + num_graphs, num_graphs, 512) + 256;
}

int mpn_knn_graph_pairs(const int64_t* frame, const int64_t* gptr, const int64_t* h_gptr, int64_t num_graphs,
                        const float* reid, int64_t dim, int64_t top_k, int reciprocal, int64_t max_frame_dist,
                        int use_tensor_cores, void* ws, int64_t capacity, int64_t* out_row, int64_t* out_col,
                        float* out_dist, int64_t* graph_pair_ptr, int64_t* h_graph_pair_ptr, int64_t* h_stats,
                        void* stream) {
  MPN_CHECK_ARG(num_graphs >= 1 && h_gptr && gptr && frame && reid && ws, "knn_graph_pairs: null / empty arguments");
  MPN_CHECK_ARG(out_row && out_col && out_dist && graph_pair_ptr && h_graph_pair_ptr, "knn_graph_pairs: null outputs");
  MPN_CHECK_ARG(num_graphs <= 65535, "knn_graph_pairs: at most 65535 windows per call");
  cudaStream_t s = as_stream(stream);
  const int64_t n = h_gptr[num_graphs];
  int64_t sum_sq = 0, max_n = 0;
  for (int64_t g = 0; g < num_graphs; ++g) {
    const int64_t ng = h_gptr[g + 1] - h_gptr[g];
    MPN_CHECK_ARG(ng >= 0, "knn_graph_pairs: node_graph_ptr must be non-decreasing");
    sum_sq += ng * ng;
    max_n = ng > max_n ? ng : max_n;
  }
  if (n == 0) { for (int64_t g = 0; g <= num_graphs; ++g) h_graph_pair_ptr[g] = 0; return MPN_OK; }
  Carver cv(ws);
  float* dense = cv.take<float>(sum_sq);
  int64_t* doff = cv.take<int64_t>(num_graphs + 1);
  int64_t* moff = cv.take<int64_t>(num_graphs + 1);
  int64_t mask_words = 0;
  for (int64_t g = 0; g < num_graphs; ++g) { const int64_t ng = h_gptr[g + 1] - h_gptr[g]; mask_words += ng * ((ng + 31) >> 5); }
  uint32_t* M = cv.take<uint32_t>(mask_words + 32);
  uint32_t* MT = cv.take<uint32_t>(mask_words + 32);
  float* win_nmax = cv.take<float>(num_graphs);
  uint32_t* tk = cv.take<uint32_t>(n);
  int32_t* ti = cv.take<int32_t>(n);
  int64_t* row_start = cv.take<int64_t>(n + 1);
  const int prune = top_k >= 0 ? 1 : 0;
  // Gram distances only pre-rank (they are repaired / recomputed exactly below); without pruning every
  // distance is an output, so the exact kernel is used directly.
  const bool tc = use_tensor_cores && prune && dim % 64 == 0 && dim <= 512 && reinterpret_cast<uintptr_t>(reid) % 16 == 0;
  int32_t* status = reinterpret_cast<int32_t*>(cv.take<int32_t>(4));
  float* norm2 = nullptr;
  int32_t* amb = nullptr;
  int32_t* amb_count = nullptr;
  int rc = MPN_OK;
  MPN_CUDA(cudaMemsetAsync(status, 0, 16, s));

  graph_offsets_kernel<<<1, 32, 0, s>>>(gptr, num_graphs, doff, moff); count_launch();
  // large windows on the tensor-core path: thresholded candidate lists instead of dense N^2 blocks (MPN_KNN_DENSE=1: old path)
  const bool force_dense = getenv("MPN_KNN_DENSE") != nullptr;          // read per call: tests toggle it
  const bool tg = tc && max_n <= SEL_MAX_N && !force_dense && gram_thresholded_applies(h_gptr, num_graphs, top_k);
  int64_t scratch_rows = 0;
  // pruned builds: per-row select into the bit matrix M -> transpose -> pairs (i, j > i) kept by M[i][j] and / or M[j][i]
  if (tg) {
    rc = gram_thresholded_select(reid, dim, frame, gptr, h_gptr, num_graphs, moff, max_frame_dist, top_k,
                                 static_cast<char*>(ws) + cv.off, win_nmax, 2e-6f, M, status, &norm2, &amb, &amb_count,
                                 launch_window_max, s);
    if (rc) return rc;
    // flagged rows (uncertain top-k set, list overflow, too few candidates): exact fp32 row into a scratch slot of the
    // (otherwise unused) dense area, ranked by the dense row select
    scratch_rows = sum_sq / max_n;
    exact_rows_kernel<<<(unsigned)n, 256, 0, s>>>(reid, dim, frame, gptr, num_graphs, doff, max_frame_dist, amb, dense, max_n,
                                                  scratch_rows); count_launch();
    launch_row_select<false>(max_n, n, s, dense, gptr, num_graphs, doff, moff, top_k, amb, tk, ti, M, nullptr, nullptr, 0.f,
                             0.f, nullptr, nullptr, max_n, scratch_rows);
  } else if (tc) {
    rc = gram_dist_blocks(reid, dim, frame, gptr, h_gptr, num_graphs, doff, max_frame_dist,
                          static_cast<char*>(ws) + cv.off, dense, status, &norm2, &amb, &amb_count, s);
    if (rc) return rc;
    window_max_kernel<<<(unsigned)num_graphs, 256, 0, s>>>(norm2, gptr, win_nmax); count_launch();
    launch_row_select<true>(max_n, n, s, dense, gptr, num_graphs, doff, moff, top_k, nullptr, tk, ti, M, norm2, win_nmax, 2e-6f,
                            gram_band_keps(dim), amb, amb_count);
    // rows whose top-k set is not certain: exact fp32 distances, ranked again
    exact_rows_kernel<<<(unsigned)n, 256, 0, s>>>(reid, dim, frame, gptr, num_graphs, doff, max_frame_dist, amb, dense, 0, 0);
    count_launch();
    launch_row_select<false>(max_n, n, s, dense, gptr, num_graphs, doff, moff, top_k, amb, tk, ti, M, nullptr, nullptr, 0.f,
                             0.f, nullptr, nullptr);
  } else {
    const int64_t nt = ceil_div(max_n, DT);
    dim3 grid((unsigned)(nt * (nt + 1) / 2), (unsigned)num_graphs);
    dist_blocks_kernel<<<grid, 256, 0, s>>>(reid, dim, frame, gptr, doff, max_frame_dist, dense); count_launch();
    if (prune)
      launch_row_select<false>(max_n, n, s, dense, gptr, num_graphs, doff, moff, top_k, nullptr, tk, ti, M, nullptr, nullptr, 0.f,
                               0.f, nullptr, nullptr);
  }
  const unsigned wgrid = (unsigned)std::min<int64_t>(ceil_div(n * 32, 256), (int64_t)sm_count() * 16);
  if (prune) {
    const int64_t max_words = (max_n + 31) >> 5;
    const unsigned tgrid = (unsigned)std::min<int64_t>(std::max<int64_t>(ceil_div(max_words * max_words * 32, 256), 1), 4096);
    bit_transpose_kernel<<<dim3(tgrid, (unsigned)num_graphs), 256, 0, s>>>(M, MT, gptr, moff); count_launch();
    mask_pairs_kernel<false><<<wgrid, 256, 0, s>>>(M, MT, tg ? nullptr : dense, gptr, num_graphs, doff, moff, frame, n, max_frame_dist, reciprocal,
                                                  row_start, nullptr, nullptr, nullptr); count_launch();
  } else {
    time_valid_pairs_kernel<false><<<wgrid, 256, 0, s>>>(dense, gptr, num_graphs, doff, frame, n, max_frame_dist, row_start,
                                                        nullptr, nullptr, nullptr); count_launch();
  }
  MPN_LAUNCH_CHECK();
  rc = exclusive_scan_i64(row_start, row_start, n, s);
  if (rc) return rc;
  graph_pair_ptr_kernel<<<(unsigned)ceil_div(num_graphs + 1, 256), 256, 0, s>>>(gptr, num_graphs, n, row_start, graph_pair_ptr);
  count_launch();
  MPN_CUDA(cudaMemcpyAsync(h_graph_pair_ptr, graph_pair_ptr, 8 * (num_graphs + 1), cudaMemcpyDeviceToHost, s));
  int32_t h_flags[2] = {0, 0};                                      // fp16 overflow in the Gram kernel, #ambiguous rows
  MPN_CUDA(cudaMemcpyAsync(&h_flags[0], status, 4, cudaMemcpyDeviceToHost, s));
  if (tc) MPN_CUDA(cudaMemcpyAsync(&h_flags[1], amb_count, 4, cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaStreamSynchronize(s));
  if (tg && h_flags[1] > scratch_rows) h_flags[0] = 1;              // more flagged rows than scratch slots: exact kernel
  if (tc && h_flags[0] != 0)                                        // embeddings beyond the fp16 range: exact kernel
    return mpn_knn_graph_pairs(frame, gptr, h_gptr, num_graphs, reid, dim, top_k, reciprocal, max_frame_dist, 0, ws,
                               capacity, out_row, out_col, out_dist, graph_pair_ptr, h_graph_pair_ptr, h_stats, stream);
  // build code: 0 exact, 1 dense Gram + row select, 2 thresholded candidate lists
  if (h_stats != nullptr) { h_stats[0] = tg ? 2 : (tc ? 1 : 0); h_stats[1] = h_flags[1]; }
  const int64_t total = h_graph_pair_ptr[num_graphs];
  if (total > capacity) {
    set_error("knn_graph_pairs: %lld pairs exceed the output capacity %lld", (long long)total, (long long)capacity);
    return MPN_ENOSPC;
  }
  if (prune) {
    mask_pairs_kernel<true><<<wgrid, 256, 0, s>>>(M, MT, tg ? nullptr : dense, gptr, num_graphs, doff, moff, frame, n, max_frame_dist, reciprocal,
                                                 row_start, out_row, out_col, out_dist); count_launch();
  } else {
    time_valid_pairs_kernel<true><<<wgrid, 256, 0, s>>>(dense, gptr, num_graphs, doff, frame, n, max_frame_dist, row_start,
                                                       out_row, out_col, out_dist); count_launch();
  }
  MPN_LAUNCH_CHECK();
  if (tc && total > 0)                                              // the edge feature is always the exact distance
    return mpn_pair_reid_dist(reid, n, dim, out_row, out_col, total, out_dist, stream);
  return MPN_OK;
}

}  // extern "C"
