// Graph construction kernels: time-valid candidate pairs, per-pair ReID distance,
// KNN keep mask, order-preserving compaction, geometric edge features + assembly.
// Integer / index work here is bit-exact with the reference's CPU path by construction
// (same total order on (distance, index)); see include/mpntrack_b200.h for citations.
#include <math.h>

#include "common.cuh"
#include "knn_select.cuh"

namespace mpn {

// ------------------------------------------------------------------ time-valid pairs
// Upper end of the node range that may pair with node i (its window).
__device__ __forceinline__ int64_t window_end(const int64_t* __restrict__ gptr, int64_t g,
                                              int64_t n, int64_t i) {
  return gptr == nullptr || g <= 0 ? n : gptr[window_of(gptr, g, i) + 1];
}

template <bool kFill>
__global__ void time_valid_kernel(const int64_t* __restrict__ frame, int64_t n,
                                  const int64_t* __restrict__ gptr, int64_t g,
                                  int64_t max_dist, int64_t* __restrict__ row_cnt_or_start,
                                  int64_t* __restrict__ out_row, int64_t* __restrict__ out_col) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < n; i += nwarps) {
    const int64_t fi = frame[i];
    const int64_t end = window_end(gptr, g, n, i);
    int64_t cursor = kFill ? row_cnt_or_start[i] : 0;
    for (int64_t j0 = i + 1; j0 < end; j0 += 32) {
      const int64_t j = j0 + lane;
      const bool ok = j < end && frames_connect(fi, frame[j], max_dist);
      const unsigned m = __ballot_sync(kFullMask, ok);
      if (kFill && ok) {
        const int64_t pos = cursor + __popc(m & ((1u << lane) - 1u));
        out_row[pos] = i;
        out_col[pos] = j;
      }
      cursor += __popc(m);
    }
    if (!kFill && lane == 0) row_cnt_or_start[i] = cursor;
  }
}

// ------------------------------------------------------------------ per-pair ReID distance
// One warp per pair; lane-strided partial sums of ((a-b)+eps)^2, then a fixed xor tree.
__global__ void pair_dist_kernel(const float* __restrict__ reid, int64_t dim,
                                 const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                 int64_t npairs, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const float eps = 1e-6f;
  for (int64_t p = warp; p < npairs; p += nwarps) {
    const float* a = reid + row[p] * dim;
    const float* b = reid + col[p] * dim;
    float acc = 0.f;
    if ((dim & 3) == 0) {
      const float4* a4 = reinterpret_cast<const float4*>(a);
      const float4* b4 = reinterpret_cast<const float4*>(b);
      for (int64_t q = lane; q < (dim >> 2); q += 32) {
        const float4 u = __ldg(a4 + q), v = __ldg(b4 + q);
        float d;
        d = (u.x - v.x) + eps; acc = fmaf(d, d, acc);
        d = (u.y - v.y) + eps; acc = fmaf(d, d, acc);
        d = (u.z - v.z) + eps; acc = fmaf(d, d, acc);
        d = (u.w - v.w) + eps; acc = fmaf(d, d, acc);
      }
    } else {
      for (int64_t q = lane; q < dim; q += 32) {
        const float d = (a[q] - b[q]) + eps;
        acc = fmaf(d, d, acc);
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(kFullMask, acc, s);
    if (lane == 0) out[p] = sqrtf(acc);
  }
}

// ------------------------------------------------------------------ KNN keep mask
__global__ void fill_f32(float* __restrict__ p, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    p[i] = v;
}

__global__ void dense_scatter(const float* __restrict__ d, const int64_t* __restrict__ row,
                              const int64_t* __restrict__ col, int64_t e, int64_t n,
                              int mirror, float* __restrict__ dense) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < e;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = row[i], c = col[i];
    dense[r * n + c] = d[i];
    if (mirror) dense[c * n + r] = d[i];
  }
}

// One CTA per dense row: its k-th smallest (key, index) pair (streamed select_kth).
// thr_key[i], thr_idx[i]: entry (i, j) is within the top-k  <=>
//   key(i,j) < thr_key[i]  ||  (key(i,j) == thr_key[i] && j <= thr_idx[i]).
__global__ void __launch_bounds__(SEL_THREADS) keep_threshold_kernel(const float* __restrict__ dense, int64_t n, int64_t k,
                                                                    uint32_t* __restrict__ thr_key,
                                                                    int32_t* __restrict__ thr_idx) {
  __shared__ SelectSmem sm;
  const float* rowp = dense + (int64_t)blockIdx.x * n;
  uint32_t tau;
  int32_t found;
  select_kth(RowKeys<0>(rowp, n), rowp, n, k, sm, tau, found);
  if (threadIdx.x == 0) { thr_key[blockIdx.x] = tau; thr_idx[blockIdx.x] = found; }
}

__global__ void knn_gather_kernel(const float* __restrict__ dense, int64_t n,
                                  const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                  int64_t e, const uint32_t* __restrict__ thr_key,
                                  const int32_t* __restrict__ thr_idx, int reciprocal,
                                  int all_in, uint8_t* __restrict__ keep) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < e;
       i += (int64_t)gridDim.x * blockDim.x) {
    if (all_in) { keep[i] = 1; continue; }
    const int64_t r = row[i], c = col[i];
    const uint32_t krc = order_key(dense[r * n + c]);
    const uint32_t kcr = order_key(dense[c * n + r]);
    const bool a = krc < thr_key[r] || (krc == thr_key[r] && c <= thr_idx[r]);
    const bool b = kcr < thr_key[c] || (kcr == thr_key[c] && r <= thr_idx[c]);
    keep[i] = (reciprocal ? (a && b) : (a || b)) ? 1 : 0;
  }
}

// ------------------------------------------------------------------ compaction
__global__ void mask_to_i64(const uint8_t* __restrict__ m, int64_t n, int64_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    out[i] = m[i] ? 1 : 0;
}

__global__ void compact_kernel(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                               const float* __restrict__ dist, const uint8_t* __restrict__ keep,
                               const int64_t* __restrict__ pos, int64_t n,
                               int64_t* __restrict__ orow, int64_t* __restrict__ ocol,
                               float* __restrict__ odist) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    if (!keep[i]) continue;
    const int64_t p = pos[i];
    orow[p] = row[i];
    ocol[p] = col[i];
    if (dist != nullptr) odist[p] = dist[i];
  }
}

// ------------------------------------------------------------------ edge features
__global__ void edge_feats_kernel(const int64_t* __restrict__ row, const int64_t* __restrict__ col,
                                  int64_t np, const float* __restrict__ frame,
                                  const float* __restrict__ h, const float* __restrict__ w,
                                  const float* __restrict__ fx, const float* __restrict__ fy,
                                  float fps, const float* __restrict__ rd, int64_t ad,
                                  float* __restrict__ attr, int64_t* __restrict__ eidx) {
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < np;
       p += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = row[p], j = col[p];
    const float hi = h[i], hj = h[j];
    const float hbar = __fdiv_rn(hi + hj, 2.f);
    float f[6];
    f[0] = __fdiv_rn(frame[j], fps) - __fdiv_rn(frame[i], fps);
    f[1] = __fdiv_rn(fx[j] - fx[i], hbar);
    f[2] = __fdiv_rn(fy[j] - fy[i], hbar);
    f[3] = logf(__fdiv_rn(hj, hi));
    f[4] = logf(__fdiv_rn(w[j], w[i]));
    f[5] = rd != nullptr ? rd[p] : 0.f;
    float* a0 = attr + p * ad;
    float* a1 = attr + (p + np) * ad;
    for (int q = 0; q < ad; ++q) { a0[q] = f[q]; a1[q] = f[q]; }
    eidx[p] = i;            eidx[np + p] = j;          // row of edge_index: sources
    eidx[2 * np + p] = j;   eidx[3 * np + p] = i;      // row 1: destinations
  }
}

static inline unsigned grid_for(int64_t n, int threads, int per_sm = 8) {
  int64_t want = ceil_div(n > 0 ? n : 1, threads);
  int64_t cap = (int64_t)sm_count() * per_sm;
  return (unsigned)(want < cap ? want : cap);
}

}  // namespace mpn

using namespace mpn;

extern "C" {

int mpn_time_valid_pairs_count(const int64_t* frame_num, int64_t n, const int64_t* gptr,
                               int64_t g, int64_t max_frame_dist, int64_t* row_start,
                               int64_t* h_total, void* stream) {
  MPN_CHECK_ARG(n >= 0 && row_start != nullptr && h_total != nullptr, "time_valid_pairs_count: bad args");
  cudaStream_t s = as_stream(stream);
  if (n == 0) { *h_total = 0; MPN_CUDA(cudaMemsetAsync(row_start, 0, 8, s)); return MPN_OK; }
  MPN_CHECK_ARG(frame_num != nullptr, "time_valid_pairs_count: frame_num is null");
  time_valid_kernel<false><<<grid_for(n * 32, 256), 256, 0, s>>>(frame_num, n, gptr, g, max_frame_dist,
                                                               row_start, nullptr, nullptr); count_launch();
  MPN_LAUNCH_CHECK();
  int rc = exclusive_scan_i64(row_start, row_start, n, s);
  if (rc) return rc;
  MPN_CUDA(cudaMemcpyAsync(h_total, row_start + n, 8, cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaStreamSynchronize(s));
  return MPN_OK;
}

int mpn_time_valid_pairs_fill(const int64_t* frame_num, int64_t n, const int64_t* gptr, int64_t g,
                              int64_t max_frame_dist, const int64_t* row_start, int64_t* out_row,
                              int64_t* out_col, void* stream) {
  if (n == 0) return MPN_OK;
  MPN_CHECK_ARG(frame_num && row_start && out_row && out_col, "time_valid_pairs_fill: null pointer");
  time_valid_kernel<true><<<grid_for(n * 32, 256), 256, 0, as_stream(stream)>>>(
      frame_num, n, gptr, g, max_frame_dist, const_cast<int64_t*>(row_start), out_row, out_col); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_pair_reid_dist(const float* reid, int64_t n, int64_t dim, const int64_t* row,
                       const int64_t* col, int64_t np, float* out, void* stream) {
  MPN_CHECK_ARG(np >= 0 && dim > 0, "pair_reid_dist: bad sizes");
  if (np == 0) return MPN_OK;
  MPN_CHECK_ARG(reid && row && col && out, "pair_reid_dist: null pointer");
  (void)n;
  pair_dist_kernel<<<grid_for(np * 32, 256, 16), 256, 0, as_stream(stream)>>>(reid, dim, row, col, np, out); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int64_t mpn_knn_mask_workspace(int64_t n) {
  return align_up(n * n * 4, 256) + 2 * align_up(n * 4, 256) + 256;
}

int mpn_knn_mask(const float* d, const int64_t* row, const int64_t* col, int64_t e, int64_t n,
                 int64_t k, int reciprocal, int symmetric_edges, void* ws, uint8_t* keep,
                 void* stream) {
  MPN_CHECK_ARG(e >= 0 && n >= 0, "knn_mask: bad sizes");
  if (e == 0) return MPN_OK;
  MPN_CHECK_ARG(d && row && col && ws && keep, "knn_mask: null pointer");
  cudaStream_t s = as_stream(stream);
  Carver cv(ws);
  float* dense = cv.take<float>(n * n);
  uint32_t* tk = cv.take<uint32_t>(n);
  int32_t* ti = cv.take<int32_t>(n);
  const int all_in = k >= n;               // every rank is < k (utils/graph.py:73)
  if (!all_in && k > 0) {
    fill_f32<<<grid_for(n * n, 256), 256, 0, s>>>(dense, n * n, INFINITY); count_launch();
    dense_scatter<<<grid_for(e, 256), 256, 0, s>>>(d, row, col, e, n, symmetric_edges ? 0 : 1, dense); count_launch();
    keep_threshold_kernel<<<(unsigned)n, SEL_THREADS, 0, s>>>(dense, n, k, tk, ti); count_launch();
    knn_gather_kernel<<<grid_for(e, 256), 256, 0, s>>>(dense, n, row, col, e, tk, ti, reciprocal, 0, keep); count_launch();
  } else if (all_in) {
    knn_gather_kernel<<<grid_for(e, 256), 256, 0, s>>>(dense, n, row, col, e, tk, ti, reciprocal, 1, keep); count_launch();
  } else {
    MPN_CUDA(cudaMemsetAsync(keep, 0, e, s));
  }
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_compact_pairs(const int64_t* row, const int64_t* col, const float* dist, const uint8_t* keep,
                      int64_t n, int64_t* scan_ws, int64_t* orow, int64_t* ocol, float* odist,
                      int64_t* h_kept, void* stream) {
  MPN_CHECK_ARG(n >= 0 && h_kept != nullptr, "compact_pairs: bad args");
  if (n == 0) { *h_kept = 0; return MPN_OK; }
  MPN_CHECK_ARG(row && col && keep && scan_ws && orow && ocol, "compact_pairs: null pointer");
  cudaStream_t s = as_stream(stream);
  mask_to_i64<<<grid_for(n, 256), 256, 0, s>>>(keep, n, scan_ws); count_launch();
  int rc = exclusive_scan_i64(scan_ws, scan_ws, n, s);
  if (rc) return rc;
  compact_kernel<<<grid_for(n, 256), 256, 0, s>>>(row, col, dist, keep, scan_ws, n, orow, ocol, odist); count_launch();
  MPN_LAUNCH_CHECK();
  MPN_CUDA(cudaMemcpyAsync(h_kept, scan_ws + n, 8, cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaStreamSynchronize(s));
  return MPN_OK;
}

int mpn_edge_feats_assemble(const int64_t* row, const int64_t* col, int64_t np, const float* frame,
                            const float* h, const float* w, const float* fx, const float* fy,
                            float fps, const float* rd, int64_t ad, float* attr, int64_t* eidx,
                            void* stream) {
  MPN_CHECK_ARG(np >= 0 && (ad == 5 || ad == 6), "edge_feats_assemble: bad size");
  if (np == 0) return MPN_OK;                  // an empty tensor has a null data pointer
  MPN_CHECK_ARG((rd != nullptr && ad == 6) || (rd == nullptr && ad == 5),
                "edge_feats_assemble: attr_dim must be 6 with reid_dist, 5 without (got %lld)", (long long)ad);
  MPN_CHECK_ARG(row && col && frame && h && w && fx && fy && attr && eidx, "edge_feats_assemble: null pointer");
  edge_feats_kernel<<<grid_for(np, 256), 256, 0, as_stream(stream)>>>(row, col, np, frame, h, w, fx, fy,
                                                                    fps, rd, ad, attr, eidx); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // extern "C"

namespace mpn {
// Edge labels of the network-flow formulation (data/mot_graph.py:223-262).  'closest': a directed edge (r -> c) between
// two detections of the same identity is active iff c is r's closest same-identity partner (by node index) among its
// later (c > r) resp. earlier (c < r) neighbours.  Index distances to distinct partners are distinct, so the reference's
// arg-min has no ties; the minimum is found with integer atomics (order independent).
__global__ void label_extrema_kernel(const int64_t* __restrict__ row, const int64_t* __restrict__ col, int64_t num_edges,
                                     const int64_t* __restrict__ ids, int32_t* __restrict__ fut, int32_t* __restrict__ past) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < num_edges; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = row[e], c = col[e];
    const int64_t a = ids[r];
    if (a == -1 || a != ids[c]) continue;
    if (c > r) atomicMin(&fut[r], (int32_t)c);
    else if (c < r) atomicMax(&past[r], (int32_t)c);
  }
}

__global__ void label_assign_kernel(const int64_t* __restrict__ row, const int64_t* __restrict__ col, int64_t num_edges,
                                    const int64_t* __restrict__ ids, const int32_t* __restrict__ fut,
                                    const int32_t* __restrict__ past, int closest, float* __restrict__ labels) {
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < num_edges; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = row[e], c = col[e];
    const int64_t a = ids[r];
    bool on = a != -1 && a == ids[c];
    if (on && closest) on = c > r ? fut[r] == (int32_t)c : (c < r && past[r] == (int32_t)c);
    labels[e] = on ? 1.f : 0.f;
  }
}
}  // namespace mpn

extern "C" int mpn_assign_edge_labels(const int64_t* edge_row, const int64_t* edge_col, int64_t num_edges,
                                      const int64_t* node_ids, int64_t num_nodes, int closest, void* workspace,
                                      float* labels, void* stream) {
  using namespace mpn;
  MPN_CHECK_ARG(num_edges >= 0 && num_nodes >= 0 && num_nodes < 2147483647LL, "assign_edge_labels: bad sizes");
  if (num_edges == 0) return MPN_OK;
  MPN_CHECK_ARG(edge_row && edge_col && node_ids && labels && workspace, "assign_edge_labels: null argument");
  cudaStream_t s = as_stream(stream);
  int32_t* fut = static_cast<int32_t*>(workspace);
  int32_t* past = fut + num_nodes;
  const unsigned grid = (unsigned)std::min<int64_t>(ceil_div(num_edges, 256), (int64_t)sm_count() * 8);
  if (closest) {
    MPN_CUDA(cudaMemsetAsync(fut, 0x7f, sizeof(int32_t) * num_nodes, s));      // 0x7f7f7f7f > any node index
    MPN_CUDA(cudaMemsetAsync(past, 0xff, sizeof(int32_t) * num_nodes, s));     // -1
    label_extrema_kernel<<<grid, 256, 0, s>>>(edge_row, edge_col, num_edges, node_ids, fut, past); count_launch();
  }
  label_assign_kernel<<<grid, 256, 0, s>>>(edge_row, edge_col, num_edges, node_ids, fut, past, closest, labels); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}
