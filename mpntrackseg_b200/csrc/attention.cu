// Attentive aggregation of the node feature maps (models/mpn.py:117-137):
//   w_e  = softmax of the edge logits over each node's future (row<col) resp. past (row>col) neighbours
//          (torch_scatter.composite.scatter_softmax: exp(l - max) / (sum + 1e-12)),
//   flow = sum_e w_e * z[col_e]      (z: [N, C*H*W] feature maps),
// evaluated per (node, direction) over that node's contiguous slot range, neighbours taken in slot
// order (= the reference's scatter_add order on CPU): deterministic, no atomics.
#include <math.h>

#include "common.cuh"

namespace mpn {

constexpr int ATT_THREADS = 256;
constexpr int ATT_MAX_DEG = 1024;   // neighbours whose weights are cached in shared memory per pass

__global__ void __launch_bounds__(ATT_THREADS) attn_aggregate_kernel(
    const float* __restrict__ z, int64_t feat, const int32_t* __restrict__ slot_col,
    const int32_t* __restrict__ slot_edge, const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ in_ptr,
    const float* __restrict__ logits, int64_t num_nodes, float* __restrict__ flow_in, float* __restrict__ flow_out) {
  __shared__ float s_w[ATT_MAX_DEG];
  __shared__ int32_t s_c[ATT_MAX_DEG];
  __shared__ float s_red[32];
  const int64_t node = blockIdx.x >> 1;
  const int dir = blockIdx.x & 1;                       // 0 = flow_in (row>col), 1 = flow_out (row<col)
  const int32_t* ptr = dir == 0 ? in_ptr : out_ptr;
  float* out = (dir == 0 ? flow_in : flow_out) + node * feat;
  const int s0 = ptr[node], s1 = ptr[node + 1];
  const int deg = s1 - s0;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (deg == 0) {                                       // scatter_add zero fill
    for (int64_t i = tid; i < feat; i += ATT_THREADS) out[i] = 0.f;
    return;
  }
  // segment max
  float m = -INFINITY;
  for (int q = tid; q < deg; q += ATT_THREADS) m = fmaxf(m, logits[slot_edge[s0 + q]]);
  for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
  if (lane == 0) s_red[warp] = m;
  __syncthreads();
  m = s_red[0];
  for (int w = 1; w < ATT_THREADS / 32; ++w) m = fmaxf(m, s_red[w]);
  __syncthreads();
  // segment sum of exp, sequential order per thread then fixed tree (deterministic)
  float sum = 0.f;
  for (int q = tid; q < deg; q += ATT_THREADS) sum += expf(logits[slot_edge[s0 + q]] - m);
  for (int d = 16; d > 0; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
  if (lane == 0) s_red[warp] = sum;
  __syncthreads();
  sum = 0.f;
  for (int w = 0; w < ATT_THREADS / 32; ++w) sum += s_red[w];
  const float inv = 1.f / (sum + 1e-12f);
  // weighted sum of the neighbours' maps
  for (int q0 = 0; q0 < deg; q0 += ATT_MAX_DEG) {
    const int nq = deg - q0 < ATT_MAX_DEG ? deg - q0 : ATT_MAX_DEG;
    __syncthreads();
    for (int q = tid; q < nq; q += ATT_THREADS) {
      s_w[q] = expf(logits[slot_edge[s0 + q0 + q]] - m) * inv;
      s_c[q] = slot_col[s0 + q0 + q];
    }
    __syncthreads();
    for (int64_t i = tid; i < feat; i += ATT_THREADS) {
      float acc = q0 == 0 ? 0.f : out[i];
      for (int q = 0; q < nq; ++q) acc += z[(int64_t)s_c[q] * feat + i] * s_w[q];   // x[col] * w, then add (mpn.py:123-124)
      out[i] = acc;
    }
  }
}

// ------------------------------------------------------------------ backward (training through the mask branch)
// Given G_dir[n] = d loss / d flow_dir[n]:
//   d w_q     = < G_dir[n], z[col_q] >                        (one warp per neighbour, fixed-order tree)
//   d logit_q = w_q (d w_q - S),  S = sum_p w_p d w_p          (softmax backward; the 1e-12 in the denominator keeps this form)
//   except for the dominant slot q* (largest logit, lowest slot among ties), whose w -> 1 would cancel dw_q* - S:
//   d logit_q* = w_q* (dw_q* W' - T'),  W' = sum_{p != q*} w_p,  T' = sum_{p != q*} w_p dw_p   (0 for a 1-slot segment)
//   S, W', T' are summed in double by thread 0 in slot order.
//   d z[c]    = sum over the slots q with col_q = c of w_q G_dir(q)[row_q]   (second kernel, slots of a column in slot order)
__device__ __forceinline__ float attn_d_logit(float w, float dw, bool dominant, double S, double Wo, double To) {
  return dominant ? (float)((double)w * ((double)dw * Wo - To)) : (float)((double)w * ((double)dw - S));
}

// 5 blocks per SM: 48 registers; the serial loop of thread 0 stays rolled, so nothing spills
__global__ void __launch_bounds__(ATT_THREADS, 5) attn_backward_edge_kernel(
    const float* __restrict__ z, int64_t feat, const int32_t* __restrict__ slot_col, const int32_t* __restrict__ slot_edge,
    const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ in_ptr, const float* __restrict__ logits,
    const float* __restrict__ g_in, const float* __restrict__ g_out, float* __restrict__ w_slot,
    float* __restrict__ d_logits) {
  __shared__ float s_w[ATT_MAX_DEG];
  __shared__ float s_dw[ATT_MAX_DEG];
  __shared__ float s_red[32];
  __shared__ int s_qred[32];
  __shared__ double s_S, s_Wo, s_To;
  const int64_t node = blockIdx.x >> 1;
  const int dir = blockIdx.x & 1;
  const int32_t* ptr = dir == 0 ? in_ptr : out_ptr;
  const float* G = (dir == 0 ? g_in : g_out) + node * feat;
  const int s0 = ptr[node], s1 = ptr[node + 1];
  const int deg = s1 - s0;
  if (deg == 0) return;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float m = -INFINITY;
  for (int q = tid; q < deg; q += ATT_THREADS) m = fmaxf(m, logits[slot_edge[s0 + q]]);
  for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
  if (lane == 0) s_red[warp] = m;
  __syncthreads();
  m = s_red[0];
  for (int w = 1; w < ATT_THREADS / 32; ++w) m = fmaxf(m, s_red[w]);
  __syncthreads();
  float sum = 0.f;
  int qs = deg;                                           // the dominant slot: the first one whose logit is the max
  for (int q = tid; q < deg; q += ATT_THREADS) {
    const float l = logits[slot_edge[s0 + q]];
    sum += expf(l - m);
    if (l == m && qs == deg) qs = q;
  }
  for (int d = 16; d > 0; d >>= 1) {
    sum += __shfl_xor_sync(0xffffffffu, sum, d);
    qs = min(qs, __shfl_xor_sync(0xffffffffu, qs, d));
  }
  if (lane == 0) { s_red[warp] = sum; s_qred[warp] = qs; }
  __syncthreads();
  sum = 0.f;
  for (int w = 0; w < ATT_THREADS / 32; ++w) { sum += s_red[w]; qs = min(qs, s_qred[w]); }
  const float inv = 1.f / (sum + 1e-12f);
  if (tid == 0) { s_S = 0.0; s_Wo = 0.0; s_To = 0.0; }   // accumulated by thread 0 over the chunks of pass 0
  for (int pass = 0; pass < 2; ++pass) {                  // pass 0: S, W', T'; pass 1: d logits
    for (int q0 = 0; q0 < deg; q0 += ATT_MAX_DEG) {
      const int nq = deg - q0 < ATT_MAX_DEG ? deg - q0 : ATT_MAX_DEG;
      __syncthreads();
      for (int q = tid; q < nq; q += ATT_THREADS) s_w[q] = expf(logits[slot_edge[s0 + q0 + q]] - m) * inv;
      for (int q = warp; q < nq; q += ATT_THREADS / 32) {
        const float* zr = z + (int64_t)slot_col[s0 + q0 + q] * feat;
        float acc = 0.f;
        for (int64_t i = lane; i < feat; i += 32) acc = fmaf(G[i], zr[i], acc);
        for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if (lane == 0) s_dw[q] = acc;
      }
      __syncthreads();
      if (pass == 0) {
        if (tid == 0) {
          double S = s_S, Wo = s_Wo, To = s_To;
#pragma unroll 1
          for (int q = 0; q < nq; ++q) {
            const double wd = (double)s_w[q] * (double)s_dw[q];
            S += wd;
            if (q0 + q != qs) { Wo += (double)s_w[q]; To += wd; }
          }
          s_S = S; s_Wo = Wo; s_To = To;
        }
      } else {
        for (int q = tid; q < nq; q += ATT_THREADS) {
          w_slot[s0 + q0 + q] = s_w[q];
          d_logits[slot_edge[s0 + q0 + q]] = attn_d_logit(s_w[q], s_dw[q], q0 + q == qs, s_S, s_Wo, s_To);
        }
      }
    }
    if (pass == 0) {
      __syncthreads();
      if (deg <= ATT_MAX_DEG) {                           // one pass over the neighbours is enough: s_w / s_dw are still valid
        for (int q = tid; q < deg; q += ATT_THREADS) {
          w_slot[s0 + q] = s_w[q];
          d_logits[slot_edge[s0 + q]] = attn_d_logit(s_w[q], s_dw[q], q == qs, s_S, s_Wo, s_To);
        }
        break;
      }
    }
  }
}

__global__ void __launch_bounds__(ATT_THREADS) attn_backward_node_kernel(
    int64_t feat, const int32_t* __restrict__ slot_row, int64_t num_out, const int32_t* __restrict__ perm_c,
    const int32_t* __restrict__ ptr_c, const float* __restrict__ w_slot, const float* __restrict__ g_in,
    const float* __restrict__ g_out, float* __restrict__ dz) {
  __shared__ float s_w[ATT_MAX_DEG];
  __shared__ const float* s_g[ATT_MAX_DEG];
  const int64_t c = blockIdx.x;
  const int q_begin = ptr_c[c], q_end = ptr_c[c + 1];
  float* out = dz + c * feat;
  const int tid = threadIdx.x;
  if (q_end == q_begin) {
    for (int64_t i = tid; i < feat; i += ATT_THREADS) out[i] = 0.f;
    return;
  }
  for (int q0 = q_begin; q0 < q_end; q0 += ATT_MAX_DEG) {
    const int nq = q_end - q0 < ATT_MAX_DEG ? q_end - q0 : ATT_MAX_DEG;
    __syncthreads();
    for (int q = tid; q < nq; q += ATT_THREADS) {
      const int32_t slot = perm_c[q0 + q];
      s_w[q] = w_slot[slot];
      s_g[q] = (slot < num_out ? g_out : g_in) + (int64_t)slot_row[slot] * feat;      // the flow this slot contributed to
    }
    __syncthreads();
    for (int64_t i = tid; i < feat; i += ATT_THREADS) {
      float acc = q0 == q_begin ? 0.f : out[i];
      for (int q = 0; q < nq; ++q) acc = fmaf(s_w[q], s_g[q][i], acc);
      out[i] = acc;
    }
  }
}

}  // namespace mpn

using namespace mpn;

extern "C" int mpn_attn_aggregate_backward(const float* z, int64_t num_nodes, int64_t feat, const mpn_edge_layout* g,
                                           const float* logits, const float* g_in, const float* g_out,
                                           const int32_t* perm_c, const int32_t* ptr_c, float* w_slot, float* d_z,
                                           float* d_logits, void* stream) {
  MPN_CHECK_ARG(g != nullptr && num_nodes == g->num_nodes, "attn_aggregate_backward: layout / node count mismatch");
  if (num_nodes == 0) return MPN_OK;
  MPN_CHECK_ARG(z && g_in && g_out && d_z && feat > 0, "attn_aggregate_backward: null pointer");
  MPN_CHECK_ARG(g->num_edges == 0 || (logits && perm_c && ptr_c && w_slot && d_logits), "attn_aggregate_backward: null edge arrays");
  MPN_CHECK_ARG(2 * num_nodes < (1ll << 31), "attn_aggregate_backward: too many nodes");
  cudaStream_t s = as_stream(stream);
  if (g->num_edges > 0) {
    attn_backward_edge_kernel<<<(unsigned)(2 * num_nodes), ATT_THREADS, 0, s>>>(z, feat, g->slot_col, g->slot_edge, g->out_ptr,
                                                                               g->in_ptr, logits, g_in, g_out, w_slot, d_logits);
    count_launch();
    attn_backward_node_kernel<<<(unsigned)num_nodes, ATT_THREADS, 0, s>>>(feat, g->slot_row, g->num_out, perm_c, ptr_c, w_slot,
                                                                         g_in, g_out, d_z);
    count_launch();
  } else {
    MPN_CUDA(cudaMemsetAsync(d_z, 0, sizeof(float) * num_nodes * feat, s));
  }
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

extern "C" int mpn_attn_aggregate(const float* z, int64_t num_nodes, int64_t feat, const mpn_edge_layout* g,
                                  const float* logits, float* flow_in, float* flow_out, void* stream) {
  MPN_CHECK_ARG(g != nullptr && num_nodes == g->num_nodes, "attn_aggregate: layout / node count mismatch");
  if (num_nodes == 0) return MPN_OK;
  MPN_CHECK_ARG(z && flow_in && flow_out && feat > 0, "attn_aggregate: null pointer");
  MPN_CHECK_ARG(logits != nullptr || g->num_edges == 0, "attn_aggregate: null logits");
  MPN_CHECK_ARG(2 * num_nodes < (1ll << 31), "attn_aggregate: too many nodes");
  attn_aggregate_kernel<<<(unsigned)(2 * num_nodes), ATT_THREADS, 0, as_stream(stream)>>>(
      z, feat, g->slot_col, g->slot_edge, g->out_ptr, g->in_ptr, logits, num_nodes, flow_in, flow_out);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}
