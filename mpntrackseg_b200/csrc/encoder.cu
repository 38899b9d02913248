// Encoders: global average pool, generic Linear(+ReLU) layer (fp32 SIMT tiled GEMM),
// row gather, and the fused edge-feature MLP in slot order.
#include <algorithm>

#include "common.cuh"
#include "mlp_regs.cuh"

namespace mpn {

constexpr unsigned kFull = 0xffffffffu;

// ------------------------------------------------------------------ average pool
// x[n*c][hw] -> out[n*c] for any number of windows in one launch.  GROUP = hw/4 lanes cooperate on one channel
// (float4 each).  The windows' rows are cut into chunks of POOL_UNROLL * 32 float4 (2 KB: every load of a warp
// covers 512 contiguous bytes); the chunks of all windows form one list, and each block takes the next
// POOL_BLOCK_CHUNKS of it.  POOL_UNROLL independent 16-byte loads per thread are issued before any of them is
// consumed: the kernel is a pure HBM stream and needs the bytes in flight.
// The blocks are short (128 KB of maps, some 10-20 us at the HBM rate per SM): the pool runs on its own stream
// beside the window-graph build, whose kernels have the higher stream priority, so a build kernel waits for the pool
// blocks on an SM to end, never for the whole pool.
constexpr int POOL_THREADS = 256, POOL_UNROLL = 4, POOL_BLOCK_CHUNKS = 64, POOL_MAX_WINDOWS = 64;

struct PoolWindow {
  const float4* x;          // the window's maps, 16-byte aligned
  int64_t rows;             // n * c
  int64_t out_row;          // first output element of the window
  int32_t chunk_end;        // one past the window's last chunk in the launch's chunk list
};
struct PoolTable {          // passed by value: the table lives in the kernel's parameter space, no copy to the device
  PoolWindow w[POOL_MAX_WINDOWS];
  int count;
};

template <int GROUP>
__global__ void __launch_bounds__(POOL_THREADS) avgpool_kernel(const __grid_constant__ PoolTable t, int hw,
                                                               float* __restrict__ out) {
  constexpr int ROWS_PER_WARP = 32 / GROUP, CHUNK_ROWS = ROWS_PER_WARP * POOL_UNROLL;
  const int lane = threadIdx.x & 31;
  const int chunks = t.w[t.count - 1].chunk_end;
  const int end = min(chunks, (int)(blockIdx.x + 1) * POOL_BLOCK_CHUNKS);
  int w = 0, first = 0;                                 // window of chunk ch and its first chunk
  for (int ch = blockIdx.x * POOL_BLOCK_CHUNKS + (threadIdx.x >> 5); ch < end; ch += POOL_THREADS / 32) {
    while (ch >= t.w[w].chunk_end) first = t.w[w++].chunk_end;
    const int64_t r0 = (int64_t)(ch - first) * CHUNK_ROWS;
    const int valid = (int)min((int64_t)CHUNK_ROWS, t.w[w].rows - r0);    // rows of this chunk
    const float4* src = t.w[w].x + r0 * GROUP + lane;
    float4 v[POOL_UNROLL];
#pragma unroll
    for (int u = 0; u < POOL_UNROLL; ++u)
      v[u] = valid == CHUNK_ROWS || u * ROWS_PER_WARP + lane / GROUP < valid ? __ldcs(src + u * 32)  // streaming
                                                                            : make_float4(0.f, 0.f, 0.f, 0.f);
    float* dst = out + t.w[w].out_row + r0 + lane / GROUP;
#pragma unroll
    for (int u = 0; u < POOL_UNROLL; ++u) {
      float s = (v[u].x + v[u].y) + (v[u].z + v[u].w);
#pragma unroll
      for (int d = GROUP / 2; d > 0; d >>= 1) s += __shfl_xor_sync(kFull, s, d);
      if ((lane % GROUP) == 0 && u * ROWS_PER_WARP + lane / GROUP < valid) dst[u * ROWS_PER_WARP] = s / (float)hw;
    }
  }
}

__global__ void avgpool_scalar_kernel(const float* __restrict__ x, int64_t rows, int hw,
                                      float* __restrict__ out) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows;
       r += (int64_t)gridDim.x * blockDim.x) {
    const float* p = x + r * hw;
    float s = 0.f;
    for (int i = 0; i < hw; ++i) s += p[i];
    out[r] = s / (float)hw;
  }
}

// ------------------------------------------------------------------ generic linear
// out[m][o] = act(sum_k in[m][k] * w[o][k] + b[o]);  64x64 tile, 16-deep k slab, 4x4 per thread.
constexpr int LT = 64, LK = 16;
__global__ void __launch_bounds__(256) linear_kernel(const float* __restrict__ in, int64_t m, int64_t k,
                                                     const float* __restrict__ w,
                                                     const float* __restrict__ b, int64_t o, int relu,
                                                     float* __restrict__ out) {
  __shared__ float As[LK][LT + 4];
  __shared__ float Bs[LK][LT + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t m0 = (int64_t)blockIdx.y * LT, o0 = (int64_t)blockIdx.x * LT;
  float acc[4][4] = {};
  for (int64_t k0 = 0; k0 < k; k0 += LK) {
    for (int idx = threadIdx.x; idx < LT * LK; idx += 256) {
      const int r = idx / LK, kk = idx % LK;
      const int64_t gm = m0 + r, go = o0 + r, gk = k0 + kk;
      As[kk][r] = (gm < m && gk < k) ? in[gm * k + gk] : 0.f;
      Bs[kk][r] = (go < o && gk < k) ? w[go * k + gk] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < LK; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bb = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t gm = m0 + ty * 4 + i;
    if (gm >= m) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t go = o0 + tx * 4 + j;
      if (go >= o) continue;
      float v = acc[i][j] + (b != nullptr ? b[go] : 0.f);
      out[gm * o + go] = relu ? fmaxf(v, 0.f) : v;
    }
  }
}

// ------------------------------------------------------------------ fused edge encoder
template <int D0, int D1, int D2, int D3>
__global__ void __launch_bounds__(256) edge_encoder_kernel(
    const float* __restrict__ attr, const int32_t* __restrict__ slot_edge, int64_t e,
    const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w1,
    const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
    float* __restrict__ e_init) {
  constexpr int P1 = Pad4<D1>::value, P2 = Pad4<D2>::value, P3 = Pad4<D3>::value;
  static_assert(D3 % 4 == 0, "edge latent width must be a multiple of 4");
  __shared__ __align__(16) float s_w0[D0 * P1], s_w1[D1 * P2], s_w2[D2 * P3];
  __shared__ __align__(16) float s_b0[P1], s_b1[P2], s_b2[P3];
  stage_weight_t<D0, D1>(w0, s_w0);
  stage_weight_t<D1, D2>(w1, s_w1);
  stage_weight_t<D2, D3>(w2, s_w2);
  stage_bias<D1>(b0, s_b0);
  stage_bias<D2>(b1, s_b1);
  stage_bias<D3>(b2, s_b2);
  __syncthreads();
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < e;
       s += (int64_t)gridDim.x * blockDim.x) {
    const float* a = attr + (int64_t)(slot_edge != nullptr ? slot_edge[s] : s) * D0;
    float in[D0];
#pragma unroll
    for (int i = 0; i < D0; ++i) in[i] = a[i];
    float h1[P1], h2[P2], h3[P3];
    load_bias<P1>(h1, s_b0);
    dense_acc<D0, P1>(h1, in, s_w0);
    relu_inplace(h1);
    load_bias<P2>(h2, s_b1);
    dense_acc<D1, P2>(h2, h1, s_w1);
    relu_inplace(h2);
    load_bias<P3>(h3, s_b2);
    dense_acc<D2, P3>(h3, h2, s_w2);
    relu_inplace(h3);
    float4* dst = reinterpret_cast<float4*>(e_init + s * D3);
#pragma unroll
    for (int q = 0; q < D3 / 4; ++q) dst[q] = make_float4(h3[4 * q], h3[4 * q + 1], h3[4 * q + 2], h3[4 * q + 3]);
  }
}

__global__ void gather_rows_kernel(const float* __restrict__ in, const int32_t* __restrict__ idx,
                                   int64_t rows, int64_t width, float* __restrict__ out) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < rows * width;
       t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / width, c = t - r * width;
    out[t] = in[(int64_t)idx[r] * width + c];
  }
}

template <int GROUP>
static int launch_avgpool(const PoolTable& t, int64_t hw, float* out, cudaStream_t s) {
  const unsigned grid = (unsigned)ceil_div(t.w[t.count - 1].chunk_end, POOL_BLOCK_CHUNKS);
  avgpool_kernel<GROUP><<<grid, POOL_THREADS, 0, s>>>(t, (int)hw, out); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

static inline unsigned grid_for(int64_t n, int threads, int per_sm = 8) {
  int64_t want = ceil_div(n > 0 ? n : 1, threads);
  int64_t cap = (int64_t)sm_count() * per_sm;
  return (unsigned)(want < cap ? want : cap);
}

}  // namespace mpn

using namespace mpn;

extern "C" {

int mpn_avgpool(const float* const* x, const int64_t* n, int64_t windows, int64_t c, int64_t hw, float* out,
                void* stream) {
  MPN_CHECK_ARG(windows >= 0 && c > 0 && hw > 0 && (windows == 0 || (x && n)), "avgpool: bad sizes");
  cudaStream_t s = as_stream(stream);
  const int64_t vec = hw / 4;
  const bool vec_hw = (hw % 4 == 0) && vec >= 1 && vec <= 32 && (vec & (vec - 1)) == 0;
  const int64_t chunk_rows = POOL_UNROLL * (32 / std::max<int64_t>(vec, 1));
  PoolTable t;
  t.count = 0;
  int64_t out_row = 0;
  // one launch per POOL_MAX_WINDOWS vector-path windows; a window off 16-byte alignment takes the scalar kernel
  auto flush = [&]() -> int {
    if (t.count == 0) return MPN_OK;
    int rc = MPN_OK;
    switch (vec) {
      case 1: rc = launch_avgpool<1>(t, hw, out, s); break;
      case 2: rc = launch_avgpool<2>(t, hw, out, s); break;
      case 4: rc = launch_avgpool<4>(t, hw, out, s); break;
      case 8: rc = launch_avgpool<8>(t, hw, out, s); break;
      case 16: rc = launch_avgpool<16>(t, hw, out, s); break;
      default: rc = launch_avgpool<32>(t, hw, out, s); break;
    }
    t.count = 0;
    return rc;
  };
  for (int64_t i = 0; i < windows; ++i) {
    MPN_CHECK_ARG(n[i] >= 0, "avgpool: window %lld has %lld rows", (long long)i, (long long)n[i]);
    const int64_t rows = n[i] * c;
    if (rows == 0) continue;
    MPN_CHECK_ARG(x[i] && out, "avgpool: null pointer");
    if (vec_hw && reinterpret_cast<uintptr_t>(x[i]) % 16 == 0) {
      const int64_t prev = t.count ? t.w[t.count - 1].chunk_end : 0;
      MPN_CHECK_ARG(prev + ceil_div(rows, chunk_rows) < INT32_MAX - POOL_BLOCK_CHUNKS, "avgpool: more than 2^31 chunks in one launch");
      t.w[t.count++] = PoolWindow{reinterpret_cast<const float4*>(x[i]), rows, out_row,
                                   (int32_t)(prev + ceil_div(rows, chunk_rows))};
      if (t.count == POOL_MAX_WINDOWS) {
        const int rc = flush();
        if (rc != MPN_OK) return rc;
      }
    } else {
      avgpool_scalar_kernel<<<grid_for(rows, 256), 256, 0, s>>>(x[i], rows, (int)hw, out + out_row); count_launch();
      MPN_LAUNCH_CHECK();
    }
    out_row += rows;
  }
  return flush();
}

int mpn_linear(const float* in, int64_t m, int64_t k, const float* w, const float* b, int64_t o,
               int relu, float* out, void* stream) {
  MPN_CHECK_ARG(m >= 0 && k > 0 && o > 0, "linear: bad sizes");
  if (m == 0) return MPN_OK;
  MPN_CHECK_ARG(in && w && out, "linear: null pointer");
  dim3 grid((unsigned)ceil_div(o, LT), (unsigned)ceil_div(m, LT));
  MPN_CHECK_ARG(grid.y <= 65535u, "linear: at most %d rows per call (gridDim.y limit)", 65535 * LT);
  linear_kernel<<<grid, 256, 0, as_stream(stream)>>>(in, m, k, w, b, o, relu, out); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_gather_rows(const float* in, const int32_t* idx, int64_t rows, int64_t width, float* out,
                    void* stream) {
  if (rows == 0) return MPN_OK;
  MPN_CHECK_ARG(in && idx && out && width > 0, "gather_rows: bad args");
  gather_rows_kernel<<<grid_for(rows * width, 256), 256, 0, as_stream(stream)>>>(in, idx, rows, width, out); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_edge_encoder(const float* edge_attr, const int32_t* slot_edge, int64_t e, const int32_t* dims,
                     int32_t n_layers, const float* const* w, const float* const* b, float* e_init,
                     void* stream) {
  MPN_CHECK_ARG(e >= 0 && dims && w && b, "edge_encoder: bad args");
  const bool shipped = n_layers == 3 && dims[0] == 6 && dims[1] == 18 && dims[2] == 18 && dims[3] == 16;
  MPN_CHECK_ARG(shipped, "edge_encoder: fused kernel is built for widths 6-18-18-16 "
                         "(configs/tracking_cfg.yaml:141-144); use mpn_gather_rows + mpn_linear for others");
  if (e == 0) return MPN_OK;
  MPN_CHECK_ARG(edge_attr && e_init, "edge_encoder: null pointer");
  edge_encoder_kernel<6, 18, 18, 16><<<grid_for(e, 256, 4), 256, 0, as_stream(stream)>>>(
      edge_attr, slot_edge, e, w[0], b[0], w[1], b[1], w[2], b[2], e_init); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // extern "C"
