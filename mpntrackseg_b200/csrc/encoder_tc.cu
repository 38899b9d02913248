// Node encoder  x_init = ReLU(W1 ReLU(W0 x + b0) + b1)  (2048 -> 128 -> 32, models/mpn.py:355 with
// configs/tracking_cfg.yaml:146-148) on the tcgen05 tensor cores.
//
// One 128-node tile per group of 4 warps (thread = node row = TMEM lane), two groups per CTA.  The
// K = 2048 contraction is streamed in chunks of 64: each thread loads its row's 64 fp32 values,
// splits them into fp16 hi/lo (22 significant bits, same scheme as mp_step_tc.cu) and writes them to
// a double-buffered TMEM A operand; the matching 32 KB slice of the packed fp16 hi/lo weight image (the K stream of
// the B operand) is brought into shared memory by ONE TMA bulk copy per chunk (cp.async.bulk, completion counted in
// bytes on an mbarrier); 12 MMAs (128 x 128 x 16, hi*hi + hi*lo + lo*hi) per chunk
// accumulate in TMEM while the next chunk is being loaded.  The 128 -> 32 layer reuses the accumulator
// in place as its operand.
//
// Every operand row is split at its own power-of-two scale (pack_shift): each output row of W0 and W1 (pack_kernel)
// and each row of the hidden h (epilogue 1) with its largest |v| in [2^13, 2^14); each row of x with the largest |v|
// seen so far in [2^10, 2^11): the shift is set by the first nonzero chunk and lowered when a later chunk would pass
// 2^15, the row's accumulator then rescaled in TMEM by the same power of two (rare: a 16x jump within the row).
// Unscaled, the low half of a value below 2^-3 is subnormal and carries an absolute error of 2^-25, which the
// default weights (|w| ~ 0.02 .. 0.1) and small features already reach.  The epilogues multiply the accumulators
// by the inverse powers of two before adding the biases, so every scaling is exact, the error is relative to
// ||x_r|| ||w_o|| whatever the magnitudes, and out(x 2^p, b 2^p) = 2^p out(x, b) bit for bit (DESIGN.md section 4).
#include "common.cuh"
#include "tc_ptx.cuh"

namespace mpn {
namespace enc {

using namespace ptx;

constexpr int TS = 128, H = 128, O = 32, KC = 64;                    // tile rows, hidden, out, K per chunk
constexpr int NTHREADS = 256;
constexpr int SLAB1 = H * 32;                                         // one K=16 step of W0: 128 rows x 32 B
constexpr int CHUNK_BYTES = 2 * (KC / 16) * SLAB1;                    // hi + lo, 4 k-steps = 32 KB
constexpr int SLAB2 = O * 32;                                         // one K=16 step of W1: 32 rows x 32 B
constexpr int W2_BYTES = 2 * (H / 16) * SLAB2;                        // 16 KB
// tail floats: biases, then 2^-e of each output row of W0 and W1 (the row was packed times 2^e)
constexpr int F_B0 = 0, F_B1 = H, F_S0 = H + O, F_S1 = 2 * H + O, F_COUNT = 2 * (H + O);
constexpr int TAIL_BYTES = W2_BYTES + F_COUNT * 4;                    // W1 image + biases + row scales

constexpr int C_A = 0;            // A operand double buffer: [buf][hi 32 cols | lo 32 cols]
constexpr int C_D1 = 128;         // 128 accumulator columns, reused in place as the layer-2 operand
constexpr int C_D2 = 0;           // layer-2 accumulator (32 cols) over the dead A buffers

constexpr int SM_W = 0;                                               // [2 groups][2 bufs][CHUNK_BYTES]
constexpr int SM_TAIL = SM_W + 4 * CHUNK_BYTES;
constexpr int SM_BAR = (SM_TAIL + TAIL_BYTES + 127) / 128 * 128;      // u64 bars[2 groups][2] (MMA done), wbars[2 groups][2] (weights landed)
constexpr int SM_TMEM = SM_BAR + 8 * 8;
constexpr int SMEM_BYTES = SM_TMEM + 16;

// global image: [K0/64 chunks][hi: 4 slabs | lo: 4 slabs] then the tail (W1 hi slabs, lo slabs, b0, b1, row scales).
// One CTA per output row (W0 rows 0..127, then W1 rows 0..31): the row's largest |w| gives its shift e, the row is
// packed times 2^e and 2^-e goes to the tail.  A non-finite weight or bias sets status bit 1.
__global__ void __launch_bounds__(256) pack_kernel(const float* __restrict__ w0, const float* __restrict__ b0,
                                                   const float* __restrict__ w1, const float* __restrict__ b1, int64_t k0,
                                                   uint8_t* __restrict__ img, int32_t* __restrict__ status) {
  __shared__ float s_max[8];
  __shared__ int s_fin[8];
  const int tid = threadIdx.x, lane = tid & 31;
  const bool layer0 = blockIdx.x < H;
  const int n = layer0 ? (int)blockIdx.x : (int)blockIdx.x - H;
  const int64_t len = layer0 ? k0 : H;
  const float* w = layer0 ? w0 + (int64_t)n * k0 : w1 + (int64_t)n * H;
  float m = 0.f;
  bool fin = true;
  for (int64_t k = tid; k < len; k += 256) {
    const float a = fabsf(w[k]);
    m = fmaxf(m, a);
    fin &= a <= 3.402823466e38f;                                     // false for inf and NaN
  }
  for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
  fin = __all_sync(0xffffffffu, fin);
  if (lane == 0) { s_max[tid >> 5] = m; s_fin[tid >> 5] = fin; }
  __syncthreads();
  for (int i = 0; i < 8; ++i) { m = fmaxf(m, s_max[i]); fin &= s_fin[i] != 0; }
  const float bias = layer0 ? b0[n] : b1[n];
  if (tid == 0 && !(fin && fabsf(bias) <= 3.402823466e38f)) atomicOr(status, 1);
  const int e = pack_shift(__float_as_uint(m));
  const float up = pow2i(e);
  uint8_t* tail = img + (k0 / KC) * CHUNK_BYTES;
  for (int64_t k = tid; k < len; k += 256) {
    const float v = w[k] * up;
    const __half h = __float2half_rn(v), l = __float2half_rn(v - __half2float(h));
    const int64_t off = layer0 ? (k / KC) * CHUNK_BYTES + ((k % KC) >> 4) * SLAB1 + slab_off(n, (int)(k & 15))
                               : (k >> 4) * SLAB2 + slab_off(n, (int)(k & 15));
    uint8_t* dst = layer0 ? img + off : tail + off;
    *reinterpret_cast<__half*>(dst) = h;
    *reinterpret_cast<__half*>(dst + (layer0 ? (KC / 16) * SLAB1 : (H / 16) * SLAB2)) = l;
  }
  if (tid == 0) {
    float* ft = reinterpret_cast<float*>(tail + W2_BYTES);
    ft[(layer0 ? F_B0 : F_B1) + n] = bias;
    ft[(layer0 ? F_S0 : F_S1) + n] = pow2i(-e);
  }
}

constexpr int X_HEADROOM = 3;            // x rows are packed with their largest |v| so far in [2^10, 2^11) ...
constexpr float X_RESCALE_AT = 32768.f;  // ... until a chunk would reach 2^15

__global__ void __launch_bounds__(NTHREADS, 1) node_encoder_tc_kernel(const float* __restrict__ x, int64_t n, int64_t k0,
                                                                     const uint8_t* __restrict__ img,
                                                                     float* __restrict__ out,
                                                                     int32_t* __restrict__ status) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  const int g = warp >> 2, wq = warp & 3, gt = tid & (TS - 1);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR) + 2 * g;   // [0]/[1]: even / odd chunks
  uint64_t* wbars = reinterpret_cast<uint64_t*>(smem + SM_BAR) + 4 + 2 * g;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM_TMEM);
  const int nchunks = (int)(k0 / KC);
  const uint8_t* tail_g = img + (int64_t)nchunks * CHUNK_BYTES;
  for (int i = tid; i < TAIL_BYTES / 16; i += NTHREADS)
    reinterpret_cast<uint4*>(smem + SM_TAIL)[i] = __ldg(reinterpret_cast<const uint4*>(tail_g) + i);
  if (tid == 0) {
    for (int i = 0; i < 8; ++i) mbar_init(reinterpret_cast<uint64_t*>(smem + SM_BAR) + i, 1);
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<512>(tmem_slot);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tcol = __shfl_sync(0xffffffffu, *tmem_slot, 0) + (uint32_t)g * 256u;
  const uint32_t tlane = tcol + ((uint32_t)(wq * 32) << 16);
  const float* s_f = reinterpret_cast<const float*>(smem + SM_TAIL + W2_BYTES);
  const uint32_t wbuf = smem_u32(smem + SM_W + g * 2 * CHUNK_BYTES);
  const uint64_t dbase = smem_desc_kmajor(0, 128, 256);
  __half2 vmax = __floats2half2_rn(0.f, 0.f);
  uint32_t par[2] = {0, 0}, wpar[2] = {0, 0};

  const int64_t tiles = (n + TS - 1) / TS;
  for (int64_t t = (int64_t)blockIdx.x * 2 + g; t < tiles; t += (int64_t)gridDim.x * 2) {
    int64_t row = t * TS + gt;
    const bool valid = row < n;
    if (!valid) row = n - 1;
    int sx = 0;                                                      // the row's shift so far
    float xmax = 0.f;                                                // its largest |x| so far
    bool early = false;                                              // MMAs of chunk c-1 already waited for
    const float4* xr = reinterpret_cast<const float4*>(x + row * k0);
    auto load_w = [&](int c) {                                       // 32 KB weight chunk: one TMA bulk copy
      if (gt == 0) {
        mbar_arrive_expect_tx(&wbars[c & 1], CHUNK_BYTES);
        tma_bulk_g2s(wbuf + (c & 1) * CHUNK_BYTES, img + (int64_t)c * CHUNK_BYTES, CHUNK_BYTES, &wbars[c & 1]);
      }
    };
    float4 xv[KC / 4];
    load_w(0);
#pragma unroll
    for (int j = 0; j < KC / 4; ++j) xv[j] = __ldcs(xr + j);
    for (int c = 0; c < nchunks; ++c) {
      // ---- this chunk's A operand: split the 64 values and store them to TMEM buffer c&1
      const uint32_t abuf = tlane + C_A + (c & 1) * 64;
      float cmax = 0.f;
#pragma unroll
      for (int j = 0; j < KC / 4; ++j)
        cmax = fmaxf(cmax, fmaxf(fmaxf(fabsf(xv[j].x), fabsf(xv[j].y)), fmaxf(fabsf(xv[j].z), fabsf(xv[j].w))));
      // the first nonzero chunk sets the shift (the accumulator is still exactly 0); a chunk that would pass 2^15
      // lowers it, and the accumulator of the chunks before is rescaled to match
      const bool first = !(xmax > 0.f) && cmax > 0.f;
      const bool rescale = xmax > 0.f && cmax * pow2i(sx) >= X_RESCALE_AT;
      const int snew = first || rescale ? pack_shift(__float_as_uint(cmax)) - X_HEADROOM : sx;
      const float fix = pow2i(snew - sx);
      sx = snew;
      xmax = fmaxf(xmax, cmax);
      const float up = pow2i(sx);
#pragma unroll
      for (int q = 0; q < KC / 16; ++q) {
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 v = xv[4 * q + j];
          split2(v.x * up, v.y * up, hi[2 * j], lo[2 * j]);
          split2(v.z * up, v.w * up, hi[2 * j + 1], lo[2 * j + 1]);
          vmax = __hmax2_nan(vmax, __habs2(*reinterpret_cast<const __half2*>(&hi[2 * j])));
          vmax = __hmax2_nan(vmax, __habs2(*reinterpret_cast<const __half2*>(&hi[2 * j + 1])));
        }
        tmem_st8(abuf + 8 * q, hi);
        tmem_st8(abuf + 32 + 8 * q, lo);
      }
      mbar_wait(&wbars[c & 1], wpar[c & 1]); wpar[c & 1] ^= 1;       // this chunk's weights have landed
      tc_wait_st();
      tc_fence_before();
      early = named_barrier_or(1 + g, TS, rescale);                   // never at c = 0: no accumulator yet
      if (early) {                                                     // wait for chunk c-1, rescale the rows that ask
        mbar_wait(&bars[(c - 1) & 1], par[(c - 1) & 1]); par[(c - 1) & 1] ^= 1;
        tc_fence_after();
        const float f = rescale ? fix : 1.f;
#pragma unroll 1
        for (int ch = 0; ch < H / 16; ++ch) {
          uint32_t acc[16], a[8], b[8];
          tmem_ld16(tlane + C_D1 + 16 * ch, acc);
          tc_wait_ld();
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            a[j] = __float_as_uint(__uint_as_float(acc[j]) * f);
            b[j] = __float_as_uint(__uint_as_float(acc[j + 8]) * f);
          }
          tmem_st8(tlane + C_D1 + 16 * ch, a);
          tmem_st8(tlane + C_D1 + 16 * ch + 8, b);
        }
        tc_wait_st();
        tc_fence_before();
        named_barrier(1 + g, TS);
      }
      if (wq == 0) {
        tc_fence_after();
        if (elect_one()) {
          const uint32_t wb = wbuf + (c & 1) * CHUNK_BYTES;
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks) {
            const uint64_t dh = dbase + (uint64_t)((wb + ks * SLAB1) >> 4);
            const uint64_t dl = dbase + (uint64_t)((wb + (KC / 16 + ks) * SLAB1) >> 4);
            const uint32_t ah = tcol + C_A + (c & 1) * 64 + 8 * ks, al = ah + 32;
            mma_ts(tcol + C_D1, ah, dh, idesc_f16(128, H), (c > 0 || ks > 0) ? 1u : 0u);
            mma_ts(tcol + C_D1, ah, dl, idesc_f16(128, H), 1u);
            mma_ts(tcol + C_D1, al, dh, idesc_f16(128, H), 1u);
          }
          mma_commit(&bars[c & 1]);
        }
        __syncwarp();
      }
      // ---- next chunk: its buffers were last read by the MMAs of chunk c-1
      if (c + 1 < nchunks) {
        if (c >= 1 && !early) { mbar_wait(&bars[(c - 1) & 1], par[(c - 1) & 1]); par[(c - 1) & 1] ^= 1; }
        load_w(c + 1);
#pragma unroll
        for (int j = 0; j < KC / 4; ++j) xv[j] = __ldcs(xr + (c + 1) * (KC / 4) + j);
      }
    }
    // drain: the last two commits
    if (nchunks >= 2 && !early) { mbar_wait(&bars[(nchunks - 2) & 1], par[(nchunks - 2) & 1]); par[(nchunks - 2) & 1] ^= 1; }
    mbar_wait(&bars[(nchunks - 1) & 1], par[(nchunks - 1) & 1]); par[(nchunks - 1) & 1] ^= 1;
    tc_fence_after();
    // ---- epilogue 1: h = ReLU(D1 * 2^-(sx + e_o) + b0) -> layer-2 operand in place, split at the row's own shift.
    // Sweep 1 finds the row's largest h, sweep 2 recomputes the same values, scales them by 2^sh and splits them.
    const float down = pow2i(-sx);
    float hmax = 0.f;
#pragma unroll 1
    for (int ch = 0; ch < H / 16; ++ch) {
      uint32_t acc[16];
      tmem_ld16(tlane + C_D1 + 16 * ch, acc);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 16; ++j)
        hmax = fmaxf(hmax, fmaf(__uint_as_float(acc[j]), down * s_f[F_S0 + 16 * ch + j], s_f[F_B0 + 16 * ch + j]));
    }
    const int sh = pack_shift(__float_as_uint(hmax));
    const float hup = pow2i(sh), hdown = pow2i(-sh);
#pragma unroll
    for (int ch = 0; ch < H / 16; ++ch) {
      uint32_t acc[16];
      tmem_ld16(tlane + C_D1 + 16 * ch, acc);
      tc_wait_ld();
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int o = 16 * ch + 2 * j;
        split2_relu(fmaf(__uint_as_float(acc[2 * j]), down * s_f[F_S0 + o], s_f[F_B0 + o]) * hup,
                    fmaf(__uint_as_float(acc[2 * j + 1]), down * s_f[F_S0 + o + 1], s_f[F_B0 + o + 1]) * hup, hi[j], lo[j]);
        vmax = __hmax2_nan(vmax, *reinterpret_cast<const __half2*>(&hi[j]));
      }
      tmem_st8(tlane + C_D1 + 16 * ch, hi);
      tmem_st8(tlane + C_D1 + 16 * ch + 8, lo);
    }
    tc_wait_st();
    tc_fence_before();
    named_barrier(1 + g, TS);
    if (wq == 0) {
      tc_fence_after();
      if (elect_one()) {
        const uint32_t w2 = smem_u32(smem + SM_TAIL);
#pragma unroll
        for (int ks = 0; ks < H / 16; ++ks) {
          const uint64_t dh = dbase + (uint64_t)((w2 + ks * SLAB2) >> 4);
          const uint64_t dl = dbase + (uint64_t)((w2 + (H / 16 + ks) * SLAB2) >> 4);
          const uint32_t ah = tcol + C_D1 + 16 * ks, al = ah + 8;
          mma_ts(tcol + C_D2, ah, dh, idesc_f16(128, O), ks > 0 ? 1u : 0u);
          mma_ts(tcol + C_D2, ah, dl, idesc_f16(128, O), 1u);
          mma_ts(tcol + C_D2, al, dh, idesc_f16(128, O), 1u);
        }
        mma_commit(&bars[0]);
      }
      __syncwarp();
    }
    mbar_wait(&bars[0], par[0]); par[0] ^= 1;
    tc_fence_after();
    // ---- epilogue 2: x_init = ReLU(D2 * 2^-(sh + e_o) + b1)
#pragma unroll
    for (int ch = 0; ch < O / 16; ++ch) {
      uint32_t acc[16];
      tmem_ld16(tlane + C_D2 + 16 * ch, acc);
      tc_wait_ld();
      if (valid) {
        float4* dst = reinterpret_cast<float4*>(out + (t * TS + gt) * O + 16 * ch);
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j)
          v[j] = fmaxf(fmaf(__uint_as_float(acc[j]), hdown * s_f[F_S1 + 16 * ch + j], s_f[F_B1 + 16 * ch + j]), 0.f);
#pragma unroll
        for (int j = 0; j < 4; ++j) dst[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
      }
    }
    tc_fence_before();
    named_barrier(1 + g, TS);                                        // D2 / A buffers are free for the next tile
  }
  {
    // scaled operands stay below 2^15 and the max keeps NaN: only a non-finite x (or a row beyond the shift's reach,
    // |v| >= 2^73) gets here
    const uint32_t w = *reinterpret_cast<const uint32_t*>(&vmax);
    if ((w & 0x7FFFu) >= 0x7BFFu || ((w >> 16) & 0x7FFFu) >= 0x7BFFu) atomicOr(status, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(*tmem_slot);
}

}  // namespace enc
}  // namespace mpn

using namespace mpn;

extern "C" {

int64_t mpn_node_encoder_tc_workspace(int64_t k0) { return (k0 / enc::KC) * enc::CHUNK_BYTES + enc::TAIL_BYTES + 512; }

int mpn_node_encoder_tc(const float* x, int64_t n, int64_t k0, const float* w0, const float* b0, int64_t hidden,
                        const float* w1, const float* b1, int64_t out_dim, void* ws, float* out, int32_t* status,
                        void* stream) {
  MPN_CHECK_ARG(hidden == enc::H && out_dim == enc::O && k0 >= enc::KC && k0 % enc::KC == 0,
                "node_encoder_tc: built for K -> 128 -> 32 with K a multiple of 64 (got %lld -> %lld -> %lld)",
                (long long)k0, (long long)hidden, (long long)out_dim);
  MPN_CHECK_ARG(ws && status, "node_encoder_tc: null workspace / status");
  cudaStream_t s = as_stream(stream);
  MPN_CUDA(cudaMemsetAsync(status, 0, 4, s));
  if (n == 0) return MPN_OK;
  MPN_CHECK_ARG(x && w0 && b0 && w1 && b1 && out, "node_encoder_tc: null pointer");
  MPN_CHECK_ARG(reinterpret_cast<uintptr_t>(x) % 16 == 0, "node_encoder_tc: x must be 16-byte aligned");
  uint8_t* img = static_cast<uint8_t*>(ws);
  MPN_CUDA(cudaFuncSetAttribute(enc::node_encoder_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                enc::SMEM_BYTES));
  enc::pack_kernel<<<enc::H + enc::O, 256, 0, s>>>(w0, b0, w1, b1, k0, img, status); count_launch();
  const int64_t tiles = ceil_div(n, enc::TS);
  int grid = (int)std::min<int64_t>(ceil_div(tiles, 2), sm_count());
  enc::node_encoder_tc_kernel<<<grid, enc::NTHREADS, enc::SMEM_BYTES, s>>>(x, n, k0, img, out, status); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // extern "C"
