// ReID distance blocks on the tcgen05 tensor cores (north-star item (a)):
//   d(i,j)^2 = ||a||^2 + ||b||^2 - 2 a.b + 2 eps (sum a - sum b) + K eps^2 ,   a.b from a split-fp16 Gram MMA
// (hi*hi + hi*lo + lo*hi, fp32 accumulation).  The Gram distances are APPROXIMATE (~1e-6 relative), so they
// only pre-rank: every row whose k-th / (k+1)-th neighbour are closer than an error band is recomputed with
// the exact fp32 formula of the reference (same kernel arithmetic as knn_graph.cu) and re-ranked, and the
// distances attached to the kept pairs are always recomputed exactly.  The kept edge set is therefore the
// one the exact path produces.
// The band, beta * (||a_i||^2 + max_window ||a||^2 + K eps^2), is relative to the window's largest ||a||^2.
// The split's error is relative too only while the values sit high in the fp16 range: below 2^-3 the low half
// is subnormal and its error an absolute 2^-25.  So every window is packed times 2^p, p chosen from its largest
// |v| (pack_shift), and the Gram result is multiplied by 2^-2p, both exact (DESIGN.md section 4).
#include <limits.h>
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "knn_select.cuh"
#include "tc_ptx.cuh"

namespace mpn {
namespace gram {

using namespace ptx;

constexpr int TS = 128, KC = 64;
constexpr int SLAB = TS * 32;                               // one K=16 step of a 128-row B tile
constexpr int CHUNK_BYTES = 2 * (KC / 16) * SLAB;           // hi + lo: 32 KB

// warp per node: max |v| of its row into its window's entry (non-negative floats order like their bits).
__global__ void window_absmax_kernel(const float* __restrict__ reid, int64_t dim, const int64_t* __restrict__ gptr,
                                     int64_t num_graphs, int64_t num_nodes, uint32_t* __restrict__ win_amax) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp; i < num_nodes; i += nwarps) {
    const int64_t g = window_of(gptr, num_graphs, i);
    float m = 0.f;
    for (int64_t k = lane; k < dim; k += 32) m = fmaxf(m, fabsf(reid[i * dim + k]));
    for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
    if (lane == 0) atomicMax(&win_amax[g], __float_as_uint(m));
  }
}

// warp per node: packed fp16 hi/lo image of its row (times 2^p of its window) inside its 128-row tile, ||a||^2 and
// sum(a) (unscaled).
__global__ void pack_reid_kernel(const float* __restrict__ reid, int64_t dim, const int64_t* __restrict__ gptr,
                                 int64_t num_graphs, const int64_t* __restrict__ tile_off, int64_t num_nodes,
                                 const uint32_t* __restrict__ win_amax, uint8_t* __restrict__ img,
                                 float* __restrict__ norm2, float* __restrict__ sum1, int32_t* __restrict__ status) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int nchunks = (int)(dim / KC);
  for (int64_t i = warp; i < num_nodes; i += nwarps) {
    const int64_t g = window_of(gptr, num_graphs, i);
    const int64_t li = i - gptr[g];
    const int64_t tile = tile_off[g] + li / TS;
    const int n = (int)(li % TS);
    const float up = ldexpf(1.f, pack_shift(win_amax[g]));
    float s2 = 0.f, s1 = 0.f;
    bool ovf = false;
    for (int64_t k = lane; k < dim; k += 32) {
      const float v = reid[i * dim + k];
      ovf |= !(fabsf(v) < 65000.f);                              // outside the build's range (or NaN): the caller reruns exactly
      s2 = fmaf(v, v, s2);
      s1 += v;
      const float vs = v * up;
      const __half h = __float2half_rn(vs), l = __float2half_rn(vs - __half2float(h));
      uint8_t* base = img + (tile * nchunks + k / KC) * CHUNK_BYTES + ((k % KC) >> 4) * SLAB + slab_off(n, (int)(k & 15));
      *reinterpret_cast<__half*>(base) = h;
      *reinterpret_cast<__half*>(base + (KC / 16) * SLAB) = l;
    }
    for (int d = 16; d > 0; d >>= 1) { s2 += __shfl_xor_sync(0xffffffffu, s2, d); s1 += __shfl_xor_sync(0xffffffffu, s1, d); }
    if (lane == 0) { norm2[i] = s2; sum1[i] = s1; }
    if (ovf) atomicOr(status, 1);
  }
}

__global__ void tile_offsets_kernel(const int64_t* __restrict__ gptr, int64_t num_graphs, int64_t* __restrict__ tile_off,
                                    int64_t* __restrict__ tri_off, int mode) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int64_t acc = 0, tri = 0;
    for (int64_t g = 0; g < num_graphs; ++g) {
      const int64_t nt = (gptr[g + 1] - gptr[g] + TS - 1) / TS;
      tile_off[g] = acc; acc += nt;
      // tiles the Gram kernel walks per window: 0 = all nt x nt, 1 = nt x 2 sample column tiles, 2 = upper triangle
      tri_off[g] = tri; tri += mode == 0 ? nt * nt : (mode == 1 ? nt * 2 : nt * (nt + 1) / 2);
    }
    tile_off[num_graphs] = acc;
    tri_off[num_graphs] = tri;
  }
}

// ------------------------------------------------------------------ TMA-fed, warp-specialised Gram kernel
// Persistent CTA per SM over the flattened list of ALL 128x128 tiles of all windows (both triangles: every element
// is stored transposed, D[col][row], so that a warp's 32 rows write 32 consecutive floats -- storing the direct
// element as well would be a 32-sector scatter per instruction and was the bottleneck).  The packed
// fp16 hi/lo image of a 128-row tile serves as BOTH operands (the Gram matrix is symmetric), so nothing is split
// or staged by threads: warp 16 streams 32 KB operand chunks with TMA bulk copies into a 3-stage ring, warp 17
// issues the SS-mode MMAs (3 per K step) into one of two TMEM accumulators, warps 0-15 turn the previous
// accumulator into distances (each warp: its TMEM lane quarter x a 32-column group) and store them.
constexpr int G2_STAGES = 3, G2_EPI_WARPS = 16, G2_THREADS = 32 * (G2_EPI_WARPS + 2);
constexpr int G2_SM_BAR = G2_STAGES * 2 * CHUNK_BYTES;      // full[3], empty[3], acc_full[2], acc_empty[2]
constexpr int G2_SM_TMEM = G2_SM_BAR + 10 * 8;
constexpr int G2_SMEM_BYTES = G2_SM_TMEM + 16;

// Thresholded mode (windows of >= 8 tiles): the N^2 distances are never written.
//   MODE 1  sample pass: the two column tiles nt/4 and 3nt/4 of every row tile -> sample[N][256] (d^2, +inf where the
//           pair is not time-valid); a per-row threshold tau = an order statistic of the sample (row_threshold_kernel).
//   MODE 2  main pass over the UPPER-TRIANGULAR tiles: an entry (i, j) with d^2 <= tau_i is appended to row i's candidate
//           list, with d^2 <= tau_j to row j's (one value serves both rows, so both see the same bits).
// cand_select_kernel then ranks a row's ~100-300 candidates exactly like the dense row select would.
constexpr int SAMPLE_COLS = 2 * TS, CAND_CAP = 512, TG_MIN_TILES = 8, TG_DEFAULT_MAX_K = 64;

struct Gram2Args {
  const int64_t* frame; const int64_t* gptr; const int64_t* doff; const int64_t* tile_off; const int64_t* tri_off;
  const uint8_t* img; const float* norm2; const float* sum1;
  const uint32_t* win_amax; // [G] largest |v| of each window: the image is packed times 2^pack_shift
  int64_t num_graphs, max_dist, dim; float* dense;  // MODE 0: [sum N_g^2] approximate d^2 (+inf where not time-valid)
  float* sample;            // MODE 1: [N][SAMPLE_COLS]
  const float* tau;         // MODE 2: [N] thresholds on d^2
  uint2* cand;              // MODE 2: [N][CAND_CAP] (column index inside the window, d^2 bits)
  int32_t* cand_cnt;        // MODE 2: [N] number of appended candidates (may exceed CAND_CAP: overflow)
};

__device__ __forceinline__ int sample_tile(int s, int nt) { return s == 0 ? nt / 4 : (3 * nt) / 4; }

template <int MODE>
struct TileCursor {                                          // flattened tile id -> (window, ti, tj); ids only grow
  int64_t w = 0;
  __device__ __forceinline__ void seek(const Gram2Args& a, int64_t t, int& ti, int& tj, int& nt) {
    while (t >= a.tri_off[w + 1]) ++w;
    const int rem = (int)(t - a.tri_off[w]);
    nt = (int)(a.tile_off[w + 1] - a.tile_off[w]);
    if (MODE == 0) {
      ti = rem / nt;
      tj = rem - ti * nt;
    } else if (MODE == 1) {
      ti = rem >> 1;
      tj = sample_tile(rem & 1, nt);
    } else {                                                 // row ti owns tiles (ti, ti), (ti, ti + 1), ... of the upper triangle
      int r = rem;
      ti = 0;
      while (r >= nt - ti) { r -= nt - ti; ++ti; }
      tj = ti + r;
    }
  }
};

template <int MODE>
__global__ void __launch_bounds__(G2_THREADS, 1) gram_blocks2_kernel(Gram2Args a) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + G2_SM_BAR);
  uint64_t* empty = full + G2_STAGES;
  uint64_t* acc_full = empty + G2_STAGES;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + G2_SM_TMEM);
  if (tid == 0) {
    for (int i = 0; i < G2_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], G2_EPI_WARPS); }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc<256>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tcol = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  const int nchunks = (int)(a.dim / KC);
  const int64_t total = a.tri_off[a.num_graphs];
  TileCursor<MODE> cur;

  if (warp == G2_EPI_WARPS) {
    // ---- TMA producer
    uint32_t it = 0;
    for (int64_t t = blockIdx.x; t < total; t += gridDim.x) {
      int ti, tj, nt;
      cur.seek(a, t, ti, tj, nt);
      const uint8_t* abase = a.img + (a.tile_off[cur.w] + ti) * (int64_t)nchunks * CHUNK_BYTES;
      const uint8_t* bbase = a.img + (a.tile_off[cur.w] + tj) * (int64_t)nchunks * CHUNK_BYTES;
      for (int c = 0; c < nchunks; ++c, ++it) {
        const uint32_t s = it % G2_STAGES, ph = (it / G2_STAGES) & 1;
        mbar_wait(&empty[s], ph ^ 1);                          // the MMAs that read this stage have retired
        if (elect_one()) {
          const uint32_t dst = smem_u32(smem + s * 2 * CHUNK_BYTES);
          mbar_arrive_expect_tx(&full[s], 2 * CHUNK_BYTES);
          tma_bulk_g2s(dst, abase + (int64_t)c * CHUNK_BYTES, CHUNK_BYTES, &full[s]);
          tma_bulk_g2s(dst + CHUNK_BYTES, bbase + (int64_t)c * CHUNK_BYTES, CHUNK_BYTES, &full[s]);
        }
        __syncwarp();
      }
    }
  } else if (warp == G2_EPI_WARPS + 1) {
    // ---- MMA issuer
    const uint64_t dbase = smem_desc_kmajor(0, 128, 256);
    uint32_t it = 0, tl = 0;
    for (int64_t t = blockIdx.x; t < total; t += gridDim.x, ++tl) {
      const uint32_t buf = tl & 1, aph = (tl >> 1) & 1;
      int ti, tj, nt;
      cur.seek(a, t, ti, tj, nt);
      // (i, j) and (j, i) are computed by different tiles and must come out BIT-IDENTICAL (row j compares its own
      // copy of the pair against its own k-th value): the mirrored tile accumulates the same terms in the same order
      const bool mirrored = MODE == 0 && ti > tj;
      mbar_wait(&acc_empty[buf], aph ^ 1);                     // the epilogue has drained this accumulator
      for (int c = 0; c < nchunks; ++c, ++it) {
        const uint32_t s = it % G2_STAGES, ph = (it / G2_STAGES) & 1;
        mbar_wait(&full[s], ph);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t ab = smem_u32(smem + s * 2 * CHUNK_BYTES), bb = ab + CHUNK_BYTES;
          const uint32_t d = tcol + buf * TS;
#pragma unroll
          for (int ks = 0; ks < KC / 16; ++ks) {
            const uint64_t ah = dbase + (uint64_t)((ab + ks * SLAB) >> 4), al = dbase + (uint64_t)((ab + (KC / 16 + ks) * SLAB) >> 4);
            const uint64_t bh = dbase + (uint64_t)((bb + ks * SLAB) >> 4), bl = dbase + (uint64_t)((bb + (KC / 16 + ks) * SLAB) >> 4);
            mma_ss(d, ah, bh, idesc_f16(128, TS), (c > 0 || ks > 0) ? 1u : 0u);
            mma_ss(d, mirrored ? al : ah, mirrored ? bh : bl, idesc_f16(128, TS), 1u);
            mma_ss(d, mirrored ? ah : al, mirrored ? bl : bh, idesc_f16(128, TS), 1u);
          }
          mma_commit(&empty[s]);
          if (c == nchunks - 1) mma_commit(&acc_full[buf]);
        }
        __syncwarp();
      }
    }
  } else {
    // ---- epilogue: warp = (column group cg, TMEM lane quarter wq)
    const int wq = warp & 3, cg = warp >> 2;
    const float eps = 1e-6f;
    const float keps = (float)a.dim * eps * eps;
    uint32_t tl = 0;
    for (int64_t t = blockIdx.x; t < total; t += gridDim.x, ++tl) {
      const uint32_t buf = tl & 1, aph = (tl >> 1) & 1;
      int ti, tj, nt;
      cur.seek(a, t, ti, tj, nt);
      const int64_t n0 = a.gptr[cur.w], n = a.gptr[cur.w + 1] - n0;
      const float down = ldexpf(1.f, -2 * pack_shift(a.win_amax[cur.w]));   // the packed Gram is the true one x 2^2p
      int64_t li = (int64_t)ti * TS + wq * 32 + lane;
      const bool valid = li < n;
      if (!valid) li = n - 1;
      const float na = a.norm2[n0 + li], sa = a.sum1[n0 + li];
      const int fi = (int)a.frame[n0 + li];
      // this lane's column of the warp's 32-column group (values are exchanged with shuffles below)
      const int64_t lc = (int64_t)tj * TS + cg * 32 + lane;
      const bool vc = lc < n;
      const float nb_l = vc ? a.norm2[n0 + lc] : 0.f, sb_l = vc ? a.sum1[n0 + lc] : 0.f;
      const int fb_l = vc ? (int)a.frame[n0 + lc] : INT_MIN;
      float tau_i = 0.f, tau_l = 0.f;
      if (MODE == 2) { tau_i = a.tau[n0 + li]; tau_l = vc ? a.tau[n0 + lc] : -1.f; }
      mbar_wait(&acc_full[buf], aph);
      tc_fence_after();
      uint32_t acc0[16], acc1[16];
      const uint32_t taddr = tcol + buf * TS + cg * 32 + ((uint32_t)(wq * 32) << 16);
      tmem_ld16(taddr, acc0);
      tmem_ld16(taddr + 16, acc1);
      tc_wait_ld();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_empty[buf]);             // the accumulator may be overwritten from here on
      if (MODE == 0) {
        float* D = a.dense + a.doff[cur.w];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float nb = __shfl_sync(0xffffffffu, nb_l, j), sb = __shfl_sync(0xffffffffu, sb_l, j);
          const int fj = __shfl_sync(0xffffffffu, fb_l, j);
          const int64_t lj = (int64_t)tj * TS + cg * 32 + j;
          if (!valid || lj >= n || lj == li || (ti == tj && lj < li)) continue;   // diagonal tile: upper half, mirrored below
          int df = fi - fj; df = df < 0 ? -df : df;
          const bool conn = fj != INT_MIN && df > 0 && (a.max_dist < 0 || df <= a.max_dist);
          // ||a_lo - a_hi + eps||^2 with lo / hi = the smaller / larger node index of the pair (the reference's i < j)
          const float ds = li < lj ? sa - sb : sb - sa;
          const float d2 = (na + nb) - 2.f * (__uint_as_float(j < 16 ? acc0[j] : acc1[j - 16]) * down) + 2.f * eps * ds + keps;
          const float d2c = fmaxf(d2, 0.f);
          const float v = conn ? d2c : INFINITY;
          D[lj * n + li] = v;                                        // row lj, column li: lanes = consecutive floats
          if (ti == tj) D[li * n + lj] = v;
        }
        if (ti == tj && cg == 0 && valid) D[li * n + li] = INFINITY;
      } else if (MODE == 1) {
        // sample pass: this thread's 32 entries of its row, 128 B contiguous in sample[row][s * 128 + cg * 32 ...]
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float nb = __shfl_sync(0xffffffffu, nb_l, j), sb = __shfl_sync(0xffffffffu, sb_l, j);
          const int fj = __shfl_sync(0xffffffffu, fb_l, j);
          const int lj = tj * TS + cg * 32 + j;
          int df = fi - fj; df = df < 0 ? -df : df;
          const bool conn = fj != INT_MIN && lj != (int)li && df > 0 && (a.max_dist < 0 || df <= a.max_dist);
          const float ds = (int)li < lj ? sa - sb : sb - sa;
          const float d2 = (na + nb) - 2.f * (__uint_as_float(j < 16 ? acc0[j] : acc1[j - 16]) * down) + 2.f * eps * ds + keps;
          v[j] = conn ? fmaxf(d2, 0.f) : INFINITY;
        }
        if (valid) {
          const int sidx = tj == sample_tile(0, nt) ? 0 : 1;
          float4* dst = reinterpret_cast<float4*>(a.sample + (n0 + li) * SAMPLE_COLS + sidx * TS + cg * 32);
#pragma unroll
          for (int q = 0; q < 8; ++q) dst[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
      } else {
        // thresholded pass (upper-triangular tiles): one value per pair, offered to both rows' candidate lists.  Pairs
        // that are not time-valid are dropped by cand_select_kernel (they rarely pass the threshold).
        // Two sweeps over the 32 columns: the first only computes and votes (no memory traffic), then every lane reserves
        // list slots ONCE for its row and once for its column (two atomics per lane per tile, all in flight together),
        // the second writes the few passing entries at their ranks.
        const int row_l = (int)li, colbase = tj * TS + cg * 32;
        const bool diag = ti == tj;
        float d2v[32];
        uint32_t rowmask = 0u, colmask = 0u;                     // bit j: column j passes for my row / lane j's column: rows that pass
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float nb = __shfl_sync(0xffffffffu, nb_l, j), sb = __shfl_sync(0xffffffffu, sb_l, j);
          const float tau_j = __shfl_sync(0xffffffffu, tau_l, j);
          const int lj = colbase + j;
          d2v[j] = fmaxf((na + nb) - 2.f * (__uint_as_float(j < 16 ? acc0[j] : acc1[j - 16]) * down) + 2.f * eps * (sa - sb) + keps, 0.f);
          const bool live = valid && lj < (int)n && (!diag || lj > row_l);
          if (live && d2v[j] <= tau_i) rowmask |= 1u << j;
          const uint32_t vote = __ballot_sync(0xffffffffu, live && d2v[j] <= tau_j);
          if (lane == j) colmask = vote;
        }
        const int rcnt = __popc(rowmask), ccnt = __popc(colmask);
        const int64_t crow = n0 + (int64_t)colbase + lane;        // the row this lane reserves column-side slots for
        int rbase = 0, cbase = 0;
        if (rcnt) rbase = atomicAdd(&a.cand_cnt[n0 + li], rcnt);
        if (ccnt) cbase = atomicAdd(&a.cand_cnt[crow], ccnt);
        uint2* rlist = a.cand + (n0 + li) * CAND_CAP;
        const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          if ((rowmask >> j) & 1u) {
            const int slot = rbase + __popc(rowmask & ((1u << j) - 1u));
            if (slot < CAND_CAP) rlist[slot] = make_uint2((uint32_t)(colbase + j), __float_as_uint(d2v[j]));
          }
          const uint32_t cm = __shfl_sync(0xffffffffu, colmask, j);
          const int cb = __shfl_sync(0xffffffffu, cbase, j);
          if ((cm >> lane) & 1u) {
            const int slot = cb + __popc(cm & lt);
            if (slot < CAND_CAP) a.cand[(n0 + (int64_t)colbase + j) * CAND_CAP + slot] = make_uint2((uint32_t)row_l, __float_as_uint(d2v[j]));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<256>(*tmem_slot);
}

// ------------------------------------------------------------------ thresholded path: per-row threshold from the sample
// Warp per row: tau = the r-th smallest of the row's time-valid sample entries, r = ceil(2.5 k valid / n) + 6 -- about 2.5x
// the number of true top-k members a uniform sample of that size holds, so that P(fewer than k row entries <= tau) is
// negligible (those rows fall back to the exact path) while ~2.5 k + n / valid * 6 entries pass.
__global__ void __launch_bounds__(256) row_threshold_kernel(const float* __restrict__ sample, const int64_t* __restrict__ gptr,
                                                            int64_t num_graphs, int64_t num_nodes, int64_t k,
                                                            float* __restrict__ tau) {
  const int lane = threadIdx.x & 31;
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= num_nodes) return;
  const int64_t g = window_of(gptr, num_graphs, i);
  const int64_t n = gptr[g + 1] - gptr[g];
  float v[8];
  int nv = 0;
#pragma unroll
  for (int q = 0; q < 8; ++q) { v[q] = sample[i * SAMPLE_COLS + q * 32 + lane]; nv += isfinite(v[q]) ? 1 : 0; }
  for (int d = 16; d > 0; d >>= 1) nv += __shfl_xor_sync(0xffffffffu, nv, d);
  int r = (int)((5 * k * nv + 2 * n - 1) / (2 * n)) + 6;
  if (nv < 8 || r > nv) { if (lane == 0) tau[i] = INFINITY; return; }        // too few valid samples: keep everything
  // lane-local ascending order (odd-even transposition), then a tournament over the lanes' heads
#pragma unroll
  for (int pass = 0; pass < 8; ++pass)
#pragma unroll
    for (int q = pass & 1; q + 1 < 8; q += 2) { const float a = fminf(v[q], v[q + 1]), b = fmaxf(v[q], v[q + 1]); v[q] = a; v[q + 1] = b; }
  float m = INFINITY;
  for (int it = 0; it < r; ++it) {
    m = v[0];
    for (int d = 16; d > 0; d >>= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, d));
    const unsigned who = __ballot_sync(0xffffffffu, v[0] == m);
    if (lane == __ffs(who) - 1) {
#pragma unroll
      for (int q = 0; q + 1 < 8; ++q) v[q] = v[q + 1];
      v[7] = INFINITY;
    }
  }
  if (lane == 0) tau[i] = m;
}

// Warp per row over its candidate list: drop the entries that are not time-valid, radix-select the k-th smallest
// (d^2 bits, index), set the row of the bit matrix M, and flag the row for the exact path when the approximate
// distances cannot decide the top-k set (error band), when the list overflowed or holds fewer than k valid entries.
constexpr int CSEL_WARPS = 4;
__global__ void __launch_bounds__(32 * CSEL_WARPS) cand_select_kernel(
    const uint2* __restrict__ cand, const int32_t* __restrict__ cand_cnt, const float* __restrict__ tau,
    const int64_t* __restrict__ frame, const int64_t* __restrict__ gptr, int64_t num_graphs, int64_t num_nodes,
    const int64_t* __restrict__ moff, int64_t k, int64_t max_dist, const float* __restrict__ norm2,
    const float* __restrict__ win_nmax, float beta, float keps, uint32_t* __restrict__ M, int32_t* __restrict__ amb,
    int32_t* __restrict__ amb_count) {
  __shared__ int s_hist[CSEL_WARPS][256];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int64_t i = (int64_t)blockIdx.x * CSEL_WARPS + wib;
  if (i >= num_nodes) return;
  int* hist = s_hist[wib];
  const int64_t g = window_of(gptr, num_graphs, i);
  const int64_t n0 = gptr[g], n = gptr[g + 1] - n0, li = i - n0;
  const int words = (int)((n + 31) >> 5);
  uint32_t* mrow = M + moff[g] + li * words;
  for (int w = lane; w < words; w += 32) mrow[w] = 0u;
  const int cnt = cand_cnt[i];
  bool fallback = cnt > CAND_CAP;
  const int64_t fi = frame[i];
  constexpr int PER = CAND_CAP / 32;
  uint32_t key[PER];
  int32_t idx[PER];
  int nvalid = 0;
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const int c = q * 32 + lane;
    key[q] = 0xffffffffu; idx[q] = -1;
    if (!fallback && c < cnt) {
      const uint2 e = cand[i * CAND_CAP + c];
      if ((int64_t)e.x != li && frames_connect(fi, frame[n0 + e.x], max_dist)) { key[q] = e.y; idx[q] = (int32_t)e.x; ++nvalid; }
    }
  }
  for (int d = 16; d > 0; d >>= 1) nvalid += __shfl_xor_sync(0xffffffffu, nvalid, d);
  if (nvalid < k) fallback = true;                       // (tau = +inf rows overflow the list and come here too)
  uint32_t kth = 0xffffffffu;
  int32_t kth_idx = -1;
  float mn = INFINITY;
  if (!fallback) {
    // radix select on the d^2 bit patterns (non-negative floats order like their bits)
    uint32_t prefix = 0u, mask = 0u;
    int remaining = (int)k;
    for (int shift = 24; shift >= 0; shift -= 8) {
      for (int b = lane; b < 256; b += 32) hist[b] = 0;
      __syncwarp();
#pragma unroll
      for (int q = 0; q < PER; ++q)
        if (idx[q] >= 0 && (key[q] & mask) == prefix) atomicAdd(&hist[(key[q] >> shift) & 255u], 1);
      __syncwarp();
      int h[8], tot = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { h[q] = hist[8 * lane + q]; tot += h[q]; }
      int incl = tot;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
      const bool mine = incl >= remaining && incl - tot < remaining;               // exactly one lane
      int rem = remaining - (incl - tot), b = 0;
      if (mine) {
#pragma unroll
        for (int q = 0; q < 8; ++q) { if (h[q] >= rem) { b = q; break; } rem -= h[q]; }
      }
      const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
      remaining = __shfl_sync(0xffffffffu, rem, src);
      prefix |= (uint32_t)(8 * src + __shfl_sync(0xffffffffu, b, src)) << shift;
      mask |= 255u << shift;
      __syncwarp();
    }
    kth = prefix;
    // `remaining` of the entries equal to the k-th key are in, in index order: the remaining-th smallest index among them
    int32_t last = -1;
    for (int it = 0; it < remaining; ++it) {
      int32_t best = INT_MAX;
#pragma unroll
      for (int q = 0; q < PER; ++q) if (idx[q] >= 0 && key[q] == kth && idx[q] > last && idx[q] < best) best = idx[q];
      for (int d = 16; d > 0; d >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, d));
      last = best;
    }
    kth_idx = last;
    __syncwarp();
#pragma unroll
    for (int q = 0; q < PER; ++q) {
      if (idx[q] < 0) continue;
      const bool in = key[q] < kth || (key[q] == kth && idx[q] <= kth_idx);
      if (in) atomicOr(&mrow[idx[q] >> 5], 1u << (idx[q] & 31));
      else mn = fminf(mn, __uint_as_float(key[q]));
    }
    for (int d = 16; d > 0; d >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, d));
    // everything that is not a candidate lies above tau: without an out-of-set candidate tau itself bounds them from below
    if (!isfinite(mn)) mn = tau[i];
    const float band = beta * (norm2[i] + win_nmax[g] + keps);                      // absolute error bound on d^2
    if (isfinite(mn) && (mn - __uint_as_float(kth)) <= 2.f * band) fallback = true;
  }
  if (lane == 0) {
    int flag = 0;
    if (fallback) flag = atomicAdd(amb_count, 1) + 1;                              // slot + 1 of the row in the exact scratch
    amb[i] = flag;
  }
}

}  // namespace gram

int64_t gram_workspace_bytes(int64_t num_nodes, int64_t total_tiles, int64_t num_graphs, int64_t dim) {
  return align_up(total_tiles * (dim / gram::KC) * gram::CHUNK_BYTES, 256) + 2 * align_up(num_nodes * 4, 256) +
         2 * align_up((num_graphs + 1) * 8, 256) + align_up(num_nodes * 4, 256) + 1024 +
         // thresholded path: sample, tau, candidate lists and their counters
         align_up(num_nodes * gram::SAMPLE_COLS * 4, 256) + 2 * align_up(num_nodes * 4, 256) +
         align_up(num_nodes * (int64_t)gram::CAND_CAP * 8, 256) +
         align_up(num_graphs * 4, 256);                       // largest |v| per window (pre-scale)
}

// K eps^2 of the d^2 formula: the band's floor, the size of the d^2 terms that do not scale with the embeddings
float gram_band_keps(int64_t dim) { return (float)dim * 1e-6f * 1e-6f; }

namespace {
struct GramWs {
  uint8_t* img; float* norm2; float* sum1; int64_t* tile_off; int64_t* tri_off; int32_t* amb;
  float* sample; float* tau; int32_t* cand_cnt; uint2* cand; uint32_t* win_amax;
};
GramWs carve_gram(void* ws, int64_t n, int64_t total_tiles, int64_t num_graphs, int64_t dim) {
  Carver cv(ws);
  GramWs w;
  w.img = cv.take<uint8_t>(total_tiles * (dim / gram::KC) * gram::CHUNK_BYTES);
  w.norm2 = cv.take<float>(n);
  w.sum1 = cv.take<float>(n);
  w.tile_off = cv.take<int64_t>(num_graphs + 1);
  w.tri_off = cv.take<int64_t>(num_graphs + 1);
  w.amb = cv.take<int32_t>(n + 1);
  w.sample = cv.take<float>(n * gram::SAMPLE_COLS);
  w.tau = cv.take<float>(n);
  w.cand_cnt = cv.take<int32_t>(n);
  w.cand = cv.take<uint2>(n * (int64_t)gram::CAND_CAP);
  w.win_amax = cv.take<uint32_t>(num_graphs);
  return w;
}

// pack the embeddings into the tile image, each window times its 2^p (+ unscaled norms / sums); shared by the dense and
// the thresholded path
int gram_pack(const float* reid, int64_t dim, const int64_t* gptr, const int64_t* h_gptr, int64_t num_graphs, const GramWs& w,
              int32_t* status, int64_t* total_tiles_out, cudaStream_t s) {
  using namespace gram;
  const int64_t n = h_gptr[num_graphs];
  int64_t total_tiles = 0;
  for (int64_t g = 0; g < num_graphs; ++g) total_tiles += ceil_div(h_gptr[g + 1] - h_gptr[g], TS);
  MPN_CUDA(cudaMemsetAsync(w.img, 0, total_tiles * (dim / KC) * CHUNK_BYTES, s));
  MPN_CUDA(cudaMemsetAsync(w.amb + n, 0, 4, s));
  MPN_CUDA(cudaMemsetAsync(w.win_amax, 0, 4 * num_graphs, s));
  tile_offsets_kernel<<<1, 32, 0, s>>>(gptr, num_graphs, w.tile_off, w.tri_off, 0); count_launch();
  const unsigned pgrid = (unsigned)std::min<int64_t>(ceil_div(n * 32, 256), (int64_t)sm_count() * 16);
  window_absmax_kernel<<<pgrid, 256, 0, s>>>(reid, dim, gptr, num_graphs, n, w.win_amax); count_launch();
  pack_reid_kernel<<<pgrid, 256, 0, s>>>(reid, dim, gptr, num_graphs, w.tile_off, n, w.win_amax, w.img, w.norm2, w.sum1,
                                         status); count_launch();
  MPN_CUDA(cudaFuncSetAttribute(gram::gram_blocks2_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, G2_SMEM_BYTES));
  MPN_CUDA(cudaFuncSetAttribute(gram::gram_blocks2_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, G2_SMEM_BYTES));
  MPN_CUDA(cudaFuncSetAttribute(gram::gram_blocks2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, G2_SMEM_BYTES));
  *total_tiles_out = total_tiles;
  return MPN_OK;
}
int64_t count_tiles(const int64_t* h_gptr, int64_t num_graphs) {
  int64_t t = 0;
  for (int64_t g = 0; g < num_graphs; ++g) t += ceil_div(h_gptr[g + 1] - h_gptr[g], gram::TS);
  return t;
}
}  // namespace

// Fills the dense blocks with approximate d^2 from the Gram kernel; the caller ranks the rows and repairs the flagged ones.
int gram_dist_blocks(const float* reid, int64_t dim, const int64_t* frame, const int64_t* gptr, const int64_t* h_gptr,
                     int64_t num_graphs, const int64_t* doff, int64_t max_dist, void* ws, float* dense,
                     int32_t* status, float** norm2_out, int32_t** amb_out, int32_t** amb_count_out, cudaStream_t s) {
  using namespace gram;
  const int64_t n = h_gptr[num_graphs];
  GramWs w = carve_gram(ws, n, count_tiles(h_gptr, num_graphs), num_graphs, dim);
  int64_t total_tiles = 0;
  int rc = gram_pack(reid, dim, gptr, h_gptr, num_graphs, w, status, &total_tiles, s);
  if (rc) return rc;
  int64_t total_blocks = 0;
  for (int64_t g = 0; g < num_graphs; ++g) {
    const int64_t t = ceil_div(h_gptr[g + 1] - h_gptr[g], TS);
    total_blocks += t * t;
  }
  Gram2Args a2 = {};
  a2.frame = frame; a2.gptr = gptr; a2.doff = doff; a2.tile_off = w.tile_off; a2.tri_off = w.tri_off;
  a2.img = w.img; a2.norm2 = w.norm2; a2.sum1 = w.sum1; a2.win_amax = w.win_amax; a2.num_graphs = num_graphs; a2.max_dist = max_dist; a2.dim = dim;
  a2.dense = dense;
  const unsigned grid2 = (unsigned)std::min<int64_t>(std::max<int64_t>(total_blocks, 1), (int64_t)sm_count());
  gram_blocks2_kernel<0><<<grid2, G2_THREADS, G2_SMEM_BYTES, s>>>(a2); count_launch();
  MPN_LAUNCH_CHECK();
  *norm2_out = w.norm2; *amb_out = w.amb; *amb_count_out = w.amb + n;
  return MPN_OK;
}

// Thresholded path (every window has >= TG_MIN_TILES tiles): sample pass -> per-row thresholds -> candidate lists from the
// upper-triangular Gram tiles -> candidate select (bit matrix rows + rows flagged for the exact repair).  No N^2 output.
bool gram_thresholded_applies(const int64_t* h_gptr, int64_t num_graphs, int64_t top_k) {
  for (int64_t g = 0; g < num_graphs; ++g)
    if (h_gptr[g + 1] - h_gptr[g] < (int64_t)gram::TG_MIN_TILES * gram::TS) return false;
  // The candidate lists grow with k: measured on 4 windows x 4,500 nodes (profiles/r02_config5_sweep.md) the thresholded build
  // wins up to k = 50 (3.35 vs 4.17 ms per step at k = 25) and loses from k = 75 on (6.80 vs 5.50 ms), so the default gate is
  // TG_DEFAULT_MAX_K; MPN_KNN_THRESHOLDED=1 extends it to the structural limit CAND_CAP / 4 (tests, measurements).
  const bool force = getenv("MPN_KNN_THRESHOLDED") != nullptr;        // read per call: tests toggle it
  return top_k >= 1 && top_k <= (force ? gram::CAND_CAP / 4 : gram::TG_DEFAULT_MAX_K);
}

int gram_thresholded_select(const float* reid, int64_t dim, const int64_t* frame, const int64_t* gptr, const int64_t* h_gptr,
                            int64_t num_graphs, const int64_t* moff, int64_t max_dist, int64_t top_k, void* ws,
                            const float* win_nmax_buf, float beta, uint32_t* M, int32_t* status, float** norm2_out,
                            int32_t** amb_out, int32_t** amb_count_out, void (*window_max)(const float*, const int64_t*, int64_t, float*, cudaStream_t),
                            cudaStream_t s) {
  using namespace gram;
  const int64_t n = h_gptr[num_graphs];
  GramWs w = carve_gram(ws, n, count_tiles(h_gptr, num_graphs), num_graphs, dim);
  int64_t total_tiles = 0;
  int rc = gram_pack(reid, dim, gptr, h_gptr, num_graphs, w, status, &total_tiles, s);
  if (rc) return rc;
  float* win_nmax = const_cast<float*>(win_nmax_buf);
  window_max(w.norm2, gptr, num_graphs, win_nmax, s);
  Gram2Args a2 = {};
  a2.frame = frame; a2.gptr = gptr; a2.doff = nullptr; a2.tile_off = w.tile_off; a2.tri_off = w.tri_off;
  a2.img = w.img; a2.norm2 = w.norm2; a2.sum1 = w.sum1; a2.win_amax = w.win_amax; a2.num_graphs = num_graphs; a2.max_dist = max_dist; a2.dim = dim;
  a2.sample = w.sample; a2.tau = w.tau; a2.cand = w.cand; a2.cand_cnt = w.cand_cnt;
  const int sms = sm_count();
  // 1. sample pass
  tile_offsets_kernel<<<1, 32, 0, s>>>(gptr, num_graphs, w.tile_off, w.tri_off, 1); count_launch();
  gram_blocks2_kernel<1><<<(unsigned)std::min<int64_t>(2 * total_tiles, sms), G2_THREADS, G2_SMEM_BYTES, s>>>(a2); count_launch();
  // 2. thresholds
  row_threshold_kernel<<<(unsigned)ceil_div(n * 32, 256), 256, 0, s>>>(w.sample, gptr, num_graphs, n, top_k, w.tau); count_launch();
  // 3. candidate lists from the upper-triangular tiles
  MPN_CUDA(cudaMemsetAsync(w.cand_cnt, 0, sizeof(int32_t) * n, s));
  int64_t tri = 0;
  for (int64_t g = 0; g < num_graphs; ++g) { const int64_t t = ceil_div(h_gptr[g + 1] - h_gptr[g], TS); tri += t * (t + 1) / 2; }
  tile_offsets_kernel<<<1, 32, 0, s>>>(gptr, num_graphs, w.tile_off, w.tri_off, 2); count_launch();
  gram_blocks2_kernel<2><<<(unsigned)std::min<int64_t>(tri, sms), G2_THREADS, G2_SMEM_BYTES, s>>>(a2); count_launch();
  // 4. exact top-k over the candidates
  cand_select_kernel<<<(unsigned)ceil_div(n, CSEL_WARPS), 32 * CSEL_WARPS, 0, s>>>(
      w.cand, w.cand_cnt, w.tau, frame, gptr, num_graphs, n, moff, top_k, max_dist, w.norm2, win_nmax, beta, gram_band_keps(dim), M, w.amb,
      w.amb + n);
  count_launch();
  MPN_LAUNCH_CHECK();
  *norm2_out = w.norm2; *amb_out = w.amb; *amb_count_out = w.amb + n;
  return MPN_OK;
}

}  // namespace mpn
