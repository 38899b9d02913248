// MOTS result of the tracker on the device (SURVEY.md §2 row 13, §3.1): the reference's host stage
//   * paste every node mask into its frame     tracker/mpn_tracker.py:267-298 (torchvision paste_masks_in_image)
//   * one owner per pixel within a frame        ensure_unique_masks
//   * RLE of every mask, text of the result     pycocotools rleEncode / rleToString, save at :398-417
// The per-node 56x56 masks never leave HBM, and the RLE work is proportional to the box areas and the run counts: no
// [N,H,W] image or per-frame buffer exists.  Integer offsets come from scans; no atomics touch the outputs, so two runs
// give identical bytes.  The contract (integer box, pasted probability, ownership, RLE) is stated in DESIGN.md.
#include "common.cuh"

namespace mpn {
namespace {

// Integer box of torchvision's expand_boxes + .to(int64), computed by the caller: (x0, y0, x1, y1), inclusive.
struct IBox { int64_t x0, y0, x1, y1; };

__device__ __forceinline__ IBox load_box(const int64_t* __restrict__ boxes, int64_t i) {
  return IBox{__ldg(boxes + 4 * i), __ldg(boxes + 4 * i + 1), __ldg(boxes + 4 * i + 2), __ldg(boxes + 4 * i + 3)};
}

__device__ __forceinline__ bool box_covers(const IBox& b, int64_t y, int64_t x) {
  return y >= b.y0 && y <= b.y1 && x >= b.x0 && x <= b.x1;
}

// ATen's upsample_bilinear2d (align_corners=False, no scale factor) source index along one axis: src = max((d + 0.5)·
// (in/out) − 0.5, 0), i0 = floor(src), i1 = min(i0 + 1, in − 1), lambda = src − i0.  Explicit roundings (no FMA), so the
// index and weight are those of the unfused double arithmetic the CPU reference runs.
__device__ __forceinline__ void src_index(int in, int64_t out, int64_t d, int& i0, int& i1, double& lam) {
  double s = __dsub_rn(__dmul_rn((double)in / (double)out, (double)d + 0.5), 0.5);
  s = s < 0.0 ? 0.0 : s;
  i0 = (int)s;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  lam = s - (double)i0;
}

__device__ __forceinline__ double texel(const float* __restrict__ mask, int m, int pad, int r, int c) {
  r -= pad; c -= pad;
  return (r >= 0 && r < m && c >= 0 && c < m) ? (double)__ldg(mask + (int64_t)r * m + c) : 0.0;
}

// p(y, x): the (M + 2·pad)² zero-padded mask resized to the box's h × w by bilinear interpolation, read at
// (y − y0, x − x0).  The caller guarantees y0 <= y <= y1 and x0 <= x <= x1.  The only definition of the pasted
// probability: the dense paste, the count and the fill kernels all call it.
__device__ double paste_prob(const float* __restrict__ mask, int m, int pad, const IBox& b, int64_t y, int64_t x) {
  const int in = m + 2 * pad;
  const int64_t h = max(b.y1 - b.y0 + 1, (int64_t)1), w = max(b.x1 - b.x0 + 1, (int64_t)1);
  int r0, r1, c0, c1;
  double ly, lx;
  src_index(in, h, y - b.y0, r0, r1, ly);
  src_index(in, w, x - b.x0, c0, c1, lx);
  const double hy = 1.0 - ly, hx = 1.0 - lx;
  const double top = __dadd_rn(__dmul_rn(hx, texel(mask, m, pad, r0, c0)), __dmul_rn(lx, texel(mask, m, pad, r0, c1)));
  const double bot = __dadd_rn(__dmul_rn(hx, texel(mask, m, pad, r1, c0)), __dmul_rn(lx, texel(mask, m, pad, r1, c1)));
  return __dadd_rn(__dmul_rn(hy, top), __dmul_rn(ly, bot));
}

__global__ void paste_dense_kernel(const float* __restrict__ masks, int64_t n, int m, int pad,
                                   const int64_t* __restrict__ boxes, int64_t H, int64_t W, float* __restrict__ out) {
  const int64_t hw = H * W, total = n * hw, mm = (int64_t)m * m;
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = idx / hw, r = idx - i * hw, y = r / W, x = r - y * W;
    const IBox b = load_box(boxes, i);
    out[idx] = box_covers(b, y, x) ? (float)paste_prob(masks + i * mm, m, pad, b, y, x) : 0.f;
  }
}

// ------------------------------------------------------------------ RLE
// pycocotools rleToString: x = cnt[i] − cnt[i−2] for i > 2, 5-bit groups low first, 0x20 = more, +48.
__device__ __forceinline__ int rle_chars(int64_t x) {
  int n = 0;
  bool more = true;
  while (more) {
    const int c = (int)(x & 0x1f);
    x >>= 5;                                          // arithmetic shift: negative deltas end at x == −1
    more = (c & 0x10) ? x != -1 : x != 0;
    ++n;
  }
  return n;
}
__device__ __forceinline__ void rle_emit(int64_t x, uint8_t* __restrict__ out) {
  bool more = true;
  while (more) {
    int c = (int)(x & 0x1f);
    x >>= 5;
    more = (c & 0x10) ? x != -1 : x != 0;
    if (more) c |= 0x20;
    *out++ = (uint8_t)(c + 48);
  }
}

constexpr int kThreads = 256;
constexpr int kItems = 8;                             // consecutive pixels of one thread (box column-major order)
constexpr int kTile = kThreads * kItems;

struct RleArgs {
  const float* masks; int64_t n; int m; int pad; const int64_t* boxes; const int64_t* frame; int64_t H, W; double thr;
};

// Pixel (y, x) of node i's clamped box belongs to its mask: p_i > thr and no other detection of the frame whose box
// covers the pixel has a larger p_j, or an equal one at a lower index.  NaN compares false both ways, so a NaN p_i sets
// nothing and a NaN p_j erases nothing.
__device__ __forceinline__ bool owned(const RleArgs& a, int64_t i, const IBox& bi, int64_t lo, int64_t hi, int64_t y,
                                      int64_t x) {
  const int64_t mm = (int64_t)a.m * a.m;
  const double p = paste_prob(a.masks + i * mm, a.m, a.pad, bi, y, x);
  if (!(p > a.thr)) return false;
  for (int64_t j = lo; j < hi; ++j) {
    if (j == i) continue;
    const IBox bj = load_box(a.boxes, j);
    if (!box_covers(bj, y, x)) continue;
    const double q = paste_prob(a.masks + j * mm, a.m, a.pad, bj, y, x);
    if (q > p || (q == p && j < i)) return false;
  }
  return true;
}

// One CTA per node.  The clamped box is walked in the image's column-major order, kTile pixels at a time.  With the
// pixel flags f(k) (k = 0 .. A−1 in box order), the transitions of the image-wide run sequence are
//   end   at pos(k−1) + 1  if f(k−1) and (!f(k) or k starts a column that does not continue the previous one),
//   start at pos(k)        if f(k)   and (!f(k−1) or k starts such a column),
// where a column continues the previous one only when the box spans the full image height (runs then merge across the
// column boundary, as in rleEncode).  Transitions T_0 < T_1 < ... give the counts cnt[t] = T_t − T_{t−1} (T_{−1} = 0)
// and a last count H·W − T_last unless the mask ends on the last pixel.  A block scan places each tile's transitions
// in shared memory after the last three of the tiles before, which is all that the string length of a count needs.
//   kFill = false: area[i], number of counts and of characters (into ncnt / nchr, scanned by the caller);
//   kFill = true:  counts at cnt_ptr[i] and characters at char_ptr[i].
template <bool kFill>
__global__ void __launch_bounds__(kThreads) mots_rle_kernel(RleArgs a, int64_t* __restrict__ area, int64_t* __restrict__ ncnt,
                                                            int64_t* __restrict__ nchr, int32_t* __restrict__ bad_order,
                                                            const int64_t* __restrict__ cnt_ptr,
                                                            const int64_t* __restrict__ char_ptr,
                                                            int32_t* __restrict__ counts, uint8_t* __restrict__ chars) {
  __shared__ uint32_t s_bits[kThreads];
  __shared__ int32_t s_pos[3 + 2 * kTile];           // [0, 3): the last three transitions before the tile (0 = none)
  __shared__ int64_t s_scan[32];
  __shared__ int64_t s_tot;
  __shared__ int64_t s_range[2];
  __shared__ uint32_t s_last;
  const int t = threadIdx.x;
  const int64_t i = blockIdx.x;
  const IBox b = load_box(a.boxes, i);
  if (t == 0) {
    const int64_t f = a.frame[i];
    int64_t l = 0, r = a.n;                           // first node of the frame (frames are non-decreasing)
    while (l < r) { const int64_t c = (l + r) >> 1; if (a.frame[c] < f) l = c + 1; else r = c; }
    s_range[0] = l;
    r = a.n;                                          // one past its last node
    while (l < r) { const int64_t c = (l + r) >> 1; if (a.frame[c] <= f) l = c + 1; else r = c; }
    s_range[1] = l;
    if (!kFill && i > 0 && a.frame[i - 1] > f) *bad_order = 1;
  }
  if (t < 3) s_pos[t] = 0;
  __syncthreads();
  const int64_t lo = s_range[0], hi = s_range[1];
  const int64_t cx0 = max(b.x0, (int64_t)0), cx1 = min(b.x1 + 1, a.W);
  const int64_t cy0 = max(b.y0, (int64_t)0), cy1 = min(b.y1 + 1, a.H);
  const int64_t bh = cy1 - cy0, A = (cx1 > cx0 && bh > 0) ? (cx1 - cx0) * bh : 0;
  const bool full_height = cy0 == 0 && cy1 == a.H;
  const int64_t cbase0 = kFill ? cnt_ptr[i] : 0, chbase0 = kFill ? char_ptr[i] : 0;
  auto pos = [&](int64_t k) -> int32_t {
    const int64_t col = k / bh;
    return (int32_t)((cx0 + col) * a.H + cy0 + (k - col * bh));
  };

  int64_t g = 0, nch = 0, pix = 0;                    // transitions and characters so far, pixels set
  uint32_t carry = 0;                                 // f(k) of the last pixel of the previous tile
  for (int64_t base = 0; base < A; base += kTile) {
    const int64_t k0 = base + (int64_t)t * kItems;
    uint32_t bits = 0;
    {
      int64_t col = k0 / bh, row = k0 - col * bh;
      for (int u = 0; u < kItems && k0 + u < A; ++u) {
        if (owned(a, i, b, lo, hi, cy0 + row, cx0 + col)) bits |= 1u << u;
        if (++row == bh) { row = 0; ++col; }
      }
    }
    s_bits[t] = bits;
    const int64_t last_k = min(base + kTile, A) - 1;
    if (k0 <= last_k && last_k < k0 + kItems) s_last = (bits >> (last_k - k0)) & 1u;
    __syncthreads();
    pix += __popc(bits);
    const uint32_t prev0 = t > 0 ? (s_bits[t - 1] >> (kItems - 1)) & 1u : carry;
    // pass 1: number of transitions of this thread's pixels
    int ne = 0;
    for (int u = 0; u < kItems && k0 + u < A; ++u) {
      const int64_t k = k0 + u;
      const uint32_t f = (bits >> u) & 1u, pf = u ? (bits >> (u - 1)) & 1u : prev0;
      const bool cont = k > 0 && (full_height || k % bh != 0);
      ne += (pf && (!f || !cont)) + (f && (!pf || !cont));
    }
    const int64_t off = block_exclusive_scan<int64_t>(ne, s_scan, &s_tot);
    const int64_t tot = s_tot;
    // pass 2: their positions, after the carried three
    {
      int e = 3 + (int)off;
      for (int u = 0; u < kItems && k0 + u < A; ++u) {
        const int64_t k = k0 + u;
        const uint32_t f = (bits >> u) & 1u, pf = u ? (bits >> (u - 1)) & 1u : prev0;
        const bool cont = k > 0 && (full_height || k % bh != 0);
        if (pf && (!f || !cont)) s_pos[e++] = pos(k - 1) + 1;
        if (f && (!pf || !cont)) s_pos[e++] = pos(k);
      }
    }
    __syncthreads();
    // the counts of these transitions and the lengths of their string pieces
    int64_t nc = 0;
    for (int e = 0; e < ne; ++e) {
      const int s = 3 + (int)off + e;
      const int64_t gi = g + off + e;
      const int64_t c = (int64_t)s_pos[s] - s_pos[s - 1];
      const int64_t x = gi > 2 ? c - ((int64_t)s_pos[s - 2] - s_pos[s - 3]) : c;
      nc += rle_chars(x);
      if (kFill) counts[cbase0 + gi] = (int32_t)c;
    }
    const int64_t coff = block_exclusive_scan<int64_t>(nc, s_scan, &s_tot);
    const int64_t ctot = s_tot;
    if (kFill) {
      uint8_t* out = chars + chbase0 + nch + coff;
      for (int e = 0; e < ne; ++e) {
        const int s = 3 + (int)off + e;
        const int64_t gi = g + off + e;
        const int64_t c = (int64_t)s_pos[s] - s_pos[s - 1];
        const int64_t x = gi > 2 ? c - ((int64_t)s_pos[s - 2] - s_pos[s - 3]) : c;
        rle_emit(x, out);
        out += rle_chars(x);
      }
    }
    __syncthreads();
    if (t == 0) {                                     // carry the last three transitions
      int32_t keep[3];
      for (int q = 0; q < 3; ++q) keep[q] = s_pos[tot + q];
      for (int q = 0; q < 3; ++q) s_pos[q] = keep[q];
    }
    carry = s_last;
    g += tot;
    nch += ctot;
    __syncthreads();
  }

  if (t == 0) {
    int32_t c3[3] = {s_pos[0], s_pos[1], s_pos[2]};
    // the run still open at the end of the box closes after its last pixel; then the zeros up to H·W
    int32_t tail[2];
    int nt = 0;
    if (carry) tail[nt++] = pos(A - 1) + 1;
    if (g + nt > 0 && (int64_t)(nt ? tail[nt - 1] : c3[2]) < a.H * a.W) tail[nt++] = (int32_t)(a.H * a.W);
    for (int q = 0; q < nt; ++q) {
      const int64_t c = (int64_t)tail[q] - c3[2];
      const int64_t x = g > 2 ? c - ((int64_t)c3[1] - c3[0]) : c;
      if (kFill) {
        counts[cbase0 + g] = (int32_t)c;
        rle_emit(x, chars + chbase0 + nch);
      }
      nch += rle_chars(x);
      c3[0] = c3[1]; c3[1] = c3[2]; c3[2] = tail[q];
      ++g;
    }
  }
  if (kFill) return;
  block_exclusive_scan<int64_t>(pix, s_scan, &s_tot);          // area: the pixels set over all threads
  if (t == 0) {
    area[i] = s_tot;
    ncnt[i] = g;
    nchr[i] = nch;
  }
}

unsigned grid_for(int64_t n) {
  const int64_t g = ceil_div(n > 0 ? n : 1, 256);
  const int64_t cap = (int64_t)sm_count() * 16;
  return (unsigned)(g < cap ? g : cap);
}

int check_common(const char* what, const float* masks, int64_t n, int64_t m, int32_t pad, const int64_t* boxes,
                 int64_t h, int64_t w) {
  MPN_CHECK_ARG(n >= 0 && n < 2147483647LL, "%s: bad number of nodes %lld", what, (long long)n);
  MPN_CHECK_ARG(m >= 1 && m <= 4096 && pad >= 0 && pad <= 4096, "%s: bad mask size %lld / padding %d", what, (long long)m,
                (int)pad);
  MPN_CHECK_ARG(h >= 1 && w >= 1 && h * w <= 2147483647LL, "%s: image %lld x %lld must have 1 .. 2^31 - 1 pixels", what,
                (long long)h, (long long)w);
  MPN_CHECK_ARG(n == 0 || (masks && boxes), "%s: null masks or boxes", what);
  return MPN_OK;
}

}  // namespace
}  // namespace mpn

using namespace mpn;

extern "C" {

int mpn_paste_masks(const float* masks, int64_t num_nodes, int64_t mask_size, int32_t padding, const int64_t* boxes,
                    int64_t height, int64_t width, float* out, void* stream) {
  int rc = check_common("paste_masks", masks, num_nodes, mask_size, padding, boxes, height, width);
  if (rc) return rc;
  MPN_CHECK_ARG(num_nodes == 0 || out, "paste_masks: null output");
  if (num_nodes == 0) return MPN_OK;
  cudaStream_t s = as_stream(stream);
  paste_dense_kernel<<<grid_for(num_nodes * height * width), 256, 0, s>>>(masks, num_nodes, (int)mask_size, padding, boxes,
                                                                          height, width, out);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int64_t mpn_mots_rle_workspace(int64_t num_nodes) { (void)num_nodes; return 256; }

int mpn_mots_rle_count(const float* masks, int64_t num_nodes, int64_t mask_size, int32_t padding, const int64_t* boxes,
                       const int64_t* frame, int64_t height, int64_t width, double threshold, void* workspace,
                       int64_t* area, int64_t* cnt_ptr, int64_t* char_ptr, int64_t* h_totals, void* stream) {
  int rc = check_common("mots_rle_count", masks, num_nodes, mask_size, padding, boxes, height, width);
  if (rc) return rc;
  MPN_CHECK_ARG(workspace && cnt_ptr && char_ptr && h_totals, "mots_rle_count: null workspace, offsets or totals");
  MPN_CHECK_ARG(num_nodes == 0 || (frame && area), "mots_rle_count: null frame or area");
  cudaStream_t s = as_stream(stream);
  int32_t* bad = static_cast<int32_t*>(workspace);
  MPN_CUDA(cudaMemsetAsync(bad, 0, sizeof(int32_t), s));
  if (num_nodes > 0) {
    RleArgs a{masks, num_nodes, (int)mask_size, padding, boxes, frame, height, width, threshold};
    mots_rle_kernel<false><<<(unsigned)num_nodes, kThreads, 0, s>>>(a, area, cnt_ptr, char_ptr, bad, nullptr, nullptr,
                                                                    nullptr, nullptr);
    count_launch();
    MPN_LAUNCH_CHECK();
  }
  rc = exclusive_scan_i64(cnt_ptr, cnt_ptr, num_nodes, s);
  if (rc) return rc;
  rc = exclusive_scan_i64(char_ptr, char_ptr, num_nodes, s);
  if (rc) return rc;
  int64_t tot[2] = {0, 0};
  int32_t h_bad = 0;
  MPN_CUDA(cudaMemcpyAsync(&tot[0], cnt_ptr + num_nodes, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaMemcpyAsync(&tot[1], char_ptr + num_nodes, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaMemcpyAsync(&h_bad, bad, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaStreamSynchronize(s));
  MPN_CHECK_ARG(h_bad == 0, "mots_rle_count: frame must be non-decreasing");
  h_totals[0] = tot[0];
  h_totals[1] = tot[1];
  return MPN_OK;
}

int mpn_mots_rle_fill(const float* masks, int64_t num_nodes, int64_t mask_size, int32_t padding, const int64_t* boxes,
                      const int64_t* frame, int64_t height, int64_t width, double threshold, const int64_t* cnt_ptr,
                      const int64_t* char_ptr, int32_t* counts, uint8_t* chars, void* stream) {
  int rc = check_common("mots_rle_fill", masks, num_nodes, mask_size, padding, boxes, height, width);
  if (rc) return rc;
  if (num_nodes == 0) return MPN_OK;
  MPN_CHECK_ARG(frame && cnt_ptr && char_ptr && counts && chars, "mots_rle_fill: null frame, offsets or outputs");
  cudaStream_t s = as_stream(stream);
  RleArgs a{masks, num_nodes, (int)mask_size, padding, boxes, frame, height, width, threshold};
  mots_rle_kernel<true><<<(unsigned)num_nodes, kThreads, 0, s>>>(a, nullptr, nullptr, nullptr, nullptr, cnt_ptr, char_ptr,
                                                                 counts, chars);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // extern "C"
