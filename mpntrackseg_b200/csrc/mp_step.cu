// Fused message-passing step, fp32 SIMT variant ("v1": exact fp32 FMA arithmetic).
//
// One step = two kernels (the second needs every node's new state => grid-wide dependency):
//   mp_edge_kernel : per 128-slot tile, one thread per directed edge
//        e'   = ReLU(W1 ReLU(W0 [x_init[r] | x_lat[r] | x_init[c] | x_lat[c] | e_init | e] + b0) + b1)
//        logit = classifier(e')                                  (models/mpn.py:114)
//        m    = flowMLP_dir([x_init[c] | x_lat[c] | e'])          (models/mpn.py:86-88 / 92-94)
//        per-row sums of m over the tile (slots of a row are contiguous) -> flow / tile partials
//   mp_node_kernel : per node, x' = ReLU(Wn [flow_in | flow_out] + bn)   (models/mpn.py:97-99)
// No float atomics anywhere: the per-row sums are sequential in slot order (= the order the
// reference's CPU scatter_add uses), tile-crossing rows are finished in tile order.
#include "common.cuh"
#include "mlp_regs.cuh"

namespace mpn {

constexpr int TS = 128;  // slots per tile == threads per CTA

template <int DN_, int DE_, int EH_, int FH_, int CH_>
struct CoreWidths {
  static constexpr int DN = DN_, DE = DE_, EH = EH_, FH = FH_, CH = CH_;
  static constexpr int EIN = 4 * DN + 2 * DE;   // edge MLP input  (models/mpn.py:279-280)
  static constexpr int FIN = 2 * DN + DE;       // flow MLP input  (models/mpn.py:282)
  static_assert(DN % 4 == 0 && DE % 4 == 0 && EH % 4 == 0 && FH % 4 == 0 && CH % 4 == 0, "widths % 4");
  static_assert(DN <= 32, "one lane per node feature in the segmented sums");
  // shared memory carve-up (floats)
  static constexpr int OFF_EW0 = 0;
  static constexpr int OFF_EB0 = OFF_EW0 + EIN * EH;
  static constexpr int OFF_EW1 = OFF_EB0 + EH;
  static constexpr int OFF_EB1 = OFF_EW1 + EH * DE;
  static constexpr int OFF_FW0 = OFF_EB1 + DE;
  static constexpr int OFF_FB0 = OFF_FW0 + FIN * FH;
  static constexpr int OFF_FW1 = OFF_FB0 + FH;
  static constexpr int OFF_FB1 = OFF_FW1 + FH * DN;
  static constexpr int OFF_CW0 = OFF_FB1 + DN;
  static constexpr int OFF_CB0 = OFF_CW0 + DE * CH;
  static constexpr int OFF_CW1 = OFF_CB0 + CH;
  static constexpr int OFF_CB1 = OFF_CW1 + CH;
  static constexpr int OFF_MSG = OFF_CB1 + 4;
  static constexpr int MSG_LD = DN + 1;
  static constexpr int OFF_ROWS = OFF_MSG + TS * MSG_LD;      // int32 [TS + 2]
  static constexpr int TOTAL_FLOATS = OFF_ROWS + TS + 4;
  static constexpr size_t SMEM_BYTES = sizeof(float) * TOTAL_FLOATS;
};

struct StepArgs {
  // layout
  const int32_t* slot_row; const int32_t* slot_col; const int32_t* slot_edge;
  int64_t num_edges, num_out;
  int32_t tiles_out, tiles_in;
  // state
  const float* x_init; const float* x_lat;      // [N, DN]
  const float* e_init; const float* e_cur;      // [E, DE] slot order
  float* e_next;                                // [E, DE] (may alias e_cur)
  float* flow;                                  // [N, 2*DN]  (flow_in | flow_out)
  float* part;                                  // [tiles, 2, DN]
  float* logits;                                // row of the logits output for this step or NULL
  int agg;                                      // 0 sum, 1 mean (sums here, divided in the node kernel), 2 max
};

// RO: read through the read-only path (__ldg).  Such loads of one address may be merged by the compiler.
template <int N4, bool RO = true>
__device__ __forceinline__ void load_vec(float (&dst)[N4 * 4], const float* __restrict__ src) {
  const float4* p = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int q = 0; q < N4; ++q) {
    const float4 v = RO ? __ldg(p + q) : p[q];
    dst[4 * q] = v.x; dst[4 * q + 1] = v.y; dst[4 * q + 2] = v.z; dst[4 * q + 3] = v.w;
  }
}

template <typename W>
__global__ void __launch_bounds__(TS) mp_edge_kernel(StepArgs a, mpn_core_weights w) {
  extern __shared__ __align__(16) float smem[];
  constexpr int DN = W::DN, DE = W::DE, EH = W::EH, FH = W::FH, CH = W::CH;
  // CTAs [0, n_out_ctas) walk flow_out tiles, the rest walk flow_in tiles.
  const int total_tiles = a.tiles_out + a.tiles_in;
  int n_out_ctas = (int)(((int64_t)gridDim.x * a.tiles_out + total_tiles - 1) / total_tiles);
  if (a.tiles_out > 0 && n_out_ctas == 0) n_out_ctas = 1;
  if (a.tiles_in > 0 && n_out_ctas >= (int)gridDim.x) n_out_ctas = gridDim.x - 1;
  if (a.tiles_in == 0) n_out_ctas = gridDim.x;
  const bool dir_out = (int)blockIdx.x < n_out_ctas;
  const int cta_in_dir = dir_out ? blockIdx.x : blockIdx.x - n_out_ctas;
  const int ctas_in_dir = dir_out ? n_out_ctas : gridDim.x - n_out_ctas;
  const int tiles_dir = dir_out ? a.tiles_out : a.tiles_in;
  const int64_t seg_base = dir_out ? 0 : a.num_out;
  const int64_t seg_end = dir_out ? a.num_out : a.num_edges;
  const int tile_off = dir_out ? 0 : a.tiles_out;

  stage_weight_t<W::EIN, EH>(w.edge_w0, smem + W::OFF_EW0);
  stage_bias<EH>(w.edge_b0, smem + W::OFF_EB0);
  stage_weight_t<EH, DE>(w.edge_w1, smem + W::OFF_EW1);
  stage_bias<DE>(w.edge_b1, smem + W::OFF_EB1);
  stage_weight_t<W::FIN, FH>(dir_out ? w.fout_w0 : w.fin_w0, smem + W::OFF_FW0);
  stage_bias<FH>(dir_out ? w.fout_b0 : w.fin_b0, smem + W::OFF_FB0);
  stage_weight_t<FH, DN>(dir_out ? w.fout_w1 : w.fin_w1, smem + W::OFF_FW1);
  stage_bias<DN>(dir_out ? w.fout_b1 : w.fin_b1, smem + W::OFF_FB1);
  stage_weight_t<DE, CH>(w.cls_w0, smem + W::OFF_CW0);
  stage_bias<CH>(w.cls_b0, smem + W::OFF_CB0);
  for (int i = threadIdx.x; i < CH; i += blockDim.x) smem[W::OFF_CW1 + i] = w.cls_w1[i];
  if (threadIdx.x == 0) smem[W::OFF_CB1] = w.cls_b1[0];
  float* s_msg = smem + W::OFF_MSG;
  int32_t* s_rows = reinterpret_cast<int32_t*>(smem + W::OFF_ROWS);   // [0]=prev, [1..TS]=tile, [TS+1]=next
  __syncthreads();

  const int tid = threadIdx.x;
  for (int t = cta_in_dir; t < tiles_dir; t += ctas_in_dir) {
    const int64_t base = seg_base + (int64_t)t * TS;
    const int cnt = (int)(seg_end - base < TS ? seg_end - base : TS);
    const int64_t slot = base + tid;
    const bool valid = tid < cnt;
    int32_t r = -1, c = 0;
    if (valid) { r = a.slot_row[slot]; c = a.slot_col[slot]; }
    s_rows[1 + tid] = r;
    if (tid == 0) {
      s_rows[0] = base > seg_base ? a.slot_row[base - 1] : -1;
      s_rows[TS + 1] = base + cnt < seg_end ? a.slot_row[base + cnt] : -1;
    }
    float msg[DN];
#pragma unroll
    for (int i = 0; i < DN; ++i) msg[i] = 0.f;
    if (valid) {
      // ---- edge MLP layer 0: stream the 6 input blocks through the accumulators
      float h[EH];
      load_bias<EH>(h, smem + W::OFF_EB0);
      float v[DN];
      const float* wt = smem + W::OFF_EW0;
      load_vec<DN / 4>(v, a.x_init + (int64_t)r * DN); dense_acc<DN, EH>(h, v, wt, 0);
      load_vec<DN / 4>(v, a.x_lat + (int64_t)r * DN);  dense_acc<DN, EH>(h, v, wt, DN);
      load_vec<DN / 4>(v, a.x_init + (int64_t)c * DN); dense_acc<DN, EH>(h, v, wt, 2 * DN);
      load_vec<DN / 4>(v, a.x_lat + (int64_t)c * DN);  dense_acc<DN, EH>(h, v, wt, 3 * DN);
      float ev[DE];
      load_vec<DE / 4>(ev, a.e_init + slot * DE);      dense_acc<DE, EH>(h, ev, wt, 4 * DN);
      load_vec<DE / 4>(ev, a.e_cur + slot * DE);       dense_acc<DE, EH>(h, ev, wt, 4 * DN + DE);
      relu_inplace(h);
      // ---- edge MLP layer 1
      float e2[DE];
      load_bias<DE>(e2, smem + W::OFF_EB1);
      dense_acc<EH, DE>(e2, h, smem + W::OFF_EW1);
      relu_inplace(e2);
      float4* dst = reinterpret_cast<float4*>(a.e_next + slot * DE);
#pragma unroll
      for (int q = 0; q < DE / 4; ++q) dst[q] = make_float4(e2[4 * q], e2[4 * q + 1], e2[4 * q + 2], e2[4 * q + 3]);
      // ---- classifier
      if (a.logits != nullptr) {
        float ch[CH];
        load_bias<CH>(ch, smem + W::OFF_CB0);
        dense_acc<DE, CH>(ch, e2, smem + W::OFF_CW0);
        relu_inplace(ch);
        float lg = smem[W::OFF_CB1];
#pragma unroll
        for (int i = 0; i < CH; ++i) lg = fmaf(ch[i], smem[W::OFF_CW1 + i], lg);
        a.logits[a.slot_edge[slot]] = lg;
      }
      // ---- flow MLP of this tile's direction on [x_init[c] | x_lat[c] | e']; x[c] is read again with plain loads:
      //      merged with the edge MLP's reads, it would stay live across layer 1 and the classifier (+58 registers)
      float g[FH];
      load_bias<FH>(g, smem + W::OFF_FB0);
      const float* wf = smem + W::OFF_FW0;
      load_vec<DN / 4, false>(v, a.x_init + (int64_t)c * DN); dense_acc<DN, FH>(g, v, wf, 0);
      load_vec<DN / 4, false>(v, a.x_lat + (int64_t)c * DN);  dense_acc<DN, FH>(g, v, wf, DN);
      dense_acc<DE, FH>(g, e2, wf, 2 * DN);
      relu_inplace(g);
      load_bias<DN>(msg, smem + W::OFF_FB1);
      dense_acc<FH, DN>(msg, g, smem + W::OFF_FW1);
      relu_inplace(msg);
    }
#pragma unroll
    for (int i = 0; i < DN; ++i) s_msg[tid * W::MSG_LD + i] = msg[i];
    __syncthreads();
    // ---- per-row sums, sequential in slot order; lane = feature
    if (tid < 32 && tid < DN) {
      const int f = tid;
      const int dir_off = dir_out ? DN : 0;                 // cat(flow_in, flow_out), mpn.py:97
      const int tile_id = tile_off + t;
      int seg_first_t = 0;
      int32_t cur = s_rows[1];
      float sum = 0.f;
      for (int q = 0; q <= cnt; ++q) {
        const int32_t rq = q < cnt ? s_rows[1 + q] : -2;
        if (rq != cur) {
          const bool starts_before = seg_first_t == 0 && s_rows[0] == cur;
          const bool continues = q == cnt && s_rows[TS + 1] == cur;
          if (!starts_before && !continues) {
            a.flow[(int64_t)cur * 2 * DN + dir_off + f] = sum;
          } else {
            a.part[((int64_t)tile_id * 2 + (seg_first_t == 0 ? 0 : 1)) * DN + f] = sum;
          }
          cur = rq; sum = 0.f; seg_first_t = q;
        }
        if (q < cnt) sum = a.agg == 2 ? fmaxf(sum, s_msg[q * W::MSG_LD + f]) : sum + s_msg[q * W::MSG_LD + f];
      }
    }
    __syncthreads();
  }
}

// x_next[r] = ReLU(Wn [flow_in(r) | flow_out(r)] + bn); one warp per node.
template <typename W>
__global__ void __launch_bounds__(256) mp_node_kernel(const int32_t* __restrict__ out_ptr,
                                                      const int32_t* __restrict__ in_ptr,
                                                      int64_t num_nodes, int64_t num_out,
                                                      int32_t tiles_out, const float* __restrict__ flow,
                                                      const float* __restrict__ part,
                                                      const float* __restrict__ node_w,
                                                      const float* __restrict__ node_b,
                                                      float* __restrict__ x_next, int agg) {
  constexpr int DN = W::DN;
  __shared__ float s_w[2 * DN * DN];   // Wt[in][out]
  __shared__ float s_b[DN];
  for (int idx = threadIdx.x; idx < 2 * DN * DN; idx += blockDim.x) {     // coalesced along a weight row
    const int o = idx / (2 * DN), i = idx - o * 2 * DN;
    s_w[i * DN + o] = node_w[idx];
  }
  for (int o = threadIdx.x; o < DN; o += blockDim.x) s_b[o] = node_b[o];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp; r < num_nodes; r += nwarps) {
    float fl[2];                       // fl[0] = flow_in[lane], fl[1] = flow_out[lane]
#pragma unroll
    for (int d = 0; d < 2; ++d) {
      const int32_t* ptr = d == 0 ? in_ptr : out_ptr;
      const int64_t seg_base = d == 0 ? num_out : 0;
      const int tile_off = d == 0 ? tiles_out : 0;
      const int64_t s0 = ptr[r], s1 = ptr[r + 1];
      float v = 0.f;
      if (s1 > s0 && lane < DN) {
        const int64_t ta = (s0 - seg_base) / TS, tb = (s1 - 1 - seg_base) / TS;
        if (ta == tb) {
          v = flow[r * 2 * DN + d * DN + lane];
        } else {
          const bool first_in_tile = (s0 - seg_base) % TS == 0;
          v = part[((tile_off + ta) * 2 + (first_in_tile ? 0 : 1)) * DN + lane];
          for (int64_t t = ta + 1; t <= tb; ++t) {
            const float u = part[((tile_off + t) * 2) * DN + lane];
            v = agg == 2 ? fmaxf(v, u) : v + u;
          }
        }
        if (agg == 1) v = v / (float)(s1 - s0);            // scatter_mean: sum / count (count >= 1 here)
      }
      fl[d] = v;
    }
    float acc = lane < DN ? s_b[lane] : 0.f;
#pragma unroll
    for (int d = 0; d < 2; ++d)
#pragma unroll
      for (int i = 0; i < DN; ++i) {
        const float xi = __shfl_sync(0xffffffffu, fl[d], i);
        if (lane < DN) acc = fmaf(xi, s_w[(d * DN + i) * DN + lane], acc);
      }
    if (lane < DN) x_next[r * DN + lane] = fmaxf(acc, 0.f);
  }
}

// logits[slot_edge[s]] = classifier(e[s])  (num_enc_steps == 0, models/mpn.py:387-389)
template <typename W>
__global__ void classify_kernel(const float* __restrict__ e, const int32_t* __restrict__ slot_edge,
                                int64_t num_edges, mpn_core_weights w, float* __restrict__ logits) {
  constexpr int DE = W::DE, CH = W::CH;
  __shared__ __align__(16) float s_w0[DE * CH];
  __shared__ __align__(16) float s_b0[CH];
  __shared__ float s_w1[CH];
  stage_weight_t<DE, CH>(w.cls_w0, s_w0);
  stage_bias<CH>(w.cls_b0, s_b0);
  for (int i = threadIdx.x; i < CH; i += blockDim.x) s_w1[i] = w.cls_w1[i];
  __syncthreads();
  const float b1 = w.cls_b1[0];
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < num_edges;
       s += (int64_t)gridDim.x * blockDim.x) {
    float ev[DE], ch[CH];
    load_vec<DE / 4>(ev, e + s * DE);
    load_bias<CH>(ch, s_b0);
    dense_acc<DE, CH>(ch, ev, s_w0);
    relu_inplace(ch);
    float lg = b1;
#pragma unroll
    for (int i = 0; i < CH; ++i) lg = fmaf(ch[i], s_w1[i], lg);
    logits[slot_edge[s]] = lg;
  }
}

using Shipped = CoreWidths<32, 16, 80, 56, 8>;

static bool is_shipped(const mpn_core_weights* w) {
  return w->dn == 32 && w->de == 16 && w->edge_h == 80 && w->flow_h == 56 && w->cls_h == 8;
}

struct MpWorkspace {
  float* x_lat[2];
  float* e_state;
  float* flow;
  float* part;
};

static int64_t carve_workspace(void* ws, int64_t n, int64_t e, int dn, int de, MpWorkspace* out) {
  Carver cv(ws);
  const int64_t tiles = ceil_div(e, TS) + 2;
  float* x0 = cv.take<float>(n * dn);
  float* x1 = cv.take<float>(n * dn);
  float* es = cv.take<float>(e * de);
  float* fl = cv.take<float>(n * 2 * dn);
  float* pt = cv.take<float>(tiles * 2 * dn);
  if (out) { out->x_lat[0] = x0; out->x_lat[1] = x1; out->e_state = es; out->flow = fl; out->part = pt; }
  return cv.off;
}

}  // namespace mpn

using namespace mpn;

extern "C" {

int64_t mpn_mp_workspace(int64_t n, int64_t e) {
  return carve_workspace(nullptr, n > 0 ? n : 1, e > 0 ? e : 1, 32, 16, nullptr) + 256;
}

}  // extern "C"

namespace mpn {

static int check_core(const mpn_core_weights* w, const mpn_edge_layout* g, const char* who) {
  MPN_CHECK_ARG(w && g, "%s: null descriptor", who);
  MPN_CHECK_ARG(w->node_agg >= 0 && w->node_agg <= 2, "%s: node_agg must be 0 (sum), 1 (mean) or 2 (max)", who);
  MPN_CHECK_ARG(is_shipped(w), "%s: fused kernels are built for widths dn=32 de=16 edge_h=80 "
                "flow_h=56 cls_h=8 (got %d %d %d %d %d)", who, w->dn, w->de, w->edge_h, w->flow_h, w->cls_h);
  return MPN_OK;
}

// One launch pair. e_next may alias e_cur. logits_row: this step's row of the output or NULL.
static int launch_step(const mpn_core_weights* w, const mpn_edge_layout* g, const MpWorkspace& m,
                       const float* x_init, const float* x_cur, const float* e_init, const float* e_cur,
                       float* e_next, float* x_next, float* logits_row, cudaStream_t s) {
  using W = Shipped;
  const int64_t n = g->num_nodes, e = g->num_edges;
  MPN_CUDA(cudaFuncSetAttribute(mp_edge_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)W::SMEM_BYTES));
  const int tiles_out = (int)ceil_div(g->num_out, TS);
  const int tiles_in = (int)ceil_div(e - g->num_out, TS);
  const int total_tiles = tiles_out + tiles_in;
  int grid = sm_count() * 2;
  if (grid > total_tiles) grid = total_tiles;
  if (tiles_out > 0 && tiles_in > 0 && grid < 2) grid = 2;
  if (e > 0) {
    StepArgs a;
    a.slot_row = g->slot_row; a.slot_col = g->slot_col; a.slot_edge = g->slot_edge;
    a.num_edges = e; a.num_out = g->num_out; a.tiles_out = tiles_out; a.tiles_in = tiles_in;
    a.x_init = x_init; a.x_lat = x_cur; a.e_init = e_init; a.e_cur = e_cur; a.e_next = e_next;
    a.flow = m.flow; a.part = m.part; a.logits = logits_row; a.agg = w->node_agg;
    if (profiling()) profile_mark(0, true, s);
    mp_edge_kernel<W><<<grid, TS, W::SMEM_BYTES, s>>>(a, *w); count_launch();
    if (profiling()) profile_mark(0, false, s);
  }
  if (n > 0) {
    const unsigned ngrid = (unsigned)std::min<int64_t>(ceil_div(n * 32, 256), (int64_t)sm_count() * 8);
    if (profiling()) profile_mark(1, true, s);
    mp_node_kernel<W><<<ngrid, 256, 0, s>>>(g->out_ptr, g->in_ptr, n, g->num_out, tiles_out, m.flow,
                                            m.part, w->node_w, w->node_b, x_next, w->node_agg); count_launch();
    if (profiling()) profile_mark(1, false, s);
  }
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // namespace mpn

extern "C" {

int mpn_mp_forward(const mpn_core_weights* w, const mpn_edge_layout* g, const float* x_init,
                   const float* e_init, int32_t num_steps, int32_t first_class_step, void* ws,
                   float* logits, float* x_out, float* e_out, void* stream) {
  int rc = check_core(w, g, "mp_forward");
  if (rc) return rc;
  MPN_CHECK_ARG(num_steps >= 0, "mp_forward: num_steps < 0");
  using W = Shipped;
  const int64_t n = g->num_nodes, e = g->num_edges;
  cudaStream_t s = as_stream(stream);
  if (e == 0 && n == 0) return MPN_OK;
  MPN_CHECK_ARG(ws != nullptr, "mp_forward: null workspace");
  MpWorkspace m;
  carve_workspace(ws, n > 0 ? n : 1, e > 0 ? e : 1, W::DN, W::DE, &m);

  if (num_steps == 0) {
    if (e > 0 && logits) {
      classify_kernel<W><<<(unsigned)std::min<int64_t>(ceil_div(e, 256), (int64_t)sm_count() * 8), 256, 0, s>>>(
          e_init, g->slot_edge, e, *w, logits); count_launch();
      MPN_LAUNCH_CHECK();
    }
    if (x_out && n > 0) MPN_CUDA(cudaMemcpyAsync(x_out, x_init, sizeof(float) * n * W::DN, cudaMemcpyDeviceToDevice, s));
    if (e_out && e > 0) MPN_CUDA(cudaMemcpyAsync(e_out, e_init, sizeof(float) * e * W::DE, cudaMemcpyDeviceToDevice, s));
    return MPN_OK;
  }

  const float* x_cur = x_init;      // before step 1 the latent state is the initial encoding
  const float* e_cur = e_init;      // (models/mpn.py:358-359)
  for (int step = 1; step <= num_steps; ++step) {
    float* x_next = (step == num_steps && x_out) ? x_out : m.x_lat[step & 1];
    float* e_next = (step == num_steps && e_out) ? e_out : m.e_state;
    float* row = (logits && step >= first_class_step) ? logits + (int64_t)(step - first_class_step) * e : nullptr;
    rc = launch_step(w, g, m, x_init, x_cur, e_init, e_cur, e_next, x_next, row, s);
    if (rc) return rc;
    x_cur = x_next;
    e_cur = e_next;
  }
  return MPN_OK;
}

}  // extern "C"
