// Fused message-passing step on the 5th-gen tensor cores (tcgen05, sm_100a).
//
// One 128-edge tile = one M=128 MMA tile: TMEM lane i <-> edge slot i <-> epilogue thread i.
// The four dense layers of a step (edge MLP 160->80->16, flow MLP 80->56->32) run as
// tcgen05.mma kind::f16 with the ACTIVATIONS as the A operand (in TMEM, written by the epilogue
// threads with tcgen05.st; the gathered x[col] rows in shared memory, written by TMA) and the
// WEIGHTS resident in shared memory (B operand, K-major).
// Precision: every operand is split v ~= hi + lo in fp16 (22 significant bits; the low part is stored lifted by
// 2^10 so that it stays a normal number, tc_ptx.cuh "lifted low part") and each layer issues lo*hi + hi*lo for
// all K steps, folds them in with the accumulator input scale 2^-10, then hi*hi, with fp32 accumulation in TMEM -- single-pass bf16/tf32 breaks
// the 1e-3 parity bar after 12 recurrent steps, bf16 hi/lo is 10-20x less accurate than fp16
// hi/lo (tools/emulate_split_bf16.py).  fp16 range overflow (> 65504) is detected and reported
// through `status`; the caller then reruns on the fp32 kernels (mp_step.cu).
//
//   x[row] part of edge layer 0 is hoisted: prow[r] = W0[:, 0:64] [x_init[r] | x_lat[r]] + b0
//   (fp32, computed by the node kernel), added in the first epilogue.
//
// State lives in HBM already split: per node 128 B = [hi(32 halfs) | lo(32 halfs)], per edge
// 64 B = [hi(16) | lo(16)], so loads are plain copies into the operands and the bytes per
// edge-update stay at 200.
//
// Warp roles (768 threads, 1 CTA / SM): three groups of 8 warps; each group keeps one tile in flight
// and owns 144 of the 512 TMEM columns and 48 KB of shared memory.  Every edge row is served by two
// threads (halves A and B of the group) that split the columns of each epilogue.  After the group's
// 256 threads have written a layer's operand, an elected lane of the group's first warp issues that
// layer's MMAs and commits them to the group's mbarrier; while one group runs an epilogue the tensor
// core runs another group's layer.  The x[col] rows of the next tile are gathered by TMA during the
// current one, and its layer 1 is issued as soon as the current tile's layer 4 has retired, so the
// last epilogue and the per-row message sums run under it.
#include <cuda.h>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace mpn {
namespace tc {

using namespace ptx;

constexpr int TS = 128;
constexpr int DN = 32, DE = 16, EH = 80, FH = 56, FHP = 64, CH = 8;

// ---- shared-memory weight image (bytes). Slab = one K=16 step of a B operand: [n/8][k/8][n%8][8 halfs]
constexpr int L1_KS = 6, L1_SLAB = EH * 32;
constexpr int L2_KS = 5, L2_SLAB = DE * 32;
constexpr int L3_KS = 5, L3_SLAB = FHP * 32;
constexpr int L4_KS = 4, L4_SLAB = DN * 32;
constexpr int OFF_L1H = 0, OFF_L1L = OFF_L1H + L1_KS * L1_SLAB;
constexpr int OFF_L2H = OFF_L1L + L1_KS * L1_SLAB, OFF_L2L = OFF_L2H + L2_KS * L2_SLAB;
constexpr int OFF_L3H = OFF_L2L + L2_KS * L2_SLAB, OFF_L3L = OFF_L3H + L3_KS * L3_SLAB;
constexpr int OFF_L4H = OFF_L3L + L3_KS * L3_SLAB, OFF_L4L = OFF_L4H + L4_KS * L4_SLAB;
constexpr int OFF_F32 = OFF_L4L + L4_KS * L4_SLAB;          // fp32 tail
constexpr int F_B1 = 0, F_FB0 = F_B1 + DE, F_FB1 = F_FB0 + FHP, F_CW0 = F_FB1 + DN, F_CB0 = F_CW0 + DE * CH,
              F_CW1 = F_CB0 + CH, F_CB1 = F_CW1 + CH, F_COUNT = F_CB1 + 4;
constexpr int IMG_BYTES = (OFF_F32 + F_COUNT * 4 + 127) / 128 * 128;
// ---- weight image of the node kernel: node Linear 64 -> 32 (K steps 0..3) and the hoisted row term 32 -> 80 (K steps 0..1)
constexpr int NW_KS = 4, NW_SLAB = DN * 32;
constexpr int PW_KS = 2, PW_SLAB = EH * 32;
constexpr int NOFF_NWH = 0, NOFF_NWL = NOFF_NWH + NW_KS * NW_SLAB;
constexpr int NOFF_PWH = NOFF_NWL + NW_KS * NW_SLAB, NOFF_PWL = NOFF_PWH + PW_KS * PW_SLAB;
constexpr int NOFF_F32 = NOFF_PWL + PW_KS * PW_SLAB;       // bn[32]
constexpr int NIMG_BYTES = (NOFF_F32 + DN * 4 + 127) / 128 * 128;

// =================================================================== range bookkeeping
// Per forward: sched[t] = s_t (exponent of the step's scale), amax[t] = float bits of the largest true activation
// the edge kernel of step t saw, xmax[t] = largest |x_lat| consumed by step t (t = 1..num_steps; all zeroed at start);
// amax[0] = largest |x_init|, |e_init| (the constant rows, recorded by prep_nodes_kernel and split_edges_kernel);
// fmax[t] = largest flow row sum (or granule partial) the edge kernel of step t wrote.
constexpr int MAX_STEPS = 1000;
// The lifted low halves keep 22 bits for any operand whose high half is a normal fp16 number (>= 2^-14), so the scale
// can leave generous headroom at no cost in precision: the lagged maximum is brought to <= 2^6 (1024x headroom for the
// growth of one step); values down to 2^-20 of the maximum still have all their bits.
constexpr float SCALE_TARGET = 64.f;
constexpr int INIT_SHIFT = 8;                // the constant x_init / e_init rows are stored x 2^-8, their weight slabs carry 2^(8 - s_t):
                                             // the slabs stay normal fp16 numbers for s_t up to 22 (values up to ~2.7e8); beyond that the
                                             // constant-row terms fade out (they are < 2^-22 of the latent terms there)
// Resolution floor: a value carried as v x 2^-s keeps 22 bits only while its high half is a normal fp16 number; below
// that both halves are subnormal and the absolute resolution is 2^(s - 34), the same for every row of the batch.  Above
// s = 17 that floor, carried through the recurrence, reaches the 1e-3 parity bar for rows whose own values are of
// order 1 (a quiet window batched with a loud one: its logit error triples at s = 19 and is 7x the bar at s = 22, on
// a B200).  Such a step sets status bit 2, which sends engine 'auto' to the fp32 kernels like an fp16 overflow.
constexpr int S_RESOLVED = 17;
// The constant rows are stored x 2^-INIT_SHIFT once per forward, whatever the step scale (which never goes below 0), so
// they have the same floor: below 2^-14 stored their absolute resolution is 2^-34 (2^-26 in true units).  They are
// resolved as S_RESOLVED resolves rows of order 1 -- floor at most 2^-17 of the value -- when the largest stored
// |x_init|, |e_init| is at least 2^(S_RESOLVED - 34); a smaller nonzero maximum sets status bit 2 (all-zero rows are exact).
__device__ __forceinline__ bool init_rows_unresolved(float init_max) {
  const float m = init_max * pow2i(-INIT_SHIFT);
  return m > 0.f && m < pow2i(S_RESOLVED - 34);
}
constexpr int FLOW_SHIFT = 7;                // a flow vector sums up to ~100 messages: operand scale 2^-(s_t + 7)
// Flows far below that (a flow MLP whose output layer is small next to the rest of the network) would leave their low
// bits to fp16 subnormals in the node Linear's operand.  When the largest flow piece of the step lies below 2^-FLOW_LIFT
// there, the node kernel lowers the flow scale so that it lands in [2^-5, 2^-4) (exact: powers of two, fp32 epilogue).
constexpr int FLOW_LIFT = 10;
// s_{t+1} from what is known when the node kernel of step t starts: the edge kernel's activation maximum of step t
// and the node-state maxima of steps t and t-1 (their ratio predicts the growth of the state being produced).
__device__ __forceinline__ int scale_for(float a_t, float x_t, float x_tm1) {
  float growth = x_tm1 > 0.f ? x_t / x_tm1 : 4.f;
  growth = fminf(fmaxf(growth, 1.f), 64.f);
  const float lag = fmaxf(a_t, x_t * growth);
  if (!(lag > SCALE_TARGET)) return 0;
  int e;
  frexpf(lag / SCALE_TARGET, &e);       // lag / target = m * 2^e, m in [0.5, 1)
  return e > 100 ? 100 : e;
}
__device__ __forceinline__ void atomic_max_f32(uint32_t* addr, float v) {   // v >= 0: integer order = float order
  const uint32_t m = __reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(v, 0.f)));
  if ((threadIdx.x & 31) == 0 && m != 0u) atomicMax(addr, m);
}

// =================================================================== weight packing (once per forward)
// One image per direction (flow_out / flow_in); layers 1-2 and the classifier are shared.
__global__ void pack_weights_kernel(mpn_core_weights w, uint8_t* __restrict__ img_out, uint8_t* __restrict__ img_in,
                                    uint8_t* __restrict__ img_node, int32_t* __restrict__ status) {
  // bad: a weight whose fp16 image, times the largest factor its slab carries (2^INIT_SHIFT for the constant-row slabs,
  // 1 elsewhere), is not finite; or a non-finite bias or fp32 tail weight
  int bad = 0;
  auto fits = [&](float v, float f) { if (!(fabsf(v) * f < 65000.f)) bad = 1; };
  auto finite = [&](float v) { if (!isfinite(v)) bad = 1; };
  const float init_f = pow2i(INIT_SHIFT);
  {
    auto putn = [&](int off_h, int off_l, int slab_bytes, int n, int k, float v) {
      const __half h = __float2half_rn(v);
      const __half l = __float2half_rn((v - __half2float(h)) * LO_SCALE);
      const int o = (k >> 4) * slab_bytes + slab_off(n, k & 15);
      *reinterpret_cast<__half*>(img_node + off_h + o) = h;
      *reinterpret_cast<__half*>(img_node + off_l + o) = l;
    };
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int i = tid; i < DN * 2 * DN; i += nt) { fits(w.node_w[i], 1.f); putn(NOFF_NWH, NOFF_NWL, NW_SLAB, i / (2 * DN), i % (2 * DN), w.node_w[i]); }
    for (int i = tid; i < EH * DN; i += nt) {            // edge layer 0, input columns 32..63 (x_lat[row])
      const int n = i / DN, k = i % DN;
      fits(w.edge_w0[n * 160 + 32 + k], 1.f);
      putn(NOFF_PWH, NOFF_PWL, PW_SLAB, n, k, w.edge_w0[n * 160 + 32 + k]);
    }
    for (int i = tid; i < DN; i += nt) { finite(w.node_b[i]); reinterpret_cast<float*>(img_node + NOFF_F32)[i] = w.node_b[i]; }
  }
  for (int dir = 0; dir < 2; ++dir) {
    uint8_t* img = dir == 0 ? img_out : img_in;
    const float* f0 = dir == 0 ? w.fout_w0 : w.fin_w0;
    const float* f1 = dir == 0 ? w.fout_w1 : w.fin_w1;
    const float* fb0 = dir == 0 ? w.fout_b0 : w.fin_b0;
    const float* fb1 = dir == 0 ? w.fout_b1 : w.fin_b1;
    auto put = [&](int off_h, int off_l, int slab_bytes, int n, int k, float v, float f) {
      fits(v, f);
      const __half h = __float2half_rn(v);
      const __half l = __float2half_rn((v - __half2float(h)) * LO_SCALE);
      const int o = (k >> 4) * slab_bytes + slab_off(n, k & 15);
      *reinterpret_cast<__half*>(img + off_h + o) = h;
      *reinterpret_cast<__half*>(img + off_l + o) = l;
    };
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    for (int i = tid; i < EH * 96; i += nt) {            // edge layer 0, input columns 64..159
      const int n = i / 96, k = i % 96, ks = k >> 4;     // K steps 0, 1 (x_init[col]) and 4 (e_init): constant rows
      put(OFF_L1H, OFF_L1L, L1_SLAB, n, k, w.edge_w0[n * 160 + 64 + k], ks <= 1 || ks == 4 ? init_f : 1.f);
    }
    for (int i = tid; i < DE * EH; i += nt) {            // edge layer 1
      const int n = i / EH, k = i % EH;
      put(OFF_L2H, OFF_L2L, L2_SLAB, n, k, w.edge_w1[n * EH + k], 1.f);
    }
    for (int i = tid; i < FHP * 80; i += nt) {           // flow layer 0 (rows padded 56 -> 64)
      const int n = i / 80, k = i % 80;
      // rows 56..63 are padding for the flow MLP; the edge kernel puts the classifier's first layer there (it reads
      // only the e' K step, columns 64..79)
      float v = n < FH ? f0[n * 80 + k] : 0.f;
      if (n >= FH && k >= 64) v = w.cls_w0[(n - FH) * DE + (k - 64)];
      put(OFF_L3H, OFF_L3L, L3_SLAB, n, k, v, k < DN ? init_f : 1.f);   // K steps 0, 1: x_init[col]
    }
    for (int i = tid; i < DN * FHP; i += nt) {           // flow layer 1 (K padded 56 -> 64)
      const int n = i / FHP, k = i % FHP;
      put(OFF_L4H, OFF_L4L, L4_SLAB, n, k, k < FH ? f1[n * FH + k] : 0.f, 1.f);
    }
    float* ft = reinterpret_cast<float*>(img + OFF_F32);
    for (int i = tid; i < F_COUNT; i += nt) {
      float v = 0.f;
      if (i < F_FB0) v = w.edge_b1[i - F_B1];
      else if (i < F_FB1) v = (i - F_FB0) < FH ? fb0[i - F_FB0] : 0.f;
      else if (i < F_CW0) v = fb1[i - F_FB1];
      else if (i < F_CB0) { const int q = i - F_CW0, in = q / CH, o = q % CH; v = w.cls_w0[o * DE + in]; }
      else if (i < F_CW1) v = w.cls_b0[i - F_CB0];
      else if (i < F_CB1) v = w.cls_w1[i - F_CW1];
      else if (i == F_CB1) v = w.cls_b1[0];
      finite(v);
      ft[i] = v;
    }
  }
  if (bad) atomicOr(status, 1);
}

// =================================================================== node-side kernels
__device__ __forceinline__ void store_split_row(__half* __restrict__ row64, int lane, float v, int* ovf) {
  const __half h = __float2half_rn(v);
  const __half l = __float2half_rn((v - __half2float(h)) * LO_SCALE);
  row64[lane] = h;
  row64[32 + lane] = l;
  if (!(fabsf(v) < 65000.f)) *ovf = 1;
}

// Once per forward: split x_init, and the hoisted row terms
//   pinit[r] = W0[:, 0:32] x_init[r] + b0 ; prow[r] = pinit[r] + W0[:, 32:64] x_init[r]  (x_lat = x_init before step 1)
__global__ void __launch_bounds__(256) prep_nodes_kernel(const float* __restrict__ x_init, int64_t n,
                                                         const float* __restrict__ w0, const float* __restrict__ b0,
                                                         __half* __restrict__ xi, __half* __restrict__ xl0,
                                                         float* __restrict__ pinit, float* __restrict__ prow,
                                                         uint32_t* __restrict__ xmax, uint32_t* __restrict__ init_max,
                                                         int32_t* __restrict__ status) {
  __shared__ float s_w[64 * EH];     // [i][o], i over W0 columns 0..63
  __shared__ float s_b[EH];
  int ovf = 0;                       // also a non-finite W0[:, 0:64] or b0: they enter the hoisted row term in fp32, unchecked elsewhere
  for (int idx = threadIdx.x; idx < 64 * EH; idx += blockDim.x) {        // coalesced along a weight row
    const int o = idx / 64, i = idx - o * 64;
    const float v = w0[o * 160 + i];
    if (!isfinite(v)) ovf = 1;
    s_w[i * EH + o] = v;
  }
  for (int o = threadIdx.x; o < EH; o += blockDim.x) { s_b[o] = b0[o]; if (!isfinite(s_b[o])) ovf = 1; }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  float mx = 0.f;
  for (int64_t r = warp; r < n; r += nwarps) {
    const float v = x_init[r * DN + lane];
    mx = fmaxf(mx, fabsf(v));
    store_split_row(xi + r * 64, lane, v * pow2i(-INIT_SHIFT), &ovf);
    store_split_row(xl0 + r * 64, lane, v, &ovf);
    float a0[3], a1[3];
#pragma unroll
    for (int q = 0; q < 3; ++q) { const int o = lane + 32 * q; a0[q] = o < EH ? s_b[o] : 0.f; a1[q] = 0.f; }
#pragma unroll
    for (int i = 0; i < DN; ++i) {
      const float xv = __shfl_sync(0xffffffffu, v, i);
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const int o = lane + 32 * q;
        if (o < EH) { a0[q] = fmaf(xv, s_w[i * EH + o], a0[q]); a1[q] = fmaf(xv, s_w[(32 + i) * EH + o], a1[q]); }
      }
    }
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const int o = lane + 32 * q;
      if (o < EH) { pinit[r * EH + o] = a0[q]; prow[r * EH + o] = a0[q] + a1[q]; }
    }
  }
  atomic_max_f32(xmax + 1, mx);                                         // the state consumed by step 1 (scale s_1 = 0)
  atomic_max_f32(init_max, mx);
  if (ovf) atomicOr(status, 1);
}

// Per step: x' = ReLU(Wn [flow_in | flow_out] + bn)  (models/mpn.py:97-99), then the split copy of
// x' for the next step's gathers and prow[r] = pinit[r] + W0[:, 32:64] x'.
//
// Tile = 128 nodes, TMEM lane = node = thread; two groups of 4 warps per CTA, one tile in flight each.  A thread
// gathers its node's two flow vectors (the row sum, or the granule partials added in granule order), splits them
// into the A operand in TMEM, the node Linear runs as 12 MMAs (N = 32),
// the epilogue writes x' (fp32 on the last step, split rows in the next step's scale) and leaves the scaled split x'
// in TMEM as the A operand of the hoisted row term (6 MMAs, N = 80), whose epilogue adds pinit and stores prow.
constexpr int NT2_THREADS = 256;
constexpr int N2_A1H = 0, N2_A1L = 32, N2_D1 = 64, N2_D2 = 96, N2_COLS = 176;
constexpr int NSM_BAR = (NIMG_BYTES + 15) / 16 * 16, NSM_TMEM = NSM_BAR + 2 * 8, NSMEM_BYTES = NSM_TMEM + 16;

__global__ void __launch_bounds__(NT2_THREADS, 1) node_tc2_kernel(
    const int32_t* __restrict__ out_ptr, const int32_t* __restrict__ in_ptr, int64_t num_nodes, int64_t num_out,
    int32_t chunks_out, int chunk_shift, const float* __restrict__ flow, const float* __restrict__ part,
    const uint8_t* __restrict__ wimg, const float* __restrict__ pinit, uint4* __restrict__ xl_next,
    float* __restrict__ prow, float* __restrict__ x_out, int32_t step, int32_t* __restrict__ sched,
    const uint32_t* __restrict__ amax, uint32_t* __restrict__ xmax, const uint32_t* __restrict__ fmax, int32_t agg,
    int32_t* __restrict__ status) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + NSM_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + NSM_TMEM);
  // scale inputs first: their latency overlaps the image copy
  const float a_t = __uint_as_float(amax[step]), x_t = __uint_as_float(xmax[step]);
  const float x_tm1 = step > 1 ? __uint_as_float(xmax[step - 1]) : 0.f;
  for (int i = tid; i < NIMG_BYTES / 16; i += NT2_THREADS)
    reinterpret_cast<uint4*>(smem)[i] = __ldg(reinterpret_cast<const uint4*>(wimg) + i);
  if (tid == 0) { mbar_init(&bars[0], 1); mbar_init(&bars[1], 1); mbar_fence_init(); }
  if (warp == 0) tmem_alloc<512>(tmem_slot);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tmem_slot;
  const int s_next = scale_for(a_t, x_t, x_tm1);
  const float sig_next = pow2i(-s_next);
  if (blockIdx.x == 0 && tid == 0) sched[step + 1] = s_next;
  // the flow vectors enter the node Linear in the scale of the step that produced the messages, 2^-FLOW_SHIFT lower,
  // or lifted (FLOW_LIFT)
  int s_flow = sched[step] + FLOW_SHIFT;
  {
    const float f_op = __uint_as_float(fmax[step]) * pow2i(-s_flow);
    if (f_op > 0.f && f_op < pow2i(-FLOW_LIFT)) {
      int e;
      frexpf(f_op, &e);                                                  // f_op in [2^(e-1), 2^e)
      s_flow = max(s_flow + e + 4, -100);
    }
  }
  const float sig_flow = pow2i(-s_flow), inv_sig_flow = pow2i(s_flow);

  const int g = warp >> 2, wq = warp & 3;
  const uint32_t tcol = __shfl_sync(0xffffffffu, tbase, 0) + (uint32_t)g * N2_COLS;
  const uint32_t tlane = tcol + ((uint32_t)(wq * 32) << 16);
  uint64_t* d_ready = &bars[g];
  uint32_t pd = 0;
  const float* s_bn = reinterpret_cast<const float*>(smem + NOFF_F32);
  const uint64_t dzero = smem_desc_kmajor(0, 128, 256);
  const uint32_t img = smem_u32(smem);
  const int64_t gmask = ((int64_t)1 << chunk_shift) - 1;
  float mx = 0.f;
  int ovf = 0;

  auto issue = [&](int layer) {                                         // after the group's operands are in TMEM
    tc_wait_st();
    tc_fence_before();
    named_barrier(1 + g, 128);
    if (wq == 0) {
      tc_fence_after();
      if (elect_one()) {
        auto bd = [&](int off) { return dzero + (uint64_t)((img + off) >> 4); };
        if (layer == 1) {
          constexpr uint32_t id = idesc_f16(128, DN);
#pragma unroll
          for (int ks = 0; ks < NW_KS; ++ks) {
            mma_ts(tcol + N2_D1, tcol + N2_A1L + 8 * ks, bd(NOFF_NWH + ks * NW_SLAB), id, ks == 0 ? 0u : 1u);
            mma_ts(tcol + N2_D1, tcol + N2_A1H + 8 * ks, bd(NOFF_NWL + ks * NW_SLAB), id, 1u);
          }
          mma_ts_sd(tcol + N2_D1, tcol + N2_A1H, bd(NOFF_NWH), id);
#pragma unroll
          for (int ks = 1; ks < NW_KS; ++ks) mma_ts(tcol + N2_D1, tcol + N2_A1H + 8 * ks, bd(NOFF_NWH + ks * NW_SLAB), id, 1u);
        } else {
          constexpr uint32_t id = idesc_f16(128, EH);
#pragma unroll
          for (int ks = 0; ks < PW_KS; ++ks) {
            mma_ts(tcol + N2_D2, tcol + N2_D1 + 16 + 8 * ks, bd(NOFF_PWH + ks * PW_SLAB), id, ks == 0 ? 0u : 1u);
            mma_ts(tcol + N2_D2, tcol + N2_D1 + 8 * ks, bd(NOFF_PWL + ks * PW_SLAB), id, 1u);
          }
          mma_ts_sd(tcol + N2_D2, tcol + N2_D1, bd(NOFF_PWH), id);
          mma_ts(tcol + N2_D2, tcol + N2_D1 + 8, bd(NOFF_PWH + PW_SLAB), id, 1u);
        }
        mma_commit(d_ready);
      }
      __syncwarp();
    }
  };
  // 32 floats of one row (128 B, per-thread contiguous)
  auto load_row = [&](const float* p, float (&v)[DN]) {
#pragma unroll
    for (int q = 0; q < DN / 4; ++q) {
      const float4 t = *reinterpret_cast<const float4*>(p + 4 * q);
      v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
    }
  };
  // one direction's flow vector of node r -> split halves -> A operand columns [col_h, col_h + 16), [col_l, col_l + 16).
  // The first three pieces (row sum, or granule partials) are loaded together from always-valid addresses and masked,
  // so that their latencies overlap; rows that span more than three granules (degree > 32) take the loop.
  auto gather_flow = [&](int64_t r, int d, int64_t s0, int64_t s1, bool live, int col_h, int col_l) {
    const int64_t seg_base = d == 0 ? num_out : 0;
    const int64_t chunk_off = d == 0 ? chunks_out : 0;
    const bool has = live && s1 > s0;
    const int64_t rel0 = s0 - seg_base;
    const int64_t ca = rel0 >> chunk_shift, cb = has ? (s1 - 1 - seg_base) >> chunk_shift : ca;
    const int64_t more = cb - ca;
    const bool first_in_chunk = (rel0 & gmask) == 0;
    const float* p0 = more == 0 ? flow + r * 2 * DN + d * DN : part + ((chunk_off + ca) * 2 + (first_in_chunk ? 0 : 1)) * DN;
    const float* pp = part + ((chunk_off + ca + 1) * 2) * DN;
    float v[DN], u1[DN], u2[DN];
    load_row(has ? p0 : flow, v);
    load_row(has && more >= 1 ? pp : flow, u1);
    load_row(has && more >= 2 ? pp + 2 * DN : flow, u2);
    const bool k1 = has && more >= 1, k2 = has && more >= 2;
    if (agg == 2) {
#pragma unroll
      for (int i = 0; i < DN; ++i) v[i] = fmaxf(fmaxf(has ? v[i] : 0.f, k1 ? u1[i] : 0.f), k2 ? u2[i] : 0.f);
    } else {
#pragma unroll
      for (int i = 0; i < DN; ++i) v[i] = ((has ? v[i] : 0.f) + (k1 ? u1[i] : 0.f)) + (k2 ? u2[i] : 0.f);   // + 0 is exact: granule order kept
    }
    for (int64_t t = ca + 3; t <= cb; ++t) {
      load_row(part + ((chunk_off + t) * 2) * DN, u1);
#pragma unroll
      for (int i = 0; i < DN; ++i) v[i] = agg == 2 ? fmaxf(v[i], u1[i]) : v[i] + u1[i];
    }
    if (agg == 1 && has) {                                              // scatter_mean: sum / count
      const float inv = 1.f / (float)(s1 - s0);
#pragma unroll
      for (int i = 0; i < DN; ++i) v[i] *= inv;
    }
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float a = v[2 * j] * sig_flow, b = v[2 * j + 1] * sig_flow;
      split2s(a, b, hi[j], lo[j]);
      if (!(fmaxf(a, b) < 65000.f)) ovf = 1;
    }
    const uint32_t h0[8] = {hi[0], hi[1], hi[2], hi[3], hi[4], hi[5], hi[6], hi[7]};
    const uint32_t h1[8] = {hi[8], hi[9], hi[10], hi[11], hi[12], hi[13], hi[14], hi[15]};
    const uint32_t l0[8] = {lo[0], lo[1], lo[2], lo[3], lo[4], lo[5], lo[6], lo[7]};
    const uint32_t l1[8] = {lo[8], lo[9], lo[10], lo[11], lo[12], lo[13], lo[14], lo[15]};
    tmem_st8(tlane + col_h, h0); tmem_st8(tlane + col_h + 8, h1);
    tmem_st8(tlane + col_l, l0); tmem_st8(tlane + col_l + 8, l1);
  };

  const int64_t tiles = (num_nodes + TS - 1) / TS;
  for (int64_t t = (int64_t)blockIdx.x * 2 + g; t < tiles; t += (int64_t)gridDim.x * 2) {
    const int64_t r = t * TS + wq * 32 + lane;
    const bool live = r < num_nodes;
    const int64_t rc = live ? r : num_nodes - 1;
    const int32_t i0 = in_ptr[rc], i1 = in_ptr[rc + 1], o0 = out_ptr[rc], o1 = out_ptr[rc + 1];
    // ---- flows -> A operand: K order [flow_in | flow_out] (models/mpn.py:97)
    gather_flow(rc, 0, i0, i1, live, N2_A1H, N2_A1L);
    gather_flow(rc, 1, o0, o1, live, N2_A1H + 16, N2_A1L + 16);
    issue(1);
    // the hoisted-term inputs of this node: all 20 loads in flight while the node Linear runs
    float pin[EH];
#pragma unroll
    for (int q = 0; q < EH / 4; ++q) {
      const float4 v = *reinterpret_cast<const float4*>(pinit + rc * EH + 4 * q);
      pin[4 * q] = v.x; pin[4 * q + 1] = v.y; pin[4 * q + 2] = v.z; pin[4 * q + 3] = v.w;
    }
    // ---- epilogue 1: x' = ReLU(D1 + bn); split rows in the next step's scale (global + A operand of the row term)
    mbar_wait(d_ready, pd); pd ^= 1;
    tc_fence_after();
    {
      uint32_t acc[32];
      tmem_ld16(tlane + N2_D1, *reinterpret_cast<uint32_t(*)[16]>(&acc[0]));
      tmem_ld16(tlane + N2_D1 + 16, *reinterpret_cast<uint32_t(*)[16]>(&acc[16]));
      tc_wait_ld();
      float xn[DN];
#pragma unroll
      for (int i = 0; i < DN; ++i) { xn[i] = fmaxf(fmaf(__uint_as_float(acc[i]), inv_sig_flow, s_bn[i]), 0.f); mx = live ? fmaxf(mx, xn[i]) : mx; }
      if (live && x_out != nullptr) {
#pragma unroll
        for (int q = 0; q < DN / 4; ++q)
          reinterpret_cast<float4*>(x_out + r * DN)[q] = make_float4(xn[4 * q], xn[4 * q + 1], xn[4 * q + 2], xn[4 * q + 3]);
      }
      uint32_t hi[16], lo[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float a = xn[2 * j] * sig_next, b = xn[2 * j + 1] * sig_next;
        split2s(a, b, hi[j], lo[j]);
        if (!(fmaxf(a, b) < 65000.f)) ovf = live ? 1 : ovf;
      }
      const uint32_t h0[8] = {hi[0], hi[1], hi[2], hi[3], hi[4], hi[5], hi[6], hi[7]};
      const uint32_t h1[8] = {hi[8], hi[9], hi[10], hi[11], hi[12], hi[13], hi[14], hi[15]};
      const uint32_t l0[8] = {lo[0], lo[1], lo[2], lo[3], lo[4], lo[5], lo[6], lo[7]};
      const uint32_t l1[8] = {lo[8], lo[9], lo[10], lo[11], lo[12], lo[13], lo[14], lo[15]};
      tmem_st8(tlane + N2_D1, h0); tmem_st8(tlane + N2_D1 + 8, h1);                 // K = 32: hi 16 columns
      tmem_st8(tlane + N2_D1 + 16, l0); tmem_st8(tlane + N2_D1 + 24, l1);           //         lo 16 columns
      issue(2);
      if (live) {                                                        // [hi(32 halfs) | lo(32 halfs)] = 128 B
        uint4* dst = xl_next + r * 8;
        dst[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);     dst[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
        dst[2] = make_uint4(hi[8], hi[9], hi[10], hi[11]);   dst[3] = make_uint4(hi[12], hi[13], hi[14], hi[15]);
        dst[4] = make_uint4(lo[0], lo[1], lo[2], lo[3]);     dst[5] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
        dst[6] = make_uint4(lo[8], lo[9], lo[10], lo[11]);   dst[7] = make_uint4(lo[12], lo[13], lo[14], lo[15]);
      }
    }
    // ---- epilogue 2: prow = (pinit + W0[:, 32:64] x') * sigma_next = fma(pinit, sigma, D2)  (D2 is in the scaled domain)
    mbar_wait(d_ready, pd); pd ^= 1;
    tc_fence_after();
#pragma unroll
    for (int ch = 0; ch < EH / 16; ++ch) {
      uint32_t acc[16];
      tmem_ld16(tlane + N2_D2 + 16 * ch, acc);
      tc_wait_ld();
      if (live) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int c = 16 * ch + 4 * q;
          reinterpret_cast<float4*>(prow + r * EH + 16 * ch)[q] =
              make_float4(fmaf(pin[c], sig_next, __uint_as_float(acc[4 * q])), fmaf(pin[c + 1], sig_next, __uint_as_float(acc[4 * q + 1])),
                          fmaf(pin[c + 2], sig_next, __uint_as_float(acc[4 * q + 2])), fmaf(pin[c + 3], sig_next, __uint_as_float(acc[4 * q + 3])));
        }
      }
    }
    tc_fence_before();
    named_barrier(1 + g, 128);                                          // D2 / A columns are rewritten by the next tile
  }
  atomic_max_f32(xmax + step + 1, mx);
  if (ovf) atomicOr(status, 1);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc<512>(tbase);
}

// e (fp32 [E,16], slot order) -> split rows [hi(16) | lo(16)] halfs
__global__ void split_edges_kernel(const float* __restrict__ e, int64_t num_edges, uint4* __restrict__ out,
                                   uint32_t* __restrict__ init_max, int32_t* __restrict__ status) {
  int ovf = 0;
  float mx = 0.f;
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < num_edges; s += (int64_t)gridDim.x * blockDim.x) {
    const float4* p = reinterpret_cast<const float4*>(e + s * DE);
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 v = __ldg(p + q);
      const float sc = pow2i(-INIT_SHIFT);
      split2s(v.x * sc, v.y * sc, hi[2 * q], lo[2 * q]);
      split2s(v.z * sc, v.w * sc, hi[2 * q + 1], lo[2 * q + 1]);
      const float m = fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w)));   // fmaxf drops NaN:
      if (!(m < 65000.f) || isnan(v.x + v.y + v.z + v.w)) ovf = 1;                           // the sum keeps it
      mx = fmaxf(mx, m);
    }
    out[s * 4 + 0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    out[s * 4 + 1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
    out[s * 4 + 2] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    out[s * 4 + 3] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
  atomic_max_f32(init_max, mx);
  if (ovf) atomicOr(status, 1);
}

// split rows -> fp32 (final edge state for callers that ask for it)
__global__ void unsplit_edges_kernel(const uint4* __restrict__ in, int64_t num_edges, float* __restrict__ e,
                                     const int32_t* __restrict__ sched, int32_t last_step) {
  const float inv = pow2i(sched[last_step]);                             // the state is stored in the last step's scale
  for (int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; s < num_edges; s += (int64_t)gridDim.x * blockDim.x) {
    const uint4 h0 = in[s * 4], h1 = in[s * 4 + 1], l0 = in[s * 4 + 2], l1 = in[s * 4 + 3];
    const uint32_t hw[8] = {h0.x, h0.y, h0.z, h0.w, h1.x, h1.y, h1.z, h1.w};
    const uint32_t lw[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&hw[j]));
      const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&lw[j]));
      e[s * DE + 2 * j] = fmaf(b.x, 1.f / LO_SCALE, a.x) * inv;
      e[s * DE + 2 * j + 1] = fmaf(b.y, 1.f / LO_SCALE, a.y) * inv;
    }
  }
}

// =================================================================== the edge kernel
struct TcArgs {
  const int32_t* slot_row; const int32_t* slot_col; const int32_t* slot_edge;
  int64_t num_edges, num_out;
  int32_t tiles_out, tiles_in;
  int64_t chunks_out;    // number of 32-slot chunks of the flow_out group
  const uint4* xi;       // [N][8]  x_init split rows (128 B)
  const uint4* xl;       // [N][8]  x_lat split rows
  const float* prow;     // [N][80] hoisted row term (incl. bias)
  const uint4* ei;       // [E][4]  e_init split rows (64 B)
  const uint4* es_in;    // [E][4]  e split rows
  uint4* es_out;         // may alias es_in
  float* flow; float* part; float* logits;
  const uint8_t* wimg_out; const uint8_t* wimg_in;
  int32_t* status;
  int32_t step;              // 1-based step index
  const int32_t* sched;      // sched[t] = s_t, see "range bookkeeping"
  uint32_t* amax;            // amax[step] receives the largest true activation of this launch; amax[0]: constant rows
  uint32_t* fmax;            // fmax[step] receives the largest flow piece (true value) this launch wrote
  int32_t agg;               // 0 sum, 1 mean (summed here, divided by the node kernel), 2 max
};

__device__ __forceinline__ void ld_f32x16(float (&d)[16], const float* __restrict__ p) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(p + 4 * q);
    d[4 * q] = v.x; d[4 * q + 1] = v.y; d[4 * q + 2] = v.z; d[4 * q + 3] = v.w;
  }
}
__device__ __forceinline__ void ld_f32x8(float (&d)[8], const float* __restrict__ p) {
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const float4 v = *reinterpret_cast<const float4*>(p + 4 * q);
    d[4 * q] = v.x; d[4 * q + 1] = v.y; d[4 * q + 2] = v.z; d[4 * q + 3] = v.w;
  }
}

// Resource plan of mp_edge_tc3_kernel, three tiles in flight per SM:
//  * the gathered x[col] rows are fetched by TMA (tile::gather4, 4 rows per instruction, 8 lanes per warp issue)
//    straight into 128B-swizzled K-major shared-memory tiles and consumed by SS-mode MMAs (layers 1 and 3) - no
//    per-thread loads, no register / TMEM staging of the widest operand;
//  * the tile's own edge rows (e_init, e) go global -> registers -> TMEM by the half of the group that is idle
//    during epilogue 2;
//  * a tile needs 144 TMEM columns and 48 KB of shared memory, so THREE groups of 8 warps keep three tiles in
//    flight per SM (24 warps); every edge row is served by two threads (halves A/B split the columns);
//  * layer 1 of the next tile is issued as soon as layer 4 of the current one has retired, so epilogue 4 and the
//    row sums run under it; row sums are split over all 8 warps (16 features each, 16-slot partial granule);
//  * the classifier's first layer rides in the 8 padding columns of flow layer 0 (computed by the tensor core).
constexpr int NG3 = 3, GT3 = 2 * TS, NTHREADS3 = NG3 * GT3;
constexpr int CHUNK3 = 16, CHUNK3_SHIFT = 4;                                   // row-sum partial granule (slots)
constexpr int T3_D1 = 0, T3_D2 = 80, T3_A3 = 96, T3_D3 = 0, T3_D4 = 80, T3_EH = 112, T3_EL = 128, T3_COLS = 144;
constexpr int A_SLAB = TS * 32;                                                // one K=16 step of a 128-row A tile
// group region: x_init[col] tile (128 rows x [hi 64 B | lo 64 B], SW128), x_lat[col] tile, message buffers
constexpr int G3_XI = 0, G3_XL = 4 * A_SLAB, G3_MSG = 8 * A_SLAB, G3_BYTES = 12 * A_SLAB;
constexpr int SM3_GRP = (IMG_BYTES + 1023) / 1024 * 1024;                      // swizzled tiles need 1 KB alignment
constexpr int SM3_BAR = SM3_GRP + NG3 * G3_BYTES;                              // d_ready[3], xc_ready[3]
constexpr int SM3_TMEM = SM3_BAR + 8 * 8;
constexpr int SM3_ROWS = SM3_TMEM + 16;                                         // int32 [24 warps][32]: slot -> row of the warp's quarter
constexpr int SMEM3_BYTES = SM3_ROWS + NG3 * 8 * 32 * 4;

__global__ void __launch_bounds__(NTHREADS3, 1) mp_edge_tc3_kernel(TcArgs a, const __grid_constant__ CUtensorMap tm_xi,
                                                                    const __grid_constant__ CUtensorMap tm_xl) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

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

  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM3_BAR);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM3_TMEM);
  uint32_t* s_fmax = tmem_slot + 1;                                     // largest flow piece this CTA wrote (scaled)
  // this step's scale (uniform): operands are true values x sigma
  const int s_cur = a.sched[a.step];
  const int s_prev = a.step > 1 ? a.sched[a.step - 1] : INIT_SHIFT;   // step 1 reads e_init rows as the latent state
  const float sigma = pow2i(-s_cur), inv_sigma = pow2i(s_cur);
  {
    const uint4* src = reinterpret_cast<const uint4*>(dir_out ? a.wimg_out : a.wimg_in);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    // The slabs that multiply the constant x_init / e_init rows (stored x 2^-INIT_SHIFT) carry 2^(INIT_SHIFT - s) themselves,
    // and the biases carry sigma; the classifier's output layer undoes it (all powers of two: exact).
    const __half2 sg = __float2half2_rn(pow2i(INIT_SHIFT - s_cur));
    for (int i = tid; i < IMG_BYTES / 16; i += NTHREADS3) {
      uint4 v = __ldg(src + i);
      const int o = i * 16;
      if (o < OFF_F32) {
        bool init_slab = false;
        if (o < OFF_L2H) { const int ks = (o % (L1_KS * L1_SLAB)) / L1_SLAB; init_slab = ks <= 1 || ks == 4; }
        else if (o >= OFF_L3H && o < OFF_L4H) { const int ks = ((o - OFF_L3H) % (L3_KS * L3_SLAB)) / L3_SLAB; init_slab = ks <= 1; }
        if (init_slab) {
          __half2* h = reinterpret_cast<__half2*>(&v);
#pragma unroll
          for (int q = 0; q < 4; ++q) h[q] = __hmul2(h[q], sg);
        }
      } else if (s_cur != 0) {
        float* f = reinterpret_cast<float*>(&v);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int fi = (o - OFF_F32) / 4 + q;
          if (fi < F_CW0 || (fi >= F_CB0 && fi < F_CW1)) f[q] *= sigma;            // b1, fb0, fb1, cb0
          else if (fi >= F_CW1 && fi < F_CB1) f[q] *= inv_sigma;                   // cw1
        }
      }
      dst[i] = v;
    }
    // s_cur > INIT_SHIFT + 14: the slab factor 2^(INIT_SHIFT - s) is a subnormal fp16 number (or 0 beyond 2^-24) and the
    // constant-row terms lose bits / vanish; such steps are already flagged by S_RESOLVED
  }
  if (blockIdx.x == 0 && tid == 0 && (s_cur > S_RESOLVED || (a.step == 1 && init_rows_unresolved(__uint_as_float(a.amax[0])))))
    atomicOr(a.status, 2);
  if (tid == 0) {
    for (int i = 0; i < NG3; ++i) { mbar_init(&bars[i], 1); mbar_init(&bars[NG3 + i], 4); }
    mbar_fence_init();
    *s_fmax = 0u;
  }
  if (warp == 0) tmem_alloc<512>(tmem_slot);
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tbase = *tmem_slot;
  const float* s_f = reinterpret_cast<const float*>(smem + OFF_F32);

  const int g = warp >> 3;
  const bool half_b = ((warp >> 2) & 1) != 0;
  const int hb = half_b ? 1 : 0;
  const int wq = warp & 3;
  const int gt = wq * 32 + lane;                                       // edge row inside the tile = TMEM lane
  const uint32_t tcol = __shfl_sync(0xffffffffu, tbase, 0) + (uint32_t)g * T3_COLS;
  const uint32_t tlane = tcol + ((uint32_t)(wq * 32) << 16);
  uint8_t* grp = smem + SM3_GRP + g * G3_BYTES;
  const uint32_t grp_addr = smem_u32(grp);
  // this warp's private message buffer: 32 rows x 16 features (its half of the columns), bank-conflict-free
  // both for the row-major writes (lane = row) and the feature-major reads of the row sums
  // Layout: row R (64 B) sits at physical row P = R ^ (R >> 4) (odd / even rows swapped in the upper granule, so that the two
  // half-warps of the row sums hit disjoint banks) with its four 16-byte chunks XOR-swizzled by (P >> 1) & 3 (conflict-free
  // 16-byte row writes).
  float* s_msg = reinterpret_cast<float*>(grp + G3_MSG) + (wq * 2 + hb) * 32 * 16;
  int32_t* s_rows = reinterpret_cast<int32_t*>(smem + SM3_ROWS) + warp * 32;
  uint64_t* d_ready = &bars[g];
  uint64_t* xc_ready = &bars[NG3 + g];                                  // 4 gathering warps arrive + 32 KB of TMA bytes
  uint32_t px = 0;
  const int64_t chunk_off = dir_out ? 0 : a.chunks_out;
  const int dir_off = dir_out ? DN : 0;
  const int bar_grp = 1 + g;
  uint32_t pd = 0;
  __half2 vmax = __floats2half2_rn(0.f, 0.f);

  const uint64_t dzero = smem_desc_kmajor(0, 128, 256);
  const uint64_t dsw = smem_desc_sw128(0);
  const uint32_t img = smem_u32(smem);
  // A layer = for every K step the two cross terms lo'.Whi + hi.Wlo' (they carry the 2^LO_SHIFT lift), then hi.Whi, whose
  // first MMA takes the accumulated cross terms in with the input scale 2^-LO_SHIFT.  *_x: x[col] K steps (A in the
  // group's swizzled shared-memory tiles), *_t: K steps whose A operand lives in TMEM.
  auto cross_x = [&](uint32_t d, uint32_t ah, uint32_t al, int off_h, int off_l, uint32_t idesc, bool first) {
    const uint64_t adh = dsw + (uint64_t)(ah >> 4), adl = dsw + (uint64_t)(al >> 4);
    const uint64_t bdh = dzero + (uint64_t)((img + off_h) >> 4), bdl = dzero + (uint64_t)((img + off_l) >> 4);
    mma_ss(d, adl, bdh, idesc, first ? 0u : 1u);
    mma_ss(d, adh, bdl, idesc, 1u);
  };
  auto cross_t = [&](uint32_t d, uint32_t ah, uint32_t al, int off_h, int off_l, uint32_t idesc, bool first) {
    const uint64_t bdh = dzero + (uint64_t)((img + off_h) >> 4), bdl = dzero + (uint64_t)((img + off_l) >> 4);
    mma_ts(d, al, bdh, idesc, first ? 0u : 1u);
    mma_ts(d, ah, bdl, idesc, 1u);
  };
  auto main_x = [&](uint32_t d, uint32_t ah, int off_h, uint32_t idesc, bool first) {
    const uint64_t adh = dsw + (uint64_t)(ah >> 4), bdh = dzero + (uint64_t)((img + off_h) >> 4);
    if (first) mma_ss_sd(d, adh, bdh, idesc);
    else mma_ss(d, adh, bdh, idesc, 1u);
  };
  auto main_t = [&](uint32_t d, uint32_t ah, int off_h, uint32_t idesc, bool first) {
    const uint64_t bdh = dzero + (uint64_t)((img + off_h) >> 4);
    if (first) mma_ts_sd(d, ah, bdh, idesc);
    else mma_ts(d, ah, bdh, idesc, 1u);
  };
  auto issue_layer = [&](int layer) {
    if (layer == 1) { mbar_wait(xc_ready, px); px ^= 1; }               // the tile's x[col] rows have landed (TMA)
    tc_fence_after();
    if (elect_one()) {
      const uint32_t cb = tcol;
      // x[col] K steps 0,1: x_init, 2,3: x_lat; hi at +0, lo at +64 B of a 128-B row
      auto xa = [&](int ks) { return grp_addr + (ks >> 1) * (G3_XL - G3_XI) + (ks & 1) * 32; };
      if (layer == 1) {
        constexpr uint32_t id = idesc_f16(128, EH);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) cross_x(cb + T3_D1, xa(ks), xa(ks) + 64, OFF_L1H + ks * L1_SLAB, OFF_L1L + ks * L1_SLAB, id, ks == 0);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
          cross_t(cb + T3_D1, cb + T3_EH + 8 * ks, cb + T3_EL + 8 * ks, OFF_L1H + (4 + ks) * L1_SLAB, OFF_L1L + (4 + ks) * L1_SLAB, id, false);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) main_x(cb + T3_D1, xa(ks), OFF_L1H + ks * L1_SLAB, id, ks == 0);
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) main_t(cb + T3_D1, cb + T3_EH + 8 * ks, OFF_L1H + (4 + ks) * L1_SLAB, id, false);
      } else if (layer == 2) {
        constexpr uint32_t id = idesc_f16(128, DE);
#pragma unroll
        for (int ks = 0; ks < L2_KS; ++ks)
          cross_t(cb + T3_D2, cb + T3_D1 + 16 * ks, cb + T3_D1 + 16 * ks + 8, OFF_L2H + ks * L2_SLAB, OFF_L2L + ks * L2_SLAB, id, ks == 0);
#pragma unroll
        for (int ks = 0; ks < L2_KS; ++ks) main_t(cb + T3_D2, cb + T3_D1 + 16 * ks, OFF_L2H + ks * L2_SLAB, id, ks == 0);
      } else if (layer == 3) {
        constexpr uint32_t id = idesc_f16(128, FHP);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) cross_x(cb + T3_D3, xa(ks), xa(ks) + 64, OFF_L3H + ks * L3_SLAB, OFF_L3L + ks * L3_SLAB, id, ks == 0);
        cross_t(cb + T3_D3, cb + T3_A3, cb + T3_A3 + 8, OFF_L3H + 4 * L3_SLAB, OFF_L3L + 4 * L3_SLAB, id, false);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) main_x(cb + T3_D3, xa(ks), OFF_L3H + ks * L3_SLAB, id, ks == 0);
        main_t(cb + T3_D3, cb + T3_A3, OFF_L3H + 4 * L3_SLAB, id, false);
      } else {
        constexpr uint32_t id = idesc_f16(128, DN);
#pragma unroll
        for (int ks = 0; ks < L4_KS; ++ks)
          cross_t(cb + T3_D4, cb + T3_D3 + 16 * ks, cb + T3_D3 + 16 * ks + 8, OFF_L4H + ks * L4_SLAB, OFF_L4L + ks * L4_SLAB, id, ks == 0);
#pragma unroll
        for (int ks = 0; ks < L4_KS; ++ks) main_t(cb + T3_D4, cb + T3_D3 + 16 * ks, OFF_L4H + ks * L4_SLAB, id, ks == 0);
      }
      mma_commit(d_ready);
    }
    __syncwarp();
  };
  auto publish_and_issue = [&](int layer) {
    tc_wait_st();
    tc_fence_before();
    named_barrier(bar_grp, GT3);
    if (!half_b && wq == 0) issue_layer(layer);
  };
  auto epilogue_chunk = [&](int col, const float* add) {
    uint32_t acc[16];
    tmem_ld16(tlane + col, acc);
    tc_wait_ld();
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      split2s_relu_add(__uint_as_float(acc[2 * j]), __uint_as_float(acc[2 * j + 1]), add[2 * j], add[2 * j + 1], hi[j], lo[j]);
      vmax = __hmax2(vmax, *reinterpret_cast<const __half2*>(&hi[j]));
    }
    tmem_st8(tlane + col, hi);
    tmem_st8(tlane + col + 8, lo);
  };

  // x[col] rows of this quarter's 32 edges -> the group's swizzled operand tiles, 4 rows per TMA gather; half A
  auto fetch_nodes = [&](int32_t c) {
    const int l4 = (lane & 7) * 4;
    const int32_t c0 = __shfl_sync(0xffffffffu, c, l4), c1 = __shfl_sync(0xffffffffu, c, l4 + 1);
    const int32_t c2 = __shfl_sync(0xffffffffu, c, l4 + 2), c3 = __shfl_sync(0xffffffffu, c, l4 + 3);
    if (lane == 0) mbar_arrive_expect_tx(xc_ready, 32 * 256);
    __syncwarp();
    if (lane < 8) {
      const uint32_t dst = grp_addr + G3_XI + (wq * 32 + l4) * 128;
      tma_gather4(dst, &tm_xi, xc_ready, c0, c1, c2, c3);
      tma_gather4(dst + (G3_XL - G3_XI), &tm_xl, xc_ready, c0, c1, c2, c3);
    }
  };
  // this thread's edge row [e_init | e] (split halves) -> TMEM operand columns; half B
  const __half2 rho = __float2half2_rn(pow2i(s_prev - s_cur));
  struct EdgeRow { uint4 v[8]; };
  auto load_edge_row = [&](int64_t base, int cnt) {
    EdgeRow r;
    const int64_t sl = base + (gt < cnt ? gt : cnt - 1);
    const uint4* p0 = a.ei + sl * 4;
    const uint4* p1 = a.es_in + sl * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) { r.v[j] = __ldg(p0 + j); r.v[4 + j] = p1[j]; }
    if (s_cur != s_prev) {                                             // uniform; e was stored in the previous step's scale
#pragma unroll
      for (int j = 4; j < 8; ++j) {
        __half2* h = reinterpret_cast<__half2*>(&r.v[j]);
#pragma unroll
        for (int q = 0; q < 4; ++q) h[q] = __hmul2(h[q], rho);
      }
    }
    return r;
  };
  auto store_edge_row = [&](const EdgeRow& r) {
    const uint32_t h0[8] = {r.v[0].x, r.v[0].y, r.v[0].z, r.v[0].w, r.v[1].x, r.v[1].y, r.v[1].z, r.v[1].w};
    const uint32_t l0[8] = {r.v[2].x, r.v[2].y, r.v[2].z, r.v[2].w, r.v[3].x, r.v[3].y, r.v[3].z, r.v[3].w};
    const uint32_t h1[8] = {r.v[4].x, r.v[4].y, r.v[4].z, r.v[4].w, r.v[5].x, r.v[5].y, r.v[5].z, r.v[5].w};
    const uint32_t l1[8] = {r.v[6].x, r.v[6].y, r.v[6].z, r.v[6].w, r.v[7].x, r.v[7].y, r.v[7].z, r.v[7].w};
    tmem_st8(tlane + T3_EH, h0);
    tmem_st8(tlane + T3_EL, l0);
    tmem_st8(tlane + T3_EH + 8, h1);
    tmem_st8(tlane + T3_EL + 8, l1);
  };

  struct TileIdx { int64_t base; int cnt; int32_t r, x, nb; bool have; };   // x: col (half A) / slot_edge (half B)
  auto load_idx = [&](int p) {
    TileIdx t;
    t.have = NG3 * p + g < tiles_dir;
    t.base = 0; t.cnt = 0; t.r = 0; t.x = 0; t.nb = -1;
    if (t.have) {
      t.base = seg_base + (int64_t)(NG3 * p + g) * TS;
      t.cnt = (int)(seg_end - t.base < TS ? seg_end - t.base : TS);
      const int64_t slot = gt < t.cnt ? t.base + gt : t.base + t.cnt - 1;
      t.r = a.slot_row[slot];
      if (!half_b) t.x = a.slot_col[slot];
      else if (a.logits != nullptr) t.x = a.slot_edge[slot];
      const int64_t cs = t.base + wq * 32;
      const int cw = t.cnt - wq * 32;
      // one predicated load (lane 0: the slot before the quarter, lane 31: the slot after it)
      const bool want = (lane == 0 && cw > 0 && cs > seg_base) || (lane == 31 && cw >= 32 && cs + 32 < seg_end);
      if (want) t.nb = a.slot_row[lane == 0 ? cs - 1 : cs + 32];
    }
    return t;
  };
  // Row sums of this warp's 16 message features over its quarter's 32 slots, in slot order: lanes (sub, f) walk the
  // two 16-slot granules.  A row's segment that lies inside one granule is written to `flow`; pieces that touch a
  // granule edge go to the granule's two partial slots and are combined by the node kernel in fixed order.
  auto row_sums = [&](const TileIdx& t) {
    const int sub = lane >> 4, fl = lane & 15;
    int cwq = t.cnt - wq * 32;
    cwq = cwq < 0 ? 0 : (cwq > 32 ? 32 : cwq);
    int cw = cwq - 16 * sub;
    cw = cw < 0 ? 0 : (cw > 16 ? 16 : cw);
    const int32_t nb_prev = __shfl_sync(0xffffffffu, t.nb, 0);
    const int32_t nb_next = __shfl_sync(0xffffffffu, t.nb, 31);
    const int32_t r15 = __shfl_sync(0xffffffffu, t.r, 15);
    const int32_t r16 = __shfl_sync(0xffffffffu, t.r, 16);
    const int32_t r_prev = sub ? r15 : nb_prev;
    const int32_t r_next = sub ? nb_next : (cwq > 16 ? r16 : -1);
    const int32_t r_after = __shfl_down_sync(0xffffffffu, t.r, 1);
    const bool seg_end_here = fl < cw && (fl == cw - 1 || r_after != t.r);       // lane doubles as the row index here
    const unsigned ends = (__ballot_sync(0xffffffffu, seg_end_here) >> (16 * sub)) & 0xffffu;
    const int64_t chunk_id = chunk_off + ((t.base + wq * 32 - seg_base) >> CHUNK3_SHIFT) + sub;
    const int f = 16 * hb + fl;
    // message (16 sub + q, fl): physical row 16 sub + (q ^ sub), chunk (fl >> 2) ^ ((q >> 1) & 3)
    const float* mb = s_msg + 256 * sub + (fl & 3);
    const int rs = 16 * sub;                                                     // (q ^ sub) * 16 = 16 q +- 16 sub
    const int c4 = 4 * (fl >> 2);
    const int32_t* rows = s_rows + 16 * sub;
    const bool agg_max = a.agg == 2;
    float sum = 0.f;
    bool first_seg = true;
#pragma unroll
    for (int q = 0; q < CHUNK3; ++q) {
      const float mq = mb[16 * q + ((q & 1) ? -rs : rs) + (c4 ^ (4 * ((q >> 1) & 3)))];
      sum = agg_max ? fmaxf(sum, mq) : sum + mq;
      if ((ends >> q) & 1u) {
        const int32_t rq = rows[q];
        const bool starts_before = first_seg && r_prev == rq;
        const bool continues = q == cw - 1 && r_next == rq;
        atomicMax(s_fmax, __float_as_uint(sum));                       // sum >= 0: integer order = float order
        if (!starts_before && !continues) a.flow[(int64_t)rq * 2 * DN + dir_off + f] = sum * inv_sigma;
        else a.part[(chunk_id * 2 + (first_seg ? 0 : 1)) * DN + f] = sum * inv_sigma;
        sum = 0.f;
        first_seg = false;
      }
    }
    __syncwarp();
  };
  auto load_prow16 = [&](float* add, int32_t r, int ch) {
    const float4* prp = reinterpret_cast<const float4*>(a.prow + (int64_t)r * EH + 16 * ch);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 v = __ldg(prp + j);
      add[4 * j] = v.x; add[4 * j + 1] = v.y; add[4 * j + 2] = v.z; add[4 * j + 3] = v.w;
    }
  };

  TileIdx cur = load_idx(cta_in_dir);
  TileIdx nxt = load_idx(cta_in_dir + ctas_in_dir);
  if (cur.have) {
    if (!half_b) {
      fetch_nodes(cur.x);
    } else {
      const EdgeRow er = load_edge_row(cur.base, cur.cnt);
      store_edge_row(er);
    }
    publish_and_issue(1);
  }
  int p = cta_in_dir;
  while (cur.have) {
    const bool valid = gt < cur.cnt;
    p += ctas_in_dir;
    TileIdx nn = load_idx(p + ctas_in_dir);
    if (nxt.have) {                                                   // next tile's hoisted row terms -> L1
      const char* pr = reinterpret_cast<const char*>(a.prow + (int64_t)nxt.r * EH) + (half_b ? 192 : 0);
      asm volatile("prefetch.global.L1 [%0];" ::"l"(pr));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(pr + 127));
    }
    if (half_b && nn.have && (lane & 1) == 0) {                       // pull the edge rows two tiles ahead into L2
      const int64_t sl = nn.base + (gt < nn.cnt ? gt : nn.cnt - 1);
      asm volatile("prefetch.global.L2 [%0];" ::"l"(a.ei + sl * 4));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(a.es_in + sl * 4));
    }

    // ---- epilogue 1: + hoisted x[row] term (A: columns 0..47, B: 48..79)
    {
      const int ch0 = half_b ? 3 : 0;
      float add[16];
      load_prow16(add, cur.r, ch0);
      mbar_wait(d_ready, pd); pd ^= 1;
      tc_fence_after();
      epilogue_chunk(T3_D1 + 16 * ch0, add);
      load_prow16(add, cur.r, ch0 + 1);
      epilogue_chunk(T3_D1 + 16 * (ch0 + 1), add);
      if (!half_b) {
        load_prow16(add, cur.r, 2);
        epilogue_chunk(T3_D1 + 32, add);
      }
    }
    publish_and_issue(2);

    // ---- epilogue 2 (half A): e' -> state + layer-3 operand; half B stages the next tile's edge rows in TMEM
    if (!half_b) {
      mbar_wait(d_ready, pd); pd ^= 1;
      tc_fence_after();
      uint32_t acc[16];
      tmem_ld16(tlane + T3_D2, acc);
      float add[16];
      ld_f32x16(add, s_f + F_B1);
      tc_wait_ld();
      uint32_t hi[8], lo[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        split2s_relu_add(__uint_as_float(acc[2 * j]), __uint_as_float(acc[2 * j + 1]), add[2 * j], add[2 * j + 1], hi[j], lo[j]);
        vmax = __hmax2(vmax, *reinterpret_cast<const __half2*>(&hi[j]));
      }
      tmem_st8(tlane + T3_A3, hi);
      tmem_st8(tlane + T3_A3 + 8, lo);
      publish_and_issue(3);
      if (valid) {
        uint4* dst = a.es_out + (cur.base + gt) * 4;
        dst[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        dst[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
        dst[2] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        dst[3] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
      }
    } else {
      if (nxt.have) {                                                  // layer 1 (the only reader) has retired
        const EdgeRow er = load_edge_row(nxt.base, nxt.cnt);
        store_edge_row(er);
      }
      mbar_wait(d_ready, pd); pd ^= 1;
      tc_fence_after();
      publish_and_issue(3);
    }
    // ---- epilogue 3: g -> layer-4 operand (A: columns 0..31, B: 32..63; 56..63 carry the classifier's first layer)
    mbar_wait(d_ready, pd); pd ^= 1;
    tc_fence_after();
    if (!half_b && nxt.have) fetch_nodes(nxt.x);                       // layer 3 was the last reader of x[col]
    {
      const int ch0 = half_b ? 2 : 0;
      float add[16];
      ld_f32x16(add, s_f + F_FB0 + 16 * ch0);
      epilogue_chunk(T3_D3 + 16 * ch0, add);
      ld_f32x16(add, s_f + F_FB0 + 16 * (ch0 + 1));                    // B: entries 8..15 are zero (padding)
      if (!half_b) {
        epilogue_chunk(T3_D3 + 16, add);
      } else {
        uint32_t acc[16];
        tmem_ld16(tlane + T3_D3 + 48, acc);
        float cb0[CH], cw1[CH];
        ld_f32x8(cb0, s_f + F_CB0);
        ld_f32x8(cw1, s_f + F_CW1);
        tc_wait_ld();
        uint32_t hi[8], lo[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          split2s_relu_add(__uint_as_float(acc[2 * j]), __uint_as_float(acc[2 * j + 1]), add[2 * j], add[2 * j + 1], hi[j], lo[j]);
          vmax = __hmax2(vmax, *reinterpret_cast<const __half2*>(&hi[j]));
        }
#pragma unroll
        for (int j = 4; j < 8; ++j) { hi[j] = 0u; lo[j] = 0u; }        // K padding of layer 4
        tmem_st8(tlane + T3_D3 + 48, hi);
        tmem_st8(tlane + T3_D3 + 56, lo);
        if (valid && a.logits != nullptr) {
          float lg = s_f[F_CB1];
#pragma unroll
          for (int o = 0; o < CH; ++o) lg = fmaf(fmaxf(__uint_as_float(acc[8 + o]) + cb0[o], 0.f), cw1[o], lg);
          a.logits[cur.x] = lg;
        }
      }
    }
    publish_and_issue(4);

    // ---- layer 4 retired -> its operand columns are free: start the next tile's layer 1, then finish this tile
    mbar_wait(d_ready, pd); pd ^= 1;
    tc_fence_after();
    if (nxt.have) publish_and_issue(1);
    {
      uint32_t acc[16];
      tmem_ld16(tlane + T3_D4 + 16 * hb, acc);
      float add[16];
      ld_f32x16(add, s_f + F_FB1 + 16 * hb);
      tc_wait_ld();
      // slots past the end of the slot range need no masking: nothing after the last row end is ever stored
      float m[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) m[j] = fmaxf(__uint_as_float(acc[j]) + add[j], 0.f);
      const int prow_ = lane ^ (lane >> 4);
      float* mrow = s_msg + 16 * prow_;
      const int sw = (prow_ >> 1) & 3;
#pragma unroll
      for (int c = 0; c < 4; ++c)
        *reinterpret_cast<float4*>(mrow + 4 * (c ^ sw)) = make_float4(m[4 * c], m[4 * c + 1], m[4 * c + 2], m[4 * c + 3]);
      s_rows[lane] = cur.r;
    }
    __syncwarp();
    row_sums(cur);
    cur = nxt; nxt = nn;
  }
  {
    // __hmax2 drops NaN, so this sees an fp16 overflow (an inf or a value at the top of the range) but not a NaN.  It need
    // not: every input, weight and bias is checked finite and inside the fp16 range before step 1 (prep_nodes_kernel,
    // split_edges_kernel, pack_weights_kernel), and from such operands the edge kernel cannot produce a NaN before an
    // activation has overflowed, which this test sees.
    const uint32_t w = *reinterpret_cast<const uint32_t*>(&vmax);
    if ((w & 0x7FFFu) >= 0x7BFFu || ((w >> 16) & 0x7FFFu) >= 0x7BFFu) atomicOr(a.status, 1);
    const float2 vm = __half22float2(vmax);
    atomic_max_f32(a.amax + a.step, fminf(fmaxf(vm.x, vm.y), 65504.f) * inv_sigma);
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0 && *s_fmax != 0u) atomicMax(a.fmax + a.step, __float_as_uint(__uint_as_float(*s_fmax) * inv_sigma));
  if (warp == 0) tmem_dealloc<512>(tbase);
}

// 2-D tensor map over split node rows [n][64 halfs] for the TMA row gather (box = one row, 128B swizzle)
static int make_row_map(CUtensorMap* out, const void* base, int64_t n) {
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  if (encode == nullptr) {
    cudaDriverEntryPointQueryResult q;
    void* fn = nullptr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || fn == nullptr) return -1;
    encode = reinterpret_cast<EncodeFn>(fn);
  }
  const cuuint64_t dims[2] = {64, (cuuint64_t)n};
  const cuuint64_t strides[1] = {128};
  const cuuint32_t box[2] = {64, 1};
  const cuuint32_t estr[2] = {1, 1};
  return encode(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS ? 0 : -1;
}

struct TcWorkspace {
  __half* xi; __half* xl[2];
  float* pinit; float* prow;
  uint4* ei; uint4* es;
  float* flow; float* part;
  uint8_t* wimg_out; uint8_t* wimg_in; uint8_t* wimg_node;
  int32_t* sched; uint32_t* amax; uint32_t* xmax; uint32_t* fmax;   // range bookkeeping, MAX_STEPS + 8 entries each (contiguous)
};

static int64_t carve(void* ws, int64_t n, int64_t e, TcWorkspace* out) {
  Carver cv(ws);
  const int64_t chunks = ceil_div(e, CHUNK3) + 8;
  TcWorkspace w;
  w.xi = cv.take<__half>(n * 64);
  w.xl[0] = cv.take<__half>(n * 64);
  w.xl[1] = cv.take<__half>(n * 64);
  w.pinit = cv.take<float>(n * EH);
  w.prow = cv.take<float>(n * EH);
  w.ei = cv.take<uint4>(e * 4);
  w.es = cv.take<uint4>(e * 4);
  w.flow = cv.take<float>(n * 2 * DN);
  w.part = cv.take<float>(chunks * 2 * DN);
  w.wimg_out = cv.take<uint8_t>(IMG_BYTES);
  w.wimg_in = cv.take<uint8_t>(IMG_BYTES);
  w.wimg_node = cv.take<uint8_t>(NIMG_BYTES);
  w.sched = cv.take<int32_t>(4 * (MAX_STEPS + 8));
  w.amax = reinterpret_cast<uint32_t*>(w.sched) + (MAX_STEPS + 8);
  w.xmax = w.amax + (MAX_STEPS + 8);
  w.fmax = w.xmax + (MAX_STEPS + 8);
  if (out) *out = w;
  return cv.off;
}

}  // namespace tc
}  // namespace mpn

using namespace mpn;

extern "C" {

int64_t mpn_mp_tc_workspace(int64_t n, int64_t e) {
  return tc::carve(nullptr, n > 0 ? n : 1, e > 0 ? e : 1, nullptr) + 256;
}

int mpn_mp_tc_read_schedule(const void* ws, int64_t n, int64_t e, int32_t num_steps, int32_t* h_sched, float* h_amax,
                            float* h_xmax, void* stream) {
  MPN_CHECK_ARG(ws && num_steps >= 1 && num_steps <= tc::MAX_STEPS, "mp_tc_read_schedule: bad arguments");
  tc::TcWorkspace m;
  tc::carve(const_cast<void*>(ws), n > 0 ? n : 1, e > 0 ? e : 1, &m);
  cudaStream_t s = as_stream(stream);
  if (h_sched) MPN_CUDA(cudaMemcpyAsync(h_sched, m.sched, sizeof(int32_t) * (num_steps + 2), cudaMemcpyDeviceToHost, s));
  if (h_amax) MPN_CUDA(cudaMemcpyAsync(h_amax, m.amax, sizeof(float) * (num_steps + 2), cudaMemcpyDeviceToHost, s));
  if (h_xmax) MPN_CUDA(cudaMemcpyAsync(h_xmax, m.xmax, sizeof(float) * (num_steps + 2), cudaMemcpyDeviceToHost, s));
  MPN_CUDA(cudaStreamSynchronize(s));
  return MPN_OK;
}

int mpn_mp_forward_tc(const mpn_core_weights* w, const mpn_edge_layout* g, const float* x_init, const float* e_init,
                      int32_t num_steps, int32_t first_class_step, void* ws, float* logits, float* x_out,
                      float* e_out, int32_t* status, void* stream) {
  MPN_CHECK_ARG(w && g, "mp_forward_tc: null descriptor");
  MPN_CHECK_ARG(w->dn == 32 && w->de == 16 && w->edge_h == 80 && w->flow_h == 56 && w->cls_h == 8,
                "mp_forward_tc: built for widths dn=32 de=16 edge_h=80 flow_h=56 cls_h=8 (got %d %d %d %d %d)", w->dn,
                w->de, w->edge_h, w->flow_h, w->cls_h);
  MPN_CHECK_ARG(w->node_agg >= 0 && w->node_agg <= 2, "mp_forward_tc: node_agg must be 0 (sum), 1 (mean) or 2 (max)");
  MPN_CHECK_ARG(num_steps >= 1 && num_steps <= tc::MAX_STEPS, "mp_forward_tc: num_steps must be in 1..%d (use mpn_mp_forward for 0)",
                tc::MAX_STEPS);
  MPN_CHECK_ARG(ws && status, "mp_forward_tc: null workspace / status");
  const int64_t n = g->num_nodes, e = g->num_edges;
  cudaStream_t s = as_stream(stream);
  MPN_CUDA(cudaMemsetAsync(status, 0, 4, s));
  if (n == 0) return MPN_OK;
  tc::TcWorkspace m;
  tc::carve(ws, n, e > 0 ? e : 1, &m);

  MPN_CUDA(cudaFuncSetAttribute(tc::mp_edge_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::SMEM3_BYTES));
  MPN_CUDA(cudaMemsetAsync(m.sched, 0, 4 * (tc::MAX_STEPS + 8) * 4, s));
  const int sms = sm_count();
  tc::pack_weights_kernel<<<16, 256, 0, s>>>(*w, m.wimg_out, m.wimg_in, m.wimg_node, status); count_launch();
  const unsigned ngrid = (unsigned)std::min<int64_t>(ceil_div(n * 32, 256), (int64_t)sms * 4);
  const unsigned ngrid_node2 = (unsigned)std::min<int64_t>(ceil_div(ceil_div(n, tc::TS), 2), (int64_t)sms);
  tc::prep_nodes_kernel<<<ngrid, 256, 0, s>>>(x_init, n, w->edge_w0, w->edge_b0, m.xi, m.xl[0], m.pinit, m.prow, m.xmax, m.amax, status);
  count_launch();
  if (e > 0) {
    const unsigned egrid = (unsigned)std::min<int64_t>(ceil_div(e, 256), (int64_t)sms * 8);
    tc::split_edges_kernel<<<egrid, 256, 0, s>>>(e_init, e, m.ei, m.amax, status); count_launch();
  }
  MPN_LAUNCH_CHECK();

  const int tiles_out = (int)ceil_div(g->num_out, tc::TS);
  const int tiles_in = (int)ceil_div(e - g->num_out, tc::TS);
  const int triples = (tiles_out + 2) / 3 + (tiles_in + 2) / 3;
  int grid3 = sms;
  if (grid3 > triples) grid3 = triples;
  if (tiles_out > 0 && tiles_in > 0 && grid3 < 2) grid3 = 2;

  CUtensorMap tm_xi, tm_xl[2];
  if (e > 0) {
    if (tc::make_row_map(&tm_xi, m.xi, n) || tc::make_row_map(&tm_xl[0], m.xl[0], n) || tc::make_row_map(&tm_xl[1], m.xl[1], n)) {
      set_error("mpn_mp_forward_tc: cuTensorMapEncodeTiled failed");
      return MPN_ECUDA;
    }
  }
  const int chunk_shift = tc::CHUNK3_SHIFT;
  const int64_t chunk = (int64_t)1 << chunk_shift;
  for (int step = 1; step <= num_steps; ++step) {
    const __half* xl_cur = m.xl[(step - 1) & 1];
    __half* xl_next = m.xl[step & 1];
    if (e > 0) {
      tc::TcArgs a;
      a.slot_row = g->slot_row; a.slot_col = g->slot_col; a.slot_edge = g->slot_edge;
      a.num_edges = e; a.num_out = g->num_out; a.tiles_out = tiles_out; a.tiles_in = tiles_in;
      a.chunks_out = ceil_div(g->num_out, chunk);
      a.xi = reinterpret_cast<const uint4*>(m.xi);
      a.xl = reinterpret_cast<const uint4*>(xl_cur);
      a.prow = m.prow;
      a.ei = m.ei;
      a.es_in = step == 1 ? m.ei : m.es;
      a.es_out = m.es;
      a.flow = m.flow; a.part = m.part;
      a.logits = (logits && step >= first_class_step) ? logits + (int64_t)(step - first_class_step) * e : nullptr;
      a.wimg_out = m.wimg_out; a.wimg_in = m.wimg_in;
      a.status = status;
      a.step = step; a.sched = m.sched; a.amax = m.amax; a.fmax = m.fmax; a.agg = w->node_agg;
      if (profiling()) profile_mark(0, true, s);
      tc::mp_edge_tc3_kernel<<<grid3, tc::NTHREADS3, tc::SMEM3_BYTES, s>>>(a, tm_xi, tm_xl[(step - 1) & 1]);
      count_launch();
      if (profiling()) profile_mark(0, false, s);
    }
    if (profiling()) profile_mark(1, true, s);
    tc::node_tc2_kernel<<<ngrid_node2, tc::NT2_THREADS, tc::NSMEM_BYTES, s>>>(
        g->out_ptr, g->in_ptr, n, g->num_out, (int32_t)ceil_div(g->num_out, chunk), chunk_shift, m.flow, m.part,
        m.wimg_node, m.pinit, reinterpret_cast<uint4*>(xl_next), m.prow, step == num_steps ? x_out : nullptr, step,
        m.sched, m.amax, m.xmax, m.fmax, w->node_agg, status);
    count_launch();
    if (profiling()) profile_mark(1, false, s);
    MPN_LAUNCH_CHECK();
  }
  if (e_out && e > 0) {
    const unsigned egrid = (unsigned)std::min<int64_t>(ceil_div(e, 256), (int64_t)sms * 8);
    tc::unsplit_edges_kernel<<<egrid, 256, 0, s>>>(m.es, e, e_out, m.sched, num_steps); count_launch();
    MPN_LAUNCH_CHECK();
  }
  return MPN_OK;
}

}  // extern "C"
