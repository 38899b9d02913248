// Weighted binary cross-entropy over the classified steps (pl_module/pl_module.py:88-105):
//   pos_weight = (#edges - #positives) / #positives   (0 when there is no positive label)
//   loss = weight * sum_steps mean_edges BCEWithLogits(logits_s, labels, pos_weight)
// plus d loss / d logits (the seed of the backward pass).  Reductions are fixed-order (deterministic).
// Per edge: term (1 - y) softplus(x) + pw y softplus(-x), gradient weight / E ((1 - y) sigmoid(x) - pw y sigmoid(-x)).
#include <math.h>

#include "common.cuh"

namespace mpn {

constexpr int LB = 256;

__device__ __forceinline__ double block_sum(double v, double* sm) {
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x == 0) for (int w = 0; w < LB / 32; ++w) t += sm[w];
  __syncthreads();
  return t;                                            // valid in thread 0
}

// softplus(x) = log(1 + e^x) and sigmoid(x) = 1 / (1 + e^-x), both accurate relative to their value for every x
// (sigmoid(x) of a very negative x is e^x, not the difference 1 - sigmoid(-x), which rounds to 0 below x = -17)
__device__ __forceinline__ float softplus(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }
__device__ __forceinline__ float sigmoid(float x) {
  const float t = expf(-fabsf(x));                                 // no overflow: e^x / (1 + e^x) below 0
  return x < 0.f ? t / (1.f + t) : 1.f / (1.f + t);
}

__global__ void __launch_bounds__(LB) label_partials_kernel(const float* __restrict__ labels, int64_t e,
                                                            double* __restrict__ partial) {
  __shared__ double sm[LB / 32];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * LB + threadIdx.x; i < e; i += (int64_t)gridDim.x * LB) s += labels[i];
  s = block_sum(s, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void __launch_bounds__(LB) bce_partials_kernel(const float* __restrict__ logits, const float* __restrict__ labels,
                                                          int64_t steps, int64_t e, const double* __restrict__ label_partial,
                                                          int nlabel, float weight, double* __restrict__ partial,
                                                          float* __restrict__ grad, float* __restrict__ pos_weight_out) {
  __shared__ double sm[LB / 32];
  __shared__ float s_pw;
  if (threadIdx.x == 0) {
    double pos = 0.0;
    for (int i = 0; i < nlabel; ++i) pos += label_partial[i];       // same order in every block
    s_pw = pos > 0.0 ? (float)(((double)e - pos) / pos) : 0.f;
    if (blockIdx.x == 0 && pos_weight_out != nullptr) *pos_weight_out = s_pw;
  }
  __syncthreads();
  const float pw = s_pw;
  const float inv_e = 1.f / (float)e;
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * LB + threadIdx.x; i < steps * e; i += (int64_t)gridDim.x * LB) {
    const float x = logits[i], y = labels[i % e];
    const float wn = 1.f - y, wp = pw * y;                           // weights of the negative / positive side
    // (1 - y) sp(x) + pw y sp(-x): no term cancels, and a side of weight 0 adds 0 even where its softplus is inf
    s += (double)((wn != 0.f ? wn * softplus(x) : 0.f) + (wp != 0.f ? wp * softplus(-x) : 0.f));
    if (grad != nullptr) grad[i] = weight * inv_e * (wn * sigmoid(x) - wp * sigmoid(-x));
  }
  s = block_sum(s, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = s;
}

__global__ void bce_final_kernel(const double* __restrict__ partial, int n, int64_t e, float weight,
                                 float* __restrict__ loss) {
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < n; ++i) t += partial[i];
    *loss = (float)(weight * t / (double)e);
  }
}

}  // namespace mpn

using namespace mpn;

extern "C" {

int64_t mpn_weighted_bce_workspace(void) { return 2 * 1024 * 8 + 256; }

int mpn_weighted_bce(const float* logits, const float* labels, int64_t steps, int64_t e, float weight, void* ws,
                     float* loss, float* pos_weight, float* grad, void* stream) {
  MPN_CHECK_ARG(steps >= 0 && e >= 0 && loss != nullptr && ws != nullptr, "weighted_bce: bad arguments");
  cudaStream_t s = as_stream(stream);
  if (steps == 0 || e == 0) { MPN_CUDA(cudaMemsetAsync(loss, 0, 4, s)); return MPN_OK; }
  MPN_CHECK_ARG(logits && labels, "weighted_bce: null pointer");
  double* lp = static_cast<double*>(ws);
  double* bp = lp + 1024;
  const int nl = (int)std::min<int64_t>(ceil_div(e, LB), 1024);
  const int nb = (int)std::min<int64_t>(ceil_div(steps * e, LB), 1024);
  label_partials_kernel<<<nl, LB, 0, s>>>(labels, e, lp); count_launch();
  bce_partials_kernel<<<nb, LB, 0, s>>>(logits, labels, steps, e, lp, nl, weight, bp, grad, pos_weight); count_launch();
  bce_final_kernel<<<1, 32, 0, s>>>(bp, nb, e, weight, loss); count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // extern "C"
