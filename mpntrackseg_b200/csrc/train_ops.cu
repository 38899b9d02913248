// Building blocks of the training step (forward with stored activations + backward), fp32,
// deterministic (no float atomics; every reduction runs in a fixed order):
//   mpn_gemm          C = act(op(A) op(B) + bias)  with optional transposes / accumulation / ReLU-mask on A
//   mpn_gather_cols   out[e, off:off+w] = src[idx[e], :]
//   mpn_segment_reduce out[n, off:off+w] (+)= sum / mean / max over the node's contiguous (optionally permuted) segment
//   (mpn_segment_sum is its sum mode)
//   mpn_segment_grad  gradient of a mean / max segment reduction back to the segment's slots (a gather, no scatter)
//   mpn_batchnorm_*   BatchNorm1d with batch statistics (+ ReLU, + dropout) and its backward
//   mpn_dropout_*     inverted dropout after a ReLU, Philox4x32 masks, and its backward
//   mpn_relu_mask     g *= (y > 0)
//   mpn_adam_step     fused Adam with L2 weight decay (torch.optim.Adam semantics) on flat buffers
// They serve pl_module/pl_module.py:122-135 (loss.backward + optimizer step) for the core network.
// Philox4x32-10 of the cuRAND device API (the generator header alone: curand_kernel.h would also link its other
// generators' precomputed tables, ~200 KB, into the module)
#include <curand_philox4x32_x.h>
#include <math.h>

#include "common.cuh"

namespace mpn {

constexpr int GT = 64, GK = 16;

// C[m][n] = sum_k A(m,k) B(k,n);  A(m,k) = ta ? a[k*lda + m] : a[m*lda + k],  B(k,n) = tb ? b[n*ldb + k] : b[k*ldb + n]
// optional: A is multiplied elementwise by (mask_a > 0) (ReLU backward of the producer), bias[n], ReLU, C += .
__global__ void __launch_bounds__(256) gemm_kernel(const float* __restrict__ a, int64_t lda, int ta,
                                                   const float* __restrict__ mask_a, int64_t ldm,
                                                   const float* __restrict__ b, int64_t ldb, int tb,
                                                   const float* __restrict__ bias, int relu, int accumulate,
                                                   float* __restrict__ c, int64_t ldc, int64_t m, int64_t n, int64_t k,
                                                   int64_t k_per_split, float* __restrict__ partial) {
  __shared__ float As[GK][GT + 4];
  __shared__ float Bs[GK][GT + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int64_t m0 = (int64_t)blockIdx.y * GT, n0 = (int64_t)blockIdx.x * GT;
  const int64_t kbeg = (int64_t)blockIdx.z * k_per_split;
  const int64_t kend = kbeg + k_per_split < k ? kbeg + k_per_split : k;
  float acc[4][4] = {};
  for (int64_t k0 = kbeg; k0 < kend; k0 += GK) {
    for (int idx = threadIdx.x; idx < GT * GK; idx += 256) {
      int r, kk;
      if (ta) { r = idx % GT; kk = idx / GT; } else { r = idx / GK; kk = idx % GK; }   // coalesced along the contiguous dim
      const int64_t gm = m0 + r, gk = k0 + kk;
      float v = 0.f;
      if (gm < m && gk < kend) {
        v = ta ? a[gk * lda + gm] : a[gm * lda + gk];
        if (mask_a != nullptr) v = (ta ? mask_a[gk * ldm + gm] : mask_a[gm * ldm + gk]) > 0.f ? v : 0.f;
      }
      As[kk][r] = v;
    }
    for (int idx = threadIdx.x; idx < GT * GK; idx += 256) {
      int r, kk;
      if (tb) { r = idx / GK; kk = idx % GK; } else { r = idx % GT; kk = idx / GT; }
      const int64_t gn = n0 + r, gk = k0 + kk;
      Bs[kk][r] = (gn < n && gk < kend) ? (tb ? b[gn * ldb + gk] : b[gk * ldb + gn]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < GK; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(ar[i], br[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t gm = m0 + ty * 4 + i;
    if (gm >= m) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t gn = n0 + tx * 4 + j;
      if (gn >= n) continue;
      if (partial != nullptr) { partial[((int64_t)blockIdx.z * m + gm) * n + gn] = acc[i][j]; continue; }
      float v = acc[i][j] + (bias != nullptr ? bias[gn] : 0.f);
      if (accumulate) v += c[gm * ldc + gn];
      c[gm * ldc + gn] = relu ? fmaxf(v, 0.f) : v;
    }
  }
}

// c = act(sum_z partial[z] + bias) (+ c): the split-K slices are added in ascending z (deterministic)
__global__ void gemm_reduce_kernel(const float* __restrict__ partial, int splits, const float* __restrict__ bias, int relu,
                                   int accumulate, float* __restrict__ c, int64_t ldc, int64_t m, int64_t n) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m * n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t gm = t / n, gn = t - gm * n;
    float v = 0.f;
    for (int z = 0; z < splits; ++z) v += partial[(int64_t)z * m * n + t];
    v += bias != nullptr ? bias[gn] : 0.f;
    if (accumulate) v += c[gm * ldc + gn];
    c[gm * ldc + gn] = relu ? fmaxf(v, 0.f) : v;
  }
}

// column sums of (A .* (mask > 0)) -> out[n] (+)= ...; one CTA per 32 columns, rows walked in a fixed order
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ a, int64_t lda,
                                                     const float* __restrict__ mask, int64_t ldm, int64_t m,
                                                     int64_t n, int64_t rows_per_slice, float* __restrict__ partial) {
  __shared__ float part[8][33];
  const int col = blockIdx.x * 32 + (threadIdx.x & 31), rgrp = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_slice;
  const int64_t r1 = r0 + rows_per_slice < m ? r0 + rows_per_slice : m;
  float s = 0.f;
  if (col < n)
    for (int64_t r = r0 + rgrp; r < r1; r += 8) {
      float v = a[r * lda + col];
      if (mask != nullptr && !(mask[r * ldm + col] > 0.f)) v = 0.f;
      s += v;
    }
  part[rgrp][threadIdx.x & 31] = s;
  __syncthreads();
  if (rgrp == 0 && col < n) {
    float t = 0.f;
    for (int g = 0; g < 8; ++g) t += part[g][threadIdx.x & 31];
    partial[(int64_t)blockIdx.y * n + col] = t;
  }
}

__global__ void colsum_reduce_kernel(const float* __restrict__ partial, int slices, int64_t n, int accumulate,
                                     float* __restrict__ out) {
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
    float t = 0.f;
    for (int y = 0; y < slices; ++y) t += partial[(int64_t)y * n + c];     // ascending slices: deterministic
    out[c] = accumulate ? out[c] + t : t;
  }
}

__global__ void gather_cols_kernel(const float* __restrict__ src, int64_t lds, int64_t w, const int32_t* __restrict__ idx,
                                   int64_t rows, float* __restrict__ out, int64_t ldo, int64_t off) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < rows * w; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / w, c = t - r * w;
    const int64_t s = idx != nullptr ? idx[r] : r;
    out[r * ldo + off + c] = src[s * lds + c];
  }
}

// out[node, off + f] (+)= reduce_{q in [ptr[node], ptr[node+1])} in[(perm ? perm[q] : q) * ld + in_off + f], in slot order.
// MODE 0: sum; 1: mean (0 for an empty segment); 2: max, the first strictly larger value in ascending q (torch_scatter's
// scatter_max on the CPU), 0 for an empty segment; argmax (MODE 2, may be null) receives the input row of the
// maximum, or -1 for an empty segment.  A template, so that the sum the backward runs most carries no mode branch.
template <int MODE>
__global__ void segment_sum_kernel(const float* __restrict__ in, int64_t ld, int64_t in_off, int64_t w,
                                   const int32_t* __restrict__ ptr, const int32_t* __restrict__ perm, int64_t nodes,
                                   int accumulate, float* __restrict__ out, int64_t ldo, int64_t off,
                                   int32_t* __restrict__ argmax) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nodes * w; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t node = t / w, f = t - node * w;
    float s = 0.f;
    if (MODE != 2) {
      for (int q = ptr[node]; q < ptr[node + 1]; ++q) s += in[(int64_t)(perm != nullptr ? perm[q] : q) * ld + in_off + f];
      if (MODE == 1 && ptr[node + 1] > ptr[node]) s /= (float)(ptr[node + 1] - ptr[node]);
    } else {
      int32_t arg = -1;
      for (int q = ptr[node]; q < ptr[node + 1]; ++q) {
        const int32_t r = perm != nullptr ? perm[q] : q;
        const float v = in[(int64_t)r * ld + in_off + f];
        if (arg < 0 || v > s) { s = v; arg = r; }
      }
      if (argmax != nullptr) argmax[t] = arg;
    }
    float* o = out + node * ldo + off + f;
    *o = accumulate ? *o + s : s;
  }
}

// Backward of a mean / max segment reduction for the slots q in [q0, q1) (one thread per slot and feature):
//   mean: out[q, f] = g[row[q], f] / |segment of row[q]|;   max: out[q, f] = argmax[row[q], f] == q ? g[row[q], f] : 0
__global__ void segment_grad_kernel(const float* __restrict__ g, int64_t ldg, const int32_t* __restrict__ row,
                                    const int32_t* __restrict__ ptr, const int32_t* __restrict__ argmax, int64_t q0,
                                    int64_t q1, int64_t w, int mode, float* __restrict__ out, int64_t ldo) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < (q1 - q0) * w; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t q = q0 + t / w, f = t % w;
    const int64_t r = row[q];
    const float gv = g[r * ldg + f];
    out[q * ldo + f] = mode == 1 ? gv / (float)(ptr[r + 1] - ptr[r]) : (argmax[r * w + f] == q ? gv : 0.f);
  }
}

// ---- BatchNorm1d (batch statistics) and dropout

// Keep decision of element `elem` of dropout call `call` in the forward numbered *counter: one Philox4x32-10 draw per
// four consecutive elements, so a mask depends on (seed, counter, call, element) only, never on the launch shape.
__device__ __forceinline__ bool dropout_keep(uint64_t seed, const int64_t* __restrict__ counter, int call, int64_t elem,
                                             float p) {
  const uint64_t ctr = (uint64_t)*counter;
  const uint4 c = make_uint4((uint32_t)(elem >> 2), (uint32_t)call, (uint32_t)ctr, (uint32_t)(ctr >> 32));
  const uint4 r = curand_Philox4x32_10(c, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const uint32_t k = elem & 3;
  const uint32_t v = k == 0 ? r.x : k == 1 ? r.y : k == 2 ? r.z : r.w;
  return (float)(v >> 8) * (1.f / 16777216.f) >= p;              // uniform in [0, 1) with 24 bits
}

// Per-slice column partials over rows [r0, r1) in a fixed order (the layout of colsum_kernel):
//   what 0: sum z;  1: sum (z - mean)^2;  2: sum g' and sum g' xhat  with g' = y > 0 ? g * gscale : 0,
//   xhat = (z - mean) invstd.  partial: [slices][n] (what 2: a second [slices][n] block follows).  The sums run in
//   double: a thread adds up to rows_per_slice / 8 rows (977 at 10^6 rows), and an fp32 sum of that many equal values
//   drifts by ~1e-5 of the mean, which a column of large offset turns into an error of the normalised output.
__global__ void __launch_bounds__(256) bn_partial_kernel(const float* __restrict__ z, int64_t ldz,
                                                         const float* __restrict__ g, int64_t ldg,
                                                         const float* __restrict__ y, int64_t ldy,
                                                         const float* __restrict__ stats, float gscale, int64_t m,
                                                         int64_t n, int64_t rows_per_slice, int what,
                                                         double* __restrict__ partial) {
  __shared__ double part[2][8][33];
  const int col = blockIdx.x * 32 + (threadIdx.x & 31), rgrp = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_slice;
  const int64_t r1 = r0 + rows_per_slice < m ? r0 + rows_per_slice : m;
  double s0 = 0.0, s1 = 0.0;
  if (col < n) {
    const float mu = what > 0 ? stats[col] : 0.f, is = what == 2 ? stats[n + col] : 0.f;
    for (int64_t r = r0 + rgrp; r < r1; r += 8) {
      const float d = z[r * ldz + col] - mu;
      if (what == 0) s0 += d;
      else if (what == 1) s0 += d * d;
      else if (y[r * ldy + col] > 0.f) {
        const float gp = g[r * ldg + col] * gscale;
        s0 += gp;
        s1 += gp * (d * is);
      }
    }
  }
  part[0][rgrp][threadIdx.x & 31] = s0;
  part[1][rgrp][threadIdx.x & 31] = s1;
  __syncthreads();
  if (rgrp == 0 && col < n) {
    double t0 = 0.0, t1 = 0.0;
    for (int k = 0; k < 8; ++k) { t0 += part[0][k][threadIdx.x & 31]; t1 += part[1][k][threadIdx.x & 31]; }
    partial[(int64_t)blockIdx.y * n + col] = t0;
    if (what == 2) partial[((int64_t)gridDim.y + blockIdx.y) * n + col] = t1;
  }
}

// Slices added in ascending order, then per column:
//   what 0: stats[0:n] = mean;
//   what 1: stats[n:2n] = 1 / sqrt(var + eps) with the biased variance, running_mean / running_var updated with the
//           unbiased one (torch.nn.BatchNorm1d), and *num_batches_tracked += 1 (also for m == 0, which changes nothing
//           else);
//   what 2: ggamma += sum g' xhat, gbeta += sum g', stats[2n:3n] / stats[3n:4n] = their means over the rows.
__global__ void bn_finalize_kernel(const double* __restrict__ partial, int slices, int64_t m, int64_t n, int what,
                                   float eps, float momentum, float* __restrict__ stats, float* __restrict__ running_mean,
                                   float* __restrict__ running_var, int64_t* __restrict__ num_batches_tracked,
                                   float* __restrict__ ggamma, float* __restrict__ gbeta) {
  if (what == 1 && num_batches_tracked != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *num_batches_tracked += 1;
  if (m == 0) return;
  for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
    double d0 = 0.0, d1 = 0.0;
    for (int k = 0; k < slices; ++k) d0 += partial[(int64_t)k * n + c];
    if (what == 2)
      for (int k = 0; k < slices; ++k) d1 += partial[(int64_t)(slices + k) * n + c];
    const float t0 = (float)d0, t1 = (float)d1;
    if (what == 0) {
      stats[c] = (float)(d0 / (double)m);
    } else if (what == 1) {
      const float var = (float)(d0 / (double)m);
      stats[n + c] = 1.f / sqrtf(var + eps);
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * stats[c];
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * (var * (float)m / (float)(m - 1));
    } else {
      gbeta[c] += t0;
      ggamma[c] += t1;
      stats[2 * n + c] = t0 / (float)m;
      stats[3 * n + c] = t1 / (float)m;
    }
  }
}

// y = ReLU(gamma (z - mean) invstd + beta), then (p > 0) y * keep / (1 - p); mask (may be null) receives keep.
__global__ void bn_apply_kernel(const float* __restrict__ z, int64_t ldz, int64_t m, int64_t n,
                                const float* __restrict__ stats, const float* __restrict__ gamma,
                                const float* __restrict__ beta, float p, uint64_t seed, const int64_t* __restrict__ counter,
                                int call, float* __restrict__ y, int64_t ldy, uint8_t* __restrict__ mask) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m * n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / n, c = t - r * n;
    float v = fmaxf(gamma[c] * ((z[r * ldz + c] - stats[c]) * stats[n + c]) + beta[c], 0.f);
    if (p > 0.f) {
      const bool keep = dropout_keep(seed, counter, call, t, p);
      v = keep ? v / (1.f - p) : 0.f;
      if (mask != nullptr) mask[t] = keep;
    }
    y[r * ldy + c] = v;
  }
}

// gz = gamma invstd (g' - mean(g') - xhat mean(g' xhat)),  g' = y > 0 ? g * gscale : 0
__global__ void bn_backward_kernel(const float* __restrict__ z, int64_t ldz, const float* __restrict__ g, int64_t ldg,
                                   const float* __restrict__ y, int64_t ldy, int64_t m, int64_t n,
                                   const float* __restrict__ stats, const float* __restrict__ gamma, float gscale,
                                   float* __restrict__ gz, int64_t ldgz) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m * n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / n, c = t - r * n;
    const float is = stats[n + c];
    const float xhat = (z[r * ldz + c] - stats[c]) * is;
    const float gp = y[r * ldy + c] > 0.f ? g[r * ldg + c] * gscale : 0.f;
    gz[r * ldgz + c] = gamma[c] * is * (gp - stats[2 * n + c] - xhat * stats[3 * n + c]);
  }
}

// in place: y = y * keep / (1 - p)  (y is a ReLU output); mask (may be null) receives keep
__global__ void dropout_kernel(float* __restrict__ y, int64_t ldy, int64_t m, int64_t n, float p, uint64_t seed,
                               const int64_t* __restrict__ counter, int call, uint8_t* __restrict__ mask) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m * n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / n, c = t - r * n;
    const bool keep = dropout_keep(seed, counter, call, t, p);
    float* o = y + r * ldy + c;
    *o = keep ? *o / (1.f - p) : 0.f;
    if (mask != nullptr) mask[t] = keep;
  }
}

// out = y > 0 ? g * scale : 0   (ReLU + dropout backward from the stored output)
__global__ void dropout_backward_kernel(const float* __restrict__ g, int64_t ldg, const float* __restrict__ y,
                                        int64_t ldy, int64_t m, int64_t n, float scale, float* __restrict__ out,
                                        int64_t ldo) {
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < m * n; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / n, c = t - r * n;
    out[r * ldo + c] = y[r * ldy + c] > 0.f ? g[r * ldg + c] * scale : 0.f;
  }
}

__global__ void relu_mask_kernel(float* __restrict__ g, const float* __restrict__ y, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (!(y[i] > 0.f)) g[i] = 0.f;
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay,
                            float bc1, float bc2, float grad_scale) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i] * grad_scale + weight_decay * p[i];           // torch.optim.Adam: L2 term added to the gradient
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// step counter on the device (CUDA-graph replays of a training step must not bake the step number in)
__global__ void bump_step_kernel(int64_t* step) { *step += 1; }
__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay,
                                const int64_t* __restrict__ step, float grad_scale) {
  const float t = (float)*step;
  const float bc1 = 1.f - powf(beta1, t), bc2 = 1.f - powf(beta2, t);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i] * grad_scale + weight_decay * p[i];
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

static void keep_async_pool() {
  static bool done = false;
  if (done) return;
  int dev = 0;
  cudaMemPool_t pool;
  if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  done = true;
}

static inline unsigned flat_grid(int64_t n) {
  return (unsigned)std::min<int64_t>(ceil_div(n > 0 ? n : 1, 256), (int64_t)sm_count() * 8);
}

}  // namespace mpn

using namespace mpn;

extern "C" {

int mpn_gemm(const float* a, int64_t lda, int trans_a, const float* mask_a, int64_t ldm, const float* b, int64_t ldb,
             int trans_b, const float* bias, int relu, int accumulate, float* c, int64_t ldc, int64_t m, int64_t n,
             int64_t k, void* stream) {
  MPN_CHECK_ARG(m >= 0 && n >= 0 && k >= 0, "gemm: negative size");
  if (m == 0 || n == 0) return MPN_OK;
  MPN_CHECK_ARG(c != nullptr && (k == 0 || (a && b)), "gemm: null pointer");
  MPN_CHECK_ARG(ceil_div(m, GT) <= 65535, "gemm: at most %d rows per call (gridDim.y limit)", 65535 * GT);
  cudaStream_t s = as_stream(stream);
  keep_async_pool();
  const int64_t tiles = ceil_div(n, GT) * ceil_div(m, GT);
  // few output tiles but a long contraction (weight gradients: contraction over the edges): split K
  int64_t splits = 1;
  if (tiles < 2 * sm_count() && k >= 2048) {
    splits = std::min<int64_t>(ceil_div(4 * (int64_t)sm_count(), tiles), ceil_div(k, 512));
    if (splits > 256) splits = 256;
  }
  if (splits <= 1) {
    dim3 grid((unsigned)ceil_div(n, GT), (unsigned)ceil_div(m, GT), 1);
    gemm_kernel<<<grid, 256, 0, s>>>(a, lda, trans_a, mask_a, ldm, b, ldb, trans_b, bias, relu, accumulate, c, ldc, m, n, k,
                                     k, nullptr);
    count_launch();
  } else {
    const int64_t kps = align_up(ceil_div(k, splits), GK);
    splits = ceil_div(k, kps);
    float* partial = nullptr;
    MPN_CUDA(cudaMallocAsync(&partial, sizeof(float) * splits * m * n, s));
    dim3 grid((unsigned)ceil_div(n, GT), (unsigned)ceil_div(m, GT), (unsigned)splits);
    gemm_kernel<<<grid, 256, 0, s>>>(a, lda, trans_a, mask_a, ldm, b, ldb, trans_b, nullptr, 0, 0, c, ldc, m, n, k, kps,
                                     partial);
    count_launch();
    gemm_reduce_kernel<<<flat_grid(m * n), 256, 0, s>>>(partial, (int)splits, bias, relu, accumulate, c, ldc, m, n);
    count_launch();
    MPN_CUDA(cudaFreeAsync(partial, s));
  }
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_colsum(const float* a, int64_t lda, const float* mask, int64_t ldm, int64_t m, int64_t n, int accumulate,
               float* out, void* stream) {
  if (n == 0) return MPN_OK;
  MPN_CHECK_ARG(out != nullptr && (m == 0 || a != nullptr), "colsum: null pointer");
  cudaStream_t s = as_stream(stream);
  keep_async_pool();
  const int64_t slices = std::max<int64_t>(1, std::min<int64_t>(ceil_div(m, 256), 128));
  const int64_t rps = ceil_div(m > 0 ? m : 1, slices);
  float* partial = nullptr;
  MPN_CUDA(cudaMallocAsync(&partial, sizeof(float) * slices * n, s));
  dim3 grid((unsigned)ceil_div(n, 32), (unsigned)slices);
  colsum_kernel<<<grid, 256, 0, s>>>(a, lda, mask, ldm, m, n, rps, partial);
  count_launch();
  colsum_reduce_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(partial, (int)slices, n, accumulate, out);
  count_launch();
  MPN_CUDA(cudaFreeAsync(partial, s));
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_gather_cols(const float* src, int64_t lds, int64_t width, const int32_t* idx, int64_t rows, float* out,
                    int64_t ldo, int64_t col_off, void* stream) {
  if (rows == 0 || width == 0) return MPN_OK;
  MPN_CHECK_ARG(src && out, "gather_cols: null pointer");
  gather_cols_kernel<<<flat_grid(rows * width), 256, 0, as_stream(stream)>>>(src, lds, width, idx, rows, out, ldo, col_off);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_segment_reduce(const float* in, int64_t ld, int64_t in_off, int64_t width, const int32_t* ptr, const int32_t* perm,
                       int64_t nodes, int accumulate, float* out, int64_t ldo, int64_t col_off, int mode, int32_t* argmax,
                       void* stream) {
  if (nodes == 0 || width == 0) return MPN_OK;
  MPN_CHECK_ARG(ptr && out, "segment_sum: null pointer");
  MPN_CHECK_ARG(mode >= 0 && mode <= 2, "segment_sum: mode must be 0 (sum), 1 (mean) or 2 (max)");
  auto kernel = mode == 0 ? segment_sum_kernel<0> : mode == 1 ? segment_sum_kernel<1> : segment_sum_kernel<2>;
  kernel<<<flat_grid(nodes * width), 256, 0, as_stream(stream)>>>(in, ld, in_off, width, ptr, perm, nodes, accumulate, out,
                                                                ldo, col_off, argmax);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_segment_sum(const float* in, int64_t ld, int64_t in_off, int64_t width, const int32_t* ptr, const int32_t* perm,
                    int64_t nodes, int accumulate, float* out, int64_t ldo, int64_t col_off, void* stream) {
  return mpn_segment_reduce(in, ld, in_off, width, ptr, perm, nodes, accumulate, out, ldo, col_off, 0, nullptr, stream);
}

int mpn_segment_grad(const float* g, int64_t ldg, const int32_t* row, const int32_t* ptr, const int32_t* argmax,
                     int64_t q0, int64_t q1, int64_t width, int mode, float* out, int64_t ldo, void* stream) {
  if (q1 <= q0 || width == 0) return MPN_OK;
  MPN_CHECK_ARG(mode == 1 || mode == 2, "segment_grad: mode must be 1 (mean) or 2 (max)");
  MPN_CHECK_ARG(g && row && out && (mode == 1 ? ptr != nullptr : argmax != nullptr), "segment_grad: null pointer");
  segment_grad_kernel<<<flat_grid((q1 - q0) * width), 256, 0, as_stream(stream)>>>(g, ldg, row, ptr, argmax, q0, q1, width,
                                                                                 mode, out, ldo);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

// slices of the column reductions of the BatchNorm kernels (as mpn_colsum)
static inline int64_t bn_slices(int64_t m) { return std::max<int64_t>(1, std::min<int64_t>(ceil_div(m, 256), 128)); }

int mpn_batchnorm_forward(const float* z, int64_t ldz, int64_t m, int64_t n, const float* gamma, const float* beta,
                          float eps, float momentum, float* running_mean, float* running_var, int64_t* num_batches_tracked,
                          float* stats, float p, uint64_t seed, const int64_t* counter, int call, float* y, int64_t ldy,
                          uint8_t* mask, void* stream) {
  MPN_CHECK_ARG(m != 1, "Expected more than 1 value per channel when training, got input size [1, %lld]", (long long)n);
  MPN_CHECK_ARG(m >= 0 && n > 0 && p >= 0.f && p < 1.f, "batchnorm_forward: bad sizes or dropout probability");
  MPN_CHECK_ARG(stats && running_mean && running_var && num_batches_tracked && (m == 0 || (z && gamma && beta && y)),
                "batchnorm_forward: null pointer");
  MPN_CHECK_ARG(p == 0.f || counter != nullptr, "batchnorm_forward: dropout needs the forward counter");
  cudaStream_t s = as_stream(stream);
  if (m == 0) {                                       // empty batch: only the batch counter moves (torch 2.11)
    bn_finalize_kernel<<<1, 32, 0, s>>>(nullptr, 0, 0, n, 1, eps, momentum, stats, running_mean, running_var,
                                        num_batches_tracked, nullptr, nullptr);
    count_launch();
    MPN_LAUNCH_CHECK();
    return MPN_OK;
  }
  keep_async_pool();
  const int64_t slices = bn_slices(m), rps = ceil_div(m, slices);
  double* partial = nullptr;
  MPN_CUDA(cudaMallocAsync(&partial, sizeof(double) * slices * n, s));
  const dim3 grid((unsigned)ceil_div(n, 32), (unsigned)slices);
  const unsigned fgrid = (unsigned)ceil_div(n, 256);
  for (int what = 0; what < 2; ++what) {              // mean, then the variance around it (two passes)
    bn_partial_kernel<<<grid, 256, 0, s>>>(z, ldz, nullptr, 0, nullptr, 0, stats, 1.f, m, n, rps, what, partial);
    bn_finalize_kernel<<<fgrid, 256, 0, s>>>(partial, (int)slices, m, n, what, eps, momentum, stats, running_mean,
                                             running_var, num_batches_tracked, nullptr, nullptr);
    count_launch(2);
  }
  bn_apply_kernel<<<flat_grid(m * n), 256, 0, s>>>(z, ldz, m, n, stats, gamma, beta, p, seed, counter, call, y, ldy, mask);
  count_launch();
  MPN_CUDA(cudaFreeAsync(partial, s));
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_batchnorm_backward(const float* z, int64_t ldz, const float* g, int64_t ldg, const float* y, int64_t ldy, int64_t m,
                           int64_t n, const float* gamma, float* stats, float gscale, float* ggamma, float* gbeta,
                           float* gz, int64_t ldgz, void* stream) {
  if (m == 0 || n == 0) return MPN_OK;
  MPN_CHECK_ARG(z && g && y && gamma && stats && ggamma && gbeta && gz, "batchnorm_backward: null pointer");
  cudaStream_t s = as_stream(stream);
  keep_async_pool();
  const int64_t slices = bn_slices(m), rps = ceil_div(m, slices);
  double* partial = nullptr;
  MPN_CUDA(cudaMallocAsync(&partial, sizeof(double) * 2 * slices * n, s));
  bn_partial_kernel<<<dim3((unsigned)ceil_div(n, 32), (unsigned)slices), 256, 0, s>>>(z, ldz, g, ldg, y, ldy, stats, gscale,
                                                                                     m, n, rps, 2, partial);
  bn_finalize_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(partial, (int)slices, m, n, 2, 0.f, 0.f, stats, nullptr,
                                                               nullptr, nullptr, ggamma, gbeta);
  bn_backward_kernel<<<flat_grid(m * n), 256, 0, s>>>(z, ldz, g, ldg, y, ldy, m, n, stats, gamma, gscale, gz, ldgz);
  count_launch(3);
  MPN_CUDA(cudaFreeAsync(partial, s));
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_dropout_forward(float* y, int64_t ldy, int64_t m, int64_t n, float p, uint64_t seed, const int64_t* counter,
                        int call, uint8_t* mask, void* stream) {
  if (m == 0 || n == 0) return MPN_OK;
  MPN_CHECK_ARG(y && counter, "dropout_forward: null pointer");
  MPN_CHECK_ARG(p > 0.f && p < 1.f, "dropout_forward: p must lie in (0, 1)");
  dropout_kernel<<<flat_grid(m * n), 256, 0, as_stream(stream)>>>(y, ldy, m, n, p, seed, counter, call, mask);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_dropout_backward(const float* g, int64_t ldg, const float* y, int64_t ldy, int64_t m, int64_t n, float scale,
                         float* out, int64_t ldo, void* stream) {
  if (m == 0 || n == 0) return MPN_OK;
  MPN_CHECK_ARG(g && y && out, "dropout_backward: null pointer");
  dropout_backward_kernel<<<flat_grid(m * n), 256, 0, as_stream(stream)>>>(g, ldg, y, ldy, m, n, scale, out, ldo);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_relu_mask(float* g, const float* y, int64_t n, void* stream) {
  if (n == 0) return MPN_OK;
  MPN_CHECK_ARG(g && y, "relu_mask: null pointer");
  relu_mask_kernel<<<flat_grid(n), 256, 0, as_stream(stream)>>>(g, y, n);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int64_t step, float grad_scale, void* stream) {
  if (n == 0) return MPN_OK;
  MPN_CHECK_ARG(params && grads && exp_avg && exp_avg_sq && step >= 1, "adam_step: bad arguments");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adam_kernel<<<flat_grid(n), 256, 0, as_stream(stream)>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                          weight_decay, bc1, bc2, grad_scale);
  count_launch();
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

int mpn_adam_step_dev(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float lr, float beta1,
                      float beta2, float eps, float weight_decay, int64_t* d_step, float grad_scale, void* stream) {
  MPN_CHECK_ARG(d_step != nullptr, "adam_step_dev: null step counter");
  bump_step_kernel<<<1, 1, 0, as_stream(stream)>>>(d_step); count_launch();
  if (n > 0) {
    MPN_CHECK_ARG(params && grads && exp_avg && exp_avg_sq, "adam_step_dev: bad arguments");
    adam_dev_kernel<<<flat_grid(n), 256, 0, as_stream(stream)>>>(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                                weight_decay, d_step, grad_scale);
    count_launch();
  }
  MPN_LAUNCH_CHECK();
  return MPN_OK;
}

}  // extern "C"
