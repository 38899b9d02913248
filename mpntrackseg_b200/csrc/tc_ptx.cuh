// Thin inline-PTX wrappers for sm_100a: mbarrier, tcgen05 (TMEM alloc / ld / st / mma / commit),
// proxy fences.  Shapes used: 32x32b TMEM accesses (thread = its own TMEM lane), kind::f16 MMA
// with A in TMEM and B in shared memory (K-major, no swizzle).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mpn {
namespace ptx {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  const uint32_t a = smem_u32(bar);
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(a), "r"(parity), "r"(20000u)      // suspend-time hint (ns): sleep in hardware instead of re-polling
        : "memory");
  }
}

// ---------------------------------------------------------------- fences
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- TMEM allocation (one warp)
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(COLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS));
}

// ---------------------------------------------------------------- TMEM <-> registers (32x32b)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(taddr), "r"(v[0]),
               "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
               : "memory");
}

// ---------------------------------------------------------------- MMA
// Shared-memory matrix descriptor, K-major, no swizzle: 8x16B core matrices; LBO = byte distance
// between the two K halves of a 16-wide K step, SBO = byte distance between 8-row groups.
__device__ __forceinline__ uint64_t smem_desc_kmajor(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;   // descriptor version 1 (sm_100)
  return d;
}
// Byte offset of element (n, k16) inside one K = 16 step of such an operand ("slab"), laid out [n/8][k16/8][n%8][k16%8]:
// 8-row x 16-B core matrices, the two K halves LBO = 128 B apart and the 8-row groups SBO = 256 B apart.
__device__ __forceinline__ int slab_off(int n, int k16) {
  return (n >> 3) * 256 + (k16 >> 3) * 128 + (n & 7) * 16 + (k16 & 7) * 2;
}
// Instruction descriptor, kind::f16: fp16 A/B (K-major), fp32 accumulate, M x N tile.
__host__ __device__ constexpr uint32_t idesc_f16(int m, int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// D[tmem] (+)= A[tmem] * B[smem]^T ; issued by ONE thread.
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T ; both operands through shared-memory matrix descriptors.
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// K-major operand tile in the 128-byte swizzle (rows at a 128-B pitch, 8-row atoms of 1 KB; the layout TMA writes
// with CU_TENSOR_MAP_SWIZZLE_128B).  A K step of 16 halves is +32 B on the start address.
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy of a contiguous global range into shared memory; completion counted in bytes on `bar`
__device__ __forceinline__ void tma_bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// TMA row gather: rows r0..r3 of a 2-D tensor map (box {row length, 1}) -> 4 consecutive tile rows at dst
__device__ __forceinline__ void tma_gather4(uint32_t dst, const void* tmap, uint64_t* bar, int32_t r0, int32_t r1,
                                            int32_t r2, int32_t r3) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(dst), "l"(tmap), "r"(smem_u32(bar)), "r"(0), "r"(r0), "r"(r1), "r"(r2), "r"(r3)
      : "memory");
}
// mbarrier arrives once all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// one lane of the (converged) warp
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void named_barrier(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
// named barrier that also returns whether `v` was true in any participating thread
__device__ __forceinline__ bool named_barrier_or(int id, int threads, bool v) {
  uint32_t r;
  asm volatile("{\n\t.reg .pred p, q;\n\tsetp.ne.u32 q, %1, 0;\n\tbar.red.or.pred p, %2, %3, q;\n\tselp.u32 %0, 1, 0, p;\n\t}"
               : "=r"(r)
               : "r"((uint32_t)v), "r"(id), "r"(threads)
               : "memory");
  return r != 0;
}

// ---------------------------------------------------------------- fp16 hi/lo split
// v ~= hi + lo with hi = fp16(v), lo = fp16(v - hi): 22 significant bits.
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(a - hf.x, b - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ReLU fused into the split: hi = fp16_rz(max(v,0)) (truncation keeps lo >= 0), lo = fp16_rn(max(v - hi, 0)).
__device__ __forceinline__ void split2_relu(float a, float b, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(b), "f"(a));
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(b - hf.y), "f"(a - hf.x));
}

// Power-of-two pre-scale of an operand row (or block) whose largest |v| is `amax_bits` (fp32 bits): 2^p * max |v|
// lies in [2^13, 2^14), so every split2 operand keeps a resolution of 2^-25 relative to 2^13 ... 2^14 of the
// largest value, and hi stays far from the fp16 maximum.  |p| <= 62 keeps 2^-2p a normal fp32 number.
constexpr int PACK_SHIFT_MAX = 62;
__device__ __forceinline__ int pack_shift(uint32_t amax_bits) {
  const float m = __uint_as_float(amax_bits);
  if (!(m > 0.f) || !isfinite(m)) return 0;                      // all zero (or non-finite: the caller's status says so)
  int e;
  frexpf(m, &e);                                                 // m in [2^(e-1), 2^e)
  return max(-PACK_SHIFT_MAX, min(PACK_SHIFT_MAX, 14 - e));
}
// 2^e for -126 <= e <= 127 (exact)
__device__ __forceinline__ float pow2i(int e) { return __int_as_float((e + 127) << 23); }

// ---------------------------------------------------------------- fp16 hi/lo split with a lifted low part
// v ~= hi + lo' * 2^-LO_SHIFT with lo' = fp16((v - hi) * 2^LO_SHIFT).  The low part is then a NORMAL fp16 number whenever
// hi is (|lo'| <= |hi| / 2 for the rn split, < |hi| for the truncating ReLU split, so it can never overflow), i.e. the
// pair keeps 22 significant bits over the whole fp16 exponent range instead of losing low bits to subnormals below
// ~0.1.  The MMAs accumulate the two cross terms (lo'.hi, hi.lo') first and fold them in with the accumulator input
// scale of tcgen05.mma (D = A.B + D * 2^-LO_SHIFT, `mma_*_sd`).
constexpr int LO_SHIFT = 10;
constexpr float LO_SCALE = 1024.f;
__device__ __forceinline__ void split2s(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(a, b);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn((a - hf.x) * LO_SCALE, (b - hf.y) * LO_SCALE);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}
// ReLU fused into the lifted split of (a + ba, b + bb), as in split2_relu: hi = fp16_rz(max(v, 0)),
// lo' = fp16_rn(max((v - hi) * 2^LO_SHIFT, 0)).  The add, subtract and lift run on the packed fp32x2 pipe (FADD2 / FMUL2:
// one instruction per pair): 7 instructions per pair instead of 10.  Every packed operation is the IEEE rn operation of
// its two lanes, so the result is bit-identical to the scalar form.
__device__ __forceinline__ unsigned long long pack2(float x, float y) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(x), "f"(y));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long r, float& x, float& y) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(x), "=f"(y) : "l"(r));
}
__device__ __forceinline__ void split2s_relu_add(float a, float b, float ba, float bb, uint32_t& hi, uint32_t& lo) {
  unsigned long long t, d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(t) : "l"(pack2(a, b)), "l"(pack2(ba, bb)));
  float tx, ty;
  unpack2(t, tx, ty);
  asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(ty), "f"(tx));
  const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(t), "l"(pack2(hf.x, hf.y)));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(d), "l"(pack2(LO_SCALE, LO_SCALE)));
  float dx, dy;
  unpack2(d, dx, dy);
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(dy), "f"(dx));
}
// D = A.B + D * 2^-LO_SHIFT (kind::f16 accumulator input scale)
__device__ __forceinline__ void mma_ts_sd(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p, 10;\n\t}" ::"r"(d_tmem),
      "r"(a_tmem), "l"(b_desc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void mma_ss_sd(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p, 10;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc)
      : "memory");
}

}  // namespace ptx
}  // namespace mpn
