// Common device-side PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (UMMA + TMEM) and small numeric helpers.  Everything here is hand-written
// inline PTX; no CUTLASS/CuTe dependency.
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>

// 16-bit storage type of this build of the library.  The library is compiled twice from the same sources:
// libidiff_b200.so (fp16 activations / weights, the reference's autocast type, inference.py:94) and
// libidiff_b200_bf16.so (-DIDIFF_STORAGE_BF16=1, BASELINE config 3).  Accumulation, statistics and the
// sampler state are fp32 in both; only the operand format of the UMMAs and the pack / unpack at the
// edges of each kernel differ, so every kernel below is written against h16 / pack_half2 / unpack_half2.
#ifndef IDIFF_STORAGE_BF16
#define IDIFF_STORAGE_BF16 0
#endif
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>

namespace idiff {

#define IDIFF_DEVICE __device__ __forceinline__

IDIFF_DEVICE uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

IDIFF_DEVICE bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ----------------------------------------------------------------------------------
// mbarrier
// ----------------------------------------------------------------------------------
IDIFF_DEVICE void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
IDIFF_DEVICE void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
}
IDIFF_DEVICE void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
IDIFF_DEVICE void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
IDIFF_DEVICE bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (try_wait may suspend the thread for a system-defined time; a polling loop over
// several barriers wants the immediate answer).
IDIFF_DEVICE bool mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug must surface as a trapped launch (an error code at the C ABI),
// never as a hung GPU.  ~4 s at 2 GHz.
IDIFF_DEVICE void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && (clock64() - t0) > 8000000000LL) {
      printf("idiff: mbarrier timeout block=(%d,%d,%d) thread=%d bar=%u parity=%u\n", blockIdx.x,
             blockIdx.y, blockIdx.z, threadIdx.x, smem_u32(bar), parity);
      __trap();
    }
  }
}

// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads)
IDIFF_DEVICE void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
}

// ----------------------------------------------------------------------------------
// TMA tiled loads (global -> shared, completion on an mbarrier)
// ----------------------------------------------------------------------------------
IDIFF_DEVICE void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
IDIFF_DEVICE void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];\n" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
IDIFF_DEVICE void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                              int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];\n" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
IDIFF_DEVICE void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                              int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6}], [%2];\n" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// TMA tiled stores (shared -> global, bulk async-group completion)
IDIFF_DEVICE void tma_store_2d(const CUtensorMap* m, const void* src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];\n" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1)
               : "memory");
}
IDIFF_DEVICE void tma_store_4d(const CUtensorMap* m, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];\n" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
IDIFF_DEVICE void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;\n" ::: "memory"); }
// all bulk groups of this thread have finished READING shared memory (buffers reusable)
IDIFF_DEVICE void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;\n" ::: "memory"); }

// ----------------------------------------------------------------------------------
// tcgen05: TMEM allocation, UMMA issue / commit, TMEM <-> register moves
// ----------------------------------------------------------------------------------
template <uint32_t kCols>
IDIFF_DEVICE void tmem_alloc(uint32_t* smem_dst) {  // whole warp, .sync.aligned
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(
                   smem_u32(smem_dst)),
               "n"(kCols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
template <uint32_t kCols>
IDIFF_DEVICE void tmem_dealloc(uint32_t taddr) {  // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(taddr), "n"(kCols)
               : "memory");
}
IDIFF_DEVICE void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
}
IDIFF_DEVICE void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem], kind::f16 (fp16/bf16 inputs, fp32 accumulate)
IDIFF_DEVICE void umma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier once all previously issued UMMAs of this thread have completed
IDIFF_DEVICE void umma_commit(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(
          smem_u32(bar))
      : "memory");
}
IDIFF_DEVICE void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }
IDIFF_DEVICE void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread `lane` of the warp receives row
// (lane quarter given by warp_id % 4 in the address) and columns [col, col+32).
IDIFF_DEVICE void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
IDIFF_DEVICE void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n" ::"r"(
          taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]),
      "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]),
      "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]),
      "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

// ----------------------------------------------------------------------------------
// UMMA descriptors (bit layout: PTX ISA "tcgen05 shared memory / instruction descriptor")
// ----------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_128B canonical layouts.
//   bits [0,14)  start address >> 4        bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4   bits [46,48) version = 1 (sm_100)
//   bits [61,64) layout type (2 = SWIZZLE_128B)
IDIFF_DEVICE uint64_t make_smem_desc_sw128(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= 1ull << 46;
  d |= 2ull << 61;
  return d;
}
// Instruction descriptor for kind::f16: fp32 accumulate; ab_fmt 0 = fp16, 1 = bf16.
//   [4,6) c fmt (1 = f32)  [7,10) a fmt  [10,13) b fmt  [15] a major  [16] b major (1 = MN-major)
//   [17,23) N >> 3         [24,29) M >> 4
__host__ __device__ constexpr uint32_t make_idesc_f16(uint32_t M, uint32_t N, uint32_t ab_fmt,
                                                      uint32_t a_mn_major, uint32_t b_mn_major) {
  return (1u << 4) | (ab_fmt << 7) | (ab_fmt << 10) | (a_mn_major << 15) | (b_mn_major << 16) |
         ((N >> 3) << 17) | ((M >> 4) << 24);
}

// ----------------------------------------------------------------------------------
// numerics
// ----------------------------------------------------------------------------------
#if IDIFF_STORAGE_BF16
using h16 = __nv_bfloat16;
constexpr uint32_t UMMA_AB_FMT = 1;  // kind::f16 operand format field: bf16
IDIFF_DEVICE uint32_t pack_half2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
IDIFF_DEVICE float2 unpack_half2(uint32_t u) {  // bf16 is the upper half of an fp32: two integer ops
  return make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
}
IDIFF_DEVICE float h2f(h16 x) { return __bfloat162float(x); }
IDIFF_DEVICE h16 f2h(float x) { return __float2bfloat16_rn(x); }
#else
using h16 = __half;
constexpr uint32_t UMMA_AB_FMT = 0;  // fp16
IDIFF_DEVICE uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
IDIFF_DEVICE float2 unpack_half2(uint32_t u) {
  __half2 h = *reinterpret_cast<__half2*>(&u);
  return __half22float2(h);
}
IDIFF_DEVICE float h2f(h16 x) { return __half2float(x); }
IDIFF_DEVICE h16 f2h(float x) { return __float2half_rn(x); }
#endif
IDIFF_DEVICE float silu_f(float x) { return x / (1.0f + __expf(-x)); }
// Exact (erf) GELU of attention.py:43, x * 0.5 * (1 + erf(x / sqrt 2)), with erf from
// Abramowitz-Stegun 7.1.26 (|error| <= 1.5e-7, far below the fp16 output resolution): one MUFU.RCP,
// one MUFU.EX2 and ten FMAs instead of libdevice erff (~2x the instructions).  1 + erf is formed
// without cancellation on the negative side: 1 + erf(-z) = poly(t) * exp(-z^2).
IDIFF_DEVICE float gelu_erf_f(float x) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float t;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  float poly = fmaf(t, 1.061405429f, -1.453152027f);
  poly = fmaf(poly, t, 1.421413741f);
  poly = fmaf(poly, t, -0.284496736f);
  poly = fmaf(poly, t, 0.254829592f);
  poly *= t;
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(z * z * -1.4426950408889634f));
  const float pe = poly * e;                       // = 1 - erf(z)
  const float one_plus_erf = (x >= 0.f) ? (2.0f - pe) : pe;
  return 0.5f * x * one_plus_erf;
}
IDIFF_DEVICE float exp2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

}  // namespace idiff
