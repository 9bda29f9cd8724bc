// Attention v2 for sm_100a (head_dim 40: the 64x64-resolution level that carries 83 % of the
// attention time).  Two 128-query tiles per CTA, 64-key blocks, TWO CTAs PER SM.
//
// Why it looks like this (measurements: tools/micro/umma_bench.cu, IDIFF_ATT2_TRACE timelines,
// profiles/README.md):
//   * d=40 attention is bounded by the MUFU pipe (16 ex2/clk/SM = 2048 clk per 128 keys of a 256-query
//     CTA), but what the first versions actually spent was hand-off latency: every mbarrier wait /
//     arrive, fence.proxy.async, tcgen05.wait::ld and tcgen05.commit round trip costs 100-350 clk,
//     one tcgen05.mma costs >= 45 clk whatever its N, and with two softmax warps per scheduler there
//     is nothing to issue meanwhile.  A traced 64-key step took ~3300 clk of which ~1700 were the 64
//     exponentials; removing the exponentials, the P.V products or the loads each changed nothing.
//   * So the kernel is sized to run two CTAs per SM (<= 113 KB shared memory, 256 TMEM columns,
//     <= 104 registers in the softmax warps): four softmax warps per scheduler from two independent
//     CTAs cover each other's hand-offs, two UMMA issuer threads share the tensor pipe, and one CTA's
//     prologue / epilogue overlaps the other's main loop.
//   * Row sums are accumulated in registers (fp32) instead of a second UMMA per k-step against a
//     block of ones: that halves the UMMA count.
//   * lazy rescaling: the running maximum used for the exponent is only advanced when it grew by
//     more than 2^8 in the exp2 domain, so the O rescale in TMEM is rare (P <= 256 fits fp16).
//   * the UMMA issuer is event-driven: each Q tile advances on its own barriers.
// Warp roles (384 threads = 3 warpgroups): warp 0 TMA producer, warp 1 TMEM allocator + UMMA issuer
// (warps 2-3 idle; the group releases registers with setmaxnreg.dec), warps 4..7 softmax of Q tile 0,
// warps 8..11 softmax of Q tile 1 (one thread per query row).
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {
namespace att2 {

constexpr int THREADS = 384;  // 3 warpgroups: {TMA, UMMA, 2 idle} + softmax(Q0) + softmax(Q1)
constexpr int BQ = 128;
constexpr int BKV = 64;

struct Params {
  int heads, nq, n0, n1, kv1_broadcast;
  float scale_log2e;
  h16* out;
  int out_ld;
  // instance-isolation mask of the gated self-attention (attention.py:187-255): query i may attend key j iff
  // (mask_q[b][i] & mask_k[b][j]) != 0, or j is the visual token i itself (the reference's 1e-9 diagonal)
  const uint32_t* mask_q;  // [batch][nq]
  const uint32_t* mask_k;  // [batch][n0 + n1]
};

template <int D>
struct Cfg {
  static_assert(D <= 64, "attention2 handles one 64-wide d chunk");
  static constexpr int KSTEPS = (D + 15) / 16;
  static constexpr int DV = 64;
  static constexpr int STAGES = 3;
  static constexpr int Q_BYTES = BQ * 128;     // per Q tile
  static constexpr int KV_BYTES = BKV * 128;   // one of K or V: 64 keys x 128 B (64 halves, d <= 64)
  static constexpr int P_BYTES = BQ * 128;     // P of one tile: 128 rows x 64 keys
  static constexpr int BAR_BYTES = 512;
  static constexpr int TRACE_BYTES = 2048;     // TRACE instantiation only
  // 2 x (this + 1 KiB the system reserves per CTA) must fit the SM's 228 KiB: no alignment slack, the
  // kernel checks that the dynamic shared memory window starts 1024-byte aligned.
  static constexpr int SMEM_BYTES = 2 * Q_BYTES + STAGES * 2 * KV_BYTES + 2 * P_BYTES + BAR_BYTES;
  // TMEM columns (256 allocated): S[tile] 64 each, then O[tile] 64 each
  static constexpr int S_COL = 0, O_COL = 128;
  static constexpr int TMEM_COLS = 256;
};

IDIFF_DEVICE void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
IDIFF_DEVICE void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}

// tcgen05.wait::ld that names the registers of the load it completes, so the compiler cannot move a
// consumer of those registers above the wait (the load of block j+1 is in flight during block j).
IDIFF_DEVICE void tmem_ld_wait_dep(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;\n"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]),
                 "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]),
                 "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]),
                 "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]),
                 "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}
IDIFF_DEVICE void st_shared_v4(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}

// ---- packed fp32x2 arithmetic (FFMA2 / FADD2: two lanes per issue slot) and the FMA-pipe exp2 ----
IDIFF_DEVICE uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
IDIFF_DEVICE void unpack_f32x2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
IDIFF_DEVICE uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
IDIFF_DEVICE uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
IDIFF_DEVICE float max3_f(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
// 2^x for two values on the FMA pipe (the MUFU pipe, 16 ex2 / clk / SM, is what bounds head_dim 40): round
// to nearest integer with the 1.5 * 2^23 trick, degree-3 minimax polynomial of 2^r on [-0.5, 0.5]
// (max relative error 7.5e-5, well below the fp16 rounding of P), exponent added in the integer domain.
// Inputs are clamped at -125 (2^-125 ~ 0 next to the row maximum's 2^0..2^8).
IDIFF_DEVICE uint64_t exp2_poly_x2(uint64_t t2) {
  float t0, t1;
  unpack_f32x2(t2, t0, t1);
  t0 = fmaxf(t0, -125.0f);
  t1 = fmaxf(t1, -125.0f);
  const uint64_t tc = pack_f32x2(t0, t1);
  const uint64_t magic = pack_f32x2(12582912.0f, 12582912.0f);
  const uint64_t nmagic = pack_f32x2(-12582912.0f, -12582912.0f);
  const uint64_t z2 = add_f32x2(tc, magic);                                     // integer part in the low mantissa bits
  const uint64_t n2 = add_f32x2(z2, nmagic);                                    // ... as a float
  const uint64_t r2 = fma_f32x2(n2, pack_f32x2(-1.0f, -1.0f), tc);              // r = t - n in [-0.5, 0.5]
  uint64_t p2 = fma_f32x2(r2, pack_f32x2(0.0551716685f, 0.0551716685f), pack_f32x2(0.2426111251f, 0.2426111251f));
  p2 = fma_f32x2(p2, r2, pack_f32x2(0.6932609677f, 0.6932609677f));
  p2 = fma_f32x2(p2, r2, pack_f32x2(0.9999280572f, 0.9999280572f));
  float p0, p1, z0, z1;
  unpack_f32x2(p2, p0, p1);
  unpack_f32x2(z2, z0, z1);
  const float e0 = __int_as_float(__float_as_int(p0) + (__float_as_int(z0) << 23));
  const float e1 = __int_as_float(__float_as_int(p1) + (__float_as_int(z1) << 23));
  return pack_f32x2(e0, e1);
}

// exponentials of one 64-key block of a row: P (fp16 pairs) and their fp32 sum.  MASK bit (u mod 8) = pair u
// takes the FMA-pipe exp2.
template <uint32_t MASK>
IDIFF_DEVICE float exp_block(const uint32_t (&sv)[2][32], float c, float mc, uint32_t (&pk)[32]) {
  uint64_t sumA = 0ull, sumB = 0ull;  // two independent packed accumulators (bit pattern of +0.0f pairs)
  const uint64_t c2 = pack_f32x2(c, c), nmc2 = pack_f32x2(-mc, -mc);
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      const uint64_t t2 = fma_f32x2(pack_f32x2(__uint_as_float(sv[hh][2 * u]), __uint_as_float(sv[hh][2 * u + 1])), c2, nmc2);
      uint64_t e2;
      if ((MASK >> (u & 7)) & 1u) {
        e2 = exp2_poly_x2(t2);
      } else {
        float t0, t1;
        unpack_f32x2(t2, t0, t1);
        e2 = pack_f32x2(exp2_approx(t0), exp2_approx(t1));
      }
      if (u & 1) sumB = add_f32x2(sumB, e2);
      else sumA = add_f32x2(sumA, e2);
      float e0, e1;
      unpack_f32x2(e2, e0, e1);
      pk[hh * 16 + u] = pack_half2(e0, e1);
    }
  }
  float sa0, sa1, sb0, sb1;
  unpack_f32x2(sumA, sa0, sa1);
  unpack_f32x2(sumB, sb0, sb1);
  return (sa0 + sa1) + (sb0 + sb1);
}

// TRACE (IDIFF_ATT2_TRACE=1): one CTA records clock stamps of blocks 16..23 in shared memory and prints
// them at exit -- a timeline of the hand-offs that costs the measured kernel nothing but a few STS.
// POLY: bit u of the mask = pair u (mod 8) of every 8 score pairs takes the FMA-pipe exp2 instead of MUFU.
// MASKED: the instance-isolation mask of Params::mask_q / mask_k is applied to the scores.
template <int D, bool TRACE = false, uint32_t POLY = 0, bool MASKED = false>
__global__ void __launch_bounds__(THREADS, 2)
attention2_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK0,
                  const __grid_constant__ CUtensorMap tmV0, const __grid_constant__ CUtensorMap tmK1,
                  const __grid_constant__ CUtensorMap tmV1, const Params p) {
  using C = Cfg<D>;
  constexpr int STAGES = C::STAGES;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) {  // SWIZZLE_128B tiles need it; no slack is budgeted (see Cfg)
    if (threadIdx.x == 0) printf("idiff: attention2 shared memory window not 1024-byte aligned\n");
    __trap();
  }
  uint8_t* sQ = smem;                                  // [2][16 KiB]
  uint8_t* sK = sQ + 2 * C::Q_BYTES;                   // [STAGES][8 KiB]
  uint8_t* sV = sK + STAGES * C::KV_BYTES;             // [STAGES][8 KiB]
  uint8_t* sP = sV + STAGES * C::KV_BYTES;             // [tile][16 KiB]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * C::P_BYTES);
  uint64_t* q_full = bars;               // 1
  uint64_t* k_full = bars + 1;           // STAGES
  uint64_t* v_full = k_full + STAGES;    // STAGES
  uint64_t* kv_empty = v_full + STAGES;  // STAGES
  uint64_t* s_full = kv_empty + STAGES;  // [tile]
  uint64_t* s_free = s_full + 2;         // [tile] (128 arrivals)
  uint64_t* p_full = s_free + 2;         // [tile] (128 arrivals)
  uint64_t* pv_done = p_full + 2;        // [tile]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 2);
  uint32_t* trace_buf = reinterpret_cast<uint32_t*>(sP + 2 * C::P_BYTES + C::BAR_BYTES);  // TRACE only
  const bool traced = TRACE && blockIdx.x == 3 && blockIdx.y == 2 && blockIdx.z == 0;
  auto stamp = [&](int slot) {
    if (TRACE && traced) trace_buf[slot] = clock();
  };

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * 2 * BQ;
  const int h = blockIdx.y;
  const int b = blockIdx.z;
  const int T0 = (p.n0 + BKV - 1) / BKV;
  const int T1 = (p.n1 + BKV - 1) / BKV;
  const int T = T0 + T1;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK0);
    tma_prefetch_desc(&tmV0);
    mbar_init(q_full, 1);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 128);
      mbar_init(&p_full[i], 128);
      mbar_init(&pv_done[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<C::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Register re-partition between warpgroups (the setmaxnreg must sit at the head of each role
  // branch so that ptxas allocates the branch bodies against the new limits).
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 32;\n");
  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(q_full, 2 * C::Q_BYTES);
      tma_load_4d(sQ, &tmQ, q_full, 0, h, q0, b);
      tma_load_4d(sQ + C::Q_BYTES, &tmQ, q_full, 0, h, q0 + BQ, b);
      for (int j = 0; j < T; ++j) {
        const int s = j % STAGES;
        mbar_wait(&kv_empty[s], ((j / STAGES) & 1) ^ 1);
        const bool seg1 = j >= T0;
        const int row = (seg1 ? (j - T0) : j) * BKV;
        const int bb = seg1 ? (p.kv1_broadcast ? 0 : b) : b;
        mbar_expect_tx(&k_full[s], C::KV_BYTES);
        tma_load_4d(sK + s * C::KV_BYTES, seg1 ? &tmK1 : &tmK0, &k_full[s], 0, h, row, bb);
        mbar_expect_tx(&v_full[s], C::KV_BYTES);
        tma_load_4d(sV + s * C::KV_BYTES, seg1 ? &tmV1 : &tmV0, &v_full[s], 0, h, row, bb);
      }
    }
  } else if (warp == 1) {
    // ===================== UMMA issuer =====================
    // All 32 lanes walk the event loop with warp-uniform control flow (every barrier probe is made uniform
    // by a vote) and ONE elected lane issues: as a single-lane loop the descriptors lived in vector registers
    // and every tcgen05.mma cost ~10 instructions (R2UR moves + an ELECT retry loop) on the one thread whose
    // instruction latency paces both Q tiles of the CTA -- 14 UMMAs, 4-5 commits and ~8 barrier probes per
    // 64-key step.  Uniform, the UMMAs of a product issue back to back from uniform registers (gemm2.cu, same
    // measurement).  Stage / phase of every ring are running counters (no div / mod by 3).
    {
      constexpr uint32_t idesc_qk = make_idesc_f16(BQ, BKV, UMMA_AB_FMT, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_f16(BQ, C::DV, UMMA_AB_FMT, 0, /*B MN-major*/ 1);
      // Every descriptor here shares its high word (SBO = 1024 B, version 1, SWIZZLE_128B); the low
      // word is (address >> 4) | (LBO >> 4) << 16, so stepping an operand by X bytes is lo += X >> 4.
      constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);
      constexpr uint32_t LBO_K = (16u >> 4) << 16;             // K-major operands (unused field)
      constexpr uint32_t LBO_V = ((BKV * 128u) >> 4) << 16;    // MN-major V: next 64-wide d chunk (unused)
      const uint32_t q_lo0 = (smem_u32(sQ) >> 4) | LBO_K;
      const uint32_t p_lo0 = (smem_u32(sP) >> 4) | LBO_K;
      const uint32_t k_lo0 = (smem_u32(sK) >> 4) | LBO_K;
      const uint32_t v_lo0 = (smem_u32(sV) >> 4) | LBO_V;
      auto umma_lo = [&](uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t acc) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
            "mov.b64 da, {%1, %3};\n\t"
            "mov.b64 db, {%2, %3};\n\t"
            "setp.ne.b32 p, %5, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}\n" ::"r"(d_tmem),
            "r"(a_lo), "r"(b_lo), "r"(DESC_HI), "r"(idesc), "r"(acc)
            : "memory");
      };
      // per Q tile: next block of Q.K^T / P.V, and the ring stage / phase of its K and V tiles
      int qk_n[2] = {0, 0}, pv_n[2] = {0, 0};
      uint32_t qk_s[2] = {0, 0}, qk_ph[2] = {0, 0}, pv_s[2] = {0, 0}, pv_ph[2] = {0, 0};
      mbar_wait(q_full, 0);
      long long t_idle = 0;
      while (pv_n[0] < T || pv_n[1] < T) {
        bool progress = false;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          // ---- S[q] = Q_q . K(n)^T once S[q] has been pulled into registers and K(n) has landed ----
          const int nq = qk_n[q];
          bool go = false;
          if (nq < T) go = (nq == 0 || mbar_test(&s_free[q], (nq - 1) & 1)) && mbar_test(&k_full[qk_s[q]], qk_ph[q]);
          if (__any_sync(0xffffffffu, go)) {  // completion is monotonic: any lane's observation holds for all
            tc_fence_after();
            if (TRACE && lane == 0 && nq >= 16 && nq < 24) stamp(128 + (q * 8 + nq - 16) * 4 + 0);
            if (elect_one()) {
              const uint32_t q_lo = q_lo0 + q * (C::Q_BYTES >> 4);
              const uint32_t k_lo = k_lo0 + qk_s[q] * (C::KV_BYTES >> 4);
              const uint32_t d_tmem = tmem_base + C::S_COL + q * 64;
#pragma unroll
              for (int kk = 0; kk < C::KSTEPS; ++kk) umma_lo(d_tmem, q_lo + kk * 2, k_lo + kk * 2, idesc_qk, kk > 0 ? 1u : 0u);
              umma_commit(&s_full[q]);
            }
            __syncwarp();
            if (TRACE && lane == 0 && nq >= 16 && nq < 24) stamp(128 + (q * 8 + nq - 16) * 4 + 1);
            qk_n[q] = nq + 1;
            if (++qk_s[q] == STAGES) {
              qk_s[q] = 0;
              qk_ph[q] ^= 1;
            }
            progress = true;
          }
          // ---- O[q] += P[q] . V(n) once P[q] is in shared memory and V(n) has landed ----
          const int np = pv_n[q];
          go = false;
          if (np < qk_n[q]) go = mbar_test(&p_full[q], np & 1) && mbar_test(&v_full[pv_s[q]], pv_ph[q]);
          if (__any_sync(0xffffffffu, go)) {
            tc_fence_after();
            if (TRACE && lane == 0 && np >= 16 && np < 24) stamp(128 + (q * 8 + np - 16) * 4 + 2);
            if (elect_one()) {
              const uint32_t v_lo = v_lo0 + pv_s[q] * (C::KV_BYTES >> 4);
              const uint32_t p_lo = p_lo0 + q * (C::P_BYTES >> 4);
              const uint32_t o_tmem = tmem_base + C::O_COL + q * 64;
              const uint32_t acc0 = np > 0 ? 1u : 0u;
#pragma unroll
              for (int kk = 0; kk < BKV / 16; ++kk)
                umma_lo(o_tmem, p_lo + kk * 2, v_lo + kk * (2048 >> 4), idesc_pv, kk > 0 ? 1u : acc0);
              umma_commit(&pv_done[q]);
              if (pv_n[q ^ 1] > np) umma_commit(&kv_empty[pv_s[q]]);  // both tiles are past block np
            }
            __syncwarp();
            if (TRACE && lane == 0 && np >= 16 && np < 24) stamp(128 + (q * 8 + np - 16) * 4 + 3);
            pv_n[q] = np + 1;
            if (++pv_s[q] == STAGES) {
              pv_s[q] = 0;
              pv_ph[q] ^= 1;
            }
            progress = true;
          }
        }
        if (progress) {
          t_idle = 0;
        } else {  // bounded like mbar_wait: a protocol bug traps instead of hanging the GPU
          if (t_idle == 0) t_idle = clock64();
          else if (clock64() - t_idle > 8000000000LL) {
            if (lane == 0)
              printf("idiff: attention2 issue loop stalled block=(%d,%d,%d) qk=(%d,%d) pv=(%d,%d)\n", blockIdx.x,
                     blockIdx.y, blockIdx.z, qk_n[0], qk_n[1], pv_n[0], pv_n[1]);
            __trap();
          }
        }
      }
    }
    __syncwarp();
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;\n");
    // ===================== softmax / correction / epilogue =====================
    const int q = (warp - 4) >> 2;  // Q tile of this warp group
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const uint32_t s_addr = tmem_base + lane_off + C::S_COL + q * 64;
    const uint32_t o_addr = tmem_base + lane_off + C::O_COL + q * 64;
    const float c = p.scale_log2e;
    const uint32_t p_row = smem_u32(sP + q * C::P_BYTES + r * 128);
    const uint32_t sw = r & 7;

    float m_used = -INFINITY;  // maximum the exponent is taken against (raw score units)
    float l = 0.0f;            // running row sum of exp
    uint32_t qword = 0xffffffffu;
    if (MASKED) {
      const int qrow_m = q0 + q * BQ + r;
      qword = qrow_m < p.nq ? __ldg(p.mask_q + (long)b * p.nq + qrow_m) : 0xffffffffu;
    }

    for (int j = 0; j < T; ++j) {
      const bool tr = TRACE && r == 0 && j >= 16 && j < 24;
      const int tb = (q * 8 + ((j - 16) & 7)) * 8;
      if (tr) stamp(tb + 0);
      const bool seg1 = j >= T0;
      const int nv = min(BKV, (seg1 ? p.n1 : p.n0) - (seg1 ? (j - T0) : j) * BKV);
      // ---- scores of block j: TMEM -> registers, S released for Q.K(j+1)^T ----
      uint32_t sv[2][32];
      mbar_wait(&s_full[q], j & 1);
      tc_fence_after();
      if (tr) stamp(tb + 1);
      tmem_ld_32x32b_x32(s_addr, sv[0]);
      tmem_ld_32x32b_x32(s_addr + 32, sv[1]);
      tmem_ld_wait_dep(sv[0]);
      tmem_ld_wait_dep(sv[1]);
      tc_fence_before();
      mbar_arrive(&s_free[q]);
      if (tr) stamp(tb + 2);
      if (nv < BKV) {  // ragged last block of a segment: keys past the end score -inf
#pragma unroll
        for (int jj = 0; jj < BKV; ++jj)
          if (jj >= nv) sv[jj >> 5][jj & 31] = 0xff800000u;
      }
      if (MASKED) {
        // the 64 key words of this block (the same for every thread: L1 broadcast) against this row's word
        const int key0 = (seg1 ? p.n0 + (j - T0) * BKV : j * BKV);
        const uint4* kw = reinterpret_cast<const uint4*>(p.mask_k + (long)b * (p.n0 + p.n1) + key0);
        const int self_jj = seg1 ? -1 : (q0 + q * BQ + r) - key0;  // this row's own key, if it lies in the block
#pragma unroll
        for (int g = 0; g < BKV / 4; ++g) {
          uint4 w = make_uint4(0, 0, 0, 0);
          if (4 * g < nv) w = __ldg(kw + g);  // (n0 and n1 blocks start 4-word aligned: n0 % 4 == 0 is required)
          const uint32_t ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int jj = 4 * g + e;
            if ((ww[e] & qword) == 0u && jj != self_jj) sv[jj >> 5][jj & 31] = 0xff800000u;
          }
        }
      }
      float m0 = -INFINITY, m1 = -INFINITY, m2 = -INFINITY, m3 = -INFINITY;
#pragma unroll
      for (int jj = 0; jj < 32; jj += 4) {  // 3-input max: two scores per issue slot
        m0 = max3_f(m0, __uint_as_float(sv[0][jj]), __uint_as_float(sv[0][jj + 1]));
        m1 = max3_f(m1, __uint_as_float(sv[0][jj + 2]), __uint_as_float(sv[0][jj + 3]));
        m2 = max3_f(m2, __uint_as_float(sv[1][jj]), __uint_as_float(sv[1][jj + 1]));
        m3 = max3_f(m3, __uint_as_float(sv[1][jj + 2]), __uint_as_float(sv[1][jj + 3]));
      }
      const float m_blk = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
      // lazy maximum: only move the reference when it grew by more than 8 in the exp2 domain
      float alpha = 1.0f;
      if (m_blk > m_used && (m_blk - m_used) * c > 8.0f) {
        alpha = exp2_approx((m_used - m_blk) * c);  // first block: 2^-inf = 0 (l = 0, O is not read)
        m_used = m_blk;
      }
      // (MASKED: a block may be dead for a row before the row has seen any live key: m_used is still -inf and the
      // scores are all -inf; exponent against 0 then gives P = 0 instead of NaN)
      const float mc = (MASKED && m_used == -INFINITY) ? 0.0f : m_used * c;
      if (tr) stamp(tb + 3);
      // ---- exponentials, packed to fp16 in place; row sum in fp32 ----
      // Packed fp32x2 arithmetic for the exponent argument and the row sum (one issue slot per two scores);
      // a POLY share of the pairs takes exp2 on the FMA pipe so that MUFU (8 clk per warp instruction per
      // scheduler) and the issue slots run out together.  A ragged block (masked -inf scores) keeps MUFU
      // (a real, warp-uniform branch: as one predicated block ptxas evaluated both variants and selected).
      uint32_t pk[32];
      float blk_sum;
      if (POLY != 0 && nv == BKV) blk_sum = exp_block<POLY>(sv, c, mc, pk);
      else blk_sum = exp_block<0u>(sv, c, mc, pk);
      l = fmaf(l, alpha, blk_sum);
      if (tr) stamp(tb + 4);
      // ---- P buffer free (P.V(j-1) done); rare O rescale; P -> shared memory ----
      if (j > 0) {
        mbar_wait(&pv_done[q], (j - 1) & 1);
        tc_fence_after();
        if (__any_sync(0xffffffffu, alpha != 1.0f)) {
          // the reference maximum moved: O is scaled while no P.V of this tile is in flight
#pragma unroll
          for (int c0 = 0; c0 < 64; c0 += 16) {
            uint32_t o[16];
            tmem_ld_32x32b_x16(o_addr + c0, o);
            tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) o[jj] = __float_as_uint(__uint_as_float(o[jj]) * alpha);
            tmem_st_32x32b_x16(o_addr + c0, o);
          }
          tmem_st_wait();
        }
      }
      if (tr) stamp(tb + 5);
      // 64 keys of this row -> 128 B of the swizzled P tile (SWIZZLE_128B: 16-byte chunk i of row r
      // sits at chunk i ^ (r & 7))
#pragma unroll
      for (int i = 0; i < 8; ++i)
        st_shared_v4(p_row + ((static_cast<uint32_t>(i) ^ sw) << 4), pk[4 * i], pk[4 * i + 1], pk[4 * i + 2],
                     pk[4 * i + 3]);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(&p_full[q]);
      if (tr) stamp(tb + 6);
    }

    // epilogue: O / l -> fp16 (UMMAs of one thread complete in order: the last P.V done = all done)
    mbar_wait(&pv_done[q], (T - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.0f / l;
    const int qrow = q0 + q * BQ + r;
    const bool row_ok = qrow < p.nq;
    h16* orow = p.out + ((long)b * p.nq + qrow) * p.out_ld + h * D;
#pragma unroll
    for (int c0 = 0; c0 < 64; c0 += 32) {
      if (c0 >= D) break;
      uint32_t o[32];
      tmem_ld_32x32b_x32(o_addr + c0, o);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8) {
          if (c0 + j8 * 8 < D) {
            uint4 ov;
            ov.x = pack_half2(__uint_as_float(o[j8 * 8 + 0]) * inv_l, __uint_as_float(o[j8 * 8 + 1]) * inv_l);
            ov.y = pack_half2(__uint_as_float(o[j8 * 8 + 2]) * inv_l, __uint_as_float(o[j8 * 8 + 3]) * inv_l);
            ov.z = pack_half2(__uint_as_float(o[j8 * 8 + 4]) * inv_l, __uint_as_float(o[j8 * 8 + 5]) * inv_l);
            ov.w = pack_half2(__uint_as_float(o[j8 * 8 + 6]) * inv_l, __uint_as_float(o[j8 * 8 + 7]) * inv_l);
            *reinterpret_cast<uint4*>(orow + c0 + j8 * 8) = ov;
          }
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
  if (TRACE && traced && threadIdx.x == 0) {
    const uint32_t t0 = trace_buf[0];
    for (int q = 0; q < 2; ++q)
      for (int j = 0; j < 8; ++j) {
        const uint32_t* tr = trace_buf + (q * 8 + j) * 8;
        printf("smx q=%d j=%2d: start %6u | S ready +%4u | S in regs +%4u | max/alpha +%4u | exps done +%4u | P free +%4u "
               "| p_full +%4u\n", q, j + 16, tr[0] - t0, tr[1] - tr[0], tr[2] - tr[0], tr[3] - tr[0], tr[4] - tr[0],
               tr[5] - tr[0], tr[6] - tr[0]);
      }
    for (int q = 0; q < 2; ++q)
      for (int n = 0; n < 8; ++n) {
        const uint32_t* tr = trace_buf + 128 + (q * 8 + n) * 4;
        printf("mma q=%d n=%2d: QK issue %6u (+%3u) | PV issue %6u (+%3u)\n", q, n + 16, tr[0] - t0, tr[1] - tr[0],
               tr[2] - t0, tr[3] - tr[2]);
      }
  }
}

int attention_v2_d40(const idiff_attn_args* a, cudaStream_t stream) {
  constexpr int D = 40;
  using C = Cfg<D>;
  CUtensorMap tmQ, tmK0, tmV0, tmK1, tmV1;
  if (make_head_tmap(&tmQ, a->q, D, a->heads, a->nq, a->batch, a->q_ld, BQ)) return -1;
  if (make_head_tmap(&tmK0, a->k0, D, a->heads, a->n0, a->batch, a->k0_ld, BKV)) return -1;
  if (make_head_tmap(&tmV0, a->v0, D, a->heads, a->n0, a->batch, a->v0_ld, BKV)) return -1;
  if (a->n1 > 0) {
    const int b1 = a->kv1_batch == 1 ? 1 : a->batch;
    if (make_head_tmap(&tmK1, a->k1, D, a->heads, a->n1, b1, a->k1_ld, BKV)) return -1;
    if (make_head_tmap(&tmV1, a->v1, D, a->heads, a->n1, b1, a->v1_ld, BKV)) return -1;
  } else {
    tmK1 = tmK0;
    tmV1 = tmV0;
  }
  Params p;
  p.heads = a->heads;
  p.nq = a->nq;
  p.n0 = a->n0;
  p.n1 = a->n1;
  p.kv1_broadcast = (a->kv1_batch == 1) ? 1 : 0;
  p.scale_log2e = a->scale * 1.4426950408889634f;
  p.out = reinterpret_cast<h16*>(a->out);
  p.out_ld = a->out_ld;
  p.mask_q = reinterpret_cast<const uint32_t*>(a->mask_q);
  p.mask_k = reinterpret_cast<const uint32_t*>(a->mask_k);
  static const bool trace = getenv("IDIFF_ATT2_TRACE") != nullptr;
  const bool masked = a->mask_q != nullptr;
  // unmasked: pairs 1 and 5 of every 8 score pairs take the FMA-pipe exp2 (measured on a B200, batch 8, 4096 keys:
  // 408 us, against 420 / 430 / 456 us for 0 / 3 / 4 of 8 pairs)
  auto kern = masked ? attention2_kernel<D, false, 0u, true>
              : trace ? attention2_kernel<D, true, 0u>
                      : attention2_kernel<D, false, 0x22u>;
  const int smem_bytes = C::SMEM_BYTES + (trace ? C::TRACE_BYTES : 0);
  static bool attr_set[2] = {false, false};  // (per masked / unmasked kernel; IDIFF_ATT2_TRACE is read once)
  if (!attr_set[masked]) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
    attr_set[masked] = true;
  }
  dim3 grid((a->nq + 2 * BQ - 1) / (2 * BQ), a->heads, a->batch);
  kern<<<grid, THREADS, smem_bytes, stream>>>(tmQ, tmK0, tmV0, tmK1, tmV1, p);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace att2
}  // namespace idiff
