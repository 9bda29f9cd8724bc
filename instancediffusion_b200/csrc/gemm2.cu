// GEMM v2 for sm_100a: persistent, stream-K balanced tcgen05 GEMM / implicit-GEMM conv3x3.
//
//   out[M, N] = epilogue( A[M, K] . W[N, K]^T )        fp16 operands, fp32 accumulation in TMEM
//
// Replaces (reference file:line): attention.py:41,62,121-125,175-179,297,354,363;
// openaimodel.py:109,134,186,205,213,361-363,464; text_grounding_net.py:75-81; convnext.py:30-32,71-81.
// Design points, driven by the measured shape mix of the UNet (profiles/r1_v0_launches_forward_b8.csv;
// the round-1 one-tile-per-CTA kernel this replaced is in the git history, not in the tree):
//   * one persistent CTA per SM; work = (128 x BN tile, k-block range) segments.  Full waves of
//     tiles are processed data-parallel; the ragged last 1-2 waves are split evenly over all CTAs
//     in units of 64-wide k-blocks ("stream-K"), so 40-, 160- and 320-tile problems no longer leave
//     most SMs idle.  A tile shared by several CTAs is finished by the CTA that holds its first
//     k-blocks; the others publish fp32 partials (coalesced, L2-resident) and a per-warp flag, and
//     the owner adds them in a fixed order -> bit-reproducible.
//   * BN in {128, 160, 192, 256} chosen per N (320 = 2 x 160, 960 = 5 x 192, 1280 = 5 x 256 ...):
//     no padded columns, half the A-tile traffic of 128-wide tiles.
//   * two TMEM accumulator buffers: the epilogue of segment i overlaps the MMAs of segment i+1;
//     8 epilogue warps (2 per TMEM lane quarter) so short-K layers are not epilogue-bound.
//   * epilogue (measured with the built-in per-CTA phase trace, tools/trace_gemm.py): per-tile
//     bias / time-embedding terms come from a shared-memory table; short-K layers move the residual
//     in and the result out as TMA boxes through a swizzled staging buffer (compact rolled loop);
//     long-K convolutions keep the deep operand ring and prefetch their residual rows into
//     registers before the accumulator is ready.  One kernel per (BN, epilogue mode, TMA epilogue).
// Warp roles (384 threads = 3 warpgroups): warp 0 TMA producer, warp 1 TMEM allocator + UMMA
// issuer (warps 2-3 idle; the group gives registers back with setmaxnreg), warps 4..11 epilogue.
// conv3x3 gathers the A tile tap by tap with a 4-D TMA box over the NHWC activation; out-of-image taps
// are zero-filled by the TMA unit (no im2col buffer, no halo copy).
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

#include <stdlib.h>

namespace idiff {
namespace v2 {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int A_STAGE_BYTES = BM * BK * 2;
// Warpgroup 0 = {TMA, UMMA, 2 idle warps}; then EW epilogue warps (EW / 4 per TMEM lane quarter: two column
// halves, 224 registers per epilogue warp).  12 / 16 epilogue warps and CTA pairs (cta_group::2) were measured
// slower or no faster: profiles/README.md round 2, sections 7.3 and 7.5.
constexpr int EW = 8;
constexpr int CHUNK = 16;  // accumulator columns per tcgen05.ld
constexpr int EPI_TAB_PB = 4;  // batches a conv tile may straddle and still use the smem epilogue table

struct Params {
  int M, N, K, KB;
  int n_tiles, T, T_dp, G;
  long U_sk;  // stream-K units (k-blocks) = (T - T_dp) * KB
  // conv geometry
  int conv, H, W, Bn, PW, PH, PB, tiles_w, tiles_h, kb_per_tap;
  // epilogue
  const float* bias;
  const h16* rowadd;
  const h16* residual;
  void* out;
  int ldo, ldr, ldra, rows_per_batch, flags;
  float gate;
  // stream-K fixup
  float* ws;    // [G][BN/CHUNK][128][CHUNK] fp32 partial tiles
  int* sflags;  // [G][EW] publish flags (fixed location, self-resetting)
  unsigned long long* trace;  // optional [G][8] %globaltimer stamps (idiff_set_gemm_trace), else null
  // LayerNorm folded across GEMMs (header: ln_* fields)
  float2* ln_out;        // producer: [n_tiles * PARTS][M] partial (sum, sumsq) of the output rows
  const float2* ln_in;   // consumer: [ln_slots][M] partials of the A rows
  const float* ln_s;     // consumer: [N] column sums of the gamma-folded fp16 weights
  int ln_slots;
  float ln_eps;
};

// TMA_EPI: the epilogue moves the residual in and the result out through shared memory with
// bulk-tensor copies ([32 rows x 16 cols] boxes, one per warp and 16-column chunk) instead of one
// 16-byte global access per thread and row (which costs an L1 transaction per access: measured
// ~0.7 us per chunk, tools/trace_gemm.py).  The staging buffer takes smem from the operand ring,
// so it is used for the short-K layers (epilogue-bound); long-K convolutions keep the deep ring.
template <int BN, bool TMA_EPI>
struct Cfg {
  static constexpr int THREADS = 128 + EW * 32;
  static constexpr int PARTS = EW / 4;            // column parts of a tile (one epilogue warp per quarter and part)
  static constexpr int NCHT = BN / CHUNK;         // 16-column accumulator chunks of a tile
  static constexpr int NCH_MAX = (NCHT + PARTS - 1) / PARTS;  // ... owned by one warp, at most
  static constexpr int B_STAGE_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_STAGE_BYTES + B_STAGE_BYTES;
  static constexpr int BOX_BYTES = 32 * CHUNK * 2;                       // 1 KiB
  // TMA epilogue staging: one [32 rows x BN/2 columns] fp16 box per epilogue warp (row-major, no swizzle):
  // the residual lands in it with ONE bulk-tensor load per warp and tile, the result leaves with ONE store
  static constexpr int WBOX_BYTES = 32 * (BN / 2) * 2;
  static constexpr int STG_BYTES = TMA_EPI ? EW * WBOX_BYTES : 0;
  static constexpr int TAB_BYTES = 2 * EPI_TAB_PB * BN * 4;
  static constexpr int BAR_BYTES = 1024;  // 2*STAGES + 4 + EW mbarriers + the TMEM base slot;
                                          // 1 KiB keeps the staging boxes 1024-byte aligned (SWIZZLE_128B boxes)
  static constexpr int FIXED = 1024 + BAR_BYTES + TAB_BYTES + STG_BYTES;
  static constexpr int STAGES_FIT = (227 * 1024 - FIXED) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_FIT > 6 ? 6 : STAGES_FIT;
  static constexpr int ACC_STRIDE = (BN <= 128) ? 128 : 256;
  static constexpr int TMEM_COLS = 2 * ACC_STRIDE;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + FIXED;
  static_assert(STAGES >= 3, "operand ring too shallow");
};

struct Seg {
  int tile, kb0, kb1;
};

// Work iterator shared by the three roles: stream-K range first, then data-parallel tiles.
struct WorkIter {
  const Params& p;
  int cta;
  long u, u1;  // stream-K cursor / end (units)
  int dp_next;
  __device__ WorkIter(const Params& p_, int cta_) : p(p_), cta(cta_) {
    u = (p.U_sk * cta) / p.G;
    u1 = (p.U_sk * (cta + 1)) / p.G;
    dp_next = cta;
  }
  __device__ bool next(Seg& s) {
    if (u < u1) {
      const int t_local = (int)(u / p.KB);
      const int kb0 = (int)(u - (long)t_local * p.KB);
      const long rem = u1 - u;
      const int kb1 = (rem < (long)(p.KB - kb0)) ? (int)(kb0 + rem) : p.KB;
      s.tile = p.T_dp + t_local;
      s.kb0 = kb0;
      s.kb1 = kb1;
      u += kb1 - kb0;
      return true;
    }
    if (dp_next < p.T_dp) {
      s.tile = dp_next;
      s.kb0 = 0;
      s.kb1 = p.KB;
      dp_next += p.G;
      return true;
    }
    return false;
  }
};

IDIFF_DEVICE void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
      "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
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

IDIFF_DEVICE int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];\n" : "=r"(v) : "l"(p) : "memory");
  return v;
}
IDIFF_DEVICE void st_release_gpu(int* p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}

// ---- packed fp32x2 arithmetic (FADD2 / FFMA2: two values per issue slot) for the epilogue ----
IDIFF_DEVICE uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
IDIFF_DEVICE void f2_unpack(uint64_t v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
IDIFF_DEVICE uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
IDIFF_DEVICE uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
IDIFF_DEVICE uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// value * gelu(gate) for two elements at once: gelu_erf_f (common.cuh) restated on packed pairs.  With
// a = |g|, z = a / sqrt 2, pe = poly(t) * exp(-z^2) = 1 - erf(z):  gelu(g) = 0.5 * ((g + a) - a * pe)
// (g + a is exactly 2g or 0, so the negative side has no cancellation).  Per pair: 2 LOP, 13 packed FP
// ops and 4 MUFU against ~36 scalar instructions: the K = 320 GEGLU projection was bound by its epilogue's
// issue slots (ncu: issue 47 %, XU 31 %, tensor 37 %; profiles/r2_ncu_geglu320.summary.csv).
IDIFF_DEVICE uint64_t geglu_f2(uint64_t val, uint64_t g) {
  float g0, g1;
  f2_unpack(g, g0, g1);
  const uint64_t a = f2_pack(fabsf(g0), fabsf(g1));
  const uint64_t z = f2_mul(a, f2_pack(0.70710678118654752f, 0.70710678118654752f));
  float d0, d1, t0, t1;
  f2_unpack(f2_fma(z, f2_pack(0.3275911f, 0.3275911f), f2_pack(1.0f, 1.0f)), d0, d1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(d0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(d1));
  const uint64_t t = f2_pack(t0, t1);
  uint64_t poly = f2_fma(t, f2_pack(1.061405429f, 1.061405429f), f2_pack(-1.453152027f, -1.453152027f));
  poly = f2_fma(poly, t, f2_pack(1.421413741f, 1.421413741f));
  poly = f2_fma(poly, t, f2_pack(-0.284496736f, -0.284496736f));
  poly = f2_fma(poly, t, f2_pack(0.254829592f, 0.254829592f));
  poly = f2_mul(poly, t);
  float x0, x1, e0, e1;
  f2_unpack(f2_mul(f2_mul(z, z), f2_pack(-1.4426950408889634f, -1.4426950408889634f)), x0, x1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(x0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(x1));
  const uint64_t pe = f2_mul(poly, f2_pack(e0, e1));
  const uint64_t two_gelu = f2_fma(f2_mul(a, f2_pack(-1.0f, -1.0f)), pe, f2_add(g, a));  // (g + a) - a * pe
  return f2_mul(f2_mul(val, f2_pack(0.5f, 0.5f)), two_gelu);
}
IDIFF_DEVICE void lds_f2x2(uint32_t a, uint64_t& p0, uint64_t& p1) {  // four floats as two packed pairs
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];\n" : "=l"(p0), "=l"(p1) : "r"(a));
}

// The short-K epilogue of one warp, specialised at compile time (the all-flags loop spent ~60 of its 142
// instructions per 16-column chunk on uniform flag tests and trace hooks, and the warp is instruction-latency
// bound: two epilogue warps per scheduler, ~6.5 clk per dependent instruction; ncu source view, profiles/).
// Plain linear layer: acc (+ LayerNorm fold) + bias, optional gate * x + residual, optional row statistics.
// Packed fp32x2 arithmetic throughout.  trow: TMEM address of this warp's lane quarter; tab_s: epilogue table
// (row 0 bias, row 1 column sums); row_s: this thread's row of the staging box; c_first: first accumulator
// column of the warp; nlive: live 16-column chunks.
template <int BN, int WCOLS, bool RES, bool LNI, bool LNO>
IDIFF_DEVICE void epi_chunks_plain(uint32_t trow, uint32_t tab_s, uint32_t row_s, int c_first, int nlive, uint32_t lane,
                                   float gate, float ln_rstd, float ln_b, float& ln_ps, float& ln_pq) {
  const uint64_t gate2 = f2_pack(gate, gate), rstd2 = f2_pack(ln_rstd, ln_rstd), lnb2 = f2_pack(ln_b, ln_b);
  uint64_t ps2 = 0ull, pq2 = 0ull;  // (+0.0f, +0.0f)
#pragma unroll 1
  for (int ch = 0; ch < nlive; ++ch) {
    const int c0 = c_first + ch * CHUNK;
    uint32_t v[CHUNK];
    tmem_ld_32x32b_x16(trow + c0, v);
    tmem_ld_wait();
    uint64_t x2[CHUNK / 2];
#pragma unroll
    for (int j = 0; j < CHUNK / 2; ++j) x2[j] = f2_pack(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint64_t b0, b1;
      lds_f2x2(tab_s + (c0 + 4 * q) * 4, b0, b1);
      if (LNI) {  // y = rstd * acc + (-mean * rstd) * colsum + bias
        uint64_t s0, s1;
        lds_f2x2(tab_s + (BN + c0 + 4 * q) * 4, s0, s1);
        x2[2 * q] = f2_fma(rstd2, x2[2 * q], f2_fma(lnb2, s0, b0));
        x2[2 * q + 1] = f2_fma(rstd2, x2[2 * q + 1], f2_fma(lnb2, s1, b1));
      } else {
        x2[2 * q] = f2_add(x2[2 * q], b0);
        x2[2 * q + 1] = f2_add(x2[2 * q + 1], b1);
      }
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint32_t slot = (WCOLS == 64) ? row_s + ((static_cast<uint32_t>(ch * 2 + q) ^ (lane & 7u)) << 4)
                                          : row_s + ch * (CHUNK * 2) + (q << 4);
      uint64_t y2[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) y2[j] = x2[4 * q + j];
      if (RES) {
        uint32_t ru[4];
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n"
                     : "=r"(ru[0]), "=r"(ru[1]), "=r"(ru[2]), "=r"(ru[3]) : "r"(slot));
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = unpack_half2(ru[j]);
          y2[j] = f2_fma(gate2, y2[j], f2_pack(f.x, f.y));
        }
      }
      if (LNO) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ps2 = f2_add(ps2, y2[j]);
          pq2 = f2_fma(y2[j], y2[j], pq2);
        }
      }
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float lo, hi;
        f2_unpack(y2[j], lo, hi);
        o[j] = pack_half2(lo, hi);
      }
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(slot), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3])
                   : "memory");
    }
  }
  if (LNO) {
    float a, b;
    f2_unpack(ps2, a, b);
    ln_ps += a + b;
    f2_unpack(pq2, a, b);
    ln_pq += a + b;
  }
}

// GEGLU projection: (value (+LN) + b) * gelu(gate (+LN) + b); value chunk c0, its gates BN/2 columns further on
template <int BN, bool LNI>
IDIFF_DEVICE void epi_chunks_geglu(uint32_t trow, uint32_t tab_s, uint32_t row_s, int c_first, int nlive, uint32_t lane,
                                   float ln_rstd, float ln_b) {
  const uint64_t rstd2 = f2_pack(ln_rstd, ln_rstd), lnb2 = f2_pack(ln_b, ln_b);
#pragma unroll 1
  for (int ch = 0; ch < nlive; ++ch) {
    const int c0 = c_first + ch * CHUNK;
    uint32_t v[CHUNK], g[CHUNK];
    tmem_ld_32x32b_x16(trow + c0, v);
    tmem_ld_32x32b_x16(trow + BN / 2 + c0, g);
    tmem_ld_wait();
    float x[CHUNK];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      uint64_t xv[2], gv[2], bv0, bv1, bg0, bg1;
      xv[0] = f2_pack(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]));
      xv[1] = f2_pack(__uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3]));
      gv[0] = f2_pack(__uint_as_float(g[4 * q]), __uint_as_float(g[4 * q + 1]));
      gv[1] = f2_pack(__uint_as_float(g[4 * q + 2]), __uint_as_float(g[4 * q + 3]));
      lds_f2x2(tab_s + (c0 + 4 * q) * 4, bv0, bv1);
      lds_f2x2(tab_s + (BN / 2 + c0 + 4 * q) * 4, bg0, bg1);
      if (LNI) {
        uint64_t sv0, sv1, sg0, sg1;
        lds_f2x2(tab_s + (BN + c0 + 4 * q) * 4, sv0, sv1);
        lds_f2x2(tab_s + (BN + BN / 2 + c0 + 4 * q) * 4, sg0, sg1);
        xv[0] = f2_fma(rstd2, xv[0], f2_fma(lnb2, sv0, bv0));
        xv[1] = f2_fma(rstd2, xv[1], f2_fma(lnb2, sv1, bv1));
        gv[0] = f2_fma(rstd2, gv[0], f2_fma(lnb2, sg0, bg0));
        gv[1] = f2_fma(rstd2, gv[1], f2_fma(lnb2, sg1, bg1));
      } else {
        xv[0] = f2_add(xv[0], bv0);
        xv[1] = f2_add(xv[1], bv1);
        gv[0] = f2_add(gv[0], bg0);
        gv[1] = f2_add(gv[1], bg1);
      }
#pragma unroll
      for (int h = 0; h < 2; ++h) f2_unpack(geglu_f2(xv[h], gv[h]), x[4 * q + 2 * h], x[4 * q + 2 * h + 1]);
    }
#pragma unroll
    for (int q = 0; q < 2; ++q) {  // GEGLU boxes are 64 columns wide: SWIZZLE_128B
      const uint32_t slot = row_s + ((static_cast<uint32_t>(ch * 2 + q) ^ (lane & 7u)) << 4);
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(slot), "r"(pack_half2(x[8 * q], x[8 * q + 1])),
                   "r"(pack_half2(x[8 * q + 2], x[8 * q + 3])), "r"(pack_half2(x[8 * q + 4], x[8 * q + 5])),
                   "r"(pack_half2(x[8 * q + 6], x[8 * q + 7]))
                   : "memory");
    }
  }
}

constexpr int MODE_PLAIN = 0;  // bias / row-add table, optional SiLU, optional gate*x + residual, fp16 out
constexpr int MODE_GEGLU = 1;  // (value + b) * gelu(gate + b), fp16 out with N/2 columns
constexpr int MODE_NCHW = 2;   // fp32 (B, N, HW) output (the final conv -> eps)

template <int BN, int MODE, bool TMA_EPI>
__global__ void __launch_bounds__(128 + EW * 32, 1)
gemm2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
             const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmR,
             const Params p) {
  using C = Cfg<BN, TMA_EPI>;
  constexpr int STAGES = C::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * C::STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;       // [2]
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;  // [2]
  uint64_t* res_bar = bars + 2 * STAGES + 4;     // [EW] residual boxes landed (TMA_EPI)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + EW);
  float* s_epi = reinterpret_cast<float*>(smem + STAGES * C::STAGE_BYTES + C::BAR_BYTES);  // [2][EPI_TAB_PB][BN]
  uint8_t* s_stage = smem + STAGES * C::STAGE_BYTES + C::BAR_BYTES + C::TAB_BYTES;          // [quarter][NCHT][1 KiB]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int cta = blockIdx.x;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], EW * 32);
    }
    for (int w = 0; w < EW; ++w) mbar_init(&res_bar[w], 1);
    if (TMA_EPI) {
      tma_prefetch_desc(&tmO);
      tma_prefetch_desc(&tmR);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<C::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  auto stamp = [&](int slot) {
    if (p.trace) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      p.trace[(long)blockIdx.x * 16 + slot] = t;
    }
  };
  if (threadIdx.x == 0) {
    stamp(0);
    if (p.trace) p.trace[(long)blockIdx.x * 16 + 12] = (unsigned long long)clock64();  // SM clock at entry
  }

  auto tile_origin = [&](int tile, int& n0, int& m0, int& b0, int& h0, int& w0) {
    const int n_tile = tile % p.n_tiles;
    const int m_tile = tile / p.n_tiles;
    n0 = n_tile * BN;
    m0 = m_tile * BM;
    b0 = h0 = w0 = 0;
    if (p.conv) {
      const int tw = m_tile % p.tiles_w;
      const int th = (m_tile / p.tiles_w) % p.tiles_h;
      const int tb = m_tile / (p.tiles_w * p.tiles_h);
      b0 = tb * p.PB;
      h0 = th * p.PH;
      w0 = tw * p.PW;
    }
  };

  // Warpgroup 0 = {TMA, UMMA, 2 idle warps} gives registers to the two epilogue warpgroups
  // (setmaxnreg at the head of each role branch: 56*128 + 224*256 = the CTA's 168*384 allocation).
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 56;\n");
  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      WorkIter it(p, cta);
      Seg sg;
      uint32_t s = 0, ph = 0;  // ring position: running stage / phase (no div / mod on the refill path: every clock
                               // between "stage released" and "TMA issued" is part of the ring's turnaround)
      while (it.next(sg)) {
        int n0, m0, b0, h0, w0;
        tile_origin(sg.tile, n0, m0, b0, h0, w0);
        // conv: k-block kb = (tap, 64-channel slice cb); walked incrementally
        int tap = 0, cb = 0, ky = 0, kx = 0;
        if (p.conv) {
          tap = sg.kb0 / p.kb_per_tap;
          cb = sg.kb0 - tap * p.kb_per_tap;
          ky = tap / 3;
          kx = tap - ky * 3;
        }
        for (int kb = sg.kb0; kb < sg.kb1; ++kb) {
          mbar_wait(&empty_bar[s], ph ^ 1);
          mbar_expect_tx(&full_bar[s], C::STAGE_BYTES);
          if (p.conv) {
            tma_load_4d(sA + s * A_STAGE_BYTES, &tmA, &full_bar[s], cb * BK, w0 + kx - 1, h0 + ky - 1, b0);
            if (++cb == p.kb_per_tap) {
              cb = 0;
              if (++kx == 3) {
                kx = 0;
                ++ky;
              }
            }
          } else {
            tma_load_2d(sA + s * A_STAGE_BYTES, &tmA, &full_bar[s], kb * BK, m0);
          }
          tma_load_2d(sB + s * C::B_STAGE_BYTES, &tmB, &full_bar[s], kb * BK, n0);
          if (++s == STAGES) {
            s = 0;
            ph ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== UMMA issuer =====================
    // All 32 lanes walk the (warp-uniform) schedule and ONE elected lane issues: with a single-lane loop
    // ptxas kept the descriptors in vector registers and paid ~25 instructions (5 R2UR + an ELECT retry loop)
    // per UMMA; this way they live in uniform registers and the four UMMAs of a k-block issue back to back
    // (UTCHMMA x4, UTCBAR).  Descriptors = (low word + constant high word), one add per UMMA; running
    // stage / phase instead of div / mod.
    constexpr uint32_t idesc = make_idesc_f16(BM, BN, UMMA_AB_FMT, 0, 0);
    constexpr uint32_t DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO 1024 B, version 1, SWIZZLE_128B
    const uint32_t a_lo0 = ((smem_u32(sA) & 0x3FFFFu) >> 4) | (1u << 16);  // LBO (unused, swizzled K-major) = 16 B
    const uint32_t b_lo0 = ((smem_u32(sB) & 0x3FFFFu) >> 4) | (1u << 16);
    auto umma_lo = [&](uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t acc) {
      asm volatile(
          "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
          "mov.b64 da, {%1, %3};\n\t"
          "mov.b64 db, {%2, %3};\n\t"
          "setp.ne.b32 p, %5, 0;\n\t"
          "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}\n" ::"r"(d_tmem),
          "r"(a_lo), "r"(b_lo), "r"(DESC_HI), "r"(idesc), "r"(acc)
          : "memory");
    };
    WorkIter it(p, cta);
    Seg sg;
    uint32_t sc = 0, s = 0, ph = 0;
    bool first = true;
    while (it.next(sg)) {
      const int acc = sc & 1;
      mbar_wait(&tmem_empty[acc], ((sc >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * C::ACC_STRIDE;
      for (int kb = sg.kb0; kb < sg.kb1; ++kb) {
        mbar_wait(&full_bar[s], ph);
        if (first && lane == 0) stamp(1);
        first = false;
        tc_fence_after();
        const uint32_t a_lo = a_lo0 + s * (A_STAGE_BYTES >> 4);
        const uint32_t b_lo = b_lo0 + s * (C::B_STAGE_BYTES >> 4);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) umma_lo(d_tmem, a_lo + 2 * k, b_lo + 2 * k, (kb > sg.kb0 || k > 0) ? 1u : 0u);
          umma_commit(&empty_bar[s]);
        }
        __syncwarp();
        if (++s == STAGES) {
          s = 0;
          ph ^= 1;
        }
      }
      if (elect_one()) umma_commit(&tmem_full[acc]);
      __syncwarp();
      if (sc == 0 && lane == 0) stamp(2);
      ++sc;
    }
    __syncwarp();
  }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 224;\n");
    // ===================== epilogue (warps 4..11) =====================
    const int ew = warp - 4;       // 0..7
    const int quarter = warp & 3;  // TMEM lane quarter this warp may access
    const int part = ew >> 2;      // which column part of the tile (EW / 4 parts)
    const int r = quarter * 32 + lane;
    constexpr bool geglu = (MODE == MODE_GEGLU);
    constexpr bool nchw = (MODE == MODE_NCHW);
    const bool do_silu = (p.flags & IDIFF_EPI_SILU) != 0;
    const bool do_gelu = (p.flags & IDIFF_EPI_GELU) != 0;
    const int n_out_total = geglu ? p.N / 2 : p.N;
    constexpr int NCH = C::NCH_MAX;  // accumulator chunks owned by this warp, at most
    constexpr int PARTS = C::PARTS;
    // This warp's chunks.  Plain: the contiguous run [cb, ce) of the tile's NCHT chunks (parts differ by
    // one chunk when PARTS does not divide NCHT, e.g. BN = 160 over four parts: 2, 3, 2, 3).
    // GEGLU: value chunks [cb, ce) of the NCHT / 2 value chunks followed by their gate chunks (BN/2
    // columns further on), so
    // that a warp publishes exactly the columns its owner counterpart consumes.
    constexpr int NOUT_CH = geglu ? C::NCHT / 2 : C::NCHT;  // output chunks of a tile
    const int cb = part * NOUT_CH / PARTS, ce = (part + 1) * NOUT_CH / PARTS;
    const int nv = ce - cb;                 // output chunks of this warp
    const int nch = geglu ? 2 * nv : nv;    // accumulator chunks of this warp
    auto chunk_col = [&](int ch) -> int {
      if (!geglu) return (cb + ch) * CHUNK;
      return (ch < nv) ? (cb + ch) * CHUNK : (BN / 2 + (cb + ch - nv) * CHUNK);
    };

    WorkIter it(p, cta);
    Seg sg;
    uint32_t sc = 0;
    uint32_t res_phase = 0;  // parity of this warp's residual-landed barrier
    while (it.next(sg)) {
      const int acc = sc & 1;
      int n0, m0, b0, h0, w0;
      tile_origin(sg.tile, n0, m0, b0, h0, w0);
      const bool owner = sg.kb0 == 0;
      const bool complete = owner && sg.kb1 == p.KB;
      const bool fixup = owner && !complete;  // this CTA holds the tile's first k-blocks, others the rest
      // followers of an incomplete owner segment: the CTAs covering the tile's remaining k-blocks
      int f0 = 0, f1 = -1;
      if (owner && !complete) {
        const long tile_u0 = (long)(sg.tile - p.T_dp) * p.KB;
        f0 = (int)(((tile_u0 + sg.kb1 + 1) * p.G + p.U_sk - 1) / p.U_sk) - 1;
        f1 = (int)(((tile_u0 + p.KB) * p.G + p.U_sk - 1) / p.U_sk) - 1;
      }
      long out_row = 0;
      bool row_ok = false;
      int batch_idx = 0, pix = 0;
      if (owner) {
        if (p.conv) {
          const int pw = r % p.PW;
          const int ph_ = (r / p.PW) % p.PH;
          const int pb = r / (p.PW * p.PH);
          const int b = b0 + pb, h = h0 + ph_, w = w0 + pw;
          row_ok = (b < p.Bn) && (h < p.H) && (w < p.W);
          pix = h * p.W + w;
          out_row = (long)b * p.H * p.W + pix;
          batch_idx = b;
        } else {
          out_row = (long)m0 + r;
          row_ok = out_row < p.M;
          batch_idx = (int)(out_row / p.rows_per_batch);
          pix = (int)(out_row - (long)batch_idx * p.rows_per_batch);
        }
      }
      // Residual prefetch: the residual rows do not depend on the accumulator, so their loads are
      // issued before the wait and overlap this segment's mainloop (the chunk loop below used to
      // pay one exposed L2/HBM round trip per 16-column chunk: latency-, not bandwidth-bound).
      const int out_col_base = geglu ? (sg.tile % p.n_tiles) * (BN / 2) : n0;
      uint4 resv[TMA_EPI ? 1 : NCH][2];
      const bool has_res = owner && (TMA_EPI || row_ok) && p.residual != nullptr && !geglu;
      // staging boxes of this warp: box ch holds rows [32*quarter, +32) x 16 output columns
      uint8_t* wstage = s_stage + (TMA_EPI ? ew * C::WBOX_BYTES : 0);
      constexpr int WCOLS = geglu ? BN / 4 : BN / 2;        // output columns of this warp (one staging-box row)
      const int wcol0 = out_col_base + cb * CHUNK;          // ... starting here
      const bool wbox_live = wcol0 < n_out_total;           // (a ragged last N tile may leave a warp without columns)
      // tile-local coordinates of this warp's first row, for the output / residual tensor maps
      int tc1 = 0, tc2 = 0, tc3 = 0;
      if (TMA_EPI && owner) {
        if (p.conv) {
          const int r0 = quarter * 32;
          const int pb = r0 / (p.PW * p.PH);
          const int rem = r0 - pb * (p.PW * p.PH);
          tc1 = w0 + rem % p.PW;
          tc2 = h0 + rem / p.PW;
          tc3 = b0 + pb;
        } else {
          tc1 = m0 + quarter * 32;
        }
        // the previous tile's stores must have finished reading the boxes before they are refilled
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
        if (has_res && wbox_live && lane == 0) {
          // one box per warp; rows / columns outside the tensor arrive as zeros and still count as bytes
          mbar_expect_tx(&res_bar[ew], 32 * WCOLS * 2);
          if (p.conv) tma_load_4d(wstage, &tmR, &res_bar[ew], wcol0, tc1, tc2, tc3);
          else tma_load_2d(wstage, &tmR, &res_bar[ew], wcol0, tc1);
        }
      }
      if (!TMA_EPI && has_res) {
        const h16* res_row = p.residual + out_row * p.ldr + out_col_base;
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
          const int c0 = chunk_col(ch);
          if (ch < nv && out_col_base + c0 < n_out_total) {
            resv[ch][0] = *reinterpret_cast<const uint4*>(res_row + c0);
            if (out_col_base + c0 + 8 < n_out_total) resv[ch][1] = *reinterpret_cast<const uint4*>(res_row + c0 + 8);
          }
        }
      }
      // Per-tile epilogue table in shared memory: tab[pb][c] = bias[n0+c] (+ rowadd[b0+pb][n0+c]), so
      // the chunk loop adds its per-column terms with broadcast LDS instead of one exposed L2 round
      // trip per chunk (measured ~1 us per 16-column chunk before; tools/trace_gemm.py).
      const bool tab_rowadd = p.rowadd != nullptr && p.conv && p.PB <= EPI_TAB_PB;
      const bool slow_rowadd = p.rowadd != nullptr && !tab_rowadd;
      float* tab = s_epi + acc * (EPI_TAB_PB * BN);
      if (owner) {
        const int npb = tab_rowadd ? p.PB : 1;
        const int et = threadIdx.x - 128;  // 0..255
        for (int idx = et; idx < npb * BN; idx += EW * 32) {
          const int pb = idx / BN, c = idx - pb * BN;
          const int col = n0 + c;
          float val = 0.f;
          if (col < p.N) {
            if (p.bias) val = __ldg(p.bias + col);
            if (tab_rowadd && b0 + pb < p.Bn) val += h2f(p.rowadd[(long)(b0 + pb) * p.ldra + col]);
          }
          tab[idx] = val;
          if (p.ln_in) tab[BN + idx] = (col < p.N) ? __ldg(p.ln_s + col) : 0.f;  // row 1: sum_k W'[col, k]
        }
        asm volatile("bar.sync 1, %0;\n" ::"n"(EW * 32) : "memory");
      }
      const float* tab_row = tab + ((tab_rowadd && p.conv) ? (r / (p.PW * p.PH)) * BN : 0);
      // LayerNorm fold, consumer side: this row's mean / rstd from the producer GEMM's partial sums, added
      // in slot order (deterministic).  y = rstd * (x . W'^T - mean * colsum(W')) + (W beta + b).
      float ln_nmean = 0.f, ln_rstd = 1.f;
      if (TMA_EPI && p.ln_in != nullptr && owner) {
        float a = 0.f, q = 0.f;
        if (row_ok) {
          for (int sl = 0; sl < p.ln_slots; ++sl) {
            const float2 v = __ldcg(p.ln_in + (long)sl * p.M + out_row);
            a += v.x;
            q += v.y;
          }
        }
        const float inv_k = 1.0f / (float)p.K;
        const float mean = a * inv_k;
        ln_rstd = rsqrtf(fmaxf(q * inv_k - mean * mean, 0.f) + p.ln_eps);
        ln_nmean = -mean * ln_rstd;  // y = rstd * acc + (-mean * rstd) * colsum + bias: two FMAs per element
      }
      float ln_ps = 0.f, ln_pq = 0.f;  // producer side: partial (sum, sumsq) of this warp's output columns
      mbar_wait(&tmem_full[acc], (sc >> 1) & 1);
      if (sc == 0 && threadIdx.x == 128) stamp(3);
      tc_fence_after();
      const uint32_t trow = tmem_base + acc * C::ACC_STRIDE + (static_cast<uint32_t>(quarter * 32) << 16);

      if (!owner) {
        // ---- publish the fp32 partial of this warp's region: ws[cta][chunk][row][CHUNK] ----
        float* wsb = p.ws + (long)cta * (BN / CHUNK) * 128 * CHUNK;
#pragma unroll 1
        for (int ch = 0; ch < nch; ++ch) {
          const int c0 = chunk_col(ch);
          uint32_t v[CHUNK];
          tmem_ld_32x32b_x16(trow + c0, v);
          tmem_ld_wait();
          // layout [chunk][quad q][row][4 floats]: one warp instruction covers 512 contiguous bytes
          // (16 full sectors); row-major 64-byte rows made every lane touch its own half sector and the
          // owner's fold was bound by L2 transactions, not bytes
          float4* dst = reinterpret_cast<float4*>(wsb) + (long)(c0 / CHUNK) * 4 * 128 + r;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            __stcg(dst + q * 128, make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]),
                                        __uint_as_float(v[4 * q + 2]), __uint_as_float(v[4 * q + 3])));
        }
        tc_fence_before();
        mbar_arrive(&tmem_empty[acc]);
        // __syncwarp orders the lanes' partial stores before lane 0's release store (cumulative), so a
        // single release replaces 32 per-thread __threadfence() (MEMBAR.GPU + L1 invalidate each).
        __syncwarp();
        if (lane == 0) st_release_gpu(p.sflags + cta * EW + ew, 1);
      } else {
        // ---- owner: (optional fixup) + fused epilogue ----
        if (fixup) {
          for (int f = f0; f <= f1; ++f) {
            const int* fl = p.sflags + f * EW + ew;
            const long long t0 = clock64();
            while (ld_acquire_gpu(fl) == 0) {
              if (clock64() - t0 > 8000000000LL) {
                if (lane == 0) printf("idiff: stream-K fixup timeout cta=%d waits %d\n", cta, f);
                __trap();
              }
            }
          }
                  // Fold the followers' partial tiles into this CTA's accumulator in TMEM, in CTA order (the sum
          // is bit-reproducible), with up to FB x 4 independent 16-byte loads in flight per thread.  The
          // first version added the partials inside the epilogue's chunk loop, one dependent L2 round
          // trip per follower and chunk: with seven followers (3x3 convolutions at 8x8) the owners'
          // epilogue took 35 us of a 68 us kernel (tools/trace_gemm.py conv1280_8).  After this pass
          // the epilogue variants below see a complete accumulator.
          constexpr int FB = 4;
          const long fstride = (long)(BN / CHUNK) * 128 * CHUNK;
#pragma unroll 1
          for (int ch = 0; ch < nch; ++ch) {
            const int c0 = chunk_col(ch);
            uint32_t av[CHUNK];
            tmem_ld_32x32b_x16(trow + c0, av);
            const float4* base = reinterpret_cast<const float4*>(p.ws) + (long)(c0 / CHUNK) * 4 * 128 + r;
            float a[CHUNK];
            bool first = true;
            for (int fb = f0; fb <= f1; fb += FB) {
              float4 tq[FB][4];
#pragma unroll
              for (int k = 0; k < FB; ++k) {
                if (fb + k <= f1) {
                  const float4* src = base + (long)(fb + k) * (fstride / 4);
#pragma unroll
                  for (int q = 0; q < 4; ++q) tq[k][q] = __ldcg(src + q * 128);
                }
              }
              if (first) {
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) a[j] = __uint_as_float(av[j]);
                first = false;
              }
#pragma unroll
              for (int k = 0; k < FB; ++k) {
                if (fb + k <= f1) {
#pragma unroll
                  for (int q = 0; q < 4; ++q) {
                    a[4 * q] += tq[k][q].x; a[4 * q + 1] += tq[k][q].y;
                    a[4 * q + 2] += tq[k][q].z; a[4 * q + 3] += tq[k][q].w;
                  }
                }
              }
            }
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) av[j] = __float_as_uint(a[j]);
            tmem_st_32x32b_x16(trow + c0, av);
          }
          tmem_st_wait();
        }
        // Lean epilogue: all per-tile pointers are formed once, bias / row-add / residual arrive as
        // 16-byte vector loads per 16-column chunk, and mode switches are warp-uniform branches
        // outside the per-element loops (the first version spent ~40 instructions per element on
        // address arithmetic and predicates and was issue-bound; see profiles/).
        if (sc == 0 && threadIdx.x == 128) stamp(4);
        if (TMA_EPI && has_res && wbox_live) {
          mbar_wait(&res_bar[ew], res_phase);
          res_phase ^= 1;
        }
        h16* o_row = reinterpret_cast<h16*>(p.out) + out_row * p.ldo + out_col_base;
        const h16* radd_row = p.rowadd ? p.rowadd + (long)batch_idx * p.ldra + n0 : nullptr;
        const float gate = p.gate;
        if (TMA_EPI && !nchw) {
          // Compact rolled loop (one 16-column chunk per trip, ~150 instructions, explicit
          // ld/st.shared): the unrolled variant below was instruction-fetch bound for short-K layers
          // (26 % stall_no_inst, generic LD for shared operands; profiles/).
          const int cbase = cb * CHUNK;
          const uint32_t tab_s = smem_u32(tab_row);
          const uint32_t row_s = smem_u32(wstage) + lane * (WCOLS * 2);  // this thread's row of the staging box
          auto lds4 = [](uint32_t a, float (&f)[4]) {
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];\n"
                         : "=f"(f[0]), "=f"(f[1]), "=f"(f[2]), "=f"(f[3]) : "r"(a));
          };
          // live chunks of this warp (a ragged last N tile ends early; warp-uniform)
          int nlive = 0;
          if (wbox_live) {
            nlive = (n_out_total - wcol0 + CHUNK - 1) / CHUNK;
            nlive = nlive < nv ? nlive : nv;
          }
          const bool lni = p.ln_in != nullptr, lno = p.ln_out != nullptr;
          bool fast = false;
          if constexpr (geglu) {
            fast = true;
            if (lni) epi_chunks_geglu<BN, true>(trow, tab_s, row_s, cbase, nlive, lane, ln_rstd, ln_nmean);
            else epi_chunks_geglu<BN, false>(trow, tab_s, row_s, cbase, nlive, lane, ln_rstd, ln_nmean);
          } else if (!slow_rowadd && !do_silu && !do_gelu) {
            fast = true;
            // (row statistics are only ever asked of residual-free proj_in GEMMs or of residual GEMMs; a fold
            // consumer never has a residual: five live combinations)
#define IDIFF_EPI(R, I, O) epi_chunks_plain<BN, WCOLS, R, I, O>(trow, tab_s, row_s, cbase, nlive, lane, gate, ln_rstd, ln_nmean, ln_ps, ln_pq)
            if (has_res) { if (lno) IDIFF_EPI(true, false, true); else IDIFF_EPI(true, false, false); }
            else if (lni) { if (lno) IDIFF_EPI(false, true, true); else IDIFF_EPI(false, true, false); }
            else { if (lno) IDIFF_EPI(false, false, true); else IDIFF_EPI(false, false, false); }
#undef IDIFF_EPI
          }
#pragma unroll 1
          for (int ch = 0; ch < (fast ? 0 : nlive); ++ch) {  // all-flags fallback (SiLU / GELU / per-row add layers)
            const int c0 = cbase + ch * CHUNK;
            const int out_c = out_col_base + c0;
            uint32_t v[CHUNK];
            float x[CHUNK];
            tmem_ld_32x32b_x16(trow + c0, v);
            if (geglu) {
              uint32_t g[CHUNK];
              float gx[CHUNK];
              tmem_ld_32x32b_x16(trow + BN / 2 + c0, g);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < CHUNK; ++j) {
                x[j] = __uint_as_float(v[j]);
                gx[j] = __uint_as_float(g[j]);
              }
              if (p.ln_in != nullptr) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float sv[4], sg[4], bv[4], bg[4];
                  lds4(tab_s + (BN + c0 + 4 * q) * 4, sv);
                  lds4(tab_s + (BN + BN / 2 + c0 + 4 * q) * 4, sg);
                  lds4(tab_s + (c0 + 4 * q) * 4, bv);
                  lds4(tab_s + (BN / 2 + c0 + 4 * q) * 4, bg);
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float xv = fmaf(ln_rstd, x[4 * q + j], fmaf(ln_nmean, sv[j], bv[j]));
                    const float gv = fmaf(ln_rstd, gx[4 * q + j], fmaf(ln_nmean, sg[j], bg[j]));
                    x[4 * q + j] = xv * gelu_erf_f(gv);
                  }
                }
              } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float bv[4], bg[4];
                  lds4(tab_s + (c0 + 4 * q) * 4, bv);
                  lds4(tab_s + (BN / 2 + c0 + 4 * q) * 4, bg);
#pragma unroll
                  for (int j = 0; j < 4; ++j) x[4 * q + j] = (x[4 * q + j] + bv[j]) * gelu_erf_f(gx[4 * q + j] + bg[j]);
                }
              }
            } else {
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < CHUNK; ++j) x[j] = __uint_as_float(v[j]);
              if (p.ln_in != nullptr) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float sv[4], bv[4];
                  lds4(tab_s + (BN + c0 + 4 * q) * 4, sv);
                  lds4(tab_s + (c0 + 4 * q) * 4, bv);
#pragma unroll
                  for (int j = 0; j < 4; ++j) x[4 * q + j] = fmaf(ln_rstd, x[4 * q + j], fmaf(ln_nmean, sv[j], bv[j]));
                }
              } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float bv[4];
                  lds4(tab_s + (c0 + 4 * q) * 4, bv);
#pragma unroll
                  for (int j = 0; j < 4; ++j) x[4 * q + j] += bv[j];
                }
              }
              if (slow_rowadd && row_ok) {
#pragma unroll
                for (int j = 0; j < CHUNK; ++j)
                  if (out_c + j < n_out_total) x[j] += h2f(radd_row[c0 + j]);
              }
              if (do_silu) {
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) x[j] = silu_f(x[j]);
              } else if (do_gelu) {
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) x[j] = gelu_erf_f(x[j]);
              }
            }
            // The residual (if any) was landed in the box by TMA; the result replaces it in place.  (Rows are
            // WCOLS * 2 bytes apart: 16-byte accesses of eight consecutive lanes collide two ways at most.)
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              // 64-column boxes (128-byte rows) are SWIZZLE_128B: 16-byte chunk i of row r sits at i ^ (r & 7);
              // wider rows are unswizzled (160 / 192-byte pitch: two / four-way conflicts at most)
              const uint32_t slot = (WCOLS == 64) ? row_s + ((static_cast<uint32_t>(ch * 2 + q) ^ (lane & 7u)) << 4)
                                                  : row_s + ch * (CHUNK * 2) + (q << 4);
              float y[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) y[j] = x[8 * q + j];
              if (has_res) {
                uint32_t ru[4];
                asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n"
                             : "=r"(ru[0]), "=r"(ru[1]), "=r"(ru[2]), "=r"(ru[3]) : "r"(slot));
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const float2 f = unpack_half2(ru[j]);
                  y[2 * j] = fmaf(gate, y[2 * j], f.x);
                  y[2 * j + 1] = fmaf(gate, y[2 * j + 1], f.y);
                }
              }
              if (p.ln_out != nullptr && out_c + 8 * q < n_out_total) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  ln_ps += y[j];
                  ln_pq = fmaf(y[j], y[j], ln_pq);
                }
              }
              asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(slot), "r"(pack_half2(y[0], y[1])),
                           "r"(pack_half2(y[2], y[3])), "r"(pack_half2(y[4], y[5])), "r"(pack_half2(y[6], y[7]))
                           : "memory");
            }
          }
          // one proxy fence and ONE bulk-tensor store per warp and tile (per 16-column chunk they were a
          // ~700-clock serial tail of every trip: tools/trace_gemm.py); columns / rows outside the tensor
          // are clipped by the store
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0 && wbox_live) {
            if (p.conv) tma_store_4d(&tmO, wstage, wcol0, tc1, tc2, tc3);
            else tma_store_2d(&tmO, wstage, wcol0, tc1);
          }
          if (sc == 0 && threadIdx.x == 128) stamp(11);
        } else {
        // Chunks are processed in groups of up to GROUP: all accumulator loads of a group are issued
        // before one wait, all results are staged before one proxy fence / warp sync, and the
        // group's TMA stores go out together.  (Chunk-at-a-time was a ~1200-cycle serial dependency
        // chain per 16 columns with only two warps per scheduler to hide it: tools/trace_gemm.py.)
        constexpr int GROUP = 4;
        constexpr int NV = (NOUT_CH + PARTS - 1) / PARTS;  // output chunks of this warp, at most
#pragma unroll
        for (int g0 = 0; g0 < NV; g0 += GROUP) {
          uint32_t xv[GROUP][CHUNK];
          uint32_t gv[geglu ? GROUP : 1][CHUNK];
          bool live[GROUP];
          const bool dbg = (sc == 0 && threadIdx.x == 128 && g0 == 0);  // group-level trace (slots 8..11)
          if (dbg) stamp(8);
          // ---- A: accumulator loads -----------------------------------------------------------
#pragma unroll
          for (int i = 0; i < GROUP; ++i) {
            const int ch = g0 + i;
            live[i] = (ch < nv) && (out_col_base + chunk_col(ch < nv ? ch : 0) < n_out_total);
            if (live[i]) {
              const int c0 = chunk_col(ch);
              tmem_ld_32x32b_x16(trow + c0, xv[i]);
              if (geglu) tmem_ld_32x32b_x16(trow + BN / 2 + c0, gv[geglu ? i : 0]);
            }
          }
          tmem_ld_wait();
          if (dbg) stamp(14);
          // ---- B: stream-K partials, per-column table terms, activation ---------------------------
#pragma unroll
          for (int i = 0; i < GROUP; ++i) {
            if (!live[i]) continue;
            const int c0 = chunk_col(g0 + i);
            float x[CHUNK];
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) x[j] = __uint_as_float(xv[i][j]);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 bv = *(reinterpret_cast<const float4*>(tab_row + c0) + q);
              x[4 * q] += bv.x; x[4 * q + 1] += bv.y; x[4 * q + 2] += bv.z; x[4 * q + 3] += bv.w;
            }
            if (geglu) {
              float gx[CHUNK];
#pragma unroll
              for (int j = 0; j < CHUNK; ++j) gx[j] = __uint_as_float(gv[geglu ? i : 0][j]);
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const float4 bg = *(reinterpret_cast<const float4*>(tab_row + BN / 2 + c0) + q);
                gx[4 * q] += bg.x; gx[4 * q + 1] += bg.y; gx[4 * q + 2] += bg.z; gx[4 * q + 3] += bg.w;
              }
#pragma unroll
              for (int j = 0; j < CHUNK; ++j) x[j] *= gelu_erf_f(gx[j]);
            } else {
              if (slow_rowadd && row_ok) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                  if (q == 0 || out_col_base + c0 + 8 < n_out_total) {
                    const uint4 rv = __ldg(reinterpret_cast<const uint4*>(radd_row + c0) + q);
                    const uint32_t ru[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                      const float2 f = unpack_half2(ru[j]);
                      x[8 * q + 2 * j] += f.x;
                      x[8 * q + 2 * j + 1] += f.y;
                    }
                  }
                }
              }
              if (do_silu) {
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) x[j] = silu_f(x[j]);
              } else if (do_gelu) {
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) x[j] = gelu_erf_f(x[j]);
              }
            }
#pragma unroll
            for (int j = 0; j < CHUNK; ++j) xv[i][j] = __float_as_uint(x[j]);
          }
          if (dbg) stamp(9);
          // ---- C: residual + store --------------------------------------------------------------
#pragma unroll
          for (int i = 0; i < GROUP; ++i) {
            if (!live[i]) continue;
            const int ch = g0 + i;
            const int c0 = chunk_col(ch);
            const int out_c = out_col_base + c0;
            const bool hi_ok = out_c + 8 < n_out_total;  // second 8-column group inside N (N % 8 == 0)
            if (nchw) {
              if (row_ok) {
                float* o = reinterpret_cast<float*>(p.out);
                const long hw = p.conv ? (long)p.H * p.W : (long)p.rows_per_batch;
#pragma unroll
                for (int j = 0; j < CHUNK; ++j) {
                  const int col = out_c + j;
                  if (col < n_out_total) o[((long)batch_idx * n_out_total + col) * hw + pix] = __uint_as_float(xv[i][j]);
                }
              }
            } else if (TMA_EPI) {
              // box `ch`: row `lane` is 32 B; SWIZZLE_32B puts 16-byte chunk q at (q ^ ((lane >> 2) & 1)).
              // The residual (if any) was landed here by TMA; the result replaces it in place.  Rows /
              // columns outside the tensor are clipped by the TMA store.
              uint8_t* box = wstage + ch * C::BOX_BYTES + lane * 32;
              const int swz = (lane >> 2) & 1;
#pragma unroll
              for (int q = 0; q < 2; ++q) {
                uint4* slot = reinterpret_cast<uint4*>(box + ((q ^ swz) << 4));
                float y[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) y[j] = __uint_as_float(xv[i][8 * q + j]);
                if (has_res) {
                  const uint4 rv = *slot;
                  const uint32_t ru[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 f = unpack_half2(ru[j]);
                    y[2 * j] = fmaf(gate, y[2 * j], f.x);
                    y[2 * j + 1] = fmaf(gate, y[2 * j + 1], f.y);
                  }
                }
                *slot = make_uint4(pack_half2(y[0], y[1]), pack_half2(y[2], y[3]), pack_half2(y[4], y[5]),
                                   pack_half2(y[6], y[7]));
              }
            } else if (row_ok) {
#pragma unroll
              for (int q = 0; q < 2; ++q) {
                if (q == 0 || hi_ok) {
                  float y[8];
#pragma unroll
                  for (int j = 0; j < 8; ++j) y[j] = __uint_as_float(xv[i][8 * q + j]);
                  if (has_res) {
                    const uint4 rv = resv[TMA_EPI ? 0 : ch][q];
                    const uint32_t ru[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                      const float2 f = unpack_half2(ru[j]);
                      y[2 * j] = fmaf(gate, y[2 * j], f.x);
                      y[2 * j + 1] = fmaf(gate, y[2 * j + 1], f.y);
                    }
                  }
                  if (p.ln_out != nullptr) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                      ln_ps += y[j];
                      ln_pq = fmaf(y[j], y[j], ln_pq);
                    }
                  }
                  *(reinterpret_cast<uint4*>(o_row + c0) + q) =
                      make_uint4(pack_half2(y[0], y[1]), pack_half2(y[2], y[3]), pack_half2(y[4], y[5]),
                                 pack_half2(y[6], y[7]));
                }
              }
            }
          }
          if (dbg) stamp(10);
          if (TMA_EPI && !nchw) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
#pragma unroll
              for (int i = 0; i < GROUP; ++i) {
                if (!live[i]) continue;
                const int ch = g0 + i;
                const int out_c = out_col_base + chunk_col(ch);
                if (p.conv) tma_store_4d(&tmO, wstage + ch * C::BOX_BYTES, out_c, tc1, tc2, tc3);
                else tma_store_2d(&tmO, wstage + ch * C::BOX_BYTES, out_c, tc1);
              }
            }
          }
          if (dbg) stamp(11);
        }
        }  // direct / grouped epilogue
        if (TMA_EPI && lane == 0) tma_store_commit();
        // LayerNorm fold, producer side: this warp's partial row statistics, slot = (n tile, column part);
        // consecutive lanes own consecutive rows -> one coalesced 256-byte store per warp
        if (p.ln_out != nullptr && row_ok)
          __stcg(p.ln_out + (long)((sg.tile % p.n_tiles) * PARTS + part) * p.M + out_row, make_float2(ln_ps, ln_pq));
        if (sc == 0 && threadIdx.x == 128) stamp(5);
        tc_fence_before();
        mbar_arrive(&tmem_empty[acc]);
        if (fixup) {
          // consume the followers' flags so the next launch (or graph replay) starts clean
          __syncwarp();
          if (lane == 0)
            for (int f = f0; f <= f1; ++f) st_release_gpu(p.sflags + f * EW + ew, 0);
        }
      }
      ++sc;
    }
  }

  if (TMA_EPI && warp >= 4 && lane == 0) tma_store_wait_read();  // boxes must outlive their stores
  if (threadIdx.x == 128) stamp(6);
  __syncthreads();
  if (threadIdx.x == 0) {
    stamp(7);
    if (p.trace) p.trace[(long)blockIdx.x * 16 + 13] = (unsigned long long)clock64();  // SM clock at exit
  }
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static void* g_ws = nullptr;
static unsigned long long* g_trace = nullptr;
static long g_ws_bytes = 0;
static int g_num_sms = 0;
constexpr long kFlagBytes = 64 * 1024;
// k-blocks up to which the TMA epilogue is used; the LayerNorm fold (ln_stats_in) exists only in that epilogue
constexpr int kTmaEpiMaxKB = 40;

static void choose_patch(int H, int W, int* PW, int* PH, int* PB) {
  int pw = 1;
  while (pw * 2 <= 128 && (W % (pw * 2)) == 0) pw *= 2;
  int ph = 1;
  while (pw * ph * 2 <= 128 && ph < H) ph *= 2;
  *PW = pw;
  *PH = ph;
  *PB = 128 / (pw * ph);
}

template <int BN, int MODE, bool TMA_EPI>
static int launch(const idiff_gemm_args* a, cudaStream_t stream, bool want_sk) {
  using C = Cfg<BN, TMA_EPI>;
  Params p;
  memset(&p, 0, sizeof(p));
  p.M = a->M;
  p.N = a->N;
  p.K = a->K;
  p.KB = (a->K + BK - 1) / BK;
  p.bias = a->bias;
  p.rowadd = reinterpret_cast<const h16*>(a->rowadd);
  p.residual = reinterpret_cast<const h16*>(a->residual);
  p.out = a->out;
  p.ldo = a->ldo;
  p.ldr = a->ldr;
  p.ldra = a->ldra > 0 ? a->ldra : a->N;
  p.rows_per_batch = a->rows_per_batch > 0 ? a->rows_per_batch : a->M;
  p.flags = a->flags;
  p.gate = a->gate;
  p.trace = g_trace;
  p.ln_out = reinterpret_cast<float2*>(a->ln_stats_out);
  p.ln_in = reinterpret_cast<const float2*>(a->ln_stats_in);
  p.ln_s = a->ln_colsum;
  p.ln_slots = a->ln_slots_in;
  p.ln_eps = a->ln_eps;

  CUtensorMap tmA, tmB;
  int m_tiles;
  if (a->conv_h > 0) {
    const int H = a->conv_h, W = a->conv_w, B = a->conv_b, Cn = a->conv_cin;
    IDIFF_REQUIRE(Cn % BK == 0, "conv3x3: Cin=%d must be a multiple of %d", Cn, BK);
    IDIFF_REQUIRE(a->K == 9 * Cn, "conv3x3: K=%d must equal 9*Cin=%d", a->K, 9 * Cn);
    IDIFF_REQUIRE(a->M == B * H * W, "conv3x3: M=%d must equal B*H*W=%d", a->M, B * H * W);
    p.conv = 1;
    p.H = H;
    p.W = W;
    p.Bn = B;
    choose_patch(H, W, &p.PW, &p.PH, &p.PB);
    p.tiles_w = W / p.PW;
    p.tiles_h = (H + p.PH - 1) / p.PH;
    const int tiles_b = (B + p.PB - 1) / p.PB;
    p.kb_per_tap = Cn / BK;
    p.rows_per_batch = H * W;
    m_tiles = p.tiles_w * p.tiles_h * tiles_b;
    const uint64_t dims[4] = {(uint64_t)Cn, (uint64_t)W, (uint64_t)H, (uint64_t)B};
    const uint64_t strides[3] = {(uint64_t)Cn * 2, (uint64_t)W * Cn * 2, (uint64_t)H * W * Cn * 2};
    const uint32_t box[4] = {(uint32_t)BK, (uint32_t)p.PW, (uint32_t)p.PH, (uint32_t)p.PB};
    if (encode_tmap_f16(&tmA, a->a, 4, dims, strides, box)) return -1;
  } else {
    m_tiles = (a->M + BM - 1) / BM;
    const uint64_t dims[2] = {(uint64_t)a->K, (uint64_t)a->M};
    const uint64_t strides[1] = {(uint64_t)a->lda * 2};
    const uint32_t box[2] = {(uint32_t)BK, (uint32_t)BM};
    if (encode_tmap_f16(&tmA, a->a, 2, dims, strides, box)) return -1;
  }
  {
    const uint64_t dims[2] = {(uint64_t)a->K, (uint64_t)a->N};
    const uint64_t strides[1] = {(uint64_t)a->ldw * 2};
    const uint32_t box[2] = {(uint32_t)BK, (uint32_t)BN};
    if (encode_tmap_f16(&tmB, a->w, 2, dims, strides, box)) return -1;
  }
  p.n_tiles = (a->N + BN - 1) / BN;
  p.T = p.n_tiles * m_tiles;

  if (g_num_sms == 0) {
    int dev = 0;
    IDIFF_CHECK_CUDA(cudaGetDevice(&dev));
    IDIFF_CHECK_CUDA(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
  }
  // Stream-K needs the fixup workspace (flags in its first 64 KiB, partial tiles after); short-K
  // problems (fixup cost ~ mainloop) and exact multiples of the SM count stay data-parallel.
  const long ws_need = kFlagBytes + (long)g_num_sms * 128 * BN * sizeof(float);
  // per-call scratch (idiff_gemm_args.workspace: one per stream, so concurrent streams never share flags)
  // takes precedence over the process-wide default of idiff_set_gemm_workspace
  void* ws_ptr = a->workspace ? a->workspace : g_ws;
  const long ws_bytes = a->workspace ? a->workspace_bytes : g_ws_bytes;
  const bool use_sk = want_sk && ws_ptr && ws_bytes >= ws_need && p.KB >= 8 && (p.T % g_num_sms) != 0 &&
                      (long)p.T * p.KB >= g_num_sms;
  if (use_sk) {
    p.G = g_num_sms;
    const int waves = p.T / p.G;
    p.T_dp = (waves >= 2) ? (waves - 1) * p.G : 0;
    p.U_sk = (long)(p.T - p.T_dp) * p.KB;
    p.sflags = reinterpret_cast<int*>(ws_ptr);
    p.ws = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(ws_ptr) + kFlagBytes);
  } else {
    p.G = g_num_sms < p.T ? g_num_sms : p.T;
    p.T_dp = p.T;
    p.U_sk = 0;
  }

  // output / residual views for the TMA epilogue: one [32 rows x BN/2 (GEGLU: BN/4) columns] box per warp,
  // row-major in shared memory (no swizzle)
  CUtensorMap tmO = tmA, tmR = tmA;
  if (TMA_EPI) {
    const int n_out = (MODE == MODE_GEGLU) ? a->N / 2 : a->N;
    const uint32_t wcols = (MODE == MODE_GEGLU) ? BN / 4 : BN / 2;
    auto make = [&](CUtensorMap* m, const void* base, int ld) -> int {
      if (p.conv) {
        const int pws = p.PW < 32 ? p.PW : 32;
        const uint64_t dims[4] = {(uint64_t)n_out, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.Bn};
        const uint64_t strides[3] = {(uint64_t)ld * 2, (uint64_t)p.W * ld * 2, (uint64_t)p.H * p.W * ld * 2};
        const uint32_t box[4] = {wcols, (uint32_t)pws, (uint32_t)(32 / pws), 1u};
        return encode_tmap_f16_sw(m, base, 4, dims, strides, box, wcols == 64 ? 128 : 0);
      }
      const uint64_t dims[2] = {(uint64_t)n_out, (uint64_t)a->M};
      const uint64_t strides[1] = {(uint64_t)ld * 2};
      const uint32_t box[2] = {wcols, 32u};
      return encode_tmap_f16_sw(m, base, 2, dims, strides, box, wcols == 64 ? 128 : 0);
    };
    if (make(&tmO, a->out, a->ldo)) return -1;
    if (a->residual && make(&tmR, a->residual, a->ldr)) return -1;
  }

  static bool attr_set = false;
  if (!attr_set) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(gemm2_kernel<BN, MODE, TMA_EPI>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  gemm2_kernel<BN, MODE, TMA_EPI><<<p.G, C::THREADS, C::SMEM_BYTES, stream>>>(tmA, tmB, tmO, tmR, p);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// Tile width and schedule.  A small cost model in SM clocks, calibrated on tools/bench_kernels.py and
// tools/trace_gemm.py at the UNet's shapes:
//   * one 64-deep k-block of a 128 x BN tile costs max(UMMA time 2*BN, operand bytes / ~50 B/clk/SM);
//   * data-parallel: ceil(T / SMs) rounds of (KB k-blocks + ~600 clk of pipeline fill) and one exposed
//     epilogue (~1000 clk per 32 columns);
//   * stream-K: the k-blocks of the last partial round are spread evenly, but the fixup is expensive --
//     ~30k clk of flag / partial-tile round trips plus the owner pulling every follower's fp32 tile
//     through one SM's L2 port (~40 B/clk).  It only wins for long-K tiles (3x3 convolutions at the
//     16x16 / 8x8 levels); for K <= 2560 it was 10-20 us slower than two plain rounds.
struct Plan {
  int bn;
  bool sk;
};
static int count_m_tiles(const idiff_gemm_args* a) {
  if (a->conv_h > 0) {
    int pw, ph, pb;
    choose_patch(a->conv_h, a->conv_w, &pw, &ph, &pb);
    return (a->conv_w / pw) * ((a->conv_h + ph - 1) / ph) * ((a->conv_b + pb - 1) / pb);
  }
  return (a->M + BM - 1) / BM;
}
static Plan plan_gemm(const idiff_gemm_args* a, int fixed_bn) {  // fixed_bn: 0 = choose the tile width
  const char* force = getenv("IDIFF_GEMM_PLAN");  // "bn,sk" overrides the model (tests, tuning); bn 0 = keep
  if (g_num_sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  const int sms = g_num_sms;
  const int KB = (a->K + BK - 1) / BK;
  const int m_tiles = count_m_tiles(a);
  const int cands[4] = {256, 192, 160, 128};
  long min_pad = -1;
  for (int i = 0; i < 4; ++i) {
    const long pad = (long)((a->N + cands[i] - 1) / cands[i]) * cands[i];
    if (min_pad < 0 || pad < min_pad) min_pad = pad;
  }
  Plan best = {fixed_bn ? fixed_bn : 128, false};
  double best_cost = -1;
  for (int i = 0; i < 4; ++i) {
    const int bn = cands[i];
    if (fixed_bn && bn != fixed_bn) continue;
    if (!fixed_bn && a->N <= 128 && bn != 128) continue;
    const long pad = (long)((a->N + bn - 1) / bn) * bn;
    if (!fixed_bn && pad > min_pad + min_pad / 14) continue;  // more than ~7 % wasted columns
    const long T = (long)((a->N + bn - 1) / bn) * m_tiles;
    // constants refitted in round 2 against tools/plan_sweep.py (every linear / conv shape of the forward x
    // {128,160,192,256} x {rounds, stream-K}: the model's picks cost 9.40 ms per forward against 9.28 for the
    // per-shape optimum and 9.52 with the round-1 constants): operand ring ~80 B/clk/SM, epilogue ~47 clk per
    // output column, stream-K fixed cost ~20k clk
    const double t_kb = fmax(2.0 * bn, (16384.0 + 128.0 * bn) / 80.0);
    const double t_epi = 1500.0 * bn / 32.0;
    const double t_tile = KB * t_kb + 600.0;
    const long rounds = (T + sms - 1) / sms;
    const double cost_dp = rounds * t_tile + t_epi;
    if (best_cost < 0 || cost_dp < best_cost) {
      best_cost = cost_dp;
      best = {bn, false};
    }
    if (KB >= 8 && (T % sms) != 0 && T * KB >= sms) {
      const long full = T / sms;
      const long t_dp = full >= 2 ? (full - 1) * sms : 0;
      const long t_sk = T - t_dp;
      const double followers = t_sk < sms ? (double)(sms - t_sk) / t_sk : 1.0;
      const double cost_sk = (full >= 2 ? (full - 1) : 0) * t_tile + (double)t_sk * KB / sms * t_kb + t_epi + 20000.0 +
                             followers * 128.0 * bn * 4.0 / 40.0;
      if (cost_sk < best_cost) {
        best_cost = cost_sk;
        best = {bn, true};
      }
    }
  }
  if (force) {
    int fbn = 0, fsk = 0;
    if (sscanf(force, "%d,%d", &fbn, &fsk) == 2) {
      if (!fixed_bn && (fbn == 256 || fbn == 192 || fbn == 160 || fbn == 128)) best.bn = fbn;
      best.sk = fsk != 0;
    }
  }
  return best;
}

struct Resolved {
  int bn, mode;
  bool tma_epi, sk;
};

static Resolved resolve(const idiff_gemm_args* a) {
  Resolved r;
  // GEGLU: one 256-column accumulator tile = 128 value columns + their 128 gates (packing.py)
  if (a->flags & IDIFF_EPI_GEGLU) {
    const bool sk = plan_gemm(a, 256).sk;
    r = {256, MODE_GEGLU, true, sk};
    return r;
  }
  if (a->flags & IDIFF_OUT_F32_NCHW) {
    r = {128, MODE_NCHW, false, plan_gemm(a, 128).sk};
    return r;
  }
  // short K: the epilogue dominates -> TMA-staged epilogue (shallower operand ring);
  // long K (3x3 convolutions): deep operand ring, direct epilogue hidden behind the next mainloop
  const bool tma_epi = ((a->K + BK - 1) / BK) <= kTmaEpiMaxKB;
  const Plan pl = plan_gemm(a, false);
  r = {pl.bn, MODE_PLAIN, tma_epi, pl.sk};
  return r;
}

template <int BN>
static int launch_plain(const Resolved& r, const idiff_gemm_args* a, cudaStream_t stream) {
  return r.tma_epi ? launch<BN, MODE_PLAIN, true>(a, stream, r.sk) : launch<BN, MODE_PLAIN, false>(a, stream, r.sk);
}

// One instantiation per (tile width, epilogue mode, TMA epilogue): each kernel carries only its own mode's code (an
// all-modes kernel was ~140 KB of SASS and stalled on instruction fetch: 26 % stall_no_inst, profiles/).
int gemm_v2(const idiff_gemm_args* a, cudaStream_t stream) {
  const Resolved r = resolve(a);
  if (r.mode == MODE_GEGLU) return launch<256, MODE_GEGLU, true>(a, stream, r.sk);
  if (r.mode == MODE_NCHW) return launch<128, MODE_NCHW, false>(a, stream, r.sk);
  switch (r.bn) {
    case 256: return launch_plain<256>(r, a, stream);
    case 192: return launch_plain<192>(r, a, stream);
    case 160: return launch_plain<160>(r, a, stream);
    default: return launch_plain<128>(r, a, stream);
  }
}

// slots of the LayerNorm partial statistics a producer GEMM with these arguments writes per row
int ln_slots_of(const idiff_gemm_args* a) {
  const Resolved r = resolve(a);
  return ((a->N + r.bn - 1) / r.bn) * (EW / 4);  // (n tile, column part): Cfg::PARTS
}

}  // namespace v2
}  // namespace idiff

extern "C" int idiff_gemm(const idiff_gemm_args* a, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(a && a->a && a->w && a->out, "idiff_gemm: null pointer argument");
  IDIFF_REQUIRE(a->M > 0 && a->N > 0 && a->K > 0, "idiff_gemm: bad shape M=%d N=%d K=%d", a->M, a->N, a->K);
  const bool geglu = (a->flags & IDIFF_EPI_GEGLU) != 0;
  const bool nchw = (a->flags & IDIFF_OUT_F32_NCHW) != 0;
  if (geglu) {
    IDIFF_REQUIRE(a->N % 256 == 0, "idiff_gemm: GEGLU needs N %% 256 == 0 (N=%d)", a->N);
    IDIFF_REQUIRE(!a->residual && !a->rowadd && !nchw, "idiff_gemm: GEGLU excludes residual/rowadd/NCHW");
  }
  if (!nchw) {
    IDIFF_REQUIRE(a->N % 8 == 0, "idiff_gemm: N=%d must be a multiple of 8 for fp16 output", a->N);
    IDIFF_REQUIRE(a->ldo % 8 == 0, "idiff_gemm: ldo=%d must be a multiple of 8", a->ldo);
    IDIFF_REQUIRE((reinterpret_cast<uintptr_t>(a->out) & 15) == 0, "idiff_gemm: out not 16B aligned");
    if (a->residual) {
      IDIFF_REQUIRE(a->ldr % 8 == 0 && (reinterpret_cast<uintptr_t>(a->residual) & 15) == 0,
                    "idiff_gemm: residual must be 16B aligned with ldr %% 8 == 0");
    }
  } else {
    IDIFF_REQUIRE(!a->residual, "idiff_gemm: NCHW fp32 output excludes residual");
  }
  if (a->workspace) {
    IDIFF_REQUIRE((reinterpret_cast<uintptr_t>(a->workspace) & 255) == 0, "idiff_gemm: workspace must be 256B aligned");
  }
  if (a->ln_stats_in) {
    IDIFF_REQUIRE(a->ln_colsum && a->ln_slots_in > 0 && a->ln_slots_in <= 64, "idiff_gemm: LayerNorm fold needs ln_colsum and 1..64 slots");
    IDIFF_REQUIRE(a->conv_h == 0 && !nchw && !a->rowadd, "idiff_gemm: LayerNorm fold applies to plain / GEGLU linear layers");
    IDIFF_REQUIRE((a->K + v2::BK - 1) / v2::BK <= v2::kTmaEpiMaxKB, "idiff_gemm: LayerNorm fold needs K <= %d (K=%d)",
                  v2::BK * v2::kTmaEpiMaxKB, a->K);
    IDIFF_REQUIRE((reinterpret_cast<uintptr_t>(a->ln_stats_in) & 7) == 0, "idiff_gemm: ln_stats_in must be 8B aligned");
  }
  if (a->ln_stats_out) {
    IDIFF_REQUIRE(a->conv_h == 0 && !nchw && !geglu, "idiff_gemm: row statistics are produced by plain linear layers");
    IDIFF_REQUIRE((reinterpret_cast<uintptr_t>(a->ln_stats_out) & 7) == 0, "idiff_gemm: ln_stats_out must be 8B aligned");
  }
  return v2::gemm_v2(a, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int idiff_gemm_ln_slots(const idiff_gemm_args* a) {
  using namespace idiff;
  IDIFF_REQUIRE(a && a->M > 0 && a->N > 0 && a->K > 0, "idiff_gemm_ln_slots: bad arguments");
  return v2::ln_slots_of(a);
}

extern "C" int idiff_set_gemm_workspace(void* ptr, long bytes) {
  using namespace idiff;
  if (ptr) {
    IDIFF_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 255) == 0, "idiff_set_gemm_workspace: pointer must be 256B aligned");
    // flags live inside the workspace and must start at zero
    IDIFF_CHECK_CUDA(cudaMemset(ptr, 0, (size_t)bytes));
  }
  v2::g_ws = ptr;
  v2::g_ws_bytes = ptr ? bytes : 0;
  return 0;
}

// Debug / profiling hook: when set, every GEMM CTA writes %globaltimer stamps (kernel entry, first
// operand tile landed, first segment issued, first accumulator ready, fixup done, first epilogue
// done, role loops done, exit, then per-chunk epilogue phases) to trace[cta*16 ..].  NULL disables.
extern "C" int idiff_set_gemm_trace(void* ptr) {
  idiff::v2::g_trace = reinterpret_cast<unsigned long long*>(ptr);
  return 0;
}

extern "C" long idiff_gemm_workspace_bytes(void) {
  // 148 SMs x 128 x 256 fp32 partial tiles + flags, rounded up
  return 256L * 128 * 256 * 4 + (1 << 20);
}
