// Flash-style attention on tcgen05 for sm_100a: O = softmax(Q K^T * scale) V per (batch, head).
//
// One CTA owns a 128-query tile of one (batch, head).  S = Q K^T and O live in TMEM; the
// probabilities P go back through shared memory as the (K-major, 128B-swizzled) A operand of
// the P.V UMMA; V is consumed as an MN-major B operand straight from its token-major tile, so
// no transposed copy of V is ever made.
//   warp 0      TMA producer (Q once, then K/V tiles through a ring)
//   warp 1      TMEM allocator + UMMA issuer
//   warps 2..5  online softmax: one thread per query row (tcgen05.ld 32x32b), exp2 on the raw
//               scores with the running row maximum, P -> smem, O rescale in TMEM when the
//               maximum moved, final O / l -> fp16
// Keys/values are read from up to two segments (visual tokens, then the 184 UniFusion object
// tokens of GatedSelfAttentionDense) -- the concatenation of attention.py:306 never exists.
//
// Replaces F.scaled_dot_product_attention at attention.py:134-144, 257-267 (+ the head
// split/merge permutes at :130-132,144,183-185,267).
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {

namespace att2 {
int attention_v2_d40(const idiff_attn_args* a, cudaStream_t stream);  // attention2.cu
}

constexpr int ATT_THREADS = 192;
constexpr int BQ = 128;

struct AttnKParams {
  int heads, nq, n0, n1, kv1_broadcast;
  float scale_log2e;
  h16* out;
  int out_ld;
};

// 64 keys per tile keep the footprint of head_dim 80 at 112 KiB of shared memory and 256 TMEM columns, so two
// CTAs are resident per SM and cover each other's softmax / hand-off latency (what took attention2 from 566 to
// 414 us).  128-key tiles, one CTA per SM, measured slower: profiles/README.md round 2, section 7.9.
template <int D>
struct AttnCfg {
  static constexpr int ND = (D + 63) / 64;           // 64-wide d chunks (one TMA box each)
  static constexpr int KSTEPS = (D + 15) / 16;       // UMMA k-steps of QK^T (zero padded)
  static constexpr int BKV = 64;                     // keys per tile
  static constexpr int DV = ND * 64;                 // UMMA N of the PV product
  static constexpr int STAGES = (D <= 64) ? 3 : 2;
  static constexpr int Q_BYTES = ND * BQ * 128;
  static constexpr int KV_TILE_BYTES = ND * BKV * 128;  // one of K or V
  static constexpr int P_BYTES = (BKV / 64) * BQ * 128;
  static constexpr int SMEM_BYTES = Q_BYTES + STAGES * 2 * KV_TILE_BYTES + P_BYTES + 256;  // (no alignment slack)
  static constexpr int TMEM_S0 = 0;
  static constexpr int TMEM_S1 = BKV;
  static constexpr int TMEM_O = 2 * BKV;
  static constexpr int TMEM_COLS = (2 * BKV + DV <= 256) ? 256 : 512;
  static_assert(2 * BKV + DV <= 512, "TMEM budget");
  // two CTAs per SM: 228 KiB per SM, 1 KiB reserved per CTA
  static constexpr int MIN_CTAS = (SMEM_BYTES <= 113 * 1024 && TMEM_COLS <= 256) ? 2 : 1;
};

template <int D>
__global__ void __launch_bounds__(ATT_THREADS, AttnCfg<D>::MIN_CTAS)
attention_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK0,
                 const __grid_constant__ CUtensorMap tmV0, const __grid_constant__ CUtensorMap tmK1,
                 const __grid_constant__ CUtensorMap tmV1, const AttnKParams p) {
  using Cfg = AttnCfg<D>;
  constexpr int ND = Cfg::ND, BKV = Cfg::BKV, STAGES = Cfg::STAGES, DV = Cfg::DV;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) {  // SWIZZLE_128B tiles need it; no slack is budgeted (see Cfg)
    if (threadIdx.x == 0) printf("idiff: attention shared memory base not 1024-byte aligned\n");
    __trap();
  }
  uint8_t* sQ = smem;
  uint8_t* sK = sQ + Cfg::Q_BYTES;
  uint8_t* sV = sK + STAGES * Cfg::KV_TILE_BYTES;
  uint8_t* sP = sV + STAGES * Cfg::KV_TILE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + Cfg::P_BYTES);
  uint64_t* q_full = bars;                 // 1
  uint64_t* k_full = bars + 1;             // STAGES
  uint64_t* v_full = k_full + STAGES;      // STAGES
  uint64_t* kv_empty = v_full + STAGES;    // STAGES
  uint64_t* s_full = kv_empty + STAGES;    // 2
  uint64_t* p_full = s_full + 2;           // 1 (128 arrivals)
  uint64_t* pv_done = p_full + 1;          // 1
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(pv_done + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int q0 = blockIdx.x * BQ;
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
    mbar_init(&s_full[0], 1);
    mbar_init(&s_full[1], 1);
    mbar_init(p_full, 128);
    mbar_init(pv_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(q_full, Cfg::Q_BYTES);
      for (int c = 0; c < ND; ++c) tma_load_4d(sQ + c * BQ * 128, &tmQ, q_full, c * 64, h, q0, b);
      for (int j = 0; j < T; ++j) {
        const int s = j % STAGES;
        const uint32_t ph = (j / STAGES) & 1;
        mbar_wait(&kv_empty[s], ph ^ 1);
        const bool seg1 = j >= T0;
        const int row = (seg1 ? (j - T0) : j) * BKV;
        const int bb = seg1 ? (p.kv1_broadcast ? 0 : b) : b;
        const CUtensorMap* mk = seg1 ? &tmK1 : &tmK0;
        const CUtensorMap* mv = seg1 ? &tmV1 : &tmV0;
        mbar_expect_tx(&k_full[s], Cfg::KV_TILE_BYTES);
        for (int c = 0; c < ND; ++c)
          tma_load_4d(sK + s * Cfg::KV_TILE_BYTES + c * BKV * 128, mk, &k_full[s], c * 64, h, row, bb);
        mbar_expect_tx(&v_full[s], Cfg::KV_TILE_BYTES);
        for (int c = 0; c < ND; ++c)
          tma_load_4d(sV + s * Cfg::KV_TILE_BYTES + c * BKV * 128, mv, &v_full[s], c * 64, h, row, bb);
      }
    }
  } else if (warp == 1) {
    // ===================== UMMA issuer =====================
    // all 32 lanes walk the (warp-uniform) schedule, one elected lane issues: the descriptors then live in
    // uniform registers and the UMMAs of a product issue back to back (see gemm2.cu: as a single-lane loop every
    // tcgen05.mma cost ~20 instructions of R2UR moves and an ELECT retry loop on the pacing thread)
    {
      constexpr uint32_t idesc_qk = make_idesc_f16(BQ, BKV, UMMA_AB_FMT, 0, 0);
      constexpr uint32_t idesc_pv = make_idesc_f16(BQ, DV, UMMA_AB_FMT, 0, /*B MN-major*/ 1);
      const uint32_t q_base = smem_u32(sQ);
      const uint32_t p_base = smem_u32(sP);
      auto issue_qk = [&](int j) {
        const int s = j % STAGES;
        mbar_wait(&k_full[s], (j / STAGES) & 1);
        tc_fence_after();
        const uint32_t k_base = smem_u32(sK + s * Cfg::KV_TILE_BYTES);
        const uint32_t d_tmem = tmem_base + ((j & 1) ? Cfg::TMEM_S1 : Cfg::TMEM_S0);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < Cfg::KSTEPS; ++kk) {
            const uint64_t adesc =
                make_smem_desc_sw128(q_base + (kk >> 2) * (BQ * 128) + (kk & 3) * 32, 16, 1024);
            const uint64_t bdesc =
                make_smem_desc_sw128(k_base + (kk >> 2) * (BKV * 128) + (kk & 3) * 32, 16, 1024);
            umma_f16_ss(d_tmem, adesc, bdesc, idesc_qk, kk > 0 ? 1u : 0u);
          }
          umma_commit(&s_full[j & 1]);
        }
        __syncwarp();
      };
      mbar_wait(q_full, 0);
      issue_qk(0);
      for (int j = 0; j < T; ++j) {
        if (j + 1 < T) issue_qk(j + 1);
        const int s = j % STAGES;
        mbar_wait(p_full, j & 1);
        mbar_wait(&v_full[s], (j / STAGES) & 1);
        tc_fence_after();
        const uint32_t v_base = smem_u32(sV + s * Cfg::KV_TILE_BYTES);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < BKV / 16; ++kk) {
            const uint64_t adesc =
                make_smem_desc_sw128(p_base + (kk >> 2) * (BQ * 128) + (kk & 3) * 32, 16, 1024);
            // V tile: [BKV keys][64 d] rows of 128 B per d-chunk = MN-major, 8-key atoms of 1024 B,
            // next 64-wide d chunk BKV*128 B further on (LBO).
            const uint64_t bdesc = make_smem_desc_sw128(v_base + kk * 2048, BKV * 128, 1024);
            umma_f16_ss(tmem_base + Cfg::TMEM_O, adesc, bdesc, idesc_pv, (j > 0 || kk > 0) ? 1u : 0u);
          }
          umma_commit(&kv_empty[s]);
          umma_commit(pv_done);
        }
        __syncwarp();
      }
    }
    __syncwarp();
  } else {
    // ===================== softmax / correction / epilogue =====================
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const uint32_t lane_off = static_cast<uint32_t>(quarter * 32) << 16;
    const float c = p.scale_log2e;
    float m_run = -INFINITY;
    float l_run = 0.f;
    uint8_t* p_row = sP + r * 128;
    const int sw = r & 7;

    for (int j = 0; j < T; ++j) {
      const bool seg1 = j >= T0;
      const int row0 = (seg1 ? (j - T0) : j) * BKV;
      const int nvalid = min(BKV, (seg1 ? p.n1 : p.n0) - row0);
      mbar_wait(&s_full[j & 1], (j >> 1) & 1);
      tc_fence_after();
      const uint32_t s_addr = tmem_base + lane_off + ((j & 1) ? Cfg::TMEM_S1 : Cfg::TMEM_S0);

      // pass 1: row maximum over the valid keys
      float m_tile = -INFINITY;
#pragma unroll
      for (int c0 = 0; c0 < BKV; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(s_addr + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 32; ++jj)
          if (c0 + jj < nvalid) m_tile = fmaxf(m_tile, __uint_as_float(v[jj]));
      }
      const float m_new = fmaxf(m_run, m_tile);
      const float alpha = exp2_approx((m_run - m_new) * c);  // m_run = -inf -> 0
      const float mc = m_new * c;

      // pass 2: p = 2^(s*c - m*c), packed to fp16 pairs
      uint32_t pk[BKV / 2];
      float l_tile = 0.f;
#pragma unroll
      for (int c0 = 0; c0 < BKV; c0 += 32) {
        uint32_t v[32];
        tmem_ld_32x32b_x32(s_addr + c0, v);
        tmem_ld_wait();
#pragma unroll
        for (int jj = 0; jj < 32; jj += 2) {
          float p0 = (c0 + jj < nvalid) ? exp2_approx(fmaf(__uint_as_float(v[jj]), c, -mc)) : 0.f;
          float p1 = (c0 + jj + 1 < nvalid) ? exp2_approx(fmaf(__uint_as_float(v[jj + 1]), c, -mc)) : 0.f;
          l_tile += p0 + p1;
          pk[(c0 + jj) >> 1] = pack_half2(p0, p1);
        }
      }
      l_run = l_run * alpha + l_tile;
      m_run = m_new;

      if (j > 0) {
        // PV(j-1) must have retired before P is overwritten / O rescaled
        mbar_wait(pv_done, (j - 1) & 1);
        tc_fence_after();
        if (__any_sync(0xffffffffu, alpha != 1.0f)) {
#pragma unroll
          for (int c0 = 0; c0 < DV; c0 += 32) {
            uint32_t o[32];
            tmem_ld_32x32b_x32(tmem_base + lane_off + Cfg::TMEM_O + c0, o);
            tmem_ld_wait();
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) o[jj] = __float_as_uint(__uint_as_float(o[jj]) * alpha);
            tmem_st_32x32b_x32(tmem_base + lane_off + Cfg::TMEM_O + c0, o);
          }
          tmem_st_wait();
        }
      }
      // P row -> smem, K-major 128B-swizzled: 16-byte chunk i of the row lands at (i ^ (r & 7))
#pragma unroll
      for (int i = 0; i < BKV / 8; ++i) {
        uint4 val = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        uint8_t* dst = p_row + (i >> 3) * (BQ * 128) + (((i & 7) ^ sw) << 4);
        *reinterpret_cast<uint4*>(dst) = val;
      }
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(p_full);
    }

    // epilogue: O / l -> fp16
    mbar_wait(pv_done, (T - 1) & 1);
    tc_fence_after();
    const float inv_l = 1.0f / l_run;
    const int qrow = q0 + r;
    const bool row_ok = qrow < p.nq;
    h16* orow = p.out + ((long)b * p.nq + qrow) * p.out_ld + h * D;
#pragma unroll
    for (int c0 = 0; c0 < DV; c0 += 32) {
      if (c0 >= D) break;
      uint32_t o[32];
      tmem_ld_32x32b_x32(tmem_base + lane_off + Cfg::TMEM_O + c0, o);
      tmem_ld_wait();
      if (row_ok) {
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8) {
          if (c0 + j8 * 8 >= D) break;
          uint4 ov;
          ov.x = pack_half2(__uint_as_float(o[j8 * 8 + 0]) * inv_l, __uint_as_float(o[j8 * 8 + 1]) * inv_l);
          ov.y = pack_half2(__uint_as_float(o[j8 * 8 + 2]) * inv_l, __uint_as_float(o[j8 * 8 + 3]) * inv_l);
          ov.z = pack_half2(__uint_as_float(o[j8 * 8 + 4]) * inv_l, __uint_as_float(o[j8 * 8 + 5]) * inv_l);
          ov.w = pack_half2(__uint_as_float(o[j8 * 8 + 6]) * inv_l, __uint_as_float(o[j8 * 8 + 7]) * inv_l);
          *reinterpret_cast<uint4*>(orow + c0 + j8 * 8) = ov;
        }
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

template <int D>
static int launch_attention(const idiff_attn_args* a, cudaStream_t stream) {
  using Cfg = AttnCfg<D>;
  CUtensorMap tmQ, tmK0, tmV0, tmK1, tmV1;
  if (make_head_tmap(&tmQ, a->q, D, a->heads, a->nq, a->batch, a->q_ld, BQ)) return -1;
  if (make_head_tmap(&tmK0, a->k0, D, a->heads, a->n0, a->batch, a->k0_ld, Cfg::BKV)) return -1;
  if (make_head_tmap(&tmV0, a->v0, D, a->heads, a->n0, a->batch, a->v0_ld, Cfg::BKV)) return -1;
  if (a->n1 > 0) {
    const int b1 = a->kv1_batch == 1 ? 1 : a->batch;
    if (make_head_tmap(&tmK1, a->k1, D, a->heads, a->n1, b1, a->k1_ld, Cfg::BKV)) return -1;
    if (make_head_tmap(&tmV1, a->v1, D, a->heads, a->n1, b1, a->v1_ld, Cfg::BKV)) return -1;
  } else {
    tmK1 = tmK0;
    tmV1 = tmV0;
  }
  AttnKParams p;
  p.heads = a->heads;
  p.nq = a->nq;
  p.n0 = a->n0;
  p.n1 = a->n1;
  p.kv1_broadcast = (a->kv1_batch == 1) ? 1 : 0;
  p.scale_log2e = a->scale * 1.4426950408889634f;
  p.out = reinterpret_cast<h16*>(a->out);
  p.out_ld = a->out_ld;
  static bool attr_set = false;
  if (!attr_set) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(attention_kernel<D>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          Cfg::SMEM_BYTES));
    attr_set = true;
  }
  dim3 grid((a->nq + BQ - 1) / BQ, a->heads, a->batch);
  attention_kernel<D><<<grid, ATT_THREADS, Cfg::SMEM_BYTES, stream>>>(tmQ, tmK0, tmV0, tmK1, tmV1, p);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace idiff

extern "C" int idiff_attention(const idiff_attn_args* a, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(a && a->q && a->k0 && a->v0 && a->out, "idiff_attention: null pointer argument");
  IDIFF_REQUIRE(a->nq > 0 && a->n0 > 0 && a->n1 >= 0 && a->batch > 0 && a->heads > 0,
                "idiff_attention: bad shape");
  IDIFF_REQUIRE(a->n1 == 0 || (a->k1 && a->v1), "idiff_attention: segment 1 pointers missing");
  IDIFF_REQUIRE(a->out_ld % 8 == 0 && (reinterpret_cast<uintptr_t>(a->out) & 15) == 0,
                "idiff_attention: out must be 16B aligned, out_ld %% 8 == 0");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  if (a->mask_q || a->mask_k) {
    IDIFF_REQUIRE(a->mask_q && a->mask_k, "idiff_attention: mask_q and mask_k come together");
    IDIFF_REQUIRE(a->head_dim == 40, "idiff_attention: the instance-isolation mask exists at the 64x64 level only "
                                     "(head_dim 40; attention.py:197), got head_dim %d", a->head_dim);
    IDIFF_REQUIRE(a->n0 % 4 == 0 && (a->n0 + a->n1) % 4 == 0 && (reinterpret_cast<uintptr_t>(a->mask_k) & 15) == 0,
                  "idiff_attention: mask_k must be 16B aligned with n0 and n0 + n1 multiples of 4");
    return att2::attention_v2_d40(a, s);
  }
  switch (a->head_dim) {
    case 40: return att2::attention_v2_d40(a, s);  // attention2.cu: two Q tiles per CTA, FMA-pipe exponentials
    case 80: return launch_attention<80>(a, s);
    case 160: return launch_attention<160>(a, s);
    default: return set_error("idiff_attention: unsupported head_dim %d (40/80/160)", a->head_dim);
  }
}
