// HBM-bound normalisation passes over fp16 token-major (NHWC) activations.
//   GroupNorm32 / Normalize : util.py:223-225 (eps 1e-5, fp32 statistics), attention.py:75-76 (eps 1e-6)
//   LayerNorm               : attention.py:294-295, 320-322
// Statistics are accumulated in fp32 in a fixed order (no floating-point atomics), so results
// are bit-reproducible and independent of how many samples share a launch.  SiLU
// (openaimodel.py:184,208,462) is fused into the GroupNorm apply pass.
//
// Thread mapping (both GroupNorm passes): a CTA has k * CV threads, CV = C/8 16-byte vectors per
// pixel; thread (r, cv) owns vector cv of pixels r, r+k, ... of the CTA's pixel chunk, so every
// warp-wide request is a run of consecutive 16-byte vectors and each thread keeps several
// independent loads in flight.
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {

constexpr int GN_MAX_GROUPS = 32;
constexpr int GN_MAX_CHUNKS = 64;  // pixel chunks per sample (two per lane in the apply pass's statistics reduction)

IDIFF_DEVICE void unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = unpack_half2(u[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}

// grid (chunks, B), block k*CV.  partial: [B][groups][GN_MAX_CHUNKS] (sum, sumsq) pairs, chunk fastest, so that the
// apply pass reduces a group's chunks with coalesced loads and a butterfly.  (Measured, round 2: 512-thread CTAs with
// eight loads in flight per thread and half as many chunks were SLOWER -- 4096x320: 42 vs 38 us for the pair -- the
// pass is bound by CTA count / tail, not by loads in flight; profiles/r2_ncu_gn_stats_kernel.summary.csv.)
__global__ void __launch_bounds__(512)
gn_stats_kernel(const uint4* __restrict__ x, float* __restrict__ partial, int hw, int C, int groups,
                int pix_per_block, int k) {
  extern __shared__ float red[];  // [k][C][2]
  const int CV = C >> 3;
  const int r = threadIdx.x / CV;
  const int cv = threadIdx.x - r * CV;
  const int b = blockIdx.y;
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(hw, p0 + pix_per_block);
  const uint4* xb = x + (long)b * hw * CV + cv;
  float s[8], ss[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = ss[j] = 0.f;
  int pix = p0 + r;
  for (; pix + 7 * k < p1; pix += 8 * k) {
    uint4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = xb[(long)(pix + u * k) * CV];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      float f[8];
      unpack8(v[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += f[j];
        ss[j] += f[j] * f[j];
      }
    }
  }
  for (; pix < p1; pix += k) {
    float f[8];
    unpack8(xb[(long)pix * CV], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[j] += f[j];
      ss[j] += f[j] * f[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[((r * C) + cv * 8 + j) * 2] = s[j];
    red[((r * C) + cv * 8 + j) * 2 + 1] = ss[j];
  }
  __syncthreads();
  // one FULL warp per group (round robin), fixed summation order.  blockDim = k*CV is generally not a
  // multiple of 32 (e.g. 240 for C=320): the trailing partial warp must not take part -- it would
  // shuffle with absent lanes and write the same `partial` slots as a full warp.
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nfull = blockDim.x >> 5;
  const int cpg = C / groups;
  if (nfull == 0) {  // fewer than 32 threads (tiny maps through the C ABI): serial, still fixed order
    if (threadIdx.x == 0) {
      for (int g = 0; g < groups; ++g) {
        float a = 0.f, q = 0.f;
        for (int i = 0; i < cpg * k; ++i) {
          const int rr = i / cpg, c = g * cpg + (i - rr * cpg);
          a += red[(rr * C + c) * 2];
          q += red[(rr * C + c) * 2 + 1];
        }
        float* dst = partial + (((long)b * groups + g) * GN_MAX_CHUNKS + blockIdx.x) * 2;
        dst[0] = a;
        dst[1] = q;
      }
    }
    return;
  }
  if (warp >= nfull) return;
  for (int g = warp; g < groups; g += nfull) {
    float a = 0.f, q = 0.f;
    for (int i = lane; i < cpg * k; i += 32) {
      const int rr = i / cpg, c = g * cpg + (i - rr * cpg);
      a += red[(rr * C + c) * 2];
      q += red[(rr * C + c) * 2 + 1];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (lane == 0) {
      float* dst = partial + (((long)b * groups + g) * GN_MAX_CHUNKS + blockIdx.x) * 2;
      dst[0] = a;
      dst[1] = q;
    }
  }
}

// grid (chunks, B), block k*CV
__global__ void __launch_bounds__(512)
gn_apply_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, const float* __restrict__ gamma,
                const float* __restrict__ beta, const float* __restrict__ partial, int hw, int C,
                int groups, float eps, int fuse_silu, int pix_per_block, int k, int stat_chunks) {
  __shared__ float s_mean[GN_MAX_GROUPS], s_rstd[GN_MAX_GROUPS];
  const int CV = C >> 3;
  const int b = blockIdx.y;
  const int cpg = C / groups;
  // statistics: one warp per group, lane = pixel chunk (one coalesced load, fixed-order butterfly) -- the round-1
  // prologue walked up to 64 chunks serially in every CTA before the first pixel moved
  {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nfull = blockDim.x >> 5;
    const float inv_n = 1.0f / (float)((long)cpg * hw);
    if (nfull == 0) {  // fewer than 32 threads (tiny maps through the C ABI): serial, same order
      if (threadIdx.x == 0)
        for (int g = 0; g < groups; ++g) {
          float a = 0.f, q = 0.f;
          for (int ch = 0; ch < stat_chunks; ++ch) {
            const float2 v = *reinterpret_cast<const float2*>(partial + (((long)b * groups + g) * GN_MAX_CHUNKS + ch) * 2);
            a += v.x;
            q += v.y;
          }
          const float mean = a * inv_n;
          s_mean[g] = mean;
          s_rstd[g] = rsqrtf(fmaxf(q * inv_n - mean * mean, 0.f) + eps);
        }
    } else if (warp < nfull) {
      for (int g = warp; g < groups; g += nfull) {
        float2 v = make_float2(0.f, 0.f);
        if (lane < stat_chunks) v = *reinterpret_cast<const float2*>(partial + (((long)b * groups + g) * GN_MAX_CHUNKS + lane) * 2);
        if (lane + 32 < stat_chunks) {
          const float2 w = *reinterpret_cast<const float2*>(partial + (((long)b * groups + g) * GN_MAX_CHUNKS + lane + 32) * 2);
          v.x += w.x;
          v.y += w.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          v.x += __shfl_xor_sync(0xffffffffu, v.x, o);
          v.y += __shfl_xor_sync(0xffffffffu, v.y, o);
        }
        if (lane == 0) {
          const float mean = v.x * inv_n;
          s_mean[g] = mean;
          s_rstd[g] = rsqrtf(fmaxf(v.y * inv_n - mean * mean, 0.f) + eps);
        }
      }
    }
  }
  __syncthreads();
  const int r = threadIdx.x / CV;
  const int cv = threadIdx.x - r * CV;
  float sa[8], sb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int c = cv * 8 + j;
    const int g = c / cpg;
    const float a = s_rstd[g] * gamma[c];
    sa[j] = a;
    sb[j] = beta[c] - s_mean[g] * a;
  }
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(hw, p0 + pix_per_block);
  const long base = (long)b * hw * CV + cv;
  auto norm_store = [&](const uint4& v, long idx) {
    float f[8];
    unpack8(v, f);
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float r0 = f[2 * j] * sa[2 * j] + sb[2 * j];
      float r1 = f[2 * j + 1] * sa[2 * j + 1] + sb[2 * j + 1];
      if (fuse_silu) {
        r0 = silu_f(r0);
        r1 = silu_f(r1);
      }
      o[j] = pack_half2(r0, r1);
    }
    y[idx] = make_uint4(o[0], o[1], o[2], o[3]);
  };
  int pix = p0 + r;
  for (; pix + 7 * k < p1; pix += 8 * k) {
    uint4 v[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) v[u] = x[base + (long)(pix + u * k) * CV];
#pragma unroll
    for (int u = 0; u < 8; ++u) norm_store(v[u], base + (long)(pix + u * k) * CV);
  }
  for (; pix < p1; pix += k) norm_store(x[base + (long)pix * CV], base + (long)pix * CV);
}

// ---------------------------------------------------------------------------------------------
// Single-pass GroupNorm (the default where one wave holds the whole launch).  One thread-block cluster per
// (sample, slab of CS channels = whole groups): every CTA of the cluster streams its share of the
// pixels once from global memory into shared memory while accumulating per-channel sums, the
// per-group partial sums of the CL CTAs are exchanged through distributed shared memory and added in
// rank order (deterministic), and the tile is normalised (+SiLU) straight from shared memory.
// 4 B per element of global traffic and one launch instead of 6 B and two.
// grid (CL * nslabs, B), cluster (CL, 1, 1), block k*CV with CV = CS/8.
// dynamic smem: tile [rows][CV] uint4, then red [k][CS][2] floats.
// ---------------------------------------------------------------------------------------------
constexpr int GNF_MAX_SLAB_GROUPS = 8;

IDIFF_DEVICE void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
IDIFF_DEVICE float ld_dsmem_f32(const float* local, uint32_t rank) {
  uint32_t raddr;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;\n" : "=r"(raddr) : "r"(smem_u32(local)), "r"(rank));
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];\n" : "=f"(v) : "r"(raddr) : "memory");
  return v;
}

__global__ void __launch_bounds__(512)
gn_fused_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, const float* __restrict__ gamma,
                const float* __restrict__ beta, int hw, int C, int groups, float eps, int fuse_silu, int CS,
                int CL, int k) {
  extern __shared__ __align__(16) uint8_t gnf_smem[];
  __shared__ float cta_part[GNF_MAX_SLAB_GROUPS * 2];  // this CTA's (sum, sumsq) per group of the slab
  __shared__ float s_mean[GNF_MAX_SLAB_GROUPS], s_rstd[GNF_MAX_SLAB_GROUPS];
  const int CV = CS >> 3;       // 16-byte vectors per pixel of the slab
  const int CVT = C >> 3;       // ... of the whole tensor
  const int rank = blockIdx.x % CL;
  const int slab = blockIdx.x / CL;
  const int b = blockIdx.y;
  const int rows = hw / CL;     // pixels of this CTA (host guarantees divisibility)
  const int cpg = C / groups;
  const int ng = CS / cpg;      // groups in the slab
  uint4* tile = reinterpret_cast<uint4*>(gnf_smem);
  float* red = reinterpret_cast<float*>(gnf_smem + (size_t)rows * CV * sizeof(uint4));

  const int r = threadIdx.x / CV;
  const int cv = threadIdx.x - r * CV;
  const uint4* xb = x + ((long)b * hw + (long)rank * rows) * CVT + slab * CV + cv;
  float s[8], ss[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = ss[j] = 0.f;
  int pix = r;
  for (; pix + 3 * k < rows; pix += 4 * k) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = xb[(long)(pix + u * k) * CVT];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      tile[(pix + u * k) * CV + cv] = v[u];
      float f[8];
      unpack8(v[u], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += f[j];
        ss[j] += f[j] * f[j];
      }
    }
  }
  for (; pix < rows; pix += k) {
    const uint4 v = xb[(long)pix * CVT];
    tile[pix * CV + cv] = v;
    float f[8];
    unpack8(v, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      s[j] += f[j];
      ss[j] += f[j] * f[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    red[((r * CS) + cv * 8 + j) * 2] = s[j];
    red[((r * CS) + cv * 8 + j) * 2 + 1] = ss[j];
  }
  __syncthreads();
  // one warp per group of the slab (round robin), fixed summation order
  // full warps only (blockDim = k*CV need not be a multiple of 32; gn_fused_geometry guarantees >= 32)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  for (int g = warp; warp < nwarps && g < ng; g += nwarps) {
    float a = 0.f, q = 0.f;
    for (int i = lane; i < cpg * k; i += 32) {
      const int rr = i / cpg, c = g * cpg + (i - rr * cpg);
      a += red[(rr * CS + c) * 2];
      q += red[(rr * CS + c) * 2 + 1];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      q += __shfl_xor_sync(0xffffffffu, q, o);
    }
    if (lane == 0) {
      cta_part[g * 2] = a;
      cta_part[g * 2 + 1] = q;
    }
  }
  cluster_sync_all();  // every CTA's partials are written and visible cluster-wide
  if (threadIdx.x < ng) {
    float a = 0.f, q = 0.f;
    for (int rk = 0; rk < CL; ++rk) {  // rank order: the same sum in every CTA of the cluster
      a += ld_dsmem_f32(&cta_part[threadIdx.x * 2], rk);
      q += ld_dsmem_f32(&cta_part[threadIdx.x * 2 + 1], rk);
    }
    const float inv_n = 1.0f / (float)((long)cpg * hw);
    const float mean = a * inv_n;
    const float var = fmaxf(q * inv_n - mean * mean, 0.f);
    s_mean[threadIdx.x] = mean;
    s_rstd[threadIdx.x] = rsqrtf(var + eps);
  }
  cluster_sync_all();  // (also a CTA barrier) no CTA leaves while its partials may still be read
  float sa[8], sb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int cl = cv * 8 + j;          // channel within the slab
    const int c = slab * CS + cl;       // channel of the tensor
    const float a = s_rstd[cl / cpg] * gamma[c];
    sa[j] = a;
    sb[j] = beta[c] - s_mean[cl / cpg] * a;
  }
  uint4* yb = y + ((long)b * hw + (long)rank * rows) * CVT + slab * CV + cv;
  for (pix = r; pix < rows; pix += k) {
    float f[8];
    unpack8(tile[pix * CV + cv], f);  // written by this very thread above
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float r0 = f[2 * j] * sa[2 * j] + sb[2 * j];
      float r1 = f[2 * j + 1] * sa[2 * j + 1] + sb[2 * j + 1];
      if (fuse_silu) {
        r0 = silu_f(r0);
        r1 = silu_f(r1);
      }
      o[j] = pack_half2(r0, r1);
    }
    yb[(long)pix * CVT] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm.  Fast path: C in {320, 640, 1280} = 40 * LPR: LPR lanes cooperate on a row, five
// 16-byte vectors per lane held in registers, 32/LPR rows per warp.  Generic path: one warp per row.
// ---------------------------------------------------------------------------------------------
template <int LPR>
__global__ void __launch_bounds__(256)
layernorm40_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, const float* __restrict__ gamma,
                   const float* __restrict__ beta, int rows, float eps) {
  constexpr int C = 40 * LPR;
  constexpr int CV = C / 8;  // 5 * LPR
  constexpr int RPW = 32 / LPR;
  const int warp_global = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPR, l = lane - sub * LPR;
  const int row = warp_global * RPW + sub;
  const bool ok = row < rows;
  float v[40];
  if (ok) {
    uint4 u[5];
#pragma unroll
    for (int i = 0; i < 5; ++i) u[i] = x[(long)row * CV + l + i * LPR];
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      float f[8];
      unpack8(u[i], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[i * 8 + j] = f[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < 40; ++j) v[j] = 0.f;
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 40; ++j) s += v[j];
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s * (1.0f / C);
  float ss = 0.f;
#pragma unroll
  for (int j = 0; j < 40; ++j) {
    const float d = v[j] - mean;
    ss += d * d;
  }
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = rsqrtf(ss * (1.0f / C) + eps);
  if (ok) {
#pragma unroll
    for (int i = 0; i < 5; ++i) {
      const int c0 = (l + i * LPR) * 8;
      const float4 g0 = *reinterpret_cast<const float4*>(gamma + c0);
      const float4 g1 = *reinterpret_cast<const float4*>(gamma + c0 + 4);
      const float4 b0 = *reinterpret_cast<const float4*>(beta + c0);
      const float4 b1 = *reinterpret_cast<const float4*>(beta + c0 + 4);
      const float g[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
      const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float r0 = (v[i * 8 + 2 * j] - mean) * rstd * g[2 * j] + bb[2 * j];
        const float r1 = (v[i * 8 + 2 * j + 1] - mean) * rstd * g[2 * j + 1] + bb[2 * j + 1];
        o[j] = pack_half2(r0, r1);
      }
      y[(long)row * CV + l + i * LPR] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}

constexpr int LN_MAX_VEC = 5;  // generic path: C <= 1280
__global__ void __launch_bounds__(256)
layernorm_generic_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, const float* __restrict__ gamma,
                         const float* __restrict__ beta, int rows, int C, float eps) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int CV = C >> 3;
  float v[LN_MAX_VEC * 8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAX_VEC; ++i) {
    const int cv = lane + i * 32;
    if (cv < CV) {
      float f[8];
      unpack8(x[(long)row * CV + cv], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[i * 8 + j] = f[j];
        s += f[j];
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)C;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < LN_MAX_VEC; ++i) {
    const int cv = lane + i * 32;
    if (cv < CV) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[i * 8 + j] - mean;
        ss += d * d;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = rsqrtf(ss / (float)C + eps);
#pragma unroll
  for (int i = 0; i < LN_MAX_VEC; ++i) {
    const int cv = lane + i * 32;
    if (cv < CV) {
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = cv * 8 + 2 * j;
        const float r0 = (v[i * 8 + 2 * j] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
        const float r1 = (v[i * 8 + 2 * j + 1] - mean) * rstd * __ldg(gamma + c + 1) + __ldg(beta + c + 1);
        o[j] = pack_half2(r0, r1);
      }
      y[(long)row * CV + cv] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}

// Row statistics for the folded LayerNorm (include/idiff_b200.h idiff_gemm_args.ln_*): one warp per row,
// (sum, sum of squares) in fp32, fixed order.  Only used where the stream was not written by idiff_gemm
// (module-level entry points); inside the UNet the producing GEMM's epilogue writes the statistics.
__global__ void __launch_bounds__(256)
row_stats_kernel(const uint4* __restrict__ x, float2* __restrict__ stats, int rows, int CV) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float a = 0.f, q = 0.f;
  for (int cv = lane; cv < CV; cv += 32) {
    float f[8];
    unpack8(x[(long)row * CV + cv], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      a += f[j];
      q = fmaf(f[j], f[j], q);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  if (lane == 0) stats[row] = make_float2(a, q);
}

}  // namespace idiff

extern "C" int idiff_row_stats(const void* x, void* stats, int rows, int channels, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(x && stats && rows > 0, "idiff_row_stats: bad arguments");
  IDIFF_REQUIRE(channels % 8 == 0 && channels > 0, "idiff_row_stats: C=%d must be a multiple of 8", channels);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  row_stats_kernel<<<(rows + 7) / 8, 256, 0, s>>>(reinterpret_cast<const uint4*>(x), reinterpret_cast<float2*>(stats),
                                                  rows, channels / 8);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

// geometry shared by the GroupNorm launches and the workspace-size query
static void gn_geometry(int batch, int hw, int channels, int* k, int* ppb, int* chunks) {
  const int CV = channels / 8;
  int kk = 256 / CV;
  if (kk < 1) kk = 1;
  if (kk > hw) kk = hw;
  // aim at >= ~4 CTAs per SM over the whole launch, at most GN_MAX_CHUNKS chunks per sample
  int want = (148 * 4 + batch - 1) / batch;
  if (want > idiff::GN_MAX_CHUNKS) want = idiff::GN_MAX_CHUNKS;
  if (want < 1) want = 1;
  int p = (hw + want - 1) / want;
  p = ((p + kk - 1) / kk) * kk;  // multiple of k
  if (p < kk) p = kk;
  *k = kk;
  *ppb = p;
  *chunks = (hw + p - 1) / p;
}

// Single-pass variant: slab width CS (whole groups and whole 16-byte vectors), cluster size CL (pixels
// split over CL CTAs), k pixel rows per block pass.  Returns false when the shape does not fit.
static bool gn_fused_geometry(int batch, int hw, int channels, int groups, int* CS, int* CL, int* k, size_t* smem) {
  const int cpg = channels / groups;
  int unit = cpg;  // lcm(cpg, 8)
  while (unit % 8 != 0) unit += cpg;
  if (channels % unit != 0 || unit / cpg > idiff::GNF_MAX_SLAB_GROUPS) return false;
  int cs = unit;
  while (cs * 2 <= 160 && channels % (cs * 2) == 0 && (cs * 2) / cpg <= idiff::GNF_MAX_SLAB_GROUPS) cs *= 2;
  const int CV = cs / 8;
  int kk = 512 / CV;
  if (kk < 1) return false;
  int cl = 1;
  const size_t budget = 160 * 1024;
  while (cl < 8 && ((size_t)(hw / cl) * cs * 2 > budget)) cl *= 2;
  if (hw % cl != 0 || (size_t)(hw / cl) * cs * 2 > budget) return false;
  // fill the machine: more CTAs per sample while the launch is below one wave
  while (cl < 8 && hw % (cl * 2) == 0 && (long)batch * (channels / cs) * cl < 128 && hw / (cl * 2) >= kk) cl *= 2;
  if (kk > hw / cl) kk = hw / cl;
  if (kk < 1 || kk * CV < 32) return false;  // the group reduction needs at least one full warp
  *CS = cs;
  *CL = cl;
  *k = kk;
  *smem = (size_t)(hw / cl) * cs * 2 + (size_t)kk * cs * 2 * sizeof(float);
  // Measured (profiles/README.md, NEXT.md): with these 100-190 KB tiles the single pass wins only while
  // the whole launch is resident at once; beyond one wave the two-kernel path is faster.
  if ((long)batch * (channels / cs) * cl > 148) return false;
  return *smem <= 200 * 1024;
}

extern "C" int idiff_groupnorm(const void* x, void* y, const float* gamma, const float* beta,
                               float* stats_ws, int batch, int hw, int channels, int groups,
                               float eps, int fuse_silu, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(x && y && gamma && beta && stats_ws, "idiff_groupnorm: null pointer argument");
  IDIFF_REQUIRE(groups > 0 && groups <= GN_MAX_GROUPS && channels % groups == 0,
                "idiff_groupnorm: bad groups=%d for C=%d", groups, channels);
  IDIFF_REQUIRE(channels % 8 == 0 && channels <= 4096, "idiff_groupnorm: C=%d must be a multiple of 8, <= 4096", channels);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  {
    // Single-pass cluster kernel wherever the launch fits one wave (gn_fused_geometry): measured 42 -> 31 us at
    // 4096x320, 36 -> 21 at 1024x640, 26 -> 16 at 256x1280, 22 -> 12 at 64x1280 (batch 8; profiles/README.md);
    // IDIFF_GN_FUSED=0 forces the two-kernel path (read per call so tests can cover both).
    const char* fe = getenv("IDIFF_GN_FUSED");
    const bool fused_on = !(fe && fe[0] == '0');
    int CS, CL, kf;
    size_t smem_f;
    if (fused_on && gn_fused_geometry(batch, hw, channels, groups, &CS, &CL, &kf, &smem_f)) {
      static bool fattr = false;
      if (!fattr) {
        IDIFF_CHECK_CUDA(cudaFuncSetAttribute(gn_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        fattr = true;
      }
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(CL * (channels / CS), batch);
      cfg.blockDim = dim3(kf * (CS / 8));
      cfg.dynamicSmemBytes = smem_f;
      cfg.stream = s;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = CL;
      attr[0].val.clusterDim.y = 1;
      attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      IDIFF_CHECK_CUDA(cudaLaunchKernelEx(&cfg, gn_fused_kernel, reinterpret_cast<const uint4*>(x),
                                          reinterpret_cast<uint4*>(y), gamma, beta, hw, channels, groups, eps,
                                          fuse_silu, CS, CL, kf));
      return 0;
    }
  }
  int k, ppb, chunks;
  gn_geometry(batch, hw, channels, &k, &ppb, &chunks);
  const int threads = k * (channels / 8);
  const size_t smem = (size_t)k * channels * 2 * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(gn_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    attr_set = true;
  }
  IDIFF_REQUIRE(smem <= 96 * 1024, "idiff_groupnorm: shared memory %zu too large", smem);
  dim3 grid(chunks, batch);
  gn_stats_kernel<<<grid, threads, smem, s>>>(reinterpret_cast<const uint4*>(x), stats_ws, hw, channels, groups, ppb, k);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  gn_apply_kernel<<<grid, threads, 0, s>>>(reinterpret_cast<const uint4*>(x), reinterpret_cast<uint4*>(y), gamma, beta,
                                           stats_ws, hw, channels, groups, eps, fuse_silu, ppb, k, chunks);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" long idiff_groupnorm_ws_floats(int batch, int groups) {
  return (long)batch * idiff::GN_MAX_CHUNKS * groups * 2;
}

extern "C" int idiff_layernorm(const void* x, void* y, const float* gamma, const float* beta,
                               int rows, int channels, float eps, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(x && y && gamma && beta, "idiff_layernorm: null pointer argument");
  IDIFF_REQUIRE(channels % 8 == 0 && channels <= 8 * 32 * LN_MAX_VEC,
                "idiff_layernorm: unsupported C=%d", channels);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const uint4* xi = reinterpret_cast<const uint4*>(x);
  uint4* yo = reinterpret_cast<uint4*>(y);
  const int warps_per_block = 8;
  auto blocks = [&](int rows_per_warp) {
    const int rpb = warps_per_block * rows_per_warp;
    return (rows + rpb - 1) / rpb;
  };
  if (channels == 320) {
    layernorm40_kernel<8><<<blocks(4), 256, 0, s>>>(xi, yo, gamma, beta, rows, eps);
  } else if (channels == 640) {
    layernorm40_kernel<16><<<blocks(2), 256, 0, s>>>(xi, yo, gamma, beta, rows, eps);
  } else if (channels == 1280) {
    layernorm40_kernel<32><<<blocks(1), 256, 0, s>>>(xi, yo, gamma, beta, rows, eps);
  } else {
    layernorm_generic_kernel<<<blocks(1), 256, 0, s>>>(xi, yo, gamma, beta, rows, channels, eps);
  }
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}
