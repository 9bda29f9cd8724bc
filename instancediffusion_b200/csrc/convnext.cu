// ConvNeXt mask encoder of UniFusion (mask conditioning, non-zero `segs`): the pieces that are not a
// GEMM.  Reference: ldm/modules/diffusionmodules/convnext.py:15-123 and
// text_grounding_net.py:226-231, 277-287.  The encoder runs once per sample (its input never changes
// across denoising steps), so these are plain coalesced HBM kernels; the pointwise convolutions, the
// 4x4 / 2x2 patchify convolutions and the MLP are tcgen05 GEMMs (gemm2.cu, GELU epilogue flag).
//
//   segs (B,30,S,S) fp32 --nearest resize to 512, conv3x3 30->3-->  NHWC fp16 (B,512,512,3)   [segs_inconv]
//   patchify p x p (stride p)  -> [B*(H/p)*(W/p), p*p*C] rows for the strided-conv GEMMs       [patchify]
//   depthwise 7x7, padding 3, NHWC                                                             [dwconv7x7]
//   token reinterpretation reshape(B,-1,64).permute(0,2,1) + null substitution + pos embedding [seg_tokens]
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {

// ---------------------------------------------------------------------------------------------
// segs -> in_conv (text_grounding_net.py:227-228): F.interpolate(segs, 512, mode="nearest") then
// Conv2d(30, 3, 3, 1, 1), fp32 arithmetic, NHWC fp16 out.  Also accumulates sum(resized segs) per sample
// (the `masks_segs` test of :279).  One thread per output pixel; a warp reads 32 consecutive x.
// w: [3][CI][3][3] fp32 (the module's layout), staged in shared memory.
// ---------------------------------------------------------------------------------------------
constexpr int INCONV_MAX_CI = 32;
__global__ void __launch_bounds__(256)
segs_inconv_kernel(const float* __restrict__ segs, const float* __restrict__ w, const float* __restrict__ bias,
                   h16* __restrict__ y, float* __restrict__ seg_sum, int B, int CI, int S, int R,
                   long sb, long sc, long sy, long sx) {
  __shared__ float sw[3 * INCONV_MAX_CI * 9];
  __shared__ float red[8];
  for (int i = threadIdx.x; i < 3 * CI * 9; i += blockDim.x) sw[i] = w[i];
  __syncthreads();
  const int b = blockIdx.z;
  const int oy = blockIdx.y;
  const int ox = blockIdx.x * blockDim.x + threadIdx.x;
  const float ratio = (float)S / (float)R;  // torch 'nearest': src = min(floor(dst * in/out), in-1)
  float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, centre_sum = 0.f;
  if (ox < R) {
    int iy[3], ix[3];
    bool vy[3], vx[3];
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int yy = oy + t - 1, xx = ox + t - 1;
      vy[t] = yy >= 0 && yy < R;
      vx[t] = xx >= 0 && xx < R;
      iy[t] = min((int)floorf((float)(vy[t] ? yy : 0) * ratio), S - 1);
      ix[t] = min((int)floorf((float)(vx[t] ? xx : 0) * ratio), S - 1);
    }
    const float* sbp = segs + (long)b * sb;
    for (int c = 0; c < CI; ++c) {
      const float* p = sbp + (long)c * sc;
      const float* w0 = sw + (0 * CI + c) * 9;
      const float* w1 = sw + (1 * CI + c) * 9;
      const float* w2 = sw + (2 * CI + c) * 9;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float v = (vy[ky] && vx[kx]) ? __ldg(p + (long)iy[ky] * sy + (long)ix[kx] * sx) : 0.f;
          acc0 = fmaf(v, w0[ky * 3 + kx], acc0);
          acc1 = fmaf(v, w1[ky * 3 + kx], acc1);
          acc2 = fmaf(v, w2[ky * 3 + kx], acc2);
          if (ky == 1 && kx == 1) centre_sum += v;
        }
      }
    }
    h16* o = y + (((long)b * R + oy) * R + ox) * 3;
    o[0] = f2h(acc0 + bias[0]);
    o[1] = f2h(acc1 + bias[1]);
    o[2] = f2h(acc2 + bias[2]);
  }
  // per-sample sum of the resized masks (block reduce, one atomic per block; masks are >= 0 in practice,
  // so the order of this fp32 sum cannot change the `> 0` test it feeds)
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) centre_sum += __shfl_xor_sync(0xffffffffu, centre_sum, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = centre_sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) t += red[i];
    if (t != 0.f) atomicAdd(seg_sum + b, t);
  }
}

// ---------------------------------------------------------------------------------------------
// patchify: NHWC (B,H,W,C) -> [B*(H/p)*(W/p), p*p*C], column (ky*p + kx)*C + c.  The stride-p, kernel-p
// convolutions of ConvNeXt (stem 4x4 s4, convnext.py:71-74; downsample 2x2 s2, :77-81) become GEMMs over
// these rows.  VEC = 8 halves per thread when C % 8 == 0, scalar otherwise (the C = 3 stem).
// ---------------------------------------------------------------------------------------------
template <int VEC>
__global__ void patchify_kernel(const h16* __restrict__ x, h16* __restrict__ y, int B, int H, int W, int C,
                                int p) {
  const int CV = C / VEC;
  const int Ho = H / p, Wo = W / p;
  const long total = (long)B * Ho * Wo * p * p * CV;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    long t = i / CV;
    const int kx = (int)(t % p);
    t /= p;
    const int ky = (int)(t % p);
    t /= p;
    const int ox = (int)(t % Wo);
    t /= Wo;
    const int oy = (int)(t % Ho);
    const int b = (int)(t / Ho);
    const long src = ((((long)b * H + oy * p + ky) * W) + ox * p + kx) * CV + cv;
    if (VEC == 8) reinterpret_cast<uint4*>(y)[i] = reinterpret_cast<const uint4*>(x)[src];
    else y[i] = x[src];
  }
}

// ---------------------------------------------------------------------------------------------
// depthwise 7x7, padding 3 (convnext.py:28,38), NHWC fp16 in/out, fp32 accumulation.
// w: fp32 [49][C] (tap-major, repacked on the host from (C,1,7,7)); bias fp32 [C].
// One thread = 8 channels of one output pixel: 49 16-byte loads, weights through the read-only path.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
dwconv7x7_kernel(const uint4* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                 uint4* __restrict__ y, int B, int H, int W, int C) {
  const int CV = C >> 3;
  const long total = (long)B * H * W * CV;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    long t = i / CV;
    const int ox = (int)(t % W);
    t /= W;
    const int oy = (int)(t % H);
    const int b = (int)(t / H);
    float acc[8];
    {
      const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + cv * 8));
      const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + cv * 8 + 4));
      acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w;
      acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
    }
    for (int ky = 0; ky < 7; ++ky) {
      const int iy = oy + ky - 3;
      if (iy < 0 || iy >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 7; ++kx) {
        const int ix = ox + kx - 3;
        if (ix < 0 || ix >= W) continue;
        const uint4 v = x[(((long)b * H + iy) * W + ix) * CV + cv];
        const float* wp = w + (long)(ky * 7 + kx) * C + cv * 8;
        const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp));
        const float4 w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
        const float2 f0 = unpack_half2(v.x), f1 = unpack_half2(v.y), f2 = unpack_half2(v.z), f3 = unpack_half2(v.w);
        acc[0] = fmaf(f0.x, w0.x, acc[0]); acc[1] = fmaf(f0.y, w0.y, acc[1]);
        acc[2] = fmaf(f1.x, w0.z, acc[2]); acc[3] = fmaf(f1.y, w0.w, acc[3]);
        acc[4] = fmaf(f2.x, w1.x, acc[4]); acc[5] = fmaf(f2.y, w1.y, acc[5]);
        acc[6] = fmaf(f3.x, w1.z, acc[6]); acc[7] = fmaf(f3.y, w1.w, acc[7]);
      }
    }
    y[i] = make_uint4(pack_half2(acc[0], acc[1]), pack_half2(acc[2], acc[3]), pack_half2(acc[4], acc[5]),
                      pack_half2(acc[6], acc[7]));
  }
}

// ---------------------------------------------------------------------------------------------
// seg tokens (text_grounding_net.py:229-230, 277-285).  The reference reinterprets the contiguous NCHW
// feature map (B, C, P) -- C = 768 channels, P = 16*16 pixels -- as (B, C*P/T, T) and permutes to
// (B, T, F) with T = 64 tokens, F = C*P/T = 3072: token t, feature r reads flat[r*T + t], i.e. channel
// c = (r*T + t) / P, pixel q = (r*T + t) % P.  Then: has_seg ? feat : null_seg, plus pos_embedding.
// feat: fp16 NHWC [B, P, C]; null_pos: fp16 [T, F] = null_seg + pos (precomputed); pos: fp32 [T, F];
// seg_sum: fp32 [B]; out: fp16 [B*T, F].
// ---------------------------------------------------------------------------------------------
__global__ void seg_tokens_kernel(const h16* __restrict__ feat, const h16* __restrict__ null_pos,
                                  const float* __restrict__ pos, const float* __restrict__ seg_sum,
                                  h16* __restrict__ out, int B, int P, int C, int T) {
  const int F = C * P / T;
  const long total = (long)B * T * F;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int r = (int)(i % F);
    const long bt = i / F;
    const int t = (int)(bt % T);
    const int b = (int)(bt / T);
    if (seg_sum[b] > 0.f) {
      const long flat = (long)r * T + t;
      const int c = (int)(flat / P), q = (int)(flat - (long)c * P);
      out[i] = f2h(h2f(feat[((long)b * P + q) * C + c]) + pos[(long)t * F + r]);
    } else {
      out[i] = null_pos[(long)t * F + r];
    }
  }
}

static int grid_for(long total, int block) {
  long g = (total + block - 1) / block;
  if (g > 148L * 32) g = 148L * 32;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace idiff

extern "C" int idiff_segs_inconv(const float* segs, const long* strides, const float* w, const float* bias,
                                 void* y, float* seg_sum, int batch, int cin, int in_size, int out_size,
                                 void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(segs && strides && w && bias && y && seg_sum, "idiff_segs_inconv: null pointer argument");
  IDIFF_REQUIRE(cin > 0 && cin <= INCONV_MAX_CI, "idiff_segs_inconv: cin=%d must be in [1, %d]", cin, INCONV_MAX_CI);
  IDIFF_REQUIRE(batch > 0 && in_size > 0 && out_size > 0, "idiff_segs_inconv: bad sizes");
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  IDIFF_CHECK_CUDA(cudaMemsetAsync(seg_sum, 0, sizeof(float) * batch, s));
  dim3 grid((out_size + 255) / 256, out_size, batch);
  segs_inconv_kernel<<<grid, 256, 0, s>>>(segs, w, bias, reinterpret_cast<h16*>(y), seg_sum, batch, cin, in_size,
                                          out_size, strides[0], strides[1], strides[2], strides[3]);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_patchify(const void* x, void* y, int batch, int h, int w, int c, int p, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(x && y, "idiff_patchify: null pointer argument");
  IDIFF_REQUIRE(p > 0 && h % p == 0 && w % p == 0, "idiff_patchify: H=%d W=%d must be multiples of p=%d", h, w, p);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const h16* xi = reinterpret_cast<const h16*>(x);
  h16* yo = reinterpret_cast<h16*>(y);
  if (c % 8 == 0) {
    const long total = (long)batch * h * w * (c / 8);
    patchify_kernel<8><<<grid_for(total, 256), 256, 0, s>>>(xi, yo, batch, h, w, c, p);
  } else {
    const long total = (long)batch * h * w * c;
    patchify_kernel<1><<<grid_for(total, 256), 256, 0, s>>>(xi, yo, batch, h, w, c, p);
  }
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_dwconv7x7(const void* x, const float* w, const float* bias, void* y, int batch, int h, int w_,
                               int c, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(x && w && bias && y, "idiff_dwconv7x7: null pointer argument");
  IDIFF_REQUIRE(c % 8 == 0, "idiff_dwconv7x7: C=%d must be a multiple of 8", c);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const long total = (long)batch * h * w_ * (c / 8);
  dwconv7x7_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const uint4*>(x), w, bias,
                                                        reinterpret_cast<uint4*>(y), batch, h, w_, c);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_seg_tokens(const void* feat, const void* null_pos, const float* pos, const float* seg_sum,
                                void* out, int batch, int pixels, int channels, int tokens, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(feat && null_pos && pos && seg_sum && out, "idiff_seg_tokens: null pointer argument");
  IDIFF_REQUIRE(tokens > 0 && ((long)channels * pixels) % tokens == 0,
                "idiff_seg_tokens: C*P=%ld must be a multiple of the token count %d", (long)channels * pixels, tokens);
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const long total = (long)batch * channels * pixels;
  seg_tokens_kernel<<<grid_for(total, 256), 256, 0, s>>>(reinterpret_cast<const h16*>(feat),
                                                         reinterpret_cast<const h16*>(null_pos), pos, seg_sum,
                                                         reinterpret_cast<h16*>(out), batch, pixels, channels, tokens);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}
