// First-stage decoder (AutoencoderKL.decode, ldm/models/autoencoder.py:33-37; Decoder, ldm/modules/
// diffusionmodules/model.py:462-569) -- the pieces that are not idiff_gemm / idiff_groupnorm calls:
//   * latent prologue: z / scale_factor, post_quant_conv (1x1, 4 -> 4), fp32 NCHW -> fp16 NHWC padded to
//     the 64-channel granularity of the conv3x3 kernel's A operand;
//   * row softmax of the single-head mid-block attention (AttnBlock, model.py:150-202): the scores of one
//     image are a [HW, HW] GEMM output (head_dim 512 does not fit the flash kernels' TMEM budget and the
//     block runs once per image), normalised in place.
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {

// grid-stride over pixels; one thread per (pixel): reads C_in <= 8 planes, writes one 128-byte row
__global__ void __launch_bounds__(256)
vae_latent_in_kernel(const float* __restrict__ z, const float* __restrict__ w, const float* __restrict__ bias,
                     float inv_scale, uint4* __restrict__ out, int B, int C, int HW) {
  __shared__ float sw[64], sb[8];
  if (threadIdx.x < C * C) sw[threadIdx.x] = w[threadIdx.x];
  if (threadIdx.x < C) sb[threadIdx.x] = bias[threadIdx.x];
  __syncthreads();
  const long total = (long)B * HW;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int b = (int)(i / HW);
    const int pix = (int)(i - (long)b * HW);
    float zi[8], o[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) zi[c] = (c < C) ? z[((long)b * C + c) * HW + pix] * inv_scale : 0.f;
#pragma unroll
    for (int co = 0; co < 8; ++co) {
      float a = 0.f;
      if (co < C) {
        a = sb[co];
#pragma unroll
        for (int ci = 0; ci < 8; ++ci)
          if (ci < C) a = fmaf(sw[co * C + ci], zi[ci], a);
      }
      o[co] = a;
    }
    uint4* row = out + i * 8;  // 64 halves = 8 x 16 bytes
    row[0] = make_uint4(pack_half2(o[0], o[1]), pack_half2(o[2], o[3]), pack_half2(o[4], o[5]), pack_half2(o[6], o[7]));
    const uint4 zero = make_uint4(0, 0, 0, 0);
#pragma unroll
    for (int q = 1; q < 8; ++q) row[q] = zero;
  }
}

// one CTA per row; the row lives in shared memory as fp32 between the passes
__global__ void __launch_bounds__(256)
softmax_rows_kernel(h16* __restrict__ x, int n, long ld) {
  extern __shared__ float srow[];
  __shared__ float red[8];
  h16* row = x + (long)blockIdx.x * ld;
  const int nv = n >> 3;  // n % 8 == 0
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float m = -INFINITY;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 u = reinterpret_cast<const uint4*>(row)[v];
    const uint32_t uu[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = unpack_half2(uu[j]);
      srow[v * 8 + 2 * j] = f.x;
      srow[v * 8 + 2 * j + 1] = f.y;
      m = fmaxf(m, fmaxf(f.x, f.y));
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) m = fmaxf(m, red[i]);
  __syncthreads();
  float s = 0.f;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float e = exp2_approx((srow[v * 8 + j] - m) * 1.4426950408889634f);
      srow[v * 8 + j] = e;
      s += e;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += red[i];  // fixed order
  const float inv = 1.0f / s;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = pack_half2(srow[v * 8 + 2 * j] * inv, srow[v * 8 + 2 * j + 1] * inv);
    reinterpret_cast<uint4*>(row)[v] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

}  // namespace idiff

extern "C" int idiff_vae_latent_in(const float* z, const float* w, const float* bias, float inv_scale, void* out,
                                   int batch, int channels, int hw, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(z && w && bias && out, "idiff_vae_latent_in: null pointer argument");
  IDIFF_REQUIRE(channels >= 1 && channels <= 8, "idiff_vae_latent_in: 1..8 latent channels supported (got %d)", channels);
  const long total = (long)batch * hw;
  const int blocks = (int)((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  vae_latent_in_kernel<<<blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(z, w, bias, inv_scale,
      reinterpret_cast<uint4*>(out), batch, channels, hw);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_softmax_rows(void* x, int rows, int n, long ld, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(x && rows > 0, "idiff_softmax_rows: bad arguments");
  IDIFF_REQUIRE(n > 0 && n % 8 == 0 && n <= 40960, "idiff_softmax_rows: n=%d must be a multiple of 8, <= 40960", n);
  IDIFF_REQUIRE(ld % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "idiff_softmax_rows: rows must be 16B aligned");
  const size_t smem = (size_t)n * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(softmax_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set = true;
  }
  softmax_rows_kernel<<<rows, 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<h16*>(x), n, ld);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}
