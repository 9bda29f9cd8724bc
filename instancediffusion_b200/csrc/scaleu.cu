// ScaleU skip-connection rescale (openaimodel.py:519-539) with Fourier_filter (:25-48) in closed
// form -- HBM-bound, two passes, no FFT:
//   filter(x) = x + (s-1) * P_low(x),  P_low = Re IDFT of the bins (fy,fx) in {-1,0}^2
// Per (b,c) plane seven real sums are needed:
//   S0=sum x, Ac=sum x cos(tx), As=sum x sin(tx), Bc=sum x cos(py), Bs=sum x sin(py),
//   Cc=sum x cos(tx+py), Cs=sum x sin(tx+py),   tx=2*pi*x/W, py=2*pi*y/H
// and P_low(y,x) = (S0 + Ac cos tx + As sin tx + Bc cos py + Bs sin py
//                   + Cc cos(tx+py) + Cs sin(tx+py)) / (H*W).
// Pass 1 writes per-chunk partial sums (fixed summation order, no atomics: bit-reproducible);
// pass 2 writes the concatenated tensor [h * (tanh(b)+1) | filter(skip)] that the next ResBlock
// reads.  Thread mapping as in norm.cu: thread (r, cv) owns 16-byte vector cv of pixels r, r+k, ...
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {

constexpr float kTwoPiF = 6.283185307179586f;
constexpr int SU_MAX_CHUNKS = 32;

IDIFF_DEVICE void su_unpack8(const uint4& v, float (&f)[8]) {
  const uint32_t u[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float2 t = unpack_half2(u[j]);
    f[2 * j] = t.x;
    f[2 * j + 1] = t.y;
  }
}

// grid (chunks, B), block k*CV2; partial: [B][chunks][C2][8]
__global__ void __launch_bounds__(512)
scaleu_coef_kernel(const uint4* __restrict__ skip, float* __restrict__ partial, int H, int W, int C,
                   int pix_per_block, int k) {
  __shared__ float tab[4 * 128];  // cos tx, sin tx, cos py, sin py
  extern __shared__ float red[];  // [k][C][7]
  float* ctx = tab;
  float* stx = tab + 128;
  float* cpy = tab + 256;
  float* spy = tab + 384;
  for (int i = threadIdx.x; i < W; i += blockDim.x) sincosf(kTwoPiF * i / W, &stx[i], &ctx[i]);
  for (int i = threadIdx.x; i < H; i += blockDim.x) sincosf(kTwoPiF * i / H, &spy[i], &cpy[i]);
  __syncthreads();
  const int CV = C >> 3;
  const int r = threadIdx.x / CV;
  const int cv = threadIdx.x - r * CV;
  const int b = blockIdx.y;
  const int hw = H * W;
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(hw, p0 + pix_per_block);
  const uint4* xb = skip + (long)b * hw * CV + cv;
  float acc[7][8];
#pragma unroll
  for (int q = 0; q < 7; ++q)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[q][j] = 0.f;
  auto accumulate = [&](const uint4& v, int pix) {
    const int yy = pix / W, xx = pix - yy * W;
    const float cx = ctx[xx], sx = stx[xx], cy = cpy[yy], sy = spy[yy];
    const float wgt[7] = {1.f, cx, sx, cy, sy, cx * cy - sx * sy, sx * cy + cx * sy};
    float f[8];
    su_unpack8(v, f);
#pragma unroll
    for (int q = 0; q < 7; ++q)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[q][j] += f[j] * wgt[q];
  };
  int pix = p0 + r;
  for (; pix + k < p1; pix += 2 * k) {
    const uint4 v0 = xb[(long)pix * CV];
    const uint4 v1 = xb[(long)(pix + k) * CV];
    accumulate(v0, pix);
    accumulate(v1, pix + k);
  }
  for (; pix < p1; pix += k) accumulate(xb[(long)pix * CV], pix);
#pragma unroll
  for (int q = 0; q < 7; ++q)
#pragma unroll
    for (int j = 0; j < 8; ++j) red[((long)r * C + cv * 8 + j) * 7 + q] = acc[q][j];
  __syncthreads();
  // fixed-order reduction over the k pixel rows; one (channel, coefficient) per thread-iteration
  for (int i = threadIdx.x; i < C * 7; i += blockDim.x) {
    float a = 0.f;
    for (int rr = 0; rr < k; ++rr) a += red[(long)rr * C * 7 + i];
    const int c = i / 7, q = i - c * 7;
    partial[(((long)b * gridDim.x + blockIdx.x) * C + c) * 8 + q] = a;
  }
}

// partial [B][chunks][C][8] -> coef [B][C][8], fixed order (one thread per (b, c, q))
__global__ void __launch_bounds__(256)
scaleu_reduce_kernel(const float* __restrict__ partial, float* __restrict__ coef, int chunks, int C, int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C * 8) return;
  const int b = i / (C * 8);
  const int rem = i - b * C * 8;
  float a = 0.f;
  for (int ch = 0; ch < chunks; ++ch) a += partial[((long)b * chunks + ch) * C * 8 + rem];
  coef[i] = a;
}

// grid (chunks, B), block k*CVO, CVO = (C1+C2)/8
__global__ void __launch_bounds__(512)
scaleu_apply_kernel(const uint4* __restrict__ h, const uint4* __restrict__ skip, uint4* __restrict__ out,
                    const float* __restrict__ b1, const float* __restrict__ partial, float s_minus_1,
                    int H, int W, int C1, int C2, int pix_per_block, int k, int coef_chunks) {
  __shared__ float tab[4 * 128];
  float* ctx = tab;
  float* stx = tab + 128;
  float* cpy = tab + 256;
  float* spy = tab + 384;
  for (int i = threadIdx.x; i < W; i += blockDim.x) sincosf(kTwoPiF * i / W, &stx[i], &ctx[i]);
  for (int i = threadIdx.x; i < H; i += blockDim.x) sincosf(kTwoPiF * i / H, &spy[i], &cpy[i]);
  __syncthreads();
  const int CV1 = C1 >> 3, CV2 = C2 >> 3, CVO = CV1 + CV2;
  const int r = threadIdx.x / CVO;
  const int cv = threadIdx.x - r * CVO;
  const int b = blockIdx.y;
  const int hw = H * W;
  const int p0 = blockIdx.x * pix_per_block;
  const int p1 = min(hw, p0 + pix_per_block);
  const long obase = (long)b * hw * CVO + cv;
  if (cv < CV1) {
    float sc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) sc[j] = b1[cv * 8 + j];
    const uint4* hb = h + (long)b * hw * CV1 + cv;
    for (int pix = p0 + r; pix < p1; pix += k) {
      float f[8];
      su_unpack8(hb[(long)pix * CV1], f);
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = pack_half2(f[2 * j] * sc[2 * j], f[2 * j + 1] * sc[2 * j + 1]);
      out[obase + (long)pix * CVO] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  } else {
    const int cv2 = cv - CV1;
    const float scale = s_minus_1 / (float)hw;
    float cf[8][7];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int q = 0; q < 7; ++q) cf[j][q] = 0.f;
    for (int ch = 0; ch < coef_chunks; ++ch) {
      const float* src = partial + (((long)b * coef_chunks + ch) * C2 + cv2 * 8) * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 a = *reinterpret_cast<const float4*>(src + j * 8);
        const float4 c = *reinterpret_cast<const float4*>(src + j * 8 + 4);
        cf[j][0] += a.x; cf[j][1] += a.y; cf[j][2] += a.z; cf[j][3] += a.w;
        cf[j][4] += c.x; cf[j][5] += c.y; cf[j][6] += c.z;
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int q = 0; q < 7; ++q) cf[j][q] *= scale;
    const uint4* sb = skip + (long)b * hw * CV2 + cv2;
    for (int pix = p0 + r; pix < p1; pix += k) {
      const int yy = pix / W, xx = pix - yy * W;
      const float cx = ctx[xx], sx = stx[xx], cy = cpy[yy], sy = spy[yy];
      const float cxy = cx * cy - sx * sy, sxy = sx * cy + cx * sy;
      float f[8];
      su_unpack8(sb[(long)pix * CV2], f);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        f[j] += cf[j][0] + cf[j][1] * cx + cf[j][2] * sx + cf[j][3] * cy + cf[j][4] * sy + cf[j][5] * cxy +
                cf[j][6] * sxy;
      uint32_t o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = pack_half2(f[2 * j], f[2 * j + 1]);
      out[obase + (long)pix * CVO] = make_uint4(o[0], o[1], o[2], o[3]);
    }
  }
}

static void su_geometry(int batch, int hw, int cv, int max_chunks, int* k, int* ppb, int* chunks) {
  int kk = 256 / cv;  // (512-thread CTAs with half as many chunks measured slower, like the GroupNorm passes)
  if (kk < 1) kk = 1;
  if (kk > hw) kk = hw;
  int want = (148 * 3 + batch - 1) / batch;
  if (want > max_chunks) want = max_chunks;
  if (want < 1) want = 1;
  int p = (hw + want - 1) / want;
  p = ((p + kk - 1) / kk) * kk;
  if (p < kk) p = kk;
  *k = kk;
  *ppb = p;
  *chunks = (hw + p - 1) / p;
}

}  // namespace idiff

extern "C" long idiff_scaleu_ws_floats(int batch, int c2) {
  return (long)batch * (idiff::SU_MAX_CHUNKS + 1) * c2 * 8;  // per-chunk partials + the reduced coefficients
}

extern "C" int idiff_scaleu_concat(const void* h, const void* skip, void* out, const float* b1, float s,
                                   float* coef_ws, int batch, int height, int width, int c1, int c2,
                                   void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(h && skip && out && b1 && coef_ws, "idiff_scaleu_concat: null pointer argument");
  IDIFF_REQUIRE(c1 % 8 == 0 && c2 % 8 == 0, "idiff_scaleu_concat: channels must be multiples of 8");
  IDIFF_REQUIRE(height <= 128 && width <= 128, "idiff_scaleu_concat: H,W <= 128 supported");
  IDIFF_REQUIRE((c1 + c2) / 8 <= 512 && c2 / 8 <= 512, "idiff_scaleu_concat: too many channels");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int hw = height * width;
  int k1, ppb1, chunks1;
  su_geometry(batch, hw, c2 / 8, SU_MAX_CHUNKS, &k1, &ppb1, &chunks1);
  const size_t smem = (size_t)k1 * c2 * 7 * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(scaleu_coef_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    attr_set = true;
  }
  IDIFF_REQUIRE(smem <= 160 * 1024, "idiff_scaleu_concat: shared memory %zu too large", smem);
  scaleu_coef_kernel<<<dim3(chunks1, batch), k1 * (c2 / 8), smem, st>>>(reinterpret_cast<const uint4*>(skip), coef_ws,
      height, width, c2, ppb1, k1);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  float* coef = coef_ws + (long)batch * SU_MAX_CHUNKS * c2 * 8;
  scaleu_reduce_kernel<<<(batch * c2 * 8 + 255) / 256, 256, 0, st>>>(coef_ws, coef, chunks1, c2, batch);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  int k2, ppb2, chunks2;
  su_geometry(batch, hw, (c1 + c2) / 8, 4096, &k2, &ppb2, &chunks2);
  scaleu_apply_kernel<<<dim3(chunks2, batch), k2 * ((c1 + c2) / 8), 0, st>>>(reinterpret_cast<const uint4*>(h),
      reinterpret_cast<const uint4*>(skip), reinterpret_cast<uint4*>(out), b1, coef, s - 1.0f, height, width, c1, c2,
      ppb2, k2, 1);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}
