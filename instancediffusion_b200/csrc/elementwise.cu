// HBM-bound helpers of the sampling hot path (ScaleU lives in scaleu.cu): layout
// conversion, nearest-2x upsample, stride-2 im2col, UniFusion Fourier embedder, timestep
// embedding and the fused PLMS sampler update.  Reference citations are at each kernel.
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {


// ---------------------------------------------------------------------------------------------
// layout conversion
// ---------------------------------------------------------------------------------------------
__global__ void nchw_f32_to_nhwc_f16_kernel(const float* __restrict__ x, h16* __restrict__ y, int B,
                                            int C, int HW, int CP) {
  const long total = (long)B * HW * CP;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % CP);
    const long bp = i / CP;
    const int b = (int)(bp / HW);
    const int pix = (int)(bp - (long)b * HW);
    y[i] = (c < C) ? f2h(x[((long)b * C + c) * HW + pix]) : f2h(0.f);
  }
}
__global__ void nhwc_f16_to_nchw_f32_kernel(const h16* __restrict__ x, float* __restrict__ y, int B,
                                            int C, int HW) {
  __shared__ float tile[32][33];
  // grid: (HW/32, C/32, B)
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int pix = p0 + j, c = c0 + threadIdx.x;
    tile[j][threadIdx.x] = (pix < HW && c < C) ? h2f(x[((long)b * HW + pix) * C + c]) : 0.f;
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int c = c0 + j, pix = p0 + threadIdx.x;
    if (pix < HW && c < C) y[((long)b * C + c) * HW + pix] = tile[threadIdx.x][j];
  }
}

// F.interpolate(scale_factor=2, mode="nearest") (openaimodel.py:107), NHWC, 8 channels/thread
__global__ void upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int B, int H, int W,
                                  int CV) {
  const long total = (long)B * 4 * H * W * CV;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    long t = i / CV;
    const int ox = (int)(t % (2 * W));
    t /= (2 * W);
    const int oy = (int)(t % (2 * H));
    const int b = (int)(t / (2 * H));
    y[i] = x[(((long)b * H + (oy >> 1)) * W + (ox >> 1)) * CV + cv];
  }
}

// im2col for conv3x3 stride 2 pad 1 (openaimodel.py:130-134): out [B*Ho*Wo, 9*C]
// pad_lo = 1: padding 1 on every side (openaimodel.py:130-134); pad_lo = 0: the first-stage encoder's
// asymmetric F.pad (0,1,0,1) + stride-2 padding-0 convolution (diffusionmodules/model.py:70-74)
__global__ void im2col_s2_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int B, int H, int W,
                                 int CV, int pad_lo) {
  const int Ho = H >> 1, Wo = W >> 1;
  const long total = (long)B * Ho * Wo * 9 * CV;
  const uint4 zero = make_uint4(0, 0, 0, 0);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    long t = i / CV;
    const int tap = (int)(t % 9);
    t /= 9;
    const int ox = (int)(t % Wo);
    t /= Wo;
    const int oy = (int)(t % Ho);
    const int b = (int)(t / Ho);
    const int iy = 2 * oy - pad_lo + tap / 3, ix = 2 * ox - pad_lo + tap % 3;
    y[i] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? x[(((long)b * H + iy) * W + ix) * CV + cv] : zero;
  }
}

// ---------------------------------------------------------------------------------------------
// UniFusion Fourier embedder + null substitution + text concat
// (text_grounding_net.py:216-225, 248-276; util.py:12-26).  One block per (b, slot) row.
// ---------------------------------------------------------------------------------------------
__constant__ float c_freqs[16];

__global__ void __launch_bounds__(256)
fourier_embed_kernel(const float* __restrict__ coords, const float* __restrict__ masks,
                     const float* __restrict__ text, const float* __restrict__ null_text,
                     const float* __restrict__ null_pos, h16* __restrict__ out, int D,
                     int text_dim, int out_ld, int mask_mode, int dropped) {
  __shared__ float red[8];
  __shared__ float s_mpos;
  const int row = blockIdx.x;
  const float m = masks[row];
  const float* xr = coords + (long)row * D;
  float mpos;
  if (dropped) {
    mpos = 0.f;
  } else if (mask_mode == 0) {
    mpos = m;
  } else {
    float s = 0.f;
    for (int j = threadIdx.x; j < D; j += blockDim.x) s += xr[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
      s_mpos = ((t + m) > 0.f) ? 1.f : 0.f;
    }
    __syncthreads();
    mpos = s_mpos;
  }
  h16* orow = out + (long)row * out_ld;
  if (text) {
    for (int j = threadIdx.x; j < text_dim; j += blockDim.x)
      orow[j] = f2h(text[(long)row * text_dim + j] * m + (1.f - m) * null_text[j]);
  }
  const int E = 32 * D;
  for (int e = threadIdx.x; e < E; e += blockDim.x) {
    const int k = e / (2 * D);
    const int rem = e - k * 2 * D;
    const int is_cos = rem >= D;
    const int j = is_cos ? rem - D : rem;
    const float arg = c_freqs[k] * xr[j];
    const float val = is_cos ? cosf(arg) : sinf(arg);
    orow[text_dim + e] = f2h(val * mpos + (1.f - mpos) * null_pos[e]);
  }
}

// timestep_embedding (util.py:160-180): [cos(t f) | sin(t f)], f_k = exp(-ln(1e4) k / half)
__global__ void timestep_embedding_kernel(const float* __restrict__ t, h16* __restrict__ out, int B,
                                          int dim) {
  const int half_dim = dim >> 1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * half_dim) return;
  const int b = i / half_dim, k = i - b * half_dim;
  const float f = expf(-9.210340371976184f * (float)k / (float)half_dim);
  const float arg = t[b] * f;
  out[(long)b * dim + k] = f2h(cosf(arg));
  out[(long)b * dim + half_dim + k] = f2h(sinf(arg));
}

// ---------------------------------------------------------------------------------------------
// fused PLMS update (plms.py:121-165; plms_instance.py:166-210)
// ---------------------------------------------------------------------------------------------
__global__ void plms_update_kernel(const float* __restrict__ x, const float* __restrict__ e_c,
                                   const float* __restrict__ e_u, float gs, const float* __restrict__ o1,
                                   const float* __restrict__ o2, const float* __restrict__ o3, float c0,
                                   float c1, float c2, float c3, float sqrt_at, float sqrt_aprev,
                                   float sqrt_1m_at, float sqrt_1m_aprev, float* __restrict__ e_out,
                                   float* __restrict__ x_out, long n) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    float e = e_c[i];
    if (e_u) {
      const float u = e_u[i];
      e = u + gs * (e - u);
    }
    float ep = c0 * e;
    if (o1) ep += c1 * o1[i];
    if (o2) ep += c2 * o2[i];
    if (o3) ep += c3 * o3[i];
    const float pred_x0 = (x[i] - sqrt_1m_at * ep) / sqrt_at;
    const float xp = sqrt_aprev * pred_x0 + sqrt_1m_aprev * ep;
    if (e_out) e_out[i] = e;
    x_out[i] = xp;
  }
}

__global__ void latent_mean_kernel(const float* const* __restrict__ xs, int count, float* __restrict__ out,
                                   long n) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    float s = 0.f;
    for (int k = 0; k < count; ++k) s += xs[k][i];
    out[i] = s / (float)count;
  }
}

__global__ void silu_f16_kernel(const h16* __restrict__ x, h16* __restrict__ y, long n) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    y[i] = f2h(silu_f(h2f(x[i])));
}

static inline int grid_for(long total, int threads) {
  long g = (total + threads - 1) / threads;
  if (g > 148 * 16) g = 148 * 16;
  if (g < 1) g = 1;
  return (int)g;
}

// ---------------------------------------------------------------------------------------------
// instance-isolation attention mask (utils/input.py:34-37, attention.py:203-247)
// ---------------------------------------------------------------------------------------------
// one thread per (b, k, a, c) element of att_masks
__global__ void boxes_to_attmask_kernel(const float* __restrict__ boxes, const int* __restrict__ counts,
                                        float* __restrict__ att, int B, int K, int S) {
  const long total = (long)B * K * S * S;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % S);
    long t = i / S;
    const int a = (int)(t % S);
    t /= S;
    const int k = (int)(t % K);
    const int b = (int)(t / K);
    float v = 0.f;
    if (k < counts[b]) {
      const float* bx = boxes + ((long)b * K + k) * 4;
      // int(np.round(box * image_size)): round half to even, computed in double like numpy on python floats
      const int x1 = (int)rint((double)bx[0] * S), y1 = (int)rint((double)bx[1] * S);
      const int x2 = (int)rint((double)bx[2] * S), y2 = (int)rint((double)bx[3] * S);
      if (a >= x1 && a < x2 && c >= y1 && c < y2) v = 1.f;  // att_masks[idx][x1:x2, y1:y2] = 1 (x on the first axis)
    }
    att[i] = v;
  }
}

// one thread per (b, token): token < P visual, then 4*K object tokens, then `tail`
__global__ void attmask_words_kernel(const float* __restrict__ att, const int* __restrict__ active,
                                     uint32_t* __restrict__ mq, uint32_t* __restrict__ mk, int B, int K, int P, int tail) {
  const int NK = P + 4 * K + tail;
  const long total = (long)B * NK;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int b = (int)(i / NK);
    const int t = (int)(i - (long)b * NK);
    uint32_t w;
    if (!active[b]) {
      w = 0xffffffffu;
      if (t < P) mq[(long)b * P + t] = w;
    } else if (t < P) {
      w = 0;
      for (int k = 0; k < K; ++k)
        if (att[((long)b * K + k) * P + t] > 0.f) w |= 1u << k;
      mq[(long)b * P + t] = w | 0x80000000u;
    } else if (t < P + 4 * K) {
      const int g = (t - P) / K, k = (t - P) - g * K;
      w = (g == 0 || g == 3) ? (1u << k) : 0x80000000u;  // [box | point | scribble | mask]: only box and mask tokens are masked
    } else {
      w = 0x80000000u;
    }
    mk[i] = w;
  }
}

}  // namespace idiff

using namespace idiff;

extern "C" int idiff_nchw_f32_to_nhwc_f16(const float* x, void* y, int batch, int c, int hw, int c_pad,
                                          void* stream) {
  IDIFF_REQUIRE(x && y && c_pad >= c, "idiff_nchw_f32_to_nhwc_f16: bad arguments");
  const long total = (long)batch * hw * c_pad;
  nchw_f32_to_nhwc_f16_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x,
      reinterpret_cast<h16*>(y), batch, c, hw, c_pad);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_nhwc_f16_to_nchw_f32(const void* x, float* y, int batch, int c, int hw, void* stream) {
  IDIFF_REQUIRE(x && y, "idiff_nhwc_f16_to_nchw_f32: null pointer argument");
  dim3 grid((hw + 31) / 32, (c + 31) / 32, batch);
  nhwc_f16_to_nchw_f32_kernel<<<grid, dim3(32, 8), 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const h16*>(x),
      y, batch, c, hw);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_upsample_nearest2x(const void* x, void* y, int batch, int h, int w, int c, void* stream) {
  IDIFF_REQUIRE(x && y && c % 8 == 0, "idiff_upsample_nearest2x: bad arguments");
  const long total = (long)batch * 4 * h * w * (c / 8);
  upsample2x_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4*>(x),
      reinterpret_cast<uint4*>(y), batch, h, w, c / 8);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_im2col_s2(const void* x, void* y, int batch, int h, int w, int c, void* stream) {
  IDIFF_REQUIRE(x && y && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "idiff_im2col_s2: bad arguments");
  const long total = (long)batch * (h / 2) * (w / 2) * 9 * (c / 8);
  im2col_s2_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4*>(x),
      reinterpret_cast<uint4*>(y), batch, h, w, c / 8, 1);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_im2col_s2_pad01(const void* x, void* y, int batch, int h, int w, int c, void* stream) {
  IDIFF_REQUIRE(x && y && c % 8 == 0 && h % 2 == 0 && w % 2 == 0, "idiff_im2col_s2_pad01: bad arguments");
  const long total = (long)batch * (h / 2) * (w / 2) * 9 * (c / 8);
  im2col_s2_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const uint4*>(x),
      reinterpret_cast<uint4*>(y), batch, h, w, c / 8, 0);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_fourier_embed(const float* coords, const float* masks, const float* text,
                                   const float* null_text, const float* null_pos, void* out, int rows,
                                   int coord_dim, int text_dim, int out_ld, int mask_mode, int dropped,
                                   void* stream) {
  IDIFF_REQUIRE(coords && masks && null_pos && out, "idiff_fourier_embed: null pointer argument");
  IDIFF_REQUIRE(!text || null_text, "idiff_fourier_embed: text given without null_text");
  static bool freqs_set = false;
  if (!freqs_set) {
    float f[16];
    for (int k = 0; k < 16; ++k) f[k] = (float)pow(100.0, (double)k / 16.0);  // util.py:17
    IDIFF_CHECK_CUDA(cudaMemcpyToSymbol(c_freqs, f, sizeof(f)));
    freqs_set = true;
  }
  fourier_embed_kernel<<<rows, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(coords, masks, text, null_text,
      null_pos, reinterpret_cast<h16*>(out), coord_dim, text ? text_dim : 0, out_ld, mask_mode, dropped);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_timestep_embedding(const float* t, void* out, int batch, int dim, void* stream) {
  IDIFF_REQUIRE(t && out && dim % 2 == 0, "idiff_timestep_embedding: bad arguments");
  const int total = batch * dim / 2;
  timestep_embedding_kernel<<<(total + 127) / 128, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(t,
      reinterpret_cast<h16*>(out), batch, dim);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_plms_update(const float* x, const float* e_c, const float* e_u, float gs,
                                 const float* old1, const float* old2, const float* old3, float c0,
                                 float c1, float c2, float c3, float a_t, float a_prev,
                                 float sqrt_one_minus_at, float* e_out, float* x_out, long n, void* stream) {
  IDIFF_REQUIRE(x && e_c && x_out && n > 0, "idiff_plms_update: bad arguments");
  plms_update_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(x, e_c, e_u, gs, old1, old2,
      old3, c0, c1, c2, c3, sqrtf(a_t), sqrtf(a_prev), sqrt_one_minus_at, sqrtf(1.0f - a_prev), e_out, x_out, n);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_latent_mean(const float* const* xs_dev, int count, float* out, long n, void* stream) {
  IDIFF_REQUIRE(xs_dev && out && count > 0, "idiff_latent_mean: bad arguments");
  latent_mean_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(xs_dev, count, out, n);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_silu_f16(const void* x, void* y, long n, void* stream) {
  IDIFF_REQUIRE(x && y && n > 0, "idiff_silu_f16: bad arguments");
  silu_f16_kernel<<<grid_for(n, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const h16*>(x),
      reinterpret_cast<h16*>(y), n);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_boxes_to_attmask(const float* boxes, const int* counts, float* att_masks, int batch, int max_objs,
                                      int size, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(boxes && counts && att_masks && batch > 0 && max_objs > 0 && size > 0, "idiff_boxes_to_attmask: bad arguments");
  const long total = (long)batch * max_objs * size * size;
  boxes_to_attmask_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(boxes, counts,
      att_masks, batch, max_objs, size);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_attmask_words(const float* att_masks, const int* active, void* mask_q, void* mask_k, int batch,
                                   int n_objs, int pixels, int tail, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(att_masks && active && mask_q && mask_k, "idiff_attmask_words: null pointer argument");
  IDIFF_REQUIRE(n_objs > 0 && n_objs <= 30 && pixels > 0 && tail >= 0, "idiff_attmask_words: 1..30 instances supported (got %d)", n_objs);
  const long total = (long)batch * (pixels + 4 * n_objs + tail);
  attmask_words_kernel<<<grid_for(total, 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(att_masks, active,
      reinterpret_cast<uint32_t*>(mask_q), reinterpret_cast<uint32_t*>(mask_k), batch, n_objs, pixels, tail);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}
