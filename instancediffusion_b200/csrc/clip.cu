// CLIP text-encoder pieces (SURVEY.md section 8f-3: the per-phrase pooled feature of utils/model.py:130-152 and the
// prompt context of ldm/modules/encoders/modules.py:144-172 -- both Hugging Face `CLIPTextModel`, transformers 4.27
// pinned by the reference's requirements.txt:247; architecture restated in oracle/torch_oracle.py: clip_text_forward).
//
// The encoder runs once per phrase / prompt, on 77 tokens: its linear layers go through idiff_gemm (QuickGELU as a
// SiLU epilogue on pre-scaled weights), its LayerNorms through idiff_layernorm.  What is left are two kernels no
// tensor core is needed for:
//   embed_tokens_kernel            token embedding gather + position embedding -> 16-bit rows
//   causal_attention_small_kernel  softmax(q k^T scale + causal mask) v for <= 128 tokens per sequence: one CTA per
//                                  (sequence, head), K / V of the head in shared memory (fp32), one thread per query
//                                  row with an online softmax in registers -- 1.5 MFLOP per (sequence, head) at
//                                  77 x 77 x 64, launch-latency-sized work
#include "../../include/idiff_b200.h"
#include "common.cuh"
#include "host.cuh"

namespace idiff {

__global__ void __launch_bounds__(128)
embed_tokens_kernel(const long long* __restrict__ ids, const uint4* __restrict__ tok, const uint4* __restrict__ pos,
                    uint4* __restrict__ out, int rows, int T, int vocab, int CV) {
  const int row = blockIdx.x;
  if (row >= rows) return;
  long long id = ids[row];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);  // (an id outside the table cannot be reported from here: clamped)
  const int t = row % T;
  for (int v = threadIdx.x; v < CV; v += blockDim.x) {
    const uint4 a = tok[(long)id * CV + v];
    const uint4 b = pos[(long)t * CV + v];
    const uint32_t au[4] = {a.x, a.y, a.z, a.w}, bu[4] = {b.x, b.y, b.z, b.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fa = unpack_half2(au[j]), fb = unpack_half2(bu[j]);
      o[j] = pack_half2(fa.x + fb.x, fa.y + fb.y);
    }
    out[(long)row * CV + v] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// q / k / v: 16-bit [batch * T, >= heads * D] with a common row stride `ld` (the fused QKV GEMM output);
// out [batch * T, heads * D] with row stride ld_out.  key_len (optional): keys at positions >= key_len[b] are masked
// (padding); the causal mask (key j visible to query i iff j <= i) always applies (modeling_clip: causal_attention_mask).
template <int D>
__global__ void __launch_bounds__(128)
causal_attention_small_kernel(const h16* __restrict__ q, const h16* __restrict__ k, const h16* __restrict__ v,
                              h16* __restrict__ out, const int* __restrict__ key_len, int ld, int ld_out, int T,
                              float scale_log2e) {
  extern __shared__ float cas_smem[];
  float* sK = cas_smem;                 // [T][D]
  float* sV = cas_smem + (size_t)T * D;  // [T][D]
  const int b = blockIdx.y, h = blockIdx.x;
  const int len = key_len ? min(key_len[b], T) : T;
  constexpr int VPR = D / 8;  // 16-byte vectors per row of one head
  for (int i = threadIdx.x; i < T * VPR; i += blockDim.x) {
    const int r = i / VPR, c = i - r * VPR;
    const long off = (long)(b * T + r) * ld + h * D + c * 8;
    const uint4 kv = *reinterpret_cast<const uint4*>(k + off);
    const uint4 vv = *reinterpret_cast<const uint4*>(v + off);
    const uint32_t ku[4] = {kv.x, kv.y, kv.z, kv.w}, vu[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 fk = unpack_half2(ku[j]), fv = unpack_half2(vu[j]);
      sK[r * D + c * 8 + 2 * j] = fk.x;
      sK[r * D + c * 8 + 2 * j + 1] = fk.y;
      sV[r * D + c * 8 + 2 * j] = fv.x;
      sV[r * D + c * 8 + 2 * j + 1] = fv.y;
    }
  }
  __syncthreads();
  const int i = threadIdx.x;  // query row
  if (i >= T) return;
  float qr[D], acc[D];
  {
    const h16* qrow = q + (long)(b * T + i) * ld + h * D;
#pragma unroll
    for (int c = 0; c < VPR; ++c) {
      const uint4 qv = *reinterpret_cast<const uint4*>(qrow + c * 8);
      const uint32_t qu[4] = {qv.x, qv.y, qv.z, qv.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_half2(qu[j]);
        qr[c * 8 + 2 * j] = f.x * scale_log2e;  // scores in the exp2 domain
        qr[c * 8 + 2 * j + 1] = f.y * scale_log2e;
      }
    }
  }
#pragma unroll
  for (int d = 0; d < D; ++d) acc[d] = 0.f;
  float m = -INFINITY, l = 0.f;
  const int last = min(i, len - 1);  // keys 0..last (the query's own position is always visible when len > i)
  for (int j = 0; j <= last; ++j) {
    const float* kr = sK + j * D;  // every thread of a warp reads the same row: shared-memory broadcast
    float s = 0.f;
#pragma unroll
    for (int d = 0; d < D; ++d) s = fmaf(qr[d], kr[d], s);
    const float m_new = fmaxf(m, s);
    const float alpha = exp2_approx(m - m_new);  // first key: 2^-inf = 0
    const float p = exp2_approx(s - m_new);
    l = fmaf(l, alpha, p);
    const float* vr = sV + j * D;
#pragma unroll
    for (int d = 0; d < D; ++d) acc[d] = fmaf(acc[d], alpha, p * vr[d]);
    m = m_new;
  }
  const float inv_l = l > 0.f ? 1.0f / l : 0.f;  // (len == 0: no visible key, zeros)
  h16* orow = out + (long)(b * T + i) * ld_out + h * D;
#pragma unroll
  for (int c = 0; c < VPR; ++c) {
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = pack_half2(acc[c * 8 + 2 * j] * inv_l, acc[c * 8 + 2 * j + 1] * inv_l);
    *reinterpret_cast<uint4*>(orow + c * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

}  // namespace idiff

extern "C" int idiff_embed_tokens(const long long* ids, const void* tok_table, const void* pos_table, void* out, int rows,
                                  int tokens_per_seq, int vocab, int channels, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(ids && tok_table && pos_table && out, "idiff_embed_tokens: null pointer argument");
  IDIFF_REQUIRE(rows > 0 && tokens_per_seq > 0 && vocab > 0 && channels > 0 && channels % 8 == 0 && rows % tokens_per_seq == 0,
                "idiff_embed_tokens: bad shape rows=%d tokens=%d vocab=%d C=%d (C %% 8 == 0, rows %% tokens == 0)", rows,
                tokens_per_seq, vocab, channels);
  embed_tokens_kernel<<<rows, 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(ids,
      reinterpret_cast<const uint4*>(tok_table), reinterpret_cast<const uint4*>(pos_table),
      reinterpret_cast<uint4*>(out), rows, tokens_per_seq, vocab, channels / 8);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int idiff_causal_attention_small(const void* q, const void* k, const void* v, void* out, const int* key_len,
                                            int ld_qkv, int ld_out, int batch, int tokens, int heads, int head_dim,
                                            float scale, void* stream) {
  using namespace idiff;
  IDIFF_REQUIRE(q && k && v && out, "idiff_causal_attention_small: null pointer argument");
  IDIFF_REQUIRE(batch > 0 && heads > 0 && tokens > 0 && tokens <= 128,
                "idiff_causal_attention_small: tokens=%d must be in 1..128 (one thread per query row)", tokens);
  IDIFF_REQUIRE(head_dim == 64, "idiff_causal_attention_small: head_dim %d not built (64: CLIP ViT-L/14 text)", head_dim);
  IDIFF_REQUIRE(ld_qkv % 8 == 0 && ld_out % 8 == 0 && ld_qkv >= heads * head_dim && ld_out >= heads * head_dim,
                "idiff_causal_attention_small: row strides must be multiples of 8 and cover heads * head_dim");
  IDIFF_REQUIRE(((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(k) | reinterpret_cast<uintptr_t>(v) |
                  reinterpret_cast<uintptr_t>(out)) & 15) == 0, "idiff_causal_attention_small: pointers must be 16-byte aligned");
  const size_t smem = (size_t)2 * tokens * head_dim * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    IDIFF_CHECK_CUDA(cudaFuncSetAttribute(causal_attention_small_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          2 * 128 * 64 * (int)sizeof(float)));
    attr_set = true;
  }
  causal_attention_small_kernel<64><<<dim3(heads, batch), 128, smem, reinterpret_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const h16*>(q),
      reinterpret_cast<const h16*>(k), reinterpret_cast<const h16*>(v), reinterpret_cast<h16*>(out), key_len, ld_qkv,
      ld_out, tokens, scale * 1.4426950408889634f);
  IDIFF_CHECK_CUDA(cudaGetLastError());
  return 0;
}
