// Error text + TMA descriptor encoding (driver entry point resolved at run time, so the
// library links against cudart only and loads on a GPU-less box).
#include "host.cuh"

#include <mutex>
#include <string.h>

#include "../../include/idiff_b200.h"

namespace idiff {

static thread_local char g_err[1024] = "";

int set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return -1;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, []() {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = (EncodeTiledFn)p;
  });
  return fn;
}

int encode_tmap_f16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box) {
  return encode_tmap_f16_sw(map, base, rank, dims, strides_bytes, box, 128);
}

int encode_tmap_f16_sw(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes) {
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                      : CU_TENSOR_MAP_SWIZZLE_NONE;
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return set_error("cuTensorMapEncodeTiled driver entry point unavailable (no CUDA driver?)");
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t bx[5];
  cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
  }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0)
    return set_error("tensor map base %p not 16-byte aligned", base);
  for (int i = 0; i + 1 < rank; ++i)
    if (gstr[i] % 16 != 0) return set_error("tensor map stride %d = %llu not a multiple of 16", i,
                                            (unsigned long long)gstr[i]);
  CUresult r = fn(map, IDIFF_STORAGE_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, const_cast<void*>(base),
                  gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    return set_error("cuTensorMapEncodeTiled failed: CUresult %d (rank %d dims %llu,%llu,%llu,%llu box %u,%u,%u,%u)",
                     (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                     (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
                     box[0], rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
  }
  return 0;
}

int make_head_tmap(CUtensorMap* m, const void* base, int d, int heads, int rows, int batch, int ld, int box_rows) {
  const uint64_t dims[4] = {(uint64_t)d, (uint64_t)heads, (uint64_t)rows, (uint64_t)batch};
  const uint64_t strides[3] = {(uint64_t)d * 2, (uint64_t)ld * 2, (uint64_t)rows * ld * 2};
  const uint32_t box[4] = {64u, 1u, (uint32_t)box_rows, 1u};
  return encode_tmap_f16(m, base, 4, dims, strides, box);
}

}  // namespace idiff

extern "C" const char* idiff_last_error(void) { return idiff::g_err; }
extern "C" int idiff_version(void) { return 2; }
extern "C" int idiff_storage_dtype(void) { return IDIFF_STORAGE_BF16 ? IDIFF_DTYPE_BF16 : IDIFF_DTYPE_F16; }
