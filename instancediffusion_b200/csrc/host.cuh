// Host-side helpers shared by the launchers: error reporting and TMA tensor-map encoding.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#ifndef IDIFF_STORAGE_BF16
#define IDIFF_STORAGE_BF16 0  // see common.cuh: 16-bit storage type of this build
#endif

namespace idiff {

int set_error(const char* fmt, ...);  // always returns -1

#define IDIFF_CHECK_CUDA(expr)                                                              \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess)                                                                  \
      return idiff::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),       \
                              __FILE__, __LINE__);                                          \
  } while (0)

#define IDIFF_REQUIRE(cond, ...)                       \
  do {                                                 \
    if (!(cond)) return idiff::set_error(__VA_ARGS__); \
  } while (0)

// Encode a tiled fp16 tensor map with 128B swizzle and zero OOB fill.
// dims/strides innermost-first; strides[i] (bytes) is the stride of dim i+1 (rank-1 entries).
int encode_tmap_f16(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                    const uint64_t* strides_bytes, const uint32_t* box);
// same with an explicit swizzle span (128 / 64 / 32 bytes, 0 = none)
int encode_tmap_f16_sw(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes, const uint32_t* box, int swizzle_bytes);

// 4-D view (d, head, token, batch) of a 16-bit [batch*rows, ld] matrix whose head h occupies
// columns [h*d, (h+1)*d) from `base`; boxes of 64 d x 1 head x box_rows tokens (the attention kernels).
int make_head_tmap(CUtensorMap* m, const void* base, int d, int heads, int rows, int batch, int ld, int box_rows);

}  // namespace idiff
