// Host-side helpers shared by the C-ABI translation units.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/vqa_b200.h"

namespace vqa {

int set_error(int code, const char* fmt, ...);   // records a thread-local message, returns code
int sm_count();                                   // SMs of the current device (cached per device)
// TMA descriptor of a bf16 matrix (gemm.cu): `inner` contiguous elements per row, `outer` rows of pitch ld elements,
// `batch` such matrices bstride elements apart; box = box_inner x box_outer (x 1).
int make_tmap(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_inner,
              uint32_t box_outer, uint64_t batch, uint64_t bstride,
              CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B);

#define VQA_CUDA_CHECK(expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) return ::vqa::set_error((int)_e, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define VQA_LAUNCH_CHECK(name)                                                                 \
  do {                                                                                         \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) return ::vqa::set_error((int)_e, "launch %s: %s", name, cudaGetErrorString(_e)); \
  } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

}  // namespace vqa
