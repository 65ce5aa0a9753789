// Host-side TMA tensor-map construction (cuTensorMapEncodeTiled resolved through the runtime's
// driver entry point, so the library links against cudart only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <stdexcept>
#include <string>

// Host code: a failing CUDA runtime call throws, naming the call and the line.
#define CUDA_OK(x)                                                                                   \
  do {                                                                                               \
    cudaError_t e_ = (x);                                                                            \
    if (e_ != cudaSuccess)                                                                           \
      throw std::runtime_error(std::string(#x) + ": " + cudaGetErrorString(e_) + " @" + std::to_string(__LINE__)); \
  } while (0)

namespace mmee {

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p)
      throw std::runtime_error("cuTensorMapEncodeTiled entry point not available");
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// 2-byte elements (bf16 / fp16), row-major [rows, cols] with row pitch `pitch_elems`;
// box = [box_rows, 64 cols] (128 B inner extent) with SWIZZLE_128B.  OOB elements read as zero.
inline CUtensorMap make_tmap_2d_sw128(const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                                      uint32_t box_rows, CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  CUtensorMap m;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode_fn()(&m, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
  return m;
}

// 1-byte elements, row-major [rows, cols] with row pitch `pitch_bytes` (multiple of 16); box = [box_rows, box_bytes]
// with box_bytes = 128 (SWIZZLE_128B) or 64 (SWIZZLE_64B).
inline CUtensorMap make_tmap_2d_u8(const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_bytes,
                                   uint32_t box_rows, uint32_t box_bytes) {
  CUtensorMap m;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {pitch_bytes};
  cuuint32_t box[2] = {box_bytes, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE,
                               box_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled(u8) failed: " + std::to_string((int)r));
  return m;
}

// 3-D variant: [d2][d1 rows][d0 cols], box = [1][box_rows][64].
inline CUtensorMap make_tmap_3d_sw128(const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t pitch1_elems,
                                      uint64_t pitch2_elems, uint32_t box_rows,
                                      CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  CUtensorMap m;
  cuuint64_t gdim[3] = {d0, d1, d2};
  cuuint64_t gstride[2] = {pitch1_elems * 2, pitch2_elems * 2};
  cuuint32_t box[3] = {64, box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = get_encode_fn()(&m, dt, 3, const_cast<void*>(base), gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw std::runtime_error("cuTensorMapEncodeTiled(3d) failed: " + std::to_string((int)r));
  return m;
}

}  // namespace mmee
