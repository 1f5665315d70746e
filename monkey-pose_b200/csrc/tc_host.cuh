// Host-side helpers for the tcgen05 kernels: TMA tensor-map encoding (through the driver entry
// point, so the library does not link libcuda directly) and operand packing conventions.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>

namespace hgru {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// Tensor map over a bf16 "chunked NHWC" operand [N][CG][H][W][8], viewed as 8-byte elements
// (dim0 = 2*W so one pixel-chunk of 16 B is two elements); box = (2*cols, rows, 2 chunks, 1).
// Out-of-bounds box elements are zero-filled: that implements the conv's SAME padding.
inline int make_act_tensor_map(CUtensorMap* map, const void* base, int N, int CG, int H, int W,
                               int box_cols, int box_rows, int box_chunks = 2) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return -1;
  cuuint64_t gdim[4] = {static_cast<cuuint64_t>(2 * W), static_cast<cuuint64_t>(H),
                        static_cast<cuuint64_t>(CG), static_cast<cuuint64_t>(N)};
  cuuint64_t gstr[3] = {static_cast<cuuint64_t>(W) * 16, static_cast<cuuint64_t>(H) * W * 16,
                        static_cast<cuuint64_t>(CG) * H * W * 16};
  cuuint32_t box[4] = {static_cast<cuuint32_t>(2 * box_cols), static_cast<cuuint32_t>(box_rows),
                       static_cast<cuuint32_t>(box_chunks), 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT64, 4, const_cast<void*>(base), gdim, gstr, box,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

// Tensor map over a K-major bf16 matrix [rows][K] (row pitch K*2 bytes, K % 8 == 0) with boxes of
// (64 K-elements = 128 bytes) x box_rows and the 128-byte swizzle: the canonical SW128 UMMA tile.
inline int make_kmajor_bf16_map(CUtensorMap* map, const void* base, size_t rows, size_t K, int box_rows) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return -1;
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstr[1] = {static_cast<cuuint64_t>(K) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

// Tensor map over a bf16 NHWC activation [N][H][W][C] (C % 64 == 0) for implicit-GEMM convolutions: box =
// (64 channels = 128 bytes) x box_w x box_h x box_n pixels with the 128-byte swizzle, so a box lands as box_w *
// box_h * box_n rows of a K-major SW128 UMMA tile in pixel order; out-of-image pixels are zero-filled (= SAME).
inline int make_nhwc_bf16_map(CUtensorMap* map, const void* base, int N, int H, int W, int C, int box_w, int box_h,
                              int box_n) {
  EncodeTiledFn enc = get_encode_tiled();
  if (!enc) return -1;
  cuuint64_t gdim[4] = {static_cast<cuuint64_t>(C), static_cast<cuuint64_t>(W), static_cast<cuuint64_t>(H),
                        static_cast<cuuint64_t>(N)};
  cuuint64_t gstr[3] = {static_cast<cuuint64_t>(C) * 2, static_cast<cuuint64_t>(W) * C * 2,
                        static_cast<cuuint64_t>(H) * W * C * 2};
  cuuint32_t box[4] = {64, static_cast<cuuint32_t>(box_w), static_cast<cuuint32_t>(box_h),
                       static_cast<cuuint32_t>(box_n)};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : static_cast<int>(r);
}

}  // namespace hgru
