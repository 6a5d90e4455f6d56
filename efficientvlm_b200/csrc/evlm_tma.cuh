// Host-side TMA tensor-map construction and the UMMA shared-memory descriptors shared by the tcgen05 kernels.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>
#include <cuda_runtime.h>
#include <mutex>
#include "evlm_common.cuh"

namespace evlm {

static inline PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  });
  return fn;
}

// 2-D bf16 tensor map over a row-major [rows, cols] matrix with leading dimension ld (elements);
// box = {64 cols (128 B, SWIZZLE_128B), box_rows}.
static inline int make_tmap_bf16(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) return (int)cudaErrorNotSupported;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : EVLM_EINVAL;
}

// 2-D e4m3 tensor map (UINT8: the TMA unit only moves bytes) over a row-major [rows, cols] matrix with a row pitch of ld bytes;
// box = {128 cols (128 B, SWIZZLE_128B), box_rows} — the byte geometry of the bf16 map above.  Columns >= cols are filled with 0.
static inline int make_tmap_e4m3(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) return (int)cudaErrorNotSupported;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld};
  cuuint32_t box[2] = {128u, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : EVLM_EINVAL;
}

// Tensor map for EPILOGUE STORES of a row-major [rows, cols] matrix (bf16 or fp32): box = {16 cols, 32 rows}, i.e. one
// epilogue warp's chunk; the 32-byte (bf16) / 64-byte (fp32) box rows are swizzled so that a thread writing its own row and
// the TMA engine reading the box are both bank-conflict free.  Needs a 16-byte aligned base and row pitch.
static inline int make_tmap_store(CUtensorMap* tm, const void* base, int64_t rows, int64_t cols, int64_t ld, bool is_f32) {
  auto fn = get_encode_fn();
  if (!fn) return (int)cudaErrorNotSupported;
  const int es = is_f32 ? 4 : 2;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * es};
  cuuint32_t box[2] = {16u, 32u};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = fn(tm, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, is_f32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B,
                  CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : EVLM_EINVAL;
}

// 3-D fp32 tensor map over the attention maps [items = B*H][Lq][ldp] for the forward's probability stores: box = {16 cols, box_rows, 1
// item}, SWIZZLE_64B like the GEMM epilogue's fp32 chunk stage.  The TMA unit clips rows >= Lq (a query tile never spills into the
// next head's map) and columns >= ldp.  Needs ldp % 4 == 0 and a 16-byte aligned base.
static inline int make_tmap_probs(CUtensorMap* tm, const void* base, int64_t ldp, int64_t Lq, int64_t items, int box_rows) {
  auto fn = get_encode_fn();
  if (!fn) return (int)cudaErrorNotSupported;
  cuuint64_t dims[3] = {(cuuint64_t)ldp, (cuuint64_t)Lq, (cuuint64_t)items};
  cuuint64_t strides[2] = {(cuuint64_t)ldp * 4, (cuuint64_t)ldp * 4 * (cuuint64_t)Lq};
  cuuint32_t box[3] = {16u, (cuuint32_t)box_rows, 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : EVLM_EINVAL;
}

static inline int device_num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// UMMA shared-memory descriptors for bf16 tiles in the 128B-swizzled canonical layouts (rows of 128 bytes, 8-row atoms):
//   K-major : tile = [MN rows][64 k];   SBO = 1024 B between 8-row groups; a K step of 16 elements = +32 B
//   MN-major: tile = [K rows][64 mn];   SBO = 1024 B between 8-row K groups, LBO = stride between 64-wide MN blocks;
//             a K step of 16 rows = +2048 B
__device__ __forceinline__ uint64_t make_desc_kmajor(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint64_t make_desc_mnmajor(uint32_t saddr, uint32_t lbo_bytes = 8192) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) |
         (2ull << 61);
}
// instruction descriptor: D = f32, A = B = bf16
__device__ __forceinline__ uint32_t make_idesc_bf16(int M, int N, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

}  // namespace evlm
