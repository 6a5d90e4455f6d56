// evlm_quant_rows_e4m3: bf16 / fp32 rows -> e4m3 rows + one fp32 scale per row (include/evlm.h, ABI v9).
//
// The formula is fixed so that a host mirror reproduces it bit for bit (tests/test_fp8_host.py, tests/test_gpu_fp8.py):
//   amax = max |x|;  inv = 448 / amax (round-to-nearest division);  q = cvt.rn.satfinite.e4m3(x * inv);  scale = amax / 448
// torch: torch.clamp(x.float() * inv, -448, 448).to(torch.float8_e4m3fn) — the clamp stands in for satfinite (torch's cast gives NaN
// above 464).  A zero row gives q = 0 and scale = 0.
//
// One CTA per row, 8 elements per thread and pass: the row is read twice (the second pass hits L1 / L2), written once as 8-byte groups.
#include "evlm_common.cuh"
#include "../../include/evlm.h"
#include <atomic>

namespace evlm {
extern std::atomic<unsigned long long> g_launch_count;

constexpr int QR_THREADS = 128;

// two floats -> two e4m3 bytes (lo in the low byte), round to nearest even, saturating to +-448
__device__ __forceinline__ uint32_t cvt_e4m3x2(float lo, float hi) {
  uint16_t r;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(r) : "f"(hi), "f"(lo));
  return r;
}

// the 8 elements of group [k, k + 8) (zeros at and beyond `cols`)
template <typename T>
__device__ __forceinline__ void load8(const T* row, int64_t k, int64_t cols, bool vec, float (&v)[8]) {
  if (vec && k + 8 <= cols) {
    if constexpr (sizeof(T) == 2) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(row + k));
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = unpack_bf16x2(w[j]);
        v[2 * j] = f.x;
        v[2 * j + 1] = f.y;
      }
    } else {
      const float4 a = __ldg(reinterpret_cast<const float4*>(row + k)), b = __ldg(reinterpret_cast<const float4*>(row + k + 4));
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (k + j < cols) {
        if constexpr (sizeof(T) == 2) v[j] = __bfloat162float(row[k + j]);
        else v[j] = row[k + j];
      } else {
        v[j] = 0.f;
      }
    }
  }
}

template <typename T>
__global__ void __launch_bounds__(QR_THREADS) quant_rows_e4m3_kernel(const T* __restrict__ x, int64_t ldx, int64_t cols, uint8_t* __restrict__ q,
                                                                     int64_t ldq, float* __restrict__ scale) {
  __shared__ float red[32];
  const int64_t r = blockIdx.x;
  const T* row = x + r * ldx;
  uint8_t* qrow = q + r * ldq;
  const bool vec = (reinterpret_cast<uintptr_t>(row) & 15) == 0;   // any pitch: rows that start 16-byte aligned take vector loads
  float amax = 0.f;
  for (int64_t k = (int64_t)threadIdx.x * 8; k < cols; k += QR_THREADS * 8) {
    float v[8];
    load8<T>(row, k, cols, vec, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) amax = fmaxf(amax, fabsf(v[j]));
  }
  amax = block_max(amax, red);
  const float inv = amax > 0.f ? __fdiv_rn(448.f, amax) : 0.f;
  if (threadIdx.x == 0) scale[r] = amax > 0.f ? __fdiv_rn(amax, 448.f) : 0.f;
  // every 8-byte group of the padded row [0, ldq): the pad bytes become 0 (the loads give 0 beyond `cols`)
  for (int64_t k = (int64_t)threadIdx.x * 8; k < ldq; k += QR_THREADS * 8) {
    float v[8];
    load8<T>(row, k, cols, vec, v);
    uint32_t lo = cvt_e4m3x2(__fmul_rn(v[0], inv), __fmul_rn(v[1], inv)) | (cvt_e4m3x2(__fmul_rn(v[2], inv), __fmul_rn(v[3], inv)) << 16);
    uint32_t hi = cvt_e4m3x2(__fmul_rn(v[4], inv), __fmul_rn(v[5], inv)) | (cvt_e4m3x2(__fmul_rn(v[6], inv), __fmul_rn(v[7], inv)) << 16);
    *reinterpret_cast<uint2*>(qrow + k) = make_uint2(lo, hi);
  }
}

}  // namespace evlm

extern "C" int evlm_quant_rows_e4m3(const void* x, int32_t x_dtype, int64_t ldx, int64_t rows, int64_t cols, void* q, int64_t ldq, float* scale,
                                    void* stream) {
  using namespace evlm;
  if (!x || !q || !scale || rows <= 0 || cols <= 0 || ldx < cols || ldq < cols) return EVLM_EINVAL;
  if (x_dtype != EVLM_BF16 && x_dtype != EVLM_F32) return EVLM_EINVAL;
  if ((ldq % 16) || (reinterpret_cast<uintptr_t>(q) & 15) || rows > 0x7fffffff) return EVLM_EINVAL;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  uint8_t* qp = reinterpret_cast<uint8_t*>(q);
  if (x_dtype == EVLM_F32)
    quant_rows_e4m3_kernel<float><<<(unsigned)rows, QR_THREADS, 0, st>>>(reinterpret_cast<const float*>(x), ldx, cols, qp, ldq, scale);
  else
    quant_rows_e4m3_kernel<__nv_bfloat16><<<(unsigned)rows, QR_THREADS, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(x), ldx, cols, qp, ldq,
                                                                                 scale);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  EVLM_CUDA_RETURN();
}
