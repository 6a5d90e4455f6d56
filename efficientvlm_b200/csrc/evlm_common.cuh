// Shared device helpers for the evlm sm_100a kernels: PTX wrappers (mbarrier, TMA, tcgen05),
// bf16 packing, warp/block reductions and the counter-based dropout RNG.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#define EVLM_OK 0
#define EVLM_EINVAL (-1)      // bad argument / shape (maps to ValueError on the host side)
#define EVLM_EUNSUPPORTED (-2)

#define EVLM_CUDA_RETURN()                                   \
  do {                                                       \
    cudaError_t _e = cudaGetLastError();                     \
    return _e == cudaSuccess ? EVLM_OK : (int)_e;            \
  } while (0)

namespace evlm {

// ---------------------------------------------------------------------------------------------
// small math
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + __expf(-x)); }
// quick_gelu (CLIP): x * sigmoid(1.702 x)                      reference: eff_vit.py:210,218 (ACT2FN)
__device__ __forceinline__ float quick_gelu(float x) { return x * sigmoidf_(1.702f * x); }
__device__ __forceinline__ float quick_gelu_grad(float x) {
  float s = sigmoidf_(1.702f * x);
  return s + 1.702f * x * s * (1.f - s);
}
// erf GELU (BERT): 0.5 x (1 + erf(x / sqrt 2))                 reference: eff_bert.py:441 (ACT2FN['gelu'])
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_erf_grad(float x) {
  float cdf = 0.5f * (1.f + erff(x * 0.70710678118654752f));
  float pdf = 0.39894228040143268f * __expf(-0.5f * x * x);
  return cdf + x * pdf;
}

// ---- fast variants for the GEMM epilogues (outputs are rounded to bf16, so ~1e-6 absolute error is invisible) ----
__device__ __forceinline__ float fast_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float fast_ex2(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float fast_sigmoid(float x) { return fast_rcp(1.f + fast_ex2(-1.4426950408889634f * x)); }
// quick_gelu value and derivative from one sigmoid
__device__ __forceinline__ void fast_quick_gelu(float x, float& y, float& dy) {
  const float s = fast_rcp(1.f + fast_ex2(-2.4554669595930157f * x));   // sigmoid(1.702 x): the two constants folded into one multiply
  y = x * s;
  dy = s + 1.702f * y * (1.f - s);
}
// erf-GELU value and derivative sharing one exponential: erf via Abramowitz-Stegun 7.1.26 (|err| < 1.5e-7),
// gelu(x) = x Phi(x), gelu'(x) = Phi(x) + x phi(x), with exp(-x^2/2) used by both erf(x/sqrt2) and phi(x).
__device__ __forceinline__ void fast_gelu_erf(float x, float& y, float& dy) {
  const float ax = fabsf(x) * 0.70710678118654752f;
  const float ex = fast_ex2(-0.72134752044448170f * x * x);  // exp(-x^2 / 2)
  const float t = fast_rcp(1.f + 0.3275911f * ax);
  const float poly = t * (0.254829592f + t * (-0.284496736f + t * (1.421413741f + t * (-1.453152027f + t * 1.061405429f))));
  const float erf_abs = 1.f - poly * ex;
  const float cdf = 0.5f * (1.f + copysignf(erf_abs, x));
  y = x * cdf;
  dy = cdf + x * 0.39894228040143268f * ex;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// Block-wide sum; `red` must hold >= 32 floats of shared memory. All threads get the result.
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float t = (lane < nw) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;
}
__device__ __forceinline__ float block_max(float v, float* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  float t = (lane < nw) ? red[lane] : -INFINITY;
  t = warp_max(t);
  return t;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float2 unpack_bf16x2(uint32_t u) {
  __nv_bfloat162 v = *reinterpret_cast<__nv_bfloat162*>(&u);
  return __bfloat1622float2(v);
}
__device__ __forceinline__ float bf16_to_f(__nv_bfloat16 v) { return __bfloat162float(v); }

// ---------------------------------------------------------------------------------------------
// Counter-based RNG for dropout: Philox2x32-10 keyed by (seed), counter = (element index / 4, stream).
// The same (seed, stream, index) regenerates the same keep/drop decision in the backward pass, so
// no mask tensor is ever stored.
// ---------------------------------------------------------------------------------------------
// Optional device-resident seed offset (evlm_rng_bind): a captured CUDA graph bakes the by-value seeds of its
// launches in, so a replayed training step advances this one device word instead (evlm_rng_advance is itself a
// capturable launch) and every dropout site of the replay sees fresh, but forward/backward-consistent, seeds.
// One copy of the pointer per translation unit; evlm_rng_bind() sets them all.  Unbound = offset 0.
static __device__ const unsigned long long* g_rng_state = nullptr;
__device__ __forceinline__ uint64_t rng_offset() {
  const unsigned long long* p = g_rng_state;
  return p ? *p : 0ull;
}
static inline cudaError_t tu_rng_bind(const void* state_dev) {
  return cudaMemcpyToSymbol(g_rng_state, &state_dev, sizeof(state_dev));
}
// Dropout draws four 16-bit uniforms per counter from Philox2x32-10 (one 32x32 multiply per round: half the integer work of
// the 4x32 variant; 16 bits resolve the keep probability to 1.5e-5, far below what a dropout mask can express).
// counter = (idx4 low word, idx4 high word ^ stream hash), key = seed low ^ seed high rotated.
__device__ __forceinline__ uint2 philox2x32_10(uint2 ctr, uint32_t key) {
  const uint32_t M = 0xD256D193u, W = 0x9E3779B9u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi = __umulhi(M, ctr.x), lo = M * ctr.x;
    ctr = make_uint2(hi ^ key ^ ctr.y, lo);
    key += W;
  }
  return ctr;
}
__device__ __forceinline__ uint2 dropout_bits(uint64_t seed, uint32_t stream, uint64_t idx4) {
  const uint32_t key = (uint32_t)seed ^ __funnelshift_l((uint32_t)(seed >> 32), (uint32_t)(seed >> 32), 13) ^ 0x65766c6du;
  return philox2x32_10(make_uint2((uint32_t)idx4, (uint32_t)(idx4 >> 32) ^ (stream * 0x85EBCA6Bu + 0xC2B2AE35u)), key);
}
// 4 uniforms in [0,1) for elements idx4*4 .. idx4*4+3 (one Philox call).
__device__ __forceinline__ float4 dropout_uniform4(uint64_t seed, uint32_t stream, uint64_t idx4) {
  const uint2 r = dropout_bits(seed, stream, idx4);
  const float s = 1.0f / 65536.0f;
  return make_float4((float)(r.x & 0xFFFFu) * s, (float)(r.x >> 16) * s, (float)(r.y & 0xFFFFu) * s, (float)(r.y >> 16) * s);
}
// Uniform in [0,1) for element `idx` of dropout stream `stream` under `seed` (same value dropout_uniform4 gives that element).
__device__ __forceinline__ float dropout_uniform(uint64_t seed, uint32_t stream, uint64_t idx) {
  const uint2 r = dropout_bits(seed, stream, idx >> 2);
  const uint32_t w = (idx & 2) ? r.y : r.x;
  return (float)((idx & 1) ? (w >> 16) : (w & 0xFFFFu)) * (1.0f / 65536.0f);
}

// ---------------------------------------------------------------------------------------------
// PTX wrappers: shared-address conversion, mbarrier, TMA, tcgen05
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Wait with a watchdog: a pipeline bug traps (CUDA error on the host) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3fffu) == 0 && globaltimer_ns() - t0 > 4000000000ull) {  // 4 s
      printf("evlm: mbarrier watchdog (block %d thread %d bar %u parity %u)\n", blockIdx.x, threadIdx.x, bar, parity);
      __trap();
    }
  }
}

// 2-D TMA load global -> shared (tile mode), completion on an mbarrier. c0 = innermost coordinate.
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void* tmap, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(tmap), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tmap) : "memory");
}

// --- tcgen05 / TMEM ---
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 inputs, fp32 accumulate, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A * B with e4m3 inputs (kind::f8f6f4; the instruction descriptor carries the formats), fp32 accumulate.
__device__ __forceinline__ void umma_e4m3(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread have completed.
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// TMEM -> registers: this thread's lane (row), 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

}  // namespace evlm
