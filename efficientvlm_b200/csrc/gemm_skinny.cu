// evlm_gemm_bf16's small-M path: D[M <= 32, N] = epilogue(A[M,K] * B[N,K]^T) for the single-token decode steps of the caption / answer
// generators (model_generation.py:233-300: one new token per sequence and step, M = batch).
//
// Such a product is a WEIGHT STREAM: 2*N*K bytes of B against 2*M*K bytes of A, a few FLOP per byte.  The tcgen05 kernel would put a
// 128-row tile (3/4 of it padding) on N/128 CTAs — 6 of 148 SMs for a 768-wide projection, each pulling its whole weight slab through one
// TMA pipeline (10-17 us per launch in profiles/r02_launch_summary_caption.txt).  Here the weights are spread over the whole machine:
//   * a CTA (8 warps) owns 64 output columns and ONE K SLICE; the `ks` CTAs that share a column block form a thread-block cluster
//     (ks = 1, 2, 4 or 8, chosen so that about two CTAs per SM exist).  Splitting K rather than N keeps the activation re-read small:
//     a CTA reads 32 x K/ks activations for 64 x K/ks weights (an 8-column CTA over all of K would read four times more A than B);
//   * warp w owns columns 16 (w % 4) .. +15 and every second 32-wide k chunk of the slice: a lane loads 16 contiguous bytes of two weight
//     rows and of two / four activation rows straight into mma.sync.m16n8k16 fragments — the k order inside a chunk is permuted
//     identically for A and B (lane (g, t) holds k = 8t..8t+7; registers x,y feed the first k16 step, z,w the second), which a dot
//     product does not see; three chunks are in flight per warp;
//   * partial sums go to the CTA's shared memory; after a cluster barrier CTA r reduces columns 64 r / ks .. of ALL ks CTAs through
//     distributed shared memory, applies the forward epilogue of evlm_gemm_args (bias, q-scale, saved pre-activation, gate,
//     activation, residual) and stores bf16 or fp32.  No global workspace, no atomics, deterministic.
// Bound: HBM / L2 weight stream; no tensor-core ambition (mma.sync is only the cheapest way to do the 32 x 16 x 32 dot products).
//
// F8 (evlm_gemm_fp8): A and B are e4m3 with one scale per row of A and per row of B.  The byte geometry is unchanged — a lane's 16-byte
// load now holds 16 k-elements, a 64-byte chunk 64 — and mma.sync.m16n8k32.e4m3 takes the fragments in the same register pattern.  The
// reduced sum is multiplied by a_scale[m] * b_scale[n] before the epilogue.
#include "evlm_common.cuh"
#include "../../include/evlm.h"
#include <cooperative_groups.h>
#include <atomic>
#include <cstdlib>
#include <type_traits>

namespace evlm {
extern std::atomic<unsigned long long> g_launch_count;

constexpr int SK_WARPS = 8;
constexpr int SK_THREADS = SK_WARPS * 32;
constexpr int SK_UNROLL = 3;

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void mma_e4m3_16832(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k32.row.col.f32.e4m3.e4m3.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
template <bool F8>
__device__ __forceinline__ void mma_16(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  if constexpr (F8) mma_e4m3_16832(c, a0, a1, a2, a3, b0, b1);
  else mma_bf16_16816(c, a0, a1, a2, a3, b0, b1);
}

// The first r (1..15) bytes of a 16-byte group, the rest zero (e4m3: r elements).
__device__ __forceinline__ uint4 keep_first_bytes(uint4 v, const int r) {
  auto m = [r](int i) -> uint32_t {       // mask of word i (bytes 4 i .. 4 i + 3)
    const int n = r - 4 * i;
    return n >= 4 ? 0xffffffffu : n <= 0 ? 0u : (0xffffffffu >> (32 - 8 * n));
  };
  return make_uint4(v.x & m(0), v.y & m(1), v.z & m(2), v.w & m(3));
}
// The first r (1..7) bf16 elements of an 8-element group, the rest zero.
__device__ __forceinline__ uint4 keep_first_elems(uint4 v, const int r) {
  const uint32_t m0 = r >= 2 ? 0xffffffffu : 0x0000ffffu;
  const uint32_t m1 = r >= 4 ? 0xffffffffu : r == 3 ? 0x0000ffffu : 0u;
  const uint32_t m2 = r >= 6 ? 0xffffffffu : r == 5 ? 0x0000ffffu : 0u;
  const uint32_t m3 = r == 7 ? 0x0000ffffu : 0u;
  return make_uint4(v.x & m0, v.y & m1, v.z & m2, v.w & m3);
}
template <bool F8>
__device__ __forceinline__ uint4 keep_first(uint4 v, const int r) {
  if constexpr (F8) return keep_first_bytes(v, r);
  else return keep_first_elems(v, r);
}

template <int MB, bool F8>
__global__ void __launch_bounds__(SK_THREADS) gemm_skinny_kernel(const evlm_gemm_args g, const int ks, const int chunks_per_slice,
                                                                 const float* __restrict__ a_scale, const float* __restrict__ b_scale) {
  using T = typename std::conditional<F8, uint8_t, __nv_bfloat16>::type;
  constexpr int EL = 16 / sizeof(T);             // k-elements per 16-byte lane load (a chunk is 4 EL elements)
  namespace cg = cooperative_groups;
  constexpr int ROWS = MB * 16, COLS = 64, LDP = COLS + 2;
  __shared__ __align__(16) float part[2][ROWS][LDP];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int gq = lane >> 2, t = lane & 3;
  const int rank = blockIdx.x;                   // k slice == rank inside the cluster (cluster dims (ks, 1, 1), grid (ks, col blocks))
  const int n0 = blockIdx.y * COLS, nw = (warp & 3) * 16, khalf = warp >> 2;
  const T* A = reinterpret_cast<const T*>(g.A);
  const T* B = reinterpret_cast<const T*>(g.B);
  const int nchunks = (g.K + 4 * EL - 1) / (4 * EL);
  const int c_begin = rank * chunks_per_slice, c_end = min(nchunks, c_begin + chunks_per_slice);
  float acc[MB][2][4];
#pragma unroll
  for (int mb = 0; mb < MB; ++mb)
#pragma unroll
    for (int nb = 0; nb < 2; ++nb)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[mb][nb][j] = 0.f;
  // row pointers of this lane (nullptr: beyond M / N, contributes zeros)
  const T* arow[MB][2];
  const T* brow[2];
#pragma unroll
  for (int mb = 0; mb < MB; ++mb) {
    const int m = mb * 16 + gq;
    arow[mb][0] = m < g.M ? A + (int64_t)m * g.lda : nullptr;
    arow[mb][1] = m + 8 < g.M ? A + (int64_t)(m + 8) * g.lda : nullptr;
  }
#pragma unroll
  for (int nb = 0; nb < 2; ++nb) {
    const int n = n0 + nw + nb * 8 + gq;
    brow[nb] = n < g.N ? B + (int64_t)n * g.ldb : nullptr;
  }
  const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
  // The main loop takes the whole EL-element groups [0, K8); a partial last group (K % EL != 0) is added after it, masked in registers.
  const int K8 = g.K & ~(EL - 1);
  for (int c0 = c_begin + khalf; c0 < c_end; c0 += 2 * SK_UNROLL) {
    uint4 av[SK_UNROLL][MB][2], bv[SK_UNROLL][2];
#pragma unroll
    for (int u = 0; u < SK_UNROLL; ++u) {
      const int c = c0 + 2 * u;
      const int k = c * 4 * EL + t * EL;   // a lane's EL elements are all below K8 or all at / beyond it
      const bool kok = c < c_end && k < K8;
#pragma unroll
      for (int nb = 0; nb < 2; ++nb) bv[u][nb] = (kok && brow[nb]) ? __ldg(reinterpret_cast<const uint4*>(brow[nb] + k)) : zero4;
#pragma unroll
      for (int mb = 0; mb < MB; ++mb) {
        av[u][mb][0] = (kok && arow[mb][0]) ? __ldg(reinterpret_cast<const uint4*>(arow[mb][0] + k)) : zero4;
        av[u][mb][1] = (kok && arow[mb][1]) ? __ldg(reinterpret_cast<const uint4*>(arow[mb][1] + k)) : zero4;
      }
    }
#pragma unroll
    for (int u = 0; u < SK_UNROLL; ++u)
#pragma unroll
      for (int mb = 0; mb < MB; ++mb)
#pragma unroll
        for (int nb = 0; nb < 2; ++nb) {
          mma_16<F8>(acc[mb][nb], av[u][mb][0].x, av[u][mb][1].x, av[u][mb][0].y, av[u][mb][1].y, bv[u][nb].x, bv[u][nb].y);
          mma_16<F8>(acc[mb][nb], av[u][mb][0].z, av[u][mb][1].z, av[u][mb][0].w, av[u][mb][1].w, bv[u][nb].z, bv[u][nb].w);
        }
  }
  // Partial last group [K8, K): it sits in chunk ct at lane column tt, which belongs to this slice's warps of one k half.  The 16-byte
  // load stays inside the row's pitch (16-byte aligned base and pitch, checked by gemm_skinny_try); the elements at K and beyond are
  // zeroed in registers on both operands, so whatever the pitch padding holds (NaN included) never reaches the product.
  if (K8 != g.K) {
    const int ct = K8 / (4 * EL), tt = (K8 % (4 * EL)) / EL, r = g.K - K8;
    if (ct >= c_begin && ct < c_end && ((ct - c_begin) & 1) == khalf) {
      const bool mine = t == tt;
      uint4 at[MB][2], bt[2];
#pragma unroll
      for (int nb = 0; nb < 2; ++nb)
        bt[nb] = (mine && brow[nb]) ? keep_first<F8>(__ldg(reinterpret_cast<const uint4*>(brow[nb] + K8)), r) : zero4;
#pragma unroll
      for (int mb = 0; mb < MB; ++mb)
#pragma unroll
        for (int h = 0; h < 2; ++h)
          at[mb][h] = (mine && arow[mb][h]) ? keep_first<F8>(__ldg(reinterpret_cast<const uint4*>(arow[mb][h] + K8)), r) : zero4;
#pragma unroll
      for (int mb = 0; mb < MB; ++mb)
#pragma unroll
        for (int nb = 0; nb < 2; ++nb) {
          mma_16<F8>(acc[mb][nb], at[mb][0].x, at[mb][1].x, at[mb][0].y, at[mb][1].y, bt[nb].x, bt[nb].y);
          mma_16<F8>(acc[mb][nb], at[mb][0].z, at[mb][1].z, at[mb][0].w, at[mb][1].w, bt[nb].z, bt[nb].w);
        }
    }
  }
  // partial sums -> shared memory (accumulator fragment: c0,c1 = (row g, cols 2t, 2t+1); c2,c3 = (row g+8, same cols))
#pragma unroll
  for (int mb = 0; mb < MB; ++mb)
#pragma unroll
    for (int nb = 0; nb < 2; ++nb) {
      *reinterpret_cast<float2*>(&part[khalf][mb * 16 + gq][nw + nb * 8 + 2 * t]) = make_float2(acc[mb][nb][0], acc[mb][nb][1]);
      *reinterpret_cast<float2*>(&part[khalf][mb * 16 + gq + 8][nw + nb * 8 + 2 * t]) = make_float2(acc[mb][nb][2], acc[mb][nb][3]);
    }
  cg::cluster_group cluster = cg::this_cluster();
  if (ks > 1) cluster.sync();
  else __syncthreads();
  // CTA `rank` finishes columns [rank * cw, (rank + 1) * cw) of the block: sum over the ks slices (distributed shared memory), then the
  // forward epilogue of evlm_gemm_args, one thread per output element:
  //   v = acc (+bias); v *= alpha for n < alpha_cols; [aux_out = v]; gate(pre) -> act -> gate(post) -> (+ residual) -> D
  const int cw = COLS / ks;
  for (int e = threadIdx.x; e < ROWS * cw; e += SK_THREADS) {
    const int m = e / cw, cn = rank * cw + (e - m * cw), n = n0 + cn;
    if (m >= g.M || n >= g.N) continue;
    float v = 0.f;
    if (ks > 1) {
      for (int r = 0; r < ks; ++r) {
        const float* rp = cluster.map_shared_rank(&part[0][0][0], r);
        v += rp[m * LDP + cn] + rp[(ROWS + m) * LDP + cn];
      }
    } else {
      v = part[0][m][cn] + part[1][m][cn];
    }
    if constexpr (F8) v *= __ldg(a_scale + m) * __ldg(b_scale + n);
    if (g.bias) v += __ldg(g.bias + n);
    if (n < g.alpha_cols) v *= g.alpha;
    if (g.act != EVLM_ACT_NONE || g.gate_mode != EVLM_GATE_NONE) {
      if (g.aux_out) reinterpret_cast<__nv_bfloat16*>(g.aux_out)[(int64_t)m * g.ld_aux_out + n] = __float2bfloat16(v);
      const float z = g.gate_mode != EVLM_GATE_NONE ? __ldg(g.gate + n) : 1.f;
      float x = g.gate_mode == EVLM_GATE_PRE_ACT ? v * z : v, y, dy;
      if (g.act == EVLM_ACT_QUICK_GELU) fast_quick_gelu(x, y, dy);
      else if (g.act == EVLM_ACT_GELU_ERF) fast_gelu_erf(x, y, dy);
      else y = x;
      v = g.gate_mode == EVLM_GATE_POST_ACT ? y * z : y;
    }
    if (g.residual) {
      const int64_t ri = (int64_t)m * g.ldr + n;
      v += g.res_dtype == EVLM_F32 ? reinterpret_cast<const float*>(g.residual)[ri]
                                   : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(g.residual)[ri]);
    }
    const int64_t di = (int64_t)m * g.ldd + n;
    if (g.d_dtype == EVLM_F32) reinterpret_cast<float*>(g.D)[di] = v;
    else reinterpret_cast<__nv_bfloat16*>(g.D)[di] = __float2bfloat16(v);
  }
  if (ks > 1) cluster.sync();      // nobody leaves while its shared memory may still be read by a peer
}

// Returns -1 when the product is not a small-M forward one (the caller then runs the tcgen05 kernel), else the launch status.
// Any K >= 1 is taken; the kernel's 16-byte operand loads need 16-byte aligned bases and row pitches of A and B (ops.alloc16 and the
// weight shadows provide them), a partial last 16-byte group is masked in registers.  a_scale == nullptr: bf16 operands; else e4m3.
int gemm_skinny_try(const evlm_gemm_args* a, const float* a_scale, const float* b_scale, void* stream) {
  const bool f8 = a_scale != nullptr;
  const int esz = f8 ? 1 : 2;
  static const bool off = getenv("EVLM_GEMM_NO_SKINNY") != nullptr;   // profiling knob: every product on the tcgen05 kernel
  if (off || a->M > 32 || a->a_mn || a->b_mn || a->epi_mode != EVLM_EPI_FORWARD || a->splits > 1 || a->accumulate ||
      a->dropout_p > 0.f || a->m_limit || a->n_limit || a->k_limit || a->K < 1)
    return -1;
  if ((reinterpret_cast<uintptr_t>(a->A) & 15) || (reinterpret_cast<uintptr_t>(a->B) & 15) || ((a->lda * esz) & 15) || ((a->ldb * esz) & 15))
    return -1;
  const int col_blocks = (a->N + 63) / 64, nchunks = (a->K * esz + 63) / 64;
  int ks = 1;                                    // k slices per column block: about two CTAs per SM, at least 4 chunks per slice
  while (ks < 8 && col_blocks * ks < 2 * 148 && nchunks / (ks * 2) >= 4) ks *= 2;
  const int cps = (nchunks + ks - 1) / ks;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)ks, (unsigned)col_blocks, 1);
  cfg.blockDim = dim3(SK_THREADS, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = static_cast<cudaStream_t>(stream);
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (ks > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = (unsigned)ks;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  cudaError_t e;
  if (f8)
    e = a->M > 16 ? cudaLaunchKernelEx(&cfg, gemm_skinny_kernel<2, true>, *a, ks, cps, a_scale, b_scale)
                  : cudaLaunchKernelEx(&cfg, gemm_skinny_kernel<1, true>, *a, ks, cps, a_scale, b_scale);
  else
    e = a->M > 16 ? cudaLaunchKernelEx(&cfg, gemm_skinny_kernel<2, false>, *a, ks, cps, a_scale, b_scale)
                  : cudaLaunchKernelEx(&cfg, gemm_skinny_kernel<1, false>, *a, ks, cps, a_scale, b_scale);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  if (e != cudaSuccess) return (int)e;
  EVLM_CUDA_RETURN();
}

}  // namespace evlm
