// evlm_gemm_bf16: persistent, warp-specialised bf16 GEMM on Blackwell tensor cores.
//
//   D[M,N] = epilogue( A[M,K] * B[N,K]^T )          A, B bf16; fp32 accumulation in TMEM.
//
// Design (sm_100a only):
//   * one CTA per SM (persistent), static round-robin over (tile, k-split) work items;
//   * warp 0 = TMA producer (cp.async.bulk.tensor, 128B-swizzled boxes, mbarrier complete_tx),
//     warp 1 = tcgen05.mma issuer (one elected lane; cta_group::1, UMMA 128 x BLOCK_N x 16),
//     warps 2..17 = epilogue: four warps per TMEM lane quadrant, each owning a quarter of the tile's columns
//     (tcgen05.ld 32x32b, fused bias / q-scale / gate / activation / dropout / residual, vector stores);
//     accumulators are double-buffered in TMEM so the epilogue of tile i overlaps the main loop of tile i+1;
//   * the epilogue flavour is a template parameter (linear / activation-forward / activation-backward) so the
//     plain GEMMs do not carry the activation code's registers;
//   * both operands may be K-major (row-major [rows, K]) or MN-major (row-major [K, rows]) — the
//     latter lets dgrad read W[N,K] and wgrad read dY[M,N] / X[M,K] in place, with no transposes:
//     the UMMA shared-memory descriptors carry the major-ness (instruction descriptor bits 15/16).
//
// Shared-memory operand layouts (bf16, SWIZZLE_128B, atoms of 8 rows x 128 B):
//   K-major  : one TMA box {64 k, ROWS}     -> [ROWS][64 k]; UMMA desc SBO = 1024 B, k-step = +32 B
//   MN-major : ROWS/64 boxes {64 mn, 64 k}  -> [ROWS/64][64 k][64 mn]; LBO = 8192 B (next 64-mn block),
//              SBO = 1024 B (next 8 k rows), k-step = +2048 B (16 k rows)
#include "evlm_common.cuh"
#include "evlm_tma.cuh"
#include "../../include/evlm.h"
#include <atomic>
#include <cstdlib>
#include <mutex>

namespace evlm {

std::atomic<unsigned long long> g_launch_count{0};
// gemm_skinny.cu: M <= 32 forward products (decode steps); a_scale != nullptr: e4m3 operands
int gemm_skinny_try(const evlm_gemm_args* a, const float* a_scale, const float* b_scale, void* stream);

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;                 // bf16: 64 elements = 128-byte rows (one SWIZZLE_128B atom)
constexpr int UMMA_K = 16;
// F8 (evlm_gemm_fp8, e4m3 operands): the same 128-byte rows hold 128 elements; a stage is four kind::f8f6f4 MMAs of K = 32, the
// descriptor advancing 32 B per step exactly as for bf16, so stage bytes, swizzle and descriptors are shared.
constexpr int BLOCK_K_F8 = 128;
constexpr int NUM_EPI_WARPS = 16;  // 16 warps: the epilogue is latency-bound per warp, thread-level parallelism hides it
constexpr int NUM_EPI_THREADS = NUM_EPI_WARPS * 32;
constexpr int NUM_THREADS = 64 + NUM_EPI_THREADS;
enum { EPI_LINEAR = 0, EPI_ACT_FWD = 1, EPI_ACT_BWD = 2 };

// DB ("double-buffered epilogue"): every epilogue warp owns TWO 2 KB chunk buffers.  Chunk c lives in buffer c & 1: its row-major
// side operand (fp32 residual / saved bf16 pre-activation) is brought in by a TMA box load issued one chunk earlier, the outputs are
// written over it in place and leave as TMA box stores that get a whole chunk to drain before the buffer is loaded again.  No side
// operand passes through the LSU or waits in registers.  The second buffer costs one mainloop stage.
template <int BLOCK_N, bool DB = false>
struct GemmCfg {
  static constexpr int kStages = DB ? ((BLOCK_N == 256) ? 3 : 5) : ((BLOCK_N == 256) ? 4 : 6);
  static constexpr int kABytes = BLOCK_M * BLOCK_K * 2;
  static constexpr int kBBytes = BLOCK_N * BLOCK_K * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kTmemCols = 2 * BLOCK_N;  // double-buffered accumulator (power of two: 256 / 512)
  static constexpr int kEpiStageBytes = NUM_EPI_WARPS * 32 * 16 * 4 * (DB ? 2 : 1);  // per-warp [32][16] fp32 chunk buffer(s)
  static constexpr int kColStageBytes = 2 * BLOCK_N * 4;              // bias | gate of the current tile's columns, per column quarter
  static constexpr int kBarBytes = 512;                               // pipeline + accumulator + 16 side-load barriers + TMEM pointer
  static constexpr int kSmemBytes = kStages * kStageBytes + kEpiStageBytes + kColStageBytes + kBarBytes;
};

struct GemmParams {
  CUtensorMap tma_a;
  CUtensorMap tma_b;
  CUtensorMap tma_d;      // epilogue stores of D   (valid when tma_d_ok)
  CUtensorMap tma_aux;    // epilogue stores of aux_out (valid when tma_aux_ok)
  CUtensorMap tma_side;   // DB epilogue: box loads of the side operand (residual, or aux_in for the activation backward)
  int tma_d_ok, tma_aux_ok;
  int side_kind;          // DB epilogue: 0 none, 1 fp32 box (2 KB), 2 bf16 box (1 KB)
  evlm_gemm_args g;
  int m_tiles, n_tiles, k_blocks, splits, kb_per_split;
  const float* a_scale;   // F8: [M] row scales of A
  const float* b_scale;   // F8: [N] row scales of B (output channels)
};

// value and derivative of the activation (fast formulations, see evlm_common.cuh)
__device__ __forceinline__ void act_both(int act, float x, float& y, float& dy) {
  if (act == EVLM_ACT_QUICK_GELU) fast_quick_gelu(x, y, dy);
  else if (act == EVLM_ACT_GELU_ERF) fast_gelu_erf(x, y, dy);
  else { y = x; dy = 1.f; }
}

// activation over one chunk with the (uniform) activation kind and gate position hoisted out of the element loop
template <int ACT>
__device__ __forceinline__ void act_one(float x, float& y, float& dy) {
  if constexpr (ACT == EVLM_ACT_QUICK_GELU) fast_quick_gelu(x, y, dy);
  else if constexpr (ACT == EVLM_ACT_GELU_ERF) fast_gelu_erf(x, y, dy);
  else { y = x; dy = 1.f; }
}
template <int ACT, int N>
__device__ __forceinline__ void act_fwd_chunk(float (&v)[N], const float (&z)[N], bool pre) {
  float dummy;
  if (pre) {               // y = act(z x)
#pragma unroll
    for (int j = 0; j < N; ++j) act_one<ACT>(v[j] * z[j], v[j], dummy);
  } else {                 // y = z act(x)
#pragma unroll
    for (int j = 0; j < N; ++j) {
      float y;
      act_one<ACT>(v[j], y, dummy);
      v[j] = y * z[j];
    }
  }
}
// v: dL/d(act output) in, dL/d(pre-activation) out;  u: saved pre-activation in, gate-gradient integrand out
template <int ACT, int N>
__device__ __forceinline__ void act_bwd_chunk(float (&v)[N], float (&u)[N], const float (&z)[N], bool pre) {
  if (pre) {               // y = act(z u): du = dg act'(zu) z ; dz-integrand = dg act'(zu) u
#pragma unroll
    for (int j = 0; j < N; ++j) {
      float y, d;
      act_one<ACT>(z[j] * u[j], y, d);
      const float t = v[j] * d;
      v[j] = t * z[j];
      u[j] = t * u[j];
    }
  } else {                 // y = z act(u): du = dg z act'(u) ; dz-integrand = dg act(u)
#pragma unroll
    for (int j = 0; j < N; ++j) {
      float y, d;
      act_one<ACT>(u[j], y, d);
      const float dg = v[j];
      v[j] = dg * z[j] * d;
      u[j] = dg * y;
    }
  }
}

// ---- epilogue I/O ------------------------------------------------------------------------------------------------
// tcgen05.ld 32x32b hands every thread ONE ROW of the accumulator (CH = 16 consecutive columns).  Reading / writing the
// row-major global operands (D, residual, aux_in, aux_out) straight from that layout makes each warp instruction touch
// 32 different rows (32 L1 wavefronts, half-used sectors).  So every row-major access goes through a per-warp shared
// memory stage [32 rows][16 fp32] instead: the row-owning thread reads/writes its row there, and the warp moves the
// stage to/from global memory with lane -> (row = 8 i + lane / 4, 4-column group = lane % 4): 64 contiguous bytes per
// row, fully used sectors, 4x fewer wavefronts.  The stage is XOR-swizzled per 16-byte group so both access patterns
// are bank-conflict free.
constexpr int CH = 16;
constexpr int STAGE_FLOATS = 32 * CH;
__device__ __forceinline__ float4* stage_at(float* st, int r, int grp) {
  return reinterpret_cast<float4*>(st + r * CH + ((grp ^ ((r >> 1) & 3)) << 2));
}
__device__ __forceinline__ void stage_put_row(float* st, int lane, const float (&v)[CH]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) *stage_at(st, lane, q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}
__device__ __forceinline__ void stage_get_row(float* st, int lane, float (&v)[CH]) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float4 x = *stage_at(st, lane, q);
    v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
  }
}
// Geometry of one 32-row x CH-column chunk as the coalesced phase sees it.
struct ChunkGeom {
  int row0;    // global row of stage row 0
  int col0;    // global column of stage column 0
  int rows;    // valid rows (<= 32)
  int ncols;   // valid columns (<= CH)
};
// Coalesced global -> registers (issued early; the values are parked in the stage later).  T = float or bf16.
template <typename T>
__device__ __forceinline__ void coalesced_load(const T* base, int64_t ld, const ChunkGeom& cg, int lane, bool vec_ok, float4 (&x)[4]) {
  const int grp = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i * 8 + (lane >> 2);
    x[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r >= cg.rows) continue;
    const T* sp = base + (int64_t)(cg.row0 + r) * ld + cg.col0 + grp * 4;
    if (vec_ok && grp * 4 + 4 <= cg.ncols) {
      if constexpr (sizeof(T) == 4) {
        x[i] = __ldg(reinterpret_cast<const float4*>(sp));
      } else {
        const uint2 q = __ldg(reinterpret_cast<const uint2*>(sp));
        const float2 a = unpack_bf16x2(q.x), b = unpack_bf16x2(q.y);
        x[i] = make_float4(a.x, a.y, b.x, b.y);
      }
    } else {
      float t0 = 0.f, t1 = 0.f, t2 = 0.f, t3 = 0.f;
      if constexpr (sizeof(T) == 4) {
        if (grp * 4 + 0 < cg.ncols) t0 = sp[0];
        if (grp * 4 + 1 < cg.ncols) t1 = sp[1];
        if (grp * 4 + 2 < cg.ncols) t2 = sp[2];
        if (grp * 4 + 3 < cg.ncols) t3 = sp[3];
      } else {
        if (grp * 4 + 0 < cg.ncols) t0 = __bfloat162float(sp[0]);
        if (grp * 4 + 1 < cg.ncols) t1 = __bfloat162float(sp[1]);
        if (grp * 4 + 2 < cg.ncols) t2 = __bfloat162float(sp[2]);
        if (grp * 4 + 3 < cg.ncols) t3 = __bfloat162float(sp[3]);
      }
      x[i] = make_float4(t0, t1, t2, t3);
    }
  }
}
// registers (coalesced layout) -> stage -> this thread's row
__device__ __forceinline__ void stage_in(float* st, int lane, const float4 (&x)[4], float (&v)[CH]) {
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) *stage_at(st, i * 8 + (lane >> 2), lane & 3) = x[i];
  __syncwarp();
  stage_get_row(st, lane, v);
}
template <typename T>
__device__ __forceinline__ void store_elem(T* dp, float t, bool add) {
  if constexpr (sizeof(T) == 4) {
    if (add) atomicAdd(dp, t);
    else *dp = t;
  } else {
    *dp = __float2bfloat16(t);
  }
}
// this thread's row -> stage -> coalesced global store (or fp32 reduction when `add`).  T = float or bf16.
template <typename T>
__device__ __forceinline__ void stage_out(float* st, int lane, const float (&v)[CH], T* base, int64_t ld, const ChunkGeom& cg, bool vec_ok,
                                          bool add) {
  __syncwarp();
  stage_put_row(st, lane, v);
  __syncwarp();
  const int grp = lane & 3;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int r = i * 8 + (lane >> 2);
    if (r >= cg.rows) continue;
    const float4 x = *stage_at(st, r, grp);
    T* dp = base + (int64_t)(cg.row0 + r) * ld + cg.col0 + grp * 4;
    if (vec_ok && grp * 4 + 4 <= cg.ncols) {
      if constexpr (sizeof(T) == 4) {
        if (add)
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dp), "f"(x.x), "f"(x.y), "f"(x.z), "f"(x.w) : "memory");
        else
          *reinterpret_cast<float4*>(dp) = x;
      } else {
        *reinterpret_cast<uint2*>(dp) = make_uint2(pack_bf16x2(x.x, x.y), pack_bf16x2(x.z, x.w));
      }
    } else {
      if (grp * 4 + 0 < cg.ncols) store_elem(dp + 0, x.x, add);
      if (grp * 4 + 1 < cg.ncols) store_elem(dp + 1, x.y, add);
      if (grp * 4 + 2 < cg.ncols) store_elem(dp + 2, x.z, add);
      if (grp * 4 + 3 < cg.ncols) store_elem(dp + 3, x.w, add);
    }
  }
}
// ---- TMA epilogue stores: the row-owning thread parks its row in the warp's stage in the tensor map's swizzled box layout
// (fp32: [32][64 B] SWIZZLE_64B = stage_at(); bf16: [32][32 B] SWIZZLE_32B), one lane issues a bulk tensor store of the
// [32 x 16] box.  No read-back through shared memory, no per-lane global stores, no bounds predicates (the TMA unit clips
// rows >= M and columns >= N), and the L1 sees 1/4 of the staged path's traffic.
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_box(const CUtensorMap* tm, uint32_t saddr, int col0, int row0, bool add) {
  if (add)
    asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(tm)),
                 "r"(saddr), "r"(col0), "r"(row0)
                 : "memory");
  else
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(tm)), "r"(saddr),
                 "r"(col0), "r"(row0)
                 : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// fp32 box: whole 2 KB stage.  bf16 box: 1 KB at byte offset `boff` (0 or 1024) of the stage.
__device__ __forceinline__ void stage_out_tma_f32(float* st, int lane, const float (&v)[CH], const CUtensorMap* tm, const ChunkGeom& cg, bool add) {
  stage_put_row(st, lane, v);
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) tma_store_box(tm, smem_u32(st), cg.col0, cg.row0, add);
}
__device__ __forceinline__ void stage_out_tma_bf16(float* st, int boff, int lane, const float (&v)[CH], const CUtensorMap* tm,
                                                   const ChunkGeom& cg) {
  uint8_t* base = reinterpret_cast<uint8_t*>(st) + boff;
  uint8_t* row = base + lane * 32;
  const int sw = (lane >> 2) & 1;
  *reinterpret_cast<uint4*>(row + ((0 ^ sw) << 4)) =
      make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  *reinterpret_cast<uint4*>(row + ((1 ^ sw) << 4)) =
      make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) tma_store_box(tm, smem_u32(base), cg.col0, cg.row0, false);
}

// 16-byte (fp32) / 8-byte (bf16) vector access is legal for every (row, 4-column group) of a tensor iff base and row
// pitch are multiples of it (chunk columns start at multiples of 16).
template <typename T>
__device__ __forceinline__ bool vec_ok_for(const T* base, int64_t ld) {
  return ((reinterpret_cast<uintptr_t>(base) | (uintptr_t)(ld * (int64_t)sizeof(T))) & (4 * sizeof(T) - 1)) == 0;
}
// per-column vector from global memory: every lane reads the same addresses (broadcast)
__device__ __forceinline__ void load_cols_f32(const float* sp, float (&u)[CH], int ncols) {
  if (ncols == CH && ((reinterpret_cast<uintptr_t>(sp) & 15) == 0)) {
#pragma unroll
    for (int j = 0; j < CH; j += 4) {
      float4 q = __ldg(reinterpret_cast<const float4*>(sp + j));
      u[j] = q.x; u[j + 1] = q.y; u[j + 2] = q.z; u[j + 3] = q.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < CH; ++j) u[j] = j < ncols ? sp[j] : 0.f;
  }
}
// per-column vectors (bias, gate) from the tile's shared-memory copy: every lane reads the same addresses (broadcast)
__device__ __forceinline__ void load_cols_smem(const float* sp, float (&u)[CH]) {
#pragma unroll
  for (int j = 0; j < CH; j += 4) {
    const float4 q = *reinterpret_cast<const float4*>(sp + j);
    u[j] = q.x; u[j + 1] = q.y; u[j + 2] = q.z; u[j + 3] = q.w;
  }
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// (acc_zero: a k-limited work item with no k-blocks at all — the accumulator was never written and stands for 0)
__device__ __forceinline__ void tmem_load_chunk(uint32_t taddr, float (&v)[CH], bool acc_zero = false) {
  if (acc_zero) {
#pragma unroll
    for (int j = 0; j < CH; ++j) v[j] = 0.f;
    return;
  }
  uint32_t r[CH];
  tmem_ld_32x32b_x16(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < CH; ++j) v[j] = __uint_as_float(r[j]);
}

// F8: the accumulator of e4m3 products times a_scale[row] * b_scale[col], before anything else of the epilogue
template <bool F8>
__device__ __forceinline__ void apply_f8_scales(const GemmParams& p, int row, const ChunkGeom& cg, float (&v)[CH]) {
  if constexpr (F8) {
    const float sa = row < p.g.M ? __ldg(p.a_scale + row) : 0.f;
    const float* sp = p.b_scale + cg.col0;
    if (cg.ncols == CH) {   // (col0 is a multiple of 16 and the scale vector is allocated 16-byte aligned)
#pragma unroll
      for (int j = 0; j < CH; j += 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(sp + j));
        v[j] *= sa * q.x; v[j + 1] *= sa * q.y; v[j + 2] *= sa * q.z; v[j + 3] *= sa * q.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < CH; ++j) v[j] *= sa * (j < cg.ncols ? sp[j] : 0.f);
    }
  }
}

// One 32-row x CH-column chunk through the epilogue; `row` is this thread's row, `cg` the chunk as a whole.
template <int EPI, bool F8>
__device__ __forceinline__ void epilogue_chunk(const GemmParams& p, uint32_t taddr, float* st, const float* bias_s, const float* gate_s,
                                               int lane, int row, const ChunkGeom& cg, int split, bool add, float keep_scale, bool acc_zero) {
  const evlm_gemm_args& g = p.g;
  const int col0 = cg.col0, ncols = cg.ncols;
  if (p.tma_d_ok | p.tma_aux_ok) {   // the previous chunk's bulk stores have finished reading this warp's stage
    if (lane == 0) tma_store_wait_read();
    __syncwarp();
  }
  float v[CH];
  if constexpr (EPI != EPI_ACT_BWD) {
    // the residual tile is requested before the accumulator is read so that its latency hides behind the math
    const bool has_res = g.residual != nullptr && split == 0;
    float4 pre[4];
    if (has_res) {
      if (g.res_dtype == EVLM_F32) {
        const float* rp = reinterpret_cast<const float*>(g.residual);
        coalesced_load<float>(rp, g.ldr, cg, lane, vec_ok_for(rp, g.ldr), pre);
      } else {
        const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(g.residual);
        coalesced_load<__nv_bfloat16>(rp, g.ldr, cg, lane, vec_ok_for(rp, g.ldr), pre);
      }
    }
    if constexpr (EPI == EPI_LINEAR) {
      // plain GEMMs: no column stage (its two barriers per tile cost more than the bias load they would hide)
      tmem_load_chunk(taddr, v, acc_zero);
      apply_f8_scales<F8>(p, row, cg, v);
      if (g.bias != nullptr && split == 0) {
        float b[CH];
        load_cols_f32(g.bias + col0, b, ncols);
#pragma unroll
        for (int j = 0; j < CH; ++j) v[j] += b[j];
      }
    } else {
      tmem_load_chunk(taddr, v, acc_zero);
      apply_f8_scales<F8>(p, row, cg, v);
      float b[CH];   // zeros when there is no bias
      load_cols_smem(bias_s, b);
#pragma unroll
      for (int j = 0; j < CH; ++j) v[j] += b[j];
    }
    if (g.alpha_cols > 0) {
#pragma unroll
      for (int j = 0; j < CH; ++j)
        if (col0 + j < g.alpha_cols) v[j] *= g.alpha;
    }
    if constexpr (EPI == EPI_ACT_FWD) {
      if (g.aux_out != nullptr) {
        __nv_bfloat16* ap = reinterpret_cast<__nv_bfloat16*>(g.aux_out);
        if (p.tma_aux_ok) stage_out_tma_bf16(st, 0, lane, v, &p.tma_aux, cg);
        else stage_out<__nv_bfloat16>(st, lane, v, ap, g.ld_aux_out, cg, vec_ok_for(ap, g.ld_aux_out), false);
      }
      float z[CH];   // ones when there is no gate
      load_cols_smem(gate_s, z);
      const bool pre = g.gate_mode == EVLM_GATE_PRE_ACT;
      if (g.act == EVLM_ACT_QUICK_GELU) act_fwd_chunk<EVLM_ACT_QUICK_GELU>(v, z, pre);
      else if (g.act == EVLM_ACT_GELU_ERF) act_fwd_chunk<EVLM_ACT_GELU_ERF>(v, z, pre);
      else act_fwd_chunk<EVLM_ACT_NONE>(v, z, pre);
    }
    if (g.dropout_p > 0.f) {
      // dropout stream element index = row * N + col
      const uint64_t seed = g.dropout_seed + rng_offset();
      const uint64_t e0 = (uint64_t)row * (uint64_t)g.N + (uint64_t)col0;
      if ((e0 & 3) == 0) {
#pragma unroll
        for (int j = 0; j < CH; j += 4) {
          float4 u = dropout_uniform4(seed, g.dropout_stream, (e0 + j) >> 2);
          v[j] = u.x >= g.dropout_p ? v[j] * keep_scale : 0.f;
          v[j + 1] = u.y >= g.dropout_p ? v[j + 1] * keep_scale : 0.f;
          v[j + 2] = u.z >= g.dropout_p ? v[j + 2] * keep_scale : 0.f;
          v[j + 3] = u.w >= g.dropout_p ? v[j + 3] * keep_scale : 0.f;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CH; ++j) {
          float u = dropout_uniform(seed, g.dropout_stream, e0 + j);
          v[j] = u >= g.dropout_p ? v[j] * keep_scale : 0.f;
        }
      }
    }
    if (has_res) {
      float q[CH];
      if (EPI == EPI_ACT_FWD && p.tma_aux_ok && g.aux_out != nullptr) {   // the aux box issued above still occupies the stage
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
      }
      stage_in(st, lane, pre, q);
#pragma unroll
      for (int j = 0; j < CH; ++j) v[j] += q[j];
    }
  } else {  // EPI_ACT_BWD: acc = dL/d(act output); aux_in = saved pre-activation u
    float u[CH], z[CH];
    {
      const __nv_bfloat16* ip = reinterpret_cast<const __nv_bfloat16*>(g.aux_in);
      float4 pre[4];
      coalesced_load<__nv_bfloat16>(ip, g.ld_aux_in, cg, lane, vec_ok_for(ip, g.ld_aux_in), pre);
      tmem_load_chunk(taddr, v, acc_zero);
      stage_in(st, lane, pre, u);
    }
    load_cols_smem(gate_s, z);
    const bool want_e = g.aux_out != nullptr;
    const bool pre = g.gate_mode == EVLM_GATE_PRE_ACT;
    if (g.act == EVLM_ACT_QUICK_GELU) act_bwd_chunk<EVLM_ACT_QUICK_GELU>(v, u, z, pre);
    else if (g.act == EVLM_ACT_GELU_ERF) act_bwd_chunk<EVLM_ACT_GELU_ERF>(v, u, z, pre);
    else act_bwd_chunk<EVLM_ACT_NONE>(v, u, z, pre);
    if (want_e) {
      __nv_bfloat16* ap = reinterpret_cast<__nv_bfloat16*>(g.aux_out);
      if (p.tma_aux_ok) stage_out_tma_bf16(st, 0, lane, u, &p.tma_aux, cg);
      else stage_out<__nv_bfloat16>(st, lane, u, ap, g.ld_aux_out, cg, vec_ok_for(ap, g.ld_aux_out), false);
    }
  }
  if (g.d_dtype == EVLM_F32) {
    float* dp = reinterpret_cast<float*>(g.D);
    if (p.tma_d_ok) {
      if (p.tma_aux_ok && g.aux_out != nullptr) {   // (not a combination the host side issues: the aux box still occupies the stage)
        if (lane == 0) tma_store_wait_read();
        __syncwarp();
      }
      stage_out_tma_f32(st, lane, v, &p.tma_d, cg, add);
    } else {
      stage_out<float>(st, lane, v, dp, g.ldd, cg, vec_ok_for(dp, g.ldd), add);
    }
  } else {
    __nv_bfloat16* dp = reinterpret_cast<__nv_bfloat16*>(g.D);
    if (p.tma_d_ok) stage_out_tma_bf16(st, 1024, lane, v, &p.tma_d, cg);
    else stage_out<__nv_bfloat16>(st, lane, v, dp, g.ldd, cg, vec_ok_for(dp, g.ldd), false);
  }
}

// ---- double-buffered epilogue (GemmCfg<.., DB = true>) -------------------------------------------------------------------------
template <int N>
__device__ __forceinline__ void tma_store_wait_read_n() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// bf16 [32][32 B] SWIZZLE_32B box: this thread's row (16 values)
__device__ __forceinline__ void box_get_row_bf16(const uint8_t* base, int lane, float (&v)[CH]) {
  const uint8_t* row = base + lane * 32;
  const int sw = (lane >> 2) & 1;
  const uint4 a = *reinterpret_cast<const uint4*>(row + ((0 ^ sw) << 4));
  const uint4 b = *reinterpret_cast<const uint4*>(row + ((1 ^ sw) << 4));
  const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float2 f = unpack_bf16x2(w[j]);
    v[2 * j] = f.x;
    v[2 * j + 1] = f.y;
  }
}
__device__ __forceinline__ void box_put_row_bf16(uint8_t* base, int lane, const float (&v)[CH]) {
  uint8_t* row = base + lane * 32;
  const int sw = (lane >> 2) & 1;
  *reinterpret_cast<uint4*>(row + ((0 ^ sw) << 4)) =
      make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  *reinterpret_cast<uint4*>(row + ((1 ^ sw) << 4)) =
      make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
}
// One chunk.  `buf` holds this chunk's side operand (when has_side) and receives its outputs; `nbuf` is the other buffer: the
// previous chunk's stores are drained from it and the NEXT chunk's side operand is requested into it before anything else happens,
// so that load has this whole chunk to land.
template <int EPI, bool F8>
__device__ __forceinline__ void epilogue_chunk_db(const GemmParams& p, uint32_t taddr, uint8_t* buf, uint8_t* nbuf, const float* bias_s,
                                                  const float* gate_s, int lane, int row, const ChunkGeom& cg, int split, bool add,
                                                  float keep_scale, bool has_side, uint32_t side_bar, uint32_t side_phase, uint32_t next_bar,
                                                  bool next_side, int next_col0, int next_row0, bool acc_zero) {
  const evlm_gemm_args& g = p.g;
  const int col0 = cg.col0, ncols = cg.ncols;
  const bool two_groups = g.aux_out != nullptr;      // (D box) + (aux box) bulk groups per chunk
  if (lane == 0) {
    if (p.side_kind != 0) {
      tma_store_wait_read_n<0>();                    // the previous chunk's boxes have left `nbuf`
      if (next_side) {
        mbar_expect_tx(next_bar, p.side_kind == 1 ? 2048u : 1024u);
        tma_load_2d(smem_u32(nbuf), &p.tma_side, next_col0, next_row0, next_bar);
      }
    } else if (two_groups) {
      tma_store_wait_read_n<2>();                    // the chunk before the previous one has left `buf`
    } else {
      tma_store_wait_read_n<1>();
    }
  }
  __syncwarp();
  float v[CH];
  if constexpr (EPI != EPI_ACT_BWD) {
    float q[CH];
    if (has_side) {
      mbar_wait(side_bar, side_phase);
      if (p.side_kind == 1) stage_get_row(reinterpret_cast<float*>(buf), lane, q);
      else box_get_row_bf16(buf, lane, q);
    }
    tmem_load_chunk(taddr, v, acc_zero);
    apply_f8_scales<F8>(p, row, cg, v);
    if constexpr (EPI == EPI_LINEAR) {
      if (g.bias != nullptr && split == 0) {
        float b[CH];
        load_cols_f32(g.bias + col0, b, ncols);
#pragma unroll
        for (int j = 0; j < CH; ++j) v[j] += b[j];
      }
    } else {
      float b[CH];   // zeros when there is no bias
      load_cols_smem(bias_s, b);
#pragma unroll
      for (int j = 0; j < CH; ++j) v[j] += b[j];
    }
    if (g.alpha_cols > 0) {
#pragma unroll
      for (int j = 0; j < CH; ++j)
        if (col0 + j < g.alpha_cols) v[j] *= g.alpha;
    }
    if (has_side) __syncwarp();                      // every lane has taken its side row: the buffer may be overwritten
    if constexpr (EPI == EPI_ACT_FWD) {
      if (g.aux_out != nullptr) box_put_row_bf16(buf, lane, v);       // saved pre-activation, bytes [0, 1 KB)
      float z[CH];   // ones when there is no gate
      load_cols_smem(gate_s, z);
      const bool pre = g.gate_mode == EVLM_GATE_PRE_ACT;
      if (g.act == EVLM_ACT_QUICK_GELU) act_fwd_chunk<EVLM_ACT_QUICK_GELU>(v, z, pre);
      else if (g.act == EVLM_ACT_GELU_ERF) act_fwd_chunk<EVLM_ACT_GELU_ERF>(v, z, pre);
      else act_fwd_chunk<EVLM_ACT_NONE>(v, z, pre);
    }
    if (g.dropout_p > 0.f) {
      const uint64_t seed = g.dropout_seed + rng_offset();
      const uint64_t e0 = (uint64_t)row * (uint64_t)g.N + (uint64_t)col0;
      if ((e0 & 3) == 0) {
#pragma unroll
        for (int j = 0; j < CH; j += 4) {
          float4 u = dropout_uniform4(seed, g.dropout_stream, (e0 + j) >> 2);
          v[j] = u.x >= g.dropout_p ? v[j] * keep_scale : 0.f;
          v[j + 1] = u.y >= g.dropout_p ? v[j + 1] * keep_scale : 0.f;
          v[j + 2] = u.z >= g.dropout_p ? v[j + 2] * keep_scale : 0.f;
          v[j + 3] = u.w >= g.dropout_p ? v[j + 3] * keep_scale : 0.f;
        }
      } else {
#pragma unroll
        for (int j = 0; j < CH; ++j) {
          float u = dropout_uniform(seed, g.dropout_stream, e0 + j);
          v[j] = u >= g.dropout_p ? v[j] * keep_scale : 0.f;
        }
      }
    }
    if (has_side) {
#pragma unroll
      for (int j = 0; j < CH; ++j) v[j] += q[j];
    }
    if (g.d_dtype == EVLM_F32) stage_put_row(reinterpret_cast<float*>(buf), lane, v);
    else box_put_row_bf16(buf + 1024, lane, v);
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      if (EPI == EPI_ACT_FWD && g.aux_out != nullptr) tma_store_box(&p.tma_aux, smem_u32(buf), cg.col0, cg.row0, false);
      tma_store_box(&p.tma_d, smem_u32(buf) + (g.d_dtype == EVLM_F32 ? 0u : 1024u), cg.col0, cg.row0, add);
    }
  } else {  // EPI_ACT_BWD: acc = dL/d(act output); side = saved pre-activation u (bf16 box, always present)
    float u[CH], z[CH];
    mbar_wait(side_bar, side_phase);
    box_get_row_bf16(buf, lane, u);
    tmem_load_chunk(taddr, v, acc_zero);
    load_cols_smem(gate_s, z);
    const bool pre = g.gate_mode == EVLM_GATE_PRE_ACT;
    if (g.act == EVLM_ACT_QUICK_GELU) act_bwd_chunk<EVLM_ACT_QUICK_GELU>(v, u, z, pre);
    else if (g.act == EVLM_ACT_GELU_ERF) act_bwd_chunk<EVLM_ACT_GELU_ERF>(v, u, z, pre);
    else act_bwd_chunk<EVLM_ACT_NONE>(v, u, z, pre);
    __syncwarp();                                    // (rows are private, but keep the in-place overwrite behind every lane's read)
    if (g.aux_out != nullptr) box_put_row_bf16(buf, lane, u);          // gate-gradient integrand, bytes [0, 1 KB)
    if (g.d_dtype == EVLM_F32) {
      // (an fp32 D box needs the whole buffer: the host side never combines it with aux_out in DB mode)
      stage_put_row(reinterpret_cast<float*>(buf), lane, v);
    } else {
      box_put_row_bf16(buf + 1024, lane, v);
    }
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      if (g.aux_out != nullptr) tma_store_box(&p.tma_aux, smem_u32(buf), cg.col0, cg.row0, false);
      tma_store_box(&p.tma_d, smem_u32(buf) + (g.d_dtype == EVLM_F32 ? 0u : 1024u), cg.col0, cg.row0, add);
    }
  }
}

template <int BLOCK_N, bool A_MN, bool B_MN, int EPI, bool DB, bool F8>
__global__ void __launch_bounds__(NUM_THREADS, 1) gemm_tcgen05_kernel(const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg<BLOCK_N, DB>;
  constexpr int BK = F8 ? BLOCK_K_F8 : BLOCK_K;   // elements per k block (128 bytes per operand row either way)
  extern __shared__ __align__(1024) uint8_t smem_raw[];   // SWIZZLE_128B operand tiles need 1024-byte alignment
  const uint32_t smem_base = smem_u32(smem_raw);
  if ((smem_base & 1023u) != 0) __trap();
  uint8_t* smem_aligned = smem_raw;
  float* epi_stage = reinterpret_cast<float*>(smem_aligned + Cfg::kStages * Cfg::kStageBytes);
  float* col_stage = epi_stage + Cfg::kEpiStageBytes / 4;
  const uint32_t bar_off = Cfg::kStages * Cfg::kStageBytes + Cfg::kEpiStageBytes + Cfg::kColStageBytes;
  const uint32_t bar_base = smem_base + bar_off;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::kStages + s); };
  auto tfull_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + s); };
  auto tempty_bar = [&](int s) { return bar_base + 8u * (2 * Cfg::kStages + 2 + s); };
  auto side_bar_of = [&](int epi_warp) { return bar_base + 8u * (2 * Cfg::kStages + 4 + 2 * epi_warp); };   // DB: one per chunk buffer
  volatile uint32_t* tmem_ptr_smem =
      reinterpret_cast<volatile uint32_t*>(smem_aligned + bar_off + 8 * (2 * Cfg::kStages + 4 + 2 * NUM_EPI_WARPS));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const evlm_gemm_args& g = p.g;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tma_a);
    tma_prefetch_desc(&p.tma_b);
    if (p.tma_d_ok) tma_prefetch_desc(&p.tma_d);
    if (p.tma_aux_ok) tma_prefetch_desc(&p.tma_aux);
    if (DB && p.side_kind != 0) tma_prefetch_desc(&p.tma_side);
    if (DB)
      for (int s = 0; s < NUM_EPI_WARPS; ++s) { mbar_init(side_bar_of(s), 1); mbar_init(side_bar_of(s) + 8, 1); }
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(tfull_bar(s), 1);
      mbar_init(tempty_bar(s), NUM_EPI_THREADS);
    }
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(smem_u32((const void*)tmem_ptr_smem), Cfg::kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  // zero-skip: device-side limits shrink the tile grid / the k loop (all roles derive the same schedule from the same scalars)
  int m_tiles_e = p.m_tiles, n_tiles_e = p.n_tiles, k_blocks_e = p.k_blocks, kbps_e = p.kb_per_split;
  if (g.m_limit) m_tiles_e = min(m_tiles_e, (max(0, __ldg(g.m_limit)) + BLOCK_M - 1) / BLOCK_M);
  if (g.n_limit) n_tiles_e = min(n_tiles_e, (max(0, __ldg(g.n_limit)) + BLOCK_N - 1) / BLOCK_N);
  if (g.k_limit) {
    k_blocks_e = min(k_blocks_e, (max(0, __ldg(g.k_limit)) + BK - 1) / BK);
    kbps_e = (k_blocks_e + p.splits - 1) / p.splits;
  }
  const int total_work = m_tiles_e * n_tiles_e * p.splits;
  const int kb_per_split = kbps_e;
  const int k_blocks_eff = k_blocks_e;
  const int n_tiles_eff = n_tiles_e;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        const int split = w % p.splits;
        const int t = w / p.splits;
        const int n0 = (t % n_tiles_eff) * BLOCK_N;
        const int m0 = (t / n_tiles_eff) * BLOCK_M;
        const int kb0 = split * kb_per_split;
        const int kb1 = min(k_blocks_eff, kb0 + kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(empty_bar(s), ph ^ 1);
          const uint32_t sa = smem_base + s * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
          mbar_expect_tx(full_bar(s), Cfg::kStageBytes);
          const int k0 = kb * BK;
          if (!A_MN) {
            tma_load_2d(sa, &p.tma_a, k0, m0, full_bar(s));
          } else {
#pragma unroll
            for (int i = 0; i < BLOCK_M / 64; ++i) tma_load_2d(sa + i * 8192, &p.tma_a, m0 + 64 * i, k0, full_bar(s));
          }
          if (!B_MN) {
            tma_load_2d(sb, &p.tma_b, k0, n0, full_bar(s));
          } else {
#pragma unroll
            for (int i = 0; i < BLOCK_N / 64; ++i) tma_load_2d(sb + i * 8192, &p.tma_b, n0 + 64 * i, k0, full_bar(s));
          }
          if (++s == Cfg::kStages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      // instruction descriptor: D=f32, A=B=bf16, majors, N>>3, M>>4
      // (F8, kind::f8f6f4: bits 7-9 / 10-12 = A / B format, E4M3 = 0; the other fields are laid out as for kind::f16)
      const uint32_t idesc = (1u << 4) | (F8 ? 0u : (1u << 7) | (1u << 10)) | ((A_MN ? 1u : 0u) << 15) | ((B_MN ? 1u : 0u) << 16) |
                             ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(BLOCK_M >> 4) << 24);
      int s = 0;
      uint32_t ph = 0;
      int as = 0;
      uint32_t aph = 0;
      for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
        const int split = w % p.splits;
        const int kb0 = split * kb_per_split;
        const int kb1 = min(k_blocks_eff, kb0 + kb_per_split);
        mbar_wait(tempty_bar(as), aph ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(as * BLOCK_N);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t sa = smem_base + s * Cfg::kStageBytes;
          const uint32_t sb = sa + Cfg::kABytes;
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = A_MN ? make_desc_mnmajor(sa + k * 2048) : make_desc_kmajor(sa + k * 32);
            const uint64_t bdesc = B_MN ? make_desc_mnmajor(sb + k * 2048) : make_desc_kmajor(sb + k * 32);
            if constexpr (F8) umma_e4m3(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            else umma_bf16(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(empty_bar(s));  // frees the smem stage once these MMAs have read it
          if (++s == Cfg::kStages) { s = 0; ph ^= 1; }
        }
        umma_commit(tfull_bar(as));  // accumulator complete
        if (++as == 2) { as = 0; aph ^= 1; }
      }
    }
  } else {
    // ============ epilogue (warps 2..17): quadrant = warp % 4, column quarter = (warp - 2) / 4 ============
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    const int part = (warp - 2) >> 2;
    float* st = epi_stage + (warp - 2) * STAGE_FLOATS;
    // Per-column operands (bias, gate) of this warp's column quarter live in shared memory for the duration of a tile:
    // the 128 threads of the quarter fetch one value each for the NEXT tile while the current one is processed, so the
    // chunk loop never waits on a global load for them (the streaming stores keep evicting them from L1).
    constexpr int CPP = BLOCK_N / 4;                 // columns per quarter
    float* cv = col_stage + part * 2 * CPP;          // [bias CPP | gate CPP]
    const int tq = quad * 32 + lane;                 // thread index within the quarter
    auto fetch_col = [&](int w) -> float {
      const int split = w % p.splits;
      const int n0 = ((w / p.splits) % n_tiles_eff) * BLOCK_N;
      const int col = n0 + part * CPP + (tq % CPP);
      if (tq < CPP) return (EPI != EPI_ACT_BWD && g.bias != nullptr && split == 0 && col < g.N) ? __ldg(g.bias + col) : 0.f;
      if (tq < 2 * CPP) return (EPI != EPI_LINEAR && g.gate_mode != EVLM_GATE_NONE && col < g.N) ? __ldg(g.gate + col) : 1.f;
      return 0.f;
    };
    float col_next = (EPI != EPI_LINEAR && (int)blockIdx.x < total_work) ? fetch_col(blockIdx.x) : 0.f;
    int as = 0;
    uint32_t aph = 0;
    const bool add = p.splits > 1 || g.accumulate;
    const float keep_scale = g.dropout_p > 0.f ? 1.f / (1.f - g.dropout_p) : 1.f;
    // DB: the chunks this warp processes form one sequence across tiles; chunk i uses buffer i & 1 and, while it is processed,
    // the side operand of chunk i + 1 (possibly the first chunk of the warp's next tile) is already on its way.
    uint8_t* dbuf = reinterpret_cast<uint8_t*>(epi_stage) + (warp - 2) * 4096;
    const uint32_t side_bar = side_bar_of(warp - 2);   // + 8 * buffer
    uint32_t side_uses[2] = {0u, 0u};                   // side loads consumed from each buffer so far (parity = barrier phase)
    int cb = 0;
    // geometry of chunk number `ci` (0 .. CPP/CH-1) of work item `w` for THIS warp; false when it does not exist
    auto chunk_geom = [&](int w, int ci, ChunkGeom& o, int& split_o) -> bool {
      if (w >= total_work || ci >= CPP / CH) return false;
      const int t = w / p.splits;
      o.row0 = (t / n_tiles_eff) * BLOCK_M + quad * 32;
      o.rows = min(32, g.M - o.row0);
      o.col0 = (t % n_tiles_eff) * BLOCK_N + part * CPP + ci * CH;
      o.ncols = min(CH, g.N - o.col0);
      split_o = w % p.splits;
      return o.rows > 0 && o.ncols > 0;
    };
    auto side_wanted = [&](int split) -> bool { return p.side_kind != 0 && (EPI == EPI_ACT_BWD || split == 0); };
    // the chunk after (w, ci) in this warp's sequence
    auto next_chunk = [&](int& w, int& ci, ChunkGeom& o, int& split_o) -> bool {
      for (;;) {
        if (++ci >= CPP / CH) { ci = 0; w += gridDim.x; }
        if (w >= total_work) return false;
        if (chunk_geom(w, ci, o, split_o)) return true;
        if (o.rows <= 0) { ci = CPP / CH; }      // the whole tile is beyond M for this warp: skip it
        else if (o.ncols <= 0) { ci = CPP / CH; }
      }
    };
    if constexpr (DB) {
      // prologue: request the side operand of the warp's very first chunk
      int sp0 = 0;
      ChunkGeom g0;
      if (p.side_kind != 0) {
        int wi = blockIdx.x, ci = -1;
        // (ci = -1, so next_chunk() starts the search at chunk 0 of the first work item)
        if (wi < total_work && next_chunk(wi, ci, g0, sp0) && side_wanted(sp0) && lane == 0) {
          mbar_expect_tx(side_bar, p.side_kind == 1 ? 2048u : 1024u);
          tma_load_2d(smem_u32(dbuf), &p.tma_side, g0.col0, g0.row0, side_bar);
        }
      }
    }
    for (int w = blockIdx.x; w < total_work; w += gridDim.x) {
      const int t = w / p.splits;
      const int n0 = (t % n_tiles_eff) * BLOCK_N;
      const int m0 = (t / n_tiles_eff) * BLOCK_M;
      const int split = w % p.splits;
      if constexpr (EPI != EPI_LINEAR) {
        named_bar_sync(1 + part, 128);               // the quarter's four warps are done reading the previous tile's values
        if (tq < 2 * CPP) cv[tq] = col_next;
        named_bar_sync(1 + part, 128);
        if (w + (int)gridDim.x < total_work) col_next = fetch_col(w + gridDim.x);
      }
      mbar_wait(tfull_bar(as), aph);
      tc_fence_after();
      const bool acc_zero = min(k_blocks_eff, split * kb_per_split + kb_per_split) <= split * kb_per_split;
      ChunkGeom cg;
      cg.row0 = m0 + quad * 32;
      cg.rows = min(32, g.M - cg.row0);      // <= 0: this warp's 32 rows are all beyond M
      if (cg.rows > 0) {
#pragma unroll 1
        for (int c = part * (BLOCK_N / 4); c < (part + 1) * (BLOCK_N / 4); c += CH) {
          cg.col0 = n0 + c;
          if (cg.col0 >= g.N) break;
          cg.ncols = min(CH, g.N - cg.col0);
          if constexpr (DB) {
            ChunkGeom ng;
            int nw = w, nci = (c - part * CPP) / CH, nsplit = 0;
            const bool has_next = next_chunk(nw, nci, ng, nsplit);
            const bool hs = side_wanted(split);
            epilogue_chunk_db<EPI, F8>(p, tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BLOCK_N + c), dbuf + cb * 2048,
                                   dbuf + (cb ^ 1) * 2048, cv + (c - part * CPP), cv + CPP + (c - part * CPP), lane, cg.row0 + lane, cg, split,
                                   add, keep_scale, hs, side_bar + 8u * cb, side_uses[cb] & 1u, side_bar + 8u * (cb ^ 1),
                                   has_next && side_wanted(nsplit), ng.col0, ng.row0, acc_zero);
            if (hs) ++side_uses[cb];
            cb ^= 1;
          } else {
            epilogue_chunk<EPI, F8>(p, tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * BLOCK_N + c), st, cv + (c - part * CPP),
                                cv + CPP + (c - part * CPP), lane, cg.row0 + lane, cg, split, add, keep_scale, acc_zero);
          }
        }
      }
      tc_fence_before();
      mbar_arrive(tempty_bar(as));
      if (++as == 2) { as = 0; aph ^= 1; }
    }
    if ((p.tma_d_ok | p.tma_aux_ok) && lane == 0) tma_store_wait_all();   // bulk stores must be complete before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
template <int BLOCK_N, bool A_MN, bool B_MN, int EPI, bool DB = false, bool F8 = false>
static int launch(const GemmParams& p, int grid, cudaStream_t st) {
  using Cfg = GemmCfg<BLOCK_N, DB>;
  static_assert(Cfg::kSmemBytes <= 232448, "shared memory budget");
  auto kern = gemm_tcgen05_kernel<BLOCK_N, A_MN, B_MN, EPI, DB, F8>;
  static std::once_flag once;
  static cudaError_t attr_err = cudaSuccess;
  std::call_once(once, [&] { attr_err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes); });
  if (attr_err != cudaSuccess) return (int)attr_err;
  kern<<<grid, NUM_THREADS, Cfg::kSmemBytes, st>>>(p);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  EVLM_CUDA_RETURN();
}

template <int BLOCK_N>
static int dispatch(const GemmParams& p, int grid, cudaStream_t st, int a_mn, int b_mn, int epi, bool db) {
  // instantiated combinations: the forward / dgrad / wgrad layouts the host side actually issues
  if (db) {
    if (!a_mn && !b_mn) return epi == EPI_ACT_FWD ? launch<BLOCK_N, false, false, EPI_ACT_FWD, true>(p, grid, st)
                               : epi == EPI_LINEAR ? launch<BLOCK_N, false, false, EPI_LINEAR, true>(p, grid, st) : EVLM_EUNSUPPORTED;
    if (!a_mn && b_mn && epi == EPI_ACT_BWD) return launch<BLOCK_N, false, true, EPI_ACT_BWD, true>(p, grid, st);
    return EVLM_EUNSUPPORTED;
  }
  if (!a_mn && !b_mn) return epi == EPI_ACT_FWD ? launch<BLOCK_N, false, false, EPI_ACT_FWD>(p, grid, st)
                             : epi == EPI_LINEAR ? launch<BLOCK_N, false, false, EPI_LINEAR>(p, grid, st) : EVLM_EUNSUPPORTED;
  if (!a_mn && b_mn) return epi == EPI_ACT_BWD ? launch<BLOCK_N, false, true, EPI_ACT_BWD>(p, grid, st)
                            : epi == EPI_LINEAR ? launch<BLOCK_N, false, true, EPI_LINEAR>(p, grid, st) : EVLM_EUNSUPPORTED;
  if (epi != EPI_LINEAR) return EVLM_EUNSUPPORTED;
  if (a_mn && b_mn) return launch<BLOCK_N, true, true, EPI_LINEAR>(p, grid, st);
  return launch<BLOCK_N, true, false, EPI_LINEAR>(p, grid, st);
}
// F8: the forward configurations inference reaches (the double-buffered epilogue serves the K <= 1024 residual projections)
template <int BLOCK_N>
static int dispatch_f8(const GemmParams& p, int grid, cudaStream_t st, int epi, bool db) {
  if (epi == EPI_LINEAR)
    return db ? launch<BLOCK_N, false, false, EPI_LINEAR, true, true>(p, grid, st) : launch<BLOCK_N, false, false, EPI_LINEAR, false, true>(p, grid, st);
  if (epi == EPI_ACT_FWD && !db) return launch<BLOCK_N, false, false, EPI_ACT_FWD, false, true>(p, grid, st);
  return EVLM_EUNSUPPORTED;
}

static int gemm_tcgen05_run(const evlm_gemm_args* a, const float* a_scale, const float* b_scale, void* stream);

}  // namespace evlm

extern "C" int evlm_abi_version(void) { return EVLM_ABI_VERSION; }
extern "C" unsigned long long evlm_launch_count(void) { return evlm::g_launch_count.load(); }
extern "C" void evlm_reset_launch_count(void) { evlm::g_launch_count.store(0); }

extern "C" int evlm_gemm_bf16(const evlm_gemm_args* a, void* stream) {
  using namespace evlm;
  if (!a || !a->A || !a->B || !a->D) return EVLM_EINVAL;
  if (a->M <= 0 || a->N <= 0 || a->K <= 0) return EVLM_EINVAL;
  // TMA: 16-byte aligned base and row pitch
  if ((reinterpret_cast<uintptr_t>(a->A) & 15) || (reinterpret_cast<uintptr_t>(a->B) & 15)) return EVLM_EINVAL;
  if ((a->lda % 8) || (a->ldb % 8)) return EVLM_EINVAL;
  if (a->d_dtype != EVLM_BF16 && a->d_dtype != EVLM_F32) return EVLM_EINVAL;
  if ((a->splits > 1 || a->accumulate) && a->d_dtype != EVLM_F32) return EVLM_EINVAL;
  if (a->splits > 1 && (a->epi_mode != EVLM_EPI_FORWARD || a->act != EVLM_ACT_NONE || a->gate_mode != EVLM_GATE_NONE ||
                        a->dropout_p > 0.f || a->aux_out))
    return EVLM_EINVAL;  // non-linear epilogues cannot be split along K
  if (a->epi_mode == EVLM_EPI_ACT_BACKWARD && !a->aux_in) return EVLM_EINVAL;
  if (a->gate_mode != EVLM_GATE_NONE && !a->gate) return EVLM_EINVAL;
  if (a->dropout_p < 0.f || a->dropout_p >= 1.f) return EVLM_EINVAL;
  if (a->epi_mode == EVLM_EPI_FORWARD && a->act == EVLM_ACT_NONE && a->gate_mode == EVLM_GATE_NONE && a->aux_out) return EVLM_EINVAL;
  {
    const int rc_skinny = gemm_skinny_try(a, nullptr, nullptr, stream);
    if (rc_skinny != -1) return rc_skinny;
  }
  return gemm_tcgen05_run(a, nullptr, nullptr, stream);
}

extern "C" int evlm_gemm_fp8(const evlm_gemm_args* a, const float* a_scale, const float* b_scale, void* stream) {
  using namespace evlm;
  if (!a || !a->A || !a->B || !a->D || !a_scale || !b_scale) return EVLM_EINVAL;
  if (a->M <= 0 || a->N <= 0 || a->K <= 0) return EVLM_EINVAL;
  // TMA and the weight-stream kernel's 16-byte lane loads: 16-byte aligned bases and row pitches (e4m3: pitch in bytes)
  if ((reinterpret_cast<uintptr_t>(a->A) & 15) || (reinterpret_cast<uintptr_t>(a->B) & 15) || (a->lda % 16) || (a->ldb % 16)) return EVLM_EINVAL;
  if (a->lda < a->K || a->ldb < a->K) return EVLM_EINVAL;
  if (a->a_mn || a->b_mn) return EVLM_EINVAL;
  if (a->d_dtype != EVLM_BF16 && a->d_dtype != EVLM_F32) return EVLM_EINVAL;
  if (a->epi_mode != EVLM_EPI_FORWARD || a->dropout_p != 0.f || a->splits > 1 || a->accumulate || a->gate_mode != EVLM_GATE_NONE || a->gate)
    return EVLM_EINVAL;
  if (a->m_limit || a->n_limit || a->k_limit) return EVLM_EINVAL;
  if (a->act != EVLM_ACT_NONE && a->act != EVLM_ACT_QUICK_GELU && a->act != EVLM_ACT_GELU_ERF) return EVLM_EINVAL;
  if (a->act == EVLM_ACT_NONE && a->aux_out) return EVLM_EINVAL;
  if (a->residual && a->res_dtype != EVLM_BF16 && a->res_dtype != EVLM_F32) return EVLM_EINVAL;
  {
    const int rc_skinny = gemm_skinny_try(a, a_scale, b_scale, stream);
    if (rc_skinny != -1) return rc_skinny;
  }
  return gemm_tcgen05_run(a, a_scale, b_scale, stream);
}

// The tcgen05 path of evlm_gemm_bf16 (a_scale == nullptr) and evlm_gemm_fp8 (e4m3 operands, validated by the caller).
static int evlm::gemm_tcgen05_run(const evlm_gemm_args* a, const float* a_scale, const float* b_scale, void* stream) {
  const bool f8 = a_scale != nullptr;
  const int bk = f8 ? BLOCK_K_F8 : BLOCK_K;
  const int epi = a->epi_mode == EVLM_EPI_ACT_BACKWARD ? EPI_ACT_BWD
                  : (a->act != EVLM_ACT_NONE || a->gate_mode != EVLM_GATE_NONE) ? EPI_ACT_FWD : EPI_LINEAR;

  // tile shape: 128x256 when there are enough wide tiles to fill the machine, else 128x128
  const int sms = a->max_ctas > 0 ? a->max_ctas : device_num_sms();
  const int m_tiles = (a->M + BLOCK_M - 1) / BLOCK_M;
  // (split-K products: the splits multiply the work items, so wide tiles fill the machine with fewer, longer k ranges)
  const int64_t wide_items = (int64_t)m_tiles * ((a->N + 255) / 256) * (a->splits > 1 ? a->splits : 1);
  static const bool narrow_split = getenv("EVLM_GEMM_NARROW_SPLITK") != nullptr;   // profiling knob: 128-wide tiles for split-K (round 1)
  const bool wide = (a->N >= 256) && wide_items * 10 >= (int64_t)sms * 9 && (a->splits <= 1 || !narrow_split);
  const int block_n = wide ? 256 : 128;

  GemmParams p;
  p.g = *a;
  p.a_scale = a_scale;
  p.b_scale = b_scale;
  p.m_tiles = m_tiles;
  p.n_tiles = (a->N + block_n - 1) / block_n;
  p.k_blocks = (a->K + bk - 1) / bk;
  {
    int sp = a->splits > 1 ? (a->splits < p.k_blocks ? a->splits : p.k_blocks) : 1;
    p.kb_per_split = (p.k_blocks + sp - 1) / sp;
    p.splits = (p.k_blocks + p.kb_per_split - 1) / p.kb_per_split;  // no empty splits
  }
  p.g.splits = p.splits;

  int rc;
  if (f8) {   // (K-major only)
    rc = make_tmap_e4m3(&p.tma_a, a->A, a->M, a->K, a->lda, BLOCK_M);
    if (rc) return rc;
    rc = make_tmap_e4m3(&p.tma_b, a->B, a->N, a->K, a->ldb, block_n);
    if (rc) return rc;
  } else {
    if (!a->a_mn) rc = make_tmap_bf16(&p.tma_a, a->A, a->M, a->K, a->lda, BLOCK_M);
    else          rc = make_tmap_bf16(&p.tma_a, a->A, a->K, a->M, a->lda, BLOCK_K);
    if (rc) return rc;
    if (!a->b_mn) rc = make_tmap_bf16(&p.tma_b, a->B, a->N, a->K, a->ldb, block_n);
    else          rc = make_tmap_bf16(&p.tma_b, a->B, a->K, a->N, a->ldb, BLOCK_K);
    if (rc) return rc;
  }

  // epilogue stores through TMA whenever base and row pitch are 16-byte multiples (everything the host side allocates is)
  p.tma_d_ok = p.tma_aux_ok = 0;
  {
    static const bool no_tma_store = getenv("EVLM_GEMM_NO_TMA_STORE") != nullptr;   // profiling knob: staged st.global epilogue
    const int es = a->d_dtype == EVLM_F32 ? 4 : 2;
    if (!no_tma_store && (reinterpret_cast<uintptr_t>(a->D) & 15) == 0 && ((a->ldd * es) % 16) == 0) {
      rc = make_tmap_store(&p.tma_d, a->D, a->M, a->N, a->ldd, a->d_dtype == EVLM_F32);
      p.tma_d_ok = rc == 0;
    }
    if (!no_tma_store && a->aux_out && (reinterpret_cast<uintptr_t>(a->aux_out) & 15) == 0 && (a->ld_aux_out % 8) == 0) {
      rc = make_tmap_store(&p.tma_aux, a->aux_out, a->M, a->N, a->ld_aux_out, false);
      p.tma_aux_ok = rc == 0;
    }
    if (p.tma_aux_ok && a->d_dtype == EVLM_F32) p.tma_aux_ok = 0;   // the fp32 D box needs the whole stage
  }
  // Double-buffered epilogue (side operand by TMA box loads, outputs over it in place): every flavour that reads a row-major side
  // operand or writes two outputs, provided all of its epilogue tensors are TMA-addressable (16-byte base and pitch).
  p.side_kind = 0;
  bool db = false;
  {
    static const bool no_db = getenv("EVLM_GEMM_NO_DB") != nullptr;   // profiling knob: the single-buffer LSU epilogue
    const bool fwd_layout = !a->a_mn && !a->b_mn, bwd_layout = !a->a_mn && a->b_mn;
    const void* side = epi == EPI_ACT_BWD ? a->aux_in : a->residual;
    const bool side_f32 = epi != EPI_ACT_BWD && a->res_dtype == EVLM_F32;
    const int64_t side_ld = epi == EPI_ACT_BWD ? a->ld_aux_in : a->ldr;
    // Measured on the B200 (scripts/gpu_gemm_db_ab.sh, profiles/r02_gemm_db_ab.log): the activation backward gains 38 % (535 -> 739
    // TFLOP/s at 25216 x 3072 x 768) and the K = 768 residual projections 14 % (577 -> 657); where no side operand is read (activation
    // forward) or the main loop is long (K = 3072 residual GEMMs) the lost pipeline stage costs 2 - 8 %, so those keep four stages.
    const bool wants = epi == EPI_ACT_BWD || (epi == EPI_LINEAR && a->residual != nullptr && a->K <= 1024);
    const bool layout_ok = (epi == EPI_ACT_BWD) ? bwd_layout : fwd_layout;
    const bool outs_ok = p.tma_d_ok && (!a->aux_out || (p.tma_aux_ok && a->d_dtype == EVLM_BF16));
    bool side_ok = true;
    if (side) side_ok = (reinterpret_cast<uintptr_t>(side) & 15) == 0 && ((side_ld * (side_f32 ? 4 : 2)) % 16) == 0;
    if (!no_db && wants && layout_ok && outs_ok && side_ok && a->splits <= 1) {
      if (side) {
        rc = make_tmap_store(&p.tma_side, side, a->M, a->N, side_ld, side_f32);
        if (rc == 0) p.side_kind = side_f32 ? 1 : 2;
      }
      db = !side || p.side_kind != 0;
    }
  }
  const int64_t total = (int64_t)p.m_tiles * p.n_tiles * p.splits;
  const int grid = (int)(total < sms ? total : sms);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (f8) return block_n == 256 ? dispatch_f8<256>(p, grid, st, epi, db) : dispatch_f8<128>(p, grid, st, epi, db);
  return block_n == 256 ? dispatch<256>(p, grid, st, a->a_mn, a->b_mn, epi, db) : dispatch<128>(p, grid, st, a->a_mn, a->b_mn, epi, db);
}

// evlm_rng_bind() reaches the per-translation-unit seed-offset pointer through this hook (evlm_common.cuh).
namespace evlm { cudaError_t rng_bind_gemm_tcgen05(const void* state_dev) { return tu_rng_bind(state_dev); } }
