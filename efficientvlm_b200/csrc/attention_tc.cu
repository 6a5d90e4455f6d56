// tcgen05 / TMEM forward attention for key lengths <= 256 (ViT-224: 197, BERT self: <= 40, text->image cross: 197).
//
// One CTA per (batch, head, 128-query tile).  Everything between the Q/K/V loads and the context store stays on chip:
//   TMA        Q [128 x 64], K [Lkp x 64], V [Lkp x 64]  (bf16, 128B swizzle)      Lkp = round_up(Lk, 16)
//   tcgen05    S[128 x Lkp] = Q K^T  -> TMEM (fp32)           4 UMMAs  (M 128, N Lkp, K 16)
//   softmax    TMEM lane = query row; the row's 16-key chunks are dealt round-robin to TC_SPLIT threads;
//              p~ = exp2(s*c + mask - max) goes (a) back to TMEM when the probabilities are wanted and
//              (b) as bf16 (after dropout) into a 128B-swizzled K-major smem tile that aliases the dead Q/K tiles
//   P write    normalised fp32 probabilities are transposed through a per-warp smem stage so every global store is a
//              coalesced 128-byte row segment (the [B,h,Lq,Lk] rows are only 4-byte aligned for odd Lk = 197)
//   tcgen05    O[128 x 64] = P V  (V is used in place as an MN-major B operand) -> TMEM, re-using S's columns
//   epilogue   ctx = O * head_z / rowsum -> bf16, 128 contiguous bytes per thread; lse for the backward.
// Every query row is shared by TC_SPLIT threads (column groups), row max / sum exchanged through shared memory.
// Two CTAs fit per SM (<= 113 KB smem, 256 TMEM columns each) so one CTA's softmax overlaps the other's loads / MMAs.
// KD-mode attention is HBM-bound on the P write (SURVEY §8d): P is written exactly once, never re-read here.
#include "evlm_common.cuh"
#include "evlm_tma.cuh"
#include "../../include/evlm.h"
#include <atomic>
#include <cstdlib>

namespace evlm {
extern std::atomic<unsigned long long> g_launch_count;

constexpr float TC_LOG2E = 1.4426950408889634f;
constexpr float TC_LN2 = 0.6931471805599453f;
constexpr int TC_SPLIT = 2;                          // column groups: each query row is shared by TC_SPLIT threads (one per group)
constexpr int TC_SM_WARPS = 4 * TC_SPLIT;            // softmax warps: (TMEM lane quadrant) x (column group)
constexpr int TC_SM_THREADS = TC_SM_WARPS * 32;
constexpr int TC_THREADS = TC_SM_THREADS + 32;       // + 1 control warp (TMA + MMA issue)
constexpr int TC_STAGE_LD = 17;                      // padded row of the per-warp [32 x 16] transpose stage (floats)
constexpr int TC_STAGE_BYTES = TC_SM_WARPS * 32 * TC_STAGE_LD * 4;
constexpr int TC_RED_BYTES = 2 * TC_SPLIT * 128 * 4; // row max | row sum partials, [group][row]
constexpr int TC_MAX_PACK = 3;
constexpr int TC_TAIL_BYTES = TC_STAGE_BYTES + TC_RED_BYTES + TC_MAX_PACK * 256 * 4 + 64;   // + key masks (one per packed item) + barriers

struct AttnTcParams {
  CUtensorMap tq, tk, tv;
  CUtensorMap tq_pack;   // Q with a box of Lq rows: one load per packed query item
  CUtensorMap tk_pack, tv_pack;   // K / V with a box of Lk rows (pack_own_kv: one load per packed item)
  CUtensorMap tp32, tp8;          // probability maps [B*H][Lq][ldp] with boxes of 32 / 8 rows x 16 columns (valid when p_tma)
  int p_tma;
  evlm_attn_args a;
  int Lkp;        // keys padded to a multiple of 16 (UMMA N)
  int p_bytes;    // bytes of the P region (aliases Q | K)
  int v_bytes;    // bytes reserved for the V tile (multiple of 1024)
  int tmem_cols;  // power of two >= max(Lkp, 64): small key lengths leave TMEM for more co-resident CTAs
};

__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const float (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7]), "f"(v[8]), "f"(v[9]), "f"(v[10]), "f"(v[11]),
      "f"(v[12]), "f"(v[13]), "f"(v[14]), "f"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void tc_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  tmem_ld_32x32b_x16(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  tmem_ld_32x32b_x32(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void tc_named_bar(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

template <bool CAUSAL>
__global__ void __launch_bounds__(TC_THREADS, 3) attn_fwd_tc_kernel(const __grid_constant__ AttnTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  const evlm_attn_args& a = p.a;
  const uint32_t sbase = smem_u32(smem_raw);
  if ((sbase & 1023u) != 0) __trap();
  uint8_t* sptr = smem_raw;
  // layout: [ P region = Q (16 KB) | K ... ] [ V ] [ transpose stages ] [ row max / sum partials ] [ key mask 256 floats ] [ barriers ]
  const uint32_t sQ = sbase, sK = sbase + 16384, sP = sbase;
  const uint32_t sV = sbase + p.p_bytes;
  float* stage = reinterpret_cast<float*>(sptr + p.p_bytes + p.v_bytes);
  float* red_max = reinterpret_cast<float*>(sptr + p.p_bytes + p.v_bytes + TC_STAGE_BYTES);
  float* red_sum = red_max + TC_SPLIT * 128;
  float* smask = red_sum + TC_SPLIT * 128;
  const uint32_t bar0 = sbase + p.p_bytes + p.v_bytes + TC_STAGE_BYTES + TC_RED_BYTES + TC_MAX_PACK * 256 * 4;
  const uint32_t bar_load = bar0, bar_s = bar0 + 8, bar_p = bar0 + 16, bar_o = bar0 + 24;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(sptr + (bar0 - sbase) + 32);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.y, q0 = blockIdx.x * 128;
  const int Lkp = p.Lkp;
  // Packed mode: this CTA's tile rows [s*Lq, (s+1)*Lq) belong to query item pack_items[group][s]; all of them attend to the
  // K/V item of the first one.  Unpacked: one item (blockIdx.z), query tile q0.
  const bool packed = a.pack_items != nullptr;
  const int G = packed ? a.pack_width : 1;
  int items[TC_MAX_PACK];
  int nvalid = 0;
#pragma unroll
  for (int s2 = 0; s2 < TC_MAX_PACK; ++s2) {
    items[s2] = -1;
    if (packed) {
      if (s2 < G) items[s2] = __ldg(a.pack_items + (int64_t)blockIdx.z * G + s2);
    } else if (s2 == 0) {
      items[0] = blockIdx.z;
    }
    if (items[s2] >= 0) nvalid = s2 + 1;
  }
  const int b = items[0];
  const bool own_kv = packed && a.pack_own_kv;   // block-diagonal pack: member s owns tile keys [s*Lk, (s+1)*Lk)

  if (warp == TC_SM_WARPS) {
    if (lane == 0) {
      tma_prefetch_desc(&p.tq);
      tma_prefetch_desc(&p.tk);
      tma_prefetch_desc(&p.tv);
      mbar_init(bar_load, 1);
      mbar_init(bar_s, 1);
      mbar_init(bar_p, TC_SM_THREADS);
      mbar_init(bar_o, 1);
      fence_mbar_init();
      // The operand loads only need the barrier: they go out first, so their HBM round trip runs under the TMEM allocation, the
      // key-mask staging and the CTA-wide barrier below instead of after them.
      if (packed) {
        mbar_expect_tx(bar_load, nvalid * a.Lq * 128 + (own_kv ? 2 * nvalid * a.Lk * 128 : 2 * Lkp * 128));
        for (int s2 = 0; s2 < nvalid; ++s2) {
          const int itm = s2 == 0 ? items[0] : (s2 == 1 ? items[1] : items[2]);
          tma_load_2d(sQ + s2 * a.Lq * 128, &p.tq_pack, h * 64, itm * a.Lq, bar_load);
          if (own_kv) {
            const int kvi = a.kv_index ? __ldg(a.kv_index + itm) : itm;
            tma_load_2d(sK + s2 * a.Lk * 128, &p.tk_pack, h * 64, kvi * a.Lk, bar_load);
            tma_load_2d(sV + s2 * a.Lk * 128, &p.tv_pack, h * 64, kvi * a.Lk, bar_load);
          }
        }
      } else {
        mbar_expect_tx(bar_load, 16384 + 2 * Lkp * 128);
        tma_load_2d(sQ, &p.tq, h * 64, b * a.Lq + q0, bar_load);
      }
      if (!own_kv) {
        const int kvb = a.kv_index ? __ldg(a.kv_index + b) : b;   // K/V batch item of this query item / pack
        tma_load_2d(sK, &p.tk, h * 64, kvb * a.Lk, bar_load);
        tma_load_2d(sV, &p.tv, h * 64, kvb * a.Lk, bar_load);
      }
    }
    __syncwarp();
    tmem_alloc(smem_u32((const void*)tmem_ptr_smem), (uint32_t)p.tmem_cols);
    tmem_relinquish();
  }
  // additive key mask (one per packed item) in log2 units; keys beyond Lk (padding / next batch's rows) are excluded with -inf
  for (int j = threadIdx.x; j < 256 * TC_MAX_PACK; j += TC_THREADS) {
    const int s2 = j >> 8, key = j & 255;
    const int it = s2 == 0 ? items[0] : (s2 == 1 ? items[1] : items[2]);
    float m = -INFINITY;
    if (own_kv) {   // tile key `key` belongs to member key / Lk: visible to that member's rows only
      const int lk = key - s2 * a.Lk;
      if (lk >= 0 && lk < a.Lk && it >= 0) m = a.key_mask ? a.key_mask[(int64_t)it * a.Lk + lk] * TC_LOG2E : 0.f;
    } else if (key < a.Lk && it >= 0) {
      m = a.key_mask ? a.key_mask[(int64_t)it * a.Lk + key] * TC_LOG2E : 0.f;
    }
    smask[j] = m;
  }
  if (own_kv) {
    // K / V rows beyond the members' keys are never loaded: they must be finite (0 x NaN = NaN in P V), so they are zeroed
    // (a swizzled 128-byte row is still one contiguous 128-byte row)
    const int first = nvalid * a.Lk, nrows = Lkp - first;
    for (int t = threadIdx.x; t < nrows * 8 * 2; t += TC_THREADS) {
      const int which = t / (nrows * 8), rem = t - which * nrows * 8;
      uint8_t* base = sptr + (which ? p.p_bytes : 16384) + (first + (rem >> 3)) * 128 + (rem & 7) * 16;
      *reinterpret_cast<uint4*>(base) = make_uint4(0u, 0u, 0u, 0u);
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;

  if (warp == TC_SM_WARPS) {
    if (lane == 0) {
      // (the Q / K / V loads were issued before the TMEM allocation and the mask staging: see the top of the kernel)
      mbar_wait(bar_load, 0);
      tc_fence_after();
      // ---- S = Q K^T ----
      const uint32_t idesc_s = make_idesc_bf16(128, Lkp, false, false);
#pragma unroll
      for (int k = 0; k < 4; ++k) umma_bf16(tmem, make_desc_kmajor(sQ + k * 32), make_desc_kmajor(sK + k * 32), idesc_s, k > 0 ? 1u : 0u);
      umma_commit(bar_s);
      // ---- O = P V (after the softmax warps have filled the P tile) ----
      mbar_wait(bar_p, 0);
      tc_fence_after();
      const uint32_t idesc_o = make_idesc_bf16(128, 64, false, true);
      const int ksteps = Lkp >> 4;
      for (int k = 0; k < ksteps; ++k)
        umma_bf16(tmem, make_desc_kmajor(sP + (k >> 2) * 16384 + (k & 3) * 32), make_desc_mnmajor(sV + k * 2048), idesc_o, k > 0 ? 1u : 0u);
      umma_commit(bar_o);
    }
  } else {
    // ===== softmax: query row q0 + r (TMEM lane r) is shared by TC_SPLIT threads; thread (r, grp) owns the 16-key chunks
    // ===== grp, grp + TC_SPLIT, ...; row max and row sum are exchanged through shared memory between the warps of a quadrant
    const int quad = warp & 3, grp = warp >> 2;
    const int r = quad * 32 + lane;
    // row r -> (query item, query index inside the item)
    const int slot = packed ? r / a.Lq : 0;
    const int item = packed ? (slot == 0 ? items[0] : (slot == 1 ? items[1] : (slot == 2 ? items[2] : -1))) : b;
    const int qi = packed ? r - slot * a.Lq : q0 + r;
    const bool row_valid = packed ? (slot < nvalid) : (qi < a.Lq);
    const int tile_rows = packed ? nvalid * a.Lq : a.Lq - q0;   // valid rows of this CTA's tile (packed items are compact)
    const int warp_rows = min(32, tile_rows - quad * 32);        // valid query rows of this warp (<= 0: none)
    const float* mrow = smask + (packed ? min(slot, TC_MAX_PACK - 1) * 256 : 0);
    // block-diagonal pack: only the 16-key chunks that overlap this row's own keys [klo, khi) carry probability mass
    // (tcgen05.ld is warp-collective, so the skip is decided per WARP: [wlo, whi) spans the keys owned by any valid row of
    // the warp; inside it the per-member -inf mask does the rest)
    const int klo = own_kv ? slot * a.Lk : 0, khi = own_kv ? klo + a.Lk : Lkp;
    const int wlo = __reduce_min_sync(0xffffffffu, row_valid ? klo : 0x7fffffff), whi = __reduce_max_sync(0xffffffffu, row_valid ? khi : 0);
    const uint32_t trow = tmem + ((uint32_t)(quad * 32) << 16);
    const float sc2 = a.scale * TC_LOG2E;
    const float causal_neg = -10000.0f * TC_LOG2E;
    const int jlim = qi + a.causal_offset;  // keys j > jlim get the additive -10000 when CAUSAL
    const bool want_probs = a.probs != nullptr;
    const int64_t ldp = a.ldp ? a.ldp : a.Lk;   // row pitch of the probability maps
    const int n16 = Lkp >> 4;
    const bool dead = warp_rows <= 0;       // (warp-uniform) no valid query row: only the P-tile zeros and the barriers matter
    mbar_wait(bar_s, 0);
    tc_fence_after();

    // pass A: row maximum over this thread's chunks
    float m2 = -INFINITY;
    if (!dead) {
      for (int cc = grp; cc < n16; cc += TC_SPLIT) {
        if (cc * 16 + 16 <= wlo || cc * 16 >= whi) continue;
        float v[16];
        tc_ld16(trow + cc * 16, v);
#pragma unroll
        for (int j4 = 0; j4 < 16; j4 += 4) {
          const float4 m4 = *reinterpret_cast<const float4*>(mrow + cc * 16 + j4);
          const float mk[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            float x = fmaf(v[j4 + jj], sc2, mk[jj]);
            if (CAUSAL && (cc * 16 + j4 + jj) > jlim) x += causal_neg;
            m2 = fmaxf(m2, x);
          }
        }
      }
    }
    red_max[grp * 128 + r] = m2;
    tc_named_bar(1 + quad, 32 * TC_SPLIT);
#pragma unroll
    for (int g2 = 0; g2 < TC_SPLIT; ++g2) m2 = fmaxf(m2, red_max[g2 * 128 + r]);

    // pass B: p~ = 2^(x - max); partial row sum; p~ -> TMEM (fp32, for the P write) and -> smem (bf16 A operand of P V)
    float l = 0.f;
    const float keep_inv = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
    const uint64_t seed = a.dropout_seed + rng_offset();
    const uint64_t lkp4 = (uint64_t)((a.Lk + 3) & ~3);
    const uint64_t erow = (((uint64_t)(item < 0 ? 0 : item) * a.H + h) * a.Lq + qi) * lkp4;
    uint8_t* prow = sptr + r * 128;   // row r inside each 16 KB atom
    for (int cc = grp; cc < n16; cc += TC_SPLIT) {
      float v[16];
      const bool off_block = cc * 16 + 16 <= wlo || cc * 16 >= whi;     // (warp-uniform) chunk holds other pack members' keys only: P = 0
      if (!dead && !off_block) {
        tc_ld16(trow + cc * 16, v);
#pragma unroll
        for (int j4 = 0; j4 < 16; j4 += 4) {
          const float4 m4 = *reinterpret_cast<const float4*>(mrow + cc * 16 + j4);
          const float mk[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {
            float x = fmaf(v[j4 + jj], sc2, mk[jj]);
            if (CAUSAL && (cc * 16 + j4 + jj) > jlim) x += causal_neg;
            const float pv = fast_ex2(x - m2);
            l += pv;
            v[j4 + jj] = pv;
          }
        }
        if (want_probs) tmem_st_32x32b_x16(trow + cc * 16, v);
        if (a.dropout_p > 0.f) {
#pragma unroll
          for (int j = 0; j < 16; j += 4) {   // one Philox call per 4 consecutive keys (row stride padded to a multiple of 4)
            // the item's own key index (own-K/V pack: tile key - klo, a multiple of 4 since Lk % 8 == 0), so the mask does not
            // depend on the pack slot; keys left of the row's block have P = 0 and are clamped rather than wrapped
            const float4 u = dropout_uniform4(seed, a.dropout_stream, (erow + (uint64_t)max(cc * 16 + j - klo, 0)) >> 2);
            v[j] = u.x >= a.dropout_p ? v[j] * keep_inv : 0.f;
            v[j + 1] = u.y >= a.dropout_p ? v[j + 1] * keep_inv : 0.f;
            v[j + 2] = u.z >= a.dropout_p ? v[j + 2] * keep_inv : 0.f;
            v[j + 3] = u.w >= a.dropout_p ? v[j + 3] * keep_inv : 0.f;
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0.f;
      }
      // bf16, 128B-swizzled K-major tile: atom = 64 keys; 16-byte chunk index XOR (row % 8)
#pragma unroll
      for (int j8 = 0; j8 < 2; ++j8) {
        const int key = cc * 16 + j8 * 8;
        const int atom = key >> 6, chunk = (key & 63) >> 3;
        uint4 o = make_uint4(pack_bf16x2(v[j8 * 8], v[j8 * 8 + 1]), pack_bf16x2(v[j8 * 8 + 2], v[j8 * 8 + 3]),
                             pack_bf16x2(v[j8 * 8 + 4], v[j8 * 8 + 5]), pack_bf16x2(v[j8 * 8 + 6], v[j8 * 8 + 7]));
        *reinterpret_cast<uint4*>(prow + atom * 16384 + ((chunk ^ (r & 7)) << 4)) = o;
      }
    }
    red_sum[grp * 128 + r] = l;
    tc_named_bar(1 + quad, 32 * TC_SPLIT);
    l = 0.f;
#pragma unroll
    for (int g2 = 0; g2 < TC_SPLIT; ++g2) l += red_sum[g2 * 128 + r];
    const float inv_l = 1.f / l;
    // pass C: normalised probabilities -> global, coalesced through the per-warp transpose stage:
    // one store instruction covers 2 rows x 16 keys (64 contiguous bytes each)
    if (want_probs && !dead && p.p_tma) {
      // Normalised probabilities leave as TMA box stores: the thread parks its row of the 16-key chunk in the warp's swizzled
      // [32][16] stage (four 16-byte shared stores), one lane hands the box to the TMA unit (un-packed: 32 rows of one map; packed:
      // four 8-row boxes, each inside one item's rows).  No per-element global store, no read-back through shared memory; rows
      // beyond Lq and columns beyond the (padded) pitch are clipped by the tensor map.
      tmem_st_wait();
      float* st = stage + warp * 512;
      const bool issuer = packed ? ((lane & 7) == 0) : (lane == 0);
      const int g8 = lane >> 3;                       // packed: this issuer's 8-row group
      const int r8 = quad * 32 + g8 * 8;              // its first tile row
      const int s8 = packed ? r8 / a.Lq : 0;
      const int it8 = packed ? (s8 == 0 ? items[0] : (s8 == 1 ? items[1] : (s8 == 2 ? items[2] : -1))) : b;
      const bool box_ok = packed ? (s8 < nvalid && it8 >= 0) : true;
      for (int cc = grp; cc < n16; cc += TC_SPLIT) {
        if (cc * 16 >= (int)ldp) break;
        float v[16];
        tc_ld16(trow + cc * 16, v);
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] *= inv_l;
        if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the previous chunk's box has left the stage
        __syncwarp();
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4)
          *reinterpret_cast<float4*>(st + lane * 16 + ((q4 ^ ((lane >> 1) & 3)) << 2)) = make_float4(v[4 * q4], v[4 * q4 + 1], v[4 * q4 + 2], v[4 * q4 + 3]);
        fence_proxy_async();
        __syncwarp();
        if (issuer && box_ok) {
          const uint32_t src = smem_u32(st) + (packed ? (uint32_t)(g8 * 512) : 0u);
          const CUtensorMap* tm = packed ? &p.tp8 : &p.tp32;
          const int row0 = packed ? r8 - s8 * a.Lq : q0 + quad * 32;
          asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(reinterpret_cast<uint64_t>(tm)),
                       "r"(src), "r"(cc * 16), "r"(row0), "r"(it8 * a.H + h)
                       : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        }
      }
    } else if (want_probs && !dead) {
      tmem_st_wait();
      float* st = stage + warp * 32 * TC_STAGE_LD;
      // global row of every tile row of this warp (packed rows of one warp may belong to two items): lane r owns row r's offset
      const int64_t my_row = row_valid ? ((int64_t)item * a.H + h) * a.Lq + qi : -1;
      const int my_lo = own_kv ? slot * a.Lk : 0;          // first tile key of this row's own block
      const int cj = lane & 15, rh = lane >> 4;
      for (int cc = grp; cc < n16; cc += TC_SPLIT) {
        if (cc * 16 + 16 <= wlo || cc * 16 >= whi) continue;
        float v[16];
        tc_ld16(trow + cc * 16, v);
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 16; ++j) st[lane * TC_STAGE_LD + j] = v[j] * inv_l;
        __syncwarp();
        const int col = cc * 16 + cj;
        if (!packed) {
          // un-packed: the warp's tile rows are consecutive rows of one map: fixed 32-bit offsets from the first one
          if (col < ldp) {                                           // (pad columns Lk .. ldp-1 receive their exact zeros)
            float* pb = a.probs + (((int64_t)b * a.H + h) * a.Lq + q0 + quad * 32 + rh) * ldp + col;
            const float* sb = st + rh * TC_STAGE_LD + cj;
            const int step2 = 2 * (int)ldp;
            if (warp_rows >= 32) {                                   // (warp-uniform) full warp: branch-free, fully unrolled
#pragma unroll
              for (int u = 0; u < 16; ++u) pb[u * step2] = sb[u * 2 * TC_STAGE_LD];
            } else {
#pragma unroll 4
              for (int u = 0; u < 16; ++u)
                if (2 * u + rh < warp_rows) pb[u * step2] = sb[u * 2 * TC_STAGE_LD];
            }
          }
        } else {
#pragma unroll 4
          for (int u = 0; u < 16; ++u) {
            const int rr = 2 * u + rh;
            const int64_t grow = __shfl_sync(0xffffffffu, my_row, rr);
            const int lcol = col - __shfl_sync(0xffffffffu, my_lo, rr);
            if (rr < warp_rows && grow >= 0 && lcol >= 0 && lcol < (own_kv ? (int64_t)a.Lk : ldp)) a.probs[grow * ldp + lcol] = st[rr * TC_STAGE_LD + cj];
          }
        }
      }
    }
    // hand the P tile to the tensor core: generic-proxy smem writes -> async proxy, TMEM reads done
    fence_proxy_async();
    tc_fence_before();
    mbar_arrive(bar_p);
    // ---- epilogue: O -> ctx; thread (r, grp) stores 64 / TC_SPLIT columns of its row ----
    if (!dead) {
      mbar_wait(bar_o, 0);
      tc_fence_after();
      const float z = a.head_z ? __ldg(a.head_z + h) : 1.f;
      const float osc = z * inv_l;
      constexpr int OC = 64 / TC_SPLIT;
      __nv_bfloat16* cg = reinterpret_cast<__nv_bfloat16*>(a.ctx) + ((int64_t)(item < 0 ? 0 : item) * a.Lq + qi) * a.ldc + h * 64 + grp * OC;
#pragma unroll
      for (int c = 0; c < OC / 16; ++c) {
        float v[16];
        tc_ld16(trow + grp * OC + c * 16, v);
        if (row_valid) {
#pragma unroll
          for (int j = 0; j < 16; j += 8) {
            uint4 o = make_uint4(pack_bf16x2(v[j] * osc, v[j + 1] * osc), pack_bf16x2(v[j + 2] * osc, v[j + 3] * osc),
                                 pack_bf16x2(v[j + 4] * osc, v[j + 5] * osc), pack_bf16x2(v[j + 6] * osc, v[j + 7] * osc));
            *reinterpret_cast<uint4*>(cg + c * 16 + j) = o;
          }
        }
      }
      if (grp == 0 && row_valid && a.lse) a.lse[((int64_t)item * a.H + h) * a.Lq + qi] = (m2 + log2f(l)) * TC_LN2;
    }
  }
  if (p.p_tma && warp < TC_SM_WARPS) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // bulk stores complete before the CTA exits
  tc_fence_before();
  __syncthreads();
  if (warp == TC_SM_WARPS) {
    tc_fence_after();
    tmem_dealloc(tmem, (uint32_t)p.tmem_cols);
  }
}

// Returns EVLM_EUNSUPPORTED when the shape is outside this kernel's envelope (the caller then uses the tiled kernel).
int attention_fwd_tc(const evlm_attn_args* a, cudaStream_t st) {
  if (a->Lk > 256 || a->full_mask != nullptr) return EVLM_EUNSUPPORTED;
  if ((a->ldc % 8) || (reinterpret_cast<uintptr_t>(a->ctx) & 15)) return EVLM_EUNSUPPORTED;
  if (a->pack_items) {
    if (a->pack_width < 1 || a->pack_width > TC_MAX_PACK || a->pack_width * a->Lq > 128 || (a->Lq % 8) || a->pack_groups <= 0 || a->causal)
      return EVLM_EINVAL;
  }
  const bool own_kv = a->pack_items && a->pack_own_kv;
  if (own_kv && ((a->Lk % 8) || a->pack_width * a->Lk > 128)) return EVLM_EINVAL;
  AttnTcParams p;
  p.a = *a;
  p.Lkp = ((own_kv ? a->pack_width * a->Lk : a->Lk) + 15) & ~15;
  const int atoms = (p.Lkp + 63) / 64;
  const int kv_bytes = (p.Lkp * 128 + 1023) & ~1023;
  p.p_bytes = atoms * 16384;
  if (p.p_bytes < 16384 + kv_bytes) p.p_bytes = 16384 + kv_bytes;   // must also hold Q | K
  p.v_bytes = kv_bytes;
  p.tmem_cols = 64;
  while (p.tmem_cols < p.Lkp) p.tmem_cols <<= 1;
  const size_t smem = (size_t)p.p_bytes + p.v_bytes + TC_TAIL_BYTES;
  int rc = make_tmap_bf16(&p.tq, a->q, (int64_t)a->B * a->Lq, (int64_t)a->H * 64, a->ldq, 128);
  if (rc) return rc;
  const int64_t kv_items = a->kv_index ? a->kv_batches : a->B;
  if (a->pack_items) {
    rc = make_tmap_bf16(&p.tq_pack, a->q, (int64_t)a->B * a->Lq, (int64_t)a->H * 64, a->ldq, a->Lq);
    if (rc) return rc;
  }
  rc = make_tmap_bf16(&p.tk, a->k, kv_items * a->Lk, (int64_t)a->H * 64, a->ldk, own_kv ? a->Lk : p.Lkp);
  if (rc) return rc;
  rc = make_tmap_bf16(&p.tv, a->v, kv_items * a->Lk, (int64_t)a->H * 64, a->ldv, own_kv ? a->Lk : p.Lkp);
  if (rc) return rc;
  p.tk_pack = p.tk;
  p.tv_pack = p.tv;
  p.p_tma = 0;
  {
    static const bool no_tma_p = getenv("EVLM_ATTN_NO_TMA_P") != nullptr;   // profiling knob: the staged scalar-store path
    const int64_t ldp = a->ldp ? a->ldp : a->Lk;
    if (a->probs && !own_kv && !no_tma_p && (ldp % 4) == 0 && (reinterpret_cast<uintptr_t>(a->probs) & 15) == 0 &&
        (!a->pack_items || (a->Lq % 8) == 0)) {
      const int r32 = make_tmap_probs(&p.tp32, a->probs, ldp, a->Lq, (int64_t)a->B * a->H, 32);
      const int r8 = make_tmap_probs(&p.tp8, a->probs, ldp, a->Lq, (int64_t)a->B * a->H, 8);
      p.p_tma = (r32 == 0 && r8 == 0) ? 1 : 0;
    }
  }
  if (rc) return rc;
  static size_t smem_set[2] = {0, 0};
  dim3 grid(a->pack_items ? 1 : (a->Lq + 127) / 128, a->H, a->pack_items ? a->pack_groups : a->B);
  if (a->causal) {
    if (smem > smem_set[1]) {
      cudaError_t e = cudaFuncSetAttribute(attn_fwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      smem_set[1] = smem;
    }
    attn_fwd_tc_kernel<true><<<grid, TC_THREADS, smem, st>>>(p);
  } else {
    if (smem > smem_set[0]) {
      cudaError_t e = cudaFuncSetAttribute(attn_fwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return (int)e;
      smem_set[0] = smem;
    }
    attn_fwd_tc_kernel<false><<<grid, TC_THREADS, smem, st>>>(p);
  }
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? EVLM_OK : (int)e;
}

}  // namespace evlm

// evlm_rng_bind() reaches the per-translation-unit seed-offset pointer through this hook (evlm_common.cuh).
namespace evlm { cudaError_t rng_bind_attention_tc(const void* state_dev) { return tu_rng_bind(state_dev); } }
