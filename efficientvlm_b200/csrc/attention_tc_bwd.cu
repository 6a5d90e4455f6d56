// tcgen05 / TMEM backward attention for Lq, Lk <= 256 (ViT-224, BERT self-attention, text->image cross-attention).
//
// One CTA per (batch, head); key tiles (128) outer, query tiles (128) inner; all five products run on the tensor cores
// with every operand read IN PLACE from 128B-swizzled shared-memory tiles (K-major or MN-major UMMA descriptors):
//     S  = Q K^T          A = Q tile  (K-major)     B = K tile  (K-major)        -> TMEM [128 q x 128 keys]
//     G  = dO V^T         A = dO tile (K-major)     B = V tile  (K-major)        -> TMEM
//     dV += (DoP)^T dO    A = P tile  (MN-major)    B = dO tile (MN-major)       -> TMEM [128 keys x 64]
//     dK += dS^T Q        A = dS tile (MN-major)    B = Q tile  (MN-major)       -> TMEM
//     dQ += dS K          A = dS tile (K-major)     B = K tile  (MN-major)       -> TMEM [128 q x 64] per query tile
// Between the two groups, 16 warps (one thread per query row and 32-key quarter of the tile) turn S / G into P and dS:
//     P = exp(S*scale + mask - lse) (re-computed from the forward's row log-sum-exp: P is never read from HBM),
//     dS = P o (head_z * D o G + dP_ext - delta),   D = dropout mask replayed from (seed, index),
// where dP_ext is the gradient arriving on the returned attention map (attention-map distillation) and
// delta_i = <dctx_i, ctx_i> + sum_j dP_ext_ij P_ij comes from a small pre-kernel.  dQ / dK / dV leave as bf16 straight from
// TMEM: no fp32 workspace, no atomics.  TMEM: S 128 | G 128 | dV 64 | dK 64 | dQ[0] 64 | dQ[1] 64 = 512 columns.
//
// LONG variant (256 < max(Lq, Lk), Lk <= 1024: ViT-384 / ViT-480, question -> image cross attention): same tile loop, but
//   * a CTA owns a (batch, head, RANGE of key tiles) and sweeps ALL query tiles, so dK / dV of its keys are still complete in
//     TMEM when they are drained (no accumulation across CTAs);
//   * dQ cannot stay in TMEM for more than two query tiles: every (key tile, query tile) product dS K lands in one of the two
//     dQ buffers (alternating) and is drained by the elementwise warps of the NEXT iteration with red.global.add.v4.f32 into
//     the caller's fp32 dq accumulator [B*Lq, H*64] (zeroed before the launch, cast to bf16 afterwards) — L2-resident atomics,
//     issued after the warps have handed P / dS to the tensor core, i.e. off the critical path.
#include "evlm_common.cuh"
#include "evlm_tma.cuh"
#include "../../include/evlm.h"
#include <atomic>
#include <cstdlib>

namespace evlm {
extern std::atomic<unsigned long long> g_launch_count;
constexpr int EVLM_OK_LONG = 1 << 30;   // internal: the LONG variant ran; the caller still has to cast the fp32 dq accumulator

constexpr float TB_LOG2E = 1.4426950408889634f;
constexpr int TB_MATH_WARPS = 16;
constexpr int TB_MATH_THREADS = TB_MATH_WARPS * 32;
constexpr int TB_THREADS = TB_MATH_THREADS + 32;  // 16 elementwise warps + 1 control warp

struct AttnTcBwdParams {
  CUtensorMap tq, tk, tv, tdo;
  CUtensorMap tq_pack, tdo_pack;   // boxes of Lq rows: one load per packed query item
  CUtensorMap tk_pack, tv_pack;    // boxes of Lk rows (pack_own_kv: one load per packed item)
  evlm_attn_args a;
  const float* delta;
  float* dq_acc;       // LONG: fp32 [B*Lq, H*64] accumulator for dQ (zeroed by the host)
  int kt_per_cta;      // LONG: key tiles per CTA (blockIdx.y selects the range)
};

// smem map (bytes, all tiles 1024-aligned)
constexpr int TB_Q0 = 0, TB_Q1 = 16384, TB_DO0 = 32768, TB_DO1 = 49152, TB_K = 65536, TB_V = 81920, TB_P = 98304, TB_DS = 131072;
constexpr int TB_MAX_PACK = 3;
constexpr int TB_MASK = 163840;             // 3 x 256 floats: additive key mask per packed item (log2 units), -inf beyond Lk;
                                            // LONG: 1024 floats for the one item of the CTA
constexpr int TB_MASK_BYTES = 4096;
constexpr int TB_RED = TB_MASK + TB_MASK_BYTES;        // 32 floats
constexpr int TB_BARS = TB_RED + 128;       // barriers
constexpr int TB_XP = TB_BARS + 128;        // per-warp [32][17] fp32 transposition stage for the external dP tile
constexpr int TB_XP_WARP = 32 * 17 * 4;
constexpr int TB_SMEM = TB_XP + TB_MATH_WARPS * TB_XP_WARP + 1024;

__device__ __forceinline__ void tb_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  tmem_ld_32x32b_x16(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
}
__device__ __forceinline__ void tb_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  tmem_ld_32x32b_x32(taddr, r);
  tmem_ld_wait();
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
}

// PACKED is a template parameter so that the un-packed instantiation (ViT: the longest launches) does not carry the pack bookkeeping
// (member tables, per-row item look-ups, block-diagonal masks) in its registers.
template <bool CAUSAL, bool LONG, bool PACKED = false>
__global__ void __launch_bounds__(TB_THREADS, 1) attn_bwd_tc_kernel(const __grid_constant__ AttnTcBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  const evlm_attn_args& a = p.a;
  const uint32_t sbase = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* sptr = smem_raw + (sbase - smem_u32(smem_raw));
  float* smask = reinterpret_cast<float*>(sptr + TB_MASK);
  float* sred = reinterpret_cast<float*>(sptr + TB_RED);
  const uint32_t bar0 = sbase + TB_BARS;
  const uint32_t bar_kv = bar0, bar_q0 = bar0 + 8, bar_q1 = bar0 + 16, bar_sg = bar0 + 24, bar_pd = bar0 + 32, bar_mma = bar0 + 40,
                 bar_epi = bar0 + 48;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(sptr + TB_BARS + 64);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int h = blockIdx.x % a.H;
  // Packed mode (see attention_tc.cu): tile rows [s*Lq, (s+1)*Lq) belong to query item pack_items[group][s]; the group shares
  // the K/V item of its first member, and its dK / dV (summed over the members by the tensor core) go to row block `group`.
  constexpr bool packed = PACKED;
  const int grp_id = blockIdx.x / a.H;
  const int G = packed ? a.pack_width : 1;
  int items[TB_MAX_PACK];
  int nvalid = 0;
#pragma unroll
  for (int s2 = 0; s2 < TB_MAX_PACK; ++s2) {
    items[s2] = -1;
    if (packed) {
      if (s2 < G) items[s2] = __ldg(a.pack_items + (int64_t)grp_id * G + s2);
    } else if (s2 == 0) {
      items[0] = grp_id;
    }
    if (items[s2] >= 0) nvalid = s2 + 1;
  }
  const int b = items[0];
  const int Lq_tile = packed ? nvalid * a.Lq : a.Lq;     // valid query rows over all tiles of this CTA
  const bool own_kv = packed && a.pack_own_kv;            // block-diagonal pack: member s owns tile keys [s*Lk, (s+1)*Lk)
  const int Lk_tile = own_kv ? nvalid * a.Lk : a.Lk;      // valid key rows over all key tiles of this CTA
  const int nkt = (Lk_tile + 127) >> 7, nqt = packed ? 1 : (a.Lq + 127) >> 7;
  // key tiles of this CTA: all of them, or (LONG) the blockIdx.y-th range of kt_per_cta tiles
  const int kt_begin = LONG ? (int)blockIdx.y * p.kt_per_cta : 0;
  const int kt_end = LONG ? min(nkt, kt_begin + p.kt_per_cta) : nkt;
  const int n_iter = (kt_end - kt_begin) * nqt;
  constexpr int MASK_AND = LONG ? 1023 : 255;

  if (warp == TB_MATH_WARPS) {
    if (lane == 0) {
      tma_prefetch_desc(&p.tq);
      tma_prefetch_desc(&p.tk);
      tma_prefetch_desc(&p.tv);
      tma_prefetch_desc(&p.tdo);
      mbar_init(bar_kv, 1);
      mbar_init(bar_q0, 1);
      mbar_init(bar_q1, 1);
      mbar_init(bar_sg, 1);
      mbar_init(bar_pd, TB_MATH_THREADS);
      mbar_init(bar_mma, 1);
      mbar_init(bar_epi, TB_MATH_THREADS);
      fence_mbar_init();
    }
    __syncwarp();
    tmem_alloc(smem_u32((const void*)tmem_ptr_smem), 512);
    tmem_relinquish();
  }
  if (LONG) {
    for (int j = threadIdx.x; j < 1024; j += TB_THREADS)
      smask[j] = j < a.Lk ? (a.key_mask ? a.key_mask[(int64_t)b * a.Lk + j] * TB_LOG2E : 0.f) : -INFINITY;
  }
  for (int j = threadIdx.x; !LONG && j < 256 * TB_MAX_PACK; j += TB_THREADS) {
    const int s2 = j >> 8, key = j & 255;
    const int itm = s2 == 0 ? items[0] : (s2 == 1 ? items[1] : items[2]);
    float m = -INFINITY;
    if (own_kv) {   // tile key `key` belongs to member key / Lk: visible to that member's rows only
      const int lk = key - s2 * a.Lk;
      if (lk >= 0 && lk < a.Lk && itm >= 0) m = a.key_mask ? a.key_mask[(int64_t)itm * a.Lk + lk] * TB_LOG2E : 0.f;
    } else if (key < a.Lk && itm >= 0) {
      m = a.key_mask ? a.key_mask[(int64_t)itm * a.Lk + key] * TB_LOG2E : 0.f;
    }
    smask[j] = m;
  }
  if (packed) {
    // Rows of the operand tiles that no TMA load fills (empty pack slots, keys beyond the members') are reduced over by the
    // dV / dK / dQ products: they must be finite (0 x NaN = NaN), so they are zeroed once; later loads never touch them.
    const int qfirst = Lq_tile, qrows = 128 - qfirst;
    for (int t = threadIdx.x; t < qrows * 8 * 4; t += TB_THREADS) {
      const int which = t / (qrows * 8), rem = t - which * qrows * 8;
      const int off = which == 0 ? TB_Q0 : (which == 1 ? TB_Q1 : (which == 2 ? TB_DO0 : TB_DO1));
      *reinterpret_cast<uint4*>(sptr + off + (qfirst + (rem >> 3)) * 128 + (rem & 7) * 16) = make_uint4(0u, 0u, 0u, 0u);
    }
    if (own_kv) {
      const int kfirst = Lk_tile, krows = 128 - kfirst;
      for (int t = threadIdx.x; t < krows * 8 * 2; t += TB_THREADS) {
        const int which = t / (krows * 8), rem = t - which * krows * 8;
        *reinterpret_cast<uint4*>(sptr + (which ? TB_V : TB_K) + (kfirst + (rem >> 3)) * 128 + (rem & 7) * 16) = make_uint4(0u, 0u, 0u, 0u);
      }
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr_smem;
  const uint32_t T_S = tmem, T_G = tmem + 128, T_DV = tmem + 256, T_DK = tmem + 320, T_DQ = tmem + 384;

  if (warp == TB_MATH_WARPS) {
    if (lane == 0) {
      const uint32_t idesc_sg = make_idesc_bf16(128, 128, false, false);
      const uint32_t idesc_dkv = make_idesc_bf16(128, 64, true, true);    // A = P / dS tile as MN-major, B = dO / Q tile as MN-major
      const uint32_t idesc_dq = make_idesc_bf16(128, 64, false, true);    // A = dS tile K-major, B = K tile MN-major
      // prefetch the first Q / dO tile
      if (packed) {
        mbar_expect_tx(bar_q0, 2 * nvalid * a.Lq * 128);
        for (int s2 = 0; s2 < nvalid; ++s2) {
          const int itm = s2 == 0 ? items[0] : (s2 == 1 ? items[1] : items[2]);
          tma_load_2d(sbase + TB_Q0 + s2 * a.Lq * 128, &p.tq_pack, h * 64, itm * a.Lq, bar_q0);
          tma_load_2d(sbase + TB_DO0 + s2 * a.Lq * 128, &p.tdo_pack, h * 64, itm * a.Lq, bar_q0);
        }
      } else {
        mbar_expect_tx(bar_q0, 32768);
        tma_load_2d(sbase + TB_Q0, &p.tq, h * 64, b * a.Lq, bar_q0);
        tma_load_2d(sbase + TB_DO0, &p.tdo, h * 64, b * a.Lq, bar_q0);
      }
      const int kvb = a.kv_index ? __ldg(a.kv_index + b) : b;   // K/V batch item of this query item (dk / dv stay per query item)
      int it = 0;
      for (int kt = kt_begin; kt < kt_end; ++kt) {
        for (int qt = 0; qt < nqt; ++qt, ++it) {
          const uint32_t sQ = sbase + ((it & 1) ? TB_Q1 : TB_Q0), sDO = sbase + ((it & 1) ? TB_DO1 : TB_DO0);
          const uint32_t sK = sbase + TB_K, sV = sbase + TB_V, sP = sbase + TB_P, sDS = sbase + TB_DS;
          auto issue_sg = [&]() {
            mbar_wait((it & 1) ? bar_q1 : bar_q0, (it >> 1) & 1);
            if (qt == 0) mbar_wait(bar_kv, (kt - kt_begin) & 1);
            tc_fence_after();
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(T_S, make_desc_kmajor(sQ + k * 32), make_desc_kmajor(sK + k * 32), idesc_sg, k > 0 ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_bf16(T_G, make_desc_kmajor(sDO + k * 32), make_desc_kmajor(sV + k * 32), idesc_sg, k > 0 ? 1u : 0u);
            umma_commit(bar_sg);
          };
          // S / G of this iteration only need the elementwise warps to be done with the previous S / G (bar_pd, waited on last
          // iteration) and run in issue order behind the previous dV / dK / dQ products: within a key tile they are issued
          // BEFORE waiting for those products to complete.  A new key tile must wait first (its K / V loads overwrite operands).
          if (qt > 0) issue_sg();
          if (it > 0) {  // previous iteration's dV / dK / dQ products have finished reading Q, dO, K, V, P, dS
            mbar_wait(bar_mma, (it - 1) & 1);
            tc_fence_after();
          }
          if (qt == 0) {
            if (own_kv) {
              mbar_expect_tx(bar_kv, 2 * nvalid * a.Lk * 128);
              for (int s2 = 0; s2 < nvalid; ++s2) {
                const int itm = s2 == 0 ? items[0] : (s2 == 1 ? items[1] : items[2]);
                const int kvi = a.kv_index ? __ldg(a.kv_index + itm) : itm;
                tma_load_2d(sbase + TB_K + s2 * a.Lk * 128, &p.tk_pack, h * 64, kvi * a.Lk, bar_kv);
                tma_load_2d(sbase + TB_V + s2 * a.Lk * 128, &p.tv_pack, h * 64, kvi * a.Lk, bar_kv);
              }
            } else {
              mbar_expect_tx(bar_kv, 32768);
              tma_load_2d(sbase + TB_K, &p.tk, h * 64, kvb * a.Lk + kt * 128, bar_kv);
              tma_load_2d(sbase + TB_V, &p.tv, h * 64, kvb * a.Lk + kt * 128, bar_kv);
            }
          }
          {  // prefetch the next iteration's Q / dO tile into the other buffer
            const int nit = it + 1;
            if (nit < n_iter) {
              const int nq = nit % nqt;
              const uint32_t bq = (nit & 1) ? bar_q1 : bar_q0;
              if (packed) {
                mbar_expect_tx(bq, 2 * nvalid * a.Lq * 128);
                for (int s2 = 0; s2 < nvalid; ++s2) {
                  const int itm = s2 == 0 ? items[0] : (s2 == 1 ? items[1] : items[2]);
                  tma_load_2d(sbase + ((nit & 1) ? TB_Q1 : TB_Q0) + s2 * a.Lq * 128, &p.tq_pack, h * 64, itm * a.Lq, bq);
                  tma_load_2d(sbase + ((nit & 1) ? TB_DO1 : TB_DO0) + s2 * a.Lq * 128, &p.tdo_pack, h * 64, itm * a.Lq, bq);
                }
              } else {
                mbar_expect_tx(bq, 32768);
                tma_load_2d(sbase + ((nit & 1) ? TB_Q1 : TB_Q0), &p.tq, h * 64, b * a.Lq + nq * 128, bq);
                tma_load_2d(sbase + ((nit & 1) ? TB_DO1 : TB_DO0), &p.tdo, h * 64, b * a.Lq + nq * 128, bq);
              }
            }
          }
          if (qt == 0) issue_sg();
          // P and dS tiles written by the elementwise warps
          mbar_wait(bar_pd, it & 1);
          tc_fence_after();
          if (qt == 0 && kt > kt_begin) {  // the previous key tile's dV / dK have been drained from TMEM
            mbar_wait(bar_epi, (kt - kt_begin - 1) & 1);
            tc_fence_after();
          }
          // dV += P^T dO ; dK += dS^T Q      (reduction over the 128 queries of this tile: 8 steps of 16 rows = +2048 B)
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16(T_DV, make_desc_mnmajor(sP + k * 2048, 16384), make_desc_mnmajor(sDO + k * 2048), idesc_dkv, (qt > 0 || k > 0) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16(T_DK, make_desc_mnmajor(sDS + k * 2048, 16384), make_desc_mnmajor(sQ + k * 2048), idesc_dkv, (qt > 0 || k > 0) ? 1u : 0u);
          // dQ[qt] += dS K                    (reduction over the 128 keys: atom = k / 4, +32 B inside the atom)
#pragma unroll
          for (int k = 0; k < 8; ++k)
            umma_bf16(T_DQ + (LONG ? (it & 1) : qt) * 64, make_desc_kmajor(sDS + (k >> 2) * 16384 + (k & 3) * 32),
                      make_desc_mnmajor(sK + k * 2048), idesc_dq, ((!LONG && kt > 0) || k > 0) ? 1u : 0u);
          umma_commit(bar_mma);
        }
      }
    }
  } else {
    // ========== elementwise warps: thread = (query row r of the tile, 32-key quarter qtr of the 128-key tile) ==========
    const int quad = warp & 3, qtr = warp >> 2;
    const int hf = qtr >> 1;                       // which 64-key swizzle atom of the P / dS tiles
    const int r = quad * 32 + lane;
    const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
    const float sc2 = a.scale * TB_LOG2E;
    const float causal_neg = -10000.0f * TB_LOG2E;
    const float z = a.head_z ? __ldg(a.head_z + h) : 1.f;
    const float keep_inv = a.dropout_p > 0.f ? 1.f / (1.f - a.dropout_p) : 1.f;
    // dp_kd_coef: the "external dP" operand holds the distillation TARGET map T and dP = coef * (P - T) is formed here from the re-computed P
    const bool kd = a.dp_kd_coef != nullptr;
    const float kd_c = kd ? __ldg(a.dp_kd_coef) : 0.f;
    const uint64_t lkp4 = (uint64_t)((a.Lk + 3) & ~3);
    const uint64_t seed = a.dropout_seed + rng_offset();
    float dz_part = 0.f;
    uint8_t* prow = sptr + TB_P + hf * 16384 + r * 128;
    uint8_t* dsrow = sptr + TB_DS + hf * 16384 + r * 128;
    float* xp = reinterpret_cast<float*>(sptr + TB_XP + warp * TB_XP_WARP);
    // Pull this warp's [32 rows x 32 keys] block of the external dP map into L2 one iteration ahead (one lane per row, both ends
    // of its 128-byte segment): the demand loads below then pay an L2 hit instead of a DRAM round trip on the critical path.
    const int64_t ldp = a.ldp ? a.ldp : a.Lk;   // row pitch of the external dP map
    // tile row -> global row id ((item * H + h) * Lq + i) of lse / delta / probs / dP, or -1 beyond the valid rows
    auto global_row = [&](int trow) -> int64_t {
      if (trow >= Lq_tile) return -1;
      if (!packed) return ((int64_t)b * a.H + h) * a.Lq + trow;
      const int sl = trow / a.Lq;
      const int itm = sl == 0 ? items[0] : (sl == 1 ? items[1] : items[2]);
      return ((int64_t)itm * a.H + h) * a.Lq + (trow - sl * a.Lq);
    };
    auto prefetch_dp = [&](int kt_, int qt_) {
      if (a.dprobs_ext == nullptr) return;
      const int trow = qt_ * 128 + quad * 32 + lane;
      const int64_t grow = global_row(trow);
      int key = kt_ * 128 + qtr * 32;
      if (own_kv) key = max(0, key - (trow / a.Lq) * a.Lk);      // the row's keys live in its own Lk-wide block
      if (grow >= 0 && key < a.Lk) {
        const float* q0 = a.dprobs_ext + grow * ldp + key;
        const float* q1 = q0 + (min(32, a.Lk - key) - 1);
        asm volatile("prefetch.global.L2 [%0];" ::"l"(q0));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(q1));
      }
    };
    // LONG: the dS K product of local iteration `pit` (query tile pqt) sits in dQ buffer pit & 1: scale it and add it to the fp32
    // accumulator.  Warp (quad, qtr) takes rows quad*32.. and columns qtr*16..+16: 64 contiguous bytes per thread.
    auto drain_dq = [&](int pit, int pqt) {
      tc_fence_after();
      float v[16];
      tb_ld16(T_DQ + (uint32_t)((pit & 1) * 64) + lane_off + (uint32_t)(qtr * 16), v);
      const int iq = pqt * 128 + r;
      if (iq < a.Lq) {
        float* dst = p.dq_acc + ((int64_t)b * a.Lq + iq) * ((int64_t)a.H * 64) + h * 64 + qtr * 16;
#pragma unroll
        for (int j = 0; j < 16; j += 4)
          asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dst + j), "f"(v[j] * a.scale), "f"(v[j + 1] * a.scale),
                       "f"(v[j + 2] * a.scale), "f"(v[j + 3] * a.scale)
                       : "memory");
      }
    };
    // Un-packed: the external dP chunk [32 rows x 16 keys] of (key tile, query tile, 16-key chunk c) of this warp's 32 x 32 block.
    // Rows are consecutive rows of ONE map (fixed 32-bit offsets, no shuffles).  The loads are issued ONE CHUNK AHEAD of their
    // use (tpre / tpre_tag): the L2 round trip overlaps the previous chunk's arithmetic or the wait for the next S / G tile.
    auto fetch_dp = [&](int kt_, int qt_, int c_, float (&t)[16]) {
      const int rh = lane >> 4, cj = lane & 15;
      const int r0 = qt_ * 128 + quad * 32;                       // first tile row of this warp
      const int wr = min(32, Lq_tile - r0);                        // its valid rows
      const int jc = kt_ * 128 + qtr * 32 + c_ * 16 + cj;          // tile key of this lane's column
      if (!packed) {
        const bool colok = jc < a.Lk;
        const float* base = a.dprobs_ext + (((int64_t)b * a.H + h) * a.Lq + r0 + rh) * ldp + jc;
        const int step2 = 2 * (int)ldp;
#pragma unroll
        for (int u = 0; u < 16; ++u) t[u] = (colok && 2 * u + rh < wr) ? __ldg(base + u * step2) : 0.f;
        return;
      }
      // Packed tiles (Lq >= 32): the warp's 32 rows belong to at most TWO consecutive pack members.  Rows below `bnd` are rows of
      // member s0 (map row r0 - s0 Lq + rr), the others rows of member s0 + 1 (map row rr - bnd): two warp-uniform bases, no
      // per-row shuffles, and the loads can be issued a chunk ahead like the un-packed ones.
      const int s0 = r0 / a.Lq;
      const int bnd = (s0 + 1) * a.Lq - r0;
      const int it0 = s0 == 0 ? items[0] : (s0 == 1 ? items[1] : (s0 == 2 ? items[2] : -1));
      const int it1 = s0 == 0 ? items[1] : (s0 == 1 ? items[2] : -1);
      const float* b0 = a.dprobs_ext + (((int64_t)max(it0, 0) * a.H + h) * a.Lq + (r0 - s0 * a.Lq)) * ldp;
      const float* b1 = a.dprobs_ext + (((int64_t)max(it1, 0) * a.H + h) * a.Lq) * ldp;
      const int lc0 = jc - (own_kv ? s0 * a.Lk : 0), lc1 = jc - (own_kv ? (s0 + 1) * a.Lk : 0);   // column inside the member's own map
      const bool ok0 = it0 >= 0 && lc0 >= 0 && lc0 < a.Lk, ok1 = it1 >= 0 && lc1 >= 0 && lc1 < a.Lk;
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        const int rr = 2 * u + rh;
        const bool second = rr >= bnd;
        const float* src = second ? b1 + (int64_t)(rr - bnd) * ldp + lc1 : b0 + (int64_t)rr * ldp + lc0;
        t[u] = (rr < wr && (second ? ok1 : ok0)) ? __ldg(src) : 0.f;
      }
    };
    float tpre[16];
    int tpre_tag = -1;                       // (local iteration) * 2 + chunk of what tpre holds
    const bool pipe_dp = a.dprobs_ext != nullptr && (!packed || a.Lq >= 32);   // (shorter packed items: per-row shuffle path below)
    if (pipe_dp) {
      fetch_dp(kt_begin, 0, 0, tpre);
      tpre_tag = 0;
    } else {
#pragma unroll
      for (int u = 0; u < 16; ++u) tpre[u] = 0.f;
    }
    prefetch_dp(kt_begin, 0);
    int it = 0;
    for (int kt = kt_begin; kt < kt_end; ++kt) {
      const int tile_keys = min(128, Lk_tile - kt * 128);
      for (int qt = 0; qt < nqt; ++qt, ++it) {
        const int i = qt * 128 + r;                                        // row inside the CTA's query rows
        const int64_t grow_me = global_row(i);
        const bool qvalid = grow_me >= 0;
        const int warp_rows = min(32, Lq_tile - (qt * 128 + quad * 32));   // valid query rows of this warp (<= 0: none)
        const int64_t rowid = qvalid ? grow_me : 0;
        const int slot_me = packed ? min(i / a.Lq, TB_MAX_PACK - 1) : 0;
        const float* mrow = smask + slot_me * 256;
        const int lo_me = own_kv ? slot_me * a.Lk : 0;                      // first tile key of this row's own block
        const float lse2 = qvalid ? a.lse[rowid] * TB_LOG2E : 0.f;
        const float dlt = qvalid ? p.delta[rowid] : 0.f;
        // block-diagonal pack: the keys any row of this warp owns span [wlo, whi)
        int wlo = 0, whi = tile_keys;
        if (own_kv && warp_rows > 0) {
          const int r0 = qt * 128 + quad * 32;
          wlo = (r0 / a.Lq) * a.Lk;
          whi = ((r0 + warp_rows - 1) / a.Lq + 1) * a.Lk;
        }
        const bool live = warp_rows > 0 && qtr * 32 < min(tile_keys, whi) && qtr * 32 + 32 > wlo;   // anything to compute for this 32 x 32 block?
        if (qt + 1 < nqt) prefetch_dp(kt, qt + 1);
        else if (kt + 1 < kt_end) prefetch_dp(kt + 1, 0);
        if (!live) {
          // rows beyond Lq must be ZERO in P and dS (they are reduced over by the dV / dK products), key columns beyond Lk must be
          // zero in dS (reduced over by the dQ product); nothing else to do, and S / G are not even read
          mbar_wait(bar_sg, it & 1);
#pragma unroll
          for (int j8 = 0; j8 < 4; ++j8) {
            const int sw = ((((qtr & 1) * 4 + j8) ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(prow + sw) = make_uint4(0u, 0u, 0u, 0u);
            *reinterpret_cast<uint4*>(dsrow + sw) = make_uint4(0u, 0u, 0u, 0u);
          }
        } else {
          const bool has_dpe = a.dprobs_ext != nullptr;
#pragma unroll 1
          for (int c = 0; c < 2; ++c) {
            const int col = qtr * 32 + c * 16;         // column inside the 128-key tile
            const int j0 = kt * 128 + col;             // key index in the sequence
            float s[16], g[16], dpv[16];
            if (col >= min(tile_keys, whi) || col + 16 <= wlo) {   // (warp-uniform) key columns beyond Lk / owned by other pack members
              if (c == 0) {
                mbar_wait(bar_sg, it & 1);
              }
#pragma unroll
              for (int j8 = 0; j8 < 2; ++j8) {
                const int sw = ((((qtr & 1) * 4 + c * 2 + j8) ^ (r & 7)) << 4);
                *reinterpret_cast<uint4*>(prow + sw) = make_uint4(0u, 0u, 0u, 0u);
                *reinterpret_cast<uint4*>(dsrow + sw) = make_uint4(0u, 0u, 0u, 0u);
              }
              continue;
            }
            // External dP tile [32 rows x 16 keys]: fetched coalesced (half a warp per row: 64 contiguous bytes) and transposed
            // through shared memory, instead of 16 scattered 4-byte loads per row-owning thread.
            if (has_dpe) {
              float t[16];
              const int cj = lane & 15;
              if (pipe_dp) {
                if (tpre_tag == it * 2 + c) {
#pragma unroll
                  for (int u = 0; u < 16; ++u) t[u] = tpre[u];
                } else {
                  fetch_dp(kt, qt, c, t);          // a skipped chunk / dead block broke the one-ahead chain: fetch now
                }
                // put the next chunk in flight: chunk 1 of this block, or chunk 0 of the next (key tile, query tile) block
                if (c == 0) {
                  fetch_dp(kt, qt, 1, tpre);
                  tpre_tag = it * 2 + 1;
                } else {
                  const int nqt2 = qt + 1 < nqt ? qt + 1 : 0, nkt2 = qt + 1 < nqt ? kt : kt + 1;
                  if (nkt2 < kt_end) {
                    fetch_dp(nkt2, nqt2, 0, tpre);
                    tpre_tag = (it + 1) * 2;
                  }
                }
              } else {
#pragma unroll
              for (int u = 0; u < 16; ++u) {
                const int rr = 2 * u + (lane >> 4);
                const int64_t grow = __shfl_sync(0xffffffffu, grow_me, rr);   // lane rr owns tile row rr of this warp
                const int lcol = j0 + cj - __shfl_sync(0xffffffffu, lo_me, rr);
                t[u] = (grow >= 0 && lcol >= 0 && lcol < a.Lk) ? __ldg(a.dprobs_ext + grow * ldp + lcol) : 0.f;
              }
              }
              __syncwarp();
#pragma unroll
              for (int u = 0; u < 16; ++u) xp[(2 * u + (lane >> 4)) * 17 + cj] = t[u];
              __syncwarp();
#pragma unroll
              for (int j = 0; j < 16; ++j) dpv[j] = xp[lane * 17 + j];
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j) dpv[j] = 0.f;
            }
            if (c == 0) {
              mbar_wait(bar_sg, it & 1);
              tc_fence_after();
            }
            tb_ld16(T_S + lane_off + col, s);
            tb_ld16(T_G + lane_off + col, g);
#pragma unroll
            for (int j4 = 0; j4 < 16; j4 += 4) {
              const float4 m4 = *reinterpret_cast<const float4*>(mrow + ((j0 + j4) & MASK_AND));   // loaded per group of 4: 12 fewer live registers
              const float mk4[4] = {m4.x, m4.y, m4.z, m4.w};
              float dm[4] = {1.f, 1.f, 1.f, 1.f};
              if (a.dropout_p > 0.f) {   // ONE Philox call per 4 consecutive keys (index = rowid * lkp4 + the item's own key)
                // own-K/V pack: tile key - lo_me (keys left of the row's block have P = 0: clamped rather than wrapped), as the forward
                const float4 u = dropout_uniform4(seed, a.dropout_stream, ((uint64_t)rowid * lkp4 + (uint64_t)max(j0 + j4 - lo_me, 0)) >> 2);
                dm[0] = u.x >= a.dropout_p ? keep_inv : 0.f;
                dm[1] = u.y >= a.dropout_p ? keep_inv : 0.f;
                dm[2] = u.z >= a.dropout_p ? keep_inv : 0.f;
                dm[3] = u.w >= a.dropout_p ? keep_inv : 0.f;
              }
#pragma unroll
              for (int jj = 0; jj < 4; ++jj) {
                const int j = j4 + jj;
                const int key = j0 + j;
                float x = fmaf(s[j], sc2, mk4[jj]);
                if (CAUSAL && key > i + a.causal_offset) x += causal_neg;
                const float pv = (qvalid && key < Lk_tile) ? fast_ex2(x - lse2) : 0.f;   // (off-block keys: mask = -inf -> 0)
                const float pd = pv * dm[jj];
                dz_part += pd > 0.f ? pd * g[j] : 0.f;
                const float dp = z * dm[jj] * g[j] + (kd ? kd_c * (pv - dpv[j]) : dpv[j]);
                s[j] = pv > 0.f ? pv * (dp - dlt) : 0.f;   // dS (selected, not multiplied: masked / padded entries stay exactly 0)
                g[j] = pd;                // D o P
              }
            }
#pragma unroll
            for (int j8 = 0; j8 < 2; ++j8) {
              const int chunk = (qtr & 1) * 4 + c * 2 + j8;   // 16-byte chunk inside this half's 64-key atom
              const int sw = (chunk ^ (r & 7)) << 4;
              *reinterpret_cast<uint4*>(prow + sw) =
                  make_uint4(pack_bf16x2(g[j8 * 8], g[j8 * 8 + 1]), pack_bf16x2(g[j8 * 8 + 2], g[j8 * 8 + 3]),
                             pack_bf16x2(g[j8 * 8 + 4], g[j8 * 8 + 5]), pack_bf16x2(g[j8 * 8 + 6], g[j8 * 8 + 7]));
              *reinterpret_cast<uint4*>(dsrow + sw) =
                  make_uint4(pack_bf16x2(s[j8 * 8], s[j8 * 8 + 1]), pack_bf16x2(s[j8 * 8 + 2], s[j8 * 8 + 3]),
                             pack_bf16x2(s[j8 * 8 + 4], s[j8 * 8 + 5]), pack_bf16x2(s[j8 * 8 + 6], s[j8 * 8 + 7]));
            }
          }
        }
        fence_proxy_async();
        tc_fence_before();
        mbar_arrive(bar_pd);
        // LONG: the previous iteration's dQ product is complete (this iteration's S / G commit, waited on above, tracks every
        // earlier MMA of the issuing thread) and its buffer is not rewritten before every warp has arrived on the NEXT bar_pd
        if (LONG && it > 0) drain_dq(it - 1, qt > 0 ? qt - 1 : nqt - 1);
        if (qt == nqt - 1) {
          // ---- this key tile's dV (quarters 0-1) / dK (quarters 2-3): TMEM -> bf16 rows, 32 columns per warp ----
          mbar_wait(bar_mma, it & 1);
          tc_fence_after();
          const int key = kt * 128 + r;
          const bool is_dv = qtr < 2;
          const int c0 = (qtr & 1) * 32;
          const float osc = is_dv ? z : a.scale;
          int64_t kvrow = (int64_t)(packed ? grp_id : b) * a.Lk + key;   // shared-K/V pack: one dK / dV row block per group
          bool kv_ok = key < a.Lk;
          if (own_kv) {                                                  // own-K/V pack: tile key row -> (member, key) -> item rows
            const int sl = key / a.Lk;
            const int itm = sl == 0 ? items[0] : (sl == 1 ? items[1] : (sl == 2 ? items[2] : -1));
            kv_ok = sl < nvalid && itm >= 0;
            kvrow = (int64_t)(itm < 0 ? 0 : itm) * a.Lk + (key - sl * a.Lk);
          }
          __nv_bfloat16* dst = is_dv ? reinterpret_cast<__nv_bfloat16*>(a.dv) + kvrow * a.lddv + h * 64
                                     : reinterpret_cast<__nv_bfloat16*>(a.dk) + kvrow * a.lddk + h * 64;
          float v[32];
          tb_ld32((is_dv ? T_DV : T_DK) + lane_off + c0, v);
          if (kv_ok) {
#pragma unroll
            for (int j = 0; j < 32; j += 8)
              *reinterpret_cast<uint4*>(dst + c0 + j) =
                  make_uint4(pack_bf16x2(v[j] * osc, v[j + 1] * osc), pack_bf16x2(v[j + 2] * osc, v[j + 3] * osc),
                             pack_bf16x2(v[j + 4] * osc, v[j + 5] * osc), pack_bf16x2(v[j + 6] * osc, v[j + 7] * osc));
          }
          tc_fence_before();
          mbar_arrive(bar_epi);
        }
      }
    }
    if (LONG) {   // the last product (its bar_mma has been waited on by the dV / dK drain above)
      if (n_iter > 0) drain_dq(n_iter - 1, nqt - 1);
    }
    // ---- dQ: quarters 0-1 drain query tile 0, quarters 2-3 query tile 1 (the last bar_mma has already been waited on) ----
    if (!LONG && (qtr >> 1) < nqt) {
      const int tq = qtr >> 1, c0 = (qtr & 1) * 32;
      const int i = tq * 128 + r;
      int64_t qrow = -1;                                   // row of q / dq: item * Lq + index inside the item
      if (i < Lq_tile) {
        if (packed) {
          const int sl = i / a.Lq;
          qrow = (int64_t)(sl == 0 ? items[0] : (sl == 1 ? items[1] : items[2])) * a.Lq + (i - sl * a.Lq);
        } else {
          qrow = (int64_t)b * a.Lq + i;
        }
      }
      __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(a.dq) + (qrow < 0 ? 0 : qrow) * a.lddq + h * 64;
      float v[32];
      tb_ld32(T_DQ + tq * 64 + lane_off + c0, v);
      if (qrow >= 0) {
#pragma unroll
        for (int j = 0; j < 32; j += 8)
          *reinterpret_cast<uint4*>(dst + c0 + j) =
              make_uint4(pack_bf16x2(v[j] * a.scale, v[j + 1] * a.scale), pack_bf16x2(v[j + 2] * a.scale, v[j + 3] * a.scale),
                         pack_bf16x2(v[j + 4] * a.scale, v[j + 5] * a.scale), pack_bf16x2(v[j + 6] * a.scale, v[j + 7] * a.scale));
      }
    }
    if (a.dhead_z != nullptr) {
      float t = warp_sum(dz_part);
      if (lane == 0) sred[warp] = t;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (a.dhead_z != nullptr && threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < TB_MATH_WARPS; ++w) t += sred[w];
    atomicAdd(a.dhead_z + h, t);
  }
  if (warp == TB_MATH_WARPS) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

// Returns EVLM_EUNSUPPORTED outside this kernel's envelope (the caller then uses the tiled mma.sync kernel).
int attention_bwd_tc(const evlm_attn_args* a, cudaStream_t st) {
  if (a->full_mask != nullptr) return EVLM_EUNSUPPORTED;
  const bool is_long = a->Lk > 256 || a->Lq > 256;
  if (is_long) {
    static const bool disabled = getenv("EVLM_ATTN_NO_LONG") != nullptr;    // profiling knob: A/B against the tiled kernel
    if (disabled || a->Lk > 1024 || a->causal || a->pack_items) return EVLM_EUNSUPPORTED;
  }
  if (a->pack_items) {
    if (a->pack_width < 1 || a->pack_width > TB_MAX_PACK || a->pack_width * a->Lq > 128 || (a->Lq % 8) || a->pack_groups <= 0 || a->causal)
      return EVLM_EINVAL;
  }
  if ((a->lddq % 8) || (a->lddk % 8) || (a->lddv % 8) || (a->lddc % 8)) return EVLM_EUNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(a->dq) | reinterpret_cast<uintptr_t>(a->dk) | reinterpret_cast<uintptr_t>(a->dv) |
       reinterpret_cast<uintptr_t>(a->dctx)) & 15)
    return EVLM_EUNSUPPORTED;
  const bool own_kv = a->pack_items && a->pack_own_kv;
  if (own_kv && ((a->Lk % 8) || a->pack_width * a->Lk > 128)) return EVLM_EINVAL;
  AttnTcBwdParams p;
  p.a = *a;
  p.delta = a->dkv_accum;   // [B, H, Lq] floats at the head of the caller's workspace
  p.dq_acc = nullptr;
  p.kt_per_cta = 0;
  int rc = make_tmap_bf16(&p.tq, a->q, (int64_t)a->B * a->Lq, (int64_t)a->H * 64, a->ldq, 128);
  if (rc) return rc;
  rc = make_tmap_bf16(&p.tdo, a->dctx, (int64_t)a->B * a->Lq, (int64_t)a->H * 64, a->lddc, 128);
  if (rc) return rc;
  if (a->pack_items) {
    rc = make_tmap_bf16(&p.tq_pack, a->q, (int64_t)a->B * a->Lq, (int64_t)a->H * 64, a->ldq, a->Lq);
    if (rc) return rc;
    rc = make_tmap_bf16(&p.tdo_pack, a->dctx, (int64_t)a->B * a->Lq, (int64_t)a->H * 64, a->lddc, a->Lq);
    if (rc) return rc;
  }
  const int n_ctas = (a->pack_items ? a->pack_groups : a->B) * a->H;
  const int64_t kv_items = a->kv_index ? a->kv_batches : a->B;
  rc = make_tmap_bf16(&p.tk, a->k, kv_items * a->Lk, (int64_t)a->H * 64, a->ldk, own_kv ? a->Lk : 128);
  if (rc) return rc;
  rc = make_tmap_bf16(&p.tv, a->v, kv_items * a->Lk, (int64_t)a->H * 64, a->ldv, own_kv ? a->Lk : 128);
  if (rc) return rc;
  p.tk_pack = p.tk;
  p.tv_pack = p.tv;
  if (rc) return rc;
  if (is_long) {
    // dq accumulator behind delta in the caller's workspace (same layout as the tiled kernel uses: evlm_attention_bwd_workspace)
    p.dq_acc = a->dkv_accum + ((((size_t)a->B * a->H * a->Lq) + 3) & ~(size_t)3);
    if (reinterpret_cast<uintptr_t>(p.dq_acc) & 15) return EVLM_EUNSUPPORTED;
    cudaError_t e = cudaMemsetAsync(p.dq_acc, 0, (size_t)a->B * a->Lq * a->H * 64 * sizeof(float), st);
    if (e != cudaSuccess) return (int)e;
    const int nkt = (a->Lk + 127) / 128;
    // key tiles per CTA: 2 amortises the per-CTA setup and the Q / dO re-reads (measured on the ITR-384 step, 5 key tiles:
    // 2 + 2 + 1 beats 5 x 1, 126.6 vs 128.1 ms; equal on VQA-480).  EVLM_BWD_KT_PER_CTA overrides (profiling knob).
    static const int kps_env = getenv("EVLM_BWD_KT_PER_CTA") ? atoi(getenv("EVLM_BWD_KT_PER_CTA")) : 0;
    p.kt_per_cta = kps_env > 0 ? kps_env : 2;
    static bool attr_long = false;
    if (!attr_long) {
      e = cudaFuncSetAttribute(attn_bwd_tc_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TB_SMEM);
      if (e != cudaSuccess) return (int)e;
      attr_long = true;
    }
    dim3 grid(n_ctas, (nkt + p.kt_per_cta - 1) / p.kt_per_cta);
    attn_bwd_tc_kernel<false, true><<<grid, TB_THREADS, TB_SMEM, st>>>(p);
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    e = cudaGetLastError();
    return e == cudaSuccess ? EVLM_OK_LONG : (int)e;
  }
  static bool attr_set[3] = {false, false, false};
  const int variant = a->pack_items ? 2 : (a->causal ? 1 : 0);       // (packed tiles are never causal: checked by the caller)
  if (!attr_set[variant]) {
    cudaError_t e = variant == 2   ? cudaFuncSetAttribute(attn_bwd_tc_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TB_SMEM)
                    : variant == 1 ? cudaFuncSetAttribute(attn_bwd_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TB_SMEM)
                                   : cudaFuncSetAttribute(attn_bwd_tc_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TB_SMEM);
    if (e != cudaSuccess) return (int)e;
    attr_set[variant] = true;
  }
  if (variant == 2) attn_bwd_tc_kernel<false, false, true><<<n_ctas, TB_THREADS, TB_SMEM, st>>>(p);
  else if (variant == 1) attn_bwd_tc_kernel<true, false><<<n_ctas, TB_THREADS, TB_SMEM, st>>>(p);
  else attn_bwd_tc_kernel<false, false><<<n_ctas, TB_THREADS, TB_SMEM, st>>>(p);
  g_launch_count.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? EVLM_OK : (int)e;
}

}  // namespace evlm

// evlm_rng_bind() reaches the per-translation-unit seed-offset pointer through this hook (evlm_common.cuh).
namespace evlm { cudaError_t rng_bind_attention_tc_bwd(const void* state_dev) { return tu_rng_bind(state_dev); } }
