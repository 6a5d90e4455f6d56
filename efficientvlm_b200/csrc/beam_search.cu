// Beam-search decode on the device: one decode position of transformers 4.12.5's beam search for every item of the batch
// (log-softmax, repetition-penalty and min-length processors, top 2 * beams, BeamSearchScorer.process, BeamHypotheses.add / is_done),
// BeamSearchScorer.finalize, and the in-place re-order of the decoder's self-attention KV caches.  The statements mirrored are
// eff_bert.py::BertLMHeadModel._beam_search and oracle/beam_search_oracle.py; with these three kernels a decode step needs no host
// involvement, so the whole loop can run eagerly without a device -> host read or be captured in one CUDA graph.
#include "evlm_common.cuh"
#include "../../include/evlm.h"
#include <atomic>
#include <climits>

namespace evlm {
extern std::atomic<unsigned long long> g_launch_count;

constexpr int BS_THREADS = 512;            // latency-bound row sweeps: 60 elements per thread and row at V = 30 522
constexpr int BS_MAX_BEAMS = 8;
constexpr int KV_STAGE_VEC = 256;            // 16-byte vectors per staged row slice (4 KB)

__device__ __forceinline__ bool bs_better(float s1, int i1, float s2, int i2) { return s1 > s2 || (s1 == s2 && i1 < i2); }

__device__ __forceinline__ float bs_block_max(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float m = red[0];
#pragma unroll
  for (int w = 1; w < BS_THREADS / 32; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  return m;
}

__device__ __forceinline__ double bs_block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < BS_THREADS / 32; ++w) s += red[w];
  __syncthreads();
  return s;
}

// BeamHypotheses.add for one item (single thread).  Scores are doubles, as the host's Python floats are: `sum / len ** lp`.
// The list keeps insertion order; on overflow the lowest (score, list index) is deleted, the rest shift down, and `worst` becomes the
// second-lowest score.  The new hypothesis is appended last, so an overflow is resolved over beams existing entries + the new one.
__device__ void bs_hyp_add(int64_t* ht, int32_t* hl, double* hs, int& count, double& worst, int beams, int64_t width, const int64_t* src,
                           int len, double sum_logprobs, double len_pow) {
  const double score = sum_logprobs / len_pow;
  if (count < beams) {
    for (int j = 0; j < len; ++j) ht[count * width + j] = src[j];
    hl[count] = len;
    hs[count] = score;
    ++count;
    worst = fmin(score, worst);
    return;
  }
  if (!(score > worst)) return;
  int j0 = beams;                                   // index `beams` stands for the new entry
  double s0 = score;
  for (int j = beams - 1; j >= 0; --j)
    if (hs[j] <= s0) { s0 = hs[j]; j0 = j; }        // descending j with <=: the lowest index among equal lowest scores
  double s1 = INFINITY;
  for (int j = 0; j <= beams; ++j) {
    if (j == j0) continue;
    const double s = j == beams ? score : hs[j];
    if (s < s1) s1 = s;
  }
  if (j0 < beams) {
    for (int j = j0; j + 1 < beams; ++j) {
      for (int c = 0; c < hl[j + 1]; ++c) ht[j * width + c] = ht[(j + 1) * width + c];
      hl[j] = hl[j + 1];
      hs[j] = hs[j + 1];
    }
    for (int c = 0; c < len; ++c) ht[(beams - 1) * width + c] = src[c];
    hl[beams - 1] = len;
    hs[beams - 1] = score;
  }
  worst = s1;
}

// One CTA per item.  Dynamic shared memory: the item's history [beams][cur_len] (int64), the per-thread candidate lists
// [BS_THREADS][KK] (float, int), and with a repetition penalty a bitmap of the vocabulary.
template <int KK>
__global__ void __launch_bounds__(BS_THREADS) beam_step_kernel(const float* __restrict__ logits, int64_t ld, int beams, int vocab, int cur_len,
                                                               int min_length, float rp, double len_pow, int early, int64_t eos, int64_t pad,
                                                               int64_t* __restrict__ tokens, int64_t width, float* __restrict__ beam_scores,
                                                               int32_t* __restrict__ beam_src, int32_t* __restrict__ done,
                                                               int64_t* __restrict__ hyp_tokens, int32_t* __restrict__ hyp_len,
                                                               double* __restrict__ hyp_score, int32_t* __restrict__ hyp_count,
                                                               double* __restrict__ hyp_worst) {
  extern __shared__ __align__(16) unsigned char bs_smem[];
  int64_t* hist = reinterpret_cast<int64_t*>(bs_smem);
  float* lst_s = reinterpret_cast<float*>(hist + beams * cur_len);
  int* lst_i = reinterpret_cast<int*>(lst_s + BS_THREADS * KK);
  uint32_t* bits = reinterpret_cast<uint32_t*>(lst_i + BS_THREADS * KK);
  __shared__ float red[BS_THREADS / 32];
  __shared__ double red_d[BS_THREADS / 32];
  __shared__ float wred_s[BS_THREADS / 32];
  __shared__ int wred_i[BS_THREADS / 32];
  __shared__ float row_m[BS_MAX_BEAMS], row_l[BS_MAX_BEAMS];
  __shared__ float top_s[KK];
  __shared__ int top_i[KK];
  __shared__ int new_src[BS_MAX_BEAMS];
  __shared__ int64_t new_tok[BS_MAX_BEAMS];
  __shared__ float new_sc[BS_MAX_BEAMS];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int64_t r0 = (int64_t)b * beams;
  if (done[b]) {
    // A finished item is frozen: identity source, pad token, score 0.  The host loop instead points its rows at row 0 of the whole
    // batch; those rows never reach the output either way, and the identity keeps the in-place re-orders inside the item.
    if (tid < beams) {
      tokens[(r0 + tid) * width + cur_len] = pad;
      beam_scores[r0 + tid] = 0.f;
      beam_src[r0 + tid] = tid;
    }
    return;
  }
  // 1. log-softmax normaliser of each beam's row (whole row): logp = (x - max) - log(sum exp(x - max)).  The sum of 30 k terms is
  // accumulated in fp64, so log-probabilities are within a few fp32 ulps of the exact value whatever the summation order.
  for (int k = 0; k < beams; ++k) {
    const float* x = logits + (r0 + k) * ld;
    float m = -INFINITY;
    for (int v = tid; v < vocab; v += BS_THREADS) m = fmaxf(m, x[v]);
    m = bs_block_max(m, red);
    double s = 0.0;
    for (int v = tid; v < vocab; v += BS_THREADS) s += (double)expf(x[v] - m);
    s = bs_block_sum(s, red_d);
    if (tid == 0) { row_m[k] = m; row_l[k] = (float)log(s); }
  }
  for (int i = tid; i < beams * cur_len; i += BS_THREADS) hist[i] = tokens[(r0 + i / cur_len) * width + i % cur_len];
  __syncthreads();
  // 2. processors + beam score, per-thread top KK over (beam, token) in ascending flat order
  float ts[KK];
  int ti[KK];
#pragma unroll
  for (int j = 0; j < KK; ++j) { ts[j] = -INFINITY; ti[j] = INT_MAX; }
  const bool penalise = rp != 1.f;
  const int words = (vocab + 31) >> 5;
  for (int k = 0; k < beams; ++k) {
    if (penalise) {
      for (int w = tid; w < words; w += BS_THREADS) bits[w] = 0u;
      __syncthreads();
      for (int j = tid; j < cur_len; j += BS_THREADS) {
        const int64_t t = hist[k * cur_len + j];
        if (t >= 0 && t < vocab) atomicOr(&bits[t >> 5], 1u << (t & 31));
      }
      __syncthreads();
    }
    const float* x = logits + (r0 + k) * ld;
    const float m = row_m[k], l = row_l[k], bsc = beam_scores[r0 + k];
    for (int v = tid; v < vocab; v += BS_THREADS) {
      float s = (x[v] - m) - l;
      if (penalise && ((bits[v >> 5] >> (v & 31)) & 1u)) s = s < 0.f ? s * rp : s / rp;
      if (v == eos && cur_len < min_length) s = -INFINITY;
      s = s + bsc;
      const int fi = k * vocab + v;
      if (bs_better(s, fi, ts[KK - 1], ti[KK - 1])) {
        ts[KK - 1] = s;
        ti[KK - 1] = fi;
#pragma unroll
        for (int j = KK - 1; j > 0; --j) {
          if (bs_better(ts[j], ti[j], ts[j - 1], ti[j - 1])) {
            const float a = ts[j]; ts[j] = ts[j - 1]; ts[j - 1] = a;
            const int c = ti[j]; ti[j] = ti[j - 1]; ti[j - 1] = c;
          }
        }
      }
    }
    if (penalise) __syncthreads();                // the next row rebuilds the bitmap
  }
#pragma unroll
  for (int j = 0; j < KK; ++j) { lst_s[tid * KK + j] = ts[j]; lst_i[tid * KK + j] = ti[j]; }
  __syncthreads();
  // 3. merge: KK rounds of a block arg-max over the heads of the sorted per-thread lists (ties: lowest flat index)
  int head = 0;
  for (int q = 0; q < KK; ++q) {
    float s = head < KK ? lst_s[tid * KK + head] : -INFINITY;
    int i = head < KK ? lst_i[tid * KK + head] : INT_MAX;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float s2 = __shfl_xor_sync(0xffffffffu, s, o);
      const int i2 = __shfl_xor_sync(0xffffffffu, i, o);
      if (bs_better(s2, i2, s, i)) { s = s2; i = i2; }
    }
    if ((tid & 31) == 0) { wred_s[tid >> 5] = s; wred_i[tid >> 5] = i; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < BS_THREADS / 32; ++w)
        if (bs_better(wred_s[w], wred_i[w], s, i)) { s = wred_s[w]; i = wred_i[w]; }
      top_s[q] = s;
      top_i[q] = i;
    }
    __syncthreads();
    if (head < KK && lst_i[tid * KK + head] == top_i[q]) ++head;
  }
  // 4. BeamSearchScorer.process + BeamHypotheses.add / is_done (one thread: 2 * beams candidates)
  if (tid == 0) {
    int64_t* ht = hyp_tokens + r0 * width;
    int32_t* hl = hyp_len + r0;
    double* hs = hyp_score + r0;
    int count = hyp_count[b];
    double worst = hyp_worst[b];
    int kept = 0;
    for (int k = 0; k < beams; ++k) { new_src[k] = k; new_tok[k] = pad; new_sc[k] = -INFINITY; }   // only reached with NaN logits
    for (int q = 0; q < KK; ++q) {
      if (top_i[q] == INT_MAX) break;                                                               // NaN rows yield no candidate
      const int tok = top_i[q] % vocab, src = top_i[q] / vocab;
      if (tok == eos) {
        if (q >= beams) continue;
        bs_hyp_add(ht, hl, hs, count, worst, beams, width, hist + src * cur_len, cur_len, (double)top_s[q], len_pow);
      } else {
        new_sc[kept] = top_s[q];
        new_tok[kept] = tok;
        new_src[kept] = src;
        ++kept;
      }
      if (kept == beams) break;
    }
    // kept == beams always holds: each beam row contributes at most one eos candidate, so at most `beams` of the 2 * beams are eos
    hyp_count[b] = count;
    hyp_worst[b] = worst;
    if (count >= beams && (early || worst >= (double)top_s[0] / len_pow)) done[b] = 1;
  }
  __syncthreads();
  // 5. history re-order inside the item, new token at column cur_len
  for (int i = tid; i < beams * cur_len; i += BS_THREADS) {
    const int k = i / cur_len, j = i % cur_len;
    if (new_src[k] != k) tokens[(r0 + k) * width + j] = hist[new_src[k] * cur_len + j];
  }
  if (tid < beams) {
    tokens[(r0 + tid) * width + cur_len] = new_tok[tid];
    beam_scores[r0 + tid] = new_sc[tid];
    beam_src[r0 + tid] = new_src[tid];
  }
}

// BeamSearchScorer.finalize, one CTA per item: live beams of unfinished items join the hypotheses, the best one is the LAST of the
// maximal scores in list order (the host's stable `sorted(..., key=score)[-1]`), and out[b] = hypothesis, eos if shorter than
// max_length, pad.
__global__ void __launch_bounds__(32) beam_finalize_kernel(const int64_t* __restrict__ tokens, int64_t width, const float* __restrict__ beam_scores,
                                                           const int32_t* __restrict__ done, int beams, int cur_len, int max_length, double len_pow,
                                                           int64_t eos, int64_t pad, int64_t* __restrict__ hyp_tokens, int32_t* __restrict__ hyp_len,
                                                           double* __restrict__ hyp_score, int32_t* __restrict__ hyp_count,
                                                           double* __restrict__ hyp_worst, int64_t* __restrict__ out, int32_t* __restrict__ out_len) {
  __shared__ int s_best, s_len;
  const int b = blockIdx.x;
  const int64_t r0 = (int64_t)b * beams;
  int64_t* ht = hyp_tokens + r0 * width;
  if (threadIdx.x == 0) {
    int32_t* hl = hyp_len + r0;
    double* hs = hyp_score + r0;
    int count = hyp_count[b];
    double worst = hyp_worst[b];
    if (!done[b])
      for (int k = 0; k < beams; ++k)
        bs_hyp_add(ht, hl, hs, count, worst, beams, width, tokens + (r0 + k) * width, cur_len, (double)beam_scores[r0 + k], len_pow);
    hyp_count[b] = count;
    hyp_worst[b] = worst;
    int best = 0;
    for (int j = 1; j < count; ++j)
      if (hs[j] >= hs[best]) best = j;
    s_best = best;
    s_len = hl[best];
    out_len[b] = hl[best];
  }
  __syncthreads();
  const int64_t* h = ht + s_best * width;
  const int n = s_len;
  for (int c = threadIdx.x; c < max_length; c += 32) out[(int64_t)b * max_length + c] = c < n ? h[c] : (c == n ? eos : pad);
}

struct KvTable {
  void* p[EVLM_KV_REORDER_MAX_LAYERS];
};

// One CTA per (position, item, layer): every row of the item takes the position's K|V row of its source beam.  The item's rows of the
// position are staged in shared memory (4 KB slices) before any is written, so repeated sources and swaps are safe in place.
__global__ void __launch_bounds__(256) kv_beam_reorder_kernel(KvTable t, const int32_t* __restrict__ beam_src, int beams, int64_t capacity,
                                                              int64_t row_vec) {
  __shared__ uint4 stage[BS_MAX_BEAMS * KV_STAGE_VEC];
  __shared__ int src[BS_MAX_BEAMS];
  const int p = blockIdx.x, b = blockIdx.y;
  if (threadIdx.x < beams) src[threadIdx.x] = beam_src[(int64_t)b * beams + threadIdx.x];
  __syncthreads();
  bool moved = false;
  for (int k = 0; k < beams; ++k) moved |= src[k] != k;
  if (!moved) return;
  uint4* base = reinterpret_cast<uint4*>(t.p[blockIdx.z]);
  const int64_t r0 = (int64_t)b * beams;
  for (int64_t c0 = 0; c0 < row_vec; c0 += KV_STAGE_VEC) {
    const int n = (int)min((int64_t)KV_STAGE_VEC, row_vec - c0);
    for (int i = threadIdx.x; i < beams * n; i += blockDim.x) {
      const int k = i / n, c = i % n;
      stage[k * KV_STAGE_VEC + c] = base[((r0 + k) * capacity + p) * row_vec + c0 + c];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < beams * n; i += blockDim.x) {
      const int k = i / n, c = i % n;
      if (src[k] != k) base[((r0 + k) * capacity + p) * row_vec + c0 + c] = stage[src[k] * KV_STAGE_VEC + c];
    }
    __syncthreads();
  }
}

template <int KK>
static int launch_beam_step(size_t smem, const float* logits, int64_t ld, int batch, int beams, int vocab, int cur_len, int min_length, float rp,
                            double len_pow, int early, int64_t eos, int64_t pad, int64_t* tokens, int64_t width, float* beam_scores, int32_t* beam_src,
                            int32_t* done, int64_t* hyp_tokens, int32_t* hyp_len, double* hyp_score, int32_t* hyp_count, double* hyp_worst,
                            cudaStream_t st) {
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(beam_step_kernel<KK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  beam_step_kernel<KK><<<(unsigned)batch, BS_THREADS, smem, st>>>(logits, ld, beams, vocab, cur_len, min_length, rp, len_pow, early, eos, pad, tokens,
                                                                   width, beam_scores, beam_src, done, hyp_tokens, hyp_len, hyp_score, hyp_count,
                                                                   hyp_worst);
  return 0;
}
}  // namespace evlm

#define ST(s) reinterpret_cast<cudaStream_t>(s)
#define COUNT(n) evlm::g_launch_count.fetch_add(n, std::memory_order_relaxed)

extern "C" int evlm_beam_step(const float* logits, int64_t ld, int32_t batch, int32_t beams, int32_t vocab, int32_t cur_len, int32_t min_length,
                              float repetition_penalty, double cur_len_pow, int32_t early_stopping, int64_t eos, int64_t pad, int64_t* tokens,
                              int64_t width, float* beam_scores, int32_t* beam_src, int32_t* done, int64_t* hyp_tokens, int32_t* hyp_len,
                              double* hyp_score, int32_t* hyp_count, double* hyp_worst, void* stream) {
  using namespace evlm;
  if (!logits || !tokens || !beam_scores || !beam_src || !done || !hyp_tokens || !hyp_len || !hyp_score || !hyp_count || !hyp_worst)
    return EVLM_EINVAL;
  if (batch <= 0 || beams < 2 || beams > BS_MAX_BEAMS || vocab <= 2 * beams || ld < vocab || cur_len < 1 || cur_len >= width ||
      eos < 0 || eos >= vocab || (int64_t)beams * vocab > INT_MAX || !(repetition_penalty > 0.f) || !(cur_len_pow > 0.0))
    return EVLM_EINVAL;
  const int KK = 2 * beams;
  size_t smem = (size_t)beams * cur_len * sizeof(int64_t) + (size_t)BS_THREADS * KK * (sizeof(float) + sizeof(int));
  if (repetition_penalty != 1.f) smem += (size_t)((vocab + 31) / 32) * sizeof(uint32_t);
  if (smem > 200 * 1024) return EVLM_EUNSUPPORTED;
  int rc = 0;
#define BS_CASE(N)                                                                                                                          \
  case N:                                                                                                                                   \
    rc = launch_beam_step<2 * N>(smem, logits, ld, batch, beams, vocab, cur_len, min_length, repetition_penalty, cur_len_pow,              \
                                 early_stopping, eos, pad, tokens, width, beam_scores, beam_src, done, hyp_tokens, hyp_len, hyp_score,     \
                                 hyp_count, hyp_worst, ST(stream));                                                                        \
    break;
  switch (beams) {
    BS_CASE(2) BS_CASE(3) BS_CASE(4) BS_CASE(5) BS_CASE(6) BS_CASE(7) BS_CASE(8)
  }
#undef BS_CASE
  if (rc) return rc;
  COUNT(1);
  EVLM_CUDA_RETURN();
}

extern "C" int evlm_beam_finalize(const int64_t* tokens, int64_t width, const float* beam_scores, const int32_t* done, int32_t batch, int32_t beams,
                                  int32_t cur_len, int32_t max_length, double cur_len_pow, int64_t eos, int64_t pad, int64_t* hyp_tokens,
                                  int32_t* hyp_len, double* hyp_score, int32_t* hyp_count, double* hyp_worst, int64_t* out, int32_t* out_len,
                                  void* stream) {
  using namespace evlm;
  if (!tokens || !beam_scores || !done || !hyp_tokens || !hyp_len || !hyp_score || !hyp_count || !hyp_worst || !out || !out_len)
    return EVLM_EINVAL;
  if (batch <= 0 || beams < 2 || beams > BS_MAX_BEAMS || cur_len < 1 || cur_len > width || max_length < 1 || max_length > width || !(cur_len_pow > 0.0))
    return EVLM_EINVAL;
  beam_finalize_kernel<<<(unsigned)batch, 32, 0, ST(stream)>>>(tokens, width, beam_scores, done, beams, cur_len, max_length, cur_len_pow, eos, pad,
                                                               hyp_tokens, hyp_len, hyp_score, hyp_count, hyp_worst, out, out_len);
  COUNT(1);
  EVLM_CUDA_RETURN();
}

extern "C" int evlm_kv_beam_reorder(void* const* caches_host, int32_t layers, int32_t batch, int32_t beams, int64_t capacity, int64_t row_elems,
                                    int32_t len, const int32_t* beam_src, void* stream) {
  using namespace evlm;
  if (!caches_host || !beam_src || layers < 1 || layers > EVLM_KV_REORDER_MAX_LAYERS || batch <= 0 || batch > 65535 || beams < 2 ||
      beams > BS_MAX_BEAMS || len < 0 || len > capacity || row_elems <= 0 || row_elems % 8 != 0)
    return EVLM_EINVAL;
  KvTable t;
  for (int l = 0; l < layers; ++l) {
    if (!caches_host[l] || (reinterpret_cast<uintptr_t>(caches_host[l]) & 15) != 0) return EVLM_EINVAL;
    t.p[l] = caches_host[l];
  }
  if (len == 0) return EVLM_OK;
  kv_beam_reorder_kernel<<<dim3((unsigned)len, (unsigned)batch, (unsigned)layers), 256, 0, ST(stream)>>>(t, beam_src, beams, capacity,
                                                                                                       row_elems / 8);
  COUNT(1);
  EVLM_CUDA_RETURN();
}
