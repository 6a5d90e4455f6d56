/*
 * evlm.h — C ABI of libevlm_b200.so, the sm_100a kernel library behind the EfficientVLM hot path.
 *
 * The reference (swaggy-TN/EfficientVLM) is pure PyTorch and has no FFI of its own; every entry point
 * below replaces a group of library-op call sites of the reference (cited per function as
 * file:line under /root/reference).  The host side (efficientvlm_b200 python modules) binds these with ctypes
 * and exposes them behind the reference's Python class API (see INTEGRATION.md).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host; tensors are row-major, contiguous
 *     in their last dimension, leading dimensions are given in ELEMENTS;
 *   - `stream` is a cudaStream_t passed as void*; nothing is ever launched on the legacy default
 *     stream implicitly and no entry point synchronises;
 *   - return value: 0 = OK, < 0 = argument/shape error (EVLM_EINVAL -1, EVLM_EUNSUPPORTED -2; the
 *     Python binding raises ValueError, mirroring the reference's `raise ValueError` at
 *     eff_vit.py:149-169), > 0 = cudaError_t (RuntimeError);
 *   - no entry point allocates persistent device memory; workspaces are caller-provided;
 *   - re-entrant: safe to call from the autograd worker thread concurrently with the main thread.
 */
#ifndef EVLM_H_
#define EVLM_H_
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVLM_ABI_VERSION 9
int evlm_abi_version(void);
/* Number of kernel launches issued through this library by the calling process (bench gpu_launches). */
unsigned long long evlm_launch_count(void);
void evlm_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Dense contraction on tcgen05 tensor cores (bf16 x bf16 -> fp32 in TMEM), TMA-fed, persistent.
 *   D[M,N] = epilogue( sum_k A[m,k] * B[n,k] )
 * Replaces: nn.Linear call sites eff_vit.py:137-139,199,215,219; eff_bert.py:277-295,375,446,459,
 * 723,745; xvlm.py:375-382,479 and their autograd backward (dgrad / wgrad).
 *   a_mn = 0: A stored [M, lda] (K contiguous)      a_mn = 1: A stored [K, lda] (M contiguous)
 *   b_mn = 0: B stored [N, ldb] (K contiguous)      b_mn = 1: B stored [K, ldb] (N contiguous)
 * so forward = (0,0), dgrad dX = dY * W = (0,1), wgrad dW = dY^T * X = (1,1).
 * -----------------------------------------------------------------------------------------------*/
enum { EVLM_ACT_NONE = 0, EVLM_ACT_QUICK_GELU = 1, EVLM_ACT_GELU_ERF = 2 };
enum { EVLM_GATE_NONE = 0, EVLM_GATE_PRE_ACT = 1, EVLM_GATE_POST_ACT = 2 };
enum { EVLM_EPI_FORWARD = 0, EVLM_EPI_ACT_BACKWARD = 1 };
enum { EVLM_BF16 = 0, EVLM_F32 = 1 };

typedef struct evlm_gemm_args {
  int32_t M, N, K;
  const void* A; int64_t lda; int32_t a_mn;       /* bf16 */
  const void* B; int64_t ldb; int32_t b_mn;       /* bf16 */
  void* D; int64_t ldd; int32_t d_dtype;          /* EVLM_BF16 | EVLM_F32 */
  int32_t epi_mode;                               /* EVLM_EPI_* */
  /* forward epilogue: v = acc (+bias[n]); v *= alpha for n < alpha_cols; [aux_out = v];
   *   gate(pre) -> act -> gate(post) -> dropout -> (+ residual[m,n]) -> D                          */
  const float* bias;                              /* [N] or NULL */
  float alpha; int32_t alpha_cols;                /* q-scaling of eff_vit.py:137 (incl. bias) */
  int32_t act;                                    /* EVLM_ACT_* */
  const float* gate; int32_t gate_mode;           /* mlp_z / intermediate_z column gate [N] */
  void* aux_out; int64_t ld_aux_out;              /* bf16: forward = pre-activation u; act-backward = gate-grad integrand */
  const void* aux_in; int64_t ld_aux_in;          /* bf16: act-backward: saved pre-activation u */
  const void* residual; int64_t ldr; int32_t res_dtype; /* added last */
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_stream;
  /* reduction-dimension split: partial sums are red.add'ed into fp32 D (D must be pre-initialised;
   * "+=" semantics).  splits <= 1: plain store (or accumulate if `accumulate`).                   */
  int32_t splits;
  int32_t accumulate;                             /* fp32 D only: D += result */
  int32_t max_ctas;                               /* 0 = number of SMs */
  /* Zero-skip (north star: "skip fully-zeroed heads and columns"): optional DEVICE scalars that shrink the problem without a host
   * read-back.  Only tiles / k-blocks below min(dim, *limit) are scheduled; operands and outputs keep their full-size buffers, with
   * the kept rows / columns compacted to the front (evlm_compact_index, evlm_gather_*).  Output tiles are written whole, so every
   * column below the limit rounded up to the tile width (128 or 256) is defined.  k_limit == 0 gives D = epilogue(0).              */
  const int32_t* m_limit; const int32_t* n_limit; const int32_t* k_limit;
} evlm_gemm_args;

int evlm_gemm_bf16(const evlm_gemm_args* args, void* stream);

/* ABI v9 — FP8 inference (csrc/fp8.cu, the F8 instantiations of gemm_tcgen05.cu / gemm_skinny.cu).
 * evlm_quant_rows_e4m3: rows of x [rows, cols] (x_dtype EVLM_BF16 | EVLM_F32, row pitch ldx elements) -> e4m3 q [rows, ldq bytes] and one
 *   fp32 scale per row, with a fixed formula that a host mirror reproduces bit for bit:
 *     amax = max_k |x[r,k]|;  inv = 448 / amax (IEEE division);  q[r,k] = cvt.rn.satfinite.e4m3(x[r,k] * inv);  scale[r] = amax / 448
 *   (amax == 0: q = 0, scale = 0).  ldq % 16 == 0 and ldq >= cols (the TMA row pitch of the GEMM operands); bytes [cols, ldq) of every row
 *   are written as 0.  One launch serves both operands: activations (a scale per token row) and weights [N, K] (a scale per output channel).
 * evlm_gemm_fp8: D = epilogue(a_scale[m] * b_scale[n] * sum_k qa[m,k] * qb[n,k]) with A and B e4m3 (the pointers of args), both K-major,
 *   lda / ldb in bytes, multiples of 16, bases 16-byte aligned.  The forward epilogue of evlm_gemm_args applies to the scaled accumulator:
 *   bias, alpha q-scale, activation (quick-GELU / erf-GELU, optional aux_out), fp32 or bf16 residual, fp32 or bf16 D.  Everything else —
 *   epi_mode != FORWARD, dropout, splits > 1, accumulate, gates, device-side limits, MN-major operands — returns EVLM_EINVAL.
 *   M <= 32: weight-stream kernel (16-byte lane loads of 16 e4m3); otherwise tcgen05.mma.kind::f8f6f4 with 128-element k blocks. */
int evlm_quant_rows_e4m3(const void* x, int32_t x_dtype, int64_t ldx, int64_t rows, int64_t cols, void* q, int64_t ldq, float* scale,
                         void* stream);
int evlm_gemm_fp8(const evlm_gemm_args* args, const float* a_scale, const float* b_scale, void* stream);

/* fp32 SIMT contraction for the tiny, precision-critical products (ITC similarity xvlm.py:397-399 and
 * its backward): D[M,N] = alpha * A[M,K] * op(B) (+ beta*D), b_trans=1: B is [N,K]; 0: B is [K,N];
 * a_trans=1: A is [K,M]. */
int evlm_sgemm(int M, int N, int K, float alpha, const float* A, int64_t lda, int a_trans, const float* B, int64_t ldb,
               int b_trans, float beta, float* D, int64_t ldd, const float* alpha_dev, int alpha_dev_inv, void* stream);
/* alpha_dev (device scalar, may be NULL): effective alpha = alpha * alpha_dev[0] (or alpha / alpha_dev[0] when
 * alpha_dev_inv): the learnable ITC temperature (xvlm.py:399) is applied without a host read-back.
 * out[0] (+)= scale * sum_i x[i]*y[i]                                                                */
int evlm_dot(const float* x, const float* y, int64_t n, float scale, float* out, int32_t accumulate, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Elementwise / layout kernels (HBM-bound)
 * -----------------------------------------------------------------------------------------------*/
/* dst_bf16[i] = src_f32[i]; optional dropout-mask replay (p>0): dst = keep ? src/(1-p) : 0 with the
 * same (seed, stream, index) stream the forward epilogue used; rows x cols with leading dims.       */
int evlm_cast_f32_to_bf16(const float* src, int64_t lds, void* dst, int64_t ldd, int64_t rows, int64_t cols, float dropout_p,
                          uint64_t seed, uint32_t stream_id, void* stream);
/* dst_bf16[r, c] = src_f32[r, c] for every table entry, one launch (src dense [rows, cols], dst row pitch ldd elements); the table
 * lives in device memory (the bf16 weight shadows of a whole optimizer are refreshed this way after each step). */
typedef struct evlm_cast_entry {
  const float* src; void* dst; int64_t rows, cols, ldd;
} evlm_cast_entry;
int evlm_cast_table(const evlm_cast_entry* table_dev, int32_t n, void* stream);
int evlm_cast_bf16_to_f32(const void* src, int64_t lds, float* dst, int64_t ldd, int64_t rows, int64_t cols, void* stream);
/* out[n] (+)= sum_m X[m,n]   (bias / gate gradients: column sums of a [rows, cols] matrix).          */
int evlm_colsum(const void* X, int32_t x_dtype, int64_t ldx, int64_t rows, int64_t cols, float* out, int32_t accumulate,
                void* stream);
/* Zero-skip index work (eff_vit.py:214-219, eff_bert.py:553-557 multiply by z; columns with z == 0 contribute nothing forward and,
 * because the hard-concrete clamp has zero slope there (xvlm_l0_module.py:239-271), nothing backward either):
 *   evlm_compact_index: idx[0..count) = ascending positions j with z[j] != 0, idx[count..n) = the remaining positions (ascending),
 *                       count[0] = number kept.  n <= 65536.  Bit-exact index work, no host read-back.
 *   evlm_gather_rows:   dst[j, :] = j < count ? src[idx[j], :] : 0      (rows x cols, dtype EVLM_BF16 | EVLM_F32; a vector is cols = 1)
 *   evlm_gather_cols_bf16: dst[:, j] = j < count ? src[:, idx[j]] : 0
 *   evlm_scatter_rows_add: dst[idx[j], :] (+)= src[j, :] for j < count  (fp32; `accumulate` = 0 also ZEROES the rows not kept)
 *   evlm_scatter_cols_add: dst[:, idx[j]] (+)= src[:, j] for j < count  (fp32; same)                                              */
int evlm_compact_index(const float* z, int32_t n, int32_t* idx, int32_t* count, void* stream);
int evlm_gather_rows(const void* src, int64_t lds, int32_t dtype, const int32_t* idx, const int32_t* count, void* dst, int64_t ldd,
                     int64_t rows, int64_t cols, void* stream);
int evlm_gather_cols_bf16(const void* src, int64_t lds, const int32_t* idx, const int32_t* count, void* dst, int64_t ldd, int64_t rows,
                          int64_t cols, void* stream);
int evlm_scatter_rows_add(const float* src, int64_t lds, const int32_t* idx, const int32_t* count, float* dst, int64_t ldd, int64_t rows,
                          int64_t cols, int32_t accumulate, void* stream);
int evlm_scatter_cols_add(const float* src, int64_t lds, const int32_t* idx, const int32_t* count, float* dst, int64_t ldd, int64_t rows,
                          int64_t cols, int32_t accumulate, void* stream);
/* out[n] = sum_m X[m,n]*Y[m,n]  (bf16 inputs)  — dL/d head_layer_z style products.                   */
int evlm_coldot(const void* X, const void* Y, int64_t ld, int64_t rows, int64_t cols, float* out, void* stream);

/* Standalone activations for the small heads (nn.GELU in build_mlp xvlm.py:77-83; transform_act_fn eff_bert.py:724):
 * y = act(x); dx = dy * act'(x).  Any mix of fp32 / bf16 buffers (dtype flags), n elements, contiguous.   */
int evlm_act_fwd(const void* x, int32_t x_dtype, void* y, int32_t y_dtype, int64_t n, int32_t act, void* stream);
int evlm_act_bwd(const void* dy, int32_t dy_dtype, const void* x, int32_t x_dtype, void* dx, int32_t dx_dtype, int64_t n, int32_t act,
                 void* stream);

/* ViT patchify: image fp32 [B,3,R,R] -> bf16 patches [B*(R/16)^2, 3*16*16] in conv-weight order
 * (c, ky, kx) so that patches x W_pe[768, 768]^T equals Conv2d(3,768,16,16) (eff_vit.py:394-396,445). */
int evlm_im2col_patch(const float* image, void* patches, int B, int C, int R, int P, void* stream);
/* h[b,0,:] = cls + pos[0]; h[b,1+p,:] = patch[b,p,:] + pos[1+p]   (eff_vit.py:448-450), fp32 out.     */
int evlm_vit_assemble_fwd(const void* patch_emb /*bf16 [B*(N-1),H]*/, const float* cls, const float* pos, float* out, int B,
                          int N, int H, void* stream);
/* backward: dpatch (bf16) = dh[:,1:,:]; dcls += sum_b dh[b,0]; dpos[n] += sum_b dh[b,n].              */
int evlm_vit_assemble_bwd(const float* dh, void* dpatch, float* dcls, float* dpos, int B, int N, int H, void* stream);

/* BERT embeddings sum: out[b,l,:] = word[ids[b,l]] + type[tt[b,l]] + pos[pos_ids or l+past]  (eff_bert.py:204-212) */
int evlm_bert_embed_fwd(const int64_t* ids, const int64_t* type_ids, const int64_t* pos_ids, const float* word, const float* type,
                        const float* pos, float* out, int64_t rows, int L, int H, int past_len, int64_t vocab, void* stream);
int evlm_bert_embed_bwd(const float* dout, const int64_t* ids, const int64_t* type_ids, const int64_t* pos_ids, float* dword,
                        float* dtype, float* dpos, int64_t rows, int L, int H, int past_len, int64_t padding_idx, void* stream);
/* padding_idx: word row that receives no look-up gradient (nn.Embedding(padding_idx=pad_token_id), eff_bert.py:173); -1 = none */

/* ------------------------------------------------------------------------------------------------
 * LayerNorm (+ dropout) — eff_vit.py:252,264,452,467; eff_bert.py:213-214,380,461,725
 *   y = LN(x) * gamma + beta ; optional dropout on y (embeddings).  x: fp32 or bf16; y: fp32 and/or bf16.
 * -----------------------------------------------------------------------------------------------*/
int evlm_layernorm_fwd(const void* x, int32_t x_dtype, const float* gamma, const float* beta, float eps, float* y_f32,
                       void* y_bf16, float* mean, float* rstd, int64_t rows, int H, float dropout_p, uint64_t seed,
                       uint32_t stream_id, void* stream);
/* dx = LN'(dy) (+ dres); dy fp32 or bf16; writes dx fp32 and/or bf16; dgamma/dbeta are ACCUMULATED (+=).
 * If dropout_p>0 the forward's output dropout mask is replayed on dy first.                          */
int evlm_layernorm_bwd(const void* dy, int32_t dy_dtype, const void* x, int32_t x_dtype, const float* gamma, const float* mean,
                       const float* rstd, const float* dres, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta,
                       int64_t rows, int H, float dropout_p, uint64_t seed, uint32_t stream_id, void* stream);
/* ABI v6: as above, plus what the Linear layer IN FRONT of the LayerNorm needs from this pass (eff_bert.py:375-381: dense -> dropout ->
 * + residual -> LayerNorm): dx_bf16 = dropout-mask(out_dropout_p, seed, out_stream_id) applied to dx (the mask that Linear's output got in
 * the forward), and dcolsum[H] += column sums of dx_bf16 (= that Linear's bias gradient).  H % 128 == 0, H <= 1024, dx_bf16 required;
 * otherwise EVLM_EUNSUPPORTED (the caller then casts / sums separately). */
int evlm_layernorm_bwd_ex(const void* dy, int32_t dy_dtype, const void* x, int32_t x_dtype, const float* gamma, const float* mean,
                          const float* rstd, const float* dres, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta, int64_t rows,
                          int H, float dropout_p, uint64_t seed, uint32_t stream_id, float out_dropout_p, uint32_t out_stream_id,
                          float* dcolsum, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Fused multi-head attention, head_dim 64 — eff_vit.py:141-197; eff_bert.py:297-359.
 *   S = q k^T * scale (+ key_mask[b, j]) (+ causal) ; P = softmax(S) -> optional fp32 write-out
 *   ctx = dropout(P) v ; ctx *= head_z[h]
 * q: rows of [B, Lq] with row stride ldq elements, head h at column offset h*64 (same for k, v, ctx).
 * -----------------------------------------------------------------------------------------------*/
typedef struct evlm_attn_args {
  int32_t B, H, Lq, Lk;                            /* head_dim fixed 64 */
  const void* q; int64_t ldq;                      /* bf16 */
  const void* k; int64_t ldk;
  const void* v; int64_t ldv;
  void* ctx; int64_t ldc;                          /* bf16 [B*Lq, H*64] */
  float* probs;                                    /* fp32 [B,H,Lq,Lk] or NULL (fwd: out, bwd: in) */
  float* lse;                                      /* fp32 [B,H,Lq] row log-sum-exp (used when probs==NULL) */
  const float* key_mask;                           /* additive fp32 [B, Lk] or NULL */
  const float* full_mask;                          /* additive fp32 [B, Lq, Lk] or NULL (region batches) */
  int32_t causal; int32_t causal_offset;           /* key j allowed iff j <= i + causal_offset, else -10000 */
  float scale;
  const float* head_z;                             /* [H] or NULL */
  float dropout_p; uint64_t dropout_seed; uint32_t dropout_stream;
  /* backward only */
  const void* dctx; int64_t lddc;                  /* bf16 */
  const float* dprobs_ext;                         /* fp32 [B,H,Lq,Lk] or NULL: gradient arriving on the returned P */
  void* dq; int64_t lddq; void* dk; int64_t lddk; void* dv; int64_t lddv; /* bf16 out */
  float* dhead_z;                                  /* [H], accumulated (+=) or NULL */
  float* dkv_accum;                                /* fp32 workspace [2, B, H, Lk, 64] (zeroed by callee) */
  /* shared keys/values (ABI v2): query item b attends to K/V batch item kv_index[b] (int32 [B], NULL: b itself), k and v
   * then hold kv_batches*Lk rows.  Cross-attention of the ITM / MLM rows to the SAME image tokens (xvlm.py:465-476 re-feeds
   * image_embeds for every text row) needs the K/V projection once per image instead of once per row.  dk / dv stay per
   * query item ([B*Lk] rows): evlm_index_add_rows folds them back per K/V item.                                        */
  const int32_t* kv_index; int32_t kv_batches;
  /* packed query items (ABI v3, tcgen05 kernels only): a 40-token text sequence fills 31 % of the 128-row query tile, so up to
   * pack_width (<= 3, pack_width * Lq <= 128, Lq % 8 == 0) query items that attend to the SAME K/V item share one CTA:
   * pack_items int32 [pack_groups, pack_width] lists them (-1 = empty slot, first slot valid); the group's K/V item is
   * kv_index[first item] (or the first item itself).  q / ctx / probs / lse / dq stay per item; dk / dv are written per
   * GROUP ([pack_groups * Lk] rows: the sum over the group's items).                                                   */
  const int32_t* pack_items; int32_t pack_groups; int32_t pack_width;
  /* pack_own_kv = 1 (self-attention of short sequences, needs Lk % 8 == 0 and pack_width * Lk <= 128): every packed item
   * brings its OWN K/V rows; the tile is the block-diagonal attention of the pack (keys of other members are masked to
   * exactly zero probability), dk / dv are written per item like dq.  0: the members share one K/V item (above).           */
  int32_t pack_own_kv;
  /* ABI v6: row pitch (floats) of probs / dprobs_ext; 0 = Lk (dense).  The Python side allocates the maps with the pitch rounded up to 4
   * floats (197 -> 200) and hands the reference API a [..., :Lk] view: rows then start on 16-byte boundaries, so the forward can
   * leave the normalised probabilities as TMA box stores and every consumer can use vector accesses.  Pad columns are written as 0. */
  int64_t ldp;
  /* ABI v6, backward: fp32 [B, H, Lq] = sum_j dprobs_ext[.., j] * probs[.., j] supplied by the producer of dprobs_ext (the KD MSE
   * backward, evlm_mse_pair.rowdot); NULL: computed here by reading both maps.  (With dp_kd_coef: see below.) */
  const float* dp_rowdot;
  /* ABI v7, forward with Lq == 1 only (single-token decode steps, csrc/attention_decode.cu): K / V rows of item b start at row
   * kv_item(b) * kv_item_rows instead of kv_item(b) * Lk — a pre-allocated KV cache [items, capacity, ...] of which the first Lk rows
   * per item are valid.  0 = Lk.  Every other kernel answers EVLM_EUNSUPPORTED to a value that differs from Lk. */
  int64_t kv_item_rows;
  /* ABI v7, backward, attention-map distillation without a materialised gradient: with dp_kd_coef (DEVICE scalar) set, `dprobs_ext`
   * holds the TARGET map T (the teacher's, same layout as probs) and the gradient arriving on the returned map is
   * dP = dp_kd_coef[0] * (P - T), formed on the fly from the re-computed P (GeneralDistill.py:60-82: d/dP of scale * mean((P - T)^2),
   * coefficient = upstream gradient * 2 * scale / numel).  `dp_rowdot` is then required and holds the UNSCALED row sums
   * sum_j (P_ij - T_ij) P_ij (left by evlm_mse_pairs_fwd, evlm_mse_pair.rowdot).  Needs dropout_p == 0; tcgen05 kernels only
   * (EVLM_EUNSUPPORTED otherwise: the caller materialises dP). */
  const float* dp_kd_coef;
} evlm_attn_args;
/* ABI v7 — greedy token selection of the decode loop (eff_bert.py:1510-1538 with do_sample = False, repetition_penalty = 1), one launch per
 * decoded token: next_token[r] = argmax_j logits[r, j] (first maximal index); score[r] = log_softmax(logits[r])[next_token[r]];
 * tokens_to_add[r] = next * unfinished[r] + pad * (1 - unfinished[r]); unfinished_out[r] = unfinished[r] * prod_e (tokens_to_add[r] != eos[e]).
 * logits fp32 [rows, ld]; the int64 vectors have `rows` entries; eos_host: n_eos <= 4 ids in HOST memory. */
int evlm_greedy_select(const float* logits, int64_t ld, int32_t rows, int32_t vocab, const int64_t* unfinished, int64_t pad,
                       const int64_t* eos_host, int32_t n_eos, int64_t* next_token, float* score, int64_t* tokens_to_add,
                       int64_t* unfinished_out, void* stream);
/* ABI v8 — beam search on the device (transformers 4.12.5's beam_search / BeamSearchScorer / BeamHypotheses, as restated by
 * eff_bert.py::BertLMHeadModel._beam_search and oracle/beam_search_oracle.py).  rows = batch * beams, 2 <= beams <= 8.
 * Loop state (device): tokens int64 [rows, width] (history, prompt pre-filled), beam_scores fp32 [rows], beam_src int32 [rows] (source
 * beam inside the item), done int32 [batch], hyp_tokens int64 [batch, beams, width], hyp_len int32 [batch, beams], hyp_score fp64
 * [batch, beams], hyp_count int32 [batch], hyp_worst fp64 [batch] (initially 1e9).  Hypothesis scores are fp64, like the host's floats;
 * cur_len_pow = cur_len ** length_penalty, computed by the caller (the host's own pow), divides every score of the call.
 * evlm_beam_step: one decode position at history length cur_len (< width) from the step's fp32 logits [rows, ld]: log-softmax,
 *   repetition penalty on the log-probabilities of every token in the row's history, eos -> -inf while cur_len < min_length, + beam
 *   score, top 2 * beams over beams x vocab (ties: lowest flat index), BeamSearchScorer.process, BeamHypotheses.add / is_done; the
 *   history is re-ordered inside the item and the new token written at column cur_len.  Finished items keep their rows (identity
 *   source, pad token, score 0).  Requires vocab > 2 * beams. */
int evlm_beam_step(const float* logits, int64_t ld, int32_t batch, int32_t beams, int32_t vocab, int32_t cur_len, int32_t min_length,
                   float repetition_penalty, double cur_len_pow, int32_t early_stopping, int64_t eos, int64_t pad, int64_t* tokens,
                   int64_t width, float* beam_scores, int32_t* beam_src, int32_t* done, int64_t* hyp_tokens, int32_t* hyp_len,
                   double* hyp_score, int32_t* hyp_count, double* hyp_worst, void* stream);
/* BeamSearchScorer.finalize after the last step (history length cur_len <= width): unfinished items add their live beams; out int64
 * [batch, max_length] (max_length <= width) = best hypothesis (last of the maximal scores in list order), eos if it is shorter than
 * max_length, then pad; out_len int32 [batch] = its length. */
int evlm_beam_finalize(const int64_t* tokens, int64_t width, const float* beam_scores, const int32_t* done, int32_t batch, int32_t beams,
                       int32_t cur_len, int32_t max_length, double cur_len_pow, int64_t eos, int64_t pad, int64_t* hyp_tokens,
                       int32_t* hyp_len, double* hyp_score, int32_t* hyp_count, double* hyp_worst, int64_t* out, int32_t* out_len,
                       void* stream);
/* In-place re-order of `layers` self-attention KV caches (bf16 [batch * beams, capacity, row_elems], row_elems % 8 == 0, 16-byte
 * aligned; caches_host: HOST array of device pointers) in one launch: for positions < len, row r takes the row of item(r) * beams +
 * beam_src[r] (0 <= beam_src < beams).  Positions >= len are untouched. */
#define EVLM_KV_REORDER_MAX_LAYERS 32
int evlm_kv_beam_reorder(void* const* caches_host, int32_t layers, int32_t batch, int32_t beams, int64_t capacity, int64_t row_elems,
                         int32_t len, const int32_t* beam_src, void* stream);
/* dst[index[i], :] += src[i, :]  (src bf16 [n_src, row_elems], dst fp32 [n_dst, row_elems] pre-zeroed by the caller; fp32 red.add) */
int evlm_index_add_rows(const void* src_bf16, const int32_t* index, float* dst, int64_t n_src, int64_t row_elems, void* stream);
/* deterministic variant without atomics on the data: dst_bf16[u, :] = sum_{i: index[i]==u} src_bf16[i, :] (fp32 accumulate);
 * workspace: int32 [2*n_dst + 1 + n_src] (CSR lists built on the device)                                                    */
int evlm_index_fold_rows(const void* src_bf16, const int32_t* index, int64_t n_src, int64_t n_dst, int64_t row_elems, void* dst_bf16,
                         int32_t* workspace, void* stream);
int evlm_attention_fwd(const evlm_attn_args* a, void* stream);
int evlm_attention_bwd(const evlm_attn_args* a, void* stream);
size_t evlm_attention_bwd_workspace(const evlm_attn_args* a);

/* ------------------------------------------------------------------------------------------------
 * Losses — GeneralDistill.py:60-89; xvlm.py:397-416,479-483; eff_bert.py:1263-1302,1699-1702
 * -----------------------------------------------------------------------------------------------*/
/* Multi-pair MSE in ONE launch: for each pair p: out[p] = mean((s_p - t_p)^2) * scale[p].
 * Tensors may be fp32 or bf16 (per-pair dtype flags). Pair table lives in device memory.            */
typedef struct evlm_mse_pair {
  const void* s; const void* t; void* ds; /* ds: gradient buffer (same dtype as s... always fp32) or NULL */
  int64_t n; float scale; int32_t s_dtype; int32_t t_dtype; int32_t pad;
  /* ABI v6, backward only: when rowdot != NULL the pair is an attention map with rows of row_len elements (row_len % 4 == 0, n %
   * row_len == 0) and rowdot[r] += sum_j ds[r, j] * s[r, j] — the "sum_j dP_ij P_ij" term of the softmax backward, produced here
   * from values that are in registers anyway instead of by a pre-kernel that re-reads both maps (evlm_attn_args.dp_rowdot).
   * The forward leaves rowdot[r] = sum_j (s - t)[r, j] * s[r, j] (unscaled) on every path; rowdot must arrive zeroed.            */
  float* rowdot; int64_t row_len;
} evlm_mse_pair;
int evlm_mse_pairs_fwd(const evlm_mse_pair* pairs_dev, int npairs, float* out /*[npairs], zeroed by callee*/, void* stream);
/* ds_p = dout[p] * scale[p] * 2 (s_p - t_p) / n_p   (fp32 ds)                                        */
int evlm_mse_pairs_bwd(const evlm_mse_pair* pairs_dev, int npairs, const float* dout /*[npairs]*/, void* stream);

/* Row-wise softmax cross-entropy with hard labels (ignore_index), label smoothing, optional per-row
 * output; also produces row max / log-sum-exp for the backward.
 *   loss_row = -(1-ls)*logp[label] - ls/V * sum_v logp[v]      (LabelSmoothSoftmaxCEV1, eff_bert.py:1263-1302)
 * out_rows[r] (0 for ignored rows); n_valid counted on device.                                        */
int evlm_xent_fwd(const float* logits, int64_t ld, int64_t rows, int V, const int64_t* labels, int64_t ignore_index,
                  float label_smoothing, float* loss_rows, float* lse, void* stream);
/* dlogits[r,v] (+)= g_row[r] * (softmax - target)  written fp32 (ld_d) and/or bf16 (ld_b).            */
int evlm_xent_bwd(const float* logits, int64_t ld, int64_t rows, int V, const int64_t* labels, int64_t ignore_index,
                  float label_smoothing, const float* lse, const float* g_rows, float* dlogits, int64_t ld_d, int32_t accumulate,
                  void* stream);
/* Soft-target CE / KL (soft_cross_entropy, GeneralDistill.py:84-89):
 *   kl_row = sum_v softmax(t/T)_v * (log softmax(t/T)_v - log softmax(s/T)_v)                           */
int evlm_kl_fwd(const float* s_logits, const float* t_logits, int64_t ld_s, int64_t ld_t, int64_t rows, int V, float inv_temp,
                float* kl_rows, float* lse_s, float* lse_t, void* stream);
int evlm_kl_bwd(const float* s_logits, const float* t_logits, int64_t ld_s, int64_t ld_t, int64_t rows, int V, float inv_temp,
                const float* lse_s, const float* lse_t, const float* g_rows, float* dlogits, int64_t ld_d, int32_t accumulate,
                void* stream);
/* Soft-label CE used by ITC with idx (xvlm.py:404-416): loss_row = -sum_v labels[r,v]*logp[r,v]; labels fp32 dense. */
int evlm_soft_xent_fwd(const float* logits, int64_t ld, const float* labels, int64_t ld_l, int64_t rows, int V, float* loss_rows,
                       float* lse, void* stream);
int evlm_soft_xent_bwd(const float* logits, int64_t ld, const float* labels, int64_t ld_l, int64_t rows, int V, const float* lse,
                       const float* g_rows, float* dlogits, int64_t ld_d, int32_t accumulate, void* stream);
/* sum / mean helpers over fp32 vectors (loss assembly without torch reductions): out[0] (+)= scale*sum(x) */
int evlm_reduce_sum(const float* x, int64_t n, float scale, float* out, int32_t accumulate, void* stream);
/* L2 row normalisation F.normalize(x, dim=-1) (xvlm.py:375-382) fwd/bwd, fp32.                        */
int evlm_l2norm_fwd(const float* x, float* y, float* inv_norm, int64_t rows, int D, void* stream);
int evlm_l2norm_bwd(const float* dy, const float* y, const float* inv_norm, float* dx, int64_t rows, int D, void* stream);
/* ITM hard-negative sampling on device (xvlm.py:422-455 without the 2B host syncs): for each row b,
 * weights = softmax(sim[b,:]) + 1e-5 with excluded entries (same idx / diagonal) zeroed, one multinomial
 * draw per row from u[b] in [0,1).  neg_out int64 [B].                                                 */
int evlm_itm_sample_neg(const float* sim, int64_t ld, const int64_t* idx /*[B] or NULL*/, const float* u, int64_t* neg_out,
                        int B, void* stream);

/* ------------------------------------------------------------------------------------------------
 * L0 hard-concrete gates — xvlm_l0_module.py:174-271,321-341
 * -----------------------------------------------------------------------------------------------*/
/* z = clamp(sigmoid((log u - log(1-u) + loga)/beta) * (r-l) + l, 0, 1)  with l=-0.1, r=1.1             */
int evlm_l0_sample_fwd(const float* loga, const float* u, float* z, int64_t n, float temperature, void* stream);
int evlm_l0_sample_bwd(const float* loga, const float* u, const float* dz, float* dloga, int64_t n, float temperature,
                       void* stream);
/* score = 1 - clamp(sigmoid(beta*log(-l/r... ) - loga), eps, 1-eps); out[0] (+)= weight * sum(score)    */
int evlm_l0_expected_fwd(const float* loga, int64_t n, float temperature, float weight, float* out, int32_t accumulate,
                         void* stream);
/* dloga += g[0] * weight * dscore/dloga                                                              */
int evlm_l0_expected_bwd(const float* loga, int64_t n, float temperature, float weight, const float* g, float* dloga,
                         void* stream);
/* Deterministic eval mask per layer row (bit-exact with _deterministic_z): for each of `layers` rows of
 * `size` entries: n0 = round_half_even(size - sum(score)); zero the n0 smallest soft = sigmoid(loga/beta*magic)
 * (ties broken by lower index first, as torch.topk(largest=False) on CPU does).                          */
int evlm_l0_deterministic(const float* loga, float* mask, int32_t* kept_count, int layers, int size, float temperature,
                          float magical_number, void* stream);
/* loga.clamp_(log 0.01, log 100)  (constrain_parameters, xvlm_l0_module.py:168-172)                      */
int evlm_clamp_(float* x, int64_t n, float lo, float hi, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Optimizer over a flat fp32 arena — optim.py:23-69 (HF AdamW semantics: decoupled decay applied
 * AFTER the Adam update, bias correction on), apex_ddp_accelerator.py:98-101 (global-norm clip).
 * -----------------------------------------------------------------------------------------------*/
/* out[0] += sum(x^2).  Deterministic (fixed-order two-level reduction, no float atomics): data-parallel replicas must derive
 * bit-identical clip coefficients from bit-identical all-reduced gradients.  Calls must be ordered on one stream. */
int evlm_sumsq(const float* x, int64_t n, float* out /*[1], accumulated*/, void* stream);
typedef struct evlm_adamw_group {
  float* p; float* g; float* m; float* v; void* p_bf16; /* bf16 shadow or NULL */
  int64_t n; float lr; float beta1; float beta2; float eps; float weight_decay; int32_t step; int32_t pad;
} evlm_adamw_group;
/* grad_scale_dev: device scalar multiplied into every gradient (clip coefficient / loss-scale), or NULL */
int evlm_adamw_step(const evlm_adamw_group* groups_host, int ngroups, const float* grad_scale_dev, void* stream);
/* coef[0] = min(1, max_norm / (sqrt(sumsq[0]) + 1e-6))                                                  */
int evlm_clip_coef(const float* sumsq, float max_norm, float* coef, void* stream);

/* ---- CUDA-graph support: everything a replayed training step must be able to change lives in device memory ----
 * (the reference's train loop, Train.py / accelerators/apex_ddp_accelerator.py:84-101, re-issues every launch from
 * Python each step; a captured step replays fixed launches, so per-step scalars move behind device pointers.)
 * evlm_adamw_step_dev: like evlm_adamw_step, but group i takes step_size = hyper_dev[2i] (lr*sqrt(1-b2^t)/(1-b1^t))
 *   and its decoupled decay factor lr*wd = hyper_dev[2i+1] from device memory (lr/step fields of the groups ignored).
 * evlm_store_f32: dst_dev[0..n) = values_host[0..n), n <= 32, values travel as launch arguments (stream ordered,
 *   no pinned staging buffer to keep alive) - the eager refresh of hyper_dev before a replay.
 * evlm_rng_bind: every dropout site adds *state_dev to its by-value seed (NULL unbinds; default unbound = +0).
 *   Synchronous, call once outside capture.   evlm_rng_advance: *state_dev = set ? delta : *state_dev + delta
 *   as a one-thread launch (capturable: a graph advances its own dropout stream at its first node).            */
int evlm_adamw_step_dev(const evlm_adamw_group* groups_host, int ngroups, const float* grad_scale_dev, const float* hyper_dev,
                        void* stream);
int evlm_store_f32(float* dst_dev, const float* values_host, int32_t n, void* stream);
int evlm_rng_bind(const uint64_t* state_dev);
int evlm_rng_advance(uint64_t* state_dev, uint64_t delta, int32_t set, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EVLM_H_ */
