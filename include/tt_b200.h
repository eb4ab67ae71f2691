/*
 * tt_b200.h — C ABI of the B200-native two-tower hot path (libtt_b200.so).
 *
 * The reference (DiegoPaniagua23/music-recommendation-multimodal) has no FFI of its
 * own: its hot path is PyTorch library calls inside three nn.Modules and two loops.
 * Each entry point below names the reference call site (file:line under the
 * reference root) whose device work it replaces.
 *
 * Conventions (all entry points):
 *   - return 0 on success, non-zero on error; tt_last_error() returns the message
 *     for the calling thread;
 *   - every pointer is a DEVICE pointer owned by the caller unless the name ends in
 *     _host; sizes are explicit; matrices are row-major with an explicit leading
 *     dimension in ELEMENTS;
 *   - no allocation, no host synchronisation, no global mutable state: launches go
 *     to the caller's stream (a cudaStream_t passed as void*) and are CUDA-graph
 *     capturable;
 *   - "bf16" buffers are raw uint16 bfloat16 bit patterns.
 */
#ifndef TT_B200_H_
#define TT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TT_B200_VERSION 1

/* ---- library ------------------------------------------------------------------ */
const char* tt_last_error(void);
int tt_version(void);
int tt_num_sms(void);

/* ---- dense contraction on tcgen05 ------------------------------------------------
 * C[M,N] = epilogue( alpha * sum_k A[m,k] * B[n,k] )
 *
 * Replaces every cuBLAS GEMM the reference reaches through nn.Linear /
 * nn.MultiheadAttention in_proj/out_proj (src/models/user_tower.py:37-57,
 * src/models/item_tower.py:121-129), torch.matmul for the InfoNCE logits
 * (src/models/two_tower.py:106) and their autograd dgrad/wgrad counterparts
 * (src/train.py:63).
 *
 * Operand layouts (bf16):
 *   a_mn = 0 : A is [M, lda]  (K contiguous;  "K-major")
 *   a_mn = 1 : A is [K, lda]  (M contiguous; "MN-major", i.e. A^T stored) — M % 8 == 0
 *   b_mn = 0 : B is [N, ldb]  (K contiguous; nn.Linear weight layout)
 *   b_mn = 1 : B is [K, ldb]  (N contiguous) — N % 8 == 0
 *   MN-major operands are fetched in 64-element chunks: when M (N) is not a multiple of 64 the
 *   last chunk of each K row reads past it (values never stored), so the buffer must stay
 *   readable up to the next multiple of 64 after its last row.
 * Epilogue, applied in this order to v = alpha * acc:
 *   v += bias[n]; relu; dropout(seed, site, m*N+n); gate (v = gate[m,n] > 0 ? v*gate_scale : 0);
 *   v += residual[m,n]; store fp32 (optionally atomically accumulated) and/or bf16.
 */
typedef struct tt_gemm_args {
  const void* A;
  const void* B;
  int32_t lda, ldb;
  int32_t a_mn, b_mn;
  int32_t M, N, K;
  float alpha;
  const float* bias;       /* [N] or NULL */
  int32_t relu;
  float drop_p;            /* 0 => no dropout */
  uint64_t drop_seed;
  const uint64_t* drop_seed_dev; /* optional device scalar added to drop_seed (graph replay) */
  uint32_t drop_site;
  const void* gate;        /* bf16 [M, ld_gate] or NULL */
  int32_t ld_gate;
  float gate_scale;
  const float* residual;   /* fp32 [M, ld_res] or NULL */
  int32_t ld_res;
  float* out_f32;          /* fp32 [M, ld_f32] or NULL */
  int32_t ld_f32;
  void* out_bf16;          /* bf16 [M, ld_bf16] or NULL */
  int32_t ld_bf16;
  int32_t accumulate;      /* 1: out_f32 += (red.add), required when k_splits > 1 */
  int32_t k_splits;        /* 0 => choose automatically (only >1 when accumulate) */
  int32_t block_n;         /* 0 => choose automatically (64/128/256) */
  float* a_colsum;         /* optional fp32 [K]: a_colsum[k] += sum_m A[m,k] (K-major A, no split-K, K <= 2048): the bias
                            * gradient sum(dY, dim=0) that autograd's Linear backward (src/models/user_tower.py:37-45
                            * layers, src/train.py:62) takes next to dX = dY W, here from the dY tiles the dgrad GEMM
                            * stages anyway instead of a second pass over dY */
} tt_gemm_args;

int tt_gemm_bf16(const tt_gemm_args* args, void* stream);

/* ---- causal self-attention, d_head = 64 -------------------------------------------
 * Replaces F.scaled_dot_product_attention inside nn.TransformerEncoderLayer
 * (src/models/user_tower.py:37-45, 111-116) for right-padded histories.
 *   qkv  : bf16 [B*L, 3*H*64], columns [Q | K | V], head h at h*64 inside each third
 *          (the packed in_proj output, rows [Q;K;V] of in_proj_weight)
 *   ctx  : bf16 [B*L, H*64]     attention output before out_proj
 *   lse  : fp32 [B, H, L]       natural-log sum-exp of the scaled scores (for backward)
 * Dropout (p > 0) is applied to the attention probabilities with the counter-based hash
 * (seed + *seed_dev, site, ((b*H+h)*L+i)*L+j). L <= 4096: L <= 512 keeps every tile of a sequence on chip;
 * 512 < L <= 4096 runs the tiled kernels (online-softmax forward; a deterministic backward in two kernels, one per key
 * tile for dK / dV and one per query tile for dQ), which hash the element index in 64 bits. B*L <= 2^31 - 1.
 */
int tt_attn_causal_fwd(const void* qkv, void* ctx, float* lse, int B, int L, int H, float drop_p,
                       uint64_t drop_seed, const uint64_t* drop_seed_dev, uint32_t drop_site, void* stream);
int tt_attn_causal_bwd(const void* qkv, const void* ctx, const void* dctx, const float* lse,
                       void* dqkv, int B, int L, int H, float drop_p, uint64_t drop_seed,
                       const uint64_t* drop_seed_dev, uint32_t drop_site, void* stream);

/* ---- bandwidth-bound row-wise kernels ------------------------------------------------
 * Dropout everywhere is the counter-based hash of (seed [+ *seed_dev], site, element index);
 * the same triple in forward and backward reproduces the mask, so no mask is stored.
 */

/* fp32 -> bf16 copy of n (multiple of 4) elements: tensor-core operand shadows of the dense
 * weights (the reference's autocast casts, src/train.py:57). */
int tt_cast_bf16(const float* src, void* dst_bf16, int64_t n, void* stream);

/* last_idx[b] = max(sum(mask[b,:] != 0) - 1, 0); mask == NULL uses ids != 0
 * (src/models/user_tower.py:122-128). ids/mask int64 [B, L]. */
int tt_last_index(const int64_t* ids, const int64_t* mask, int B, int L, int32_t* last_idx, void* stream);

/* x0 = dropout(LayerNorm(E[ids] + P[pos])) fp32 [B*L,256]; h = LayerNorm_next(x0) bf16.
 * Replaces nn.Embedding lookup + positional add + layer_norm + dropout
 * (src/models/user_tower.py:86-93) and the first encoder norm1. */
int tt_embed_ln_fwd(const int64_t* ids, const float* E, const float* P, const float* ln_w, const float* ln_b,
                    const float* next_w, const float* next_b, int B, int L, float drop_p, uint64_t seed,
                    const uint64_t* seed_dev, uint32_t site, float* x0, void* h_bf16, void* stream);

/* tt_embed_ln_fwd for n rows at explicit positions: row r is item ids[r] at position pos[r] (int32), local table,
 * no dropout (eval). x0 fp32 [n,256], h bf16 [n,256]; each row equal bit for bit to tt_embed_ln_fwd's row at the same
 * (id, position). Same reference lines (src/models/user_tower.py:86-93); used by the session append. */
int tt_embed_ln_fwd_pos(const int64_t* ids, const int32_t* pos, const float* E, const float* P, const float* ln_w,
                        const float* ln_b, const float* next_w, const float* next_b, int n, float* x0, void* h_bf16,
                        void* stream);

/* backward of the embedding LayerNorm + lookup: dx0 -> dE (scatter-add, row 0 skipped:
 * padding_idx, src/models/user_tower.py:26), dP, d(ln_w), d(ln_b); all accumulated. */
int tt_embed_ln_bwd(const int64_t* ids, const float* E, const float* P, const float* ln_w, const float* ln_b,
                    const float* dx0, int B, int L, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                    uint32_t site, float* dE, float* dP, float* dgamma, float* dbeta, void* stream);

/* Deterministic form of tt_embed_ln_bwd for the table gradient (the reference's embedding backward is
 * autograd's embedding_dense_backward, src/models/user_tower.py:26; its CUDA form is deterministic only under
 * torch.use_deterministic_algorithms). Token t adds its gradient row into acc64[slot_of_token[t]] (int64
 * [slots, 256], slot 0 = padding: skipped) in 64-bit fixed point, 2^-40 units: integer addition is associative,
 * so the sums do not depend on the order in which duplicate ids arrive and are bit-identical from run to run.
 * slot_of_token / the distinct-id list come from tt_ids_dedup; tt_rows_scatter_add_i64 rounds every sum once to
 * fp32, adds it to the table's gradient row (one writer per row) and clears the accumulator. dP / d(ln_w) /
 * d(ln_b) as in tt_embed_ln_bwd. */
int tt_embed_ln_bwd_det(const int64_t* ids, const float* E, const float* P, const float* ln_w, const float* ln_b,
                        const float* dx0, int B, int L, float drop_p, uint64_t seed, const uint64_t* seed_dev,
                        uint32_t site, const int64_t* slot_of_token, int64_t* acc64, float* dP, float* dgamma,
                        float* dbeta, void* stream);
int tt_rows_scatter_add_i64(float* grad_local, const int64_t* uniq, const int32_t* n_uniq, int max_rows,
                            int64_t* acc64, void* stream);

/* Row chain on fp32 rows of width 256 or 512:
 *   forward : [LayerNorm] -> [ReLU] -> [dropout] -> [L2 normalise] -> out_f32 / out_bf16
 *   backward: recomputes the forward from x, then dout -> ... -> (+resid) -> dx_f32 / dx_bf16,
 *             accumulating dgamma/dbeta and (optionally) the column sums of dx_bf16; dx_bf16 may
 *             receive a second dropout mask (drop2_*), the one of the residual branch it feeds.
 * Covers nn.LayerNorm, F.normalize, the user fusion LN+ReLU and the item LN+normalise
 * (src/models/user_tower.py:47,54-55; item_tower.py:128; two_tower.py:100-101). */
typedef struct tt_chain_args {
  const float* x;
  int32_t rows, width;
  const float* ln_w;
  const float* ln_b;
  float ln_eps;
  int32_t relu;
  float drop_p;
  uint64_t drop_seed;
  const uint64_t* drop_seed_dev;
  uint32_t drop_site;
  int32_t l2norm;
  float l2_eps;
  float* out_f32;
  void* out_bf16;
  /* backward */
  const float* dout;
  const float* resid;
  float* dx_f32;
  void* dx_bf16;
  float drop2_p;
  uint32_t drop2_site;
  float* dgamma;
  float* dbeta;
  float* dx_colsum;
  /* backward, sparse residual: instead of a dense `resid`, sequence b (rows [b*seq_len, (b+1)*seq_len)) adds
   * resid_rows[b, :] to its row b*seq_len + resid_last_idx[b] only — the residual-stream gradient of the
   * single-row last layer, which is non-zero for one position per sequence. Exclusive with `resid`. */
  const float* resid_rows;
  const int32_t* resid_last_idx;
  int32_t resid_seq_len;
  /* backward: the incoming gradient as bf16 [rows, width] instead of `dout` (exactly one of the two). Under
   * autocast the reference's Linear backward returns dX in bf16 (src/train.py:57-62), so a dgrad GEMM may hand
   * its result over in that type: half the bytes written there and read here. */
  const void* dout_bf16;
} tt_chain_args;
int tt_chain_fwd(const tt_chain_args* args, void* stream);
int tt_chain_bwd(const tt_chain_args* args, void* stream);

/* cat[b] = [x[b*L + last_idx[b], :256] | G[gender[b]] (16) | C[country[b]] (32)] as bf16 [B,304]
 * (src/models/user_tower.py:132-139) and its backward (dx must be zero-initialised). */
int tt_gather_cat_fwd(const float* x, const int32_t* last_idx, const int64_t* gender, const int64_t* country,
                      const float* G, const float* C, int B, int L, void* cat_bf16, void* stream);
int tt_gather_cat_bwd(const float* dcat, const int32_t* last_idx, const int64_t* gender, const int64_t* country,
                      int B, int L, float* dx, void* dx_bf16, float* dG, float* dC, void* stream);

/* [audio | visual | text | tabular] -> bf16 [B, 4*m] (src/models/item_tower.py:147). */
int tt_concat4_bf16(const float* audio, const float* visual, const float* text, const float* tabular, int B, int m,
                    void* out_bf16, void* stream);

/* Catalog-indexing tail (src/evaluate_metrics.py:70-102): y fp32 [R, 256] = output of the item tower's last Linear
 * -> LayerNorm (item_tower.py:128) -> F.normalize eps 1e-12 (two_tower.py:168) -> NaN -> 0 (:79-81) ->
 * F.normalize eps 1e-8 (:85) -> table[ids[r], :] (fp32, the reference's cache layout) and, when table_bf16 is
 * non-NULL, the bf16 copy the scoring kernel reads. ids must be distinct (the reference indexes unique_df);
 * ids outside [0, V) are skipped. Rows not listed are left untouched (the caller zero-fills the table once). */
int tt_index_rows(const float* y, int R, const float* ln_w, const float* ln_b, const int64_t* ids, int64_t V,
                  float* table, void* table_bf16, void* stream);

/* BatchNorm1d + ReLU + Dropout on fp32 [B, C] -> bf16 (src/models/item_tower.py:124-126).
 * training != 0: batch statistics, running stats / num_batches_tracked updated (momentum 0.1,
 * unbiased variance); else running statistics. */
typedef struct tt_bn_args {
  const float* y;
  int32_t B, C;
  const float* w;
  const float* b;
  float* running_mean;
  float* running_var;
  int64_t* num_batches_tracked;
  int32_t training;
  float momentum, eps;
  float drop_p;
  uint64_t drop_seed;
  const uint64_t* drop_seed_dev;
  uint32_t drop_site;
  float* save_mean;
  float* save_rstd;
  void* out_bf16;
  /* backward */
  const float* dout;
  void* dy_bf16;
  float* dgamma;
  float* dbeta;
  float* dy_colsum;
} tt_bn_args;
int tt_bn_relu_fwd(const tt_bn_args* args, void* stream);
int tt_bn_relu_bwd(const tt_bn_args* args, void* stream);

/* Fused dense AdamW over a flat fp32 buffer (torch.optim.AdamW as used at src/train.py:302,
 * 64-65): p,g,m,v [n]; the gradient used is grad_scale * g (1 / world for a buffer that holds the SUM of the
 * ranks' gradients, e.g. the owner's shard of a row-sharded ID table); *step_dev is the 1-based step count on the
 * device; optionally writes a bf16 shadow of p[shadow_begin:shadow_end] and zeroes g. */
int tt_adamw_step(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, float grad_scale, const int64_t* step_dev, void* shadow_bf16,
                  int64_t shadow_begin, int64_t shadow_end, int zero_grad, void* stream);
/* ++*step_dev; *seed_dev += golden-ratio increment (either may be NULL). */
int tt_step_counters_advance(int64_t* step_dev, uint64_t* seed_dev, void* stream);

/* ---- last-layer specialisation (SURVEY.md §8 a5) ------------------------------------------
 * Only out[b, len_b-1] of the LAST encoder layer is read (src/models/user_tower.py:122-132), so
 * that layer needs K/V for every position but the query, attention output, out_proj, norm2 and
 * FFN for one row per sequence. Exact: identical outputs and gradients, the skipped values are
 * never consumed.
 *   tt_gather_rows      : out[b] = x[b*L + last_idx[b]] (fp32 and/or bf16 source/destination pairs)
 *   tt_scatter_rows_add : x[b*L + last_idx[b]] = rows[b] (+ previous value when accumulate)
 *   tt_attn_lastq_fwd   : q bf16 [B, H*64], K/V from qkv bf16 [B*L, 3*H*64] -> ctx bf16 [B, H*64],
 *                         lse fp32 [B, H]; keys 0..last_idx[b]
 *   tt_attn_lastq_bwd   : -> dq bf16 [B, H*64] and the K/V thirds of dqkv for EVERY position
 *                         (zeros beyond last_idx[b])
 *                         L <= 4096 for both.
 */
int tt_gather_rows(const float* x_f32, const void* x_bf16, const int32_t* last_idx, int B, int L, int W,
                   float* out_f32, void* out_bf16, void* stream);
int tt_scatter_rows_add(const float* rows, const int32_t* last_idx, int B, int L, int W, float* x, int accumulate,
                        void* stream);
int tt_attn_lastq_fwd(const void* q, const void* qkv, const int32_t* last_idx, void* ctx, float* lse, int B, int L,
                      int H, float drop_p, uint64_t seed, const uint64_t* seed_dev, uint32_t site, void* stream);
int tt_attn_lastq_bwd(const void* q, const void* qkv, const int32_t* last_idx, const void* ctx, const void* dctx,
                      const float* lse, void* dq, void* dqkv, int B, int L, int H, float drop_p, uint64_t seed,
                      const uint64_t* seed_dev, uint32_t site, void* stream);

/* ---- user sessions: one new row per user over cached keys/values -------------------------
 * Appending item p to a right-padded history of length p < L leaves every earlier position of the causal encoder
 * unchanged (src/models/user_tower.py:95-120: causal mask, key padding beyond the history), so each layer needs the
 * new row's attention over the stored K/V of positions 0..p only.
 *   tt_session_attn : qkv bf16 [n, 3*H*64] (Q | K | V of the new rows), K/V caches bf16 [capacity, H, L, 64] each,
 *                     slots / pos int32 [n]. For row r: cache[slots[r], :, pos[r]] = its K / V, then ctx bf16 [n, H*64]
 *                     = softmax(q K[0..pos]^T / 8) V[0..pos]. No dropout (eval). L <= 4096; rows with a slot outside
 *                     [0, capacity) or pos outside [0, L) touch no cache and get ctx = 0. Slots must be distinct
 *                     within a call. Bit-identical from run to run. */
int tt_session_attn(const void* qkv, void* k_cache, void* v_cache, const int32_t* slots, const int32_t* pos, int n,
                    int H, int L, int capacity, void* ctx, void* stream);

/* ---- symmetric InfoNCE (src/models/two_tower.py:106-140) --------------------------------
 * Row formulation: S [R, C] fp32 holds logits of R local rows against C (all-gathered)
 * columns, the positive of row i sits at column pos0 + i.
 * tt_infonce_rows : in place, S[i][j] = -1e4 where uid_rows[i] == uid_cols[j] and j != pos0+i
 *                   (uid_* may be NULL: no masking); row_lse[i] = logsumexp(S[i,:]);
 *                   pos_logit[i] = S[i][pos0+i].
 * tt_infonce_grad : dS[i][j] = coef * (exp(S-row_lse[i]) + exp(S-col_lse[j]) - 2*[j==pos0+i]), bf16.
 *                   col_lse[j] is the log-sum-exp of column j over ALL rows of all ranks, i.e. the
 *                   row_lse of the transposed problem.
 * tt_infonce_loss : loss = coef * sum_i (lse_a-pos_a + lse_b-pos_b)[i]   (coef = 0.5 / global batch)
 */
int tt_infonce_rows(float* S, int R, int C, int ld, const int64_t* uid_rows, const int64_t* uid_cols, int pos0,
                    float* row_lse, float* pos_logit, void* stream);
int tt_infonce_grad(const float* S, int R, int C, int ld, const float* row_lse, const float* col_lse, int pos0,
                    float coef, void* dS_bf16, int ld_d, void* stream);
/* In-batch Recall@k of `evaluate` (src/train.py:95-103) on the logits of one batch: acc[0] += #rows whose positive
 * (column pos0 + i) has fewer than k entries ahead of it in the canonical order (logit descending, column
 * ascending), acc[1] += R. acc is a device float[2] the caller zeroes once per evaluation and all-reduces (SUM)
 * over ranks at the end (:106-109). */
int tt_inbatch_recall(const float* S, int R, int C, int ld, int pos0, int k, float* acc, void* stream);
int tt_infonce_loss(const float* lse_a, const float* pos_a, const float* lse_b, const float* pos_b, int R, float coef,
                    float* loss, void* stream);

/* ---- logQ correction of in-batch negatives (Yi et al., RecSys 2019) --------------------
 * The positives of a batch are its negatives, so column j is sampled with its entity's popularity q_j; the
 * corrected loss subtracts log q_j from every logit of column j. col_off[j] = log q of column j's entity (C values),
 * row_off[p] = log q of the OTHER side's entity at global row p (indexed pos0 + i).
 * tt_infonce_rows_off : tt_infonce_rows over x_ij - col_off[j]; masked entries are -1e4 BEFORE the offset, S keeps the
 *                       uncorrected masked logits; pos_logit[i] = S[i][pos0+i] - col_off[pos0+i].
 * tt_infonce_grad_off : dS[i][j] = coef * (exp(S-col_off[j]-row_lse[i]) + exp(S-row_off[pos0+i]-col_lse[j])
 *                       - 2*[j==pos0+i]). With zero offsets both equal the plain kernels bit for bit.
 * tt_logq_table_gather : off_out[i] = table[ids[i]] for ids in [0, N), floor otherwise.
 * tt_logq_stream_update : streaming frequency estimator, one CTA. A int64 [h, 2^log2H] (last step seen), Bv fp32
 *                       [h, 2^log2H] (interval estimate); slot of id y in array k = low log2H bits of
 *                       splitmix64_finaliser(y + (k+1) * 0x9E3779B97F4A7C15). t = ++*step_dev; every slot hit by the
 *                       ids is updated once: Bv = fl(fl(one_minus_alpha * Bv) + fl(alpha * (float)(t - A))), A = t;
 *                       then off_out[i] = -logf(max_k Bv_k[slot_k(ids[i])]). Deterministic, no host reads.
 *                       1 <= h <= 4, 0 <= log2H <= 28, alpha in (0, 1], n >= 1. */
int tt_infonce_rows_off(float* S, int R, int C, int ld, const int64_t* uid_rows, const int64_t* uid_cols, int pos0,
                        const float* col_off, float* row_lse, float* pos_logit, void* stream);
int tt_infonce_grad_off(const float* S, int R, int C, int ld, const float* row_lse, const float* col_lse, int pos0,
                        float coef, const float* col_off, const float* row_off, void* dS_bf16, int ld_d, void* stream);
int tt_logq_table_gather(const int64_t* ids, int n, const float* table, int64_t N, float floor, float* off_out,
                         void* stream);
int tt_logq_stream_update(const int64_t* ids, int n, int64_t* A, float* Bv, int h, int log2H, int64_t* step_dev,
                          float alpha, float one_minus_alpha, float* off_out, void* stream);

/* ---- catalog retrieval (src/evaluate_metrics.py:106-192) ------------------------------
 * Canonical order everywhere: score descending, then item index ascending (torch.topk leaves
 * ties unspecified). Keys are 64-bit: (order-preserving score bits << 32) | (2^32-1 - index).
 *
 * tt_topk_plan_make : sizes the work decomposition and the scratch buffers for U users against
 *                     N items (this shard), K' = kprime candidates per user (8..256).
 * tt_score_topk     : fused U E^T (bf16 tensor cores, fp32 accumulate) + streaming top-K' per
 *                     user; replaces the matmul at :148, the column-0 mask at :152 and topk at
 *                     :156 without materialising the (U, N) score matrix. Runs on CTA pairs
 *                     (clusters of 2, tcgen05 cta_group::2): a work unit is 256 users x a range of
 *                     256-item steps ("tiles" in the plan below).
 *                     users_bf16 [U,256], items_bf16 [N,256]; item_base = global index of row 0
 *                     of this shard; mask_item0 excludes global item 0 (the padding id).
 *                     cand/cand_cnt/thr/smax are scratch of plan->{cand,cnt,thr,smax}_bytes (smax may be
 *                     NULL: no sample pass).
 * tt_topk_finalize  : per user, K' best keys -> exact re-score (fp32 inputs, fp64 accumulate,
 *                     rounded once to fp32) -> canonical sort -> top K (global indices, -1 pad)
 *                     and flags[u] = 1 when the certificate "no non-candidate can reach the
 *                     exact top K" fails (eps bounds |bf16-path score - exact score|).
 * tt_topk_finalize_bounded : sharded catalogs. Returns ALL K' candidates of this shard re-scored exactly
 *                     ([U, K'], canonical order, -1 / -inf padded) and out_bound[u]: every item of the shard that
 *                     is NOT in the list has exact score <= out_bound[u]. The merged top K over the shards
 *                     (tt_topk_merge_lists) is exact for user u when its K-th score beats every shard's bound;
 *                     a shard then only needs K' ~ (single-GPU K') / shards candidates.
 * tt_topk_merge     : top K of the union of G per-shard lists [G][U][K].
 * tt_topk_merge_lists : the same with input lists of K_in entries and K_out outputs (-1 / -inf padded).
 * tt_exact_topk     : brute-force exact top K of one user (fallback for flagged users);
 *                     key_scratch = N * 8 bytes.
 *
 * Excluding seen items (src/inference.py:296-302: scores[0] = -inf and scores[h] = -inf for every
 * history item h, before the top k). Excluded ids are dropped from the candidate lists before any
 * prune and before the lists are handed over, so pruning, finalize, the certificate, the bounded shard protocol and the merges all speak about the
 * admissible items only; a user with fewer than K admissible items gets a -1 / -inf tail.
 * tt_exclusions_build : ids [U, m] int64 with row pitch ld_in (0 = empty slot; ids <= 0 or >= vocab_size
 *                     are dropped), m <= 4096 -> per user a sorted, de-duplicated int32 list out_ids [U, ld]
 *                     (ld >= m), its length out_cnt [U] and a 4096-bit hashed bitmap out_bits [U, 128].
 * tt_score_topk_excl : tt_score_topk that never admits user u's excluded ids (ex_* from
 *                     tt_exclusions_build, ex_ld = its ld; all NULL = tt_score_topk). The sample pass
 *                     raises each user's rank by its excluded ids inside the sampled item steps.
 * tt_exact_topk_excl : tt_exact_topk without the ids ex_ids[0 .. *ex_cnt) (one user's row of
 *                     tt_exclusions_build's output; NULL = tt_exact_topk).
 * tt_rank_metrics   : per-row Recall@k / NDCG@k (:159-185); gain_table[r] = 1/log2(r+2) comes
 *                     from the host so rows are bit-identical to the reference's; outputs [nk][U].
 */
typedef struct tt_topk_plan {
  int32_t U, N, kprime, cap;
  int32_t n_ut, n_ranges, tiles_per_range;
  int32_t sample_stride, sample_rank, sample_tiles; /* sample pass (0 = none): every sample_stride-th item step
                                                       is scored first, keeping the maximum of each 32-score chunk;
                                                       each user's sample_rank-th largest chunk maximum becomes the
                                                       main pass's start threshold (verified later, never trusted) */
  int64_t cand_bytes, cnt_bytes, thr_bytes, smax_bytes;
} tt_topk_plan;
int tt_topk_plan_make(int U, int N, int kprime, tt_topk_plan* plan);
int tt_score_topk(const void* users_bf16, const void* items_bf16, int item_base, const tt_topk_plan* plan,
                  void* cand, int32_t* cand_cnt, void* thr, void* smax, int mask_item0, void* stream);
/* eps: bound on |bf16-path score - exact score| used by the certificate. Either a host value (eps_stats == NULL) or
 * evaluated on the device from eps_stats = {max ||bf16(u)-u||, max ||u||} written by tt_users_prepare for this pass
 * and the item-side constants ne_max = max ||bf16(e)||, de_max = max ||bf16(e)-e||: no host read precedes the launch. */
int tt_users_prepare(const float* users_f32, void* users_bf16, int U, float* stats, void* stream);
int tt_topk_finalize(const tt_topk_plan* plan, const void* cand, const int32_t* cand_cnt, const void* thr,
                     const float* users_f32, const float* items_f32, int item_base, int K, float eps,
                     const float* eps_stats, float ne_max, float de_max, int32_t* out_idx, float* out_score,
                     int32_t* flags, void* stream);
/* bounded variant: user u's list goes to out_idx / out_score + u * ld_out, its bound and flag to out_bound / flags
 * + u * ld_aux — with out_score = pack, out_idx = pack + K', out_bound = pack + 2K', flags = pack + 2K' + 1 and
 * ld_out = ld_aux = 2K' + 2 the kernel writes the exchange buffer of retrieval.sharded_topk directly. */
int tt_topk_finalize_bounded(const tt_topk_plan* plan, const void* cand, const int32_t* cand_cnt, const void* thr,
                             const float* users_f32, const float* items_f32, int item_base, float eps,
                             const float* eps_stats, float ne_max, float de_max, int32_t* out_idx, float* out_score,
                             int ld_out, float* out_bound, int32_t* flags, int ld_aux, void* stream);
/* merge of the all-gathered exchange buffer in place: packed [G][U][ld] int32 words, row = [K_in scores | K_in global
 * ids | bound | flag]; writes the merged top K_out and bad[u] = 1 where the certificate fails (K_out-th merged score
 * does not beat every shard's bound, or a shard flagged a tie flood). */
int tt_topk_merge_packed(const int32_t* packed, int ld, int G, int U, int K_in, int K_out, float* out_score,
                         int32_t* out_idx, int32_t* bad, void* stream);
int tt_topk_merge(const float* scores, const int32_t* idx, int G, int U, int K, float* out_score, int32_t* out_idx,
                  void* stream);
int tt_topk_merge_lists(const float* scores, const int32_t* idx, int G, int U, int K_in, int K_out, float* out_score,
                        int32_t* out_idx, void* stream);
int tt_exact_topk(const float* user_f32, const float* items_f32, int N, int item_base, int mask_item0, int K,
                  void* key_scratch, float* out_score, int32_t* out_idx, void* stream);
int tt_exclusions_build(const int64_t* ids, int U, int m, int ld_in, int vocab_size, int32_t* out_ids, int ld,
                        int32_t* out_cnt, uint32_t* out_bits, void* stream);
int tt_score_topk_excl(const void* users_bf16, const void* items_bf16, int item_base, const tt_topk_plan* plan,
                       void* cand, int32_t* cand_cnt, void* thr, void* smax, int mask_item0, const int32_t* ex_ids,
                       const int32_t* ex_cnt, const uint32_t* ex_bits, int ex_ld, void* stream);
int tt_exact_topk_excl(const float* user_f32, const float* items_f32, int N, int item_base, int mask_item0, int K,
                       const int32_t* ex_ids, const int32_t* ex_cnt, void* key_scratch, float* out_score,
                       int32_t* out_idx, void* stream);
int tt_rank_metrics(const int32_t* topk_idx, const int64_t* targets, int U, int K, const int32_t* k_list, int nk,
                    const float* gain_table, float* recall, float* ndcg, void* stream);

/* ---- diversified recommendations: maximal marginal relevance over each user's candidate pool ----
 * Extends the selection of src/inference.py:296-306 (masked scores, top k): instead of the k best scores, k picks
 * from the pool of the exact top P admissible candidates (pool_idx int32 / pool_score fp32 [U, P], canonical order,
 * -1 / -inf tail, as tt_topk_finalize writes them). lam = 1 - diversity and mu = 1 - lam come from the host.
 * sim(a, b) = fp32 rows of items a and b, fp64 accumulate, rounded once to fp32; m_j = max sim(c_j, s) over the items
 * s picked so far (0 before the first). Step t picks the unpicked position j with c_j >= 0 and the largest
 * obj_j = lam * r_j - mu * m_j (fp64: two correctly rounded products, one subtraction, no FMA); ties go to the smaller
 * j. out_idx int32 / out_score fp32 [U, k]: picked ids in pick order and their relevances (NOT sorted by score when
 * mu > 0), -1 / -inf where fewer than k candidates are admissible. Bit-identical from run to run.
 *   tt_mmr_select : rows from source TT_MMR_ROWS_TABLE (rows = this shard's fp32 table; id's row at id - item_base,
 *                   ids outside [item_base, item_base + num_rows) count as inadmissible) or TT_MMR_ROWS_GATHERED
 *                   (rows = fp32 [U, P, 256], row of pool position j of user u at (u * P + j) * 256; item_base and
 *                   num_rows unused). 1 <= k <= P <= 256, lam and mu in [0, 1]; U = 0 launches nothing (its
 *                   pointers may be NULL). k = 1 reads no row.
 *   tt_mmr_gather_rows : sharded catalogs: out fp32 [n, 256] row r = the table row of pool_idx[r] when this shard owns
 *                   it (item_base <= id < item_base + num_rows), zeros otherwise. The sum of every shard's buffer is
 *                   the TT_MMR_ROWS_GATHERED input, exactly (one non-zero contributor per element). */
#define TT_MMR_ROWS_TABLE 0
#define TT_MMR_ROWS_GATHERED 1
int tt_mmr_select(const int32_t* pool_idx, const float* pool_score, int U, int P, int k, double lam, double mu,
                  int source, const float* rows, int item_base, int num_rows, int32_t* out_idx, float* out_score,
                  void* stream);
int tt_mmr_gather_rows(const int32_t* pool_idx, int n, const float* table, int item_base, int num_rows, float* out,
                       void* stream);

/* ---- ID table row-sharded over the ranks of one NVLink domain ----------
 * (BASELINE.json configs[4]: 10M items; reference: nn.Embedding(vocab_size, 256, padding_idx=0) and its dense
 * gradient, src/models/user_tower.py:26,86.) The table and its gradient live in a symmetric arena (tt_symm_team
 * below): the rows are dealt ROUND-ROBIN (item popularity is Zipfian in the id: contiguous ranges would send most
 * lookups to rank 0): row id is local row id / world of rank id % world, at byte `weight_offset` / `grad_offset` of
 * that rank's copy. Rows are read from — and gradient rows added (red.global.add.v4.f32) into — the OWNER's memory
 * over NVLink. The caller separates steps with tt_symm_barrier (owners' updates visible before the next gather; all
 * ranks' gradient rows landed before the owner's AdamW). */
struct tt_symm_team;

/* Duplicate-free traffic for a row-sharded (or replicated) ID table. Histories are Zipfian in the item id: at batch
 * 256 x 200 about a third of the tokens carry a distinct id, so a step first reduces its ids to the distinct ones.
 * tt_ids_dedup   : ids[T] -> uniq[0..n) int64 (uniq[0] = 0, the padding id; order unspecified), inverse[t] = slot of
 *                  ids[t] (0 for padding / out-of-table ids), state[1] = n. Scratch: flag, slot int32 [V] and state
 *                  int32 [2], zero-filled by the caller ONCE; uniq needs T + 1 entries. Every call clears the flags
 *                  the previous call set.
 * tt_rows_gather : cache[s, :] = table row uniq[s] for s < *n_uniq — read from the owner's shard over NVLink
 *                  (team + weight_offset) or from a local table (table_local); each distinct row crosses the link
 *                  once. The embedding kernels (tt_embed_ln_fwd / _bwd) then run on `cache` with `inverse` as ids.
 * tt_rows_scatter_add : owner's gradient row uniq[s] += gacc[s, :] (red.global.add.v4.f32), then gacc[s, :] = 0, for
 *                  1 <= s < *n_uniq: gacc is the compact gradient buffer the embedding backward accumulated into
 *                  (duplicates combined locally, L2-resident), one remote reduction per distinct row remains.
 * max_rows bounds the launch (the count itself is read on the device). */
int tt_ids_dedup(const int64_t* ids, int T, int64_t V, int32_t* flag, int32_t* slot, int64_t* uniq, int32_t* state,
                 int64_t* inverse, void* stream);
int tt_rows_gather(const struct tt_symm_team* team, int64_t weight_offset, const float* table_local, const int64_t* uniq,
                   const int32_t* n_uniq, int max_rows, float* cache, void* stream);
int tt_rows_scatter_add(const struct tt_symm_team* team, int64_t grad_offset, float* grad_local, const int64_t* uniq,
                        const int32_t* n_uniq, int max_rows, float* gacc, void* stream);

/* ---- data-parallel exchanges over NVLink peer memory -------------------------------------
 * Replaces the NCCL traffic of the reference's DistributedDataParallel wrapper (src/train.py:29-35, 300: one
 * gradient all-reduce per step, then torch.optim.AdamW on every rank, :302) and of the gathered-negatives
 * exchange this repo adds (BASELINE.json configs[3]).
 *
 * A "team" describes ONE symmetric arena: the same allocation made by every rank, `bufs[r]` = rank r's copy as
 * mapped into the calling process (bufs[rank] is the local one), `multicast` = the NVLS multicast mapping of the
 * arena or NULL, `ctrl_offset` = byte offset of a tt_symm_ctrl_bytes()-sized control block inside the arena that
 * the caller zeroes once before the first collective (and never touches again). Every rank must issue the same
 * sequence of collectives on a team. All three entry points are stream-ordered and graph-capturable; they spin on
 * flags in the control block, so the ranks' kernels must be able to run concurrently (one process per GPU).
 *
 * tt_symm_allgather : rank r's n_seg (<= 4) source blocks are stored into EVERY rank's arena at
 *                     dst_offset + r * nbytes; ends with a cross-rank barrier (when the kernel completes, all
 *                     ranks' blocks are visible locally). pre_barrier != 0 adds one at the start (needed when no
 *                     collective separates this call from the peers' last reads of the destination).
 * tt_dp_adamw_step  : flat fp32 parameters, fp32 gradients and the bf16 shadow of parameters [shadow_begin, n) live
 *                     in the arena at the given byte offsets. Rank r owns elements [r*n/G, (r+1)*n/G): it reads the
 *                     MEAN over ranks of the gradient slice (multimem.ld_reduce, or peer loads in rank order),
 *                     applies torch.optim.AdamW (m, v: local moments of the slice) and stores the new values and
 *                     their bf16 copies into every rank's arena (multimem.st / peer stores). Barriers on both
 *                     sides: starts when every rank's gradients are final, completes when every rank's parameters
 *                     are. Gradients are NOT cleared (the caller zeroes its local buffer afterwards).
 *                     shard_* (shard_n > 0): this rank's rows of a row-sharded ID table in plain local memory
 *                     (parameters, gradient SUM over ranks, moments): updated by the same kernel between the two
 *                     barriers with gradient = shard_g / world, shard_g cleared in the same pass — the first barrier
 *                     guarantees every rank's gradient rows have landed, the second that every owner's rows are
 *                     final before any rank's next step gathers them.
 * tt_symm_barrier   : barrier across the team.
 * A wait longer than ~10 s (a peer died) sets the int32 at ctrl_offset + 8 and returns; callers check it. */
#define TT_SYMM_MAX_RANKS 16
typedef struct tt_symm_team {
  int32_t rank, world;
  void* bufs[TT_SYMM_MAX_RANKS];
  void* multicast;
  int64_t ctrl_offset;
} tt_symm_team;
typedef struct tt_symm_segment {
  const void* src;
  int64_t dst_offset;
  int64_t nbytes;
} tt_symm_segment;
int tt_symm_ctrl_bytes(void);
int tt_symm_allgather(const tt_symm_team* team, const tt_symm_segment* segs, int n_seg, int pre_barrier, void* stream);
int tt_dp_adamw_step(const tt_symm_team* team, int64_t flat_offset, int64_t grad_offset, int64_t shadow_offset,
                     int64_t n, int64_t shadow_begin, float* m, float* v, float lr, float beta1, float beta2, float eps,
                     float weight_decay, const int64_t* step_dev, float* shard_p, float* shard_g, float* shard_m,
                     float* shard_v, int64_t shard_n, void* stream);
int tt_symm_barrier(const tt_symm_team* team, void* stream);

#ifdef __cplusplus
}
#endif

#endif /* TT_B200_H_ */
