/* rbm.h -- C ABI of librbm_b200.so: the B200 (sm_100a) kernels behind the BERT4Rec / SASRec
 * train step and full-catalogue evaluation.
 *
 * The reference (Furyton/Recommender-Baseline-Model) has no FFI: its "operator interface" for this
 * path is the set of torch ops its modules call.  Each entry point below replaces one group of those
 * ops; the reference call site is cited as NN/<file>:<line> with
 *   NN/ = NerualNetwork/bert4rec&sas4rec/.
 * The Python host side (recommender-baseline-model_b200/) binds these with ctypes and mirrors the
 * reference's model / trainer / metric API on top (see INTEGRATION.md).
 *
 * Conventions
 *  - all pointers are DEVICE pointers unless the name ends in _host; fp32 data, int64 indices;
 *    row-major; every fp32 pointer must be 16-byte aligned and every hidden size d % 4 == 0.
 *  - `stream` is a cudaStream_t passed as void*; every call only enqueues work on it (no sync,
 *    no allocation, no global state besides the thread-local last-error string).
 *  - return 0 on success, <0 for an invalid argument / unsupported shape (no CPU fallback),
 *    >0 = cudaError_t of the launch.  rbm_last_error() describes the last failure on this thread.
 *  - dropout: keep-mask = Philox4x32-7(key=seed, counter=(element/4, site)) >= p*2^32, scaled by
 *    1/(1-p); `site` identifies the dropout call site within a step (DESIGN.md "dropout").  The
 *    backward entry points regenerate the mask from (seed, site); nothing is stored.
 */
#ifndef RBM_H
#define RBM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBM_ABI_VERSION 1

typedef void* rbm_stream_t; /* cudaStream_t */

/* activation codes for rbm_linear_* */
#define RBM_ACT_NONE 0
#define RBM_ACT_RELU 1      /* NN/models/sas_model/sas.py:12 */
#define RBM_ACT_GELU_TANH 2 /* NN/models/bert_modules/utils/gelu.py:12 */

/* LayerNorm flavours */
#define RBM_LN_TORCH 0 /* nn.LayerNorm: biased var, eps inside sqrt  (NN/models/sas_model/sas.py:39,42,50) */
#define RBM_LN_BERT 1  /* a*(x-mean)/(std_unbiased+eps)+b           (NN/models/bert_modules/utils/layer_norm.py:14-17) */

/* attention mask modes */
#define RBM_MASK_NONE 0
#define RBM_MASK_CAUSAL 1 /* future keys -> -inf                      (NN/models/sas_model/sas.py:70,75-76) */
#define RBM_MASK_KEYPAD 2 /* keys whose token == 0 -> -1e9            (NN/models/bert_modules/bert.py:38, attention/single.py:27-28) */

int rbm_abi_version(void);
const char* rbm_last_error(void);

/* ---- embedding stage ---------------------------------------------------------------------------
 * out[r,:] = keep(r) * dropout( table[tok[r],:]*scale + pos[r % L,:] ),  keep(r) = zero_pad ? tok[r]!=0 : 1
 * replaces  SAS.log2feats NN/models/sas_model/sas.py:60-67  (scale=sqrt(d), zero_pad=1)
 *           BERTEmbedding.forward NN/models/bert_modules/embedding/bert.py:29-31 (scale=1, zero_pad=0) */
int rbm_embed_fwd(const int64_t* tok, const float* table, const float* pos, float* out, int64_t rows, int L,
                  int d, int64_t vocab, float scale, int zero_pad, float p, uint64_t seed, uint64_t site,
                  rbm_stream_t stream);
/* g[r,:] = keep(r)*mask*dout[r,:]  (gradient w.r.t. the pre-dropout sum);  dpos[l,:] = sum_b g[b*L+l,:]
 * (batch-ascending order).  The table gradient is rbm_scatter_add_sorted(tok, g, alpha=scale). */
int rbm_embed_bwd(const int64_t* tok, const float* dout, float* g, float* dpos, int64_t rows, int L, int d,
                  int zero_pad, float p, uint64_t seed, uint64_t site, rbm_stream_t stream);

/* Row-sharded item table (SURVEY 8e "input lookup"): `table_shard` holds rows [v_begin, v_end) of the [vocab, d] table.  Same as
 * rbm_embed_fwd for tokens inside the shard; tokens of other shards produce exact zeros (their owner produces the value, so a
 * sum over the shards -- reduce-scatter -- is the unsharded result bit for bit).  `tok` is the rank-ordered concatenation of the
 * ranks' batches, so the dropout element index is the index in the global batch.  An empty shard (v_begin == v_end) may pass
 * table_shard = NULL. */
int rbm_embed_fwd_shard(const int64_t* tok, const float* table_shard, const float* pos, float* out, int64_t rows, int L,
                        int d, int64_t vocab, int64_t v_begin, int64_t v_end, float scale, int zero_pad, float p,
                        uint64_t seed, uint64_t site, rbm_stream_t stream);
/* rbm_embed_bwd (zero_pad = 1) on the live rows only: dout_c / g_c [cap, d] hold row rows[r] of the [B, L] batch in row r (csrc/rows.cu);
 * idx_c[r] = tok[rows[r]] (0 past *count): the (idx_c, g_c) pair goes to rbm_scatter_add_sorted with cap entries.  dpos [L, d] is
 * summed per position in ascending row order inside fixed row ranges, then over the ranges.  Dropout stream: the element's index in
 * the full batch, as in rbm_embed_fwd.  L*d*4 <= 96 KB. */
size_t rbm_embed_bwd_rows_ws_bytes(int L, int d);
int rbm_embed_bwd_rows(const int64_t* tok, const int32_t* rows, const int32_t* count, int64_t cap, const float* dout_c,
                       float* g_c, int64_t* idx_c, float* dpos, int L, int d, float p, uint64_t seed, uint64_t site,
                       void* ws, size_t ws_bytes, rbm_stream_t stream);
/* rbm_embed_bwd on a rank's slice of the global batch: `row_offset` = index of its first row in the global batch (dropout
 * element indices continue from there). */
int rbm_embed_bwd_offset(const int64_t* tok, const float* dout, float* g, float* dpos, int64_t rows, int L, int d,
                         int zero_pad, float p, uint64_t seed, uint64_t site, uint64_t row_offset, rbm_stream_t stream);

/* ---- embedding-gradient scatter-add (autograd of nn.Embedding = embedding_dense_backward; triggered by
 * loss.backward() NN/trainers/base.py:121).  grad[idx[i],:] += alpha * coef[i] * src[i,:], summed over i in
 * ASCENDING i per destination row (stable LSD radix sort of idx, then one sequential fp32 segment sum per
 * row: bit-identical to the CPU reference's index-ordered loop).  idx == padding_idx contributes nothing
 * (padding_idx < 0: none).  coef may be NULL (=1).  ws: rbm_scatter_ws_bytes(n, vocab) bytes. */
size_t rbm_scatter_ws_bytes(int64_t n, int64_t vocab);
int rbm_scatter_add_sorted(const int64_t* idx, const float* src, const float* coef, float alpha, float* grad,
                           int64_t n, int d, int64_t vocab, int64_t padding_idx, void* ws, size_t ws_bytes,
                           rbm_stream_t stream);

/* ---- LayerNorm (both flavours), stats[r] = {mean, 1/(sqrt(var+eps)) | 1/(std+eps)} saved for backward --- */
int rbm_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* stats,
                      int64_t rows, int d, float eps, int flavour, rbm_stream_t stream);
/* dx = LN'(x)*dy; dgamma/dbeta [d] (deterministic two-stage column reduction; ws >= rbm_layernorm_ws_bytes) */
size_t rbm_layernorm_ws_bytes(int64_t rows, int d);
int rbm_layernorm_bwd(const float* x, const float* gamma, const float* dy, const float* stats, float* dx,
                      float* dgamma, float* dbeta, int64_t rows, int d, float eps, int flavour, void* ws,
                      size_t ws_bytes, rbm_stream_t stream);
/* same, plus dx += dres when dres != NULL: the gradient that reaches x through the residual branch of
 * x + sublayer(LN(x)) (NN/models/bert_modules/utils/sublayer.py:16-18), folded into the one pass that writes dx */
int rbm_layernorm_bwd_residual(const float* x, const float* gamma, const float* dy, const float* dres, const float* stats,
                               float* dx, float* dgamma, float* dbeta, int64_t rows, int d, float eps, int flavour,
                               void* ws, size_t ws_bytes, rbm_stream_t stream);

/* same, plus dy2 (may be NULL): the gradient of a second consumer of the normalised output (SASRec: Q feeds the q-projection
 * and the residual, NN/models/sas_model/sas.py:72-79; the FFN input feeds conv1 and the residual, :16-20): LN'(x)*(dy + dy2) + dres */
int rbm_layernorm_bwd_fanout(const float* x, const float* gamma, const float* dy, const float* dy2, const float* dres,
                             const float* stats, float* dx, float* dgamma, float* dbeta, int64_t rows, int d, float eps,
                             int flavour, void* ws, size_t ws_bytes, rbm_stream_t stream);

/* ---- Linear with fused epilogue --------------------------------------------------------------------
 * pre = x[M,K] . w[N,K]^T + bias        (optionally stored to `pre` when act needs it in backward)
 * y   = rowkeep * dropB( residual + dropA( act(pre) ) )      rowkeep(r) = row_tok ? row_tok[r]!=0 : 1
 * Blackwell path: tcgen05.mma kind::tf32 (fp32 operands read as TF32, fp32 accumulation in TMEM), TMA-fed, whenever
 * K % 32 == 0 and N % 16 == 0; other shapes use the fp32 SIMT kernel.
 * replaces nn.Linear / Conv1d(k=1) + Dropout + activation + residual chains:
 *   NN/models/bert_modules/attention/multi_head.py:29-30,40; utils/feed_forward.py:16; utils/sublayer.py:18;
 *   transformer.py:32; NN/models/sas_model/sas.py:16-19,75,79,84 (in/out-proj of nn.MultiheadAttention). */
int rbm_linear_fwd(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t ldy,
                   float* pre, int64_t M, int N, int K, int act, const float* residual, int64_t ldres,
                   const int64_t* row_tok, float pA, uint64_t siteA, float pB, uint64_t siteB, uint64_t seed,
                   rbm_stream_t stream);
/* the same call with a scratch buffer of rbm_linear_fwd_ws_bytes(M,N,K) bytes (may be 0): wide layers (N, K >= 128) with
 * M >= 512 rows then run on the split-fp16 tiled tensor kernel, which keeps fp16 hi/lo copies of w in the scratch */
size_t rbm_linear_fwd_ws_bytes(int64_t M, int N, int K);
int rbm_linear_fwd_ws(const float* x, int64_t ldx, const float* w, const float* bias, float* y, int64_t ldy,
                      float* pre, int64_t M, int N, int K, int act, const float* residual, int64_t ldres,
                      const int64_t* row_tok, float pA, uint64_t siteA, float pB, uint64_t siteB, uint64_t seed,
                      void* ws, size_t ws_bytes, rbm_stream_t stream);
/* elementwise backward of the epilogue: dres = rowkeep*maskB*dout (may be NULL), dpre = dres*maskA*act'(pre) */
int rbm_linear_epilogue_bwd(const float* dout, const float* pre, float* dpre, float* dres, int64_t M, int N,
                            int act, const int64_t* row_tok, float pA, uint64_t siteA, float pB,
                            uint64_t siteB, uint64_t seed, rbm_stream_t stream);
/* dx[M,K] = dpre[M,N] . w[N,K]   (ws: rbm_linear_bwd_data_ws_bytes(N,K) bytes, holds w^T for the tcgen05 path) */
size_t rbm_linear_bwd_data_ws_bytes(int N, int K);
int rbm_linear_bwd_data(const float* dpre, int64_t lddpre, const float* w, float* dx, int64_t lddx, int64_t M,
                        int N, int K, void* ws, size_t ws_bytes, rbm_stream_t stream);
/* dw[N,K] = dpre^T . x ; db[N] = colsum(dpre)  (split over M, fixed-order reduction; ws from _ws_bytes) */
size_t rbm_linear_bwd_weight_ws_bytes(int64_t M, int N, int K);
int rbm_linear_bwd_weight(const float* dpre, int64_t lddpre, const float* x, int64_t ldx, float* dw, float* db,
                          int64_t M, int N, int K, void* ws, size_t ws_bytes, rbm_stream_t stream);

/* ---- short-sequence multi-head attention (L <= 256), one CTA per (sequence, head) -------------------
 * q/k/v/out are [B*L, ld*] row-major with head hh occupying columns [hh*dk, (hh+1)*dk).
 * P = dropout(softmax(mask(scale * q.k^T)));  out = P.v;  stats[(b*h+hh)*L+i] = {rowmax, 1/rowsum}.
 * replaces Attention.forward NN/models/bert_modules/attention/single.py:13-35 and the core of
 * nn.MultiheadAttention at NN/models/sas_model/sas.py:75-76. */
/* rbm_attn_fwd / rbm_attn_bwd with the queries a per-sequence compacted subset: q / out / dout / dq are [B*Lq, ld] (Lq rows per
 * sequence, zero rows after the real ones), k / v / dk / dv [B*L, ld], stats [B*h*Lq, 2], ws rbm_attn_bwd_lq_ws_bytes(B, Lq, h).
 * BERT4Rec training reads the final block's output at the labelled positions only (NN/trainers/bert.py:36-40), so that block's
 * attention needs those queries only -- against every key.  Tensor path only: d_k = 32, Lq <= L <= 256, mask NONE / KEYPAD; dropout
 * fields are indexed by (sequence-head, compact query ordinal, key position). */
int rbm_attn_lq_supported(int L, int Lq, int dk, int mask_mode);
int rbm_attn_fwd_lq(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                    const int64_t* tok, float* out, int64_t ldo, float* stats, int B, int L, int Lq, int h, int dk,
                    int mask_mode, float scale, float p, uint64_t seed, uint64_t site, rbm_stream_t stream);
size_t rbm_attn_bwd_lq_ws_bytes(int B, int Lq, int h);
int rbm_attn_bwd_lq(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                    const int64_t* tok, const float* out, int64_t ldo, const float* dout, int64_t lddo,
                    const float* stats, float* dq, int64_t lddq, float* dk_, int64_t lddk, float* dv, int64_t lddv, int B,
                    int L, int Lq, int h, int dk, int mask_mode, float scale, float p, uint64_t seed, uint64_t site, void* ws,
                    size_t ws_bytes, rbm_stream_t stream);
/* evaluation (K20): attention of the LAST query position of every sequence only -- q/out are [B, h*dk] (row b = sequence b),
 * k/v the [B*L, ld] rows of every position.  Same masks as rbm_attn_fwd (the causal mask leaves the last query every key), no
 * dropout.  Replaces the `[:, -1, :]` slice of NN/trainers/bert.py:47 and NN/models/sas_model/sas.py:111 being taken AFTER the
 * last block was computed for all L positions. */
int rbm_attn_last_query(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                        const int64_t* tok, float* out, int64_t ldo, int B, int L, int h, int dk, int mask_mode, float scale,
                        rbm_stream_t stream);
int rbm_attn_fwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                 const int64_t* tok, float* out, int64_t ldo, float* stats, int B, int L, int h, int dk,
                 int mask_mode, float scale, float p, uint64_t seed, uint64_t site, rbm_stream_t stream);
size_t rbm_attn_bwd_ws_bytes(int B, int L, int h);
int rbm_attn_bwd(const float* q, int64_t ldq, const float* k, int64_t ldk, const float* v, int64_t ldv,
                 const int64_t* tok, const float* out, int64_t ldo, const float* dout, int64_t lddo,
                 const float* stats, float* dq, int64_t lddq, float* dk_, int64_t lddk, float* dv,
                 int64_t lddv, int B, int L, int h, int dk, int mask_mode, float scale, float p, uint64_t seed,
                 uint64_t site, void* ws, size_t ws_bytes, rbm_stream_t stream);

/* ---- live-row compaction around the token-wise layers of SASRec (csrc/rows.cu) ----------------------
 * The reference zeroes the rows of padding positions after the embedding and after every block (`seqs *= ~timeline_mask`,
 * NN/models/sas_model/sas.py:67,86): those rows are exactly zero at every block input, their keys / values equal the projection
 * bias, and what the block computes for them is multiplied by zero -- value and gradient.  rows / count: rbm_compact_labels applied
 * to the token ids; cap >= *count is a host-side capacity (compact rows past *count are zero / ignored).
 *   gather : dst[r] = r < *count ? (coef ? coef[rows[r]] : 1) * src[rows[r]] : 0      [n, d] -> [cap, d]
 *   scatter: dst[rows[r]] = src[r]; rows with tok == 0 get `fill` ([d], may be NULL = zeros)   [cap, d] -> [n, d]
 *   dead_colsum: out[c] = sum over rows with tok == 0 of src[row, c] (the gradient of `fill`), fixed summation order */
int rbm_rows_gather(const float* src, int64_t ld, const int32_t* rows, const int32_t* count, int64_t cap, int d,
                    const float* coef /* [n] per-source-row factor or NULL */, float* dst, rbm_stream_t stream);
int rbm_rows_scatter(const float* src, const int32_t* rows, const int32_t* count, int64_t cap, int d, const float* fill,
                     const int64_t* tok, int64_t n, float* dst, int64_t ldd, rbm_stream_t stream);
size_t rbm_rows_dead_colsum_ws_bytes(int d);
int rbm_rows_dead_colsum(const float* src, int64_t ld, const int64_t* tok, int64_t n, int d, float* out, void* ws, size_t ws_bytes,
                         rbm_stream_t stream);
/* out[c] = sum of the first *count rows of the compact [cap, d] tensor (ws: rbm_rows_dead_colsum_ws_bytes(d)) */
int rbm_rows_live_colsum(const float* src, int64_t ld, const int32_t* count, int64_t cap, int d, float* out, void* ws,
                         size_t ws_bytes, rbm_stream_t stream);

/* compact rows <-> per-sequence padded layout [B, Lq, d]: slot o of sequence b = compact row seq_start[b] + o, zero rows past the
 * sequence's last live row (no sequence may have more than Lq live rows: the caller checks).  Each is the other's gradient. */
int rbm_rows_to_seq(const float* src, const int32_t* seq_start, int B, int Lq, int d, float* dst, rbm_stream_t stream);
int rbm_seq_to_rows(const float* src, const int32_t* rows, const int32_t* seq_start, const int32_t* count, int64_t cap, int L,
                    int Lq, int d, float* dst, rbm_stream_t stream);

/* ---- SASRec attention on the compact (live-row) layout (csrc/attention_live.cu) ---------------------
 * q [cap, h*dk] and kv [cap, 2*h*dk] (k | v) hold the live rows in ascending (sequence, position) order (rows / count / tok as
 * above); every padding position's key / value is bkv = [b_k | b_v] (the projection bias: its input row is exactly zero).  Causal
 * softmax over the live keys j <= i plus n_dead(i) copies of the padding key; dropout fields are indexed by (sequence-head, i, j)
 * over the [L x L] positions exactly as in rbm_attn_fwd.  L <= 64, d_k in {16, 32, 64, 128}.  stats [cap, h, 2].
 * Backward: dq [cap, h*dk], dkv [cap, 2*h*dk] and per-query rows dead [cap, 2*h*dk] whose column sum (rbm_rows_live_colsum) is the
 * gradient of bkv; delta [cap, h] floats and keepw [cap, h] 64-bit words are scratch.  Replaces the core of nn.MultiheadAttention at NN/models/sas_model/sas.py:75-76 on that layout. */
/* seq_start[b] = first compact row of sequence b (b = 0..B: B + 1 entries), from the ascending row ids */
int rbm_rows_seq_start(const int32_t* rows, const int32_t* count, int B, int L, int32_t* seq_start, rbm_stream_t stream);
int rbm_attn_live_fwd(const float* q, int64_t ldq, const float* kv, int64_t ldkv, const float* bkv, const int32_t* rows,
                      const int32_t* seq_start, const int64_t* tok, float* out, float* stats, int B, int L, int h, int dk,
                      float scale, float p, uint64_t seed, uint64_t site, rbm_stream_t stream);
int rbm_attn_live_bwd(const float* q, int64_t ldq, const float* kv, int64_t ldkv, const float* bkv, const int32_t* rows,
                      const int32_t* seq_start, const int64_t* tok, const float* out, const float* stats, const float* dout,
                      float* dq, float* dkv, float* dead, float* delta, uint64_t* keepw, int B, int L, int h, int dk, float scale,
                      float p, uint64_t seed, uint64_t site, rbm_stream_t stream);

/* ---- BERT4Rec output scoring fused with masked cross-entropy (logits never materialised) ------------
 * rows with labels != 0 are compacted (ascending); for those rows logits = h.w^T + bias over V1 = V+1
 * columns; loss = mean(logsumexp - target logit).
 * replaces self.out(...) NN/models/bert.py:16 + CrossEntropyLoss(ignore_index=0) NN/trainers/bert.py:11,36-40. */
/* compaction: rows_out[0..count) = ascending row ids with labels != 0, tgt_out = their labels, *count_out. */
size_t rbm_compact_ws_bytes(int64_t n);
int rbm_compact_labels(const int64_t* labels, int64_t n, int32_t* rows_out, int64_t* tgt_out, int32_t* count_out,
                       void* ws, size_t ws_bytes, rbm_stream_t stream);
size_t rbm_ce_ws_bytes(int64_t cap, int V1, int d);
/* forward: lse[cap], loss (1 float).  cap = capacity (>= count); count read from device.  A target outside [0, V1) matches
 * no column (its logit counts as 0): this is what a row-shard of the output layer passes for targets it does not own
 * (tgt - v_begin; rbm_b200.dist.vocab_parallel_cross_entropy). */
int rbm_ce_fwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w,
               const float* bias, float* lse, float* loss, int64_t cap, int V1, int d, void* ws, size_t ws_bytes,
               rbm_stream_t stream);
/* backward: dh_full[n_rows_total,d] must be pre-zeroed; rows listed in `rows` receive their gradient;
 * dw[V1,d], db[V1] overwritten.  dloss: device scalar (upstream gradient). */
int rbm_ce_bwd(const float* h, const int32_t* rows, const int64_t* tgt, const int32_t* count, const float* w,
               const float* bias, const float* lse, const float* dloss, float* dh_full, float* dw, float* db,
               int64_t cap, int V1, int d, void* ws, size_t ws_bytes, rbm_stream_t stream);

/* ---- SASRec train scoring + BCE ---------------------------------------------------------------------
 * pos_logit[r] = <f[r,:], table[pos[r],:]>, same for neg     (SAS.forward NN/models/sas_model/sas.py:93-100) */
int rbm_sas_score_fwd(const float* f, const float* table, const int64_t* pos, const int64_t* neg,
                      float* pos_logit, float* neg_logit, int64_t rows, int d, rbm_stream_t stream);
/* df[r,:] = dpl[r]*table[pos[r]] + dnl[r]*table[neg[r]]; table grads: scatter with coef=dpl / dnl, src=f */
int rbm_sas_score_bwd(const float* table, const int64_t* pos, const int64_t* neg, const float* dpl,
                      const float* dnl, float* df, int64_t rows, int d, rbm_stream_t stream);
/* loss = mean_{pos!=0} softplus(-pl) + mean_{pos!=0} softplus(nl)   (NN/trainers/sas.py:38-49);
 * also writes count (int32) of pos != 0.  ws >= rbm_bce_ws_bytes(rows). */
size_t rbm_bce_ws_bytes(int64_t rows);
int rbm_bce_pair_fwd(const float* pl, const float* nl, const int64_t* pos, float* loss, int32_t* count,
                     int64_t rows, void* ws, size_t ws_bytes, rbm_stream_t stream);
int rbm_bce_pair_bwd(const float* pl, const float* nl, const int64_t* pos, const int32_t* count,
                     const float* dloss, float* dpl, float* dnl, int64_t rows, rbm_stream_t stream);

/* ---- candidate scoring for sampled evaluation -------------------------------------------------------
 * out[u,c] = <table[cand[u,c],:], f[u,:]> (+ bias[cand[u,c]])
 * replaces SAS.predict NN/models/sas_model/sas.py:110-114 and scores.gather NN/trainers/bert.py:47-49 */
int rbm_candidate_scores(const float* f, int64_t ldf, const float* table, const float* bias, const int64_t* cand,
                         float* out, int64_t U, int C, int d, rbm_stream_t stream);

/* ---- full-catalogue scoring fused with top-k (scores never materialised) ----------------------------
 * For each user u: rank items v in [v_begin, v_end) (rows of `table`) by s = <f[u],table[v]> (+bias[v]),
 * order (score desc, id asc), id = v + id_offset; emit top_scores/top_ids [U,k] (k <= 32; unfilled slots
 * = (-inf, -1)).  ws >= rbm_score_topk_ws_bytes_d(U, v_end - v_begin, d, k). */
size_t rbm_score_topk_ws_bytes(int64_t U, int64_t n_items, int k);
/* the same for a known hidden size d (the catalogue-scale path keeps a range-scaled fp16 copy of the scored rows, n_items * d * 2
 * bytes, in the workspace; the d-less query above has to assume d = 256) */
size_t rbm_score_topk_ws_bytes_d(int64_t U, int64_t n_items, int d, int k);
int rbm_score_topk(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin,
                   int64_t v_end, int64_t id_offset, float* top_scores, int64_t* top_ids, int64_t U, int d,
                   int k, void* ws, size_t ws_bytes, rbm_stream_t stream);
/* rbm_score_topk over the catalogue minus each user's already-seen items (the "full sort" protocol of full-ranking
 * evaluation: the reference's argsort over all items, NN/trainers/utils.py:36-38, after the history is removed).  Row u of
 * excl [U, n_excl] (row stride ld_excl, int64) holds the ids user u must not be ranked, in output-id space (v + id_offset,
 * the ids this call returns), sorted ascending; duplicates are allowed and ids outside [v_begin, v_end) + id_offset never
 * match (0 / -1 padding and other shards' ids are harmless).  Result: the canonical top-k of the remaining items (same
 * order and scores as rbm_score_topk; fewer than k remaining -> trailing (-inf, -1)).  excl == NULL or n_excl == 0 gives
 * results bit-identical to rbm_score_topk.  Same workspace query. */
int rbm_score_topk_excl(const float* f, int64_t ldf, const float* table, const float* bias, int64_t v_begin, int64_t v_end,
                        int64_t id_offset, const int64_t* excl, int64_t ld_excl, int n_excl, float* top_scores,
                        int64_t* top_ids, int64_t U, int d, int k, void* ws, size_t ws_bytes, rbm_stream_t stream);
/* top-k of materialised scores [U,C] (ld = row stride), same order rule; id = column + id_offset.
 * replaces (-scores).argsort(dim=1)[:, :k]  NN/trainers/utils.py:36-38 */
int rbm_topk_rows(const float* scores, int64_t ld, float* top_scores, int64_t* top_ids, int64_t U, int64_t C,
                  int k, int64_t id_offset, rbm_stream_t stream);
/* merge S per-shard lists [S,U,k] (global ids, (-inf,-1) padding) into [U,k]; shard-count invariant */
int rbm_topk_merge(const float* scores, const int64_t* ids, float* out_scores, int64_t* out_ids, int S,
                   int64_t U, int k, rbm_stream_t stream);
/* ranking metrics, NN/trainers/utils.py:41-55.  hits[u,t] = labels[u, top_ids[u,t]-id_offset] (labels
 * [U,C] i64) or, when labels==NULL, (top_ids[u,t] == positives[u]).  For each k in ks (nk values, host
 * array, each <= K): per_user[u, j, 0..2] = Recall@k, NDCG@k, MRR@k; w_ndcg/w_mrr: [K] weight tables. */
int rbm_rank_metrics(const int64_t* top_ids, const int64_t* labels, const int64_t* positives,
                     const float* w_ndcg, const float* w_mrr, const int32_t* ks_host, int nk, float* per_user,
                     int64_t U, int K, int64_t C, int64_t id_offset, rbm_stream_t stream);
/* mean over rows of x[U,cols] accumulated in double in fixed order -> out[cols] (fp32); cols <= 256 */
size_t rbm_column_mean_ws_bytes(int64_t U, int cols);
int rbm_column_mean(const float* x, float* out, int64_t U, int cols, void* ws, size_t ws_bytes, rbm_stream_t stream);

/* ---- dense Adam over many tensors in one launch (optim.Adam NN/trainers/base.py:225-233, .step() :123) */
typedef struct {
  float* p;
  const float* g;
  float* m;
  float* v;
  int64_t n;
} rbm_adam_tensor;
/* tensors: DEVICE array of n_tensors descriptors; total_chunks = sum ceil(n/RBM_ADAM_CHUNK);
 * chunk_map: DEVICE int32 [total_chunks*2] = (tensor id, chunk id within tensor). */
#define RBM_ADAM_CHUNK 4096
int rbm_adam_multi(const rbm_adam_tensor* tensors, const int32_t* chunk_map, int total_chunks, double lr,
                   double beta1, double beta2, double eps, double weight_decay, int step, rbm_stream_t stream);
/* flat-bucket helpers for the data-parallel gradient all-reduce: copy n_tensors tensors to/from one
 * contiguous bucket (offsets in elements), optionally scaling. */
typedef struct {
  float* ptr;
  int64_t n;
  int64_t offset;
} rbm_bucket_tensor;
int rbm_bucket_pack(const rbm_bucket_tensor* tensors, const int32_t* chunk_map, int total_chunks, float* bucket,
                    float scale, int unpack, rbm_stream_t stream);

/* ---- CUDA-graph support -------------------------------------------------------------------------------
 * Dropout sites (step*64 + local id) and Adam's step arrive by value, so a captured step would replay the same masks
 * and bias corrections for ever.  After rbm_set_step_counter(ptr) -- ptr = a device uint64, or NULL to switch it off --
 * every kernel adds 64 * (*ptr) to its dropout sites and rbm_adam_multi adds *ptr to `step`; a captured graph
 * increments *ptr itself.  Eager step s and replay number s of a graph captured with step 0 are bit-identical.
 * Synchronous (cudaMemcpyToSymbol), library-wide: call it outside stream capture. */
int rbm_set_step_counter(const uint64_t* counter);

/* ---- device-side batch construction (SURVEY 8(f) #1) -------------------------------------------------
 * User histories arrive as a CSR: hist_ptr[U+1], hist_items[nnz] (int64, ids in 1..num_items, oldest first); `users[B]`
 * selects the rows of the batch.  Randomness is Philox4x32-10(key=seed, counter=(idx4, site)) with the field layout written
 * in csrc/batch.cu (and restated in oracle/batches.py), so a batch is a pure function of (histories, users, seed, site).
 *
 * Cloze masking + left padding of BertTrainDataset.__getitem__ (NN/dataloaders/bert.py:77-110): tokens/labels [B, L] int64;
 * a position is scored with probability mask_prob (label = item, else 0) and then shows [MASK] (80 %), a uniform item of
 * 1..num_items (10 %) or itself (10 %). */
int rbm_bert_cloze_batch(const int64_t* hist_ptr, const int64_t* hist_items, const int64_t* users, int B, int L,
                         double mask_prob, int64_t mask_token, int64_t num_items, uint64_t seed, uint64_t site,
                         int64_t* tokens, int64_t* labels, rbm_stream_t stream);
/* (seq, pos, neg) of sample_function / random_neq (NN/dataloaders/sas.py:65-86): the window is the last L items; seq drops
 * its last item, pos its first; neg[p] is uniform over the ids of [0, num_items] that are not in the window (L <= 256). */
int rbm_sas_train_batch(const int64_t* hist_ptr, const int64_t* hist_items, const int64_t* users, int B, int L,
                        int64_t num_items, uint64_t seed, uint64_t site, int64_t* seq, int64_t* pos, int64_t* neg,
                        rbm_stream_t stream);

/* Evaluation negatives (SURVEY 8(f) #2): `n_samples` distinct items per user that the user has not seen, for users
 * [user_begin, user_begin + num_users).  seen_ptr[U+1] / seen_items: CSR of each user's seen set, ASCENDING and unique.
 * pop_cdf == NULL: uniform over 1..num_items (RandomNegativeSampler, NN/dataloaders/negative_samplers/random.py:13-37);
 * else pop_cdf[num_items] (uint64) = inclusive prefix sums of the interaction counts of items 1..num_items and an item is
 * drawn with probability count/total (PopularNegativeSampler, popular.py:15-44).  Rejection sampling, one thread per user;
 * out [num_users, n_samples] int64 in acceptance order (-1 where 65536 attempts did not suffice).  Philox layout: csrc/batch.cu. */
int rbm_negative_samples(const int64_t* seen_ptr, const int64_t* seen_items, const uint64_t* pop_cdf, int64_t user_begin,
                         int64_t num_users, int64_t num_items, int n_samples, uint64_t seed, uint64_t site, int64_t* out,
                         rbm_stream_t stream);
/* Evaluation batch of BertEvalDataset / SASEvalDataset.__getitem__ (NN/dataloaders/bert.py:128-142, sas.py:136-153):
 * seq [B, L] = last L entries of (history ++ [mask_token] if mask_token >= 0), left-padded with 0;
 * cand [B, 1 + n_neg] = answers[u] then negatives[u, :]; labels [B, 1 + n_neg] = 1 then zeros. */
int rbm_eval_batch(const int64_t* hist_ptr, const int64_t* hist_items, const int64_t* answers, const int64_t* negatives,
                   const int64_t* users, int B, int L, int n_neg, int64_t mask_token, int64_t* seq, int64_t* cand,
                   int64_t* labels, rbm_stream_t stream);

/* ---- test / debug ---------------------------------------------------------------------------------- */
/* materialise the keep-mask (1 = keep) the kernels use for an elementwise site over n elements */
int rbm_dropout_mask(uint8_t* out, int64_t n, float p, uint64_t seed, uint64_t site, rbm_stream_t stream);
/* ... and for an attention site: out [B*h*L, L] */
int rbm_dropout_mask_attn(uint8_t* out, int64_t rows, int L, float p, uint64_t seed, uint64_t site,
                          rbm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RBM_H */
