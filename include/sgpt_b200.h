/*
 * sgpt_b200 — C ABI of the B200-native SGPT bi-encoder hot path.
 *
 * The reference (Muennighoff/sgpt @ 37c8bf09) is pure Python and has no FFI layer; its plug-in boundary is the pair
 * of duck-typed protocols in biencoder/beir/custommodels/exact_search.py:22-32 (embedder: encode_queries /
 * encode_corpus; retriever: search).  This header is the C boundary that sits *underneath* those protocols: every
 * entry point replaces the PyTorch/HF library call(s) cited next to it.  All pointers are DEVICE pointers owned by
 * the caller unless stated otherwise; no torch types cross this boundary.  Every function returns SGPT_OK (0) or an
 * error code; sgpt_last_error() returns a thread-local message.  Nothing throws.  A handle is bound to the device
 * that was current when it was created, is not thread-safe, and may be used on any stream of that device as long
 * as calls are externally ordered.
 *
 * Abbreviations in citations:  BDR = biencoder/beir/beir_dense_retriever.py, XS = .../custommodels/exact_search.py,
 * ST/ = biencoder/nli_msmarco/sentence-transformers/sentence_transformers/, HF: = transformers/models/ (third-party
 * dependency of the reference, pinned >=4.6,<5 by ST's setup.py:21).
 */
#ifndef SGPT_B200_H_
#define SGPT_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGPT_ABI_VERSION 3  /* 3: sgpt_topk_merge_packed requires sorted input lists; sgpt_debug_topk_timeline added */

#define SGPT_OK 0
#define SGPT_ERR_INVALID 1     /* bad argument / unsupported shape */
#define SGPT_ERR_CUDA 2        /* a CUDA runtime/driver call failed */
#define SGPT_ERR_UNSUPPORTED 3 /* valid request this build does not implement */

typedef void* sgpt_stream_t; /* cudaStream_t */

int sgpt_abi_version(void);
const char* sgpt_last_error(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Encoder building blocks (rows F1–F7 of SURVEY.md §8a).  Token-major, *ragged* layout: the B sequences of a batch
 * are packed back to back into T = sum(len_b) rows ("tokens"); padding never exists on the device.
 * ------------------------------------------------------------------------------------------------------------------ */

/* F1. resid[t,:] = wte[ids[t],:] (+ wpe[pos[t],:] if wpe != NULL)       HF:gpt_neo/modeling_gpt_neo.py:462-463
 *     ids,pos int32[T]; wte bf16[vocab,d]; wpe bf16[max_pos,d] or NULL (GPT-J / BLOOM); resid fp32[T,d]. */
int sgpt_embed_tokens(const int32_t* ids, const int32_t* pos, const void* wte, const void* wpe, float* resid,
                      int T, int d, int vocab, int max_pos, sgpt_stream_t stream);

/* F2/F7. y = LayerNorm(x; gamma, beta, eps) row-wise, fp32 statistics, bf16 output.   HF:gpt_neo/...:332,345,492
 *     x fp32[T,d]; gamma,beta fp32[d]; y bf16[T,d]. */
int sgpt_layernorm(const float* x, const float* gamma, const float* beta, void* y, int T, int d, float eps,
                   sgpt_stream_t stream);

/* F3/F5/F6. y = epilogue(x @ w^T + bias).   torch.nn.Linear call sites HF:gpt_neo/...:84-87,153,295-309
 *     x bf16[M,K] (row pitch ldx), w bf16[N,K] (nn.Linear weight layout, row pitch ldw), bias fp32[N] or NULL.
 *     epilogue: SGPT_EPI_BF16       out bf16[M,N]  = acc + bias
 *               SGPT_EPI_GELU_BF16  out bf16[M,N]  = gelu_new(acc + bias)       (HF activations.py NewGELUActivation)
 *               SGPT_EPI_RESID_F32  out fp32[M,N]  = resid + acc + bias         (resid fp32[M,N], may alias out)
 *     Runs on the tcgen05 tensor cores (TMA-staged tiles, TMEM accumulators). */
#define SGPT_EPI_BF16 0
#define SGPT_EPI_GELU_BF16 1
#define SGPT_EPI_RESID_F32 2
#define SGPT_EPI_RESID_BF16 3 /* out bf16[M,N] += acc + bias, in place (resid == out): bf16 residual stream */
int sgpt_linear(const void* x, int64_t ldx, const void* w, int64_t ldw, const float* bias, void* out, int64_t ldo,
                const float* resid, int M, int N, int K, int epilogue, sgpt_stream_t stream);

/* F7'. y[m,:] = LayerNorm(x[rows[m],:]) for a gathered subset of rows (bf16 out): the LM-head input of
 *      sgpt_lm_logprobs.  x fp32[T,d]; rows int32[M] (values in [0,T)); y bf16[M,d]. */
int sgpt_layernorm_gather(const float* x, const int32_t* rows, const float* gamma, const float* beta, void* y, int M,
                          int d, float eps, sgpt_stream_t stream);

/* F2'. In-place fp32 LayerNorm (BLOOM word_embeddings_layernorm, HF:bloom/modeling_bloom.py:496): x fp32[T,d]. */
int sgpt_layernorm_f32_inplace(float* x, const float* gamma, const float* beta, int T, int d, float eps,
                               sgpt_stream_t stream);

/* F3'. GPT-J fused q/k/v projection with rotary position embedding in the epilogue
 *     (HF:gptj/modeling_gptj.py:98-101 bias-free projections, :55-67 + :196-207 rotary on the first rotary_dim dims of
 *     every q and k head, interleaved pairs).  x bf16[M,d] (pitch ldx), w_qkv bf16[3d,d] rows [q|k|v],
 *     qkv bf16[M,3d]; pos int32[M]; cos_sin fp32[max_pos, rotary_dim/2, 2] = (cos, sin) of pos * 10000^(-2i/rotary_dim). */
int sgpt_linear_qkv_rotary(const void* x, int64_t ldx, const void* w_qkv, void* qkv, const int32_t* pos,
                           const float* cos_sin, int M, int d_model, int head_dim, int rotary_dim, int max_pos,
                           sgpt_stream_t stream);

/* F4. Causal self-attention over a ragged batch.    HF:gpt_neo/modeling_gpt_neo.py:105-130 (_attn)
 *     qkv bf16[T, 3*H*hd]: per token [q(H*hd) | k(H*hd) | v(H*hd)];  out bf16[T, H*hd].
 *     cu_seqlens int32[B+1] (row offsets of each sequence; cu[B] == T).
 *     scale: multiplies q.k before softmax (GPT-Neo: 1.0 — unscaled, :110; GPT-J: 1/sqrt(hd)).
 *     window: 0 = plain causal; w > 0 = GPT-Neo local attention (key j visible to query i iff i-w < j <= i, :63-66).
 *     alibi_slopes: fp32[H] or NULL; adds slope_h * (key position in its sequence) to the scaled scores (BLOOM ALiBi,
 *                   HF:bloom/modeling_bloom.py:43-86; the bias depends on the key only).
 *     impl: 0 = tcgen05 tensor-core kernel, 1 = SIMT cross-check kernel (test infrastructure). */
int sgpt_attention(const void* qkv, void* out, const int32_t* cu_seqlens, int B, int T, int H, int hd, float scale,
                   int window, int max_seqlen, const float* alibi_slopes, int impl, sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * P1/P2. Pooling over the ragged sequence dimension, fp32 accumulate.
 *     BDR:258-270 == ST/models/Pooling.py:99-125 (weightedmean), BDR:238-242 (mean), BDR:271-282 (lasttoken)
 *     x fp32[T,d] (residual stream or hidden state); pos int32[T] = index of the token in its *padded* row
 *     (weight of token t is pos[t]+1 for weightedmean); out fp32[B,d].
 *     If gamma != NULL the final LayerNorm (ln_f, F7) is applied to every row on the fly before it is pooled.
 *     clamp_denominator != 0 reproduces ST's clamp(min=1e-9) (Pooling.py:122); 0 reproduces the script (no clamp).
 *     normalize != 0 additionally L2-normalises each output row (ST/models/Normalize.py:13-14).
 * ------------------------------------------------------------------------------------------------------------------ */
#define SGPT_POOL_MEAN 0
#define SGPT_POOL_WEIGHTEDMEAN 1
#define SGPT_POOL_LASTTOKEN 2
/* All-hidden-state modes, accepted by sgpt_encode only: the mean over the L+1 hidden states (embedding output, every
 * block output, ln_f of the last) of the per-state mean / last-token embedding — BDR:243-257 (meanmean: the mask sum is
 * the same for every layer, so sum/sum == mean of means) and BDR:284-301 (lasttokenmean).  layer_idx is ignored, as in
 * the reference. */
#define SGPT_POOL_MEANMEAN 3
#define SGPT_POOL_LASTTOKENMEAN 4
int sgpt_pool(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma, const float* beta,
              float eps, float* out, float* row_stats_ws /* fp32[2*T] scratch */, int B, int T, int d, int mode,
              int clamp_denominator, int normalize, sgpt_stream_t stream);
/* Building block of the all-hidden-state modes: out = (accumulate ? out : 0) + out_scale * pool(x); mode is one of
 * MEAN / WEIGHTEDMEAN / LASTTOKEN; normalize (if set) acts on the accumulated rows, so pass it with the last state. */
int sgpt_pool_accumulate(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                         const float* beta, float eps, float* out, float* row_stats_ws, int B, int T, int d, int mode,
                         int clamp_denominator, int normalize, int accumulate, float out_scale, sgpt_stream_t stream);

/* General form: pos_weights fp32[n_pos_weights] or NULL.  With a table (mode must be WEIGHTEDMEAN) the weight of token t
 * is pos_weights[pos[t]] instead of pos[t]+1 — the learnt per-position weights of
 * ST/models/WeightedMeanPooling.py:21-37 (`position_weights[:positions]`, indexed by the position in the padded row;
 * that module always clamps the denominator, :34).  pos[t] >= n_pos_weights is the caller's error (the reference
 * asserts, :30); the kernel clamps the index instead of reading out of bounds. */
int sgpt_pool_ex(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma, const float* beta,
                 float eps, const float* pos_weights, int n_pos_weights, float* out, float* row_stats_ws, int B, int T,
                 int d, int mode, int clamp_denominator, int normalize, int accumulate, float out_scale,
                 sgpt_stream_t stream);

/* Sentence-embedding head applied after pooling: y = act(x @ w^T + bias), all fp32 (ST/models/Dense.py:40-43 with
 * key_name "sentence_embedding"; nn.Linear weight layout).  x fp32[B,in], w fp32[out,in], bias fp32[out] or NULL,
 * y fp32[B,out] (must not alias x). */
#define SGPT_ACT_IDENTITY 0
#define SGPT_ACT_TANH 1
#define SGPT_ACT_RELU 2
#define SGPT_ACT_SIGMOID 3
int sgpt_dense(const float* x, const float* w, const float* bias, float* y, int B, int in_features, int out_features,
               int activation, sgpt_stream_t stream);

/* P2 stand-alone: x[b,:] /= max(||x[b,:]||_2, 1e-12) in place (ST/models/Normalize.py:13-14;
 * SentenceTransformer.py:248-249) for embeddings that passed through a head after pooling.  x fp32[B,d]. */
int sgpt_normalize_rows(float* x, int B, int d, sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Whole-encoder handle (F1..F7 + P1 in one call).
 * ------------------------------------------------------------------------------------------------------------------ */
#define SGPT_ARCH_GPT_NEO 0
#define SGPT_ARCH_GPTJ 1
#define SGPT_ARCH_BLOOM 2

typedef struct sgpt_model_config {
  int32_t arch;
  int32_t n_layer, d_model, n_head, d_ff, vocab, max_pos;
  int32_t window;     /* GPT-Neo local-attention window (256) */
  int32_t rotary_dim; /* GPT-J */
  float ln_eps;
  int32_t max_tokens; /* workspace capacity: largest T a single sgpt_encode call may carry */
  int32_t max_batch;  /* largest B */
} sgpt_model_config;

/* Per-layer device pointers.  Linear weights are bf16 in nn.Linear layout [out,in]; biases and LayerNorm
 * parameters are fp32.  Unused entries (arch-dependent) are NULL. */
typedef struct sgpt_layer_weights {
  const float *ln1_g, *ln1_b;
  const void* w_qkv;   /* bf16[3d, d]: rows [q | k | v] */
  const float* b_qkv;  /* fp32[3d] or NULL (GPT-Neo / GPT-J have no q,k,v bias) */
  const void* w_o;     /* bf16[d, d] */
  const float* b_o;    /* fp32[d] or NULL */
  const float *ln2_g, *ln2_b;
  const void* w_fc;    /* bf16[ff, d] */
  const float* b_fc;   /* fp32[ff] */
  const void* w_proj;  /* bf16[d, ff] */
  const float* b_proj; /* fp32[d] */
  int32_t local_attention; /* GPT-Neo: 1 for "local" layers */
  int32_t _pad;
} sgpt_layer_weights;

typedef struct sgpt_model_weights {
  const void* wte; /* bf16[vocab, d] */
  const void* wpe; /* bf16[max_pos, d] or NULL */
  const float *lnf_g, *lnf_b;
  const sgpt_layer_weights* layers; /* HOST array of n_layer entries (copied at create) */
  const float *emb_ln_g, *emb_ln_b; /* BLOOM word_embeddings_layernorm, else NULL */
} sgpt_model_weights;

typedef struct sgpt_model* sgpt_model_t;

/* Replaces AutoModel.from_pretrained(...).to(device) at BDR:123 / ST/models/Transformer.py:38 (weights are handed
 * over already on the device; the handle borrows them and owns its activation workspace and the LayerNorm-folded copies
 * it derives at creation: per layer w_qkv, b_qkv, w_fc, b_fc and ln1 / ln2 are folded into library-owned buffers
 * (sgpt_fold_layernorm) and are NOT referenced after sgpt_model_create returns — the caller may free them; wte, wpe, w_o,
 * b_o, w_proj, b_proj, ln_f and the embedding LayerNorm stay borrowed).  Synchronises the device. */
int sgpt_model_create(const sgpt_model_config* cfg, const sgpt_model_weights* w, sgpt_model_t* out);
void sgpt_model_destroy(sgpt_model_t m);

/* Replaces self.model(**batch_tokens, output_hidden_states=True) + pooling, BDR:205 + BDR:233-304
 * (ST path: ST/models/Transformer.py:72 + ST/models/Pooling.py:85-168).
 *     ids,pos int32[T]; cu_seqlens int32[B+1]; out fp32[B,d].
 *     layer_idx: which entry of HF hidden_states to pool: -1 / n_layer = after ln_f (the reference default, BDR:44);
 *                0..n_layer-1 = input of block i (no final LayerNorm). */
int sgpt_encode(sgpt_model_t m, const int32_t* ids, const int32_t* pos, const int32_t* cu_seqlens, int B, int T,
                int max_seqlen, int layer_idx, int pool_mode, int clamp_denominator, int normalize, float* out,
                sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Continuation log-likelihoods with the same encoder (SURVEY.md §8f row 4; the SGPT cross-encoder scorer,
 * crossencoder/beir/sgptce.py:150-262 `_loglikelihood_tokens`).
 * ------------------------------------------------------------------------------------------------------------------ */

/* The GPT forward pass alone (F1..F6 of every block): replaces `model(inps)` at sgptce.py:76-83 up to the final
 * LayerNorm.  Leaves the fp32 residual stream [T,d] in the handle for sgpt_lm_logprobs / sgpt_model_read_residual. */
int sgpt_forward(sgpt_model_t m, const int32_t* ids, const int32_t* pos, const int32_t* cu_seqlens, int B, int T,
                 int max_seqlen, sgpt_stream_t stream);

/* token_logprobs[i] = log_softmax(LN_f(resid[rows[i]]) @ lm_head_w^T + lm_head_bias)[targets[i]]
 *     == F.log_softmax(logits, -1) (sgptce.py:221) gathered at the continuation tokens (:247), for the packed token
 *     rows `rows` of the batch the last sgpt_forward ran.  lm_head_w bf16[vocab,d] (the tied wte for GPT-Neo / BLOOM,
 *     lm_head.weight for GPT-J), lm_head_bias fp32[vocab] or NULL (GPT-J has one); rows,targets int32[M];
 *     greedy int32[M] or NULL receives argmax(logits) (:229, lowest index on ties).  The [M,vocab] logits exist only in
 *     `ws`, rows_per_chunk rows at a time (ws >= sgpt_lm_logprobs_workspace_bytes(d_model, vocab, rows_per_chunk)). */
int64_t sgpt_lm_logprobs_workspace_bytes(int d_model, int vocab, int rows_per_chunk);
int sgpt_lm_logprobs(sgpt_model_t m, const void* lm_head_w, const float* lm_head_bias, int vocab, const int32_t* rows,
                     const int32_t* targets, int M, float* token_logprobs, int32_t* greedy, void* ws, int64_t ws_bytes,
                     int rows_per_chunk, sgpt_stream_t stream);

/* Building blocks of the above.  sgpt_token_logprobs: logits fp32[M,lds] (vocab valid columns) -> log-softmax value of
 * the target column per row (+ optional argmax).  sgpt_segment_sum: out[r] = sum(x[offsets[r]..offsets[r+1])) in index
 * order — the per-request `float(logits.sum())` of sgptce.py:250; offsets int32[R+1]. */
int sgpt_token_logprobs(const float* logits, int64_t lds, int M, int vocab, const float* bias, const int32_t* targets,
                        float* logprob, int32_t* greedy, sgpt_stream_t stream);
int sgpt_segment_sum(const float* x, const int32_t* offsets, int R, float* out, sgpt_stream_t stream);

/* Installs (w != NULL) or removes (w == NULL) a learnt position-weight table for pool_mode WEIGHTEDMEAN in sgpt_encode
 * (ST/models/WeightedMeanPooling.py).  w is a DEVICE fp32[n] buffer borrowed by the handle; sgpt_encode then fails with
 * SGPT_ERR_INVALID when max_seqlen > n, like the reference's shape assert (:30). */
int sgpt_model_set_position_weights(sgpt_model_t m, const float* w, int n);

/* Debug/parity tap: copies the fp32 residual stream (hidden_states[layer] before ln_f) left by the LAST sgpt_encode
 * into dst (device, capacity_elems floats) and reports its shape. */
int sgpt_model_read_residual(sgpt_model_t m, float* dst, int64_t capacity_elems, int* T, int* d, sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * S1–S3. Exact dense retrieval over one corpus shard.
 * ------------------------------------------------------------------------------------------------------------------ */

/* inv_norm[i] = 1 / max(||x_i||_2, 1e-12) for bf16 rows (F.normalize semantics, ST/util.py:41-42).  x bf16[n,D]. */
int sgpt_row_inv_norms(const void* x, float* inv_norm, int64_t n, int D, sgpt_stream_t stream);

/* fp32 -> bf16 row conversion (round-to-nearest-even) used to store embeddings in a shard. */
int sgpt_f32_to_bf16(const float* x, void* y, int64_t count, sgpt_stream_t stream);

/* Element types of a corpus shard (and of the queries searched against it): the `elem` argument of the _ex entry
 * points below.  SGPT_ELEM_I8 = int8 rows quantized per row by sgpt_quantize_rows_i8 (D a multiple of 16, D <= 65536). */
#define SGPT_ELEM_BF16 0
#define SGPT_ELEM_I8 1

/* Symmetric per-row int8 quantization, for corpus rows and query rows alike.  x fp32[n,D] (x_is_bf16 = 0) or bf16[n,D]
 * (x_is_bf16 = 1, widened exactly); per row: s = max_j |x_j| / 127 (IEEE fp32), c_j = clamp(rint(x_j / s), -127, 127)
 * (round-half-even; s = 0 gives c = 0), inv = 1 / max(sqrt((float)sum_j c_j^2), 1e-12).  out int8[n,D], scale fp32[n]
 * = s, inv_norm fp32[n] = inv.  An int8 search then scores cos_sim = ((float)acc * inv_q) * inv_d and
 * dot = ((float)acc * s_q) * s_d with acc = sum_j cq_j cd_j exact in int32: cos_sim / dot_score of the dequantized rows
 * s * c.  Rows must be finite (not checked here: the Python layer rejects non-finite rows).  D % 16 == 0, D <= 65536. */
int sgpt_quantize_rows_i8(const void* x, int x_is_bf16, int64_t n, int D, int8_t* out, float* scale, float* inv_norm,
                          sgpt_stream_t stream);

/* S1. scores[q,j] = fixnan( <Q[q,:], C[j,:]> * q_scale[q] * c_scale[j] )      ST/util.py:24-63, XS:96-99
 *     Q bf16[nq,D], C bf16[n,D], q_scale fp32[nq]|NULL, c_scale fp32[n]|NULL (NULL = 1: dot_score),
 *     scores fp32[nq, lds]; NaN -> -1 as XS:99.  tcgen05 GEMM, corpus streamed once from HBM. */
int sgpt_scores(const void* Q, const void* C, const float* q_scale, const float* c_scale, float* scores, int64_t lds,
                int nq, int64_t n, int D, sgpt_stream_t stream);

/* S2. Row-wise exact top-k of a score matrix (torch.topk(..., largest=True, sorted=False), XS:102-108), with the
 *     winners returned in DESCENDING score order (ties: ascending id).  ids are offset by id_base (global doc ids of a
 *     shard).  scores fp32[nq, lds] (n valid columns); out_scores fp32[nq,k]; out_ids int64[nq,k].
 *     If n < k the tail is filled with (-inf, -1).  ws: scratch of sgpt_topk_workspace_bytes(nq,n,k) bytes. */
int64_t sgpt_topk_workspace_bytes(int nq, int64_t n, int k);
int sgpt_topk(const float* scores, int64_t lds, int nq, int64_t n, int k, int64_t id_base, float* out_scores,
              int64_t* out_ids, void* ws, sgpt_stream_t stream);

/* S3. Merge G candidate lists per query (cross-chunk heapq.nlargest merge XS:121-132; cross-shard merge after the
 *     all-gather): in_scores fp32[G,nq,k], in_ids int64[G,nq,k] -> out fp32/int64[nq,k], descending; entries with
 *     id < 0 are ignored, and so are entries whose id equals exclude_ids[q] (the `corpus_id != query_id` self-match
 *     rule of XS:118; exclude_ids int64[nq] or NULL). */
int sgpt_topk_merge(const float* in_scores, const int64_t* in_ids, int G, int nq, int k, float* out_scores,
                    int64_t* out_ids, const int64_t* exclude_ids, void* ws, sgpt_stream_t stream);

/* S1+S2 in one call: exact top-k of one corpus shard for a batch of queries (XS:96-108 for one chunk).
 *     Q bf16[nq,D], C bf16[n,D], q_scale/c_scale as sgpt_scores; out_scores fp32[nq,k], out_ids int64[nq,k]
 *     (descending, ids offset by id_base, tail (-inf,-1) when n < k).  ws: sgpt_search_workspace_bytes(nq,n,k). */
int64_t sgpt_search_workspace_bytes(int nq, int64_t n, int k);
int sgpt_search(const void* Q, const void* C, const float* q_scale, const float* c_scale, int nq, int64_t n, int D,
                int k, int64_t id_base, float* out_scores, int64_t* out_ids, void* ws, int64_t ws_bytes,
                sgpt_stream_t stream);

/* Same search, result as ONE packed list: out_packed uint64[nq,k], entry = (int32 global id << 32) | fp32 score bits,
 *     descending, empty slots (-inf, -1); requires id_base + n < 2^31.  This is the 8-byte entry of SURVEY.md §8e: one
 *     all-gather of Q*(k+1)*8 bytes per rank when the exchange goes through NCCL (sgpt_b200/dist.py). */
int sgpt_search_packed(const void* Q, const void* C, const float* q_scale, const float* c_scale, int nq, int64_t n,
                       int D, int k, int64_t id_base, uint64_t* out_packed, void* ws, int64_t ws_bytes,
                       sgpt_stream_t stream);
/* sgpt_search / sgpt_search_packed for either element type (SGPT_ELEM_BF16: identical to the calls above;
 * SGPT_ELEM_I8: Q int8[nq,D] and C int8[n,D] from sgpt_quantize_rows_i8, q_scale / c_scale = the inverse norms for
 * cos_sim or the scales for dot).  Same workspace size for both types.  SGPT_ERR_INVALID before any CUDA call for an
 * unknown elem, an int8 D that is not a multiple of 16 or exceeds 65536, or a null output. */
int sgpt_search_ex(const void* Q, const void* C, const float* q_scale, const float* c_scale, int nq, int64_t n, int D,
                   int k, int64_t id_base, float* out_scores, int64_t* out_ids, void* ws, int64_t ws_bytes, int elem,
                   sgpt_stream_t stream);
int sgpt_search_packed_ex(const void* Q, const void* C, const float* q_scale, const float* c_scale, int nq, int64_t n,
                          int D, int k, int64_t id_base, uint64_t* out_packed, void* ws, int64_t ws_bytes, int elem,
                          sgpt_stream_t stream);
/* S3 on packed lists: in_packed uint64[G,nq,k] (the all-gathered sgpt_search_packed outputs; chunk = shard in
 *     XS:121-132) -> out_scores fp32[nq,k], out_ids int64[nq,k]; ids < 0 and ids == exclude_ids[q] (XS:118) dropped.
 *     Every input list must be in the order sgpt_search_packed writes (score descending, id ascending on ties, empty
 *     slots last) and ids must be unique across the lists (disjoint shards): the merge ranks entries by binary search
 *     instead of selecting and sorting again. */
int sgpt_topk_merge_packed(const uint64_t* in_packed, int G, int nq, int k, float* out_scores, int64_t* out_ids,
                           const int64_t* exclude_ids, sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * §8e without a collective library call: the per-shard top-k lists are PUSHED into every rank's gather buffer by the
 * final selection kernel itself (stores through NVLink peer mappings + a system-scope release per query) and merged by
 * a kernel that acquires those per-query counters — the reference's sequential chunk/heapq merge (XS:80-132) with
 * chunk = GPU.  One context per process (= per GPU):
 *   sgpt_gather_create    allocates this rank's buffer and returns its CUDA IPC handle (SGPT_IPC_HANDLE_BYTES bytes);
 *   sgpt_gather_connect   maps the buffers of all ranks from the concatenated handles [world][SGPT_IPC_HANDLE_BYTES]
 *                         (exchanged by the host, e.g. torch.distributed.all_gather_object);
 *   sgpt_search_gather    = sgpt_search on this rank's shard + push + merge: every rank of the group must call it with
 *                         the same nq and k, in the same order; all ranks receive the identical merged top-k
 *                         (out_scores fp32[nq,k], out_ids int64[nq,k], self matches exclude_ids[q] dropped).
 * ------------------------------------------------------------------------------------------------------------------ */
#define SGPT_IPC_HANDLE_BYTES 64
typedef struct sgpt_gather* sgpt_gather_t;
int sgpt_gather_create(int rank, int world, int nq_cap, int k, sgpt_gather_t* out, void* handle_out);
int sgpt_gather_connect(sgpt_gather_t g, const void* all_handles);
void sgpt_gather_destroy(sgpt_gather_t g);
int sgpt_search_gather(sgpt_gather_t g, const void* Q, const void* C, const float* q_scale, const float* c_scale,
                       int nq, int64_t n, int D, int k, int64_t id_base, const int64_t* exclude_ids, float* out_scores,
                       int64_t* out_ids, void* ws, int64_t ws_bytes, sgpt_stream_t stream);
/* sgpt_search_gather for either element type (elem and its checks as sgpt_search_ex). */
int sgpt_search_gather_ex(sgpt_gather_t g, const void* Q, const void* C, const float* q_scale, const float* c_scale,
                          int nq, int64_t n, int D, int k, int64_t id_base, const int64_t* exclude_ids,
                          float* out_scores, int64_t* out_ids, void* ws, int64_t ws_bytes, int elem,
                          sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Residual stream in bf16 (SGPT_RESID_BF16=1 when the model handle is created; default fp32).  HF keeps hidden_states in
 * the model dtype, i.e. bf16 for the reference's bf16 configs (BASELINE configs 3-5); the `_ex` entry points take the
 * residual stream as `const void*` + a flag.  sgpt_linear(..., SGPT_EPI_RESID_BF16) adds into it with a bf16 TMA reduce.
 * ------------------------------------------------------------------------------------------------------------------ */
int sgpt_embed_tokens_ex(const int32_t* ids, const int32_t* pos, const void* wte, const void* wpe, void* resid, int T,
                         int d, int vocab, int max_pos, int resid_bf16, sgpt_stream_t stream);
int sgpt_layernorm_ex(const void* x, int x_bf16, const float* gamma, const float* beta, void* y, int T, int d, float eps,
                      sgpt_stream_t stream);
int sgpt_layernorm_gather_ex(const void* x, int x_bf16, const int32_t* row_idx, const float* gamma, const float* beta,
                             void* y, int M, int d, float eps, sgpt_stream_t stream);
int sgpt_pool_ex2(const void* x, int x_bf16, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                  const float* beta, float eps, const float* pos_weights, int n_pos_weights, float* out,
                  float* row_stats_ws, int B, int T, int d, int mode, int clamp_denominator, int normalize,
                  int accumulate, float out_scale, sgpt_stream_t stream);
int sgpt_bf16_to_f32(const void* x, float* y, int64_t count, sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * LayerNorm without a pass of its own (F2 fused into F3 / F6 / F7).  HF applies ln_1 / ln_2 as separate modules
 * (HF:gpt_neo/modeling_gpt_neo.py:332,345); here
 *   - the kernels that write the residual stream also emit xb = bf16(resid) and, per row and 128-column group, the
 *     partial sums (sum x, sum x^2): sgpt_resid_stats (after the embedding) and sgpt_linear_resid_ln (out-proj / c_proj:
 *     resid += x w^T + bias in place, one TMA load + store of the residual tile in the GEMM epilogue);
 *   - the consuming GEMM runs on xb with gamma folded into its weights (sgpt_fold_layernorm, once per model):
 *     out = act( r_t * (xb W'^T) - r_t mu_t * colsum + bias' ), (mu_t, r_t) rebuilt from the partial sums
 *     (sgpt_linear_lnfold; sgpt_linear_qkv_rotary_lnfold adds GPT-J's rotary embedding);
 *   - ln_f + pooling read the same partial sums (sgpt_pool_partials).
 * row_stats: float2[M, n_groups], n_groups = ceil(d / 128).  eps: LayerNorm epsilon.
 * ------------------------------------------------------------------------------------------------------------------ */
int sgpt_fold_layernorm(const void* w, const float* gamma, const float* beta, const float* bias, void* w_out,
                        float* colsum_out, float* bias_out, int N, int K, sgpt_stream_t stream);
int sgpt_resid_stats(const float* resid, void* xb, float* stats, int T, int d, sgpt_stream_t stream);
int sgpt_linear_lnfold(const void* x_bf16, int64_t ldx, const void* w_folded, int64_t ldw, const float* bias_folded,
                       const float* colsum, const float* row_stats, int n_groups, float eps, void* out, int64_t ldo,
                       int M, int N, int K, int gelu, sgpt_stream_t stream);
int sgpt_linear_qkv_rotary_lnfold(const void* x_bf16, int64_t ldx, const void* w_folded, const float* bias_folded,
                                  const float* colsum, const float* row_stats, int n_groups, float eps, void* qkv,
                                  const int32_t* pos, const float* cos_sin, int M, int d_model, int head_dim,
                                  int rotary_dim, int max_pos, sgpt_stream_t stream);
int sgpt_linear_resid_ln(const void* x, int64_t ldx, const void* w, int64_t ldw, const float* bias, float* resid,
                         void* xb_out, float* stats_out, int M, int N, int K, sgpt_stream_t stream);
int sgpt_pool_partials(const float* x, const int32_t* pos, const int32_t* cu_seqlens, const float* gamma,
                       const float* beta, float eps, const float* pos_weights, int n_pos_weights, float* out,
                       const float* partial_stats, int n_partials, float* sumsq_ws, int B, int T, int d, int mode,
                       int clamp_denominator, int normalize, int accumulate, float out_scale, sgpt_stream_t stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Measurement hooks (bench.py): launch counters are always on; with profiling enabled every kernel launch issued
 * through this library is bracketed by CUDA events on its stream.  sgpt_profile_read waits for them, returns the
 * summed device milliseconds and launch counts per category since the previous read, and resets the timed set.
 * Categories: 0 embed, 1 layernorm, 2 linear GEMM, 3 attention, 4 pool, 5 similarity GEMM, 6 top-k, 7 misc.
 * ------------------------------------------------------------------------------------------------------------------ */
#define SGPT_NUM_LAUNCH_CATEGORIES 8
int sgpt_profile_enable(int on);
int sgpt_profile_read(double* ms_by_cat, int64_t* timed_launches_by_cat, int64_t* total_launches_by_cat);
/* SM clock the tcgen05 GEMM kernels actually ran at: every GEMM launch has one thread read %clock64 and %globaltimer
 * at its start and end and accumulate both deltas on the device.  Returns the accumulated SM cycles and nanoseconds
 * since the previous call (cycles / ns = GHz under load, which nvidia-smi sampling cannot resolve) and resets them.
 * Synchronises the device. */
int sgpt_profile_gemm_clock(double* sm_cycles, double* nanoseconds);
/* Phase timeline of the most recent exact-selection launch (topk.cu): %globaltimer nanoseconds stamped by CTA 0 at
 * [0] kernel entry, [1] predecessor complete, [2] front/back decision, [3] list offsets, [4] keys in shared memory,
 * [5] sample pivot, [6] compaction, [7] exact k-th key, [8] winners placed + ids fetched, [9] sorted, [10] outputs
 * written.  n <= 16.  Synchronises the device.  A measurement aid, not part of any reference interface. */
int sgpt_debug_topk_timeline(uint64_t* stamps_ns, int n);

#ifdef __cplusplus
}
#endif
#endif /* SGPT_B200_H_ */
