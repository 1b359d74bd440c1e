/* rp_b200.h - C ABI of librp_b200.so: the B200 (sm_100a) kernels behind RePlay's sequential-recommender hot path.
 *
 * The reference (sb-ai-lab/RePlay @ b4e051e8) has NO FFI on this path: its extension points are Python protocols and
 * Lightning hooks (SURVEY.md §8b).  Each entry point below therefore cites the reference *Python* call it replaces;
 * INTEGRATION.md shows the ctypes stub a RePlay maintainer would add at that call site.
 *
 * Conventions (all functions):
 *   - caller owns all memory; pointers are device pointers unless the name says host; no allocation inside;
 *   - asynchronous with respect to the host, ordered on `stream` (a cudaStream_t / CUstream passed as void*);
 *   - scratch memory is passed in by the caller, sized by the matching *_workspace() function;
 *   - return value: 0 = ok, < 0 = argument / shape / alignment error (RP_E*), > 0 = a cudaError_t;
 *   - never throws, keeps no global mutable state besides cached driver entry points / device attributes;
 *   - bf16 tensors are row-major with 16-byte aligned base and row pitch.
 */
#ifndef RP_B200_H
#define RP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RP_OK 0
#define RP_EINVAL (-1)     /* null pointer / unsupported flag */
#define RP_ESHAPE (-2)     /* unsupported size */
#define RP_EALIGN (-3)     /* pointer or pitch not 16-byte aligned */
#define RP_EDRIVER (-4)    /* CUDA driver entry point unavailable / tensor-map encode failed */
#define RP_EWORKSPACE (-5) /* workspace too small */

/* library / build info: returns a static string such as "rp_b200 0.1 sm_100a" */
const char* rp_version(void);

/* ---------------------------------------------------------------------------------------------------------------
 * Predict head:  logits = hq . table^T  ->  seen-item mask  ->  top-K        (one fused pass, logits never stored)
 *   replaces  EmbeddingTyingHead.forward          replay/nn/head.py:29-34
 *                                                  replay/models/nn/sequential/sasrec/model.py:286-307 (legacy)
 *             SeenItemsFilter._compute_scores     replay/nn/lightning/postprocessor/seen_items.py:56-83
 *             RemoveSeenItems._compute_scores     replay/models/nn/sequential/postprocessors/postprocessors.py:55-95
 *             torch.topk(logits, k, dim=1)        replay/nn/lightning/callback/predictions_callback.py:90
 *                                                  replay/models/nn/sequential/callbacks/prediction_callbacks.py:93
 * ------------------------------------------------------------------------------------------------------------- */

/* seen_ids int64 [n_users, S] (any order, duplicates allowed, ids outside [0,item_count) are padding)
 *   -> out_sorted int32 [n_users, S], ascending, padding = INT32_MAX.
 * inv_map (optional, int32 [item_count]): position of each item in candidates_to_score, -1 if absent; when given the
 * output holds candidate positions instead of item ids (seen_items.py:68-71,80-81). */
int rp_seen_prepare(const int64_t* seen_ids, int n_users, int S, int item_count, const int32_t* inv_map,
                    int32_t* out_sorted, void* stream);

size_t rp_score_topk_workspace(int n_users, int n_items, int d, int K);

/* hq bf16 [n_users, d]; table bf16 [n_items, d] (the rows that are scored: all items, or the gathered candidates);
 * bias fp32 [round_up(n_items,128)] or NULL (BERT4Rec head); seen_sorted from rp_seen_prepare or NULL (no filter); candidates int64 [n_items] or NULL
 * (maps a scored column back to an item id, predictions_callback.py:91-92).
 * out_ids int64 [n_users, K], out_scores fp32 [n_users, K], sorted by (score desc, column asc).
 * d in {64,128,256,512}; 1 <= K <= 32. */
int rp_score_topk(const void* hq, const void* table, const float* bias, const int32_t* seen_sorted, int S, int n_users,
                  int n_items, int d, int K, const int64_t* candidates, int64_t* out_ids, float* out_scores,
                  void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Training head: full-catalog cross entropy fused with the logits GEMM, forward and backward
 *   replaces  logits = hidden . E^T                 replay/nn/head.py:29-34 ; replay/nn/sequential/sasrec/model.py:258-265
 *             torch.nn.CrossEntropyLoss (mean)       replay/nn/loss/ce.py:49-81
 *                                                    replay/models/nn/sequential/sasrec/lightning.py:335-355
 *                                                    replay/models/nn/sequential/bert4rec/lightning.py:332-351
 *             and autograd's backward of both.
 * hc bf16 [capacity, d]: hidden rows of the VALID targets, compacted (rows >= *n_valid are ignored but must be finite);
 * table bf16 [n_items, d] (tied item table or the untied Linear weight); bias fp32 [round_up(n_items,128)] or NULL
 * (bert4rec/model.py:363-382: logits = F.linear(h, W, b)); d_bias fp32 [n_items] is overwritten when bias is given;
 * labels int32 [capacity]; n_valid int32 [1] IN DEVICE MEMORY (keeps the step graph-capturable).
 * ------------------------------------------------------------------------------------------------------------- */
size_t rp_ce_head_workspace(int capacity_tokens, int n_items, int d);

/* loss_out fp32 [2] = { mean CE over the valid targets, 1 / n_valid }; lse fp32 [capacity];
 * cvec fp32 [round_up(capacity,128)] (per-token exponent offsets for the backward; entries >= capacity must be -inf).
 * d_hc (optional, bf16 [capacity, d], d <= 256): enables the FUSED training path - a single pass accumulates the row sums of
 * exp(s) against a fixed reference maximum together with the un-normalised gradient sum_i exp(s_i) E_i, so the separate
 * log-sum-exp pass disappears and d_hc is final after this call.  A device-side Cauchy-Schwarz bound on |s| guards the
 * trick; when it fails the two-pass kernels run instead (both variants are enqueued, the losing one exits immediately), so
 * the call stays CUDA-graph capturable.  n_valid_hint: host estimate of *n_valid (0 = unknown), load-balance only. */
int rp_ce_head_fwd(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                   int capacity, int n_items, int d, float* loss_out, float* lse, float* cvec, void* d_hc, int n_valid_hint,
                   void* workspace, size_t workspace_bytes, void* stream);

/* gradients of the mean CE for d(loss) = 1:  d_hc bf16 [capacity, d] (rows < *n_valid; already produced by the forward when
 * `fused` != 0 and the bound held, otherwise computed here); d_table fp32 [n_items, d] is OVERWRITTEN (softmax part) and
 * then atomically corrected by the one-hot part; d_bias fp32 [n_items] likewise iff bias.  `fused` must equal
 * (d_hc != NULL) of the matching forward call and then needs the same workspace.  d in {64,128,256}: fused tcgen05 passes
 * (logits never leave TMEM).  d = 512 (bias == NULL only): S plus a [128 x 512] fp32 accumulator exceed the 512 TMEM columns, so
 * the softmax numerators of a token chunk are materialised in bf16 inside the workspace (chunk sized by RP_CE_WIDE_G_BYTES,
 * default 8 GiB) and three GEMMs per chunk produce dH and dE; the workspace is then always required.
 * n_valid_hint: host estimate of *n_valid (0 = unknown), load-balance only. */
/* Per-row variants of the full-catalog head, single positive label per position:
 *   row_weight  fp32 [capacity], >= 0, in the compacted order of the valid targets (NULL = 1): loss = mean_t w_t ce_t
 *               replaces  replay/nn/loss/logout_ce.py:148-228 LogOutCEWeighted (and :10-145 LogOutCE = the plain head) ;
 *                         replay/nn/loss/ce.py:84-143 CEWeighted
 *   loss_kind 1 LogInCE   replay/nn/loss/login_ce.py:102-239: loss_t = -clamp(log(p_t + log_eps), -clamp, clamp) with p_t the
 *               softmax probability of the positive over the catalog; gradient = CE gradient of the row x p / (p + eps)
 * Same buffers and fused behaviour as rp_ce_head_fwd; rp_ce_head_bwd with the same workspace completes it. */
int rp_ce_head_fwd_w(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                     int capacity, int n_items, int d, float* loss_out, float* lse, float* cvec, void* d_hc, int n_valid_hint,
                     const float* row_weight, int loss_kind, float log_eps, float clamp, void* workspace,
                     size_t workspace_bytes, void* stream);
int rp_ce_head_bwd(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                   int capacity, int n_items, int d, const float* loss_out, const float* cvec, void* d_hc, float* d_table,
                   float* d_bias, int fused, int n_valid_hint, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Training head: full-catalog pointwise BCE fused with the logits GEMM
 *   replaces  BCE (BCEWithLogitsLoss(reduction="sum") / T_v against a one-hot row)   replay/nn/loss/bce.py:10-95
 *             legacy SasRec(loss_type="BCE")._compute_loss_bce                       sasrec/lightning.py:278-308
 *             legacy Bert4Rec(loss_type="BCE")._compute_loss_bce                     bert4rec/lightning.py:273-305
 *   loss = (1/T_v) sum_t [ sum_i softplus(s_ti) - s_t,y_t ],  s = h.E_i + b_i (fp32), never materialised.
 * Same conventions as rp_ce_head_*: hc / table / bias / labels / n_valid as there (n_valid in device memory: graph-capturable),
 * d in {64, 128, 256} (512: RP_ESHAPE).  fwd: loss_out fp32 [2] = { mean BCE, 1 / n_valid } and d_hc bf16 [capacity, d]
 * (required: one fused forward + dH pass) final after the call.  bwd (same workspace and loss_out): d_table fp32
 * [n_items, d] and d_bias fp32 [n_items] (iff bias) are OVERWRITTEN.  n_valid_hint: load balance only (0 = unknown).
 * ------------------------------------------------------------------------------------------------------------- */
size_t rp_bce_head_workspace(int capacity_tokens, int n_items, int d);
int rp_bce_head_fwd(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                    int capacity, int n_items, int d, float* loss_out, void* d_hc, int n_valid_hint, void* workspace,
                    size_t workspace_bytes, void* stream);
int rp_bce_head_bwd(const void* hc, const void* table, const float* bias, const int32_t* labels, const int32_t* n_valid,
                    int capacity, int n_items, int d, const float* loss_out, float* d_table, float* d_bias, void* workspace,
                    size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Transformer body.  All activations are token-major bf16 [T = B*L, d]; weights are the bf16 shadow of the fp32 masters.
 * ------------------------------------------------------------------------------------------------------------- */

/* Generic batched GEMM  C[m,n] = epilogue(alpha * sum_k A(m,k) B(n,k))  on tcgen05.
 *   replaces  torch.nn.MultiheadAttention in/out projections   replay/nn/sequential/sasrec/transformer.py:36-46,99-106
 *             Conv1d(d,d,1) / Linear FFN layers                  replay/nn/ffn.py:43-57 ; models/nn/sequential/sasrec/model.py:490-506
 *                                                                models/nn/sequential/bert4rec/model.py:516-527
 *             and autograd's backward of all of them (dX = dY.W, dW = dY^T.X read in place through MN-major descriptors).
 * Operand X is a 2-D bf16 array [x_rows, x_cols] with pitch ldx; x_mn = 0: stored [M or N rows, K cols] (K-major),
 * x_mn = 1: stored [K rows, M or N cols].  Batch element bz = outer*inner + in addresses rows r0 + outer*ro + in*ri and
 * columns c0 + outer*co + in*ci.  C: element offset c_off0 + outer*c_oo + in*c_oi, row pitch ldc.
 * out_mode 0: bf16 store, 1: fp32 atomic add (split_k >= 1), 2: fp32 store, 3: fp32 store of the split-K partial at
 * C + ksplit * c_split_stride (deterministic two-stage split-K; reduce with rp_reduce_splits), 4: fp32 C += x as a plain
 * read-modify-write (split_k == 1, every element has one owner).
 * Epilogue order: alpha, bias[N], act (0 none, 1 ReLU, 2 GELU-erf, 3 exp2 with a per-row offset), Philox dropout(drop_p; seed + *seed_ptr, drop_offset +
 * element offset in C), gate (x *= gate != 0 ? gate_scale : 0, same geometry as C), residual (bf16, same geometry as C),
 * post-residual dropout (post_drop_p, post_drop_offset), rowmask[rowmask_off0 + outer*rowmask_oo + m].
 * C2 (optional, bf16, geometry of C) receives the value after the bias and before the activation; gate_mode 1 multiplies
 * by gelu'(gate) instead of the (gate != 0) test. */
typedef struct rp_gemm_desc {
  const void* A; long long a_rows, a_cols, lda; int a_mn;
  const void* B; long long b_rows, b_cols, ldb; int b_mn;
  int M, N, K, batch, inner;
  int a_r0, a_ro, a_ri, a_c0, a_co, a_ci;
  int b_r0, b_ro, b_ri, b_c0, b_co, b_ci;
  void* C; long long ldc, c_off0, c_oo, c_oi; int out_mode;
  float alpha; const float* bias; int act;
  const void* residual; const uint8_t* rowmask; long long rowmask_off0, rowmask_oo;
  float drop_p; unsigned long long seed, drop_offset; const unsigned long long* seed_ptr;
  int split_k;
  const void* gate; float gate_scale;
  void* C2; int gate_mode; float post_drop_p; unsigned long long post_drop_offset;
  long long c_split_stride;
  const float* row_exp2_offset;                    /* act 3: x = exp2(x * log2(e) + row_exp2_offset[m]) */
  const int32_t* m_limit_dev; int m_limit_base;    /* device scalar: 128-row tiles with m0 + base >= *limit are skipped */
  const int32_t* k_limit_dev; int k_limit_base;    /* device scalar: the contraction stops at *limit - base, rounded up to
                                                      a whole 64-element chunk (operands beyond the limit must be finite) */
} rp_gemm_desc;
int rp_gemm(const rp_gemm_desc* g, void* stream);
/* dst[i] (+)= sum_s src[s * stride + i], i < n (n, stride multiples of 4) */
int rp_reduce_splits(const float* src, int n_splits, long long stride, long long n, float* dst, int accumulate, void* stream);

/* Fused multi-head attention forward for L <= 256, head_dim in {64,128}: S = Q.K^T, causal / key-padding mask derived
 * from pad_mask (no [B*H,L,L] mask tensor), softmax, dropout, O = P.V.
 *   replaces  torch.nn.MultiheadAttention's SDPA core + replay/nn/mask.py:18-51 (new path: causal & pad keys masked)
 *             models/nn/sequential/sasrec/model.py:229-231,435 (legacy: causal only) ; bert4rec/model.py:494 (pad keys only)
 * q/k/v: 2-D bf16 arrays whose rows are tokens; head h reads columns x_c0 + h*head_dim.  out: bf16 [B*L, ldo].
 * p_save (optional) bf16 [B*H, Lp, Lp] receives exp(s - rowmax) (Lp = round_up(L,64), must be zero-initialised once),
 * inv_sum fp32 [B*H, Lp] the reciprocal row sums - the inputs of rp_attn_softmax_bwd. */
typedef struct rp_attn_desc {
  const void* q; long long q_rows, q_cols, ldq; int q_c0;
  const void* k; long long k_rows, k_cols, ldk; int k_c0;
  const void* v; long long v_rows, v_cols, ldv; int v_c0;
  int B, H, L, head_dim;
  int causal, mask_pad_keys;
  const uint8_t* pad_mask;
  void* out; int ldo;
  void* p_save; float* inv_sum;
  float drop_p; unsigned long long seed, drop_off; const unsigned long long* seed_ptr;
  float* m_save;  /* optional fp32 [B*H, Lp]: row max in exp2 units, input of rp_attn_bwd */
  float scale;    /* softmax scale; 0 -> 1/sqrt(head_dim).  Padded head slots (true head_dim 32 / 48 / 50 inside a 64-wide
                     slot) pass 1/sqrt(true head_dim) */
} rp_attn_desc;
int rp_attn_fwd(const rp_attn_desc* a, void* stream);

/* Fused attention backward (L <= 256, head_dim 64), one CTA per (sequence, head): recomputes S^T = K.Q^T and
 * dP^T = V.dO^T on tcgen05, forms P / dS in registers from the forward's row statistics (m_save, inv_sum) and accumulates
 * dV = Pd^T.dO, dK = dS^T.Q, dQ = dS.K with the bf16 operands staged in TMEM / swizzled shared memory - the [B*H, L, L]
 * matrices of the un-fused path are never written.  Replaces autograd's backward of the SDPA core of
 * torch.nn.MultiheadAttention (replay/nn/sequential/sasrec/transformer.py:99-106 ; bert4rec/model.py:494).
 * q/k/v/d_out/out: token-major 2-D bf16 arrays; dq/dk/dv: outputs (rows b*L + i, columns x_c0 + h*64). */
typedef struct rp_attn_bwd_desc {
  const void* q; long long q_rows, q_cols, ldq; int q_c0;
  const void* k; long long k_rows, k_cols, ldk; int k_c0;
  const void* v; long long v_rows, v_cols, ldv; int v_c0;
  const void* d_out; long long do_rows, do_cols, ld_do;
  const void* out; int ldo;
  int B, H, L, head_dim;
  int causal, mask_pad_keys;
  const uint8_t* pad_mask;
  const float* m_save; const float* inv_sum;
  void* dq; int ld_dq, dq_c0;
  void* dk; int ld_dk, dk_c0;
  void* dv; int ld_dv, dv_c0;
  float drop_p; unsigned long long seed, drop_off; const unsigned long long* seed_ptr;
  float scale;    /* as in rp_attn_desc */
} rp_attn_bwd_desc;
int rp_attn_bwd(const rp_attn_bwd_desc* a, void* stream);

/* Softmax backward between the batched attention-backward GEMMs (un-fused path, any supported head_dim): in place, dpd := dS = P*(dP - sum P*dP)*scale and
 * p_save := P*dropmask/keep (the A operand of dV). */
int rp_attn_softmax_bwd(void* p_save, void* dpd, const float* inv_sum, int BH, int L, float scale, float drop_p,
                        unsigned long long seed, unsigned long long drop_off, const unsigned long long* seed_ptr,
                        void* stream);

/* predict(): attention of ONE query row per (sequence, head) - the last position - against that sequence's keys
 * (SasRec.forward_inference keeps only hidden[:, -1, :], nn/sequential/sasrec/model.py:301; legacy model.py:157).
 * q, out: compact bf16 [B, H*head_dim]; k, v: token-major 2-D arrays (rows b*L + j, head h at columns x_c0 + h*head_dim). */
int rp_attn_last(const void* q, const void* k, const void* v, long long ldk, long long ldv, int k_c0, int v_c0,
                 const uint8_t* pad_mask, int B, int H, int L, int head_dim, int mask_pad_keys, void* out, float scale /* 0: 1/sqrt(head_dim) */,
                 void* stream);

/* int64 ids / bool masks of one [B, L] batch -> int32 ids (pads -> pad_id) and the compacted valid-target list
 * (replaces the masked_fill / boolean-index preparation in nn/loss/ce.py:70-80 and models/.../sasrec/model.py:236-239).
 * labels/target_mask may be NULL (predict). */
int rp_prepare_batch(const int64_t* ids, const uint8_t* pad_mask, const int64_t* labels, const uint8_t* target_mask, int T,
                     int pad_id, int n_items, int32_t* ids32, int32_t* valid_idx, int32_t* labels_c, int32_t* n_valid,
                     int32_t* scratch /* >= ceil(T/1024) ints, needed with targets */, void* stream);

/* x[t] = table[ids[t]] * scale + pos[pos0 + t % L] -> dropout -> (zero pad rows)      nn/sequential/sasrec/agg.py:37-53,
 * models/nn/sequential/sasrec/model.py:346-357 ; and its backward (fp32 atomics into d_table, pad row frozen). */
int rp_embed_fwd(const void* table, const float* pos, const int32_t* ids, const uint8_t* pad_mask, int T, int L, int d,
                 int pos0, float scale, int zero_pad_rows, float drop_p, unsigned long long seed, unsigned long long drop_off,
                 const unsigned long long* seed_ptr, void* out, void* stream);
int rp_embed_bwd(const void* dx, const int32_t* ids, const uint8_t* pad_mask, int B, int L, int d, int pad_id, int pos0,
                 float scale, int zero_pad_rows, float drop_p, unsigned long long seed, unsigned long long drop_off,
                 const unsigned long long* seed_ptr, float* d_table, float* d_pos, void* stream);

/* torch.nn.LayerNorm forward / backward (transformer.py:47-49,60-62 eps 1e-8; model.py:248 eps 1e-5).  With `gather`
 * output row r reads input row gather[r] and only *n_rows_dev rows exist (valid-target compaction); the backward then
 * scatters dx to those rows.  add_to (optional, bf16 [*, d]) is added to dx (residual-branch gradient). */
/* PADDED FEATURE SLOTS (`hd_valid`, 0 = none): the reference's default shapes are not multiples of the 64-wide tensor-core
 * feature tiles (SasRec.from_params: embedding_dim 192 / 4 heads = head_dim 48, nn/sequential/sasrec/model.py:199-253; legacy
 * hidden_size 50, sasrec/lightning.py:30-47; examples: d = 64 / 2 heads = 32).  Such a model is stored with every head in its
 * own slot of 64 columns (128 for head_dim in (64, 128]) whose first hd_valid columns are the real features and whose padded
 * columns are ZERO in every activation, weight, bias and gradient (zero weights keep them zero through every GEMM, the
 * optimizer never moves a parameter whose gradient is zero).  The only operator that is not blind to the padding is LayerNorm:
 * its statistics run over the d_true = (d / slot) * hd_valid real features and its backward sends no gradient into padded
 * inputs - every entry point that contains a LayerNorm takes `hd_valid`; the attention takes the true softmax scale. */
int rp_layernorm_fwd(const void* x, const float* w, const float* b, float eps, int n_rows, int d, const int32_t* n_rows_dev,
                     const int32_t* gather, void* y, float* mean, float* rstd, int hd_valid, void* stream);
int rp_layernorm_bwd(const void* dy, const void* x, const float* w, const float* mean, const float* rstd, int n_rows, int d,
                     const int32_t* n_rows_dev, const int32_t* gather, const void* add_to, void* dx, float* dw, float* db,
                     int hd_valid, void* stream);

/* out = in * regenerated dropout mask / keep (and optional row mask); db[c] += column sums of a bf16 [rows, cols] array. */
int rp_dropout_bwd(const void* in, void* out, long long rows, int cols, const uint8_t* rowmask, float drop_p,
                   unsigned long long seed, unsigned long long drop_off, const unsigned long long* seed_ptr, void* stream);
int rp_colsum(const void* dy, int rows, int cols, long long ld, float* db, void* stream);
/* the same for n <= 6 tensors sharing the row count, one launch (the bias gradients of one block's backward) */
int rp_colsum_multi(int n, const void* const* dy, const int* cols, const long long* ld, float* const* db, int rows, void* stream);

/* torch.optim.Adam (models/nn/optimizer_utils/optimizer_factory.py:71-87; no weight decay) on flat fp32 buffers; refreshes
 * the bf16 shadow, optionally zeroes the gradient; lr and the step counter live in device memory. */
/* BERT4Rec embedding: where(token_mask, table[ids], mask_emb) + pos[t % L] (bert4rec/model.py:239-296) and its backward;
 * row gather / scatter with a device-side row count (dst[r] = src[idx[r]] or dst[idx[r]] = src[r]). */
int rp_bert_embed_fwd(const void* table, const void* mask_emb, const float* pos, const int32_t* ids, const uint8_t* tok_mask,
                      int T, int L, int d, float drop_p, unsigned long long seed, unsigned long long drop_off,
                      const unsigned long long* seed_ptr, void* out, void* stream);
int rp_bert_embed_bwd(const void* dx, const int32_t* ids, const uint8_t* pad_mask, const uint8_t* tok_mask, int B, int L, int d,
                      float drop_p, unsigned long long seed, unsigned long long drop_off, const unsigned long long* seed_ptr,
                      float* d_table, float* d_mask_emb, float* d_pos, void* stream);
int rp_gather_rows(const void* src, const int32_t* idx, int n_max, const int32_t* n_dev, int d, void* dst, int scatter,
                   void* stream);

/* Inference / predict(): the whole point-wise FFN in one pass  out = relu(y W1^T + b1) W2^T + b2 + y  (weights resident in shared
 * memory, hidden activation kept in TMEM, residual read from the staged y tile): y is read once and out written once.
 *   replaces (eval)  SasRecPointWiseFeedForward.forward  replay/models/nn/sequential/sasrec/model.py:496-506 ; replay/nn/ffn.py:43-57
 * y, out bf16 [T, d] (no aliasing), w1 / w2 bf16 [d, d], b1 / b2 fp32 [d], rowmask optional uint8 [T] (0 -> zero row), d in {64,128}. */
int rp_ffn_fused(const void* y, const void* w1, const float* b1, const void* w2, const float* b2, const uint8_t* rowmask, int T,
                 int d, void* out, void* stream);

/* Inference: out-projection + residual + LayerNorm + FFN of one SASRec block in one pass  (h = o Wo^T + bo + q_in ;
 * y = LN(h) ; out = relu(y W1^T + b1) W2^T + b2 + y); h and y never reach HBM.  Shapes as rp_ffn_fused; out may not alias o / q_in.
 *   replaces (eval)  replay/nn/sequential/sasrec/transformer.py:99-110 ; replay/models/nn/sequential/sasrec/model.py:435-441 */
int rp_post_attn_fused(const void* o, const void* q_in, const void* wo, const float* bo, const float* ln_w, const float* ln_b,
                       float eps, const void* w1, const float* b1, const void* w2, const float* b2, const uint8_t* rowmask, int T,
                       int d, void* out, int hd_valid, void* stream);

/* Training forward of everything after the attention of one SASRec block in one pass over the tokens:
 *   h = o Wo^T + bo + q_in ; y = LN(h) ; u = dropout1(relu(y W1^T + b1)) ; out = (y + dropout2(u W2^T + b2)) [* rowmask]
 * writing the activations the backward needs on the way (h, y, u bf16 [T, d]; LayerNorm mean / rstd fp32 [T]): 2 tensors read
 * and 4 written instead of the 14 [T, d] passes of out-projection GEMM + LayerNorm + two FFN GEMMs.  Element (row, column) of a
 * dropout site is kept iff drop_mix(drop_row_key(seed + *seed_ptr, drop_off, row), drop_col_key(column)) >= p * 2^32
 * (csrc/rp_philox.cuh) - the stream of rp_gemm's epilogue and rp_dropout_bwd, so the un-fused backward applies unchanged.  d in {64,128}; out may not alias o / q_in.
 *   replaces (train)  replay/nn/sequential/sasrec/transformer.py:99-110 ; replay/nn/ffn.py:43-57 ;
 *                     replay/models/nn/sequential/sasrec/model.py:435-441,496-506 */
int rp_post_attn_train(const void* o, const void* q_in, const void* wo, const float* bo, const float* ln_w, const float* ln_b,
                       float eps, const void* w1, const float* b1, const void* w2, const float* b2, const uint8_t* rowmask, int T,
                       int d, float drop_p, unsigned long long seed, unsigned long long drop_off1, unsigned long long drop_off2,
                       const unsigned long long* seed_ptr, void* h_save, void* y_save, void* u_save, float* mean_out,
                       float* rstd_out, void* out, int hd_valid, void* stream);

/* Backward of rp_post_attn_train in one pass over the tokens.  Given dz = d loss / d out:
 *   dzm = dz [* rowmask] ;  d_t = dropout2'(dzm) ;  du = (d_t W2) * [u != 0] / keep ;  dy = du W1 + dzm ;
 *   dh = LayerNorm-backward(dy ; h, mean, rstd, ln_w) ;  d_o = dh Wo ;  dln_w / dln_b += column sums (fp32 atomics, one per column and CTA)
 * d_t, du, dh (bf16 [T, d]) are the dY operands of rp_wgrad_group for W2 / W1 / Wo (X = u, y, o); dh is also the residual gradient
 * into the pre-attention part; d_o feeds rp_attn_bwd.  d_t may be NULL when drop_p == 0 and rowmask == NULL (then d_t == dz).
 *   replaces autograd's backward of  replay/nn/sequential/sasrec/transformer.py:107-110 ; replay/nn/ffn.py:43-57 ;
 *                                    replay/models/nn/sequential/sasrec/model.py:436-441,496-506 */
int rp_post_attn_bwd(const void* dz, const void* u, const void* h, const float* mean, const float* rstd, const float* ln_w,
                     const void* w2, const void* w1, const void* wo, const uint8_t* rowmask, int T, int d, float drop_p,
                     unsigned long long seed, unsigned long long drop_off2, const unsigned long long* seed_ptr, void* d_t, void* du,
                     void* dh, void* d_o, float* dln_w, float* dln_b, int hd_valid, void* stream);

/* Everything BEFORE the attention of one SASRec block in one pass over the tokens (training and inference):
 *   q_in = LayerNorm(x) ;  Q = q_in Wq^T + bq ;  [K | V] = x [Wk | Wv]^T + [bk | bv]      (K, V from the un-normalised x)
 * x is read once; q_in (the block's residual), Q, KV and the LayerNorm statistics are written once (LayerNorm + two GEMM
 * launches read x / q_in three times).  w_in bf16 [3d, d] = packed in_proj_weight, b_in fp32 [3d]; d in {64,128}.
 * q_in == NULL and Q == NULL: only [K | V] is computed (ln_w / ln_b unused) - predict()'s final block, whose LayerNorm and
 * Q projection run on the last position of every sequence only.
 *   replaces  replay/nn/sequential/sasrec/transformer.py:99-106 ; replay/models/nn/sequential/sasrec/model.py:434-435 */
int rp_ln_qkv_fused(const void* x, const float* ln_w, const float* ln_b, float eps, const void* w_in, const float* b_in, int T,
                    int d, void* q_in, void* Q, void* KV, float* mean_out, float* rstd_out, int hd_valid, void* stream);
/* Its backward in one pass:  dq_in = dQ Wq + dh ;  t = LayerNorm-backward(dq_in; x, mean, rstd, ln_w) ;  dx = [dK | dV] Wkv + t.
 * dln_w / dln_b fp32 [d] are ACCUMULATED (one fp32 atomic per column and CTA).  dx may not alias an input; d in {64,128}. */
int rp_pre_attn_bwd(const void* dQ, const void* dKV, const void* dh, const void* x, const float* mean, const float* rstd,
                    const float* ln_w, const void* w_in, int T, int d, void* dx, float* dln_w, float* dln_b, int hd_valid,
                    void* stream);

/* ALL weight and bias gradients of one transformer block in one launch (+ one deterministic reduction launch):
 *   dW_i[n_out_i, n_in_i] (+)= dY_i[T, n_out_i]^T . X_i[T, n_in_i] ;  db_i[n_out_i] (+)= column sums of dY_i      i < n_pairs <= 8
 * dY_i / X_i are read in place (MN-major tcgen05 operands, contraction over the tokens); the bias gradient is one extra N = 16
 * MMA per k-step against a tile of ones.  n_out, n_in multiples of 64; at most 48 output tiles of 128 x 128 in one call.
 *   replaces  autograd's weight / bias gradients of  replay/nn/sequential/sasrec/transformer.py:36-46,99-110 ;
 *             replay/nn/ffn.py:43-57 ; replay/models/nn/sequential/sasrec/model.py:407-414,490-506 ; bert4rec/model.py:471-527 */
typedef struct rp_wgrad_pair {
  const void* dY; long long dy_ld; int n_out;   /* bf16 [T, n_out], row pitch dy_ld elements */
  const void* X; long long x_ld; int n_in;      /* bf16 [T, n_in],  row pitch x_ld */
  float* dW; long long dw_ld;                   /* fp32 [n_out, n_in], row pitch dw_ld (multiple of 4) */
  float* db;                                    /* fp32 [n_out] or NULL */
} rp_wgrad_pair;
size_t rp_wgrad_group_workspace(const rp_wgrad_pair* pairs, int n_pairs);
int rp_wgrad_group(const rp_wgrad_pair* pairs, int n_pairs, int T, int accumulate, void* workspace, size_t workspace_bytes,
                   void* stream);

int rp_adam_step(float* p, float* g, float* m, float* v, void* shadow_bf16, long long n, const float* lr_dev,
                 int32_t* step_dev, float beta1, float beta2, float eps, float grad_scale, const uint8_t* frozen,
                 int zero_grad, void* stream);
/* Gradient exchange of data-parallel training over NVLink peer memory - ONE kernel inside the captured step graph.
 *   replaces  the bucketed all-reduce of Lightning DDP under loss.backward()  replay/nn/lightning/module.py:62-75 with
 *             Trainer(strategy="ddp"); replay/models/nn/sequential/sasrec/lightning.py:196-209 (SURVEY.md 2.1 / 8e)
 * bufs[w] / states[w] (host arrays of `world` device pointers): rank w's fp32 gradient buffer (n elements, 16-byte aligned)
 * and its state block (rp_peer_allreduce_state_bytes() bytes, zeroed once) as mapped into THIS process - every rank passes
 * pointers into the same symmetric allocation (replay_b200/peer.py).  world in 2..8, one node.  Result: every buffer holds
 * the element-wise sum, bit-identical on all ranks (each element is summed by one rank in rank order and broadcast).
 * Every rank must enqueue it exactly once per step; CUDA-graph capturable; the grid never exceeds the SM count. */
size_t rp_peer_allreduce_state_bytes(void);
int rp_peer_allreduce(void* const* bufs, void* const* states, int rank, int world, long long n, void* stream);
int rp_cast_bf16(const float* src, void* dst, long long n, void* stream);
int rp_counter_add(unsigned long long* counter, unsigned long long inc, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Sampled training heads (SURVEY.md §8 a9 / f.2): logits only for the positive item and n_neg sampled negatives per target.
 *   replaces  SampledLossBase.get_sampled_logits + mask_negative_logits   replay/nn/loss/base.py:40-154,157-196
 *             CESampled.forward / BCESampled.forward                      replay/nn/loss/ce.py:199-249 ; bce.py:154-218
 *             legacy _compute_loss_ce_sampled / _compute_loss_bce_sampled  replay/models/nn/sequential/sasrec/lightning.py:310-376
 * hc / labels / n_valid as for rp_ce_head_fwd (compacted valid targets).  negatives int64: neg_mode 0 = [n_neg] shared by the
 * batch (tensor-core path), 1 = [B*seq_len, n_neg] per position, 2 = [B, n_neg] per sequence (1, 2: rows addressed through
 * valid_idx[t] = flat b*seq_len + l of compacted row t; gather-dot kernels).  kind: RP_LOSS_CE_SAMPLED (negatives equal to the
 * positive or to ignore_index get logit -1e9), RP_LOSS_BCE_SAMPLED (same masking, log_eps / clamp as the reference),
 * RP_LOSS_LEGACY_CE_SAMPLED (log(vocab_size-1) - 1e6*reject - log(n_neg - #reject) correction), RP_LOSS_LEGACY_BCE_SAMPLED (no
 * masking).  One positive per position.  fwd: loss_out[0] = mean loss, loss_out[1] = 1/T_v, d(loss)/d(logits) stays in the
 * workspace; bwd: d_hc bf16 [capacity, d] rows < *n_valid, d_table fp32 ACCUMULATED (zero it first; dense rows untouched).
 * ------------------------------------------------------------------------------------------------------------- */
#define RP_LOSS_CE_SAMPLED 0
#define RP_LOSS_BCE_SAMPLED 1
#define RP_LOSS_LEGACY_CE_SAMPLED 2
#define RP_LOSS_LEGACY_BCE_SAMPLED 3
typedef struct rp_sampled_desc {
  const void* hc; const void* table; const int32_t* labels; const int32_t* valid_idx; const int64_t* negatives;
  const int32_t* n_valid;
  int capacity, n_items, d, n_neg, neg_mode, seq_len, kind, ignore_index, vocab_size;
  float log_eps, clamp;
  float* loss_out;
  void* workspace; size_t workspace_bytes;
} rp_sampled_desc;
size_t rp_sampled_head_workspace(int capacity, int d, int n_neg, int neg_mode);
int rp_sampled_head_fwd(const rp_sampled_desc* s, void* stream);
int rp_sampled_head_bwd(const rp_sampled_desc* s, void* d_hc, float* d_table, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Device-side batch construction (SURVEY.md §8 f.1).  All histories are resident in HBM as CSR: offsets [n_seq+1] int64,
 * items [offsets[n_seq]] int32.  One call builds B rows of a [B, L] batch: row b is the window of history seq_index[b]
 * starting at seq_offset[b] (NULL: the LAST L(+1) items), left-padded with pad_value.  Replaces the per-sample host path
 *   TorchSequentialDataset.__getitem__/_pad_sequence/_generate_padding_mask  replay/data/nn/torch_sequential_dataset.py:69-136
 *   SasRecTrainingDataset.__getitem__ (window L+1, inputs [:-1], labels [1:])  replay/models/nn/sequential/sasrec/dataset.py:104-126
 *   Bert4RecUniformMasker.mask + Bert4RecTrainingDataset.__getitem__          .../bert4rec/dataset.py:71-92,163-177
 *   _shift_features (predict: roll left, last = pad, token/pad masks)         .../bert4rec/dataset.py:322-351
 *   Array1DColumn.__getitem__ + NextTokenTransform (new path, torch ops)     replay/data/nn/parquet/impl/array_1d_column.py:70-84,
 *                                                                            impl/indexing.py:42-78, replay/nn/transform/next_token.py:65-96
 * and the default collate.  mode: RP_BATCH_SASREC_TRAIN -> ids, pad_mask, labels, aux_mask = target_padding_mask;
 * RP_BATCH_PREDICT -> ids, pad_mask; RP_BATCH_BERT_TRAIN -> ids (= inputs), pad_mask, labels (= positive_labels),
 * aux_mask = token_mask (0 = masked) drawn as (u * pad) >= mask_prob with the reference's two corner-case fix-ups, u from
 * `uniforms` [B, L] when given (bit-exact against the reference masker fed the same numbers) else Philox4x32-10 keyed by
 * (seed, draw0 + b); RP_BATCH_BERT_PREDICT -> shifted ids, pad_mask, aux_mask = token_mask.
 * query_out [B] (optional) = query_ids[seq_index[b]] (or the index itself when query_ids is NULL).
 * ------------------------------------------------------------------------------------------------------------- */
#define RP_BATCH_SASREC_TRAIN 0
#define RP_BATCH_PREDICT 1
#define RP_BATCH_BERT_TRAIN 2
#define RP_BATCH_BERT_PREDICT 3
int rp_build_batch(const int64_t* offsets, const int32_t* items, long long n_seq, const int32_t* seq_index,
                   const int32_t* seq_offset, int B, int L, int mode, int pad_value, float mask_prob, const float* uniforms,
                   unsigned long long seed, unsigned long long draw0, const int64_t* query_ids, int64_t* ids,
                   uint8_t* pad_mask, int64_t* labels, uint8_t* aux_mask, int64_t* query_out, void* stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Bring-up self test of the tcgen05 operand encodings (used by tests/, not by the product path).
 * A, B: bf16 [128,128]; D: fp32 [128,128].  mode bit0: B given as Bt[K,N]; bit1: A staged through TMEM;
 * bit2: A given as At[K,M].  D = A . B^T in every mode.
 * ------------------------------------------------------------------------------------------------------------- */
int rp_selftest_umma(int mode, const void* A, const void* B, float* D, void* stream);
/* TMA feed-rate probe (tools/probe_tma.py): every CTA streams `tiles` [box_rows x d] row tiles of a K-major bf16 table through
 * an 8-stage ring with no consumer. */
/* tcgen05.mma issue-rate probe (tools/probe_mma.py): mode bit0 B MN-major, bit1 A from TMEM, bit2 A MN-major; every CTA issues
 * iters x 8 MMAs (128x128x16 bf16) and writes its elapsed SM cycles to cycles_out[blockIdx.x]. */
int rp_selftest_mma_probe(int mode, int iters, int grid, long long* cycles_out, void* stream);
int rp_selftest_tma_probe(const void* table, long long rows, int d, int box_rows, int tiles, int same_tile, int grid,
                          void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RP_B200_H */
