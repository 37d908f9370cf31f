/* tome_b200.h -- C ABI of the B200-native ToMe transformer block.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has NO native layer: its interface for this
 * path is a set of Python/JAX functions and Flax modules (paths relative to
 * /root/reference/multi_modal_transformers/).  Each entry point below names the reference lines whose arithmetic
 * it replaces; the Python mirror of the reference API (package multi_modal_transformers_tokenmerge_b200) and an
 * XLA-FFI shim (INTEGRATION.md) bind exactly these symbols.
 *
 * Conventions
 *   - every pointer is DEVICE memory owned by the caller unless the name ends in _host; the library allocates
 *     nothing, keeps no state except a thread-local error string, and never synchronises the stream;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and the call returns at once;
 *   - return value: TOME_OK (0) or an error code; the text is available from tome_last_error();
 *     nothing throws or aborts across this boundary;
 *   - activations are bf16 (TOME_BF16) or fp32 (TOME_F32) where a dtype field exists; token sizes, LayerNorm
 *     statistics, log-sum-exp, biases and gradients of parameters are always fp32; indices are int32;
 *   - strides and leading dimensions are in ELEMENTS.
 */
#ifndef TOME_B200_H
#define TOME_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TOME_ABI_VERSION 18

enum tome_status { TOME_OK = 0, TOME_ERR_INVALID = 1, TOME_ERR_CUDA = 2, TOME_ERR_UNSUPPORTED = 3 };
enum tome_dtype { TOME_BF16 = 0, TOME_F32 = 1, TOME_U8 = 2 /* raw pixels: image front end only */ };
enum tome_major { TOME_MAJOR_K = 0, TOME_MAJOR_MN = 1 };
enum tome_merge_mode { TOME_MERGE_SUM = 0, TOME_MERGE_WAVG = 1 };

const char* tome_last_error(void);
int tome_abi_version(void);

/* ------------------------------------------------------------------------------------------------------------
 * 1. Bipartite soft matching          tokenizers/token_compression.py:54-112
 * ------------------------------------------------------------------------------------------------------------ */

/* r = min(r, (tokens - protected) / 2), clamped at 0            token_compression.py:60-67 */
int tome_clamp_r(int tokens, int r, int class_token, int distill_token);

/* Token sets for matching INSIDE each set (ABI 15): the sequence is n_sets consecutive sets in order, set s holding tokens
 * [set_start[s], set_start[s] + set_n[s]), set_start[0] = 0, the sets covering `tokens` without gap or overlap.  Set s loses
 * set_r[s] tokens, 0 <= set_r[s] <= set_n[s] / 2: its part of the output is bipartite_soft_matching + merge of the set's
 * slice on its own (even / odd split relative to set_start[s], the same tie rules and fp32 rank-order adds), the parts
 * concatenated in set order; a set with set_r[s] == 0 is copied unchanged.  So a token never merges with a token of another
 * set: with one set per frame and modality the block-causal group mask keeps holding after a merge.  Not combinable with
 * class_token / distill_token (TOME_ERR_INVALID).  A NULL `sets` pointer below means one set spanning the sequence: the
 * behaviour and results of ABI 14. */
#define TOME_MAX_TOKEN_SETS 16
typedef struct {
  int n_sets;
  int set_start[TOME_MAX_TOKEN_SETS];
  int set_n[TOME_MAX_TOKEN_SETS];
  int set_r[TOME_MAX_TOKEN_SETS];
} tome_token_sets_t;

/* Where the matching metric comes from.  metric[b,t,d] = (1/heads) * sum_h src[b,t,h,d]; with heads == 1 this is a
 * plain [B,T,Dm] tensor (the `metric` argument of bipartite_soft_matching); with heads > 1 it is "keys averaged
 * over heads" read in place from a packed qkv buffer (intended call site tome_attention.py:249-256). */
typedef struct {
  int batch, tokens, dim, heads;
  int dtype; /* tome_dtype of src */
  long long batch_stride, token_stride, head_stride;
  int class_token, distill_token;
  const tome_token_sets_t* sets; /* NULL: one set (set_r is ignored here apart from its range check) */
} tome_metric_desc_t;

/* L2-normalise rows (no epsilon), split even/odd, scores = a b^T in fp32, protect row/column 0, then
 * node_max[b,i] = max_j scores, node_idx[b,i] = first arg max.                       token_compression.py:72-83
 * node_max f32 [B,Ta], node_idx i32 [B,Ta]  (Ta = ceil(T/2), Tb = floor(T/2)).
 * With sets: every set is scored against its own odd tokens only; node_max / node_idx are [B, sum_s ceil(n_s/2)], set after
 * set, node_idx local to the set; scores_out is [B, sum_s ceil(n_s/2) * floor(n_s/2)], each set's [ceil, floor] block in
 * turn.  A one-token set has no partner: node_max = -inf, node_idx = 0.
 * scores_out: optional f32 [B,Ta,Tb] dump of the exact fp32 scores the arg max was taken from (parity protocol:
 * "indices bit-exact from the same fp32 scores"); pass NULL on the fast path and the scores never touch HBM.
 * dim: even, 2 .. 296.  workspace: required, tome_sim_argmax_workspace_bytes(desc) bytes, 16-byte aligned; a NULL or
 * smaller one is TOME_ERR_INVALID.  The rows are normalised once into the workspace, then scored:
 *   dim == 64  each row as three bf16 planes (hi + mid + lo: the fp32 value), a b^T on the tensor cores (tcgen05);
 *   otherwise  fp32 planes, a b^T as fp32 FMAs on CUDA cores (even and odd k summed separately).
 * (ABI 14: the workspace became required.  Dims 297 .. 448 ran only without a workspace before and are now refused.) */
size_t tome_sim_argmax_workspace_bytes(const tome_metric_desc_t* desc);
int tome_sim_argmax(const tome_metric_desc_t* desc, const void* src, float* node_max, int32_t* node_idx,
                    float* scores_out, void* workspace, size_t workspace_bytes, void* stream);

/* The index set bipartite_soft_matching closes over (token_compression.py:84-88) plus derived maps the merge
 * kernels use.  All int32, device. */
typedef struct {
  int32_t* edge_idx; /* [B,Ta]   argsort(node_max) reversed: value descending, ties by index descending;
                                 edge_idx[:, :r] = src_idx, edge_idx[:, r:] = unm_idx                       */
  int32_t* dst_idx;  /* [B,r]    node_idx[src_idx]                                                          */
  int32_t* row_map;  /* [B,T]    row of the merged output that input token t lands in (unmerge gather map)  */
  int32_t* dst_off;  /* [B,Tb+1] CSR offsets: sources merged into odd token j are dst_src[dst_off[j]..)     */
  int32_t* dst_src;  /* [B,r]    even-set indices grouped by destination, in rank order inside a group      */
} tome_plan_t;
/* With sets the arrays are concatenated set by set inside each batch row, indices local to the set: edge_idx [B, sum
 * ceil(n_s/2)] (the identity order for a set with r = 0), dst_idx / dst_src [B, sum r_s], dst_off [B, sum (floor(n_s/2) + 1)];
 * row_map [B,T] holds GLOBAL output rows, so tome_merge_bwd and tome_chain_row_maps read it as they read a one-set plan. */

typedef struct {
  int batch, tokens, r; /* r already clamped (tome_clamp_r), r >= 1; with sets: sum_s set_r[s] */
  int distill_token;
  const tome_token_sets_t* sets; /* NULL: one set */
} tome_plan_shape_t;

/* Edge ranking and index split.                                                       token_compression.py:84-88 */
int tome_select_topr(const tome_plan_shape_t* shape, const float* node_max, const int32_t* node_idx,
                     const tome_plan_t* plan, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 2. Merge / unmerge                   tokenizers/token_compression.py:90-129
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int batch, tokens, channels, r;
  int distill_token;
  int dtype; /* of x / x_out / dy / dx */
  int mode;  /* TOME_MERGE_SUM: merge(x, "sum") :90-109;  TOME_MERGE_WAVG: merge_wavg :114-129 */
  const tome_token_sets_t* sets; /* NULL: one set; else r = sum_s set_r[s] and the plan has the per-set layout above */
} tome_merge_shape_t;

/* x [B,T,C] -> x_out [B,T-r,C].  WAVG: x_out = merge(x*size)/merge(size), size_out = merge(size), fp32 arithmetic in
 * the reference's order (sources added to their destination sequentially in rank order).  size / size_out are
 * f32 [B,T] / [B,T-r]; size == NULL means all ones (token_compression.py:121-122).  SUM ignores both.
 * gid/pos (optional, may be NULL): per-token group id (u8) and position-in-group (i32) carried through the merge:
 * an output row keeps the group/position of its unmerged or destination token. */
int tome_merge_fwd(const tome_merge_shape_t* shape, const tome_plan_t* plan, const void* x, const float* size,
                   void* x_out, float* size_out, const uint8_t* gid, const int32_t* pos, uint8_t* gid_out,
                   int32_t* pos_out, void* stream);

/* Backward of tome_merge_fwd w.r.t. x (autodiff of token_compression.py:95-108,125-127):
 * dx[b,t] = w * dy[b,row_map[b,t]],  w = size[b,t] / size_out[b,row] for WAVG, 1 for SUM.
 * With mode SUM this is also the ToMe-paper `unmerge` (not in the reference; SURVEY.md A.7). */
int tome_merge_bwd(const tome_merge_shape_t* shape, const tome_plan_t* plan, const float* size, const float* size_out,
                   const void* dy, void* dx, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 3. Dense layers                      attention_blocks/tome_attention.py:145-164,287-299; attention.py:32-37
 * ------------------------------------------------------------------------------------------------------------ */

/* C[M,N] = epilogue(A[M,K] * B[N,K]^T), bf16 operands, fp32 accumulation (tcgen05, accumulators in TMEM).
 * An operand is K-major (row index = M or N, K contiguous) or MN-major (row index = K, M or N contiguous), so the
 * Flax kernel layout [in, out] serves forward (B MN-major), dgrad (B K-major) and wgrad (A, B MN-major) as is.
 * epilogue, in order: + bias[N]; ReLU; * (gate > 0 ? gate_scale : 0); dropout; + residual; cast to c_dtype.
 * k_splits > 1 (fp32 C only) splits the reduction and sums the partials in a fixed order (weight gradients);
 * k_splits == 0 lets the library choose; with accumulate != 0 the result is ADDED to C (fp32 C only). */
#define TOME_GEMM_MAX_SHIFTS 16
typedef struct {
  int m, n, k;
  const void* a; long long lda; int a_major;
  const void* b; long long ldb; int b_major;
  void* c; long long ldc; int c_dtype;
  const float* bias;
  const void* residual; long long ldr; /* bf16 [M, ldr] */
  const void* gate; long long ldg;     /* bf16 [M, ldg] */
  float gate_scale;
  int relu;
  float dropout_rate; uint64_t dropout_seed; uint32_t dropout_site;
  int k_splits;
  int accumulate;
  /* The ReLU gate as one bit per element instead of bf16 rows ([M, ld_bits] u32 words, bit j of word w = column 32 w + j):
   * a ReLU epilogue with relu_bits_out != NULL also writes bit = (output > 0) (after dropout, so the dropped elements are
   * gated too); a later GEMM with gate_bits != NULL multiplies by (bit ? gate_scale : 0) exactly as `gate` would, reading
   * 1/16 of the bytes.  ld_bits >= ceil(n / 32). */
  const void* gate_bits;
  void* relu_bits_out;
  long long ld_bits;
  /* Bias gradient of the layer that produced this GEMM's input gradient, without a second pass over C: when not NULL
   * (bf16 C, no split-K), row i of colsum_partial (f32 [ceil(m / 128), n], dense) receives the column sums of the
   * bf16-rounded rows 128 i .. 128 i + 127 of C, in a fixed order; tome_reduce_rows_f32 adds the rows up.
   * (MLPBlock Dense bias: attention.py:32-37 under autodiff.) */
  float* colsum_partial;
  /* Row-shifted A windows: a convolution over a zero-bordered, flattened activation grid without materialising im2col rows.
   * With a_row_shift != NULL (host array of a_shift_groups <= TOME_GEMM_MAX_SHIFTS ints; K-major A, no split-K), A is
   * [m, k / a_shift_groups] and the reduction runs over the groups g: C[i, :] = sum_g A[i + a_row_shift[g], :] * B[g-th block
   * of k / a_shift_groups rows, :], rows outside [0, m) reading as zero.  For a 3 x 3 SAME convolution on a grid of width W
   * (zero border included) a_row_shift[3 ty + tx] = (ty - 1) W + (tx - 1) and B is the Flax kernel [3, 3, in, out] as it is.
   * k / a_shift_groups must be a multiple of 64. */
  const int* a_row_shift;
  int a_shift_groups;
} tome_gemm_args_t;

size_t tome_gemm_workspace_bytes(const tome_gemm_args_t* args);
/* SMs the persistent GEMM grid may occupy from now on (process-wide; 0 = all 148).  Lowered by the data-parallel trainer
 * during backward so the overlapped NCCL all-reduce kernels have SMs of their own. */
int tome_gemm_set_sm_limit(int sms);
/* number of SMs the kernels of this library size their persistent grids for (148 on B200) */
int tome_num_sms(void);
int tome_gemm_bf16(const tome_gemm_args_t* args, void* workspace, size_t workspace_bytes, void* stream);

/* out[n] (+)= sum_m x[m,n]   (bias gradients).  x bf16 [M, ldx]; out f32 [N].  workspace: f32 [ws_rows, N] with
 * ws_rows = tome_colsum_workspace_rows(m). */
/* out[n] (+)= sum_r partial[r, n]   (f32, rows added in a fixed order: the second stage of every column sum here) */
int tome_reduce_rows_f32(int rows, int n, const float* partial, float* out, int accumulate, void* stream);
int tome_colsum_workspace_rows(int m);
int tome_colsum_bf16(int m, int n, const void* x, long long ldx, float* out, int accumulate, float* workspace,
                     void* stream);
/* y = dropout(x) (dense bf16 [M,N]; the mask of the GEMM epilogue for the same seed / site / element) and
 * out[n] (+)= sum_m y[m,n] in ONE pass: the backward of "Dropout -> Dense" (attention.py:37,60) needs both. */
int tome_dropout_colsum_bf16(int m, int n, const void* x, void* y, float rate, uint64_t seed, uint32_t site, float* out,
                             int accumulate, float* workspace, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 4. LayerNorm as configured          model_configs/attention_blocks/vanilla_decoder.yaml:7-13
 * ------------------------------------------------------------------------------------------------------------ */

/* axis = 1: statistics over TOKENS for every (batch, feature) -- what reduction_axes=[1] says (SURVEY.md A.4);
 * axis = 2: conventional statistics over features for every (batch, token) (opt-in).
 * var = max(0, E[x^2] - E[x]^2) (use_fast_variance), y = (x - mean) * rsqrt(var + eps) * gamma + beta.
 * x,y bf16 [B,T,C]; gamma,beta f32 [C]; mean,rstd f32 [B,C] (axis 1) or [B,T] (axis 2). */
int tome_layernorm_fwd(int batch, int tokens, int channels, int axis, float eps, const void* x, const float* gamma,
                       const float* beta, void* y, float* mean, float* rstd, void* stream);

/* dx = LN backward (+ dres if not NULL, the residual branch's gradient); dgamma/dbeta f32 [C] are ACCUMULATED
 * into (caller zeroes them at the start of a step).  partial: f32 workspace [2, B, C] (axis 1) or
 * [2, tome_colsum_workspace_rows(B*T), C] (axis 2). */
int tome_layernorm_bwd(int batch, int tokens, int channels, int axis, const void* x, const void* dy,
                       const float* gamma, const float* mean, const float* rstd, const void* dres, void* dx,
                       float* dgamma, float* dbeta, float* partial, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 5. Attention                         flax dot_product_attention reached from tome_attention.py:259-285;
 *                                      mask rules tokenizers/token_sequencer.py:55-183,313-321
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int batch, tokens, heads, head_dim; /* head_dim: 64 */
  /* q,k,v,out: element (b,t,h,d) at  ptr[b*batch_stride + t*token_stride + h*head_dim + d], bf16 */
  long long q_batch_stride, q_token_stride;
  long long k_batch_stride, k_token_stride;
  long long v_batch_stride, v_token_stride;
  long long o_batch_stride, o_token_stride;
  float scale; /* 1/sqrt(head_dim): query scaling of dot_product_attention */
  /* block-causal mask as a group table instead of [B,H,T,T] booleans (octo.py:66-68,119):
   * allow[gid[b,q]*num_groups + gid[b,k]] = 0 masked, 1 visible, 2 visible iff pos[b,k] <= pos[b,q].
   * gid == NULL: no mask.  masked logits become -FLT_MAX (finite, like flax's finfo.min), so a fully masked row
   * yields the uniform distribution, not NaN.  Such a row's lse is the mask constant's, below -2^90 * ln 2 (about -8.6e26)
   * for scale >= 2^-9, and a row that sees any key has an lse of the order of its logits; tome_attention_bwd and
   * tome_attention_importance recognise the row by that lse.  Its gradient is that of the uniform forward: every key
   * k < T receives dO / T (times keep[q,k] / (1 - rate) with dropout) in dV, nothing flows into dQ or dK (the masked
   * logits are constants), and its weights count 1/T per key in both importance modes. */
  const uint8_t* gid;   /* [B,T] */
  const int32_t* pos;   /* [B,T] */
  const uint8_t* allow; /* [G,G], G <= 32 */
  int num_groups;
  /* proportional attention (ToMe paper; not in the reference, SURVEY.md A.7): logits += log(size[b,k]) */
  const float* size; /* [B,T] or NULL */
  /* attention-weight dropout (flax dot_product_attention with dropout_rate > 0 and the default broadcast_dropout=True,
   * vanilla_decoder.yaml:23): weights *= keep[q,k] / (1 - rate) after the softmax, ONE mask shared by every batch row
   * and head.  keep[q,k] is regenerated from (seed, site, q, k) in forward and backward; 0 disables. */
  float dropout_rate;
  uint64_t dropout_seed;
  uint32_t dropout_site;
} tome_attn_desc_t;

/* out [B,T,H,D] bf16, lse f32 [B,H,T] (natural-log sum-exp of the biased, masked, scaled logits).
 * workspace: tome_attention_workspace_bytes(desc) bytes of 256-byte-aligned device scratch (per-tile mask words,
 * log2(size) bias and, with dropout, the keep bits: built once per call and streamed into the kernel by bulk copies);
 * contents need not be kept. */
size_t tome_attention_workspace_bytes(const tome_attn_desc_t* desc);
int tome_attention_fwd(const tome_attn_desc_t* desc, const void* q, const void* k, const void* v, void* out,
                       float* lse, void* workspace, size_t workspace_bytes, void* stream);

/* dq,dk,dv share the layout of q,k,v (their own strides below).  workspace: tome_attention_bwd_workspace_bytes(desc)
 * bytes of 256-byte-aligned device scratch (per-tile mask words, delta = rowsum(dO*O) and lse*log2e padded to 64-token
 * tiles); gradients are produced
 * without atomics or fp32 staging. */
typedef struct {
  long long dq_batch_stride, dq_token_stride;
  long long dk_batch_stride, dk_token_stride;
  long long dv_batch_stride, dv_token_stride;
  long long do_batch_stride, do_token_stride;
  /* Optional (head_dim 64 only): the q/k/v projection's bias gradient without a second pass over dq/dk/dv.  When not NULL,
   * row b * ceil(T / 128) + t of bias_partial (f32, leading dimension bias_partial_ld) receives the column sums of the t-th
   * 128-token tile of batch row b: dq at columns [q_col, q_col + H*D), dk at [k_col, ...), dv at [v_col, ...), each laid out
   * [head][d]; tome_reduce_rows_f32 adds the B * ceil(T / 128) rows up.  (DenseGeneral bias, tome_attention.py:145-164.) */
  float* bias_partial;
  long long bias_partial_ld;
  int bias_q_col, bias_k_col, bias_v_col;
} tome_attn_grad_strides_t;
size_t tome_attention_bwd_workspace_bytes(const tome_attn_desc_t* desc);
int tome_attention_bwd(const tome_attn_desc_t* desc, const tome_attn_grad_strides_t* gs, const void* q, const void* k,
                       const void* v, const void* out, const float* lse, const void* dout, void* dq, void* dk,
                       void* dv, void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 5b. Per-modality top-k pruning       tokenizers/token_compression.py:15-46 (compute_top_k_tokens): the sibling
 *                                      compression path of SURVEY.md 8(f) rank 2
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int batch, tokens, channels;
  int dtype;        /* tome_dtype of the embeddings */
  int n_sets;       /* token sets ("modalities"), in output order */
  int set_start[TOME_MAX_TOKEN_SETS]; /* tokenset_idx[s][0] */
  int set_n[TOME_MAX_TOKEN_SETS];     /* tokenset_idx[s][1] */
  int set_k[TOME_MAX_TOKEN_SETS];     /* tokenset_k[s]: 0 <= k <= n (jax.lax.top_k raises otherwise) */
  int score_planes; /* importance is [score_planes, B, T]; planes are summed in order before ranking (1 = plain [B,T]) */
} tome_prune_desc_t;
/* For every set keep the k highest-scoring tokens in descending score order (equal scores: lower index first, as
 * jax.lax.top_k; NaN ranks above every number), sets concatenated in order:
 * ids i32 [B, sum k] = kept token indices, out [B, sum k, C] = embeddings gathered through ids (bit copies). */
int tome_topk_prune(const tome_prune_desc_t* desc, const void* embeddings, const float* importance, void* out,
                    int32_t* ids, void* stream);
/* What a stack of pruning layers needs around the gather (compressed_attention.py:396-402, one prune per layer):
 * row_map i32 [B, T] = output row of every token, -1 for a pruned one (the inverse of ids [B, kept]); gid_out / pos_out
 * (optional) = the mask group / position of the kept tokens, carried with them. */
int tome_prune_row_map(int batch, int tokens, int kept, const int32_t* ids, const uint8_t* gid, const int32_t* pos,
                       int32_t* row_map, uint8_t* gid_out, int32_t* pos_out, void* stream);
/* Backward of the gather (autodiff of token_compression.py:41-44): dx [B, T, C] = dy [B, kept, C] rows through row_map,
 * zero rows for pruned tokens. */
int tome_prune_bwd(int batch, int tokens, int kept, int channels, int dtype, const int32_t* row_map, const void* dy, void* dx,
                   void* stream);

/* Token importance from the attention weights   attention_blocks/compressed_attention.py:303-306:
 *   importance [B, T] = mean over heads ( mean over one token axis ( softmax weights [B, H, Tq, Tk] ) ).
 * TOME_IMPORTANCE_ROW_MEAN: the inner mean runs over the KEYS, the expression as the reference writes it (rows of a
 * softmax sum to one, so every score is 1 / T up to rounding; kept for fidelity).  TOME_IMPORTANCE_RECEIVED: over the
 * QUERIES -- the attention a token receives, a usable ranking for tome_topk_prune.  desc / q / k as tome_attention_fwd
 * (mask and log(size) bias included), lse [B, H, T] = what that call wrote; weights are the undropped ones. */
enum tome_importance_mode { TOME_IMPORTANCE_ROW_MEAN = 0, TOME_IMPORTANCE_RECEIVED = 1 };
int tome_attention_importance(const tome_attn_desc_t* desc, const void* q, const void* k, const float* lse, int mode,
                              float* importance, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 6. Small fused steps around the block
 * ------------------------------------------------------------------------------------------------------------ */

/* y[b,t,:] = x[b,t,:] + pos_embedding[t,:]     attention.py:97-100 (x f32 or bf16 -> y bf16) */
int tome_add_pos_embedding(int batch, int tokens, int channels, const void* x, int x_dtype, const float* pos_embedding,
                           void* y, void* stream);
/* dpe[t,:] += sum_b dy[b,t,:]  (f32 accumulate) */
int tome_pos_embedding_bwd(int batch, int tokens, int channels, const void* dy, float* dpe, void* stream);

/* origin[b,i] <- row of the final sequence that original token readout_idx[i] ended up in: chains the per-layer
 * row maps (row_maps_host: host array of `layers` device pointers, entry l is i32 [B, tokens_host[l]] or NULL when
 * layer l merged nothing).  Replaces unmerge + jnp.take(embeddings, readout_idx) of octo.py:123-124. */
int tome_chain_row_maps(int batch, int layers, const int32_t* const* row_maps_host, const int* tokens_host,
                        const int32_t* readout_idx, int n_readout, int32_t* origin, void* stream);

/* Synthetic stand-in for octo.py:167-174: out[b,i,:] = x[b,origin[b,i],:]; loss = mean((out - target)^2);
 * writes dx (bf16 [B,T,C], zero except gathered rows, summed where two readouts share a row), loss f32 [1 + B]
 * (loss[0] = the mean; loss[1..B] = per-row partial sums, reduced in a fixed order), and optionally the gathered
 * rows `out` f32 [B,n,C]. target f32 [B,n,C]. */
int tome_readout_mse(int batch, int tokens, int channels, int n_readout, const void* x, const int32_t* origin,
                     const float* target, float* loss, void* dx, float* out, void* stream);

/* Action heads on the pooled readout rows and their training losses (SURVEY.md 8(f) rank 3).
 *   TOME_HEAD_CONTINUOUS_L2:  action_heads/continuous.py:16-25 + models/octo/octo.py:157-165, 253-263
 *       pooled = mean over all n_readout rows; z = pooled W + b; out = tanh(z / max_action) * max_action  (f32 [B, features]);
 *       loss_b = sum_a (out - actions[b,a])^2, loss[0] = mean_b loss_b.  groups must be 1; actions f32 [B, features].
 *   TOME_HEAD_CATEGORICAL_CE: action_heads/categorical.py:12-40 + models/octo/octo.py:178-190, 292-303
 *       readout i belongs to action group i / (n_readout / groups) ("(action timestep)"); pooled[g] = mean of the group;
 *       out = logits = pooled[g] W + b (f32 [B, groups, features], features = num_bins);
 *       label = one_hot(digitize(actions[b,g], linspace(-max_action, max_action, features + 1)), features) -- literally:
 *       digitize is 1-based, so bin k maps to class k + 1 and the top bin / out-of-range values to an all-zero label, whose
 *       cross-entropy is 0; loss[0] = mean over (b, g) of -sum_f label_f log_softmax(logits)_f.  actions f32 [B, groups].
 * x is the FINAL sequence of the stack ([B, tokens, C], bf16 or f32) and origin i32 [B, n_readout] the row each readout
 * token ended up in (tome_chain_row_maps; arange(n_readout) for an already gathered readout tensor, tokens = n_readout).
 * w f32 [C, features] (Flax Dense kernel layout), bias f32 [features] or NULL.  loss f32 [1 + B] as tome_readout_mse
 * (NULL: inference).  workspace (tome_action_head_workspace_bytes; NULL when no backward follows) keeps pooled and
 * dL/dz for tome_action_head_bwd, which ACCUMULATES into dw [C, features] / dbias [features] (summed over the batch in a
 * fixed order) and OVERWRITES dx (x's dtype and shape; zero except the readout rows; NULL to skip). */
#define TOME_HEAD_CONTINUOUS_L2 0
#define TOME_HEAD_CATEGORICAL_CE 1
typedef struct {
  int batch, tokens, channels;
  int x_dtype;      /* tome_dtype of x / dx */
  int n_readout;
  int groups;       /* 1 (continuous) or action_space_dim (categorical) */
  int features;     /* Dense features: action dimensions (continuous) or num_bins (categorical) */
  int kind;         /* TOME_HEAD_* */
  float max_action;
} tome_head_desc_t;
size_t tome_action_head_workspace_bytes(const tome_head_desc_t* desc);
int tome_action_head_fwd(const tome_head_desc_t* desc, const void* x, const int32_t* origin, const float* w,
                         const float* bias, const float* actions, float* out, float* loss, void* workspace,
                         size_t workspace_bytes, void* stream);
int tome_action_head_bwd(const tome_head_desc_t* desc, const int32_t* origin, const float* w, const void* workspace,
                         float* dw, float* dbias, void* dx, void* stream);

/* The attention step of MultiHeadAttentionPooling (attention_blocks/attention.py:139-147; forward): the learnt query
 * [embed_dim] is projected once (wq f32 [embed_dim, heads * head_dim] = the Flax query kernel [E, H, D] flattened, bq f32
 * [H * D] or NULL; scaled by 1 / sqrt(head_dim)), then one softmax over the n_keys (<= 64) key rows of every (batch row, head)
 * and the weighted sum of the value rows.  kv: bf16 [batch, n_keys, kv_ld], keys at column 0, values at column v_col (each
 * [H, D] wide: the output of one GEMM over the concatenated key | value kernels).  q_scratch f32 [H * D]; out bf16
 * [batch, H * D], the input of the out projection (:147), LayerNorm (:148) and MLPBlock (:149) -- the library's GEMM /
 * LayerNorm entry points. */
int tome_attention_pool_fwd(int batch, int n_keys, int heads, int head_dim, int embed_dim, const float* learnt_q,
                            const float* wq, const float* bq, const void* kv, long long kv_ld, int v_col, float* q_scratch,
                            void* out, void* stream);

/* Diffusion action head, training path: DiffusionActionHead.denoise_loss over OctoDenoise / FourierFeatures / MLPBlock
 * (action_heads/diffusion.py:29-64, 94-143; the head octo_base.yaml selects).  The random draws are the caller's:
 * time i32 [B] in [0, diffusion_steps), noise f32 [B, A]; alpha_hats f32 [diffusion_steps] is the cumulative product of
 * 1 - cosine_beta_schedule (diffusion.py:16-26, 85-92).
 *   noisy = sqrt(ah[t]) actions + sqrt(1 - ah[t]) noise;  emb = mean over the readout rows (x / origin as tome_action_head_fwd);
 *   ff = [cos | sin](2 pi t fourier_kernel);  te = Dense_1(relu(Dense_0(ff)))          time encoder MLPBlock
 *   pred = Dense_1(relu(Dense_0([noisy | te | emb])))                                  denoiser MLPBlock (num_blocks = 1)
 *   loss[0] = mean_b sum_a 0.5 (pred - noise)^2, loss[1 + b] = per-row sums            optax.l2_loss
 * The MLPBlocks' Dropouts are inactive, as in the reference (OctoDenoise calls them without `train`).
 * Parameters: one flat fp32 vector + its bf16 copy (GEMM operands), layout
 *   fourier_kernel [F/2] | tw1 [F, Ht] tb1 [Ht] | tw2 [Ht, To] tb2 [To] | w1 [A + To + C, H] b1 [H] | w2 [H, A] b2 [A]
 * (kernels [in, out] as Flax stores them; tome_diffusion_head_param_offset(desc, i) gives the offset of the i-th array,
 * i = 9: the total).  backward ACCUMULATES into grads_f32 (same layout) and OVERWRITES dx (bf16 [B, tokens, C], zero
 * except the readout rows; NULL to skip); it needs the workspace forward wrote. */
typedef struct {
  int batch, tokens, channels;   /* x bf16 [B, tokens, C]; channels % 8 == 0 */
  int n_readout;
  int action_dim;                /* A: denoiser mlp_block.dense_out.features; multiple of 8 (diffusion.yaml: 8) */
  int fourier_dim;               /* F: FourierFeatures.output_dim, multiple of 16 */
  int time_hidden, time_out;     /* Ht, To: time_encoder.mlp_block dense / dense_out features */
  int hidden;                    /* H: denoiser mlp_block.dense.features */
  int diffusion_steps;
} tome_diffusion_desc_t;
long long tome_diffusion_head_param_count(const tome_diffusion_desc_t* desc);
long long tome_diffusion_head_param_offset(const tome_diffusion_desc_t* desc, int which);
size_t tome_diffusion_head_workspace_bytes(const tome_diffusion_desc_t* desc);
int tome_diffusion_head_fwd(const tome_diffusion_desc_t* desc, const float* params_f32, const void* params_bf16, const void* x,
                            const int32_t* origin, const float* actions, const float* noise, const int32_t* time,
                            const float* alpha_hats, float* pred, float* loss, void* workspace, size_t workspace_bytes,
                            void* stream);
int tome_diffusion_head_bwd(const tome_diffusion_desc_t* desc, const float* params_f32, const void* params_bf16,
                            const int32_t* origin, const int32_t* time, void* workspace, float* grads_f32, void* dx,
                            void* stream);

/* Diffusion action head, inference: DiffusionActionHead.predict_action (action_heads/diffusion.py:146-213), the whole reverse
 * process in one call.  Starting from init, for t = steps - 1 .. 0 (step i = steps - 1 - t):
 *   eps = the denoiser of tome_diffusion_head_fwd on [sample | te(t) | emb];  sample = clip(c1 (sample - c2 eps) + c3 noise_i)
 * with coef[t] = {c1 = 1/sqrt(alpha_t), c2 = (1 - alpha_t)/sqrt(1 - alpha_hat_t), c3 = sqrt(beta_t)} computed by the caller,
 * noise_i = noise ([B, A], reused by every step as the reference does at :179) or noise + i B A ([steps, B, A]), clip to
 * [-clip, clip] (:189).  x / origin as tome_diffusion_head_fwd; actions f32 [B, A] out.  The denoiser input's first A columns
 * run in fp32 (W1[:A], W2 and b2 from params_f32); the readout mean and the time embedding through bf16 GEMMs as in training.
 * One kernel runs every step, so the call makes six launches whatever `steps` is.  It needs action_dim <= 64, hidden <= 2048
 * and W1[:A] and W2 in fp32 (8 A H bytes) within 227 KB of shared memory, else TOME_ERR_UNSUPPORTED.
 * Deterministic: the same inputs give the same bits, whatever the batch size. */
typedef struct {
  const float* init;    /* f32 [B, A]: the Gaussian start (diffusion.py:203) */
  const float* noise;   /* f32 [B, A] (noise_per_step = 0) or [steps, B, A] (noise_per_step = 1) */
  int noise_per_step;
  const float* coef;    /* f32 [steps, 3]: c1, c2, c3 of time step t in row t */
  float clip;           /* > 0; the reference clips to 5.0 */
} tome_ddpm_sample_t;
size_t tome_diffusion_head_sample_workspace_bytes(const tome_diffusion_desc_t* desc);
int tome_diffusion_head_sample(const tome_diffusion_desc_t* desc, const float* params_f32, const void* params_bf16, const void* x,
                               const int32_t* origin, const tome_ddpm_sample_t* sample, float* actions, void* workspace,
                               size_t workspace_bytes, void* stream);

/* AdamW on an fp32 master vector with a bf16 working copy refreshed in the same pass (bf16_copy may be NULL).
 * grad_scale multiplies the gradient first (1/world_size after a sum all-reduce).  Per element, with g = grad_scale * grad:
 *   m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;  p -= lr * ((m / bc1) / (sqrt(v / bc2) + eps) + wd * p)
 * with bc1 = 1 - b1^step, bc2 = 1 - b2^step computed in fp32 on the host.
 *
 * opts == NULL is exactly this plain step (ABI 16).  opts adds, without any host synchronisation (ABI 17):
 *   - the global L2 norm of g over all n elements, written to grad_norm when given.  It is a fixed-order reduction (a
 *     compile-time partition into chunks, fp32 inside a chunk, fp64 across chunks), so the same gradient bits give the same
 *     norm bits whatever the GPU, its SM count or tome_gemm_set_sm_limit: data-parallel replicas that all-reduced the same
 *     gradient stay identical.  Computed when max_grad_norm > 0, skip_nonfinite or grad_norm != NULL;
 *   - clipping as optax.clip_by_global_norm: g unchanged when norm < max_grad_norm, else g * (max_grad_norm / norm);
 *   - skipping as optax.apply_if_finite: a NaN / Inf in g leaves param, m, v, bf16_copy and steps[0] untouched and adds 1 to
 *     steps[1];
 *   - steps != NULL: bias correction uses t = steps[0] + 1 (applied steps only) instead of `step`, computed on the device in
 *     fp64 and rounded to fp32, and the call adds 1 to steps[0] when it applies the step;
 *   - decay_ranges: weight decay only inside these element ranges (e.g. the Dense kernels; not LayerNorm, biases or embeddings).
 * Malformed options return TOME_ERR_INVALID before any CUDA call. */
#define TOME_ADAMW_MAX_DECAY_RANGES 512
typedef struct {
  float max_grad_norm;            /* > 0: clip g to this global L2 norm; 0: no clipping; negative or non-finite: refused */
  int skip_nonfinite;             /* 1: a g with a NaN / Inf leaves every buffer untouched (needs steps) */
  const long long* decay_ranges;  /* HOST array [2 * n_decay_ranges]: sorted, disjoint, non-empty half-open ranges [lo, hi) in
                                     [0, n) that get weight decay; NULL: every element */
  int n_decay_ranges;             /* 0 .. TOME_ADAMW_MAX_DECAY_RANGES */
  float* grad_norm;               /* device f32 [1], optional: the norm of g before clipping */
  int* steps;                     /* device i32 [2] {applied, skipped}, optional; required when skip_nonfinite */
  void* workspace;                /* 16-byte aligned, tome_adamw_workspace_bytes(n) bytes; needed when the norm or steps is used */
  size_t workspace_bytes;
} tome_adamw_opts_t;
size_t tome_adamw_workspace_bytes(long long n);
int tome_adamw_step(long long n, float* param, const float* grad, float* m, float* v, void* bf16_copy, float lr,
                    float beta1, float beta2, float eps, float weight_decay, float grad_scale, int step,
                    const tome_adamw_opts_t* opts, void* stream);

/* dst_bf16[i] = (bf16) src_f32[i] */
int tome_cast_f32_to_bf16(long long n, const float* src, void* dst, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 7. The whole stack: StackedEncoder1DBlock of ToMeEncoder1DBlock, unrolled with shrinking T
 *    attention.py:41-119, tome_attention.py:305-383, placement per SURVEY.md A.7
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int batch, tokens, channels, heads, head_dim, mlp_dim, layers;
  int r;              /* tokens merged per layer (clamped per layer) */
  int ln_axis;        /* 1 = tokens (reference yaml), 2 = features */
  float ln_eps;       /* 1e-6 */
  int prop_attn;      /* logits += log(size) */
  int class_token, distill_token;
  int num_groups;     /* 0: no mask */
  int n_readout;
  float dropout_rate; /* hidden dropout after out-proj, ReLU and dense_out (attention.py:34,37,60); 0 in parity mode */
  uint64_t dropout_seed;
  float attn_dropout_rate; /* attention-weight dropout (self_attention.dropout_rate, vanilla_decoder.yaml:23), same seed */
  int head;           /* loss on the readout rows: 0 = synthetic MSE against target [B,n_readout,C] (tome_readout_mse);
                         1 + TOME_HEAD_*: that action head and its loss (tome_action_head_*), target = actions;
                         3: the diffusion head's denoise loss (tome_diffusion_head_*), target = [actions | noise] */
  int head_groups;    /* tome_head_desc_t.groups */
  int head_features;  /* tome_head_desc_t.features / tome_diffusion_desc_t.action_dim */
  float max_action;
  int head_fourier_dim, head_time_hidden, head_time_out, head_hidden, diffusion_steps; /* tome_diffusion_desc_t (head 3) */
  /* Per-modality top-k PRUNING per layer instead of merging (the sibling compression path: token_compression.py:15-46 applied
   * by every layer, compressed_attention.py:303-308, 396-402; grammar of token_sequencer.py:222-238).  prune_sets > 0 selects it
   * (r must be 0, prop_attn 0): the sequence is prune_sets consecutive token sets; set i holds prune_set_n[i] tokens at layer 0
   * and every layer drops its prune_set_c[i] least important ones (scores: prune_importance, a tome_importance_mode), keeping
   * the rest in descending score order.  The reference prunes the attention output before the out projection and then adds
   * the UNPRUNED residual (a shape error as written); here the same token choice is applied after the residual add, which is
   * what pruning both branches alike gives. */
  int prune_sets;
  int prune_set_n[TOME_MAX_TOKEN_SETS];
  int prune_set_c[TOME_MAX_TOKEN_SETS];
  int prune_importance;
  /* set_merge != 0 (with prune_sets > 0): every layer MERGES prune_set_c[i] tokens inside set i instead of pruning them --
   * bipartite soft matching on the keys averaged over heads, merge_wavg after the attention residual, sizes carried (prop_attn
   * allowed), group id / position carried as by the global merge (tome_token_sets_t).  r must be 0, no class / distill token,
   * prune_set_c[i] <= floor(n_i(l) / 2) at every layer l, and layer_gid / layer_pos are not taken. */
  int set_merge;
} tome_stack_cfg_t;

/* Per-layer parameter offsets (elements) into one flat fp32 vector (master weights / gradients / Adam moments)
 * and the same offsets into a flat bf16 working copy.  Kernels are stored [in, out] (Flax layout):
 * wqkv [C, 3*H*D] = concat(query, key, value kernels), wo [H*D, C], w1 [C, Dff], w2 [Dff, C].
 * Layout of one layer: ln1_scale[C] ln1_bias[C] wqkv bqkv[3HD] wo bo[C] ln2_scale[C] ln2_bias[C] w1 b1[Dff] w2 b2[C];
 * the vector starts with pos_embedding [T0, C]; with cfg.head > 0 it ends with the head's parameters (tome_stack_head_offset;
 * -1 without a head): Dense kernel [C, features] and bias [features], or the diffusion head's vector (its own layout).  tome_stack_param_count gives the total. */
long long tome_stack_param_count(const tome_stack_cfg_t* cfg);
long long tome_stack_head_offset(const tome_stack_cfg_t* cfg);
long long tome_stack_layer_offset(const tome_stack_cfg_t* cfg, int layer); /* offset of ln1_scale of `layer` */

/* bytes of activation workspace the executor needs (saved activations for backward + scratch) */
size_t tome_stack_workspace_bytes(const tome_stack_cfg_t* cfg);

typedef struct {
  const float* params_f32;    /* flat fp32 (biases, LN, pos-embedding are read from here) */
  const void* params_bf16;    /* flat bf16 copy (GEMM operands) */
  const void* x;              /* [B,T0,C] input embeddings */
  int x_dtype;
  const uint8_t* gid;         /* [T0] group ids (same for every batch row at layer 0) or NULL */
  const int32_t* pos;         /* [T0] */
  const uint8_t* allow;       /* [G,G] */
  const int32_t* readout_idx; /* [n_readout] original positions of the readout tokens */
  const float* target;        /* loss target or NULL: [B,n_readout,C] (head 0), actions [B,features] (continuous head),
                                 [B,groups] (categorical head), [2,B,A] = actions then noise (diffusion head) */
  void* workspace; size_t workspace_bytes;
  /* outputs */
  void* x_final;              /* bf16 [B,T_L,C] (points into workspace when NULL is passed: see tome_stack_final) */
  float* readout;             /* f32 [B,n_readout,C] or NULL */
  float* loss;                /* f32 [1 + B] (see tome_readout_mse) */
  float* grads_f32;           /* flat fp32 gradient vector (backward; accumulated into, caller zeroes) */
  void* const* layer_done_events; /* optional host array [layers+1] of cudaEvent_t recorded as each layer's (and
                                     finally the pos-embedding's) gradients become final, for all-reduce overlap */
  float* head_out;            /* f32 [B, head_groups, head_features]: actions (continuous), logits (categorical) or the
                                 predicted denoise term [B, A] (diffusion); required when cfg.head > 0 */
  const int32_t* head_time;   /* diffusion head: i32 [B] sampled time steps */
  const float* head_alpha_hats; /* diffusion head: f32 [diffusion_steps] */
  void* grad_trace;           /* optional (parity tests), bf16 [layers, B * T0 * C]: backward copies dL/dx_out of layer l (its
                                 first B * T_out(l) * C elements) into slot l before it consumes it, so a checker can run
                                 each layer's backward on the implementation's own incoming gradient */
  /* Pruning stacks: the per-layer attention masks of the compression grammar (TokenSequence.generate_attention_mask(layer = l),
   * token_sequencer.py:222-238, 313-321, what compressed_attention.py:399 passes as masks[layer_idx]) as group ids / positions:
   * u8 / i32 [sum over layers of T_in(l)], layer after layer, the same for every batch row.  NULL: the layer-0 gid / pos are
   * carried with the kept tokens instead (a kept token keeps its own group and position). */
  const uint8_t* layer_gid;
  const int32_t* layer_pos;
} tome_stack_io_t;

int tome_stack_forward(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, void* stream);
/* runs loss gradient + full backward; tome_stack_forward must have run on the same workspace */
int tome_stack_backward(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, void* stream);
/* device pointers into the workspace, valid after forward: final tokens/sizes and per-layer plan dumps (tests) */
int tome_stack_tokens_at(const tome_stack_cfg_t* cfg, int layer); /* T entering `layer`; layer == layers: final T */
const void* tome_stack_final_x(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io);
/* bf16 [B, T_in(layer), C]: the tokens entering `layer` (after the position embedding for layer 0); layer == layers: final x */
const void* tome_stack_layer_x_in(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
/* f32 [B, T_in(layer)] token sizes entering `layer`, or NULL while every size is still 1 */
const float* tome_stack_layer_size_in(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
const float* tome_stack_final_size(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io);
const int32_t* tome_stack_layer_edge_idx(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
const int32_t* tome_stack_layer_dst_idx(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
const float* tome_stack_layer_node_max(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
const int32_t* tome_stack_layer_node_idx(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
/* u32 [B * T_out(layer), ceil(mlp_dim / 32)]: bit j of word w = element 32 w + j of MLP-1's output survived ReLU (and hidden
 * dropout), i.e. the gate the MLP backward of attention.py:32-34 uses; lets a checker take the SAME gate decisions. */
const uint32_t* tome_stack_layer_relu_bits(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
/* pruning stacks: f32 [B, T_in(layer)] importance scores the layer ranked, i32 [B, T_out(layer)] the token indices it kept */
const float* tome_stack_layer_importance(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);
const int32_t* tome_stack_layer_prune_ids(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, int layer);

/* Forward-only executor: the forward of tome_stack_forward over a workspace that keeps nothing for backward.  The residual
 * stream, sizes and group ids ping-pong between two buffers and every layer reuses one set of scratch; only each merging or
 * pruning layer's row map (4 B T_in(l) bytes) stays, for the readout origins, so the workspace does not otherwise grow with
 * `layers`.  Every stack kind tome_stack_forward accepts runs here.
 *   - Dropout is off: cfg->dropout_rate and attn_dropout_rate are not applied, so one cfg serves a training executor and its
 *     predictor.  The reference's Octo.generate_readouts passes train=True even when predicting (octo.py:120); stochastic
 *     prediction as it does is tome_stack_forward with the dropout rates set.
 *   - At dropout 0 x_final, readout and head_out (heads 1 and 2) equal tome_stack_forward's bit for bit.
 *   - Outputs, each optional except head_out when cfg->head > 0: io->x_final (bf16 [B, T_L, C]), io->readout (f32
 *     [B, n_readout, C]), io->head_out: tanh actions [B, A] (head 1), logits [B, groups, bins] (head 2), or actions [B, A]
 *     sampled by tome_diffusion_head_sample with `sample` (head 3; sample must be NULL for any other head).
 *   - io->target, loss, grads_f32, grad_trace, head_time, head_alpha_hats and layer_done_events are not read.
 *   - io->workspace holds tome_stack_predict_workspace_bytes(cfg) bytes.  The tome_stack_layer_* / tome_stack_final_*
 *     accessors describe the training workspace and are invalid on a predict workspace. */
size_t tome_stack_predict_workspace_bytes(const tome_stack_cfg_t* cfg);
int tome_stack_predict(const tome_stack_cfg_t* cfg, const tome_stack_io_t* io, const tome_ddpm_sample_t* sample, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 7b. Image patch-embed front end (forward)   tokenizers/images/image_tokenizer.py:35-71 (image_to_patches), :74-140
 *     (encode_patch_position), :148-190 (ResNetV2Block), :216-309 (ImageTokenizer); config form of
 *     model_configs/tokenizers/images/gato_resnet.yaml.  SURVEY.md 8(f) rank 4: the compute ahead of the block.
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct {
  int batch, n_images;   /* images [B, N, H, W, C_in], square */
  int image_size;        /* H = W, a multiple of patch_size */
  int channels_in;
  int image_dtype;       /* TOME_U8 (raw pixels 0..255) or TOME_F32 (the reference's float pixels) */
  int normalize;         /* 2 * (x / 255) - 1 before the first convolution (image_tokenizer.py:67) */
  int patch_size;        /* patches in row-major (h, w) order, each embedded on its own */
  int conv_kernel, conv_stride;   /* input convolution, padding VALID (gato_resnet.yaml: 12, 2) */
  int features;          /* channels of every convolution (64); a multiple of 8 and of num_groups */
  int pool_window;       /* max pool, stride 1, VALID (3) */
  int num_blocks;        /* x [GroupNorm -> gelu(tanh) -> Conv 3x3 SAME]; the pooled tensor is added back after the last */
  int num_groups;        /* GroupNorm groups (32).  Flax semantics: the statistics of a group run over EVERY axis but the
                            batch one, i.e. over the N images, all patches, H, W and the group's channels of a batch row */
  float gn_eps;
  int embed_dim;         /* output Dense features (768); a multiple of 8 */
  int position_interval; /* rows of the two position-embedding tables */
  int token_rows;        /* position tokens are given per patch for every image alike (1: evaluation mode, the interval
                            midpoints) or per (batch row, image) (batch * n_images: training mode, sampled by the caller) */
  int out_dtype;         /* TOME_BF16 or TOME_F32 */
  int chunk_rows;        /* batch rows processed per pass (bounds the workspace); 0 = the library chooses (~1 GiB of im2col rows).
                            GroupNorm statistics are per batch row, so the result does not depend on it */
} tome_image_tokenizer_desc_t;

/* Flat parameter vector (f32 master and bf16 working copy, same offsets): conv0 kernel [k*k*C_in, F] (= Flax [k, k, C_in, F]),
 * conv0 bias [F]; per block: GroupNorm scale [F], bias [F], conv kernel [9F, F], conv bias [F]; dense kernel [o*o*F, E],
 * dense bias [E]; row embedding [P, E]; column embedding [P, E]   (o = (patch - k) / stride + 1 - (pool_window - 1)). */
enum tome_image_tokenizer_param { TOME_IT_CONV0_KERNEL = 0, TOME_IT_CONV0_BIAS, TOME_IT_DENSE_KERNEL, TOME_IT_DENSE_BIAS,
                                  TOME_IT_ROW_EMBED, TOME_IT_COL_EMBED,
                                  TOME_IT_BLOCK0 = 16 /* + 4 * block + {0: gn scale, 1: gn bias, 2: conv kernel, 3: conv bias} */ };
long long tome_image_tokenizer_param_count(const tome_image_tokenizer_desc_t* desc);
long long tome_image_tokenizer_param_offset(const tome_image_tokenizer_desc_t* desc, int which);
size_t tome_image_tokenizer_workspace_bytes(const tome_image_tokenizer_desc_t* desc);
/* out [B, N, n_patches, E] = ImageTokenizer(image).  row_tokens / col_tokens: i32 [token_rows, n_patches] indices into the
 * embedding tables (evaluation mode: image_tokenizer.py:111-113; the Python mirror computes them).  The convolutions and the
 * Dense run on the tcgen05 GEMM (input convolution: im2col rows; 3 x 3 convolutions with features % 64 == 0: row-shifted windows
 * of the zero-bordered activation, tome_gemm_args_t.a_row_shift), bf16 activations, fp32 accumulation.  workspace: 256-byte aligned, tome_image_tokenizer_workspace_bytes(desc) bytes. */
int tome_image_tokenizer_fwd(const tome_image_tokenizer_desc_t* desc, const void* image, const float* params_f32,
                             const void* params_bf16, const int32_t* row_tokens, const int32_t* col_tokens, void* out,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 7c. Pixels to actions in one call (ABI 18): Octo.generate_readouts (models/octo/octo.py:91-126) under
 *     predict_continuous_action / predict_diffusion_action -- image front end -> sequence assembly -> forward-only stack -> head
 * ------------------------------------------------------------------------------------------------------------ */
/* One non-image token set of the sequence (text or readouts): bf16 [B or 1, n, C] rows copied to sequence rows
 * first_row .. first_row + n - 1.  batch_stride (elements, a multiple of 8) is 0 to give every batch row the same n rows
 * (readout embeddings) or >= n * C.  rows is 16-byte aligned. */
typedef struct {
  const void* rows;
  long long batch_stride;
  int n;
  int first_row;
} tome_policy_rows_t;

typedef struct {
  tome_image_tokenizer_desc_t image;  /* batch == cfg->batch, embed_dim == cfg->channels, out_dtype == TOME_BF16 */
  const float* image_params_f32;      /* the front end's flat parameters (section 7b) and their bf16 copy */
  const void* image_params_bf16;
  const void* pixels;                 /* [B, N, H, W, C_in], u8 or f32 as image.image_dtype */
  const int32_t* row_tokens;          /* i32 [image.token_rows, n_patches] (device), as tome_image_tokenizer_fwd */
  const int32_t* col_tokens;
  const int32_t* image_rows;          /* HOST i32 [N * n_patches]: sequence row of image token n * n_patches + p (the grammar's
                                         image positions in order, TokenSequence.get_modality_idx("images")); at most 32 runs
                                         of consecutive rows */
  int n_sets;                         /* 0 .. TOME_MAX_TOKEN_SETS */
  tome_policy_rows_t sets[TOME_MAX_TOKEN_SETS];
} tome_policy_inputs_t;

/* tome_policy_predict runs, on `stream`: the image front end of section 7b writing each bf16 token (b, n, p) straight into row
 * image_rows[n * n_patches + p] of an assembled [B, T0, C] sequence; one kernel copying every non-image set into its rows; then
 * tome_stack_predict on that sequence (io->x and io->x_dtype are not read; every other io field and `sample` as there).  The
 * sequence, and with it every output, equals TokenSequence.assemble_embeddings of the front end's bf16 tokens fed to
 * tome_stack_predict, bit for bit.
 * Workspace (io->workspace, 256-byte aligned, tome_policy_predict_workspace_bytes bytes): the sequence, then one region the
 * front end's scratch and the predict layout share, so the size is the sequence plus the larger of
 * tome_image_tokenizer_workspace_bytes and tome_stack_predict_workspace_bytes.
 * Validation runs on the host before any CUDA call and returns TOME_ERR_INVALID naming the fault: batch differs between cfg and
 * the descriptor, embed_dim != channels, out_dtype not bf16, an image row outside [0, T0), image and set rows not covering
 * [0, T0) exactly once, a malformed set; shapes the front end, the stack or the sampler refuse keep their own errors.
 * Graph capture: for fixed pointers and shapes the call allocates nothing, never synchronises, reads no device memory on the
 * host and launches the same kernels with the same parameters every time, so a caller may capture it in a CUDA graph and
 * replay it with new pixels, sets and draws written into the same buffers.  The first call must run eagerly, before any
 * capture: it sets kernel attributes (shared-memory limits) and loads the modules, which a capturing stream cannot do. */
size_t tome_policy_predict_workspace_bytes(const tome_stack_cfg_t* cfg, const tome_policy_inputs_t* inputs);
int tome_policy_predict(const tome_stack_cfg_t* cfg, const tome_policy_inputs_t* inputs, const tome_stack_io_t* io,
                        const tome_ddpm_sample_t* sample, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * 8. Launch accounting and per-op timing (measurement aid; off by default, never on the product path's hot loop)
 * ------------------------------------------------------------------------------------------------------------ */
enum tome_prof_tag { TOME_PROF_GEMM = 0, TOME_PROF_ATTN_FWD, TOME_PROF_ATTN_BWD, TOME_PROF_MERGE_FWD, TOME_PROF_MERGE_BWD,
                     TOME_PROF_SIM, TOME_PROF_SELECT, TOME_PROF_LN, TOME_PROF_COLSUM, TOME_PROF_OTHER, TOME_PROF_IMPORTANCE,
                     TOME_PROF_PRUNE, TOME_PROF_NTAGS };
/* number of kernels this library has launched in this process (reset != 0 zeroes the counter after reading) */
long long tome_launch_count(int reset);
/* record ONE CUDA event at the end of every op on its stream (up to max_records ops): op i is timed from the end of op
 * i-1 (the first from a start event), so markers perturb short kernels half as much and inter-op gaps are charged to
 * the op that follows them.  Meant for a single stream (the stack executor's). */
int tome_profile_enable(int max_records);
int tome_profile_disable(void);
/* per tag: total milliseconds, total algorithmic work (FLOPs for GEMM / attention / sim, bytes for merge / LN /
 * colsum), number of ops; clears the records.  Arrays must hold TOME_PROF_NTAGS entries. */
int tome_profile_collect(int n_tags, float* ms, double* work, int* count);

#ifdef __cplusplus
}
#endif
#endif /* TOME_B200_H */
