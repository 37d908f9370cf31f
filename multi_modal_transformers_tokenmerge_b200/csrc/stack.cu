// The whole stack as one native executor: StackedEncoder1DBlock of ToMeEncoder1DBlock, unrolled because the token
// count shrinks by r per layer (an nn.scan carry cannot do that: SURVEY.md 3.3).
//
//   x = x + pos_embedding                                                       attention.py:97-100
//   per layer:  h   = LN1(x)                                                    attention.py:58
//               qkv = h Wqkv + b ; o = attention(q, k, v, group mask, log size) tome_attention.py:145-164, 259-285
//               x1  = x + dropout(o Wo + bo)                                    :287-299, attention.py:60-63
//               metric = mean_heads(k) -> match -> x1m, size = merge_wavg(x1)   tome_attention.py:249-256 (intent),
//                                                                               token_compression.py:54-129
//               y   = x1m + dropout(W2 dropout(relu(W1 LN2(x1m) + b1)) + b2)    attention.py:66-69, :32-37
//   readout rows gathered through the chained row maps, synthetic MSE loss      octo.py:123-124, 167-174
//
// Host code only: it sequences the kernels of this library on one stream and owns the layout of the activation
// workspace (everything saved for backward lives there; the library allocates nothing).  Every launch has static
// shapes, so a whole step can be captured in a CUDA graph by the caller.
#include <string.h>

#include <vector>

#include "common.cuh"
#include "host_util.h"

namespace tome {

// dropout sites: hidden dropout uses 3 * layer + {0: out-proj, 1: MLP hidden, 2: MLP out}; attention-weight dropout of layer l
// draws from site kAttnDropSite + l
constexpr uint32_t kAttnDropSite = 0x40000000u;

struct LayerShape {
  int t_in, r, t_out;
};

struct LayerBufs {
  // saved for backward
  __nv_bfloat16 *x_in, *h, *qkv, *attn_o, *x1m, *h2, *m1, *x_out;
  uint32_t* m1_bits;  // [B*To, F/32]: one bit per element of m1 (ReLU and dropout survive), the gate of the MLP dgrad
  float *ln1_mean, *ln1_rstd, *ln2_mean, *ln2_rstd, *lse;
  float *size_in, *size_out;  // size_in == nullptr at layer 0 (all ones)
  uint8_t *gid_in, *gid_out;
  int32_t *pos_in, *pos_out;
  float* node_max;
  int32_t* node_idx;
  tome_plan_t plan;
  float* importance;     // pruning stacks: [B, T] scores ranked by this layer
  int32_t* prune_ids;    // pruning stacks: [B, To] kept token indices
};

struct StackLayout {
  std::vector<LayerShape> shapes;
  std::vector<LayerBufs> L;
  __nv_bfloat16 *x1_scratch, *g0, *g1, *g2, *g3, *big;
  float *ws_gemm, *ws_colsum, *ws_ln;
  float* ws_colpart;   // [ceil(B T0 / 128), widest N]: per-row-tile column sums written by a GEMM epilogue
  uint8_t *ws_attn, *ws_sim;
  size_t ws_attn_bytes, ws_sim_bytes;
  int32_t* origin;
  uint8_t* ws_head;      // pooled readouts + dL/dz of the action head (cfg.head > 0)
  size_t ws_head_bytes;
  size_t ws_gemm_bytes;
  size_t total;
};

struct ParamOffsets {
  long long ln1_scale, ln1_bias, wqkv, bqkv, wo, bo, ln2_scale, ln2_bias, w1, b1, w2, b2, end;
};

static ParamOffsets layer_offsets(const tome_stack_cfg_t* c, int layer) {
  const long long C = c->channels, HD = (long long)c->heads * c->head_dim, F = c->mlp_dim;
  const long long per = C + C + C * 3 * HD + 3 * HD + HD * C + C + C + C + C * F + F + F * C + C;
  ParamOffsets o;
  long long p = (long long)c->tokens * C + per * layer;
  o.ln1_scale = p; p += C;
  o.ln1_bias = p; p += C;
  o.wqkv = p; p += C * 3 * HD;
  o.bqkv = p; p += 3 * HD;
  o.wo = p; p += HD * C;
  o.bo = p; p += C;
  o.ln2_scale = p; p += C;
  o.ln2_bias = p; p += C;
  o.w1 = p; p += C * F;
  o.b1 = p; p += F;
  o.w2 = p; p += F * C;
  o.b2 = p; p += C;
  o.end = p;
  return o;
}

// descriptor of the action head over the final sequence of `tokens` rows (cfg.head = 1 + TOME_HEAD_*)
static tome_head_desc_t head_desc(const tome_stack_cfg_t* c, int tokens) {
  tome_head_desc_t h;
  h.batch = c->batch; h.tokens = tokens; h.channels = c->channels; h.x_dtype = TOME_BF16;
  h.n_readout = c->n_readout; h.groups = c->head_groups; h.features = c->head_features;
  h.kind = c->head - 1; h.max_action = c->max_action;
  return h;
}

static tome_diffusion_desc_t diffusion_desc(const tome_stack_cfg_t* c, int tokens) {
  tome_diffusion_desc_t d;
  d.batch = c->batch; d.tokens = tokens; d.channels = c->channels; d.n_readout = c->n_readout;
  d.action_dim = c->head_features; d.fourier_dim = c->head_fourier_dim; d.time_hidden = c->head_time_hidden;
  d.time_out = c->head_time_out; d.hidden = c->head_hidden; d.diffusion_steps = c->diffusion_steps;
  return d;
}

static int check_cfg(const tome_stack_cfg_t* c) {
  TOME_CHECK(c != nullptr, TOME_ERR_INVALID, "stack: null config");
  TOME_CHECK(c->batch > 0 && c->tokens >= 2 && c->layers >= 1 && c->layers <= 64, TOME_ERR_INVALID,
             "stack: need batch > 0, tokens >= 2, 1 <= layers <= 64");
  TOME_CHECK(c->channels % 8 == 0 && c->mlp_dim % 8 == 0 && c->channels > 0 && c->mlp_dim > 0, TOME_ERR_INVALID,
             "stack: channels and mlp_dim must be positive multiples of 8");
  TOME_CHECK(c->head_dim >= 8 && c->head_dim <= 256 && c->head_dim % 8 == 0, TOME_ERR_UNSUPPORTED,
             "stack: head_dim %d not supported (64 on tensor cores; other multiples of 8 up to 256 on the generic attention path)",
             c->head_dim);
  TOME_CHECK(c->heads > 0, TOME_ERR_INVALID, "stack: heads must be positive");
  TOME_CHECK(c->ln_axis == 1 || c->ln_axis == 2, TOME_ERR_INVALID, "stack: ln_axis must be 1 (tokens) or 2 (features)");
  TOME_CHECK(c->r >= 0, TOME_ERR_INVALID, "stack: r must be >= 0");
  TOME_CHECK(c->num_groups >= 0 && c->num_groups <= 32, TOME_ERR_INVALID, "stack: num_groups must be in [0, 32]");
  TOME_CHECK(c->dropout_rate >= 0.f && c->dropout_rate < 1.f, TOME_ERR_INVALID, "stack: dropout_rate must be in [0, 1)");
  TOME_CHECK(c->attn_dropout_rate >= 0.f && c->attn_dropout_rate < 1.f, TOME_ERR_INVALID, "stack: attn_dropout_rate must be in [0, 1)");
  TOME_CHECK(c->n_readout >= 0, TOME_ERR_INVALID, "stack: n_readout must be >= 0");
  TOME_CHECK(c->prune_sets >= 0 && c->prune_sets <= TOME_MAX_TOKEN_SETS, TOME_ERR_INVALID, "stack: prune_sets must be in [0, %d]",
             TOME_MAX_TOKEN_SETS);
  TOME_CHECK(!c->set_merge || c->prune_sets > 0, TOME_ERR_INVALID, "stack: set_merge needs the token sets (prune_sets > 0)");
  if (c->prune_sets > 0 && c->set_merge) {
    TOME_CHECK(c->r == 0 && !c->class_token && !c->distill_token, TOME_ERR_INVALID,
               "stack: a set-merging stack (set_merge) takes r = 0 and no class / distill token");
    long long total = 0;
    for (int i = 0; i < c->prune_sets; ++i) {
      TOME_CHECK(c->prune_set_n[i] >= 1 && c->prune_set_c[i] >= 0, TOME_ERR_INVALID, "stack: token set %d: n >= 1, c >= 0", i);
      // every layer merges c tokens of the set's n(l) = n - l c: bipartite matching needs c <= floor(n(l) / 2)
      const long long n_last = (long long)c->prune_set_n[i] - (long long)(c->layers - 1) * c->prune_set_c[i];
      TOME_CHECK(n_last >= 1 && c->prune_set_c[i] <= n_last / 2, TOME_ERR_INVALID,
                 "stack: token set %d (%d tokens) cannot merge %d tokens in each of %d layers (c <= floor(n / 2) at every layer)", i,
                 c->prune_set_n[i], c->prune_set_c[i], c->layers);
      total += c->prune_set_n[i];
    }
    TOME_CHECK(total == c->tokens, TOME_ERR_INVALID, "stack: the token sets hold %lld tokens, the sequence %d", total, c->tokens);
  } else if (c->prune_sets > 0) {
    TOME_CHECK(c->r == 0 && c->prop_attn == 0 && !c->class_token && !c->distill_token, TOME_ERR_INVALID,
               "stack: a pruning stack (prune_sets > 0) takes r = 0, prop_attn = 0 and no class / distill token");
    TOME_CHECK(c->prune_importance == TOME_IMPORTANCE_ROW_MEAN || c->prune_importance == TOME_IMPORTANCE_RECEIVED, TOME_ERR_INVALID,
               "stack: unknown prune_importance %d", c->prune_importance);
    TOME_CHECK(c->head_dim == 64 || c->head_dim == 128 || c->head_dim == 256, TOME_ERR_UNSUPPORTED,
               "stack: pruning stacks need head_dim 64, 128 or 256 (tome_attention_importance)");
    long long total = 0;
    for (int i = 0; i < c->prune_sets; ++i) {
      TOME_CHECK(c->prune_set_n[i] >= 1 && c->prune_set_c[i] >= 0, TOME_ERR_INVALID, "stack: token set %d: n >= 1, c >= 0", i);
      // the grammar's token count at the last layer's input must stay positive and its top_k valid (token_compression.py:31)
      TOME_CHECK((long long)c->prune_set_n[i] - (long long)c->layers * c->prune_set_c[i] >= 0 &&
                 (long long)c->prune_set_n[i] - (long long)(c->layers - 1) * c->prune_set_c[i] >= 1, TOME_ERR_INVALID,
                 "stack: token set %d (%d tokens) cannot drop %d tokens in each of %d layers", i, c->prune_set_n[i],
                 c->prune_set_c[i], c->layers);
      total += c->prune_set_n[i];
    }
    TOME_CHECK(total == c->tokens, TOME_ERR_INVALID, "stack: the token sets hold %lld tokens, the sequence %d", total, c->tokens);
  }
  TOME_CHECK(c->head >= 0 && c->head <= 3, TOME_ERR_INVALID,
             "stack: head must be 0 (synthetic readout MSE), 1 (continuous l2), 2 (categorical cross-entropy) or 3 (diffusion)");
  if (c->head == 3) {
    TOME_CHECK(c->n_readout > 0, TOME_ERR_INVALID, "stack: an action head needs readout tokens");
    tome_diffusion_desc_t d = diffusion_desc(c, 1);
    if (tome_diffusion_head_param_count(&d) < 0) return TOME_ERR_INVALID;  // message set by the head's own check
  } else if (c->head > 0) {
    TOME_CHECK(c->n_readout > 0, TOME_ERR_INVALID, "stack: an action head needs readout tokens");
    tome_head_desc_t h = head_desc(c, 1);
    if (tome_action_head_workspace_bytes(&h) == 0) return TOME_ERR_INVALID;  // message set by the head's own check
  }
  return TOME_OK;
}

// The token sets entering `layer` of a pruning or set-merging stack (token_sequencer.py:236: n - layer * c), each losing c.
static tome_token_sets_t layer_sets(const tome_stack_cfg_t* c, int layer) {
  tome_token_sets_t ts;
  memset(&ts, 0, sizeof(ts));
  ts.n_sets = c->prune_sets;
  for (int i = 0, start = 0; i < c->prune_sets; ++i) {
    ts.set_start[i] = start;
    ts.set_n[i] = c->prune_set_n[i] - layer * c->prune_set_c[i];
    ts.set_r[i] = c->prune_set_c[i];
    start += ts.set_n[i];
  }
  return ts;
}

static bool merges_in_sets(const tome_stack_cfg_t* c) { return c->prune_sets > 0 && c->set_merge; }

static std::vector<LayerShape> layer_shapes(const tome_stack_cfg_t* c) {
  std::vector<LayerShape> s(c->layers);
  int t = c->tokens;
  for (int l = 0; l < c->layers; ++l) {
    s[l].t_in = t;
    s[l].r = tome_clamp_r(t, c->r, c->class_token, c->distill_token);
    if (c->prune_sets > 0) {
      s[l].r = 0;
      for (int i = 0; i < c->prune_sets; ++i) s[l].r += c->prune_set_c[i];
    }
    s[l].t_out = t - s[l].r;
    t = s[l].t_out;
  }
  return s;
}

// One function computes the layout for both the size query (base == nullptr) and the real pointers.
static StackLayout make_layout(const tome_stack_cfg_t* c, void* workspace) {
  StackLayout S;
  S.shapes = layer_shapes(c);
  S.L.resize(c->layers);
  Bump b{reinterpret_cast<uint8_t*>(workspace)};
  const size_t B = c->batch, C = c->channels, HD = (size_t)c->heads * c->head_dim, F = c->mlp_dim, T0 = c->tokens;
  const size_t wide = 3 * HD > F ? 3 * HD : F;
  __nv_bfloat16* x_prev = b.take<__nv_bfloat16>(B * T0 * C);  // x0 = x + pos_embedding
  float* size_prev = nullptr;
  uint8_t* gid_prev = c->num_groups ? b.take<uint8_t>(B * T0) : nullptr;
  int32_t* pos_prev = c->num_groups ? b.take<int32_t>(B * T0) : nullptr;
  for (int l = 0; l < c->layers; ++l) {
    LayerBufs& Lb = S.L[l];
    const size_t T = S.shapes[l].t_in, To = S.shapes[l].t_out, r = S.shapes[l].r;
    // plan arrays: even tokens (node_max, node_idx, edge_idx) and dst_off entries, summed over the token sets when merging in sets
    size_t ta = (T + 1) / 2, n_off = T / 2 + 1;
    if (merges_in_sets(c)) {
      const tome_token_sets_t ts = layer_sets(c, l);
      ta = n_off = 0;
      for (int i = 0; i < ts.n_sets; ++i) {
        ta += (ts.set_n[i] + 1) / 2;
        n_off += ts.set_n[i] / 2 + 1;
      }
    }
    const size_t st_in = c->ln_axis == 1 ? B * C : B * T, st_out = c->ln_axis == 1 ? B * C : B * To;
    Lb.x_in = x_prev;
    Lb.size_in = size_prev;
    Lb.gid_in = gid_prev;
    Lb.pos_in = pos_prev;
    Lb.ln1_mean = b.take<float>(st_in);
    Lb.ln1_rstd = b.take<float>(st_in);
    Lb.h = b.take<__nv_bfloat16>(B * T * C);
    Lb.qkv = b.take<__nv_bfloat16>(B * T * 3 * HD);
    Lb.attn_o = b.take<__nv_bfloat16>(B * T * HD);
    Lb.lse = b.take<float>(B * c->heads * T);
    Lb.x1m = b.take<__nv_bfloat16>(B * To * C);
    memset(&Lb.plan, 0, sizeof(Lb.plan));
    Lb.node_max = nullptr;
    Lb.node_idx = nullptr;
    Lb.importance = nullptr;
    Lb.prune_ids = nullptr;
    if (r > 0 && c->prune_sets > 0 && !c->set_merge) {
      Lb.importance = b.take<float>(B * T);
      Lb.prune_ids = b.take<int32_t>(B * To);
      Lb.plan.row_map = b.take<int32_t>(B * T);
      Lb.size_out = nullptr;
      Lb.gid_out = c->num_groups ? b.take<uint8_t>(B * To) : nullptr;
      Lb.pos_out = c->num_groups ? b.take<int32_t>(B * To) : nullptr;
    } else if (r > 0) {
      Lb.node_max = b.take<float>(B * ta);
      Lb.node_idx = b.take<int32_t>(B * ta);
      Lb.plan.edge_idx = b.take<int32_t>(B * ta);
      Lb.plan.dst_idx = b.take<int32_t>(B * r);
      Lb.plan.row_map = b.take<int32_t>(B * T);
      Lb.plan.dst_off = b.take<int32_t>(B * n_off);
      Lb.plan.dst_src = b.take<int32_t>(B * r);
      Lb.size_out = b.take<float>(B * To);
      Lb.gid_out = c->num_groups ? b.take<uint8_t>(B * To) : nullptr;
      Lb.pos_out = c->num_groups ? b.take<int32_t>(B * To) : nullptr;
    } else {
      Lb.size_out = Lb.size_in;
      Lb.gid_out = Lb.gid_in;
      Lb.pos_out = Lb.pos_in;
    }
    Lb.ln2_mean = b.take<float>(st_out);
    Lb.ln2_rstd = b.take<float>(st_out);
    Lb.h2 = b.take<__nv_bfloat16>(B * To * C);
    Lb.m1 = b.take<__nv_bfloat16>(B * To * F);
    Lb.m1_bits = b.take<uint32_t>(B * To * ((F + 31) / 32));
    Lb.x_out = b.take<__nv_bfloat16>(B * To * C);
    x_prev = Lb.x_out;
    size_prev = Lb.size_out;
    gid_prev = Lb.gid_out;
    pos_prev = Lb.pos_out;
  }
  S.x1_scratch = b.take<__nv_bfloat16>(B * T0 * C);
  S.g0 = b.take<__nv_bfloat16>(B * T0 * C);
  S.g1 = b.take<__nv_bfloat16>(B * T0 * C);
  S.g2 = b.take<__nv_bfloat16>(B * T0 * C);
  S.g3 = b.take<__nv_bfloat16>(B * T0 * HD);
  S.big = b.take<__nv_bfloat16>(B * T0 * wide);
  {  // attention scratch (forward: per-tile metadata; backward: delta + metadata), sized for the widest layer
    tome_attn_desc_t ad;
    memset(&ad, 0, sizeof(ad));
    ad.batch = c->batch; ad.tokens = c->tokens; ad.heads = c->heads; ad.head_dim = c->head_dim;
    ad.dropout_rate = c->attn_dropout_rate;
    const size_t f = tome_attention_workspace_bytes(&ad), bw = tome_attention_bwd_workspace_bytes(&ad);
    S.ws_attn_bytes = f > bw ? f : bw;
    S.ws_attn = b.take<uint8_t>(S.ws_attn_bytes);
  }
  {  // normalised (and, on the tensor-core path, bf16-split) matching metric: tome_sim_argmax's workspace
    tome_metric_desc_t md;
    memset(&md, 0, sizeof(md));
    md.batch = c->batch; md.tokens = c->tokens; md.dim = c->head_dim; md.heads = c->heads; md.dtype = TOME_BF16;
    S.ws_sim_bytes = tome_sim_argmax_workspace_bytes(&md);
  }
  S.ws_sim = b.take<uint8_t>(S.ws_sim_bytes);
  // split-K workspace: the largest weight gradient, at most 64 splits are ever chosen but 148 tiles bound the product
  size_t wmax = C * 3 * HD;
  if (C * F > wmax) wmax = C * F;
  if (HD * C > wmax) wmax = HD * C;
  S.ws_gemm_bytes = wmax * sizeof(float) * 64;
  S.ws_gemm = b.take<float>(wmax * 64);
  S.ws_colsum = b.take<float>(256 * wide);
  {  // rows: 128-row tiles of the flattened [B T0, N] GEMM outputs, or (batch row, 128-token tile) pairs of attention backward
    const size_t r1 = (B * T0 + 127) / 128, r2 = B * ((T0 + 127) / 128);
    S.ws_colpart = b.take<float>((r1 > r2 ? r1 : r2) * wide);
  }
  const size_t ln_rows = c->ln_axis == 1 ? B : 256;
  S.ws_ln = b.take<float>(2 * ln_rows * C);
  S.origin = b.take<int32_t>(B * (c->n_readout > 0 ? c->n_readout : 1));
  S.ws_head_bytes = 0;
  S.ws_head = nullptr;
  if (c->head == 3) {
    tome_diffusion_desc_t d = diffusion_desc(c, 1);
    S.ws_head_bytes = tome_diffusion_head_workspace_bytes(&d);
    S.ws_head = b.take<uint8_t>(S.ws_head_bytes);
  } else if (c->head > 0) {
    tome_head_desc_t h = head_desc(c, 1);
    S.ws_head_bytes = tome_action_head_workspace_bytes(&h);
    S.ws_head = b.take<uint8_t>(S.ws_head_bytes);
  }
  S.total = b.total();
  return S;
}

__global__ void broadcast_groups_kernel(int B, int T, const uint8_t* __restrict__ gid, const int32_t* __restrict__ pos,
                                        uint8_t* __restrict__ gid_out, int32_t* __restrict__ pos_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B * T) {
    gid_out[i] = gid[i % T];
    pos_out[i] = pos[i % T];
  }
}

// Layer l's attention over its packed qkv: forward and backward must describe it identically (the attention-dropout
// mask is regenerated from the seed and site given here).
static tome_attn_desc_t attn_desc(const tome_stack_cfg_t* c, const tome_stack_io_t* io, const LayerBufs& Lb, int T, int l) {
  const int HD = c->heads * c->head_dim;
  tome_attn_desc_t ad;
  memset(&ad, 0, sizeof(ad));
  ad.batch = c->batch; ad.tokens = T; ad.heads = c->heads; ad.head_dim = c->head_dim;
  ad.q_batch_stride = ad.k_batch_stride = ad.v_batch_stride = (long long)T * 3 * HD;
  ad.q_token_stride = ad.k_token_stride = ad.v_token_stride = 3 * HD;
  ad.o_batch_stride = (long long)T * HD; ad.o_token_stride = HD;
  ad.scale = 1.0f / sqrtf((float)c->head_dim);
  if (c->num_groups) { ad.gid = Lb.gid_in; ad.pos = Lb.pos_in; ad.allow = io->allow; ad.num_groups = c->num_groups; }
  ad.size = c->prop_attn ? Lb.size_in : nullptr;
  ad.dropout_rate = c->attn_dropout_rate; ad.dropout_seed = c->dropout_seed; ad.dropout_site = kAttnDropSite + (uint32_t)l;
  return ad;
}

#define RC(expr)                 \
  do {                           \
    int _rc = (expr);            \
    if (_rc != TOME_OK) return _rc; \
  } while (0)

static int gemm(const tome_stack_cfg_t* c, const StackLayout& S, cudaStream_t st, int m, int n, int k, const void* a,
                long long lda, int a_major, const void* b, long long ldb, int b_major, void* out, long long ldc, int c_dtype,
                const float* bias, int relu, const void* residual, const void* gate, float gate_scale, int drop_site,
                int accumulate, const void* gate_bits = nullptr, void* relu_bits_out = nullptr, float* colsum_partial = nullptr) {
  tome_gemm_args_t g;
  memset(&g, 0, sizeof(g));
  g.m = m; g.n = n; g.k = k;
  g.a = a; g.lda = lda; g.a_major = a_major;
  g.b = b; g.ldb = ldb; g.b_major = b_major;
  g.c = out; g.ldc = ldc; g.c_dtype = c_dtype;
  g.bias = bias; g.relu = relu;
  g.residual = residual; g.ldr = n;
  g.gate = gate; g.ldg = n; g.gate_scale = gate_scale;
  g.gate_bits = gate_bits; g.relu_bits_out = relu_bits_out; g.ld_bits = (n + 31) / 32;
  g.colsum_partial = colsum_partial;
  if (drop_site >= 0 && c->dropout_rate > 0.f) {
    g.dropout_rate = c->dropout_rate;
    g.dropout_seed = c->dropout_seed;
    g.dropout_site = (uint32_t)drop_site;
  }
  g.k_splits = 0;
  g.accumulate = accumulate;
  return tome_gemm_bf16(&g, S.ws_gemm, S.ws_gemm_bytes, st);
}

}  // namespace tome

using namespace tome;

// the action head's Dense kernel [C, features] and bias [features] follow the last layer (so they ride in the last
// layer's all-reduce bucket: their gradients are the first to become final)
static long long head_param_count(const tome_stack_cfg_t* c) {
  if (c->head == 3) {
    tome_diffusion_desc_t d = diffusion_desc(c, 1);
    return tome_diffusion_head_param_count(&d);
  }
  return c->head > 0 ? (long long)c->channels * c->head_features + c->head_features : 0;
}
extern "C" long long tome_stack_param_count(const tome_stack_cfg_t* c) {
  if (check_cfg(c)) return -1;
  return layer_offsets(c, c->layers).ln1_scale + head_param_count(c);
}
extern "C" long long tome_stack_head_offset(const tome_stack_cfg_t* c) {
  if (check_cfg(c) || c->head == 0) return -1;
  return layer_offsets(c, c->layers).ln1_scale;
}
extern "C" long long tome_stack_layer_offset(const tome_stack_cfg_t* c, int layer) {
  if (check_cfg(c) || layer < 0 || layer > c->layers) return -1;
  return layer_offsets(c, layer).ln1_scale;
}
extern "C" size_t tome_stack_workspace_bytes(const tome_stack_cfg_t* c) {
  if (check_cfg(c)) return 0;
  return make_layout(c, nullptr).total;
}
extern "C" int tome_stack_tokens_at(const tome_stack_cfg_t* c, int layer) {
  if (check_cfg(c) || layer < 0 || layer > c->layers) return -1;
  auto s = layer_shapes(c);
  return layer == c->layers ? s.back().t_out : s[layer].t_in;
}

static int check_io(const tome_stack_cfg_t* c, const tome_stack_io_t* io, const StackLayout& S, bool backward) {
  TOME_CHECK(io != nullptr, TOME_ERR_INVALID, "stack: null io");
  TOME_CHECK(io->params_f32 && io->params_bf16 && io->x && io->workspace, TOME_ERR_INVALID, "stack: null params / x / workspace");
  TOME_CHECK(io->workspace_bytes >= S.total, TOME_ERR_INVALID, "stack: workspace too small (%zu < %zu)", io->workspace_bytes, S.total);
  TOME_CHECK(((uintptr_t)io->workspace & 255) == 0, TOME_ERR_INVALID, "stack: workspace must be 256-byte aligned");
  TOME_CHECK(c->num_groups == 0 || (((io->gid && io->pos) || (io->layer_gid && io->layer_pos)) && io->allow), TOME_ERR_INVALID,
             "stack: a group mask needs gid, pos (or layer_gid, layer_pos) and allow");
  TOME_CHECK(!(io->layer_gid || io->layer_pos) || (c->prune_sets > 0 && c->num_groups > 0 && io->layer_gid && io->layer_pos), TOME_ERR_INVALID,
             "stack: layer_gid / layer_pos are the per-layer masks of a pruning stack with a group mask (both or neither)");
  TOME_CHECK(!(c->set_merge && (io->layer_gid || io->layer_pos)), TOME_ERR_INVALID,
             "stack: a set-merging stack carries gid / pos through its merges and takes no layer_gid / layer_pos");
  TOME_CHECK(c->n_readout == 0 || io->readout_idx, TOME_ERR_INVALID, "stack: readout_idx missing");
  if (backward) TOME_CHECK(io->grads_f32 && io->target && io->loss && c->n_readout > 0, TOME_ERR_INVALID,
                           "stack_backward: needs grads_f32, target, loss and n_readout > 0");
  return TOME_OK;
}

extern "C" int tome_stack_forward(const tome_stack_cfg_t* c, const tome_stack_io_t* io, void* stream_) {
  clear_error();
  cudaStream_t st = (cudaStream_t)stream_;
  RC(check_cfg(c));
  StackLayout S = make_layout(c, io ? io->workspace : nullptr);
  RC(check_io(c, io, S, false));
  const int B = c->batch, C = c->channels, H = c->heads, D = c->head_dim, HD = H * D, F = c->mlp_dim;
  const float* pf = io->params_f32;
  const __nv_bfloat16* pw = reinterpret_cast<const __nv_bfloat16*>(io->params_bf16);

  RC(tome_add_pos_embedding(B, c->tokens, C, io->x, io->x_dtype, pf, S.L[0].x_in, st));
  if (c->num_groups) {
    const int n = B * c->tokens;
    ProfScope prof(PROF_OTHER, 0.0, 1, st);
    launch_k(broadcast_groups_kernel, ceil_div(n, 256), 256, 0, st, B, c->tokens, io->layer_gid ? io->layer_gid : io->gid,
             io->layer_pos ? io->layer_pos : io->pos, S.L[0].gid_in, S.L[0].pos_in);
    TOME_CUDA(cudaGetLastError());
  }
  long long grammar_off = 0;   // pruning stacks with per-layer grammar masks: offset of the NEXT layer's rows in layer_gid / layer_pos
  for (int l = 0; l < c->layers; ++l) {
    const LayerBufs& Lb = S.L[l];
    const ParamOffsets o = layer_offsets(c, l);
    const int T = S.shapes[l].t_in, r = S.shapes[l].r, To = S.shapes[l].t_out;
    const int M = B * T, Mo = B * To;
    RC(tome_layernorm_fwd(B, T, C, c->ln_axis, c->ln_eps, Lb.x_in, pf + o.ln1_scale, pf + o.ln1_bias, Lb.h, Lb.ln1_mean,
                          Lb.ln1_rstd, st));
    RC(gemm(c, S, st, M, 3 * HD, C, Lb.h, C, TOME_MAJOR_K, pw + o.wqkv, 3 * HD, TOME_MAJOR_MN, Lb.qkv, 3 * HD, TOME_BF16,
            pf + o.bqkv, 0, nullptr, nullptr, 1.f, -1, 0));
    const tome_attn_desc_t ad = attn_desc(c, io, Lb, T, l);
    RC(tome_attention_fwd(&ad, Lb.qkv, Lb.qkv + HD, Lb.qkv + 2 * HD, Lb.attn_o, Lb.lse, S.ws_attn, S.ws_attn_bytes, st));
    __nv_bfloat16* x1 = r > 0 ? S.x1_scratch : Lb.x1m;
    RC(gemm(c, S, st, M, C, HD, Lb.attn_o, HD, TOME_MAJOR_K, pw + o.wo, C, TOME_MAJOR_MN, x1, C, TOME_BF16, pf + o.bo, 0,
            Lb.x_in, nullptr, 1.f, 3 * l + 0, 0));
    grammar_off += T;
    if (r > 0 && c->prune_sets > 0 && !c->set_merge) {
      // importance from this layer's attention weights, per-set top-k, gather (compressed_attention.py:303-308)
      RC(tome_attention_importance(&ad, Lb.qkv, Lb.qkv + HD, Lb.lse, c->prune_importance, Lb.importance, st));
      tome_prune_desc_t pd;
      memset(&pd, 0, sizeof(pd));
      pd.batch = B; pd.tokens = T; pd.channels = C; pd.dtype = TOME_BF16; pd.n_sets = c->prune_sets; pd.score_planes = 1;
      const tome_token_sets_t ts = layer_sets(c, l);
      for (int i = 0; i < c->prune_sets; ++i) {
        pd.set_start[i] = ts.set_start[i];
        pd.set_n[i] = ts.set_n[i];
        pd.set_k[i] = ts.set_n[i] - ts.set_r[i];
      }
      RC(tome_topk_prune(&pd, x1, Lb.importance, Lb.x1m, Lb.prune_ids, st));
      const bool grammar = io->layer_gid != nullptr && c->num_groups > 0;
      RC(tome_prune_row_map(B, T, To, Lb.prune_ids, Lb.gid_in, Lb.pos_in, Lb.plan.row_map, grammar ? nullptr : Lb.gid_out,
                            grammar ? nullptr : Lb.pos_out, st));
      if (grammar && l + 1 < c->layers) {   // masks[layer + 1] of the compression grammar, the same for every batch row
        ProfScope prof(PROF_OTHER, 0.0, 1, st);
        launch_k(broadcast_groups_kernel, ceil_div(B * To, 256), 256, 0, st, B, To, io->layer_gid + grammar_off,
                 io->layer_pos + grammar_off, Lb.gid_out, Lb.pos_out);
        TOME_CUDA(cudaGetLastError());
      }
    } else if (r > 0) {
      // merging: over the whole sequence, or inside each token set (the sets of a set-merging stack)
      const tome_token_sets_t ts = merges_in_sets(c) ? layer_sets(c, l) : tome_token_sets_t{};
      const tome_token_sets_t* sets = merges_in_sets(c) ? &ts : nullptr;
      tome_metric_desc_t md;
      memset(&md, 0, sizeof(md));
      md.batch = B; md.tokens = T; md.dim = D; md.heads = H; md.dtype = TOME_BF16;
      md.batch_stride = (long long)T * 3 * HD; md.token_stride = 3 * HD; md.head_stride = D;
      md.class_token = c->class_token; md.distill_token = c->distill_token; md.sets = sets;
      RC(tome_sim_argmax(&md, Lb.qkv + HD, Lb.node_max, Lb.node_idx, nullptr, S.ws_sim, S.ws_sim_bytes, st));
      tome_plan_shape_t ps{B, T, r, c->distill_token, sets};
      RC(tome_select_topr(&ps, Lb.node_max, Lb.node_idx, &Lb.plan, st));
      tome_merge_shape_t ms{B, T, C, r, c->distill_token, TOME_BF16, TOME_MERGE_WAVG, sets};
      RC(tome_merge_fwd(&ms, &Lb.plan, x1, Lb.size_in, Lb.x1m, Lb.size_out, Lb.gid_in, Lb.pos_in, Lb.gid_out, Lb.pos_out, st));
    }
    RC(tome_layernorm_fwd(B, To, C, c->ln_axis, c->ln_eps, Lb.x1m, pf + o.ln2_scale, pf + o.ln2_bias, Lb.h2, Lb.ln2_mean,
                          Lb.ln2_rstd, st));
    RC(gemm(c, S, st, Mo, F, C, Lb.h2, C, TOME_MAJOR_K, pw + o.w1, F, TOME_MAJOR_MN, Lb.m1, F, TOME_BF16, pf + o.b1, 1, nullptr,
            nullptr, 1.f, 3 * l + 1, 0, nullptr, Lb.m1_bits));
    RC(gemm(c, S, st, Mo, C, F, Lb.m1, F, TOME_MAJOR_K, pw + o.w2, C, TOME_MAJOR_MN, Lb.x_out, C, TOME_BF16, pf + o.b2, 0, Lb.x1m,
            nullptr, 1.f, 3 * l + 2, 0));
  }
  const int TL = S.shapes.back().t_out;
  if (io->x_final)
    TOME_CUDA(cudaMemcpyAsync(io->x_final, S.L.back().x_out, (size_t)B * TL * C * 2, cudaMemcpyDeviceToDevice, st));
  if (c->n_readout > 0) {
    const int32_t* maps[64];
    int toks[64];
    for (int l = 0; l < c->layers; ++l) {
      maps[l] = S.shapes[l].r > 0 ? S.L[l].plan.row_map : nullptr;   // merge and prune layers both leave token -> output row
      toks[l] = S.shapes[l].t_in;
    }
    RC(tome_chain_row_maps(B, c->layers, maps, toks, io->readout_idx, c->n_readout, S.origin, st));
    if (c->head == 3) {
      // diffusion head: denoise_loss on the pooled readout rows (diffusion.py:94-143); target = [actions | noise]
      tome_diffusion_desc_t d = diffusion_desc(c, TL);
      const long long ho = layer_offsets(c, c->layers).ln1_scale;
      TOME_CHECK(io->head_out && io->target && io->loss && io->head_time && io->head_alpha_hats, TOME_ERR_INVALID,
                 "stack: the diffusion head needs head_out, target ([B, 2A] = actions | noise), loss, head_time and head_alpha_hats");
      RC(tome_diffusion_head_fwd(&d, io->params_f32 + ho, reinterpret_cast<const __nv_bfloat16*>(io->params_bf16) + ho,
                                 S.L.back().x_out, S.origin, io->target, io->target + (size_t)B * c->head_features, io->head_time,
                                 io->head_alpha_hats, io->head_out, io->loss, S.ws_head, S.ws_head_bytes, st));
      if (io->readout) RC(tome_readout_mse(B, TL, C, c->n_readout, S.L.back().x_out, S.origin, nullptr, nullptr, nullptr, io->readout, st));
    } else if (c->head > 0) {
      // action head on the pooled readout rows + its loss (continuous.py / categorical.py, octo.py:157-190)
      tome_head_desc_t h = head_desc(c, TL);
      const long long ho = layer_offsets(c, c->layers).ln1_scale;
      const bool with_loss = io->target && io->loss;
      TOME_CHECK(io->head_out, TOME_ERR_INVALID, "stack: head_out missing");
      RC(tome_action_head_fwd(&h, S.L.back().x_out, S.origin, io->params_f32 + ho, io->params_f32 + ho + (long long)C * c->head_features,
                              with_loss ? io->target : nullptr, io->head_out, with_loss ? io->loss : nullptr, S.ws_head,
                              S.ws_head_bytes, st));
      if (io->readout) RC(tome_readout_mse(B, TL, C, c->n_readout, S.L.back().x_out, S.origin, nullptr, nullptr, nullptr, io->readout, st));
    } else if (io->readout || (io->target && io->loss))
      RC(tome_readout_mse(B, TL, C, c->n_readout, S.L.back().x_out, S.origin, (io->target && io->loss) ? io->target : nullptr,
                          (io->target && io->loss) ? io->loss : nullptr, nullptr, io->readout, st));
  }
  return TOME_OK;
}

extern "C" int tome_stack_backward(const tome_stack_cfg_t* c, const tome_stack_io_t* io, void* stream_) {
  clear_error();
  cudaStream_t st = (cudaStream_t)stream_;
  RC(check_cfg(c));
  StackLayout S = make_layout(c, io ? io->workspace : nullptr);
  RC(check_io(c, io, S, true));
  const int B = c->batch, C = c->channels, H = c->heads, D = c->head_dim, HD = H * D, F = c->mlp_dim;
  const float* pf = io->params_f32;
  const __nv_bfloat16* pw = reinterpret_cast<const __nv_bfloat16*>(io->params_bf16);
  float* gr = io->grads_f32;
  const bool drop = c->dropout_rate > 0.f;
  const float inv_keep = drop ? make_dropout(c->dropout_rate, c->dropout_seed, 0).inv_keep : 1.0f;
  const int TL = S.shapes.back().t_out;

  __nv_bfloat16 *g0 = S.g0, *g1 = S.g1, *g2 = S.g2, *g3 = S.g3;
  // dL/dx_final from the readout rows: through the action head (pooled / dL/dz saved by forward), or the synthetic MSE
  // (which recomputes the loss value, harmless)
  if (c->head == 3) {
    tome_diffusion_desc_t d = diffusion_desc(c, TL);
    const long long ho = layer_offsets(c, c->layers).ln1_scale;
    TOME_CHECK(io->head_time, TOME_ERR_INVALID, "stack_backward: head_time missing");
    RC(tome_diffusion_head_bwd(&d, pf + ho, pw + ho, S.origin, io->head_time, S.ws_head, gr + ho, g0, st));
  } else if (c->head > 0) {
    tome_head_desc_t h = head_desc(c, TL);
    const long long ho = layer_offsets(c, c->layers).ln1_scale;
    RC(tome_action_head_bwd(&h, S.origin, pf + ho, S.ws_head, gr + ho, gr + ho + (long long)C * c->head_features, g0, st));
  } else {
    RC(tome_readout_mse(B, TL, C, c->n_readout, S.L.back().x_out, S.origin, io->target, io->loss, g0, nullptr, st));
  }

  // dy_eff = dropout mask applied to an incoming gradient + its column sums (the Dense bias gradient), one pass
  auto masked_colsum = [&](const __nv_bfloat16* src, __nv_bfloat16* dst, int rows, int ncols, int site, float* dbias,
                           const __nv_bfloat16** out) -> int {
    if (!drop) {
      *out = src;
      return tome_colsum_bf16(rows, ncols, src, ncols, dbias, 1, S.ws_colsum, st);
    }
    *out = dst;
    return tome_dropout_colsum_bf16(rows, ncols, src, dst, c->dropout_rate, c->dropout_seed, (uint32_t)site, dbias, 1,
                                    S.ws_colsum, st);
  };

  for (int l = c->layers - 1; l >= 0; --l) {
    const LayerBufs& Lb = S.L[l];
    const ParamOffsets o = layer_offsets(c, l);
    const int T = S.shapes[l].t_in, r = S.shapes[l].r, To = S.shapes[l].t_out;
    const int M = B * T, Mo = B * To;
    if (io->grad_trace)  // parity aid: the gradient this layer receives, before it is consumed
      TOME_CUDA(cudaMemcpyAsync(reinterpret_cast<__nv_bfloat16*>(io->grad_trace) + (size_t)l * B * c->tokens * C, g0,
                                (size_t)Mo * C * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice, st));
    // ---- MLP: y = x1m + drop2(m1 W2 + b2),  m1 = drop1(relu(h2 W1 + b1))          d_out in g0
    const __nv_bfloat16* dy2;
    RC(masked_colsum(g0, g2, Mo, C, 3 * l + 2, gr + o.b2, &dy2));
    RC(gemm(c, S, st, F, C, Mo, Lb.m1, F, TOME_MAJOR_MN, dy2, C, TOME_MAJOR_MN, gr + o.w2, C, TOME_F32, nullptr, 0, nullptr,
            nullptr, 1.f, -1, 1));
    RC(gemm(c, S, st, Mo, F, C, dy2, C, TOME_MAJOR_K, pw + o.w2, C, TOME_MAJOR_K, S.big, F, TOME_BF16, nullptr, 0, nullptr, nullptr,
            inv_keep, -1, 0, Lb.m1_bits, nullptr, S.ws_colpart));  // dm1 (pre-activation): the relu and dropout masks are the bits
    // MLP-1 forward wrote; the same epilogue leaves dm1's column sums per 128-row tile (no second pass over the 400 MB)
    RC(tome_reduce_rows_f32((Mo + 127) / 128, F, S.ws_colpart, gr + o.b1, 1, st));
    RC(gemm(c, S, st, C, F, Mo, Lb.h2, C, TOME_MAJOR_MN, S.big, F, TOME_MAJOR_MN, gr + o.w1, F, TOME_F32, nullptr, 0, nullptr,
            nullptr, 1.f, -1, 1));
    RC(gemm(c, S, st, Mo, C, F, S.big, F, TOME_MAJOR_K, pw + o.w1, F, TOME_MAJOR_K, g1, C, TOME_BF16, nullptr, 0, nullptr, nullptr,
            1.f, -1, 0));  // dh2
    // ---- LN2 (+ residual gradient d_out) -> dx1m in g2
    RC(tome_layernorm_bwd(B, To, C, c->ln_axis, Lb.x1m, g1, pf + o.ln2_scale, Lb.ln2_mean, Lb.ln2_rstd, g0, g2,
                          gr + o.ln2_scale, gr + o.ln2_bias, S.ws_ln, st));
    // ---- merge backward -> dx1 in g0
    const __nv_bfloat16* dx1;
    if (r > 0 && c->prune_sets > 0 && !c->set_merge) {
      RC(tome_prune_bwd(B, T, To, C, TOME_BF16, Lb.plan.row_map, g2, g0, st));
      dx1 = g0;
    } else if (r > 0) {
      // the global row map: the same backward with or without token sets
      const tome_token_sets_t ts = merges_in_sets(c) ? layer_sets(c, l) : tome_token_sets_t{};
      tome_merge_shape_t ms{B, T, C, r, c->distill_token, TOME_BF16, TOME_MERGE_WAVG, merges_in_sets(c) ? &ts : nullptr};
      RC(tome_merge_bwd(&ms, &Lb.plan, Lb.size_in, Lb.size_out, g2, g0, st));
      dx1 = g0;
    } else {
      dx1 = g2;
      __nv_bfloat16* t = g0; g0 = g2; g2 = t;  // keep "dx1 lives in g0"
    }
    // ---- out projection: x1 = x + drop0(o Wo + bo)
    const __nv_bfloat16* dyo;
    RC(masked_colsum(dx1, g1, M, C, 3 * l + 0, gr + o.bo, &dyo));
    RC(gemm(c, S, st, HD, C, M, Lb.attn_o, HD, TOME_MAJOR_MN, dyo, C, TOME_MAJOR_MN, gr + o.wo, C, TOME_F32, nullptr, 0, nullptr,
            nullptr, 1.f, -1, 1));
    RC(gemm(c, S, st, M, HD, C, dyo, C, TOME_MAJOR_K, pw + o.wo, C, TOME_MAJOR_K, g3, HD, TOME_BF16, nullptr, 0, nullptr, nullptr,
            1.f, -1, 0));  // d attn_o
    // ---- attention backward -> dqkv in big
    const tome_attn_desc_t ad = attn_desc(c, io, Lb, T, l);
    tome_attn_grad_strides_t gs;
    memset(&gs, 0, sizeof(gs));
    gs.dq_batch_stride = gs.dk_batch_stride = gs.dv_batch_stride = (long long)T * 3 * HD;
    gs.dq_token_stride = gs.dk_token_stride = gs.dv_token_stride = 3 * HD;
    gs.do_batch_stride = (long long)T * HD; gs.do_token_stride = HD;
    const bool fused_bias = D == 64;   // the tcgen05 kernels leave dqkv's column sums per 128-token tile
    gs.bias_partial = fused_bias ? S.ws_colpart : nullptr;
    gs.bias_partial_ld = 3 * HD; gs.bias_q_col = 0; gs.bias_k_col = HD; gs.bias_v_col = 2 * HD;
    RC(tome_attention_bwd(&ad, &gs, Lb.qkv, Lb.qkv + HD, Lb.qkv + 2 * HD, Lb.attn_o, Lb.lse, g3, S.big, S.big + HD,
                          S.big + 2 * HD, S.ws_attn, S.ws_attn_bytes, st));
    // ---- qkv projection
    if (fused_bias) RC(tome_reduce_rows_f32(B * ((T + 127) / 128), 3 * HD, S.ws_colpart, gr + o.bqkv, 1, st));
    else RC(tome_colsum_bf16(M, 3 * HD, S.big, 3 * HD, gr + o.bqkv, 1, S.ws_colsum, st));
    RC(gemm(c, S, st, C, 3 * HD, M, Lb.h, C, TOME_MAJOR_MN, S.big, 3 * HD, TOME_MAJOR_MN, gr + o.wqkv, 3 * HD, TOME_F32, nullptr, 0,
            nullptr, nullptr, 1.f, -1, 1));
    RC(gemm(c, S, st, M, C, 3 * HD, S.big, 3 * HD, TOME_MAJOR_K, pw + o.wqkv, 3 * HD, TOME_MAJOR_K, g1, C, TOME_BF16, nullptr, 0,
            nullptr, nullptr, 1.f, -1, 0));  // dh
    // ---- LN1 (+ residual gradient dx1) -> dx_in in g2, which becomes the next d_out (g0)
    RC(tome_layernorm_bwd(B, T, C, c->ln_axis, Lb.x_in, g1, pf + o.ln1_scale, Lb.ln1_mean, Lb.ln1_rstd, dx1, g2,
                          gr + o.ln1_scale, gr + o.ln1_bias, S.ws_ln, st));
    {
      __nv_bfloat16* t = g0; g0 = g2; g2 = t;
    }
    if (l == 0) RC(tome_pos_embedding_bwd(B, c->tokens, C, g0, gr, st));
    if (io->layer_done_events && io->layer_done_events[l])
      TOME_CUDA(cudaEventRecord((cudaEvent_t)io->layer_done_events[l], st));
  }
  if (io->layer_done_events && io->layer_done_events[c->layers])
    TOME_CUDA(cudaEventRecord((cudaEvent_t)io->layer_done_events[c->layers], st));
  return TOME_OK;
}

#define ACCESSOR(name, type, expr)                                                             \
  extern "C" type name(const tome_stack_cfg_t* c, const tome_stack_io_t* io, int layer) {      \
    if (check_cfg(c) || !io || layer < 0 || layer >= c->layers) return nullptr;                \
    StackLayout S = make_layout(c, io->workspace);                                             \
    return expr;                                                                               \
  }
ACCESSOR(tome_stack_layer_edge_idx, const int32_t*, S.L[layer].plan.edge_idx)
ACCESSOR(tome_stack_layer_dst_idx, const int32_t*, S.L[layer].plan.dst_idx)
ACCESSOR(tome_stack_layer_node_max, const float*, S.L[layer].node_max)
ACCESSOR(tome_stack_layer_node_idx, const int32_t*, S.L[layer].node_idx)
ACCESSOR(tome_stack_layer_relu_bits, const uint32_t*, S.L[layer].m1_bits)
ACCESSOR(tome_stack_layer_importance, const float*, S.L[layer].importance)
ACCESSOR(tome_stack_layer_prune_ids, const int32_t*, S.L[layer].prune_ids)

extern "C" const void* tome_stack_layer_x_in(const tome_stack_cfg_t* c, const tome_stack_io_t* io, int layer) {
  if (check_cfg(c) || !io || layer < 0 || layer > c->layers) return nullptr;
  StackLayout S = make_layout(c, io->workspace);
  return layer == c->layers ? S.L.back().x_out : S.L[layer].x_in;
}
extern "C" const float* tome_stack_layer_size_in(const tome_stack_cfg_t* c, const tome_stack_io_t* io, int layer) {
  if (check_cfg(c) || !io || layer < 0 || layer > c->layers) return nullptr;
  StackLayout S = make_layout(c, io->workspace);
  return layer == c->layers ? S.L.back().size_out : S.L[layer].size_in;
}
extern "C" const void* tome_stack_final_x(const tome_stack_cfg_t* c, const tome_stack_io_t* io) {
  if (check_cfg(c) || !io) return nullptr;
  return make_layout(c, io->workspace).L.back().x_out;
}
extern "C" const float* tome_stack_final_size(const tome_stack_cfg_t* c, const tome_stack_io_t* io) {
  if (check_cfg(c) || !io) return nullptr;
  return make_layout(c, io->workspace).L.back().size_out;
}
