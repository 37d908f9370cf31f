// Attention for head dimensions the tcgen05 kernels are not built for (they are specialised for D = 64, the octo-small /
// octo-base head size).  The only shape the reference itself defines -- vanilla_decoder.yaml: 3 heads x 256 over 74 tokens --
// has D = 256, so this path exists to run THAT configuration with the same semantics (group-table mask, log(size) bias,
// attention-weight dropout, lse), not to be fast: fp32 CUDA-core arithmetic, one warp per query row (forward, dQ) or per
// key row (dK/dV), lanes splitting the head dimension, online softmax per row.  Cost is O(T * D) per row per pass, which
// at the literal config (8 x 3 x 74 rows) is microseconds.  Same entry points, same results contract; chosen by head_dim.
#include <float.h>

#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int AG_MAXD = 256;          // head_dim <= 256, multiple of 8
constexpr int AG_PER_LANE = AG_MAXD / 32;
constexpr int AG_WARPS = 4;

struct AttnGenericParams {
  int batch, tokens, heads, dim;
  float scale, scale_log2;
  const uint8_t* gid; const int32_t* pos; const uint8_t* allow; int num_groups;
  const float* size;
  DropoutCfg drop;  // thresh16 == 0: no dropout
  const __nv_bfloat16 *q, *k, *v;
  long long q_bs, q_ts, k_bs, k_ts, v_bs, v_ts;
  __nv_bfloat16* out; long long o_bs, o_ts;
  float* lse;  // [B,H,T] natural log
  // backward
  const __nv_bfloat16 *o_in, *dout; long long do_bs, do_ts;
  __nv_bfloat16 *dq, *dk, *dv; long long dq_bs, dq_ts, dk_bs, dk_ts, dv_bs, dv_ts;
};

__device__ __forceinline__ bool ag_visible(const AttnGenericParams& p, int gq, int pq, int b, int kk) {
  if (p.gid == nullptr) return true;
  const int a = p.allow[gq * p.num_groups + p.gid[(long long)b * p.tokens + kk]];
  return a == 1 || (a == 2 && p.pos[(long long)b * p.tokens + kk] <= pq);
}

// keep bit of attention-weight dropout for (q, k): element k % 32 of stream (q, k / 32); `st` is advanced along k
__device__ __forceinline__ bool ag_keep(const AttnGenericParams& p, DropStream& st, int q, int kk) {
  if (p.drop.thresh16 == 0) return true;
  if ((kk & 31) == 0) st = drop_stream(p.drop, (uint32_t)q, (uint32_t)kk >> 5);
  return st.next() >= (p.drop.thresh16 << 16);
}

// ------------------------------------------------------------------------------------------------ forward: warp = query row
__global__ void __launch_bounds__(AG_WARPS * 32)
attn_generic_fwd_kernel(const AttnGenericParams p) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * AG_WARPS + (threadIdx.x >> 5), h = blockIdx.y, b = blockIdx.z;
  if (q >= p.tokens) return;
  const int T = p.tokens, D = p.dim;
  float qv[AG_PER_LANE], acc[AG_PER_LANE];
  const __nv_bfloat16* qr = p.q + b * p.q_bs + q * p.q_ts + (long long)h * D;
#pragma unroll
  for (int i = 0; i < AG_PER_LANE; ++i) {
    const int d = lane + 32 * i;
    qv[i] = d < D ? __bfloat162float(qr[d]) : 0.f;
    acc[i] = 0.f;
  }
  int gq = 0, pq = 0;
  if (p.gid) { gq = p.gid[(long long)b * T + q]; pq = p.pos[(long long)b * T + q]; }
  float m = -INFINITY, l = 0.f;
  DropStream st{0u, 1u};
  for (int kk = 0; kk < T; ++kk) {
    const __nv_bfloat16* kr = p.k + b * p.k_bs + kk * p.k_ts + (long long)h * D;
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < AG_PER_LANE; ++i) {
      const int d = lane + 32 * i;
      if (d < D) dot = fmaf(qv[i], __bfloat162float(kr[d]), dot);
    }
    dot = warp_sum(dot);
    float s2 = fmaf(dot, p.scale_log2, p.size ? log2f(p.size[(long long)b * T + kk]) : 0.f);
    if (!ag_visible(p, gq, pq, b, kk)) s2 = -FLT_MAX;   // finite, like flax's finfo.min: a fully masked row is uniform
    const bool keep = ag_keep(p, st, q, kk);
    const float m_new = fmaxf(m, s2);
    const float alpha = fast_exp2(m - m_new), pe = fast_exp2(s2 - m_new);
    l = fmaf(l, alpha, pe);                                // the row sum is that of the undropped weights
    const float pw = keep ? pe : 0.f;
    const __nv_bfloat16* vr = p.v + b * p.v_bs + kk * p.v_ts + (long long)h * D;
#pragma unroll
    for (int i = 0; i < AG_PER_LANE; ++i) {
      const int d = lane + 32 * i;
      if (d < D) acc[i] = fmaf(acc[i], alpha, pw * __bfloat162float(vr[d]));
    }
    m = m_new;
  }
  const float inv = p.drop.inv_keep / l;
  __nv_bfloat16* orow = p.out + b * p.o_bs + q * p.o_ts + (long long)h * D;
#pragma unroll
  for (int i = 0; i < AG_PER_LANE; ++i) {
    const int d = lane + 32 * i;
    if (d < D) orow[d] = __float2bfloat16(acc[i] * inv);
  }
  if (lane == 0 && p.lse) p.lse[((long long)b * p.heads + h) * T + q] = (m + log2f(l)) * 0.6931471805599453f;
}

// ------------------------------------------------------------------------------------------------ dQ: warp = query row
__global__ void __launch_bounds__(AG_WARPS * 32)
attn_generic_dq_kernel(const AttnGenericParams p) {
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * AG_WARPS + (threadIdx.x >> 5), h = blockIdx.y, b = blockIdx.z;
  if (q >= p.tokens) return;
  const int T = p.tokens, D = p.dim;
  float qv[AG_PER_LANE], dov[AG_PER_LANE], acc[AG_PER_LANE];
  const __nv_bfloat16* qr = p.q + b * p.q_bs + q * p.q_ts + (long long)h * D;
  const __nv_bfloat16* dor = p.dout + b * p.do_bs + q * p.do_ts + (long long)h * D;
  const __nv_bfloat16* orow = p.o_in + b * p.o_bs + q * p.o_ts + (long long)h * D;
  float delta = 0.f;
#pragma unroll
  for (int i = 0; i < AG_PER_LANE; ++i) {
    const int d = lane + 32 * i;
    qv[i] = d < D ? __bfloat162float(qr[d]) : 0.f;
    dov[i] = d < D ? __bfloat162float(dor[d]) : 0.f;
    if (d < D) delta = fmaf(dov[i], __bfloat162float(orow[d]), delta);
    acc[i] = 0.f;
  }
  delta = warp_sum(delta);
  const float lse2 = p.lse[((long long)b * p.heads + h) * T + q] * 1.4426950408889634f;
  int gq = 0, pq = 0;
  if (p.gid) { gq = p.gid[(long long)b * T + q]; pq = p.pos[(long long)b * T + q]; }
  DropStream st{0u, 1u};
  for (int kk = 0; kk < T; ++kk) {
    const __nv_bfloat16* kr = p.k + b * p.k_bs + kk * p.k_ts + (long long)h * D;
    const __nv_bfloat16* vr = p.v + b * p.v_bs + kk * p.v_ts + (long long)h * D;
    float dot = 0.f, dp = 0.f;
#pragma unroll
    for (int i = 0; i < AG_PER_LANE; ++i) {
      const int d = lane + 32 * i;
      if (d < D) {
        dot = fmaf(qv[i], __bfloat162float(kr[d]), dot);
        dp = fmaf(dov[i], __bfloat162float(vr[d]), dp);
      }
    }
    dot = warp_sum(dot);
    dp = warp_sum(dp);
    const bool keep = ag_keep(p, st, q, kk);
    const bool vis = ag_visible(p, gq, pq, b, kk);
    const float s2 = fmaf(dot, p.scale_log2, p.size ? log2f(p.size[(long long)b * T + kk]) : 0.f);
    const float pe = vis ? fast_exp2(s2 - lse2) : 0.f;
    const float dpd = keep ? dp * p.drop.inv_keep : 0.f;
    const float ds = pe * (dpd - delta) * p.scale;
#pragma unroll
    for (int i = 0; i < AG_PER_LANE; ++i) {
      const int d = lane + 32 * i;
      if (d < D) acc[i] = fmaf(ds, __bfloat162float(kr[d]), acc[i]);
    }
  }
  __nv_bfloat16* dqr = p.dq + b * p.dq_bs + q * p.dq_ts + (long long)h * D;
#pragma unroll
  for (int i = 0; i < AG_PER_LANE; ++i) {
    const int d = lane + 32 * i;
    if (d < D) dqr[d] = __float2bfloat16(acc[i]);
  }
}

// ------------------------------------------------------------------------------------------------ dK / dV: warp = key row
__global__ void __launch_bounds__(AG_WARPS * 32)
attn_generic_dkdv_kernel(const AttnGenericParams p) {
  const int lane = threadIdx.x & 31;
  const int kk = blockIdx.x * AG_WARPS + (threadIdx.x >> 5), h = blockIdx.y, b = blockIdx.z;
  if (kk >= p.tokens) return;
  const int T = p.tokens, D = p.dim;
  float kv[AG_PER_LANE], vv[AG_PER_LANE], dk[AG_PER_LANE], dv[AG_PER_LANE];
  const __nv_bfloat16* kr = p.k + b * p.k_bs + kk * p.k_ts + (long long)h * D;
  const __nv_bfloat16* vr = p.v + b * p.v_bs + kk * p.v_ts + (long long)h * D;
#pragma unroll
  for (int i = 0; i < AG_PER_LANE; ++i) {
    const int d = lane + 32 * i;
    kv[i] = d < D ? __bfloat162float(kr[d]) : 0.f;
    vv[i] = d < D ? __bfloat162float(vr[d]) : 0.f;
    dk[i] = dv[i] = 0.f;
  }
  const float bias2 = p.size ? log2f(p.size[(long long)b * T + kk]) : 0.f;
  const uint32_t thr = p.drop.thresh16 << 16;
  for (int q = 0; q < T; ++q) {
    const __nv_bfloat16* qr = p.q + b * p.q_bs + q * p.q_ts + (long long)h * D;
    const __nv_bfloat16* dor = p.dout + b * p.do_bs + q * p.do_ts + (long long)h * D;
    const __nv_bfloat16* orow = p.o_in + b * p.o_bs + q * p.o_ts + (long long)h * D;
    float qv[AG_PER_LANE], dov[AG_PER_LANE];
    float dot = 0.f, dp = 0.f, delta = 0.f;
#pragma unroll
    for (int i = 0; i < AG_PER_LANE; ++i) {
      const int d = lane + 32 * i;
      qv[i] = d < D ? __bfloat162float(qr[d]) : 0.f;
      dov[i] = d < D ? __bfloat162float(dor[d]) : 0.f;
      if (d < D) {
        dot = fmaf(qv[i], kv[i], dot);
        dp = fmaf(dov[i], vv[i], dp);
        delta = fmaf(dov[i], __bfloat162float(orow[d]), delta);
      }
    }
    dot = warp_sum(dot);
    dp = warp_sum(dp);
    delta = warp_sum(delta);
    bool keep = true;
    if (p.drop.thresh16) {  // element kk % 32 of stream (q, kk / 32): jump there
      DropStream st = drop_stream(p.drop, (uint32_t)q, (uint32_t)kk >> 5);
      uint32_t x = 0;
      for (int e = 0; e <= (kk & 31); ++e) x = st.next();
      keep = x >= thr;
    }
    int gq = 0, pq = 0;
    if (p.gid) { gq = p.gid[(long long)b * T + q]; pq = p.pos[(long long)b * T + q]; }
    const bool vis = ag_visible(p, gq, pq, b, kk);
    const float lse2 = p.lse[((long long)b * p.heads + h) * T + q] * 1.4426950408889634f;
    const float pe = vis ? fast_exp2(fmaf(dot, p.scale_log2, bias2) - lse2) : 0.f;
    const float pd = keep ? pe * p.drop.inv_keep : 0.f;
    const float dpd = keep ? dp * p.drop.inv_keep : 0.f;
    const float ds = pe * (dpd - delta) * p.scale;
#pragma unroll
    for (int i = 0; i < AG_PER_LANE; ++i) {
      dv[i] = fmaf(pd, dov[i], dv[i]);
      dk[i] = fmaf(ds, qv[i], dk[i]);
    }
  }
  __nv_bfloat16* dkr = p.dk + b * p.dk_bs + kk * p.dk_ts + (long long)h * D;
  __nv_bfloat16* dvr = p.dv + b * p.dv_bs + kk * p.dv_ts + (long long)h * D;
#pragma unroll
  for (int i = 0; i < AG_PER_LANE; ++i) {
    const int d = lane + 32 * i;
    if (d < D) {
      dkr[d] = __float2bfloat16(dk[i]);
      dvr[d] = __float2bfloat16(dv[i]);
    }
  }
}

static void fill_params(AttnGenericParams& p, const tome_attn_desc_t* d, const void* q, const void* k, const void* v) {
  p.batch = d->batch; p.tokens = d->tokens; p.heads = d->heads; p.dim = d->head_dim;
  p.scale = d->scale; p.scale_log2 = d->scale * 1.4426950408889634f;
  p.gid = d->gid; p.pos = d->pos; p.allow = d->allow; p.num_groups = d->num_groups; p.size = d->size;
  p.drop = make_dropout(d->dropout_rate, d->dropout_seed, d->dropout_site);
  p.q = reinterpret_cast<const __nv_bfloat16*>(q); p.k = reinterpret_cast<const __nv_bfloat16*>(k);
  p.v = reinterpret_cast<const __nv_bfloat16*>(v);
  p.q_bs = d->q_batch_stride; p.q_ts = d->q_token_stride; p.k_bs = d->k_batch_stride; p.k_ts = d->k_token_stride;
  p.v_bs = d->v_batch_stride; p.v_ts = d->v_token_stride; p.o_bs = d->o_batch_stride; p.o_ts = d->o_token_stride;
}

// called by tome_attention_fwd / _bwd for head_dim != 64
int attn_generic_fwd(const tome_attn_desc_t* d, const void* q, const void* k, const void* v, void* out, float* lse,
                     cudaStream_t stream) {
  TOME_CHECK(d->head_dim >= 8 && d->head_dim <= AG_MAXD && d->head_dim % 8 == 0, TOME_ERR_UNSUPPORTED,
             "attention: head_dim %d not supported (64 on tensor cores; multiples of 8 up to %d on the generic path)", d->head_dim, AG_MAXD);
  AttnGenericParams p;
  fill_params(p, d, q, k, v);
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.lse = lse;
  dim3 grid(ceil_div(d->tokens, AG_WARPS), d->heads, d->batch);
  launch_k(attn_generic_fwd_kernel, grid, AG_WARPS * 32, 0, stream, p);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

int attn_generic_bwd(const tome_attn_desc_t* d, const tome_attn_grad_strides_t* gs, const void* q, const void* k, const void* v,
                     const void* out, const float* lse, const void* dout, void* dq, void* dk, void* dv, cudaStream_t stream) {
  TOME_CHECK(d->head_dim >= 8 && d->head_dim <= AG_MAXD && d->head_dim % 8 == 0, TOME_ERR_UNSUPPORTED,
             "attention: head_dim %d not supported (64 on tensor cores; multiples of 8 up to %d on the generic path)", d->head_dim, AG_MAXD);
  AttnGenericParams p;
  fill_params(p, d, q, k, v);
  p.lse = const_cast<float*>(lse);
  p.o_in = reinterpret_cast<const __nv_bfloat16*>(out);
  p.dout = reinterpret_cast<const __nv_bfloat16*>(dout);
  p.do_bs = gs->do_batch_stride; p.do_ts = gs->do_token_stride;
  p.dq = reinterpret_cast<__nv_bfloat16*>(dq); p.dk = reinterpret_cast<__nv_bfloat16*>(dk); p.dv = reinterpret_cast<__nv_bfloat16*>(dv);
  p.dq_bs = gs->dq_batch_stride; p.dq_ts = gs->dq_token_stride; p.dk_bs = gs->dk_batch_stride; p.dk_ts = gs->dk_token_stride;
  p.dv_bs = gs->dv_batch_stride; p.dv_ts = gs->dv_token_stride;
  dim3 grid(ceil_div(d->tokens, AG_WARPS), d->heads, d->batch);
  launch_k(attn_generic_dq_kernel, grid, AG_WARPS * 32, 0, stream, p);
  launch_k(attn_generic_dkdv_kernel, grid, AG_WARPS * 32, 0, stream, p);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

}  // namespace tome
