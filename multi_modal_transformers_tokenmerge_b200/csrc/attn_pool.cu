// K14: the attention step of MultiHeadAttentionPooling.   attention_blocks/attention.py:122-150 (SURVEY.md 8(f) rank 3)
//
//   query = tile(learnt_q_input [1, 1, E], batch);  x = MultiHeadDotProductAttention(query, x);  ...          attention.py:139-147
//
// ONE query row per batch row attends over n keys (the readout tokens: 4 .. 64): a few thousand flops per (batch row, head),
// so this is not a tensor-core shape.  The query is batch-independent: pool_query_kernel projects the learnt input once
// (q = learnt . Wq + bq, already scaled by 1 / sqrt(D)), then one warp per (batch row, head) takes the n logits, the softmax
// and the weighted sum of the value rows, lanes splitting the head dimension.  The key / value projections before it, the
// out projection, LayerNorm and MLPBlock after it are the library's GEMM / LayerNorm entry points (the Python mirror
// attention_blocks/attention.py::MultiHeadAttentionPooling strings them together).  fp32 arithmetic on bf16 keys / values.
#include <float.h>

#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int AP_MAX_KEYS = 64;

// q[j] = scale * (sum_c learnt[c] * wq[c, j] + bq[j]),  j < H * D: one thread per output (E x HD multiply-adds in total)
__global__ void pool_query_kernel(int E, int HD, const float* __restrict__ learnt, const float* __restrict__ wq,
                                  const float* __restrict__ bq, float scale, float* __restrict__ q) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= HD) return;
  float acc = 0.f;
  for (int c = 0; c < E; ++c) acc = fmaf(learnt[c], wq[(long long)c * HD + j], acc);
  q[j] = (acc + (bq ? bq[j] : 0.f)) * scale;
}

// warp = (batch row, head).  kv bf16 [B, n, ld]: keys at column 0, values at column v_off (both [H, D] wide).
__global__ void __launch_bounds__(128)
attn_pool_kernel(int B, int n, int H, int D, const float* __restrict__ q, const __nv_bfloat16* __restrict__ kv, long long ld,
                 int v_off, __nv_bfloat16* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (w >= B * H) return;
  const int b = w / H, h = w - b * H;
  const __nv_bfloat16* kb = kv + (long long)b * n * ld + (long long)h * D;
  float logit[AP_MAX_KEYS / 32] = {-FLT_MAX, -FLT_MAX};   // key j lives in lane j % 32, slot j / 32
  for (int j = 0; j < n; ++j) {
    float dot = 0.f;
    for (int d = lane; d < D; d += 32) dot = fmaf(q[h * D + d], __bfloat162float(kb[(long long)j * ld + d]), dot);
    dot = warp_sum(dot);
    if ((j & 31) == lane) logit[j >> 5] = dot;
  }
  float m = warp_max(fmaxf(logit[0], logit[1]));
  float e0 = logit[0] == -FLT_MAX ? 0.f : __expf(logit[0] - m), e1 = logit[1] == -FLT_MAX ? 0.f : __expf(logit[1] - m);
  const float inv = 1.0f / warp_sum(e0 + e1);
  for (int d = lane; d < D; d += 32) {
    float acc = 0.f;
    for (int j = 0; j < n; ++j) {
      const float wj = __shfl_sync(0xffffffffu, (j >> 5) ? e1 : e0, j & 31) * inv;
      acc = fmaf(wj, __bfloat162float(kb[(long long)j * ld + v_off + d]), acc);
    }
    out[((long long)b * H + h) * D + d] = __float2bfloat16(acc);
  }
}

}  // namespace tome

using namespace tome;

extern "C" int tome_attention_pool_fwd(int batch, int n_keys, int heads, int head_dim, int embed_dim, const float* learnt_q,
                                       const float* wq, const float* bq, const void* kv, long long kv_ld, int v_col,
                                       float* q_scratch, void* out, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && heads > 0 && head_dim > 0 && embed_dim > 0, TOME_ERR_INVALID, "attention_pool: bad shape");
  TOME_CHECK(n_keys >= 1 && n_keys <= AP_MAX_KEYS, TOME_ERR_UNSUPPORTED, "attention_pool: 1 <= n_keys <= %d (got %d)", AP_MAX_KEYS, n_keys);
  TOME_CHECK(learnt_q && wq && kv && q_scratch && out, TOME_ERR_INVALID, "attention_pool: null argument");
  TOME_CHECK(kv_ld >= (long long)v_col + heads * head_dim && v_col >= heads * head_dim, TOME_ERR_INVALID,
             "attention_pool: kv rows hold the keys at column 0 and the values at column v_col >= heads * head_dim");
  const int HD = heads * head_dim;
  ProfScope prof(PROF_OTHER, 0.0, 2, stream);
  launch_k(pool_query_kernel, (unsigned)ceil_div(HD, 128), 128, 0, stream, embed_dim, HD, learnt_q, wq, bq, 1.0f / sqrtf((float)head_dim), q_scratch);
  TOME_CUDA(cudaGetLastError());
  launch_k(attn_pool_kernel, (unsigned)ceil_div(batch * heads, 4), 128, 0, stream, batch, n_keys, heads, head_dim, q_scratch,
           reinterpret_cast<const __nv_bfloat16*>(kv), kv_ld, v_col, reinterpret_cast<__nv_bfloat16*>(out));
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
