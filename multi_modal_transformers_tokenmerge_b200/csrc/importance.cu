// K13: token importance from the attention weights.   attention_blocks/compressed_attention.py:303-306 (SURVEY.md 8(f) rank 2)
//
//   importance_scores = mean over heads ( mean over the LAST axis ( attn_weights [B, H, Tq, Tk] ) )      -> [B, T]
//
// As written that is the mean over KEYS of rows that each sum to one, i.e. 1 / T for every token (DESIGN.md 7): mode
// TOME_IMPORTANCE_ROW_MEAN computes exactly that expression.  TOME_IMPORTANCE_RECEIVED is the same double mean with the
// inner one over QUERIES -- the attention a token receives, the quantity top-k pruning (token_compression.py:15-46) can
// rank on.  Both are sums of P[q, k] = exp(s[q, k] + log size[k] - lse[q]) with the row statistics lse the attention
// forward kernel already saved, so no softmax pass is repeated: every (q, k) element is independent.
//
// The contraction s = q . k is the one place here that is a matrix product, and it is small and feeds a transcendental
// epilogue: 16-row tiles per warp on the warp-level bf16 MMA (mma.sync m16n8k16, fp32 accumulate -- the same operand
// rounding as the attention kernels' S), A fragments of the warp's 16 rows held in registers across the sweep over the
// other axis, the swept operand staged through shared memory (cp.async, double-buffered) and read with ldmatrix.
// Sums run in a fixed order (thread-sequential over heads and column tiles, then a 4-lane butterfly) => deterministic.
// Weights are the UNDROPPED ones (the ranking must not depend on the dropout stream).
#include <float.h>

#include "attn_meta.cuh"
#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int IMP_WARPS = 4;

struct ImpParams {
  int batch, tokens, heads;
  float scale_log2;
  const __nv_bfloat16 *q, *k;
  long long q_bs, q_ts, k_bs, k_ts;
  const float* lse;     // [B, H, T] natural log (attention forward)
  const float* size;    // [B, T] or null
  const uint8_t* gid; const int32_t* pos; const uint8_t* allow; int num_groups;
  float* out;           // [B, T]
};

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t saddr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(saddr));
}
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }


// ROWS_ARE_KEYS: the warp's 16 rows are keys and it sweeps the queries (RECEIVED); otherwise rows are queries, sweep over keys.
// CTA = 4 warps x 16 rows.  The swept operand goes through shared memory in 64-row blocks (cp.async, two buffers; rows padded
// by 16 bytes so the 8 x 8 ldmatrix tiles are conflict-free) together with its per-column terms (lse or log size, group,
// position); B fragments come from ldmatrix (a row-major [n][k] tile IS the "col" B operand of m16n8k16).
template <int D, bool ROWS_ARE_KEYS, bool MASKED>
__global__ void __launch_bounds__(IMP_WARPS * 32)
attn_importance_kernel(const ImpParams p) {
  constexpr int PITCH = D + 8;   // bf16 elements per staged row
  constexpr int IMP_COLS = D > 128 ? 32 : 64;   // rows of the swept operand staged per step (static shared memory <= 48 KB)
  __shared__ __align__(16) __nv_bfloat16 ys[2][IMP_COLS * PITCH];
  __shared__ float c_term_s[2][IMP_COLS];
  __shared__ int c_gp_s[2][IMP_COLS];     // group | position << 8
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int b = blockIdx.y, T = p.tokens, G = p.num_groups;
  const int r0 = (blockIdx.x * IMP_WARPS + warp) * 16;
  const __nv_bfloat16* X = (ROWS_ARE_KEYS ? p.k + b * p.k_bs : p.q + b * p.q_bs);
  const __nv_bfloat16* Y = (ROWS_ARE_KEYS ? p.q + b * p.q_bs : p.k + b * p.k_bs);
  const long long x_ts = ROWS_ARE_KEYS ? p.k_ts : p.q_ts, y_ts = ROWS_ARE_KEYS ? p.q_ts : p.k_ts;
  const int row[2] = {r0 + g, r0 + g + 8};
  const bool row_ok[2] = {row[0] < T, row[1] < T};
  const long long bt = (long long)b * T;
  // Visibility of a column group for each of this thread's two rows, as bit masks over the (<= 32) groups: bit cg of vis1 =
  // the pair is always visible, of vis2 = visible when the key's position does not exceed the query's (causal-intra sets).
  int rp[2] = {0, 0};
  uint32_t vis1[2] = {0xffffffffu, 0xffffffffu}, vis2[2] = {0u, 0u};
  float r_term[2] = {0.f, 0.f};   // log2 size of a key row; -lse2 of a query row is set per head below
#pragma unroll
  for (int i = 0; i < 2; ++i)
    if (row_ok[i]) {
      if (MASKED) {
        const int rg = p.gid[bt + row[i]];
        rp[i] = p.pos[bt + row[i]];
        vis1[i] = 0u;
        for (int cg = 0; cg < G; ++cg) {
          const int al = ROWS_ARE_KEYS ? p.allow[cg * G + rg] : p.allow[rg * G + cg];
          vis1[i] |= (al == 1 ? 1u : 0u) << cg;
          vis2[i] |= (al == 2 ? 1u : 0u) << cg;
        }
      }
      if (ROWS_ARE_KEYS && p.size) r_term[i] = log2f(p.size[bt + row[i]]);
    }
  const int nblk = (T + IMP_COLS - 1) / IMP_COLS, n_it = p.heads * nblk;

  auto stage = [&](int it, int buf) {   // block `it` = (head, 64-row block) of the swept operand -> buffer buf
    const int h = it / nblk, c0 = (it - h * nblk) * IMP_COLS;
    constexpr int VPR = D / 8;          // 16-byte vectors per row
    for (int v = threadIdx.x; v < IMP_COLS * VPR; v += IMP_WARPS * 32) {
      const int r = v / VPR, c = v - r * VPR;
      const int yrow = min(c0 + r, T - 1);
      cp_async16(smem_u32(&ys[buf][r * PITCH + c * 8]), Y + (long long)yrow * y_ts + h * D + c * 8);
    }
    cp_async_commit();
    if (threadIdx.x < IMP_COLS) {
      const bool ok = c0 + (int)threadIdx.x < T;   // a column past T contributes exp2(-inf) = 0
      const int col = min(c0 + (int)threadIdx.x, T - 1);
      const float ct = ROWS_ARE_KEYS ? -p.lse[((long long)b * p.heads + h) * T + col] * 1.4426950408889634f
                                     : (p.size ? log2f(p.size[bt + col]) : 0.f);
      c_term_s[buf][threadIdx.x] = ok ? ct : -INFINITY;
      c_gp_s[buf][threadIdx.x] = MASKED ? ((int)p.gid[bt + col] | (p.pos[bt + col] << 8)) : 0;
    }
  };

  float acc[2] = {0.f, 0.f};
  const float inv_t = 1.0f / (float)T;
  uint32_t a[D / 16][4];
  stage(0, 0);
  for (int it = 0; it < n_it; ++it) {
    const int buf = it & 1;
    const int h = it / nblk, c0 = (it - h * nblk) * IMP_COLS;
    if (c0 == 0) {   // a new head: this warp's 16 rows of the fixed operand
#pragma unroll
      for (int kk = 0; kk < D / 16; ++kk)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int ri = i & 1;
          a[kk][i] = row_ok[ri] ? *reinterpret_cast<const uint32_t*>(X + (long long)row[ri] * x_ts + h * D + kk * 16 + (i >> 1) * 8 + 2 * t) : 0u;
        }
      if (!ROWS_ARE_KEYS) {
#pragma unroll
        for (int i = 0; i < 2; ++i)
          r_term[i] = row_ok[i] ? -p.lse[((long long)b * p.heads + h) * T + row[i]] * 1.4426950408889634f : 0.f;
        // a query with no visible key (attn_meta.cuh) weighs each of the T keys 1/T: its row sums to one
        if (MASKED && t == 0)
#pragma unroll
          for (int i = 0; i < 2; ++i) acc[i] += r_term[i] > -ATTN_MASKED_ROW_LSE2 ? 1.f : 0.f;
      }
    }
    cp_async_wait<0>();
    __syncthreads();                       // block `it` has landed; every warp is done with the other buffer
    if (it + 1 < n_it) stage(it + 1, buf ^ 1);
    if (r0 < T) {
      const uint32_t ybase = smem_u32(&ys[buf][0]) + ((lane & 7) * PITCH + (lane >> 3) * 8) * 2;
#pragma unroll 2
      for (int j = 0; j < IMP_COLS / 8; ++j) {
        if (c0 + j * 8 >= T) break;
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int kp = 0; kp < D / 32; ++kp) {
          uint32_t bf[4];
          ldmatrix_x4(bf, ybase + (j * 8 * PITCH + kp * 32) * 2);
          mma_bf16_16816(c, a[2 * kp], bf[0], bf[1]);
          mma_bf16_16816(c, a[2 * kp + 1], bf[2], bf[3]);
        }
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int cl = j * 8 + 2 * t + jj;
          const float c_term = c_term_s[buf][cl];
          const int gp = MASKED ? c_gp_s[buf][cl] : 0;
          const int cg = gp & 255, cp = gp >> 8;
          // received: a query with no visible key (attn_meta.cuh) gives 1/T to every key
          const float c_fill = ROWS_ARE_KEYS && c_term > -ATTN_MASKED_ROW_LSE2 ? inv_t : 0.f;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const float s2 = fmaf(c[2 * i + jj], p.scale_log2, c_term + r_term[i]);
            if (MASKED) {
              const bool causal_ok = ROWS_ARE_KEYS ? rp[i] <= cp : cp <= rp[i];
              const bool vis = ((vis1[i] >> cg) & 1u) || (((vis2[i] >> cg) & 1u) && causal_ok);
              acc[i] += vis ? fast_exp2(s2) : c_fill;
            } else {
              acc[i] += fast_exp2(s2);
            }
          }
        }
      }
    }
  }
  const float inv = 1.0f / ((float)p.heads * (float)T);
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    float v = acc[i];
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    if (t == 0 && row_ok[i]) p.out[bt + row[i]] = v * inv;
  }
}

}  // namespace tome

using namespace tome;

extern "C" int tome_attention_importance(const tome_attn_desc_t* d, const void* q, const void* k, const float* lse, int mode,
                                         float* importance, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(d && q && k && lse && importance, TOME_ERR_INVALID, "attention_importance: null argument");
  TOME_CHECK(d->batch > 0 && d->batch <= 65535 && d->tokens > 0 && d->heads > 0, TOME_ERR_INVALID, "attention_importance: bad shape");
  TOME_CHECK(d->head_dim == 64 || d->head_dim == 128 || d->head_dim == 256, TOME_ERR_UNSUPPORTED,
             "attention_importance: head_dim %d not supported (64, 128, 256)", d->head_dim);
  TOME_CHECK(mode == TOME_IMPORTANCE_ROW_MEAN || mode == TOME_IMPORTANCE_RECEIVED, TOME_ERR_INVALID, "attention_importance: unknown mode %d", mode);
  TOME_CHECK((d->q_token_stride | d->k_token_stride | d->q_batch_stride | d->k_batch_stride) % 8 == 0 &&
             (((uintptr_t)q | (uintptr_t)k) & 15) == 0, TOME_ERR_INVALID, "attention_importance: q / k rows must be 16-byte aligned");
  TOME_CHECK(d->num_groups <= 32, TOME_ERR_INVALID, "attention_importance: at most 32 groups");
  TOME_CHECK(!d->gid || (d->pos && d->allow && d->num_groups > 0), TOME_ERR_INVALID, "attention_importance: gid needs pos, allow, num_groups");
  ImpParams p;
  p.batch = d->batch; p.tokens = d->tokens; p.heads = d->heads;
  p.scale_log2 = d->scale * 1.4426950408889634f;
  p.q = reinterpret_cast<const __nv_bfloat16*>(q); p.k = reinterpret_cast<const __nv_bfloat16*>(k);
  p.q_bs = d->q_batch_stride; p.q_ts = d->q_token_stride; p.k_bs = d->k_batch_stride; p.k_ts = d->k_token_stride;
  p.lse = lse; p.size = d->size;
  p.gid = d->gid; p.pos = d->pos; p.allow = d->allow; p.num_groups = d->num_groups;
  p.out = importance;
  const dim3 grid(ceil_div(d->tokens, 16 * IMP_WARPS), d->batch);
  const double flops = 2.0 * d->batch * d->heads * (double)d->tokens * d->tokens * d->head_dim;
  ProfScope prof(PROF_IMPORTANCE, flops, 1, stream);
#define IMP_LAUNCH2(DD, RK)                                                                              \
  if (d->gid) launch_k(attn_importance_kernel<DD, RK, true>, grid, IMP_WARPS * 32, 0, stream, p);        \
  else launch_k(attn_importance_kernel<DD, RK, false>, grid, IMP_WARPS * 32, 0, stream, p)
#define IMP_LAUNCH(DD)                                                     \
  if (mode == TOME_IMPORTANCE_RECEIVED) { IMP_LAUNCH2(DD, true); }         \
  else { IMP_LAUNCH2(DD, false); }
  if (d->head_dim == 64) { IMP_LAUNCH(64); }
  else if (d->head_dim == 128) { IMP_LAUNCH(128); }
  else { IMP_LAUNCH(256); }
#undef IMP_LAUNCH
#undef IMP_LAUNCH2
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
