// K10: action heads on the pooled readout rows + their training losses (SURVEY.md 8(f) rank 3).
//
//   ContinuousActionHead.__call__   action_heads/continuous.py:16-25   mean over the readouts -> Dense -> tanh(z/max)*max
//   Octo.compute_l2_loss            models/octo/octo.py:157-165        sum_a (pred - action)^2, mean over the batch (:253-263)
//   CategoricalActionHead.__call__  action_heads/categorical.py:30-40  "(action timestep)" groups averaged -> Dense -> logits
//   assign_bins + Octo.compute_ce_loss  categorical.py:12-22, octo.py:178-190   digitize into uniform bins, one_hot,
//                                                                      optax.softmax_cross_entropy
//
// Every head starts with `jnp.mean(readouts, axis=-2)`; here the readouts are never gathered into their own tensor: the
// kernel reads the rows of the final (merged) sequence the readout tokens ended up in (origin[b,i], from
// tome_chain_row_maps) and averages them in fp32.  The heads are a few thousand flops per batch row, so one CTA per batch
// row does pool -> Dense -> loss -> dL/dz in one launch; backward is two launches (dW/db with a fixed summation order over
// the batch, and the scatter of dL/dpooled back into the rows).  Everything is fp32 and deterministic.
#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int HEAD_THREADS = 256;

struct HeadWs {
  float* pooled;  // [B, G, C]
  float* dz;      // [B, G, F]   dL/dz of the mean loss
  size_t total;
};
static HeadWs head_ws(const tome_head_desc_t* d, void* base) {
  Bump b{reinterpret_cast<uint8_t*>(base)};
  HeadWs w;
  w.pooled = b.take<float>((size_t)d->batch * d->groups * d->channels);
  w.dz = b.take<float>((size_t)d->batch * d->groups * d->features);
  w.total = b.total();
  return w;
}

template <bool BF16>
__device__ __forceinline__ float head_load(const void* x, long long i) {
  if constexpr (BF16) return __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(x)[i]);
  else return reinterpret_cast<const float*>(x)[i];
}

// jnp.digitize(v, jnp.linspace(-max, max, F + 1)): the number of edges <= v (edges increasing, right = False).
// linspace in fp32: edge_k = lo + k * step, the last edge is `hi` exactly.
__device__ __forceinline__ int head_digitize(float v, float max_action, int F) {
  const float lo = -max_action, hi = max_action, step = (hi - lo) / (float)F;
  int n = 0;
  for (int k = 0; k <= F; ++k) {
    const float e = k == F ? hi : __fmaf_rn((float)k, step, lo);
    n += (e <= v) ? 1 : 0;
  }
  return n;
}

template <bool BF16>
__global__ void __launch_bounds__(HEAD_THREADS)
head_fwd_kernel(const tome_head_desc_t d, const void* __restrict__ x, const int32_t* __restrict__ origin,
                const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ actions,
                float* __restrict__ out, float* __restrict__ loss, float* __restrict__ pooled_g, float* __restrict__ dz_g) {
  extern __shared__ float head_sm[];
  const int b = blockIdx.x, C = d.channels, G = d.groups, F = d.features, m = d.n_readout / d.groups;
  float* pooled = head_sm;        // [G*C]
  float* z = head_sm + G * C;     // [G*F]
  __shared__ float group_loss[64];
  // 1. pooled[g, :] = mean of the group's rows (sequential over the rows, fp32)
  const float inv_m = 1.0f / (float)m;
  for (int i = threadIdx.x; i < G * C; i += HEAD_THREADS) {
    const int g = i / C, c = i - g * C;
    float s = 0.f;
    for (int j = 0; j < m; ++j) {
      const int row = origin[b * d.n_readout + g * m + j];
      s += head_load<BF16>(x, ((long long)b * d.tokens + row) * C + c);
    }
    s *= inv_m;
    pooled[i] = s;
    if (pooled_g) pooled_g[(long long)b * G * C + i] = s;
  }
  __syncthreads();
  // 2. z[g, f] = pooled[g, :] . W[:, f] + bias[f]   (one warp per output, lanes stride the channels, fixed shuffle tree)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int o = warp; o < G * F; o += HEAD_THREADS / 32) {
    const int g = o / F, f = o - g * F;
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s = fmaf(pooled[g * C + c], w[(long long)c * F + f], s);
    s = warp_sum(s);
    if (lane == 0) z[o] = s + (bias ? bias[f] : 0.f);
  }
  __syncthreads();
  // 3. head output, loss of this batch row, dL/dz
  if (d.kind == TOME_HEAD_CONTINUOUS_L2) {
    // pred = tanh(z / max) * max (continuous.py:25); loss_b = sum_a (pred - action)^2 (octo.py:165); L = mean_b loss_b
    if (threadIdx.x < F) {
      const int f = threadIdx.x;
      const float t = tanhf(z[f] / d.max_action);
      const float pred = t * d.max_action;
      out[(long long)b * F + f] = pred;
      float l = 0.f, g = 0.f;
      if (actions) {
        const float diff = pred - actions[(long long)b * F + f];
        l = diff * diff;
        g = 2.0f * diff / (float)d.batch * (1.0f - t * t);
      }
      z[f] = l;
      if (dz_g) dz_g[(long long)b * F + f] = g;
    }
    __syncthreads();
    if (threadIdx.x == 0 && loss) {
      float t = 0.f;
      for (int f = 0; f < F; ++f) t += z[f];
      loss[1 + b] = t;
    }
  } else {
    // logits = z; label = one_hot(digitize(action), F) (all zeros when the index is >= F, as jax.nn.one_hot);
    // loss[b, g] = -sum_f label_f * log_softmax(z)_f; L = mean over (b, g)
    if (threadIdx.x < G) {
      const int g = threadIdx.x;
      float mx = -INFINITY;
      for (int f = 0; f < F; ++f) mx = fmaxf(mx, z[g * F + f]);
      float se = 0.f;
      for (int f = 0; f < F; ++f) se += expf(z[g * F + f] - mx);
      const float lse = mx + logf(se);
      int label = -1;
      if (actions) label = head_digitize(actions[(long long)b * G + g], d.max_action, F);
      const bool hot = label >= 0 && label < F;
      group_loss[g] = hot ? lse - z[g * F + label] : 0.f;
      const float gs = 1.0f / ((float)d.batch * (float)G);
      for (int f = 0; f < F; ++f) {
        const float zf = z[g * F + f];
        out[((long long)b * G + g) * F + f] = zf;
        if (dz_g) dz_g[((long long)b * G + g) * F + f] = hot ? (expf(zf - lse) - (f == label ? 1.f : 0.f)) * gs : 0.f;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0 && loss) {
      float t = 0.f;
      for (int g = 0; g < G; ++g) t += group_loss[g];
      loss[1 + b] = t;
    }
  }
}

__global__ void head_loss_final_kernel(int B, float inv_count, float* loss) {
  float t = 0.f;
  for (int b = 0; b < B; ++b) t += loss[1 + b];
  loss[0] = t * inv_count;
}

// dW[c, f] += sum_{b, g} pooled[b, g, c] * dz[b, g, f];  db[f] += sum_{b, g} dz[b, g, f].
// A CTA owns 32 consecutive outputs; its 8 warps each sum one contiguous slice of the B*G rows and the slices are added
// in warp order through shared memory, so the result does not depend on the launch (no atomics).
__global__ void __launch_bounds__(HEAD_THREADS)
head_wgrad_kernel(const tome_head_desc_t d, const float* __restrict__ pooled, const float* __restrict__ dz,
                  float* __restrict__ dw, float* __restrict__ dbias) {
  __shared__ float part[HEAD_THREADS / 32][32];
  const int C = d.channels, F = d.features, BG = d.batch * d.groups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = HEAD_THREADS / 32;
  const long long i = blockIdx.x * 32LL + lane, n_w = (long long)C * F;
  const int r0 = (int)((long long)BG * warp / nw), r1 = (int)((long long)BG * (warp + 1) / nw);
  float s = 0.f;
  if (i < n_w) {
    const int c = (int)(i / F), f = (int)(i - (long long)c * F);
    for (int r = r0; r < r1; ++r) s = fmaf(pooled[(long long)r * C + c], dz[(long long)r * F + f], s);
  } else if (i < n_w + F) {
    const int f = (int)(i - n_w);
    for (int r = r0; r < r1; ++r) s += dz[(long long)r * F + f];
  }
  part[warp][lane] = s;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
    for (int w = 0; w < nw; ++w) t += part[w][lane];
    if (i < n_w) dw[i] += t;
    else if (dbias && i < n_w + F) dbias[i - n_w] += t;
  }
}

// dx[b, origin[b, g*m + j], :] += (W dz[b, g, :]) / m   (dx zeroed by the caller of this kernel; bf16 or f32)
template <bool BF16>
__global__ void __launch_bounds__(HEAD_THREADS)
head_dgrad_kernel(const tome_head_desc_t d, const int32_t* __restrict__ origin, const float* __restrict__ w,
                  const float* __restrict__ dz, void* __restrict__ dx) {
  extern __shared__ float head_sm[];
  const int b = blockIdx.x, C = d.channels, G = d.groups, F = d.features, m = d.n_readout / d.groups;
  float* dzs = head_sm;  // [G*F]
  for (int i = threadIdx.x; i < G * F; i += HEAD_THREADS) dzs[i] = dz[(long long)b * G * F + i];
  __syncthreads();
  const float inv_m = 1.0f / (float)m;
  for (int c = threadIdx.x; c < C; c += HEAD_THREADS) {
    for (int g = 0; g < G; ++g) {
      float s = 0.f;
      for (int f = 0; f < F; ++f) s = fmaf(w[(long long)c * F + f], dzs[g * F + f], s);
      s *= inv_m;
      for (int j = 0; j < m; ++j) {  // two readouts merged into one row: the same thread adds twice, in order
        const long long xi = ((long long)b * d.tokens + origin[b * d.n_readout + g * m + j]) * C + c;
        if constexpr (BF16) {
          __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(dx) + xi;
          *p = __float2bfloat16(__bfloat162float(*p) + s);
        } else {
          reinterpret_cast<float*>(dx)[xi] += s;
        }
      }
    }
  }
}

static int check_head(const tome_head_desc_t* d) {
  TOME_CHECK(d != nullptr, TOME_ERR_INVALID, "action_head: null descriptor");
  TOME_CHECK(d->batch > 0 && d->tokens > 0 && d->channels > 0 && d->n_readout > 0, TOME_ERR_INVALID, "action_head: bad shape");
  TOME_CHECK(d->x_dtype == TOME_BF16 || d->x_dtype == TOME_F32, TOME_ERR_INVALID, "action_head: x must be bf16 or f32");
  TOME_CHECK(d->kind == TOME_HEAD_CONTINUOUS_L2 || d->kind == TOME_HEAD_CATEGORICAL_CE, TOME_ERR_INVALID,
             "action_head: kind must be TOME_HEAD_CONTINUOUS_L2 or TOME_HEAD_CATEGORICAL_CE");
  TOME_CHECK(d->groups >= 1 && d->groups <= 64 && d->n_readout % d->groups == 0, TOME_ERR_INVALID,
             "action_head: %d readouts do not split into %d groups (einops '(action timestep)', categorical.py:32-36)",
             d->n_readout, d->groups);
  TOME_CHECK(d->kind != TOME_HEAD_CONTINUOUS_L2 || d->groups == 1, TOME_ERR_INVALID,
             "action_head: the continuous head averages all readouts (continuous.py:17): groups must be 1");
  TOME_CHECK(d->features >= 1 && d->features <= 4096, TOME_ERR_INVALID, "action_head: 1 <= features <= 4096");
  TOME_CHECK(d->kind != TOME_HEAD_CONTINUOUS_L2 || d->features <= HEAD_THREADS, TOME_ERR_UNSUPPORTED,
             "action_head: continuous head supports at most %d action dimensions", HEAD_THREADS);
  TOME_CHECK(d->max_action > 0.f, TOME_ERR_INVALID, "action_head: max_action must be positive");
  const size_t smem = ((size_t)d->groups * d->channels + (size_t)d->groups * d->features) * sizeof(float);
  TOME_CHECK(smem <= 160 * 1024, TOME_ERR_UNSUPPORTED, "action_head: groups * (channels + features) too large for shared memory");
  return TOME_OK;
}

}  // namespace tome

using namespace tome;

extern "C" size_t tome_action_head_workspace_bytes(const tome_head_desc_t* d) {
  clear_error();
  if (check_head(d) != TOME_OK) return 0;
  return head_ws(d, nullptr).total;
}

extern "C" int tome_action_head_fwd(const tome_head_desc_t* d, const void* x, const int32_t* origin, const float* w,
                                    const float* bias, const float* actions, float* out, float* loss, void* workspace,
                                    size_t workspace_bytes, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int rc = check_head(d)) return rc;
  TOME_CHECK(x && origin && w && out, TOME_ERR_INVALID, "action_head_fwd: null argument");
  TOME_CHECK(!loss || actions, TOME_ERR_INVALID, "action_head_fwd: a loss needs the target actions");
  const HeadWs ws = head_ws(d, workspace);  // no workspace: nothing kept for the backward
  TOME_CHECK(!workspace || (workspace_bytes >= ws.total && ((uintptr_t)workspace & 255) == 0), TOME_ERR_INVALID,
             "action_head_fwd: workspace too small or not 256-byte aligned");
  const size_t smem = ((size_t)d->groups * d->channels + (size_t)d->groups * d->features) * sizeof(float);
  ProfScope prof(PROF_OTHER, 0.0, loss ? 2 : 1, stream);
  if (d->x_dtype == TOME_BF16) {
    TOME_CUDA(cudaFuncSetAttribute(head_fwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_k(head_fwd_kernel<true>, d->batch, HEAD_THREADS, smem, stream, *d, x, origin, w, bias, actions, out, loss, ws.pooled, ws.dz);
  } else {
    TOME_CUDA(cudaFuncSetAttribute(head_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    launch_k(head_fwd_kernel<false>, d->batch, HEAD_THREADS, smem, stream, *d, x, origin, w, bias, actions, out, loss, ws.pooled, ws.dz);
  }
  TOME_CUDA(cudaGetLastError());
  if (loss) {
    const float count = d->kind == TOME_HEAD_CONTINUOUS_L2 ? (float)d->batch : (float)d->batch * (float)d->groups;
    launch_k(head_loss_final_kernel, 1, 1, 0, stream, d->batch, 1.0f / count, loss);
    TOME_CUDA(cudaGetLastError());
  }
  return TOME_OK;
}

extern "C" int tome_action_head_bwd(const tome_head_desc_t* d, const int32_t* origin, const float* w, const void* workspace,
                                    float* dw, float* dbias, void* dx, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int rc = check_head(d)) return rc;
  TOME_CHECK(origin && w && workspace && dw, TOME_ERR_INVALID, "action_head_bwd: null argument");
  TOME_CHECK(((uintptr_t)workspace & 255) == 0, TOME_ERR_INVALID, "action_head_bwd: workspace must be 256-byte aligned");
  HeadWs ws = head_ws(d, const_cast<void*>(workspace));
  ProfScope prof(PROF_OTHER, 0.0, dx ? 3 : 1, stream);
  const long long n = (long long)d->channels * d->features + d->features;
  launch_k(head_wgrad_kernel, (unsigned)((n + 31) / 32), HEAD_THREADS, 0, stream, *d, ws.pooled, ws.dz, dw, dbias);
  TOME_CUDA(cudaGetLastError());
  if (dx) {
    const size_t esz = d->x_dtype == TOME_BF16 ? 2 : 4;
    TOME_CUDA(cudaMemsetAsync(dx, 0, (size_t)d->batch * d->tokens * d->channels * esz, stream));
    const size_t smem = (size_t)d->groups * d->features * sizeof(float);
    if (d->x_dtype == TOME_BF16) {
      TOME_CUDA(cudaFuncSetAttribute(head_dgrad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      launch_k(head_dgrad_kernel<true>, d->batch, HEAD_THREADS, smem, stream, *d, origin, w, ws.dz, dx);
    } else {
      TOME_CUDA(cudaFuncSetAttribute(head_dgrad_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      launch_k(head_dgrad_kernel<false>, d->batch, HEAD_THREADS, smem, stream, *d, origin, w, ws.dz, dx);
    }
    TOME_CUDA(cudaGetLastError());
  }
  return TOME_OK;
}
