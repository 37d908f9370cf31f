// Small HBM-bound steps around the block: position embedding (attention.py:97-100), readout gather + synthetic
// loss (octo.py:123-124, :167-174), row-map chaining, AdamW, casts.
#include "common.cuh"
#include "host_util.h"

namespace tome {

__device__ __forceinline__ void unpack8m(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 pack8m(const float (&f)[8]) {
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}

template <bool X_F32>
__global__ void add_pos_kernel(long long n8, long long tc8, const void* __restrict__ x, const float* __restrict__ pe,
                               __nv_bfloat16* __restrict__ y) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
    float f[8];
    if (X_F32) {
      const float4 a = reinterpret_cast<const float4*>(x)[2 * i], b = reinterpret_cast<const float4*>(x)[2 * i + 1];
      f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b.x; f[5] = b.y; f[6] = b.z; f[7] = b.w;
    } else {
      unpack8m(ld_nc_v4(reinterpret_cast<const uint4*>(x) + i), f);
    }
    const long long j = i % tc8;
    const float4 p0 = __ldg(reinterpret_cast<const float4*>(pe) + 2 * j), p1 = __ldg(reinterpret_cast<const float4*>(pe) + 2 * j + 1);
    f[0] += p0.x; f[1] += p0.y; f[2] += p0.z; f[3] += p0.w; f[4] += p1.x; f[5] += p1.y; f[6] += p1.z; f[7] += p1.w;
    reinterpret_cast<uint4*>(y)[i] = pack8m(f);
  }
}

__global__ void pos_bwd_kernel(int B, long long tc8, const __nv_bfloat16* __restrict__ dy, float* __restrict__ dpe) {
  const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (j >= tc8) return;
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.f;
  for (int b = 0; b < B; ++b) {
    float f[8];
    unpack8m(ld_nc_v4(reinterpret_cast<const uint4*>(dy) + (long long)b * tc8 + j), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] += f[i];
  }
  float4* o = reinterpret_cast<float4*>(dpe) + 2 * j;
  float4 o0 = o[0], o1 = o[1];
  o0.x += a[0]; o0.y += a[1]; o0.z += a[2]; o0.w += a[3]; o1.x += a[4]; o1.y += a[5]; o1.z += a[6]; o1.w += a[7];
  o[0] = o0; o[1] = o1;
}

constexpr int MAX_CHAIN = 64;
struct ChainArgs {
  const int32_t* maps[MAX_CHAIN];
  int tokens[MAX_CHAIN];
};
__global__ void chain_kernel(int B, int layers, const ChainArgs a, const int32_t* __restrict__ readout_idx, int n,
                             int32_t* __restrict__ origin) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * n) return;
  const int b = i / n;
  int pidx = readout_idx[i % n];
  for (int l = 0; l < layers; ++l)
    if (a.maps[l] && pidx >= 0) pidx = a.maps[l][(long long)b * a.tokens[l] + pidx];   // -1: pruned away by a pruning layer
  origin[i] = pidx;
}

// one CTA per batch row: gather, squared error, gradient scatter (sequential over readouts => deterministic)
__global__ void __launch_bounds__(256)
readout_mse_kernel(int B, int T, int C, int n, const __nv_bfloat16* __restrict__ x, const int32_t* __restrict__ origin,
                   const float* __restrict__ target, float* __restrict__ loss, __nv_bfloat16* __restrict__ dx,
                   float* __restrict__ out) {
  __shared__ float red[8];
  const int b = blockIdx.x;
  const float gscale = 2.0f / ((float)B * (float)n * (float)C);
  float local = 0.f;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    for (int i = 0; i < n; ++i) {
      const int row = origin[b * n + i];
      const long long xi = ((long long)b * T + row) * C + c;
      const float v = __bfloat162float(x[xi]);
      const float d = target ? v - target[((long long)b * n + i) * C + c] : 0.f;
      if (out) out[((long long)b * n + i) * C + c] = v;
      local = fmaf(d, d, local);
      if (dx) dx[xi] = __float2bfloat16(__bfloat162float(dx[xi]) + d * gscale);
    }
  }
  local = warp_sum(local);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = local;
  __syncthreads();
  if (threadIdx.x == 0 && loss) {
    float t = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    loss[1 + b] = t;
  }
}
__global__ void loss_final_kernel(int B, float inv_count, float* loss) {
  float t = 0.f;
  for (int b = 0; b < B; ++b) t += loss[1 + b];
  loss[0] = t * inv_count;
}

__global__ void adamw_kernel(long long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, __nv_bfloat16* __restrict__ w16, float lr, float b1, float b2, float eps,
                             float wd, float gs, float bc1, float bc2) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * gs;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    float pi = p[i];
    pi -= lr * ((mi / bc1) / (sqrtf(vi / bc2) + eps) + wd * pi);
    p[i] = pi;
    if (w16) w16[i] = __float2bfloat16(pi);
  }
}

__global__ void cast_kernel(long long n, const float* __restrict__ s, __nv_bfloat16* __restrict__ d) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    d[i] = __float2bfloat16(s[i]);
}

static inline int ew_grid(long long n, int threads) {
  long long b = (n + threads - 1) / threads;
  const long long cap = (long long)kNumSMs * 16;
  if (b > cap) b = cap;
  return (int)(b < 1 ? 1 : b);
}

}  // namespace tome

using namespace tome;

extern "C" int tome_add_pos_embedding(int batch, int tokens, int channels, const void* x, int x_dtype,
                                      const float* pos_embedding, void* y, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && channels > 0 && channels % 8 == 0, TOME_ERR_INVALID, "add_pos_embedding: bad shape");
  TOME_CHECK(x && pos_embedding && y, TOME_ERR_INVALID, "add_pos_embedding: null argument");
  TOME_CHECK(x_dtype == TOME_BF16 || x_dtype == TOME_F32, TOME_ERR_INVALID, "add_pos_embedding: bad dtype");
  const long long tc8 = (long long)tokens * channels / 8, n8 = tc8 * batch;
  ProfScope prof(PROF_OTHER, 0.0, 1, stream);
  if (x_dtype == TOME_F32)
    launch_k(add_pos_kernel<true>, ew_grid(n8, 256), 256, 0, stream, n8, tc8, x, pos_embedding, reinterpret_cast<__nv_bfloat16*>(y));
  else
    launch_k(add_pos_kernel<false>, ew_grid(n8, 256), 256, 0, stream, n8, tc8, x, pos_embedding, reinterpret_cast<__nv_bfloat16*>(y));
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_pos_embedding_bwd(int batch, int tokens, int channels, const void* dy, float* dpe, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && channels > 0 && channels % 8 == 0 && dy && dpe, TOME_ERR_INVALID,
             "pos_embedding_bwd: bad argument");
  const long long tc8 = (long long)tokens * channels / 8;
  ProfScope prof(PROF_OTHER, 0.0, 1, stream);
  launch_k(pos_bwd_kernel, (unsigned)((tc8 + 127) / 128), 128, 0, stream, batch, tc8, reinterpret_cast<const __nv_bfloat16*>(dy), dpe);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_chain_row_maps(int batch, int layers, const int32_t* const* row_maps_host, const int* tokens_host,
                                   const int32_t* readout_idx, int n_readout, int32_t* origin, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && layers >= 0 && layers <= MAX_CHAIN, TOME_ERR_INVALID, "chain_row_maps: layers must be in [0, %d]", MAX_CHAIN);
  TOME_CHECK(n_readout > 0 && readout_idx && origin && (layers == 0 || (row_maps_host && tokens_host)), TOME_ERR_INVALID,
             "chain_row_maps: null argument");
  ChainArgs a;
  for (int l = 0; l < MAX_CHAIN; ++l) {
    a.maps[l] = l < layers ? row_maps_host[l] : nullptr;
    a.tokens[l] = l < layers ? tokens_host[l] : 0;
  }
  const int n = batch * n_readout;
  ProfScope prof(PROF_OTHER, 0.0, 1, stream);
  launch_k(chain_kernel, ceil_div(n, 128), 128, 0, stream, batch, layers, a, readout_idx, n_readout, origin);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_readout_mse(int batch, int tokens, int channels, int n_readout, const void* x, const int32_t* origin,
                                const float* target, float* loss, void* dx, float* out, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && channels > 0 && n_readout > 0 && x && origin, TOME_ERR_INVALID, "readout_mse: bad argument");
  TOME_CHECK(!(loss || dx) || target, TOME_ERR_INVALID, "readout_mse: loss / dx need a target");
  ProfScope prof(PROF_OTHER, 0.0, loss ? 2 : 1, stream);
  if (dx) TOME_CUDA(cudaMemsetAsync(dx, 0, (size_t)batch * tokens * channels * 2, stream));
  launch_k(readout_mse_kernel, batch, 256, 0, stream, batch, tokens, channels, n_readout, reinterpret_cast<const __nv_bfloat16*>(x),
                                                origin, target, loss, reinterpret_cast<__nv_bfloat16*>(dx), out);
  TOME_CUDA(cudaGetLastError());
  if (loss) {
    launch_k(loss_final_kernel, 1, 1, 0, stream, batch, 1.0f / ((float)batch * n_readout * channels), loss);
    TOME_CUDA(cudaGetLastError());
  }
  return TOME_OK;
}

extern "C" int tome_adamw_step(long long n, float* param, const float* grad, float* m, float* v, void* bf16_copy, float lr,
                               float beta1, float beta2, float eps, float weight_decay, float grad_scale, int step,
                               void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(n > 0 && param && grad && m && v && step >= 1, TOME_ERR_INVALID, "adamw_step: bad argument");
  ProfScope prof(PROF_OTHER, 0.0, 1, stream);
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  launch_k(adamw_kernel, ew_grid(n, 256), 256, 0, stream, n, param, grad, m, v, reinterpret_cast<__nv_bfloat16*>(bf16_copy), lr, beta1,
                                                    beta2, eps, weight_decay, grad_scale, bc1, bc2);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_cast_f32_to_bf16(long long n, const float* src, void* dst, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(n > 0 && src && dst, TOME_ERR_INVALID, "cast: bad argument");
  ProfScope prof(PROF_OTHER, 0.0, 1, stream);
  launch_k(cast_kernel, ew_grid(n, 256), 256, 0, stream, n, src, reinterpret_cast<__nv_bfloat16*>(dst));
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
