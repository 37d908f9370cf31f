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

// ---- AdamW with optional global-norm clipping, non-finite skipping and a weight-decay mask ----
// The norm is a fixed-order reduction: NORM_CHUNKS contiguous chunks (a partition fixed at compile time, independent of the
// SM count and of tome_gemm_set_sm_limit), each summed in fp32 by one CTA through a fixed tree, then the partials added in
// index order in fp64 by one CTA.  The same gradient bits therefore give the same norm bits on every GPU and every rank.
constexpr int NORM_CHUNKS = 1024;
constexpr int NORM_THREADS = 256;
static_assert(NORM_CHUNKS == 4 * NORM_THREADS, "adam_control_kernel sums four partials per thread");

struct AdamControl {   // written by adam_control_kernel, read by every adamw_kernel CTA
  float scale;         // grad_scale times the clip factor
  float bc1, bc2;      // bias corrections of this step
  int skip;            // 1: this step is skipped
};

struct DecayRanges {   // n < 0: weight decay everywhere; else only inside the n sorted half-open ranges [lo, hi)
  int n;
  long long lo[TOME_ADAMW_MAX_DECAY_RANGES], hi[TOME_ADAMW_MAX_DECAY_RANGES];
};

// fixed-shape tree over one CTA of NORM_THREADS: warp butterflies, then warp 0 over the 8 warp sums
__device__ __forceinline__ float block_sum_fixed(float s, float* red) {
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x < 32) {
    t = threadIdx.x < NORM_THREADS / 32 ? red[threadIdx.x] : 0.f;
    t = warp_sum(t);
  }
  return t;   // valid in thread 0
}

// partial[c] = sum over chunk c of (gs * g)^2 in fp32, or NaN when the chunk holds a NaN / Inf.  g is 16-byte aligned.
__global__ void __launch_bounds__(NORM_THREADS) grad_sumsq_kernel(long long n, const float* __restrict__ g, float gs,
                                                                  float* __restrict__ partial) {
  __shared__ float red[NORM_THREADS / 32];
  const long long n4 = n / 4, per = (n4 + NORM_CHUNKS - 1) / NORM_CHUNKS;
  const long long lo = blockIdx.x * per, hi = min(lo + per, n4);
  float s = 0.f;
  bool bad = false;
  for (long long i = lo + threadIdx.x; i < hi; i += NORM_THREADS) {
    const uint4 u = ld_nc_v4(reinterpret_cast<const uint4*>(g) + i);
    const float x0 = __uint_as_float(u.x) * gs, x1 = __uint_as_float(u.y) * gs;
    const float x2 = __uint_as_float(u.z) * gs, x3 = __uint_as_float(u.w) * gs;
    bad |= !(isfinite(x0) && isfinite(x1) && isfinite(x2) && isfinite(x3));
    s = fmaf(x0, x0, s); s = fmaf(x1, x1, s); s = fmaf(x2, x2, s); s = fmaf(x3, x3, s);
  }
  if (blockIdx.x == NORM_CHUNKS - 1 && threadIdx.x < n - 4 * n4) {   // the n % 4 tail
    const float x = g[4 * n4 + threadIdx.x] * gs;
    bad |= !isfinite(x);
    s = fmaf(x, x, s);
  }
  bad = __syncthreads_or(bad);
  const float t = block_sum_fixed(s, red);
  if (threadIdx.x == 0) partial[blockIdx.x] = bad ? __int_as_float(0x7fc00000) : t;
}

// One CTA: the norm from the partials (fp64, fixed order), the clip factor, the skip decision, the bias corrections and the
// step counters.  partial == NULL: no norm this step (only the counters are used).
__global__ void __launch_bounds__(NORM_THREADS) adam_control_kernel(const float* __restrict__ partial, float gs, float max_norm,
                                                                    int skip_nonfinite, float b1, float b2, float bc1, float bc2,
                                                                    float* __restrict__ grad_norm, int* __restrict__ steps,
                                                                    AdamControl* __restrict__ ctl) {
  __shared__ double red[NORM_THREADS];
  double s = 0.0;
  if (partial) {
#pragma unroll
    for (int k = 0; k < 4; ++k) s += (double)partial[4 * threadIdx.x + k];
  }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int w = NORM_THREADS / 2; w > 0; w >>= 1) {
    if (threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
    __syncthreads();
  }
  if (threadIdx.x != 0) return;
  const double tot = red[0];
  const float norm = (float)sqrt(tot);
  const bool skip = skip_nonfinite && isnan(tot);   // a NaN partial marks a non-finite element; Inf is a finite overflow
  if (partial && grad_norm) *grad_norm = norm;
  // optax.clip_by_global_norm: unchanged below max_norm, else scaled by max_norm / norm (no epsilon)
  const float clip = (partial && max_norm > 0.f && !(norm < max_norm)) ? max_norm / norm : 1.f;
  if (steps) {   // bias correction counts applied steps only (optax.apply_if_finite leaves the inner state alone); in fp64,
                 // since 1 - b2^t cancels: an fp32 power would carry its rounding error into early steps 500-fold
    const int t = steps[0] + 1;
    bc1 = (float)(1.0 - pow((double)b1, (double)t));
    bc2 = (float)(1.0 - pow((double)b2, (double)t));
    steps[skip ? 1 : 0] += 1;
  }
  *ctl = AdamControl{gs * clip, bc1, bc2, skip ? 1 : 0};
}

// ctl == NULL: the host's scale and bias corrections (the ABI-16 step).  Decayed elements: p -= lr * (m^ / (sqrt(v^) + eps)
// + wd * p); others the same with wd = 0, which adds an exact zero.
__global__ void adamw_kernel(long long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                             float* __restrict__ v, __nv_bfloat16* __restrict__ w16, float lr, float b1, float b2, float eps,
                             float wd, float gs, float bc1, float bc2, const AdamControl* __restrict__ ctl,
                             const __grid_constant__ DecayRanges dr) {
  if (ctl) {
    const AdamControl c = *ctl;
    if (c.skip) return;
    gs = c.scale;
    bc1 = c.bc1;
    bc2 = c.bc2;
  }
  int r = 0;   // first range whose end lies past i; i only grows, so r only advances
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float wdi = wd;
    if (dr.n >= 0) {
      while (r < dr.n && dr.hi[r] <= i) ++r;
      wdi = (r < dr.n && dr.lo[r] <= i) ? wd : 0.f;
    }
    const float gi = g[i] * gs;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    float pi = p[i];
    pi -= lr * ((mi / bc1) / (sqrtf(vi / bc2) + eps) + wdi * pi);
    p[i] = pi;
    if (w16) w16[i] = __float2bfloat16(pi);
  }
}

static size_t adamw_carve(uint8_t* base, float** partial, AdamControl** ctl) {
  Bump b{base};
  float* pp = b.take<float>(NORM_CHUNKS);
  AdamControl* cc = b.take<AdamControl>(1);
  if (partial) *partial = pp;
  if (ctl) *ctl = cc;
  return b.total();
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

extern "C" size_t tome_adamw_workspace_bytes(long long n) {
  return n > 0 ? adamw_carve(nullptr, nullptr, nullptr) : 0;
}

extern "C" int tome_adamw_step(long long n, float* param, const float* grad, float* m, float* v, void* bf16_copy, float lr,
                               float beta1, float beta2, float eps, float weight_decay, float grad_scale, int step,
                               const tome_adamw_opts_t* opts, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(n > 0 && param && grad && m && v && step >= 1, TOME_ERR_INVALID, "adamw_step: bad argument");
  DecayRanges dr;
  dr.n = -1;
  bool norm = false, control = false;
  if (opts) {
    const tome_adamw_opts_t& o = *opts;
    TOME_CHECK(isfinite(o.max_grad_norm) && o.max_grad_norm >= 0.f, TOME_ERR_INVALID,
               "adamw_step: max_grad_norm must be finite and >= 0 (got %g)", (double)o.max_grad_norm);
    TOME_CHECK(o.skip_nonfinite == 0 || o.skip_nonfinite == 1, TOME_ERR_INVALID, "adamw_step: skip_nonfinite must be 0 or 1");
    TOME_CHECK(!o.skip_nonfinite || o.steps, TOME_ERR_INVALID, "adamw_step: skip_nonfinite needs the steps counters");
    TOME_CHECK(o.n_decay_ranges >= 0 && o.n_decay_ranges <= TOME_ADAMW_MAX_DECAY_RANGES, TOME_ERR_INVALID,
               "adamw_step: n_decay_ranges must be in [0, %d] (got %d)", TOME_ADAMW_MAX_DECAY_RANGES, o.n_decay_ranges);
    TOME_CHECK(o.decay_ranges || o.n_decay_ranges == 0, TOME_ERR_INVALID, "adamw_step: n_decay_ranges > 0 with NULL decay_ranges");
    if (o.decay_ranges) {
      dr.n = o.n_decay_ranges;
      long long prev = 0;
      for (int k = 0; k < o.n_decay_ranges; ++k) {
        const long long lo = o.decay_ranges[2 * k], hi = o.decay_ranges[2 * k + 1];
        TOME_CHECK(lo < hi, TOME_ERR_INVALID, "adamw_step: decay range %d [%lld, %lld) is empty", k, lo, hi);
        TOME_CHECK(lo >= prev, TOME_ERR_INVALID, "adamw_step: decay range %d [%lld, %lld) is unsorted or overlaps the one before",
                   k, lo, hi);
        TOME_CHECK(hi <= n, TOME_ERR_INVALID, "adamw_step: decay range %d [%lld, %lld) lies outside [0, %lld)", k, lo, hi, n);
        dr.lo[k] = lo;
        dr.hi[k] = hi;
        prev = hi;
      }
    }
    norm = o.max_grad_norm > 0.f || o.skip_nonfinite || o.grad_norm;
    control = norm || o.steps;
    if (control) {
      const size_t need = tome_adamw_workspace_bytes(n);
      TOME_CHECK(o.workspace && o.workspace_bytes >= need && reinterpret_cast<uintptr_t>(o.workspace) % 16 == 0, TOME_ERR_INVALID,
                 "adamw_step: these options need a 16-byte aligned workspace of tome_adamw_workspace_bytes(n) = %zu bytes (got %zu)",
                 need, o.workspace ? o.workspace_bytes : (size_t)0);
    }
    TOME_CHECK(!norm || reinterpret_cast<uintptr_t>(grad) % 16 == 0, TOME_ERR_INVALID,
               "adamw_step: the norm pass reads grad in 16-byte vectors: grad must be 16-byte aligned");
  }
  ProfScope prof(PROF_OTHER, 0.0, 1 + (control ? 1 : 0) + (norm ? 1 : 0), stream);
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  AdamControl* ctl = nullptr;
  if (control) {
    float* partial = nullptr;
    adamw_carve(reinterpret_cast<uint8_t*>(opts->workspace), &partial, &ctl);
    if (norm) {
      launch_k(grad_sumsq_kernel, NORM_CHUNKS, NORM_THREADS, 0, stream, n, grad, grad_scale, partial);
      TOME_CUDA(cudaGetLastError());
    }
    launch_k(adam_control_kernel, 1, NORM_THREADS, 0, stream, norm ? partial : nullptr, grad_scale, opts->max_grad_norm,
             opts->skip_nonfinite, beta1, beta2, bc1, bc2, opts->grad_norm, opts->steps, ctl);
    TOME_CUDA(cudaGetLastError());
  }
  launch_k(adamw_kernel, ew_grid(n, 256), 256, 0, stream, n, param, grad, m, v, reinterpret_cast<__nv_bfloat16*>(bf16_copy), lr, beta1,
                                                    beta2, eps, weight_decay, grad_scale, bc1, bc2, ctl, dr);
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
