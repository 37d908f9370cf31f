// K11: the diffusion action head's training path (SURVEY.md 8(f) rank 3, the head octo_base.yaml selects).
//
//   cosine_beta_schedule / alpha_hats       action_heads/diffusion.py:16-26, 85-92   (host side: the caller passes alpha_hats)
//   DiffusionActionHead.denoise_loss        diffusion.py:114-143   noisy = sqrt(ah[t]) a + sqrt(1 - ah[t]) noise;
//                                                                   loss = mean_b sum_a 0.5 (pred - noise)^2  (optax.l2_loss)
//   DiffusionActionHead.predict_denoise_term diffusion.py:94-112   embeddings = mean(readouts, axis=-2)
//   OctoDenoise.__call__                    diffusion.py:52-64     x = [noisy | time_embedding | readout_embedding] -> MLPBlock
//   FourierFeatures.__call__                diffusion.py:29-50     x = 2 pi t w^T; [cos x | sin x] -> MLPBlock
//   MLPBlock (train=False here: the denoiser calls it without `train`, so its two Dropouts are inactive)
//                                           attention_blocks/attention.py:20-39   Dense -> relu -> Dense
//
// The random draws (time step, noise) are the caller's: jax's threefry stream cannot be reproduced, so `time` and `noise`
// are inputs.  The three wide Dense layers run on the tcgen05 GEMM (bf16 operands from the caller's bf16 parameter copy,
// fused bias / ReLU epilogues, ReLU-gated dgrad, fp32-accumulating wgrad); pooling, Fourier features, the 8-wide output
// Dense, the loss and their backward are small fp32 kernels with fixed summation orders.
#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int DH_THREADS = 256;

struct DiffDims {
  long long B, T, C, n, A, F, Ht, To, H, Dc;
};
static DiffDims diff_dims(const tome_diffusion_desc_t* d) {
  DiffDims s;
  s.B = d->batch; s.T = d->tokens; s.C = d->channels; s.n = d->n_readout; s.A = d->action_dim; s.F = d->fourier_dim;
  s.Ht = d->time_hidden; s.To = d->time_out; s.H = d->hidden; s.Dc = s.A + s.To + s.C;
  return s;
}
struct DiffOffsets {
  long long fourier, tw1, tb1, tw2, tb2, w1, b1, w2, b2, end;
};
static DiffOffsets diff_offsets(const tome_diffusion_desc_t* d) {
  const DiffDims s = diff_dims(d);
  DiffOffsets o;
  long long p = 0;
  o.fourier = p; p += s.F / 2;
  o.tw1 = p; p += s.F * s.Ht;
  o.tb1 = p; p += s.Ht;
  o.tw2 = p; p += s.Ht * s.To;
  o.tb2 = p; p += s.To;
  o.w1 = p; p += s.Dc * s.H;
  o.b1 = p; p += s.H;
  o.w2 = p; p += s.H * s.A;
  o.b2 = p; p += s.A;
  o.end = p;
  return o;
}

struct DiffWs {
  __nv_bfloat16 *ff, *th, *cat, *h, *dh, *dcat, *dth;
  float *dpred, *colsum, *dff;
  size_t total;
};
static DiffWs diff_ws(const tome_diffusion_desc_t* d, void* base) {
  const DiffDims s = diff_dims(d);
  Bump b{reinterpret_cast<uint8_t*>(base)};
  DiffWs w;
  w.ff = b.take<__nv_bfloat16>(s.B * s.F);
  w.th = b.take<__nv_bfloat16>(s.B * s.Ht);
  w.cat = b.take<__nv_bfloat16>(s.B * s.Dc);
  w.h = b.take<__nv_bfloat16>(s.B * s.H);
  w.dpred = b.take<float>(s.B * s.A);
  w.dh = b.take<__nv_bfloat16>(s.B * s.H);
  w.dcat = b.take<__nv_bfloat16>(s.B * s.Dc);
  w.dth = b.take<__nv_bfloat16>(s.B * s.Ht);
  w.dff = b.take<float>(s.B * s.F);   // fp32: it feeds the Fourier-kernel gradient, a sum with cancellation
  long long widest = s.H > s.Ht ? s.H : s.Ht;
  if (s.To > widest) widest = s.To;
  w.colsum = b.take<float>((size_t)tome_colsum_workspace_rows((int)s.B) * widest);
  w.total = b.total();
  return w;
}

// cat[b] = [noisy action | (time embedding: written later by the GEMM) | mean of the readout rows];  ff[b] = [cos | sin](2 pi t w)
__global__ void __launch_bounds__(DH_THREADS)
diff_prep_kernel(const tome_diffusion_desc_t d, const __nv_bfloat16* __restrict__ x, const int32_t* __restrict__ origin,
                 const float* __restrict__ fourier, const float* __restrict__ actions, const float* __restrict__ noise,
                 const int32_t* __restrict__ time, const float* __restrict__ alpha_hats, __nv_bfloat16* __restrict__ ff,
                 __nv_bfloat16* __restrict__ cat) {
  const int b = blockIdx.x, C = d.channels, A = d.action_dim, F2 = d.fourier_dim / 2, n = d.n_readout;
  const long long Dc = (long long)A + d.time_out + C;
  const int t = min(max(time[b], 0), d.diffusion_steps - 1);
  const float ah = alpha_hats[t];
  const float a1 = sqrtf(ah), a2 = sqrtf(1.0f - ah);                       // diffusion.py:131-133
  for (int a = threadIdx.x; a < A; a += DH_THREADS)
    cat[b * Dc + a] = __float2bfloat16(a1 * actions[(long long)b * A + a] + a2 * noise[(long long)b * A + a]);   // :134
  const float inv_n = 1.0f / (float)n;
  for (int c = threadIdx.x; c < C; c += DH_THREADS) {                      // :107 jnp.mean(readouts, axis=-2)
    float s = 0.f;
    for (int j = 0; j < n; ++j) s += __bfloat162float(x[((long long)b * d.tokens + origin[b * n + j]) * C + c]);
    cat[b * Dc + A + d.time_out + c] = __float2bfloat16(s * inv_n);
  }
  for (int j = threadIdx.x; j < F2; j += DH_THREADS) {                     // :44-45
    const float ang = 6.283185307179586f * (float)t * fourier[j];
    float sn, cs;
    sincosf(ang, &sn, &cs);
    ff[(long long)b * d.fourier_dim + j] = __float2bfloat16(cs);
    ff[(long long)b * d.fourier_dim + F2 + j] = __float2bfloat16(sn);
  }
}

// pred[b] = h[b] W2 + b2 (fp32 weights); loss_b = sum_a 0.5 (pred - noise)^2; dpred = (pred - noise) / B
__global__ void __launch_bounds__(DH_THREADS)
diff_out_kernel(const tome_diffusion_desc_t d, const __nv_bfloat16* __restrict__ h, const float* __restrict__ w2,
                const float* __restrict__ b2, const float* __restrict__ noise, float* __restrict__ pred,
                float* __restrict__ loss, float* __restrict__ dpred) {
  __shared__ float lsum[DH_THREADS / 32];
  const int b = blockIdx.x, H = d.hidden, A = d.action_dim;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float part = 0.f;
  for (int a = warp; a < A; a += DH_THREADS / 32) {
    float s = 0.f;
    for (int k = lane; k < H; k += 32) s = fmaf(__bfloat162float(h[(long long)b * H + k]), w2[(long long)k * A + a], s);
    s = warp_sum(s);
    if (lane == 0) {
      const float p = s + b2[a];
      pred[(long long)b * A + a] = p;
      if (noise) {
        const float diff = p - noise[(long long)b * A + a];
        part += 0.5f * diff * diff;
        if (dpred) dpred[(long long)b * A + a] = diff / (float)d.batch;
      }
    }
  }
  if (lane == 0) lsum[warp] = part;
  __syncthreads();
  if (threadIdx.x == 0 && loss) {
    float t = 0.f;
    for (int w = 0; w < DH_THREADS / 32; ++w) t += lsum[w];
    loss[1 + b] = t;
  }
}
__global__ void diff_loss_final_kernel(int B, float* loss) {
  float t = 0.f;
  for (int b = 0; b < B; ++b) t += loss[1 + b];
  loss[0] = t / (float)B;
}

// dW2[k, a] += sum_b h[b,k] dpred[b,a];  db2[a] += sum_b dpred[b,a];  dh[b,k] = relu'(h) * sum_a dpred[b,a] W2[k,a]
__global__ void __launch_bounds__(DH_THREADS)
diff_out_bwd_kernel(const tome_diffusion_desc_t d, const __nv_bfloat16* __restrict__ h, const float* __restrict__ w2,
                    const float* __restrict__ dpred, float* __restrict__ dw2, float* __restrict__ db2,
                    __nv_bfloat16* __restrict__ dh) {
  const int H = d.hidden, A = d.action_dim, B = d.batch;
  const long long i = blockIdx.x * (long long)DH_THREADS + threadIdx.x;
  if (i < (long long)H * A) {                       // weight gradient, fixed order over the batch
    const int k = (int)(i / A), a = (int)(i - (long long)k * A);
    float s = 0.f;
    for (int b = 0; b < B; ++b) s = fmaf(__bfloat162float(h[(long long)b * H + k]), dpred[(long long)b * A + a], s);
    dw2[i] += s;
  } else if (i < (long long)H * A + A) {
    const int a = (int)(i - (long long)H * A);
    float s = 0.f;
    for (int b = 0; b < B; ++b) s += dpred[(long long)b * A + a];
    db2[a] += s;
  }
  for (long long j = i; j < (long long)B * H; j += (long long)gridDim.x * DH_THREADS) {
    const int b = (int)(j / H), k = (int)(j - (long long)b * H);
    float s = 0.f;
    if (__bfloat162float(h[j]) > 0.f)
      for (int a = 0; a < A; ++a) s = fmaf(dpred[(long long)b * A + a], w2[(long long)k * A + a], s);
    dh[j] = __float2bfloat16(s);
  }
}

// dx rows of the readouts <- dcat[:, A+To:] / n;   d fourier[j] += sum_b 2 pi t_b (cos * dsin - sin * dcos)
__global__ void __launch_bounds__(DH_THREADS)
diff_scatter_kernel(const tome_diffusion_desc_t d, const int32_t* __restrict__ origin, const __nv_bfloat16* __restrict__ dcat,
                    __nv_bfloat16* __restrict__ dx) {
  const int b = blockIdx.x, C = d.channels, n = d.n_readout;
  const long long Dc = (long long)d.action_dim + d.time_out + C;
  const float inv_n = 1.0f / (float)n;
  for (int c = threadIdx.x; c < C; c += DH_THREADS) {
    const float g = __bfloat162float(dcat[b * Dc + d.action_dim + d.time_out + c]) * inv_n;
    for (int j = 0; j < n; ++j) {
      __nv_bfloat16* p = dx + ((long long)b * d.tokens + origin[b * n + j]) * C + c;
      *p = __float2bfloat16(__bfloat162float(*p) + g);
    }
  }
}
__global__ void __launch_bounds__(DH_THREADS)
diff_fourier_bwd_kernel(const tome_diffusion_desc_t d, const int32_t* __restrict__ time, const float* __restrict__ fourier,
                        const float* __restrict__ dff, float* __restrict__ dfourier) {
  const int j = blockIdx.x * DH_THREADS + threadIdx.x, F2 = d.fourier_dim / 2;
  if (j >= F2) return;
  const float w = fourier[j];
  float s = 0.f;
  for (int b = 0; b < d.batch; ++b) {
    const float k = 6.283185307179586f * (float)time[b];
    float sn, cs;
    sincosf(k * w, &sn, &cs);
    const float dcos = dff[(long long)b * d.fourier_dim + j];
    const float dsin = dff[(long long)b * d.fourier_dim + F2 + j];
    s = fmaf(k, cs * dsin - sn * dcos, s);
  }
  dfourier[j] += s;
}

static int check_diff(const tome_diffusion_desc_t* d) {
  TOME_CHECK(d != nullptr, TOME_ERR_INVALID, "diffusion_head: null descriptor");
  TOME_CHECK(d->batch > 0, TOME_ERR_INVALID, "diffusion_head: batch must be positive");
  TOME_CHECK(d->tokens > 0 && d->n_readout > 0 && d->channels > 0 && d->channels % 8 == 0, TOME_ERR_INVALID, "diffusion_head: bad shape");
  TOME_CHECK(d->action_dim > 0 && d->action_dim % 8 == 0, TOME_ERR_INVALID,
             "diffusion_head: action_dim (%d) must be a multiple of 8 (16-byte rows of the concatenated input; diffusion.yaml uses 8)", d->action_dim);
  TOME_CHECK(d->fourier_dim > 0 && d->fourier_dim % 16 == 0, TOME_ERR_INVALID, "diffusion_head: fourier_dim must be a multiple of 16");
  TOME_CHECK(d->time_hidden > 0 && d->time_hidden % 8 == 0 && d->time_out > 0 && d->time_out % 8 == 0 && d->hidden > 0 && d->hidden % 8 == 0,
             TOME_ERR_INVALID, "diffusion_head: time_hidden, time_out and hidden must be positive multiples of 8");
  TOME_CHECK(d->diffusion_steps >= 1, TOME_ERR_INVALID, "diffusion_head: diffusion_steps must be >= 1");
  return TOME_OK;
}

static int diff_gemm(cudaStream_t st, int m, int n, int k, const void* a, long long lda, int a_major, const void* b, long long ldb,
                     int b_major, void* c, long long ldc, int c_dtype, const float* bias, int relu, const void* gate, long long ldg,
                     int accumulate) {
  tome_gemm_args_t g;
  memset(&g, 0, sizeof(g));
  g.m = m; g.n = n; g.k = k;
  g.a = a; g.lda = lda; g.a_major = a_major;
  g.b = b; g.ldb = ldb; g.b_major = b_major;
  g.c = c; g.ldc = ldc; g.c_dtype = c_dtype;
  g.bias = bias; g.relu = relu;
  g.gate = gate; g.ldg = ldg; g.gate_scale = 1.0f;
  g.k_splits = 1;   // the reductions here are a few hundred long: no split-K, no workspace
  g.accumulate = accumulate;
  return tome_gemm_bf16(&g, nullptr, 0, st);
}

}  // namespace tome

using namespace tome;

#define DH_RC(x) do { int rc__ = (x); if (rc__ != TOME_OK) return rc__; } while (0)

extern "C" long long tome_diffusion_head_param_count(const tome_diffusion_desc_t* d) {
  clear_error();
  if (check_diff(d) != TOME_OK) return -1;
  return diff_offsets(d).end;
}
extern "C" long long tome_diffusion_head_param_offset(const tome_diffusion_desc_t* d, int which) {
  clear_error();
  if (check_diff(d) != TOME_OK) return -1;
  const DiffOffsets o = diff_offsets(d);
  const long long v[10] = {o.fourier, o.tw1, o.tb1, o.tw2, o.tb2, o.w1, o.b1, o.w2, o.b2, o.end};
  return which >= 0 && which < 10 ? v[which] : -1;
}
extern "C" size_t tome_diffusion_head_workspace_bytes(const tome_diffusion_desc_t* d) {
  clear_error();
  if (check_diff(d) != TOME_OK) return 0;
  return diff_ws(d, nullptr).total;
}

extern "C" int tome_diffusion_head_fwd(const tome_diffusion_desc_t* d, const float* params_f32, const void* params_bf16_,
                                       const void* x, const int32_t* origin, const float* actions, const float* noise,
                                       const int32_t* time, const float* alpha_hats, float* pred, float* loss,
                                       void* workspace, size_t workspace_bytes, void* stream_) {
  clear_error();
  cudaStream_t st = (cudaStream_t)stream_;
  DH_RC(check_diff(d));
  TOME_CHECK(params_f32 && params_bf16_ && x && origin && actions && noise && time && alpha_hats && pred && workspace, TOME_ERR_INVALID,
             "diffusion_head_fwd: null argument");
  TOME_CHECK(((uintptr_t)workspace & 255) == 0 && workspace_bytes >= diff_ws(d, nullptr).total, TOME_ERR_INVALID,
             "diffusion_head_fwd: workspace too small or not 256-byte aligned");
  TOME_CHECK(((uintptr_t)params_bf16_ & 15) == 0, TOME_ERR_INVALID, "diffusion_head_fwd: params_bf16 must be 16-byte aligned");
  const DiffDims s = diff_dims(d);
  const DiffOffsets o = diff_offsets(d);
  const DiffWs w = diff_ws(d, workspace);
  const __nv_bfloat16* pw = reinterpret_cast<const __nv_bfloat16*>(params_bf16_);
  const int B = (int)s.B;
  {
    ProfScope prof(PROF_OTHER, 0.0, 1, st);
    launch_k(diff_prep_kernel, B, DH_THREADS, 0, st, *d, reinterpret_cast<const __nv_bfloat16*>(x), origin, params_f32 + o.fourier, actions,
                                               noise, time, alpha_hats, w.ff, w.cat);
    TOME_CUDA(cudaGetLastError());
  }
  // time encoder MLPBlock: th = relu(ff tw1 + tb1); time embedding = th tw2 + tb2, written straight into its slot of `cat`
  DH_RC(diff_gemm(st, B, (int)s.Ht, (int)s.F, w.ff, s.F, TOME_MAJOR_K, pw + o.tw1, s.Ht, TOME_MAJOR_MN, w.th, s.Ht, TOME_BF16,
                  params_f32 + o.tb1, 1, nullptr, 0, 0));
  DH_RC(diff_gemm(st, B, (int)s.To, (int)s.Ht, w.th, s.Ht, TOME_MAJOR_K, pw + o.tw2, s.To, TOME_MAJOR_MN, w.cat + s.A, s.Dc, TOME_BF16,
                  params_f32 + o.tb2, 0, nullptr, 0, 0));
  // denoiser MLPBlock: h = relu(cat w1 + b1); pred = h w2 + b2
  DH_RC(diff_gemm(st, B, (int)s.H, (int)s.Dc, w.cat, s.Dc, TOME_MAJOR_K, pw + o.w1, s.H, TOME_MAJOR_MN, w.h, s.H, TOME_BF16,
                  params_f32 + o.b1, 1, nullptr, 0, 0));
  ProfScope prof(PROF_OTHER, 0.0, loss ? 2 : 1, st);
  launch_k(diff_out_kernel, B, DH_THREADS, 0, st, *d, w.h, params_f32 + o.w2, params_f32 + o.b2, noise, pred, loss, w.dpred);
  TOME_CUDA(cudaGetLastError());
  if (loss) {
    launch_k(diff_loss_final_kernel, 1, 1, 0, st, B, loss);
    TOME_CUDA(cudaGetLastError());
  }
  return TOME_OK;
}

extern "C" int tome_diffusion_head_bwd(const tome_diffusion_desc_t* d, const float* params_f32, const void* params_bf16_,
                                       const int32_t* origin, const int32_t* time, void* workspace, float* grads_f32, void* dx,
                                       void* stream_) {
  clear_error();
  cudaStream_t st = (cudaStream_t)stream_;
  DH_RC(check_diff(d));
  TOME_CHECK(params_f32 && params_bf16_ && origin && time && workspace && grads_f32, TOME_ERR_INVALID, "diffusion_head_bwd: null argument");
  TOME_CHECK(((uintptr_t)workspace & 255) == 0, TOME_ERR_INVALID, "diffusion_head_bwd: workspace must be 256-byte aligned");
  const DiffDims s = diff_dims(d);
  const DiffOffsets o = diff_offsets(d);
  const DiffWs w = diff_ws(d, workspace);
  const __nv_bfloat16* pw = reinterpret_cast<const __nv_bfloat16*>(params_bf16_);
  float* gr = grads_f32;
  const int B = (int)s.B;
  {
    ProfScope prof(PROF_OTHER, 0.0, 1, st);
    const long long nthr = s.H * s.A + s.A > s.B * s.H ? s.H * s.A + s.A : s.B * s.H;
    launch_k(diff_out_bwd_kernel, (unsigned)((nthr + DH_THREADS - 1) / DH_THREADS), DH_THREADS, 0, st, 
        *d, w.h, params_f32 + o.w2, w.dpred, gr + o.w2, gr + o.b2, w.dh);
    TOME_CUDA(cudaGetLastError());
  }
  // denoiser Dense_0: dW1 += cat^T dh, db1 += colsum(dh), dcat = dh W1^T
  DH_RC(diff_gemm(st, (int)s.Dc, (int)s.H, B, w.cat, s.Dc, TOME_MAJOR_MN, w.dh, s.H, TOME_MAJOR_MN, gr + o.w1, s.H, TOME_F32, nullptr, 0,
                  nullptr, 0, 1));
  DH_RC(tome_colsum_bf16(B, (int)s.H, w.dh, s.H, gr + o.b1, 1, w.colsum, st));
  DH_RC(diff_gemm(st, B, (int)s.Dc, (int)s.H, w.dh, s.H, TOME_MAJOR_K, pw + o.w1, s.H, TOME_MAJOR_K, w.dcat, s.Dc, TOME_BF16, nullptr, 0,
                  nullptr, 0, 0));
  if (dx) {
    ProfScope prof(PROF_OTHER, 0.0, 2, st);
    TOME_CUDA(cudaMemsetAsync(dx, 0, (size_t)s.B * s.T * s.C * 2, st));
    launch_k(diff_scatter_kernel, B, DH_THREADS, 0, st, *d, origin, w.dcat, reinterpret_cast<__nv_bfloat16*>(dx));
    TOME_CUDA(cudaGetLastError());
  }
  // time encoder: dte = dcat[:, A:A+To];  dW_t2 += th^T dte, db_t2 += colsum(dte), dth = relu'(th) * (dte W_t2^T)
  const __nv_bfloat16* dte = w.dcat + s.A;
  DH_RC(diff_gemm(st, (int)s.Ht, (int)s.To, B, w.th, s.Ht, TOME_MAJOR_MN, dte, s.Dc, TOME_MAJOR_MN, gr + o.tw2, s.To, TOME_F32, nullptr, 0,
                  nullptr, 0, 1));
  DH_RC(tome_colsum_bf16(B, (int)s.To, dte, s.Dc, gr + o.tb2, 1, w.colsum, st));
  DH_RC(diff_gemm(st, B, (int)s.Ht, (int)s.To, dte, s.Dc, TOME_MAJOR_K, pw + o.tw2, s.To, TOME_MAJOR_K, w.dth, s.Ht, TOME_BF16, nullptr, 0,
                  w.th, s.Ht, 0));
  DH_RC(diff_gemm(st, (int)s.F, (int)s.Ht, B, w.ff, s.F, TOME_MAJOR_MN, w.dth, s.Ht, TOME_MAJOR_MN, gr + o.tw1, s.Ht, TOME_F32, nullptr, 0,
                  nullptr, 0, 1));
  DH_RC(tome_colsum_bf16(B, (int)s.Ht, w.dth, s.Ht, gr + o.tb1, 1, w.colsum, st));
  DH_RC(diff_gemm(st, B, (int)s.F, (int)s.Ht, w.dth, s.Ht, TOME_MAJOR_K, pw + o.tw1, s.Ht, TOME_MAJOR_K, w.dff, s.F, TOME_F32, nullptr, 0,
                  nullptr, 0, 0));
  ProfScope prof(PROF_OTHER, 0.0, 1, st);
  launch_k(diff_fourier_bwd_kernel, (unsigned)((s.F / 2 + DH_THREADS - 1) / DH_THREADS), DH_THREADS, 0, st, *d, time, params_f32 + o.fourier,
                                                                                                      w.dff, gr + o.fourier);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// One step of the sampler's update (DiffusionActionHead.predict_action, action_heads/diffusion.py:182-190; algorithm 2 of
// arXiv:2006.11239):  out = clip(c1 * (sample - c2 * denoise_term) + c3 * noise, -clip, clip), the coefficients taken from
// the schedule by the caller (c1 = 1 / sqrt(alpha_t), c2 = (1 - alpha_t) / sqrt(1 - alpha_hat_t), c3 = sqrt(beta_t)).
namespace tome {
__global__ void ddpm_step_kernel(long long n, const float* __restrict__ sample, const float* __restrict__ eps,
                                 const float* __restrict__ noise, float c1, float c2, float c3, float clip, float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = c1 * (sample[i] - c2 * eps[i]) + c3 * noise[i];
  out[i] = fminf(fmaxf(v, -clip), clip);
}
}  // namespace tome

extern "C" int tome_ddpm_step(long long n, const float* sample, const float* denoise_term, const float* noise, float c1, float c2,
                              float c3, float clip, float* out, void* stream_) {
  clear_error();
  cudaStream_t st = (cudaStream_t)stream_;
  TOME_CHECK(n > 0 && sample && denoise_term && noise && out, TOME_ERR_INVALID, "ddpm_step: bad argument");
  TOME_CHECK(clip > 0.f, TOME_ERR_INVALID, "ddpm_step: clip must be positive");
  ProfScope prof(PROF_OTHER, 0.0, 1, st);
  launch_k(tome::ddpm_step_kernel, (unsigned)((n + 255) / 256), 256, 0, st, n, sample, denoise_term, noise, c1, c2, c3, clip, out);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
