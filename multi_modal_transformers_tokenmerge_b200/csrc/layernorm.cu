// K8: LayerNorm exactly as the reference configures it (vanilla_decoder.yaml:7-13): reduction_axes=[1] -- the
// statistics run over the TOKEN axis for every (batch, feature) pair -- scale/bias per feature, epsilon 1e-6,
// flax's fast variance max(0, E[x^2] - E[x]^2).  axis = 2 is the conventional per-token LayerNorm (opt-in).
//
// HBM-bound.  axis 1: one CTA owns a (batch, 64-feature) slab = T rows x 128 bytes; 8 threads x 16 bytes cover a
// row segment (one full 128-byte line), 32 row groups stride over T.  The slab (T x 128 B <= 1 MB) is read twice, the
// second time from L2.  Also here: column sums (bias gradients) with the same slab walk.
#include <string.h>

#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int LN_THREADS = 256;
constexpr int LN_RG = 32;     // row groups
constexpr int LN_SLAB = 64;   // features per CTA (8 threads x 8 bf16)

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
  f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}

// ------------------------------------------------------------------------------------------------ axis 1 forward
__global__ void __launch_bounds__(LN_THREADS)
ln_seq_fwd_kernel(int T, int C, float eps, const __nv_bfloat16* __restrict__ x, const float* __restrict__ gamma,
                  const float* __restrict__ beta, __nv_bfloat16* __restrict__ y, float* __restrict__ mean,
                  float* __restrict__ rstd) {
  __shared__ float s_sum[LN_RG][LN_SLAB + 1];
  __shared__ float s_sq[LN_RG][LN_SLAB + 1];
  __shared__ float s_mean[LN_SLAB], s_rstd[LN_SLAB];
  const int b = blockIdx.y, c0 = blockIdx.x * LN_SLAB;
  const int ct = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = c0 + ct * 8;
  const bool active = c < C;
  const __nv_bfloat16* xb = x + (long long)b * T * C + c;
  float sum[8], sq[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) sum[i] = sq[i] = 0.f;
  if (active) {
    for (int t = rg; t < T; t += LN_RG) {
      float f[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(xb + (long long)t * C)), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sum[i] += f[i];
        sq[i] = fmaf(f[i], f[i], sq[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    s_sum[rg][ct * 8 + i] = sum[i];
    s_sq[rg][ct * 8 + i] = sq[i];
  }
  __syncthreads();
  if (threadIdx.x < LN_SLAB) {
    float a = 0.f, q = 0.f;
    for (int g = 0; g < LN_RG; ++g) {
      a += s_sum[g][threadIdx.x];
      q += s_sq[g][threadIdx.x];
    }
    const float mu = a / (float)T;
    const float var = fmaxf(q / (float)T - mu * mu, 0.f);
    const float rs = rsqrtf(var + eps);
    s_mean[threadIdx.x] = mu;
    s_rstd[threadIdx.x] = rs;
    if (c0 + threadIdx.x < C) {
      mean[(long long)b * C + c0 + threadIdx.x] = mu;
      rstd[(long long)b * C + c0 + threadIdx.x] = rs;
    }
  }
  __syncthreads();
  if (!active) return;
  float mu[8], sc[8], sh[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    mu[i] = s_mean[ct * 8 + i];
    sc[i] = s_rstd[ct * 8 + i] * gamma[c + i];
    sh[i] = beta[c + i];
  }
  __nv_bfloat16* yb = y + (long long)b * T * C + c;
  for (int t = rg; t < T; t += LN_RG) {
    float f[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(xb + (long long)t * C)), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = fmaf(f[i] - mu[i], sc[i], sh[i]);
    *reinterpret_cast<uint4*>(yb + (long long)t * C) = pack8(f);
  }
}

// ------------------------------------------------------------------------------------------------ axis 1 backward
// per (b, c):  A = sum_t dy,  Bq = sum_t dy * xhat;   dx = rstd*gamma*(dy - A/T - xhat*Bq/T) (+ dres)
// partial[0][b][c] = A (-> dbeta), partial[1][b][c] = Bq (-> dgamma); reduced over b by reduce_rows_kernel.
__global__ void __launch_bounds__(LN_THREADS)
ln_seq_bwd_kernel(int B, int T, int C, const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                  const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ rstd,
                  const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx, float* __restrict__ partial) {
  __shared__ float s_a[LN_RG][LN_SLAB + 1];
  __shared__ float s_b[LN_RG][LN_SLAB + 1];
  __shared__ float s_A[LN_SLAB], s_B[LN_SLAB];
  const int b = blockIdx.y, c0 = blockIdx.x * LN_SLAB;
  const int ct = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = c0 + ct * 8;
  const bool active = c < C;
  const long long base = (long long)b * T * C + c;
  float mu[8], rs[8];
  float sa[8], sb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sa[i] = sb[i] = 0.f;
    mu[i] = active ? mean[(long long)b * C + c + i] : 0.f;
    rs[i] = active ? rstd[(long long)b * C + c + i] : 0.f;
  }
  if (active) {
    for (int t = rg; t < T; t += LN_RG) {
      float fx[8], fd[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + base + (long long)t * C)), fx);
      unpack8(__ldg(reinterpret_cast<const uint4*>(dy + base + (long long)t * C)), fd);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sa[i] += fd[i];
        sb[i] = fmaf(fd[i], (fx[i] - mu[i]) * rs[i], sb[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    s_a[rg][ct * 8 + i] = sa[i];
    s_b[rg][ct * 8 + i] = sb[i];
  }
  __syncthreads();
  if (threadIdx.x < LN_SLAB) {
    float a = 0.f, q = 0.f;
    for (int g = 0; g < LN_RG; ++g) {
      a += s_a[g][threadIdx.x];
      q += s_b[g][threadIdx.x];
    }
    s_A[threadIdx.x] = a;
    s_B[threadIdx.x] = q;
    if (c0 + threadIdx.x < C) {
      partial[(long long)b * C + c0 + threadIdx.x] = a;
      partial[(long long)(B + b) * C + c0 + threadIdx.x] = q;
    }
  }
  __syncthreads();
  if (!active) return;
  const float inv_t = 1.0f / (float)T;
  float k0[8], k1[8], k2[8];  // dx = k0*dy + k1*xhat + k2
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float g = rs[i] * gamma[c + i];
    k0[i] = g;
    k1[i] = -g * s_B[ct * 8 + i] * inv_t;
    k2[i] = -g * s_A[ct * 8 + i] * inv_t;
  }
  for (int t = rg; t < T; t += LN_RG) {
    float fx[8], fd[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + base + (long long)t * C)), fx);
    unpack8(__ldg(reinterpret_cast<const uint4*>(dy + base + (long long)t * C)), fd);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = fmaf(k0[i], fd[i], fmaf(k1[i], (fx[i] - mu[i]) * rs[i], k2[i]));
    if (dres) {
      float fr[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(dres + base + (long long)t * C)), fr);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] += fr[i];
    }
    *reinterpret_cast<uint4*>(dx + base + (long long)t * C) = pack8(o);
  }
}

// out_p[n] (+)= sum_r ws[p][r, n]   for plane p = blockIdx.y (fp32, fixed order); planes are `plane_stride` floats apart.
// G row groups of 32 threads: each thread adds every G-th row of its column (four loads in flight), then the groups are added
// in order.  G = 8 for the short partial lists of LayerNorm / the chunked column sums, 32 for the per-tile partials a GEMM or
// attention-backward epilogue leaves (1 000+ rows: 22 -> 7 us).
template <int G>
__global__ void __launch_bounds__(32 * G)
reduce_rows_kernel(int R, int N, const float* __restrict__ ws, long long plane_stride, float* __restrict__ out0,
                   float* __restrict__ out1, int accumulate) {
  __shared__ float s[G][33];
  const int n = blockIdx.x * 32 + (threadIdx.x & 31), rgp = threadIdx.x >> 5;
  const float* w = ws + blockIdx.y * plane_stride;
  float* out = blockIdx.y ? out1 : out0;
  float a = 0.f;
  if (n < N) {
    int r = rgp;
    for (; r + 3 * G < R; r += 4 * G) {
      const float v0 = w[(long long)r * N + n], v1 = w[(long long)(r + G) * N + n], v2 = w[(long long)(r + 2 * G) * N + n],
                  v3 = w[(long long)(r + 3 * G) * N + n];
      a += v0; a += v1; a += v2; a += v3;
    }
    for (; r < R; r += G) a += w[(long long)r * N + n];
  }
  s[rgp][threadIdx.x & 31] = a;
  __syncthreads();
  if (rgp == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int g = 0; g < G; ++g) t += s[g][threadIdx.x & 31];
    out[n] = accumulate ? out[n] + t : t;
  }
}

// ------------------------------------------------------------------------------------------------ axis 1, shared-memory slabs
// The kernels above read their (batch, 64-feature) slab twice through L2 and keep few loads in flight per thread.  When
// the slab fits in shared memory (T <= LN_SMEM_T_FWD / _BWD) it is instead brought in ONCE by TMA -- 64-row boxes, one
// mbarrier per box, so the statistics pass starts on the first box while the others are still in flight -- and the
// second pass runs out of shared memory.  HBM/L2 traffic per element: forward 1 read + 1 write (was 2 + 1), backward
// 3 reads + 1 write (was 5 + 1).
constexpr int LN_BOX = 64;                       // token rows per TMA box (box = 64 rows x 128 bytes = 8 KB, 128B swizzle)
constexpr int LN_SMEM_T_FWD = 1536, LN_SMEM_T_BWD = 640;
__host__ __device__ constexpr int ln_boxes(int T) { return (T + LN_BOX - 1) / LN_BOX; }

__device__ __forceinline__ uint4 slab_ld(const uint8_t* slab, int t, int ct) {  // row t, 16-byte chunk ct of the swizzled slab
  return *reinterpret_cast<const uint4*>(slab + (size_t)t * 128 + ((ct ^ (t & 7)) << 4));
}

// CL: the tokens of one (batch, slab) are split over the gridDim.z CTAs of a thread-block cluster, `nb` boxes each (long
// sequences with few batch rows: one CTA per slab left most of the machine idle -- 0.08 of the HBM peak at T = 8192, B = 4).
// Every CTA reduces its own rows, the partial sums are exchanged through distributed shared memory and added in rank
// order by every CTA (identical statistics everywhere, deterministic), rank 0 stores them.
template <bool CL>
__global__ void __launch_bounds__(LN_THREADS)
ln_seq_fwd_smem_kernel(const __grid_constant__ CUtensorMap tm_x, int T, int C, int nb, float eps, const float* __restrict__ gamma,
                       const float* __restrict__ beta, __nv_bfloat16* __restrict__ y, float* __restrict__ mean,
                       float* __restrict__ rstd) {
  extern __shared__ uint8_t ln_smem_raw[];
  uint8_t* slab = ln_smem_raw + ((1024u - (smem_u32(ln_smem_raw) & 1023u)) & 1023u);
  const int t0 = CL ? (int)blockIdx.z * nb * LN_BOX : 0;   // first token row of this CTA
  uint64_t* bars = reinterpret_cast<uint64_t*>(slab + (size_t)nb * LN_BOX * 128);
  __shared__ float s_sum[LN_RG][LN_SLAB + 1];
  __shared__ float s_sq[LN_RG][LN_SLAB + 1];
  __shared__ float s_mean[LN_SLAB], s_rstd[LN_SLAB];
  __shared__ float s_part[2][LN_SLAB];   // CL: this CTA's partial sums, read by its cluster peers
  const int b = blockIdx.y, c0 = blockIdx.x * LN_SLAB;
  const int ct = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = c0 + ct * 8;
  const bool active = c < C;
  if (threadIdx.x == 0) {
    for (int k = 0; k < nb; ++k) mbar_init(&bars[k], 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < nb; ++k) {
      mbar_expect_tx(&bars[k], LN_BOX * 128);
      tma_load_3d(slab + (size_t)k * LN_BOX * 128, &tm_x, &bars[k], c0, t0 + k * LN_BOX, b);  // rows past T / columns past C arrive as zeros
    }
  }
  float sum[8], sq[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) sum[i] = sq[i] = 0.f;
  for (int k = 0; k < nb; ++k) {
    mbar_wait(&bars[k], 0);
#pragma unroll
    for (int u = 0; u < LN_BOX / LN_RG; ++u) {
      const int t = k * LN_BOX + u * LN_RG + rg;   // zero rows past T add nothing
      float f[8];
      unpack8(slab_ld(slab, t, ct), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sum[i] += f[i];
        sq[i] = fmaf(f[i], f[i], sq[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    s_sum[rg][ct * 8 + i] = sum[i];
    s_sq[rg][ct * 8 + i] = sq[i];
  }
  __syncthreads();
  if (CL) {
    if (threadIdx.x < LN_SLAB) {
      float a = 0.f, q = 0.f;
      for (int g = 0; g < LN_RG; ++g) {
        a += s_sum[g][threadIdx.x];
        q += s_sq[g][threadIdx.x];
      }
      s_part[0][threadIdx.x] = a;
      s_part[1][threadIdx.x] = q;
    }
    cluster_sync_all();   // every CTA's partials are in its shared memory
  }
  if (threadIdx.x < LN_SLAB) {
    float a = 0.f, q = 0.f;
    if (CL) {
      for (uint32_t r = 0; r < gridDim.z; ++r) {
        a += ld_shared_cluster_f32(map_to_cta(&s_part[0][threadIdx.x], r));
        q += ld_shared_cluster_f32(map_to_cta(&s_part[1][threadIdx.x], r));
      }
    } else {
      for (int g = 0; g < LN_RG; ++g) {
        a += s_sum[g][threadIdx.x];
        q += s_sq[g][threadIdx.x];
      }
    }
    const float mu = a / (float)T;
    const float var = fmaxf(q / (float)T - mu * mu, 0.f);
    const float rs = rsqrtf(var + eps);
    s_mean[threadIdx.x] = mu;
    s_rstd[threadIdx.x] = rs;
    if (c0 + threadIdx.x < C && (!CL || blockIdx.z == 0)) {
      mean[(long long)b * C + c0 + threadIdx.x] = mu;
      rstd[(long long)b * C + c0 + threadIdx.x] = rs;
    }
  }
  if (CL) cluster_sync_all();   // nobody leaves (or reuses s_part) while a peer may still read it
  else __syncthreads();
  if (!active) return;
  float mu[8], sc[8], sh[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    mu[i] = s_mean[ct * 8 + i];
    sc[i] = s_rstd[ct * 8 + i] * gamma[c + i];
    sh[i] = beta[c + i];
  }
  __nv_bfloat16* yb = y + (long long)b * T * C + c;
  const int t_end = min(T - t0, nb * LN_BOX);   // rows of this CTA that exist
#pragma unroll 4
  for (int t = rg; t < t_end; t += LN_RG) {
    float f[8];
    unpack8(slab_ld(slab, t, ct), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = fmaf(f[i] - mu[i], sc[i], sh[i]);
    st_na_v4(yb + (long long)(t0 + t) * C, pack8(f));
  }
}

// Backward keeps TWO slabs (x and dy), so it works on 32-feature slabs: 2 x T x 64 bytes (69 KB at T = 536) lets three
// CTAs share an SM, and their load / statistics / write phases overlap.  (With 64-feature slabs only one CTA fits and
// the kernel was slower than the L2 version.)  64-byte rows need no swizzle: 8 consecutive threads read 128 contiguous
// bytes.  Two CTAs with adjacent slabs fetch the two halves of the same 128-byte lines at about the same time.
constexpr int LNB_CPR = 4;                      // 16-byte chunks per row
constexpr int LNB_SLAB = LNB_CPR * 8;           // 32 features
constexpr int LNB_RG = LN_THREADS / LNB_CPR;    // 64 row groups = one 64-row box per step
static_assert(LNB_RG == LN_BOX, "one row per thread per box");
constexpr int LNB_MAX_BOXES = 10;               // the backward slab path keeps one residual row per box in registers: T <= 640

template <bool CL>   // as in the forward kernel: tokens split over a cluster, `nb` boxes (<= LNB_MAX_BOXES) per CTA
__global__ void __launch_bounds__(LN_THREADS)
ln_seq_bwd_smem_kernel(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_dy, int B, int T, int C, int nb,
                       const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ rstd,
                       const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx, float* __restrict__ partial) {
  extern __shared__ uint8_t ln_smem_raw[];
  uint8_t* slab_x = ln_smem_raw + ((128u - (smem_u32(ln_smem_raw) & 127u)) & 127u);
  const int t0 = CL ? (int)blockIdx.z * nb * LN_BOX : 0;   // first token row of this CTA
  constexpr int BOX_BYTES = LN_BOX * LNB_SLAB * 2;  // 4 KB
  uint8_t* slab_d = slab_x + (size_t)nb * BOX_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(slab_d + (size_t)nb * BOX_BYTES);
  __shared__ float s_a[LN_THREADS / 32][LNB_SLAB + 1];   // per-warp partial sums (the 8 row groups of a warp are shuffle-reduced first)
  __shared__ float s_b[LN_THREADS / 32][LNB_SLAB + 1];
  __shared__ float s_A[LNB_SLAB], s_B[LNB_SLAB];
  __shared__ float s_part[2][LNB_SLAB];   // CL: this CTA's partial sums, read by its cluster peers
  const int b = blockIdx.y, c0 = blockIdx.x * LNB_SLAB;
  const int ct = threadIdx.x & (LNB_CPR - 1), rg = threadIdx.x / LNB_CPR;
  const int c = c0 + ct * 8;
  const bool active = c < C;
  if (threadIdx.x == 0) {
    for (int k = 0; k < nb; ++k) mbar_init(&bars[k], 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int k = 0; k < nb; ++k) {
      mbar_expect_tx(&bars[k], 2 * BOX_BYTES);
      tma_load_3d(slab_x + (size_t)k * BOX_BYTES, &tm_x, &bars[k], c0, t0 + k * LN_BOX, b);  // rows past T / columns past C arrive as zeros
      tma_load_3d(slab_d + (size_t)k * BOX_BYTES, &tm_dy, &bars[k], c0, t0 + k * LN_BOX, b);
    }
  }
  // the residual-branch gradient rows this thread will add in the second pass: requested NOW, so their latency hides
  // behind the TMA loads and the statistics pass (nb <= LNB_MAX_BOXES on this path)
  const long long base = (long long)b * T * C + c;
  uint4 rv[LNB_MAX_BOXES];
#pragma unroll
  for (int k = 0; k < LNB_MAX_BOXES; ++k) {
    const int t = t0 + k * LN_BOX + rg;
    rv[k] = (dres && active && k < nb && t < T) ? ld_nc_v4(dres + base + (long long)t * C) : make_uint4(0u, 0u, 0u, 0u);
  }
  float mu[8], rs[8];
  float sa[8], sb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sa[i] = sb[i] = 0.f;
    mu[i] = active ? mean[(long long)b * C + c + i] : 0.f;
    rs[i] = active ? rstd[(long long)b * C + c + i] : 0.f;
  }
  const size_t my = (size_t)rg * (LNB_SLAB * 2) + ct * 16;  // this thread's 16 bytes inside a box
  for (int k = 0; k < nb; ++k) {
    mbar_wait(&bars[k], 0);
    float fx[8], fd[8];   // row k * 64 + rg; rows past T hold dy = 0 and add nothing
    unpack8(*reinterpret_cast<const uint4*>(slab_x + (size_t)k * BOX_BYTES + my), fx);
    unpack8(*reinterpret_cast<const uint4*>(slab_d + (size_t)k * BOX_BYTES + my), fd);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      sa[i] += fd[i];
      sb[i] = fmaf(fd[i], (fx[i] - mu[i]) * rs[i], sb[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {  // lanes l, l^4, l^8, l^16 hold the same features of different row groups
#pragma unroll
    for (int o = LNB_CPR; o < 32; o <<= 1) {
      sa[i] += __shfl_xor_sync(0xffffffffu, sa[i], o);
      sb[i] += __shfl_xor_sync(0xffffffffu, sb[i], o);
    }
  }
  if ((threadIdx.x & 31) < LNB_CPR) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      s_a[threadIdx.x >> 5][ct * 8 + i] = sa[i];
      s_b[threadIdx.x >> 5][ct * 8 + i] = sb[i];
    }
  }
  __syncthreads();
  if (CL) {
    if (threadIdx.x < LNB_SLAB) {
      float a = 0.f, q = 0.f;
#pragma unroll
      for (int g = 0; g < LN_THREADS / 32; ++g) {
        a += s_a[g][threadIdx.x];
        q += s_b[g][threadIdx.x];
      }
      s_part[0][threadIdx.x] = a;
      s_part[1][threadIdx.x] = q;
    }
    cluster_sync_all();
  }
  if (threadIdx.x < LNB_SLAB) {
    float a = 0.f, q = 0.f;
    if (CL) {
      for (uint32_t r = 0; r < gridDim.z; ++r) {
        a += ld_shared_cluster_f32(map_to_cta(&s_part[0][threadIdx.x], r));
        q += ld_shared_cluster_f32(map_to_cta(&s_part[1][threadIdx.x], r));
      }
    } else {
#pragma unroll
      for (int g = 0; g < LN_THREADS / 32; ++g) {
        a += s_a[g][threadIdx.x];
        q += s_b[g][threadIdx.x];
      }
    }
    s_A[threadIdx.x] = a;
    s_B[threadIdx.x] = q;
    if (c0 + threadIdx.x < C && (!CL || blockIdx.z == 0)) {
      partial[(long long)b * C + c0 + threadIdx.x] = a;
      partial[(long long)(B + b) * C + c0 + threadIdx.x] = q;
    }
  }
  if (CL) cluster_sync_all();   // nobody leaves while a peer may still read its partial sums
  else __syncthreads();
  if (!active) return;
  const float inv_t = 1.0f / (float)T;
  float k0[8], k1[8], k2[8];  // dx = k0*dy + k1*xhat + k2
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float g = rs[i] * gamma[c + i];
    k0[i] = g;
    k1[i] = -g * s_B[ct * 8 + i] * inv_t;
    k2[i] = -g * s_A[ct * 8 + i] * inv_t;
  }
#pragma unroll
  for (int k = 0; k < LNB_MAX_BOXES; ++k) {
    const int t = t0 + k * LN_BOX + rg;
    if (k < nb && t < T) {
      float fx[8], fd[8], o[8];
      unpack8(*reinterpret_cast<const uint4*>(slab_x + (size_t)k * BOX_BYTES + my), fx);
      unpack8(*reinterpret_cast<const uint4*>(slab_d + (size_t)k * BOX_BYTES + my), fd);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = fmaf(k0[i], fd[i], fmaf(k1[i], (fx[i] - mu[i]) * rs[i], k2[i]));
      if (dres) {
        float fr[8];
        unpack8(rv[k], fr);
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] += fr[i];
      }
      st_na_v4(dx + base + (long long)t * C, pack8(o));
    }
  }
}

// ------------------------------------------------------------------------------------------------ column sums
// ws[chunk, n] = sum over the rows of this chunk of x[m, n]
__global__ void __launch_bounds__(LN_THREADS)
colsum_partial_kernel(int M, int N, long long ldx, int rows_per_chunk, const __nv_bfloat16* __restrict__ x,
                      float* __restrict__ ws) {
  __shared__ float s_sum[LN_RG][LN_SLAB + 1];
  const int chunk = blockIdx.y, c0 = blockIdx.x * LN_SLAB;
  const int ct = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = c0 + ct * 8;
  const int m0 = chunk * rows_per_chunk, m1 = min(M, m0 + rows_per_chunk);
  float sum[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) sum[i] = 0.f;
  if (c < N) {
    for (int m = m0 + rg; m < m1; m += LN_RG) {
      float f[8];
      unpack8(ld_nc_v4(x + (long long)m * ldx + c), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) sum[i] += f[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) s_sum[rg][ct * 8 + i] = sum[i];
  __syncthreads();
  if (threadIdx.x < LN_SLAB && c0 + threadIdx.x < N) {
    float a = 0.f;
    for (int g = 0; g < LN_RG; ++g) a += s_sum[g][threadIdx.x];
    ws[(long long)chunk * N + c0 + threadIdx.x] = a;
  }
}

// y = dropout(x) with the GEMM epilogue's stream for element (m, n), and ws[chunk, n] = sum over the chunk's rows of y:
// the backward of a "dropout -> Dense" pair needs both, and one pass over x serves them (it used to be two kernels
// and two reads).
__global__ void __launch_bounds__(LN_THREADS)
dropout_colsum_kernel(int M, int N, int rows_per_chunk, const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ y,
                      DropoutCfg d, float* __restrict__ ws) {
  __shared__ float s_sum[LN_RG][LN_SLAB + 1];
  const int chunk = blockIdx.y, c0 = blockIdx.x * LN_SLAB;
  const int ct = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = c0 + ct * 8;
  const int m0 = chunk * rows_per_chunk, m1 = min(M, m0 + rows_per_chunk);
  float sum[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) sum[i] = 0.f;
  if (c < N) {
#pragma unroll 4
    for (int m = m0 + rg; m < m1; m += LN_RG) {
      float f[8];
      unpack8(ld_nc_v4(x + (long long)m * N + c), f);
      const uint32_t keep = dropout_keep8(d, (uint32_t)m, (uint32_t)c);
#pragma unroll
      for (int i = 0; i < 8; ++i) f[i] = ((keep >> i) & 1u) ? f[i] * d.inv_keep : 0.f;
      const uint4 o = pack8(f);
      st_na_v4(y + (long long)m * N + c, o);
      unpack8(o, f);  // sum what the GEMMs will read (the bf16-rounded values), like the separate colsum did
#pragma unroll
      for (int i = 0; i < 8; ++i) sum[i] += f[i];
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) s_sum[rg][ct * 8 + i] = sum[i];
  __syncthreads();
  if (threadIdx.x < LN_SLAB && c0 + threadIdx.x < N) {
    float a = 0.f;
    for (int g = 0; g < LN_RG; ++g) a += s_sum[g][threadIdx.x];
    ws[(long long)chunk * N + c0 + threadIdx.x] = a;
  }
}

// ------------------------------------------------------------------------------------------------ axis 2 (features)
// one warp per token row
__global__ void __launch_bounds__(256)
ln_feat_fwd_kernel(long long rows, int C, float eps, const __nv_bfloat16* __restrict__ x, const float* __restrict__ gamma,
                   const float* __restrict__ beta, __nv_bfloat16* __restrict__ y, float* __restrict__ mean,
                   float* __restrict__ rstd) {
  const long long row = blockIdx.x * 8ll + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const __nv_bfloat16* xr = x + row * C;
  float a = 0.f, q = 0.f;
  for (int c = lane * 8; c < C; c += 256) {
    float f[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(xr + c)), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      a += f[i];
      q = fmaf(f[i], f[i], q);
    }
  }
  a = warp_sum(a);
  q = warp_sum(q);
  const float mu = a / (float)C;
  const float rs = rsqrtf(fmaxf(q / (float)C - mu * mu, 0.f) + eps);
  if (lane == 0) {
    mean[row] = mu;
    rstd[row] = rs;
  }
  for (int c = lane * 8; c < C; c += 256) {
    float f[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(xr + c)), f);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = fmaf((f[i] - mu) * rs, gamma[c + i], beta[c + i]);
    *reinterpret_cast<uint4*>(y + row * C + c) = pack8(f);
  }
}

// dx = rstd * (g - mean_c(g) - xhat * mean_c(g * xhat)),  g = dy * gamma.   Per-chunk dgamma/dbeta partials in ws.
__global__ void __launch_bounds__(256)
ln_feat_bwd_kernel(long long rows, int C, const __nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ dy,
                   const float* __restrict__ gamma, const float* __restrict__ mean, const float* __restrict__ rstd,
                   const __nv_bfloat16* __restrict__ dres, __nv_bfloat16* __restrict__ dx) {
  const long long row = blockIdx.x * 8ll + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float mu = mean[row], rs = rstd[row];
  float a = 0.f, q = 0.f;
  for (int c = lane * 8; c < C; c += 256) {
    float fx[8], fd[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + row * C + c)), fx);
    unpack8(__ldg(reinterpret_cast<const uint4*>(dy + row * C + c)), fd);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float g = fd[i] * gamma[c + i];
      a += g;
      q = fmaf(g, (fx[i] - mu) * rs, q);
    }
  }
  a = warp_sum(a) / (float)C;
  q = warp_sum(q) / (float)C;
  for (int c = lane * 8; c < C; c += 256) {
    float fx[8], fd[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + row * C + c)), fx);
    unpack8(__ldg(reinterpret_cast<const uint4*>(dy + row * C + c)), fd);
#pragma unroll
    for (int i = 0; i < 8; ++i) o[i] = rs * (fd[i] * gamma[c + i] - a - (fx[i] - mu) * rs * q);
    if (dres) {
      float fr[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(dres + row * C + c)), fr);
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] += fr[i];
    }
    *reinterpret_cast<uint4*>(dx + row * C + c) = pack8(o);
  }
}

// ws[0][chunk][c] = sum_rows dy ; ws[1][chunk][c] = sum_rows dy * xhat      (axis-2 dbeta / dgamma partials)
__global__ void __launch_bounds__(LN_THREADS)
ln_feat_param_grad_kernel(long long rows, int C, int rows_per_chunk, int n_chunks, const __nv_bfloat16* __restrict__ x,
                          const __nv_bfloat16* __restrict__ dy, const float* __restrict__ mean,
                          const float* __restrict__ rstd, float* __restrict__ ws) {
  __shared__ float s_a[LN_RG][LN_SLAB + 1];
  __shared__ float s_b[LN_RG][LN_SLAB + 1];
  const int chunk = blockIdx.y, c0 = blockIdx.x * LN_SLAB;
  const int ct = threadIdx.x & 7, rg = threadIdx.x >> 3;
  const int c = c0 + ct * 8;
  const long long m0 = (long long)chunk * rows_per_chunk;
  const long long m1 = m0 + rows_per_chunk < rows ? m0 + rows_per_chunk : rows;
  float sa[8], sb[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) sa[i] = sb[i] = 0.f;
  if (c < C) {
    for (long long m = m0 + rg; m < m1; m += LN_RG) {
      float fx[8], fd[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + m * C + c)), fx);
      unpack8(__ldg(reinterpret_cast<const uint4*>(dy + m * C + c)), fd);
      const float mu = mean[m], rs = rstd[m];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sa[i] += fd[i];
        sb[i] = fmaf(fd[i], (fx[i] - mu) * rs, sb[i]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    s_a[rg][ct * 8 + i] = sa[i];
    s_b[rg][ct * 8 + i] = sb[i];
  }
  __syncthreads();
  if (threadIdx.x < LN_SLAB && c0 + threadIdx.x < C) {
    float a = 0.f, q = 0.f;
    for (int g = 0; g < LN_RG; ++g) {
      a += s_a[g][threadIdx.x];
      q += s_b[g][threadIdx.x];
    }
    ws[(long long)chunk * C + c0 + threadIdx.x] = a;
    ws[(long long)(n_chunks + chunk) * C + c0 + threadIdx.x] = q;
  }
}

static inline int colsum_rows(long long m) {
  long long r = (m + 63) / 64;
  if (r > 256) r = 256;
  return (int)(r < 1 ? 1 : r);
}

}  // namespace tome

using namespace tome;

extern "C" int tome_colsum_workspace_rows(int m) { return colsum_rows(m); }

static int g_ln_force_cluster = 0;
/* testing aid (not in the public header): 1 = take the cluster kernels even when one CTA per slab would do; n > 1 = split the
 * tokens over exactly n CTAs */
extern "C" void tome_ln_force_cluster(int n) { g_ln_force_cluster = n < 0 ? 0 : n > 8 ? 8 : n; }

// CTAs per (batch, slab): about nine 64-row boxes per CTA (what the T = 536 shape has), at most a portable cluster of 8
static inline int ln_token_split(int boxes) {
  int s = (boxes + 8) / 9;
  return s < 1 ? 1 : s > 8 ? 8 : s;
}

template <typename K, typename... Args>
static int launch_cluster_z(K kern, dim3 grid, int smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = dim3(LN_THREADS);
  cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = grid.z;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  TOME_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  return TOME_OK;
}

extern "C" int tome_reduce_rows_f32(int rows, int n, const float* partial, float* out, int accumulate, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(rows > 0 && n > 0 && partial && out, TOME_ERR_INVALID, "reduce_rows: bad argument");
  if (rows >= 256) launch_k(reduce_rows_kernel<32>, ceil_div(n, 32), 1024, 0, stream, rows, n, partial, 0, out, out, accumulate);
  else launch_k(reduce_rows_kernel<8>, ceil_div(n, 32), 256, 0, stream, rows, n, partial, 0, out, out, accumulate);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_colsum_bf16(int m, int n, const void* x, long long ldx, float* out, int accumulate, float* workspace,
                                void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(m > 0 && n > 0 && x && out && workspace, TOME_ERR_INVALID, "colsum: bad argument");
  TOME_CHECK(n % 8 == 0 && ldx % 8 == 0, TOME_ERR_INVALID, "colsum: n and ldx must be multiples of 8");
  const int chunks = colsum_rows(m);
  ProfScope prof(PROF_COLSUM, (double)m * n * 2.0, 2, stream);
  const int rpc = ceil_div(m, chunks);
  dim3 grid(ceil_div(n, LN_SLAB), chunks);
  launch_k(colsum_partial_kernel, grid, LN_THREADS, 0, stream, m, n, ldx, rpc, reinterpret_cast<const __nv_bfloat16*>(x), workspace);
  TOME_CUDA(cudaGetLastError());
  launch_k(reduce_rows_kernel<8>, ceil_div(n, 32), 256, 0, stream, chunks, n, workspace, 0, out, out, accumulate);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_dropout_colsum_bf16(int m, int n, const void* x, void* y, float rate, uint64_t seed, uint32_t site,
                                        float* out, int accumulate, float* workspace, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(m > 0 && n > 0 && x && y && out && workspace, TOME_ERR_INVALID, "dropout_colsum: bad argument");
  TOME_CHECK(n % 8 == 0, TOME_ERR_INVALID, "dropout_colsum: n must be a multiple of 8");
  TOME_CHECK(rate >= 0.f && rate < 1.f, TOME_ERR_INVALID, "dropout_colsum: rate must be in [0, 1)");
  const DropoutCfg d = make_dropout(rate, seed, site);
  const int chunks = colsum_rows(m);
  ProfScope prof(PROF_COLSUM, (double)m * n * 4.0, 2, stream);
  const int rpc = ceil_div(m, chunks);
  dim3 grid(ceil_div(n, LN_SLAB), chunks);
  launch_k(dropout_colsum_kernel, grid, LN_THREADS, 0, stream, m, n, rpc, reinterpret_cast<const __nv_bfloat16*>(x),
                                                         reinterpret_cast<__nv_bfloat16*>(y), d, workspace);
  TOME_CUDA(cudaGetLastError());
  launch_k(reduce_rows_kernel<8>, ceil_div(n, 32), 256, 0, stream, chunks, n, workspace, 0, out, out, accumulate);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_layernorm_fwd(int batch, int tokens, int channels, int axis, float eps, const void* x,
                                  const float* gamma, const float* beta, void* y, float* mean, float* rstd, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && channels > 0, TOME_ERR_INVALID, "layernorm_fwd: bad shape");
  TOME_CHECK(channels % 8 == 0, TOME_ERR_INVALID, "layernorm_fwd: channels (%d) must be a multiple of 8", channels);
  TOME_CHECK(x && gamma && beta && y && mean && rstd, TOME_ERR_INVALID, "layernorm_fwd: null argument");
  TOME_CHECK(axis == 1 || axis == 2, TOME_ERR_INVALID, "layernorm_fwd: axis must be 1 (tokens) or 2 (features)");
  const __nv_bfloat16* xp = reinterpret_cast<const __nv_bfloat16*>(x);
  __nv_bfloat16* yp = reinterpret_cast<__nv_bfloat16*>(y);
  ProfScope prof(PROF_LN, 2.0 * batch * (double)tokens * channels * 2.0, 1, stream);
  if (axis == 1) {
    TOME_CHECK(batch <= 65535, TOME_ERR_INVALID, "layernorm_fwd: batch too large");
    dim3 grid(ceil_div(channels, LN_SLAB), batch);
    const int nb_all = ln_boxes(tokens);
    const int split = g_ln_force_cluster > 1 ? g_ln_force_cluster : ln_token_split(nb_all);   // CTAs (one cluster) per (batch, slab)
    const int nb = ceil_div(nb_all, split);
    if (((uintptr_t)x & 15) == 0 && nb * LN_BOX <= LN_SMEM_T_FWD) {
      CUtensorMap tx;
      if (int rc = make_tmap_3d_bf16(&tx, x, channels, tokens, batch, channels, (uint64_t)tokens * channels, LN_BOX)) return rc;
      const int smem = nb * LN_BOX * 128 + nb * 8 + 1024;
      if (split == 1 && !g_ln_force_cluster) {
        static DynSmemOnce once;
        TOME_CUDA(ensure_dyn_smem(ln_seq_fwd_smem_kernel<false>, smem, once));
        launch_k(ln_seq_fwd_smem_kernel<false>, grid, LN_THREADS, smem, stream, tx, tokens, channels, nb, eps, gamma, beta, yp, mean, rstd);
      } else {
        static DynSmemOnce once;
        TOME_CUDA(ensure_dyn_smem(ln_seq_fwd_smem_kernel<true>, smem, once));
        if (int rc = launch_cluster_z(ln_seq_fwd_smem_kernel<true>, dim3(grid.x, grid.y, split), smem, stream, tx, tokens, channels, nb,
                                      eps, gamma, beta, yp, mean, rstd)) return rc;
      }
    } else {
      launch_k(ln_seq_fwd_kernel, grid, LN_THREADS, 0, stream, tokens, channels, eps, xp, gamma, beta, yp, mean, rstd);
    }
  } else {
    const long long rows = (long long)batch * tokens;
    launch_k(ln_feat_fwd_kernel, (unsigned)((rows + 7) / 8), 256, 0, stream, rows, channels, eps, xp, gamma, beta, yp, mean, rstd);
  }
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_layernorm_bwd(int batch, int tokens, int channels, int axis, const void* x, const void* dy,
                                  const float* gamma, const float* mean, const float* rstd, const void* dres, void* dx,
                                  float* dgamma, float* dbeta, float* partial, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && channels > 0 && channels % 8 == 0, TOME_ERR_INVALID, "layernorm_bwd: bad shape");
  TOME_CHECK(x && dy && gamma && mean && rstd && dx && dgamma && dbeta && partial, TOME_ERR_INVALID,
             "layernorm_bwd: null argument");
  TOME_CHECK(axis == 1 || axis == 2, TOME_ERR_INVALID, "layernorm_bwd: axis must be 1 (tokens) or 2 (features)");
  const __nv_bfloat16* xp = reinterpret_cast<const __nv_bfloat16*>(x);
  const __nv_bfloat16* dyp = reinterpret_cast<const __nv_bfloat16*>(dy);
  const __nv_bfloat16* drp = reinterpret_cast<const __nv_bfloat16*>(dres);
  __nv_bfloat16* dxp = reinterpret_cast<__nv_bfloat16*>(dx);
  ProfScope prof(PROF_LN, (dres ? 4.0 : 3.0) * batch * (double)tokens * channels * 2.0, axis == 1 ? 3 : 4, stream);
  int chunks;
  if (axis == 1) {
    TOME_CHECK(batch <= 65535, TOME_ERR_INVALID, "layernorm_bwd: batch too large");
    dim3 grid(ceil_div(channels, LN_SLAB), batch);
    const int nb_all = ln_boxes(tokens);
    const int split = g_ln_force_cluster > 1 ? g_ln_force_cluster : ln_token_split(nb_all);
    const int nb = ceil_div(nb_all, split);
    if (nb <= LNB_MAX_BOXES && (((uintptr_t)x | (uintptr_t)dy) & 15) == 0) {
      CUtensorMap tx, tdy;
      if (int rc = make_tmap_3d_bf16_plain(&tx, x, channels, tokens, batch, channels, (uint64_t)tokens * channels, LNB_SLAB, LN_BOX)) return rc;
      if (int rc = make_tmap_3d_bf16_plain(&tdy, dy, channels, tokens, batch, channels, (uint64_t)tokens * channels, LNB_SLAB, LN_BOX)) return rc;
      const int smem = 2 * nb * LN_BOX * LNB_SLAB * 2 + nb * 8 + 128;
      grid = dim3(ceil_div(channels, LNB_SLAB), batch);
      if (split == 1 && !g_ln_force_cluster) {
        static DynSmemOnce once;
        TOME_CUDA(ensure_dyn_smem(ln_seq_bwd_smem_kernel<false>, smem, once));
        launch_k(ln_seq_bwd_smem_kernel<false>, grid, LN_THREADS, smem, stream, tx, tdy, batch, tokens, channels, nb, gamma, mean, rstd, drp, dxp, partial);
      } else {
        static DynSmemOnce once;
        TOME_CUDA(ensure_dyn_smem(ln_seq_bwd_smem_kernel<true>, smem, once));
        if (int rc = launch_cluster_z(ln_seq_bwd_smem_kernel<true>, dim3(grid.x, grid.y, split), smem, stream, tx, tdy, batch, tokens,
                                      channels, nb, gamma, mean, rstd, drp, dxp, partial)) return rc;
      }
    } else {
      launch_k(ln_seq_bwd_kernel, grid, LN_THREADS, 0, stream, batch, tokens, channels, xp, dyp, gamma, mean, rstd, drp, dxp, partial);
    }
    chunks = batch;
  } else {
    const long long rows = (long long)batch * tokens;
    launch_k(ln_feat_bwd_kernel, (unsigned)((rows + 7) / 8), 256, 0, stream, rows, channels, xp, dyp, gamma, mean, rstd, drp, dxp);
    TOME_CUDA(cudaGetLastError());
    chunks = colsum_rows(rows);
    const int rpc = (int)((rows + chunks - 1) / chunks);
    dim3 grid(ceil_div(channels, LN_SLAB), chunks);
    launch_k(ln_feat_param_grad_kernel, grid, LN_THREADS, 0, stream, rows, channels, rpc, chunks, xp, dyp, mean, rstd, partial);
  }
  TOME_CUDA(cudaGetLastError());
  launch_k(reduce_rows_kernel<8>, dim3(ceil_div(channels, 32), 2), 256, 0, stream, chunks, channels, partial, (long long)chunks * channels,
                                                                          dbeta, dgamma, 1);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
