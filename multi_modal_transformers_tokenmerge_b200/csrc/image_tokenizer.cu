// K12: image patch-embed front end (forward).   tokenizers/images/image_tokenizer.py:35-71 (image_to_patches), :74-140
// (encode_patch_position), :148-190 (ResNetV2Block), :216-309 (ImageTokenizer); SURVEY.md 8(f) rank 4.
//
//   image [B, N, H, W, C_in] -> patches (p x p, row-major) -> Conv k x k / stride s VALID -> max pool w x w / 1 VALID
//   -> num_blocks x [GroupNorm -> gelu(tanh) -> Conv 3x3 SAME] -> + pooled -> flatten (h, w, c) -> Dense -> + row / column
//   position embeddings -> tokens [B, N, n_patches, E].
//
// The three contractions (input convolution, block convolutions, Dense) run on the tcgen05 GEMM of gemm.cu with bf16
// operands and fp32 accumulation; the kernels here produce their A operands and consume their outputs:
//   it_pixels_bf16_kernel + it_im2col0_words_kernel   pixels (u8 / f32) -> normalised bf16 once, then the im2col rows
//                          [M0, k*k*C_in] of the input convolution by 32-bit words (patch extraction is index arithmetic: no
//                          patch tensor is ever written); it_im2col0_kernel does both per byte through a 256-entry table
//                          when an odd element offset rules the word path out
//   it_pool_kernel         conv0 output [.., o1, o1, F] -> max over w x w windows (packed bf16x2 max) -> the activation grid
//   it_gn_partial_kernel / it_gn_final_kernel   GroupNorm statistics.  Flax's GroupNorm reduces over EVERY axis but the
//                          batch one, so a (batch row, group) statistic spans all N images and all patches of that row:
//                          per-CTA per-channel partial sums in a fixed order, then one warp per (row, group)
//   it_gn_gelu_kernel      (x - mean) * rstd * scale + bias -> gelu, once per element (the statistics folded into a
//                          per-(batch row, channel) multiply-add by it_gn_fold_kernel); zeroes the grid's border
//   3 x 3 convolutions     features % 64 == 0 (the reference's 64): the block activations live on a (o2 + 2)^2 grid with a zero
//                          border, and the convolution is ONE GEMM whose nine k-blocks read the SAME matrix at rows shifted by
//                          (ty - 1)(o2 + 2) + (tx - 1) (tome_gemm_args_t.a_row_shift: a TMA row coordinate per k-block; no
//                          im2col rows, the activation is re-read from L2); it_compact_kernel then gathers the interior and
//                          adds the pooled tensor (the residual of image_tokenizer.py:170)
//   it_im2col3_kernel      other widths: the nine shifted copies of the 3x3 SAME im2col row, zero outside the o2 x o2
//                          window; one 16-byte load and one 16-byte store per thread; residual in the last GEMM's epilogue
//   it_posadd_kernel       Dense output + row_embedding[row_token] + col_embedding[col_token] -> out dtype, into
//                          out [B, N, n_patches, E] or (tome_policy_predict) straight into rows of the assembled sequence
//   it_seq_rows_kernel     the sequence's text / readout rows (tome_policy_predict), one launch for every set
// What is left HBM-bound is the input convolution (its im2col rows are k*k*C_in / (s*s*C_in) = 36x the pixels); the batch
// is processed in chunks of whole batch rows so that buffer stays near 1 GiB whatever the batch.  Measurements and the
// versions that led here: DESIGN.md 4.5, profiles/r02c_image_tokenizer.md.
#include <algorithm>

#include "common.cuh"
#include "host_util.h"
#include "image_tokenizer.h"

namespace tome {

constexpr int IT_THREADS = 256;
constexpr int IT_GN_MAX_CTAS = 64;      // CTAs per batch row in the statistics pass
constexpr size_t IT_COL_TARGET = (size_t)1 << 30;   // im2col buffer target per chunk of batch rows

struct ItGeom {
  int ppd, np;          // patches per image side / per image
  int o1, o2;           // side after the input convolution / after the pool
  int wp, pad;          // side of the grid the block activations live on: o2 + 2 with a zero border (pad = 1) when the 3 x 3
                        // convolutions run as row-shifted GEMMs (features % 64 == 0), else o2 (pad = 0, im2col rows)
  int k0;               // k*k*C_in
  int kd;               // o2*o2*F (Dense fan-in)
  long long imgs;       // B*N
  int chunk_rows;       // batch rows per chunk
  int gn_ctas;
  // workspace offsets (bytes) of one chunk
  size_t off_col, off_y0, off_pool, off_xa, off_xb, off_h, off_pix, off_dense, off_part, off_stats, off_ab, total;
};

static int it_geometry(const tome_image_tokenizer_desc_t* d, ItGeom* g, const char* who) {
  TOME_CHECK(d != nullptr, TOME_ERR_INVALID, "%s: null descriptor", who);
  TOME_CHECK(d->batch > 0 && d->n_images > 0 && d->image_size > 0 && d->channels_in > 0, TOME_ERR_INVALID, "%s: bad image shape", who);
  TOME_CHECK(d->patch_size > 0 && d->image_size % d->patch_size == 0, TOME_ERR_INVALID,
             "%s: image_size (%d) must be a multiple of patch_size (%d) (image_tokenizer.py:52)", who, d->image_size, d->patch_size);
  TOME_CHECK(d->image_dtype == TOME_U8 || d->image_dtype == TOME_F32, TOME_ERR_INVALID, "%s: image_dtype must be u8 or f32", who);
  TOME_CHECK(d->out_dtype == TOME_BF16 || d->out_dtype == TOME_F32, TOME_ERR_INVALID, "%s: out_dtype must be bf16 or f32", who);
  TOME_CHECK(d->conv_kernel > 0 && d->conv_stride > 0 && d->patch_size >= d->conv_kernel, TOME_ERR_INVALID,
             "%s: the input convolution (%d, stride %d) does not fit a %d-pixel patch", who, d->conv_kernel, d->conv_stride, d->patch_size);
  TOME_CHECK(d->pool_window >= 1, TOME_ERR_INVALID, "%s: pool_window must be >= 1", who);
  TOME_CHECK(d->num_blocks >= 1, TOME_ERR_UNSUPPORTED, "%s: num_blocks must be >= 1", who);
  TOME_CHECK(d->features > 0 && d->features % 8 == 0 && d->features <= 2048, TOME_ERR_UNSUPPORTED,
             "%s: features (%d) must be a multiple of 8, at most 2048", who, d->features);
  TOME_CHECK(d->num_groups > 0 && d->features % d->num_groups == 0, TOME_ERR_INVALID,
             "%s: features (%d) must be a multiple of num_groups (%d)", who, d->features, d->num_groups);
  TOME_CHECK(d->embed_dim > 0 && d->embed_dim % 8 == 0, TOME_ERR_UNSUPPORTED, "%s: embed_dim (%d) must be a multiple of 8", who, d->embed_dim);
  TOME_CHECK(d->position_interval > 0, TOME_ERR_INVALID, "%s: position_interval must be positive", who);
  TOME_CHECK(d->token_rows == 1 || d->token_rows == d->batch * d->n_images, TOME_ERR_INVALID,
             "%s: token_rows must be 1 or batch * n_images (got %d)", who, d->token_rows);
  g->ppd = d->image_size / d->patch_size;
  g->np = g->ppd * g->ppd;
  g->o1 = (d->patch_size - d->conv_kernel) / d->conv_stride + 1;
  g->o2 = g->o1 - (d->pool_window - 1);
  TOME_CHECK(g->o2 >= 1, TOME_ERR_INVALID, "%s: a %d-wide pool does not fit the %d x %d convolution output", who, d->pool_window, g->o1, g->o1);
  g->k0 = d->conv_kernel * d->conv_kernel * d->channels_in;
  g->kd = g->o2 * g->o2 * d->features;
  g->pad = d->features % 64 == 0 ? 1 : 0;
  TOME_CHECK(g->k0 % 16 == 0, TOME_ERR_UNSUPPORTED, "%s: conv_kernel^2 * channels_in (%d) must be a multiple of 16", who, g->k0);
  g->wp = g->o2 + 2 * g->pad;
  g->imgs = (long long)d->batch * d->n_images;
  const long long m0_row = (long long)d->n_images * g->np * g->o1 * g->o1;   // im2col rows of the input convolution per batch row
  const long long m2_row = (long long)d->n_images * g->np * g->o2 * g->o2;
  const long long m2p_row = (long long)d->n_images * g->np * g->wp * g->wp;   // rows of the (bordered) activation grid
  const size_t col_row = 2 * (size_t)std::max(m0_row * g->k0, g->pad ? 0ll : m2_row * 9 * d->features);
  long long cr = (long long)(IT_COL_TARGET / col_row);
  TOME_CHECK(d->chunk_rows >= 0, TOME_ERR_INVALID, "%s: chunk_rows must be >= 0", who);
  if (d->chunk_rows > 0) cr = d->chunk_rows;
  if (cr < 1) cr = 1;
  if (cr > d->batch) cr = d->batch;
  TOME_CHECK(m0_row * cr * (g->k0 / 8) < (1ll << 31) && m2p_row * cr * 9 * (d->features / 8) < (1ll << 31), TOME_ERR_UNSUPPORTED,
             "%s: %lld batch rows per pass need more than 2^31 16-byte vectors of im2col rows: lower chunk_rows", who, cr);
  g->chunk_rows = (int)cr;
  long long want = m2_row * (d->features / 8) / (IT_THREADS * 4);
  g->gn_ctas = (int)std::min<long long>(IT_GN_MAX_CTAS, std::max<long long>(1, want));
  Bump b{nullptr};
  g->off_col = b.reserve(col_row * cr);
  g->off_y0 = b.reserve((size_t)2 * m0_row * cr * d->features);
  g->off_pool = b.reserve((size_t)2 * m2p_row * cr * d->features);
  g->off_xa = b.reserve((size_t)2 * m2p_row * cr * d->features);
  g->off_xb = b.reserve((size_t)2 * m2p_row * cr * d->features);
  g->off_h = b.reserve((size_t)2 * m2p_row * cr * d->features);
  g->off_pix = b.reserve((size_t)2 * cr * d->n_images * d->image_size * d->image_size * d->channels_in + 16);
  g->off_dense = b.reserve((size_t)4 * cr * d->n_images * g->np * d->embed_dim);
  g->off_part = b.reserve((size_t)4 * cr * g->gn_ctas * d->features * 2);
  g->off_stats = b.reserve((size_t)4 * cr * d->num_groups * 2);
  g->off_ab = b.reserve((size_t)4 * cr * d->features * 2);
  g->total = b.total();
  return TOME_OK;
}

// Division of an index below 2^31 by a runtime constant, as one multiply-high and a shift (the index decodes below would
// otherwise spend more instructions on dividing than on moving their 16 bytes).
struct FastDiv {
  uint32_t mul, shift, d;
  __device__ __forceinline__ uint32_t div(uint32_t n) const { return d == 1 ? n : __umulhi(n, mul) >> shift; }
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const { q = div(n); r = n - q * d; }
};
static FastDiv make_fastdiv(uint32_t d) {   // exact for n < 2^31: mul = ceil(2^(31+s) / d), s = ceil(log2 d)
  FastDiv f;
  f.d = d;
  uint32_t s = 0;
  while ((1ull << s) < d) ++s;
  f.mul = d == 1 ? 0u : (uint32_t)(((1ull << (31 + s)) + d - 1) / d);
  f.shift = d == 1 ? 0u : s - 1;
  return f;
}

struct Im2col0Args {
  FastDiv vpr, o1, np, ppd, kw_c;
  int psize, stride, img_w_c, c_in, normalize;
  long long img_elems;   // H * W * C_in
};

// ---------------------------------------------------------------------------------------------------------------
// pixels -> im2col rows of the input convolution.  Row m = ((img * np + patch) * o1 + oy) * o1 + ox, column
// (dy * k + dx) * C_in + c  <-  image[img, py * p + oy * s + dy, px * p + ox * s + dx, c]: for one dy the (dx, c) run
// is contiguous in the image.  One thread writes 8 consecutive columns (16 bytes), which span at most two dy rows.
// uint8 pixels go through a 256-entry table of the normalised bf16 values (2 * (x / 255) - 1, image_tokenizer.py:67).
template <typename PixT>
__global__ void __launch_bounds__(IT_THREADS)
it_im2col0_kernel(const PixT* __restrict__ image, __nv_bfloat16* __restrict__ col, uint32_t n_vec, const Im2col0Args a) {
  __shared__ uint16_t lut[256];
  if (sizeof(PixT) == 1) {
    float x = (float)threadIdx.x;
    if (a.normalize) x = 2.0f * __fdiv_rn(x, 255.0f) - 1.0f;
    __nv_bfloat16 h = __float2bfloat16(x);
    lut[threadIdx.x] = *reinterpret_cast<uint16_t*>(&h);
    __syncthreads();
  }
  const uint32_t v = (blockIdx.x * IT_THREADS + threadIdx.x) * 2;   // two consecutive 16-byte vectors of one row (k0 / 8 is even)
  if (v >= n_vec) return;
  uint32_t m, kc, ox, oy, patch, img, py, px, dy, rem, t;
  a.vpr.divmod(v, m, kc);
  a.o1.divmod(m, t, ox);
  a.o1.divmod(t, t, oy);
  a.np.divmod(t, img, patch);
  a.ppd.divmod(patch, py, px);
  a.kw_c.divmod(kc << 3, dy, rem);
  const PixT* base = image + img * a.img_elems + (long long)(py * a.psize + oy * a.stride + dy) * a.img_w_c +
                     (long long)(px * a.psize + ox * a.stride) * a.c_in;
  uint32_t w[8];
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    if (rem >= a.kw_c.d) { rem -= a.kw_c.d; base += a.img_w_c; }
    uint32_t h16;
    if (sizeof(PixT) == 1) {
      h16 = lut[(uint32_t)base[rem]];
    } else {
      float x = (float)base[rem];
      if (a.normalize) x = 2.0f * __fdiv_rn(x, 255.0f) - 1.0f;
      __nv_bfloat16 h = __float2bfloat16(x);
      h16 = *reinterpret_cast<uint16_t*>(&h);
    }
    if (j & 1) w[j >> 1] |= h16 << 16; else w[j >> 1] = h16;
    ++rem;
  }
  st_na_v4(col + (size_t)v * 8, make_uint4(w[0], w[1], w[2], w[3]));
  st_na_v4(col + (size_t)v * 8 + 8, make_uint4(w[4], w[5], w[6], w[7]));
}

// pixels (u8 / f32) -> normalised bf16, once (8 pixels values per thread); the im2col below then moves whole 32-bit words.
template <typename PixT>
__global__ void __launch_bounds__(IT_THREADS)
it_pixels_bf16_kernel(const PixT* __restrict__ image, __nv_bfloat16* __restrict__ out, long long n, int normalize) {
  const long long i = ((long long)blockIdx.x * IT_THREADS + threadIdx.x) * 8;
  if (i >= n) return;
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float x = i + j < n ? (float)image[i + j] : 0.f;
    if (normalize) x = 2.0f * __fdiv_rn(x, 255.0f) - 1.0f;   // image_tokenizer.py:67
    __nv_bfloat16 h = __float2bfloat16(x);
    const uint32_t h16 = *reinterpret_cast<uint16_t*>(&h);
    if (j & 1) w[j >> 1] |= h16 << 16; else w[j >> 1] = h16;
  }
  if (i + 8 <= n) *reinterpret_cast<uint4*>(out + i) = make_uint4(w[0], w[1], w[2], w[3]);
  else for (int j = 0; i + j < n; ++j) reinterpret_cast<uint16_t*>(out)[i + j] = (uint16_t)(w[j >> 1] >> ((j & 1) * 16));
}

// im2col rows of the input convolution from the bf16 pixels, two elements (one 32-bit word) at a time: every offset involved
// is even (host-checked: k * C_in, W * C_in, stride * C_in and patch * C_in even), so a word never straddles a (dy) row.
__global__ void __launch_bounds__(IT_THREADS)
it_im2col0_words_kernel(const uint32_t* __restrict__ pix, __nv_bfloat16* __restrict__ col, uint32_t n_vec, const Im2col0Args a) {
  const uint32_t v = (blockIdx.x * IT_THREADS + threadIdx.x) * 2;   // two consecutive 16-byte vectors of one row
  if (v >= n_vec) return;
  uint32_t m, kc, ox, oy, patch, img, py, px, dy, rem, t;
  a.vpr.divmod(v, m, kc);
  a.o1.divmod(m, t, ox);
  a.o1.divmod(t, t, oy);
  a.np.divmod(t, img, patch);
  a.ppd.divmod(patch, py, px);
  a.kw_c.divmod(kc << 3, dy, rem);
  const uint32_t* base = pix + ((img * a.img_elems + (long long)(py * a.psize + oy * a.stride + dy) * a.img_w_c +
                                 (long long)(px * a.psize + ox * a.stride) * a.c_in) >> 1);
  const uint32_t row_words = (uint32_t)a.img_w_c >> 1, kw_words = a.kw_c.d >> 1;
  uint32_t rw = rem >> 1, w[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    if (rw >= kw_words) { rw -= kw_words; base += row_words; }
    w[j] = __ldg(base + rw);
    ++rw;
  }
  st_na_v4(col + (size_t)v * 8, make_uint4(w[0], w[1], w[2], w[3]));
  st_na_v4(col + (size_t)v * 8 + 8, make_uint4(w[4], w[5], w[6], w[7]));
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  f[0] = bf16_lo(u.x); f[1] = bf16_hi(u.x); f[2] = bf16_lo(u.y); f[3] = bf16_hi(u.y);
  f[4] = bf16_lo(u.z); f[5] = bf16_hi(u.z); f[6] = bf16_lo(u.w); f[7] = bf16_hi(u.w);
}

__device__ __forceinline__ uint32_t bf16x2_max(uint32_t a, uint32_t b) {
  uint32_t r;
  asm("max.bf16x2 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
  return r;
}

// max pool, stride 1, VALID (flax.linen.max_pool).  Thread = (output pixel, 8 channels).
__global__ void __launch_bounds__(IT_THREADS)
it_pool_kernel(const __nv_bfloat16* __restrict__ y0, __nv_bfloat16* __restrict__ pooled, uint32_t n_vec, FastDiv nchunk, int o1,
               FastDiv o2, int window, int wp, int pad) {
  const uint32_t v = blockIdx.x * IT_THREADS + threadIdx.x;
  if (v >= n_vec) return;
  uint32_t c, t, ox, oy, ip;
  nchunk.divmod(v, t, c);
  o2.divmod(t, t, ox);
  o2.divmod(t, ip, oy);
  const int F = nchunk.d << 3;
  const __nv_bfloat16* src = y0 + (((size_t)ip * o1 + oy) * o1 + ox) * F + (c << 3);
  // the maximum of bf16 values is one of them: packed bf16x2 max, no conversion
  uint4 best = *reinterpret_cast<const uint4*>(src);
  for (int dy = 0; dy < window; ++dy)
    for (int dx = (dy == 0 ? 1 : 0); dx < window; ++dx) {
      const uint4 u = *reinterpret_cast<const uint4*>(src + ((size_t)dy * o1 + dx) * F);
      best.x = bf16x2_max(best.x, u.x); best.y = bf16x2_max(best.y, u.y);
      best.z = bf16x2_max(best.z, u.z); best.w = bf16x2_max(best.w, u.w);
    }
  *reinterpret_cast<uint4*>(pooled + ((((size_t)ip * wp + oy + pad) * wp + ox + pad) * nchunk.d + c) * 8) = best;
}

// GroupNorm statistics, stage 1: x [rows_b, R, F] bf16; CTA (j, b) sums x and x^2 per CHANNEL over its slice of the R rows
// of batch row b -> part [rows_b, gridDim.x, F, 2].  Thread = (8-channel chunk, row lane); lanes are added in lane order.
__global__ void __launch_bounds__(IT_THREADS)
it_gn_partial_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ part, long long R, int nchunk, FastDiv wp, int pad) {
  __shared__ float sm[2][IT_THREADS * 8];
  const int F = nchunk << 3;
  const int lanes = blockDim.x / nchunk;
  const int c = threadIdx.x % nchunk, rl = threadIdx.x / nchunk;
  const long long r0 = R * blockIdx.x / gridDim.x, r1 = R * (blockIdx.x + 1) / gridDim.x;
  const __nv_bfloat16* xb = x + (long long)blockIdx.y * R * F + (c << 3);
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  for (long long r = r0 + rl; r < r1; r += lanes) {
    if (pad) {   // bordered grid: only the interior pixels are data
      uint32_t q, xx, yy;
      wp.divmod((uint32_t)r, q, xx);
      yy = q - wp.div(q) * wp.d;
      if (xx < (uint32_t)pad || xx >= wp.d - pad || yy < (uint32_t)pad || yy >= wp.d - pad) continue;
    }
    float f[8];
    unpack8(ld_nc_v4(xb + r * F), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) { s[j] += f[j]; q[j] = fmaf(f[j], f[j], q[j]); }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sm[0][rl * F + (c << 3) + j] = s[j];
    sm[1][rl * F + (c << 3) + j] = q[j];
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < F; ch += blockDim.x) {
    float a = 0.f, b = 0.f;
    for (int l = 0; l < lanes; ++l) { a += sm[0][l * F + ch]; b += sm[1][l * F + ch]; }
    float* o = part + (((long long)blockIdx.y * gridDim.x + blockIdx.x) * F + ch) * 2;
    o[0] = a; o[1] = b;
  }
}

// stage 2: warp = (batch row, group): lane j adds the group's channels of CTA partials j, j + 32, ... in order, then a
// fixed butterfly over the lanes -> stats [rows_b, G, 2] = (mean, 1 / sqrt(var + eps)), var = E[x^2] - mean^2 clamped at 0
// (Flax's fast variance).
__global__ void __launch_bounds__(128)
it_gn_final_kernel(const float* __restrict__ part, float* __restrict__ stats, int rows_b, int n_ctas, int F, int G, long long R,
                   float eps) {
  const int i = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (i >= rows_b * G) return;
  const int b = i / G, g = i - b * G, cg = F / G;
  float s = 0.f, q = 0.f;
  for (int j = lane; j < n_ctas; j += 32) {
    const float* p = part + (((long long)b * n_ctas + j) * F + g * cg) * 2;
    for (int ch = 0; ch < cg; ++ch) { s += p[2 * ch]; q += p[2 * ch + 1]; }
  }
  s = warp_sum(s);
  q = warp_sum(q);
  if (lane == 0) {
    const float inv_n = 1.0f / ((float)R * (float)cg);
    const float mean = s * inv_n;
    const float var = fmaxf(q * inv_n - mean * mean, 0.f);
    stats[2 * i] = mean;
    stats[2 * i + 1] = 1.0f / sqrtf(var + eps);
  }
}

__device__ __forceinline__ float gelu_tanh(float x) {   // flax.linen.gelu, approximate=True
  const float u = 0.7978845608028654f * (x + 0.044715f * x * x * x);
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));   // one SFU op; |error| ~ 2^-11, below the bf16 rounding of the result
  return 0.5f * x * (1.0f + t);
}

// h = gelu(GroupNorm(x)), once per element.  Thread = (pixel, 8 channels); ab [rows_b, F, 2] holds the per-(batch row,
// channel) affine (rstd * scale, bias - mean * rstd * scale) the preceding tiny kernel folded the statistics into.
__global__ void it_gn_fold_kernel(const float* __restrict__ stats, const float* __restrict__ scale, const float* __restrict__ bias,
                                  float* __restrict__ ab, int rows_b, int F, int G) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows_b * F) return;
  const int b = i / F, ch = i - b * F;
  const float* st = stats + 2 * ((long long)b * G + ch / (F / G));
  const float a = st[1] * scale[ch];
  ab[2 * i] = a;
  ab[2 * i + 1] = bias[ch] - st[0] * a;
}

__global__ void __launch_bounds__(IT_THREADS)
it_gn_gelu_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ ab, __nv_bfloat16* __restrict__ h, uint32_t n_vec,
                  FastDiv nchunk, FastDiv pix_per_row, FastDiv wp, int pad) {
  const uint32_t v = blockIdx.x * IT_THREADS + threadIdx.x;
  if (v >= n_vec) return;
  uint32_t m, c;
  nchunk.divmod(v, m, c);
  const uint32_t b = pix_per_row.div(m);
  if (pad) {   // the zero border the row-shifted convolution reads as SAME padding
    uint32_t q, xx, yy;
    wp.divmod(m, q, xx);
    yy = q - wp.div(q) * wp.d;
    if (xx < (uint32_t)pad || xx >= wp.d - pad || yy < (uint32_t)pad || yy >= wp.d - pad) {
      *reinterpret_cast<uint4*>(h + (size_t)v * 8) = make_uint4(0u, 0u, 0u, 0u);
      return;
    }
  }
  const float4* abp = reinterpret_cast<const float4*>(ab + ((size_t)b * (nchunk.d << 3) + (c << 3)) * 2);
  float f[8];
  unpack8(ld_nc_v4(x + (size_t)v * 8), f);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 t = __ldg(abp + j);   // (a, b) of channels 2j and 2j + 1
    f[2 * j] = gelu_tanh(fmaf(f[2 * j], t.x, t.y));
    f[2 * j + 1] = gelu_tanh(fmaf(f[2 * j + 1], t.z, t.w));
  }
  uint4 o;
  o.x = pack_bf16(f[0], f[1]); o.y = pack_bf16(f[2], f[3]); o.z = pack_bf16(f[4], f[5]); o.w = pack_bf16(f[6], f[7]);
  *reinterpret_cast<uint4*>(h + (size_t)v * 8) = o;
}

// im2col rows of the 3x3 SAME convolution: the nine shifted copies of h, zero outside the o2 x o2 window.  Thread =
// (pixel, tap, 8 channels): output vector index == thread index, so the stores are one contiguous stream.
__global__ void __launch_bounds__(IT_THREADS)
it_im2col3_kernel(const __nv_bfloat16* __restrict__ h, __nv_bfloat16* __restrict__ col, uint32_t n_vec, FastDiv nchunk, FastDiv o2) {
  const uint32_t v = blockIdx.x * IT_THREADS + threadIdx.x;
  if (v >= n_vec) return;
  uint32_t c, t, tap, m, ox, oy, q;
  nchunk.divmod(v, t, c);
  m = t / 9u;
  tap = t - m * 9u;
  o2.divmod(m, q, ox);
  oy = q - o2.div(q) * o2.d;
  const int ty = (int)(tap / 3u), tx = (int)(tap - (tap / 3u) * 3u);
  const int sy = (int)oy + ty - 1, sx = (int)ox + tx - 1;
  uint4 o = make_uint4(0u, 0u, 0u, 0u);
  if (sy >= 0 && sy < (int)o2.d && sx >= 0 && sx < (int)o2.d) {
    const long long ms = (long long)m + (long long)(ty - 1) * (int)o2.d + (tx - 1);
    o = *reinterpret_cast<const uint4*>(h + (size_t)ms * (nchunk.d << 3) + (c << 3));
  }
  st_na_v4(col + (size_t)v * 8, o);
}

// interior of the bordered grid + the residual (the pooled tensor) -> dense [pixels, F] rows (the flatten the Dense consumes).
// Thread = 16 bytes of output.
__global__ void __launch_bounds__(IT_THREADS)
it_compact_kernel(const __nv_bfloat16* __restrict__ xp, const __nv_bfloat16* __restrict__ res, __nv_bfloat16* __restrict__ out,
                  uint32_t n_vec, FastDiv nchunk, FastDiv o2, int wp, int pad) {
  const uint32_t v = blockIdx.x * IT_THREADS + threadIdx.x;
  if (v >= n_vec) return;
  uint32_t c, t, ox, oy, ip;
  nchunk.divmod(v, t, c);
  o2.divmod(t, t, ox);
  o2.divmod(t, ip, oy);
  const size_t src = ((((size_t)ip * wp + oy + pad) * wp + ox + pad) * nchunk.d + c) * 8;
  float f[8], r[8];
  unpack8(ld_nc_v4(xp + src), f);
  unpack8(ld_nc_v4(res + src), r);   // x + residual (image_tokenizer.py:170), added here instead of in the convolution's epilogue
  uint4 o;
  o.x = pack_bf16(f[0] + r[0], f[1] + r[1]); o.y = pack_bf16(f[2] + r[2], f[3] + r[3]);
  o.z = pack_bf16(f[4] + r[4], f[5] + r[5]); o.w = pack_bf16(f[6] + r[6], f[7] + r[7]);
  st_na_v4(out + (size_t)v * 8, o);
}

// tokens + row / column position embeddings (image_tokenizer.py:296-305), 4 features per thread.  kPlaced: bf16 token
// (b, n, p) goes to row place.row0[i] + (n * np + p - place.k0[i]) of the [B, T0, E] sequence `out` instead of out[b, n, p].
template <bool kPlaced>
__global__ void __launch_bounds__(IT_THREADS)
it_posadd_kernel(const float* __restrict__ dense, const float* __restrict__ row_emb, const float* __restrict__ col_emb,
                 const int32_t* __restrict__ row_tok, const int32_t* __restrict__ col_tok, void* __restrict__ out, long long n_vec,
                 int E, int np, long long img0, int per_image_tokens, int P, int out_bf16, const ItPlacement place) {
  const long long v = (long long)blockIdx.x * IT_THREADS + threadIdx.x;
  if (v >= n_vec) return;
  const int e4 = E >> 2;
  const long long m = v / e4;
  const int e = (int)(v - m * e4) << 2;
  const int p = (int)(m % np);
  const long long ti = (per_image_tokens ? (img0 + m / np) * np : 0) + p;
  int rt = row_tok[ti], ct = col_tok[ti];
  rt = min(max(rt, 0), P - 1);   // jnp indexing clamps out-of-range indices
  ct = min(max(ct, 0), P - 1);
  const float4 d = *reinterpret_cast<const float4*>(dense + m * E + e);
  const float4 r = *reinterpret_cast<const float4*>(row_emb + (long long)rt * E + e);
  const float4 c = *reinterpret_cast<const float4*>(col_emb + (long long)ct * E + e);
  const float4 y = make_float4((d.x + r.x) + c.x, (d.y + r.y) + c.y, (d.z + r.z) + c.z, (d.w + r.w) + c.w);
  if (kPlaced) {
    const long long img = img0 + m / np;
    const int k = (int)(img % place.n_images) * np + p;
    int i = 0;
    while (i + 1 < place.n_runs && k >= place.k0[i + 1]) ++i;
    const long long row = (img / place.n_images) * place.seq_tokens + place.row0[i] + (k - place.k0[i]);
    uint2 w = make_uint2(pack_bf16(y.x, y.y), pack_bf16(y.z, y.w));
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + row * E + e) = w;
  } else if (out_bf16) {
    uint2 w = make_uint2(pack_bf16(y.x, y.y), pack_bf16(y.z, y.w));
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(out) + m * E + e) = w;
  } else {
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + m * E + e) = y;
  }
}

// The non-image rows of the assembled sequence: CTA column blockIdx.y = token set, thread = 16 bytes of one (batch row,
// token) row.  A pure copy, so the rows equal TokenSequence.assemble_embeddings's bit for bit.
__global__ void __launch_bounds__(IT_THREADS)
it_seq_rows_kernel(const SeqRowSets sets, __nv_bfloat16* __restrict__ seq, int batch, int seq_tokens, int c8) {
  const int s = blockIdx.y;
  const long long v = (long long)blockIdx.x * IT_THREADS + threadIdx.x;
  const long long per_row = (long long)sets.n[s] * c8;
  if (v >= per_row * batch) return;
  const long long b = v / per_row, rem = v - b * per_row;
  const long long t = rem / c8, c = rem - t * c8;
  const __nv_bfloat16* src = reinterpret_cast<const __nv_bfloat16*>(sets.src[s]) + b * sets.batch_stride[s] + t * c8 * 8 + c * 8;
  *reinterpret_cast<uint4*>(seq + ((b * seq_tokens + sets.row0[s] + t) * c8 + c) * 8) = ld_nc_v4(src);
}

static long long it_offset(const tome_image_tokenizer_desc_t* d, const ItGeom& g, int which) {
  const long long F = d->features, E = d->embed_dim, P = d->position_interval;
  const long long conv0 = (long long)g.k0 * F + F;
  const long long block = 2 * F + 9 * F * F + F;
  const long long blocks_end = conv0 + block * d->num_blocks;
  switch (which) {
    case TOME_IT_CONV0_KERNEL: return 0;
    case TOME_IT_CONV0_BIAS: return (long long)g.k0 * F;
    case TOME_IT_DENSE_KERNEL: return blocks_end;
    case TOME_IT_DENSE_BIAS: return blocks_end + (long long)g.kd * E;
    case TOME_IT_ROW_EMBED: return blocks_end + (long long)g.kd * E + E;
    case TOME_IT_COL_EMBED: return blocks_end + (long long)g.kd * E + E + P * E;
    default: break;
  }
  if (which >= TOME_IT_BLOCK0 && which < TOME_IT_BLOCK0 + 4 * d->num_blocks) {
    const int b = (which - TOME_IT_BLOCK0) / 4, f = (which - TOME_IT_BLOCK0) % 4;
    const long long base = conv0 + block * b;
    return base + (f == 0 ? 0 : f == 1 ? F : f == 2 ? 2 * F : 2 * F + 9 * F * F);
  }
  return -1;
}

}  // namespace tome

using namespace tome;

extern "C" long long tome_image_tokenizer_param_count(const tome_image_tokenizer_desc_t* d) {
  clear_error();
  ItGeom g;
  if (it_geometry(d, &g, "image_tokenizer_param_count") != TOME_OK) return -1;
  return it_offset(d, g, TOME_IT_COL_EMBED) + (long long)d->position_interval * d->embed_dim;
}

extern "C" long long tome_image_tokenizer_param_offset(const tome_image_tokenizer_desc_t* d, int which) {
  clear_error();
  ItGeom g;
  if (it_geometry(d, &g, "image_tokenizer_param_offset") != TOME_OK) return -1;
  const long long o = it_offset(d, g, which);
  if (o < 0) set_error(TOME_ERR_INVALID, "image_tokenizer_param_offset: no parameter %d", which);
  return o;
}

extern "C" size_t tome_image_tokenizer_workspace_bytes(const tome_image_tokenizer_desc_t* d) {
  clear_error();
  ItGeom g;
  if (it_geometry(d, &g, "image_tokenizer_workspace_bytes") != TOME_OK) return 0;
  return g.total;
}

static int it_gemm(int m, int n, int k, const void* a, const void* b, void* c, int c_dtype, const float* bias, const void* residual,
                   cudaStream_t stream, const int* a_row_shift = nullptr, int shift_groups = 0) {
  tome_gemm_args_t ga;
  memset(&ga, 0, sizeof(ga));
  ga.m = m; ga.n = n; ga.k = k;
  ga.a = a; ga.lda = shift_groups ? k / shift_groups : k; ga.a_major = TOME_MAJOR_K;
  ga.a_row_shift = a_row_shift; ga.a_shift_groups = shift_groups;
  ga.b = b; ga.ldb = n; ga.b_major = TOME_MAJOR_MN;    // the Flax kernel layout [in, out] as is
  ga.c = c; ga.ldc = n; ga.c_dtype = c_dtype;
  ga.bias = bias;
  ga.residual = residual; ga.ldr = n;
  ga.k_splits = 1;
  return tome_gemm_bf16(&ga, nullptr, 0, stream);
}

// The front end; place == nullptr writes out [B, N, n_patches, E], else the bf16 sequence rows of `place`.
static int it_forward(const tome_image_tokenizer_desc_t* d, const void* image, const float* pf, const void* pb_,
                      const int32_t* row_tokens, const int32_t* col_tokens, void* out, const ItPlacement* place, void* workspace,
                      size_t workspace_bytes, cudaStream_t stream) {
  ItGeom g;
  int rc = it_geometry(d, &g, "image_tokenizer_fwd");
  if (rc != TOME_OK) return rc;
  TOME_CHECK(image && pf && pb_ && row_tokens && col_tokens && out && workspace, TOME_ERR_INVALID, "image_tokenizer_fwd: null argument");
  TOME_CHECK(workspace_bytes >= g.total, TOME_ERR_INVALID, "image_tokenizer_fwd: workspace too small (%zu < %zu)", workspace_bytes, g.total);
  TOME_CHECK((((uintptr_t)workspace) & 255) == 0 && (((uintptr_t)pb_ | (uintptr_t)pf | (uintptr_t)out) & 15) == 0, TOME_ERR_INVALID,
             "image_tokenizer_fwd: workspace must be 256-byte aligned, parameters / out 16-byte aligned");
  const __nv_bfloat16* pb = reinterpret_cast<const __nv_bfloat16*>(pb_);
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  __nv_bfloat16* col = reinterpret_cast<__nv_bfloat16*>(ws + g.off_col);
  __nv_bfloat16* y0 = reinterpret_cast<__nv_bfloat16*>(ws + g.off_y0);
  __nv_bfloat16* pooled = reinterpret_cast<__nv_bfloat16*>(ws + g.off_pool);
  __nv_bfloat16* xbuf[2] = {reinterpret_cast<__nv_bfloat16*>(ws + g.off_xa), reinterpret_cast<__nv_bfloat16*>(ws + g.off_xb)};
  float* dense = reinterpret_cast<float*>(ws + g.off_dense);
  float* part = reinterpret_cast<float*>(ws + g.off_part);
  float* stats = reinterpret_cast<float*>(ws + g.off_stats);
  float* ab = reinterpret_cast<float*>(ws + g.off_ab);
  __nv_bfloat16* hbuf = reinterpret_cast<__nv_bfloat16*>(ws + g.off_h);
  const int F = d->features, E = d->embed_dim, nchunk = F / 8;
  const int gn_threads = nchunk * std::max(1, IT_THREADS / nchunk);
  const long long pix_img = (long long)d->image_size * d->image_size * d->channels_in;
  const size_t pix_bytes = d->image_dtype == TOME_U8 ? 1 : 4;
  const size_t out_bytes = d->out_dtype == TOME_BF16 ? 2 : 4;
  auto nblk = [](long long n) { return (unsigned)((n + IT_THREADS - 1) / IT_THREADS); };

  for (int b0 = 0; b0 < d->batch; b0 += g.chunk_rows) {
    const int rows_b = std::min(g.chunk_rows, d->batch - b0);
    const long long imgs = (long long)rows_b * d->n_images, img0 = (long long)b0 * d->n_images;
    const long long m0 = imgs * g.np * g.o1 * g.o1, m2 = imgs * g.np * g.o2 * g.o2, mt = imgs * g.np;
    const long long R = (long long)d->n_images * g.np * g.o2 * g.o2;   // pixels of one batch row in the GroupNorm reduction
    const long long Rp = (long long)d->n_images * g.np * g.wp * g.wp;  // rows of one batch row on the (bordered) activation grid
    const long long m2p = imgs * g.np * g.wp * g.wp;
    const FastDiv fd_wp = make_fastdiv(g.wp);
    int shifts[9];
    for (int t9 = 0; t9 < 9; ++t9) shifts[t9] = (t9 / 3 - 1) * g.wp + (t9 % 3 - 1);
    const uint8_t* img = reinterpret_cast<const uint8_t*>(image) + (size_t)img0 * pix_img * pix_bytes;
    {
      const long long nv = m0 * (g.k0 / 8);
      Im2col0Args ia;
      ia.vpr = make_fastdiv(g.k0 / 8); ia.o1 = make_fastdiv(g.o1); ia.np = make_fastdiv(g.np); ia.ppd = make_fastdiv(g.ppd);
      ia.kw_c = make_fastdiv(d->conv_kernel * d->channels_in);
      ia.psize = d->patch_size; ia.stride = d->conv_stride; ia.img_w_c = d->image_size * d->channels_in; ia.c_in = d->channels_in;
      ia.normalize = d->normalize; ia.img_elems = pix_img;
      const bool words = (d->conv_kernel * d->channels_in) % 2 == 0 && (d->image_size * d->channels_in) % 2 == 0 &&
                         (d->conv_stride * d->channels_in) % 2 == 0 && (d->patch_size * d->channels_in) % 2 == 0 && (pix_img % 2) == 0;
      if (words) {
        // pixels -> normalised bf16 once, then the im2col moves 32-bit words (no per-byte loads, table lookups or packing)
        __nv_bfloat16* pix = reinterpret_cast<__nv_bfloat16*>(ws + g.off_pix);
        const long long np_ = imgs * pix_img;
        ProfScope prof(PROF_OTHER, (double)np_ * 3 + (double)nv * 16, 2, stream);
        if (d->image_dtype == TOME_U8)
          launch_k(it_pixels_bf16_kernel<uint8_t>, nblk((np_ + 7) / 8), IT_THREADS, 0, stream, img, pix, np_, d->normalize);
        else
          launch_k(it_pixels_bf16_kernel<float>, nblk((np_ + 7) / 8), IT_THREADS, 0, stream, reinterpret_cast<const float*>(img), pix, np_, d->normalize);
        TOME_CUDA(cudaGetLastError());
        launch_k(it_im2col0_words_kernel, nblk(nv / 2), IT_THREADS, 0, stream, reinterpret_cast<const uint32_t*>(pix), col, (uint32_t)nv, ia);
        TOME_CUDA(cudaGetLastError());
      } else {
        ProfScope prof(PROF_OTHER, (double)nv * 16, 1, stream);
        if (d->image_dtype == TOME_U8)
          launch_k(it_im2col0_kernel<uint8_t>, nblk(nv / 2), IT_THREADS, 0, stream, img, col, (uint32_t)nv, ia);
        else
          launch_k(it_im2col0_kernel<float>, nblk(nv / 2), IT_THREADS, 0, stream, reinterpret_cast<const float*>(img), col, (uint32_t)nv, ia);
        TOME_CUDA(cudaGetLastError());
      }
      rc = it_gemm((int)m0, F, g.k0, col, pb + it_offset(d, g, TOME_IT_CONV0_KERNEL), y0, TOME_BF16, pf + it_offset(d, g, TOME_IT_CONV0_BIAS),
                   nullptr, stream);
      if (rc != TOME_OK) return rc;
    }
    const FastDiv fd_chunk = make_fastdiv(nchunk), fd_o2 = make_fastdiv(g.o2);
    {
      const long long nv = m2 * nchunk;
      ProfScope prof(PROF_OTHER, (double)nv * 16 * (d->pool_window * d->pool_window + 1), 1, stream);
      launch_k(it_pool_kernel, nblk(nv), IT_THREADS, 0, stream, y0, pooled, (uint32_t)nv, fd_chunk, g.o1, fd_o2, d->pool_window, g.wp, g.pad);
      TOME_CUDA(cudaGetLastError());
    }
    const __nv_bfloat16* x = pooled;
    for (int blk = 0; blk < d->num_blocks; ++blk) {
      const int pi = TOME_IT_BLOCK0 + 4 * blk;
      {
        ProfScope prof(PROF_OTHER, (double)m2 * F * 2, 3, stream);
        launch_k(it_gn_partial_kernel, dim3(g.gn_ctas, rows_b), gn_threads, 0, stream, x, part, Rp, nchunk, fd_wp, g.pad);
        TOME_CUDA(cudaGetLastError());
        launch_k(it_gn_final_kernel, (unsigned)ceil_div(rows_b * d->num_groups, 4), 128, 0, stream, part, stats, rows_b, g.gn_ctas, F,
                 d->num_groups, R, d->gn_eps);
        TOME_CUDA(cudaGetLastError());
        launch_k(it_gn_fold_kernel, (unsigned)ceil_div(rows_b * F, 256), 256, 0, stream, stats, pf + it_offset(d, g, pi + 0),
                 pf + it_offset(d, g, pi + 1), ab, rows_b, F, d->num_groups);
        TOME_CUDA(cudaGetLastError());
      }
      {
        const long long nv = m2p * nchunk;
        ProfScope prof(PROF_OTHER, (double)nv * 32, 1, stream);
        launch_k(it_gn_gelu_kernel, nblk(nv), IT_THREADS, 0, stream, x, ab, hbuf, (uint32_t)nv, fd_chunk, make_fastdiv((uint32_t)Rp), fd_wp, g.pad);
        TOME_CUDA(cudaGetLastError());
      }
      __nv_bfloat16* y = xbuf[blk & 1];
      const bool last = blk == d->num_blocks - 1;
      if (g.pad) {
        // 3 x 3 SAME convolution as ONE GEMM over nine row-shifted windows of the bordered activation (no im2col rows): tap
        // (ty, tx) reads h at rows + (ty - 1) wp + (tx - 1); outputs on border positions are never read
        rc = it_gemm((int)m2p, F, 9 * F, hbuf, pb + it_offset(d, g, pi + 2), y, TOME_BF16, pf + it_offset(d, g, pi + 3),
                     nullptr, stream, shifts, 9);   // the residual of image_tokenizer.py:170 is added by it_compact_kernel
      } else {
        const long long nv = m2 * 9 * nchunk;
        {
          ProfScope prof(PROF_OTHER, (double)nv * 16, 1, stream);
          launch_k(it_im2col3_kernel, nblk(nv), IT_THREADS, 0, stream, hbuf, col, (uint32_t)nv, fd_chunk, fd_o2);
          TOME_CUDA(cudaGetLastError());
        }
        rc = it_gemm((int)m2, F, 9 * F, col, pb + it_offset(d, g, pi + 2), y, TOME_BF16, pf + it_offset(d, g, pi + 3),
                     last ? pooled : nullptr, stream);
      }
      if (rc != TOME_OK) return rc;
      x = y;
    }
    if (g.pad) {   // the Dense flattens (h, w, c) of the interior of x + pooled
      const long long nv = m2 * nchunk;
      ProfScope prof(PROF_OTHER, (double)nv * 48, 1, stream);
      launch_k(it_compact_kernel, nblk(nv), IT_THREADS, 0, stream, x, pooled, hbuf, (uint32_t)nv, fd_chunk, fd_o2, g.wp, g.pad);
      TOME_CUDA(cudaGetLastError());
      x = hbuf;
    }
    rc = it_gemm((int)mt, E, g.kd, x, pb + it_offset(d, g, TOME_IT_DENSE_KERNEL), dense, TOME_F32, pf + it_offset(d, g, TOME_IT_DENSE_BIAS),
                 nullptr, stream);
    if (rc != TOME_OK) return rc;
    {
      const long long nv = mt * (E / 4);
      ProfScope prof(PROF_OTHER, (double)nv * 16 * 2, 1, stream);
      if (place)
        launch_k(it_posadd_kernel<true>, nblk(nv), IT_THREADS, 0, stream, dense, pf + it_offset(d, g, TOME_IT_ROW_EMBED),
                 pf + it_offset(d, g, TOME_IT_COL_EMBED), row_tokens, col_tokens, out, nv, E, g.np, img0,
                 d->token_rows == 1 ? 0 : 1, d->position_interval, 1, *place);
      else
        launch_k(it_posadd_kernel<false>, nblk(nv), IT_THREADS, 0, stream, dense, pf + it_offset(d, g, TOME_IT_ROW_EMBED),
                 pf + it_offset(d, g, TOME_IT_COL_EMBED), row_tokens, col_tokens,
                 reinterpret_cast<uint8_t*>(out) + (size_t)img0 * g.np * E * out_bytes, nv, E, g.np, img0, d->token_rows == 1 ? 0 : 1,
                 d->position_interval, d->out_dtype == TOME_BF16 ? 1 : 0, ItPlacement{});
      TOME_CUDA(cudaGetLastError());
    }
  }
  return TOME_OK;
}

extern "C" int tome_image_tokenizer_fwd(const tome_image_tokenizer_desc_t* d, const void* image, const float* pf, const void* pb,
                                        const int32_t* row_tokens, const int32_t* col_tokens, void* out, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  clear_error();
  return it_forward(d, image, pf, pb, row_tokens, col_tokens, out, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
}

namespace tome {

int image_tokenizer_fwd_placed(const tome_image_tokenizer_desc_t* d, const void* image, const float* pf, const void* pb,
                               const int32_t* row_tokens, const int32_t* col_tokens, const ItPlacement& place, void* seq,
                               void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  TOME_CHECK(d != nullptr && d->out_dtype == TOME_BF16, TOME_ERR_INVALID, "image_tokenizer_fwd: sequence rows are bf16 (out_dtype)");
  TOME_CHECK(place.n_runs >= 1 && place.n_runs <= IT_MAX_ROW_RUNS && place.n_images == d->n_images, TOME_ERR_INVALID,
             "image_tokenizer_fwd: bad row placement");
  return it_forward(d, image, pf, pb, row_tokens, col_tokens, seq, &place, workspace, workspace_bytes, stream);
}

int fill_sequence_rows(const SeqRowSets& sets, int batch, int seq_tokens, int channels, void* seq, cudaStream_t stream) {
  if (sets.n_sets == 0) return TOME_OK;
  long long most = 0;
  for (int s = 0; s < sets.n_sets; ++s) most = std::max(most, (long long)batch * sets.n[s] * (channels / 8));
  ProfScope prof(PROF_OTHER, (double)most * sets.n_sets * 32, 1, stream);
  launch_k(it_seq_rows_kernel, dim3((unsigned)((most + IT_THREADS - 1) / IT_THREADS), sets.n_sets), IT_THREADS, 0, stream, sets,
           reinterpret_cast<__nv_bfloat16*>(seq), batch, seq_tokens, channels / 8);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

}  // namespace tome
