// K1 + K2: bipartite soft matching.
//
//   tome_sim_argmax   token_compression.py:72-83   L2-normalise, even/odd split, scores = a b^T, row max / arg max
//   tome_select_topr  token_compression.py:84-88   edge ranking (value desc, index desc on ties), index split,
//                                                  plus the derived maps the merge kernels consume
//
// Both are exact-index kernels: all comparisons are done on fp32 values with the reference's tie rules
// (arg max = first maximum; ranking = stable ascending argsort reversed; NaN ranks above everything, as in XLA /
// numpy), so indices are bit-exact given the same fp32 scores.  The similarity product is fp32 FMA on CUDA cores
// on purpose: it is 0.1 % of the block's FLOPs (SURVEY.md 8d) and fp32 keeps the arg max aligned with the fp32
// reference; the scores tile lives in registers and never reaches HBM unless scores_out is given.
#include "common.cuh"
#include "host_util.h"
#include "token_sets.cuh"

namespace tome {

// "candidate (v, j) beats the current best (bv, bj)" for a row arg max: larger value, NaN largest, first index wins.
__device__ __forceinline__ bool argmax_better(float v, int j, float bv, int bj) {
  const bool nv = v != v, nb = bv != bv;
  if (nv || nb) return nv && (!nb || j < bj);
  return v > bv || (v == bv && j < bj);
}

constexpr int SIM_TILE = 64;
constexpr int SIM_THREADS = 256;

__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}

template <typename T>
__device__ __forceinline__ float2 load2(const T* p);
template <>
__device__ __forceinline__ float2 load2<float>(const float* p) {
  return *reinterpret_cast<const float2*>(p);
}
template <>
__device__ __forceinline__ float2 load2<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
}

// ------------------------------------------------------------------------------------------------ K1, fp32 planes (dim != 64)
// The rows are normalised ONCE into the workspace (metric_norm_kernel: head mean, L2 norm, fp32, a rows and b rows in
// separate contiguous planes), so the score kernel only streams 16 KB tiles through a cp.async double buffer into the
// 4x4-per-thread fp32 loop on packed f32x2 FMAs (even-k and odd-k partial sums, added at the end).
// generic version: one warp per token row, 2 columns per lane per step (any even dim, any even strides)
template <typename T>
__global__ void __launch_bounds__(256)
metric_norm_kernel(const tome_metric_desc_t d, const __grid_constant__ SetTable tab, const T* __restrict__ src,
                   float* __restrict__ plane_a, float* __restrict__ plane_b) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tok = (long long)blockIdx.x * 8 + warp;   // b * T + t
  if (tok >= (long long)d.batch * d.tokens) return;
  const int b = (int)(tok / d.tokens), t = (int)(tok % d.tokens);
  const int dpad = (d.dim + 3) & ~3;
  const int ta = tab.a_off[tab.n], tb = tab.b_off[tab.n];
  const T* base = src + (long long)b * d.batch_stride + (long long)t * d.token_stride;
  bool odd;
  const int pr = set_plane_row(tab, t, odd);
  float* out = odd ? plane_b + ((long long)b * tb + pr) * dpad : plane_a + ((long long)b * ta + pr) * dpad;
  const float inv_h = 1.0f / (float)d.heads;
  float ss = 0.f;
  for (int c = 2 * lane; c < d.dim; c += 64) {  // pass 1: head mean -> out (un-normalised), sum of squares
    float2 acc = make_float2(0.f, 0.f);
    for (int h = 0; h < d.heads; ++h) {
      const float2 v = load2<T>(base + (long long)h * d.head_stride + c);
      acc.x += v.x;
      acc.y += v.y;
    }
    if (d.heads > 1) {  // jnp.mean over heads = sum / H
      acc.x *= inv_h;
      acc.y *= inv_h;
    }
    ss += acc.x * acc.x + acc.y * acc.y;
    *reinterpret_cast<float2*>(out + c) = acc;
  }
  ss = warp_sum(ss);
  const float nrm = sqrtf(ss);  // no epsilon (token_compression.py:72): a zero row becomes NaN
  for (int c = 2 * lane; c < dpad; c += 64) {   // pass 2: each lane rescales what it wrote
    float2 v = c < d.dim ? *reinterpret_cast<float2*>(out + c) : make_float2(0.f, 0.f);
    *reinterpret_cast<float2*>(out + c) = c < d.dim ? make_float2(v.x / nrm, v.y / nrm) : v;
  }
}

// bf16, dim == 64, 16-byte aligned rows (the stack's case): 8 lanes per token row, one 128-bit load per head per lane
__global__ void __launch_bounds__(256)
metric_norm64_kernel(const tome_metric_desc_t d, const __grid_constant__ SetTable tab, const __nv_bfloat16* __restrict__ src,
                     float* __restrict__ plane_a, float* __restrict__ plane_b) {
  const long long tok = ((long long)blockIdx.x * 256 + threadIdx.x) >> 3;   // b * T + t
  const int sub = threadIdx.x & 7;
  const bool valid = tok < (long long)d.batch * d.tokens;   // every lane stays for the shuffles
  const long long tk = valid ? tok : 0;
  const int b = (int)(tk / d.tokens), t = (int)(tk % d.tokens);
  const int ta = tab.a_off[tab.n], tb = tab.b_off[tab.n];
  const __nv_bfloat16* base = src + (long long)b * d.batch_stride + (long long)t * d.token_stride + sub * 8;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int h = 0; h < d.heads; ++h) {
    const uint4 v = ld_nc_v4(base + (long long)h * d.head_stride);
    acc[0] += bf16_lo(v.x); acc[1] += bf16_hi(v.x); acc[2] += bf16_lo(v.y); acc[3] += bf16_hi(v.y);
    acc[4] += bf16_lo(v.z); acc[5] += bf16_hi(v.z); acc[6] += bf16_lo(v.w); acc[7] += bf16_hi(v.w);
  }
  float ss = 0.f;
  const float inv_h = 1.0f / (float)d.heads;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (d.heads > 1) acc[i] *= inv_h;
    ss += acc[i] * acc[i];
  }
  ss += __shfl_xor_sync(0xffffffffu, ss, 1);
  ss += __shfl_xor_sync(0xffffffffu, ss, 2);
  ss += __shfl_xor_sync(0xffffffffu, ss, 4);
  const float nrm = sqrtf(ss);
  if (valid) {
    bool odd;
    const int pr = set_plane_row(tab, t, odd);
    float* out = (odd ? plane_b + ((long long)b * tb + pr) * 64 : plane_a + ((long long)b * ta + pr) * 64) + sub * 8;
    reinterpret_cast<float4*>(out)[0] = make_float4(acc[0] / nrm, acc[1] / nrm, acc[2] / nrm, acc[3] / nrm);
    reinterpret_cast<float4*>(out)[1] = make_float4(acc[4] / nrm, acc[5] / nrm, acc[6] / nrm, acc[7] / nrm);
  }
}

__device__ __forceinline__ void cp_async_16(void* dst_smem, const void* src, bool valid) {
  const uint32_t n = valid ? 16u : 0u;  // src-size 0: the 16 bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(n) : "memory");
}

// tile of SIM_TILE normalised rows (plane row r0 + i, dpad floats each) -> smem rows of pitch dpad + 4
__device__ __forceinline__ void load_tile_async(float* dst, const float* plane, int r0, int nrows, int dpad) {
  const int pitch = dpad + 4, vpr = dpad >> 2;
  for (int i = threadIdx.x; i < SIM_TILE * vpr; i += SIM_THREADS) {
    const int rr = i / vpr, v = i - rr * vpr;
    const bool ok = r0 + rr < nrows;
    cp_async_16(dst + rr * pitch + 4 * v, plane + (long long)(ok ? r0 + rr : 0) * dpad + 4 * v, ok);
  }
}

// Dynamic shared memory of sim_argmax_planes_kernel: the a tile and two b tiles of SIM_TILE rows, pitch pad4(dim) + 4 floats.
// It bounds the metric width the library accepts: the widest even dim whose tiles fit the 227 KB a block may opt into.
constexpr size_t sim_planes_smem(int dim) { return (size_t)3 * SIM_TILE * (((dim + 3) & ~3) + 4) * sizeof(float); }
constexpr int sim_max_dim() {
  int dim = 2;
  while (sim_planes_smem(dim + 2) <= 232448) dim += 2;
  return dim;
}
constexpr int SIM_MAX_DIM = sim_max_dim();
static_assert(SIM_MAX_DIM == 296, "include/tome_b200.h states the accepted dims of tome_sim_argmax");

__global__ void __launch_bounds__(SIM_THREADS)
sim_argmax_planes_kernel(const tome_metric_desc_t d, const __grid_constant__ SetTable tab, const float* __restrict__ plane_a,
                         const float* __restrict__ plane_b, float* __restrict__ node_max, int32_t* __restrict__ node_idx,
                         float* __restrict__ scores_out) {
  extern __shared__ float4 sm4[];
  float* sm = reinterpret_cast<float*>(sm4);
  const int dpad = (d.dim + 3) & ~3, pitch = dpad + 4;
  float* sa = sm;
  float* sb0 = sm + SIM_TILE * pitch;
  const int b = blockIdx.y;
  // CTA = (a-row tile of a token set, batch row): rows and columns are the set's own even and odd tokens
  const int set = set_of(tab.tile_off, tab.n, blockIdx.x);
  const int ta = (tab.len[set] + 1) / 2, tb = tab.len[set] / 2;
  const int a0 = (blockIdx.x - tab.tile_off[set]) * SIM_TILE;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const long long arow = (long long)b * tab.a_off[tab.n] + tab.a_off[set];   // node_max / plane A row of the set's token 0
  const float* pa = plane_a + arow * dpad;
  const float* pb = plane_b + ((long long)b * tab.b_off[tab.n] + tab.b_off[set]) * dpad;
  float* dump = scores_out ? scores_out + (long long)b * tab.sc_off[tab.n] + tab.sc_off[set] : nullptr;
  const int n_bt = (tb + SIM_TILE - 1) / SIM_TILE;

  load_tile_async(sa, pa, a0, ta, dpad);
  load_tile_async(sb0, pb, 0, tb, dpad);
  asm volatile("cp.async.commit_group;" ::: "memory");

  float best_v[4];
  int best_j[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    best_v[i] = -INFINITY;
    best_j[i] = 0x7fffffff;
  }
  for (int bt = 0; bt < n_bt; ++bt) {
    const int b0 = bt * SIM_TILE;
    float* sb = sb0 + (bt & 1) * SIM_TILE * pitch;
    if (bt + 1 < n_bt) load_tile_async(sb0 + ((bt + 1) & 1) * SIM_TILE * pitch, pb, b0 + SIM_TILE, tb, dpad);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");  // tile bt (and the a tile) have landed; tile bt+1 may be in flight
    __syncthreads();
    // packed f32x2 FMAs (scalar FFMA issues at half rate on sm_100): lane .x accumulates the even k, lane .y the odd k
    float2 acc2[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc2[i][j] = make_float2(0.f, 0.f);
    // row pointers hoisted out of the k loop: IMAD shares the FMA pipe with FFMA2, so address arithmetic inside the
    // loop costs FMA throughput one for one
    const float4* ap[4];
    const float4* bp[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      ap[i] = reinterpret_cast<const float4*>(sa + (ty + 16 * i) * pitch);
      bp[i] = reinterpret_cast<const float4*>(sb + (tx + 16 * i) * pitch);
    }
#pragma unroll 4
    for (int c4 = 0; c4 < (dpad >> 2); ++c4) {  // one 128-bit shared-memory read feeds 4 k-steps: 8 LDS.128 per 32 FFMA2
      float4 av[4], bv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) av[i] = ap[i][c4];
#pragma unroll
      for (int j = 0; j < 4; ++j) bv[j] = bp[j][c4];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          acc2[i][j] = __ffma2_rn(make_float2(av[i].x, av[i].y), make_float2(bv[j].x, bv[j].y), acc2[i][j]);
          acc2[i][j] = __ffma2_rn(make_float2(av[i].z, av[i].w), make_float2(bv[j].z, bv[j].w), acc2[i][j]);
        }
    }
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = acc2[i][j].x + acc2[i][j].y;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int ai = a0 + ty + 16 * i;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int bj = b0 + tx + 16 * j;
        if (ai < ta && bj < tb) {
          float s = acc[i][j];
          if ((d.class_token && ai == 0) || (d.distill_token && bj == 0)) s = -INFINITY;  // :77-80
          if (dump) dump[(long long)ai * tb + bj] = s;
          if (argmax_better(s, bj, best_v[i], best_j[i])) {
            best_v[i] = s;
            best_j[i] = bj;
          }
        }
      }
    }
    __syncthreads();  // tile bt fully consumed before tile bt+2 overwrites its buffer
  }
  if (n_bt == 0) asm volatile("cp.async.wait_all;" ::: "memory");   // a one-token set: no b tile, the a tile still in flight
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best_v[i], o);
      const int oj = __shfl_xor_sync(0xffffffffu, best_j[i], o);
      if (argmax_better(ov, oj, best_v[i], best_j[i])) {
        best_v[i] = ov;
        best_j[i] = oj;
      }
    }
    const int ai = a0 + ty + 16 * i;
    if (tx == 0 && ai < ta) {
      node_max[arow + ai] = best_v[i];
      node_idx[arow + ai] = best_j[i] == 0x7fffffff ? 0 : best_j[i];
    }
  }
}

// ------------------------------------------------------------------------------------------------ K1 on the tensor cores
// scores = a b^T is a dense contraction, so it belongs on tcgen05 -- but the arg max must come out of fp32 scores that
// agree with the reference's fp32 arithmetic (scores within 1e-5, indices exact from the scores the kernel itself used).
// A bf16 MMA alone cannot do that; a SPLIT one can: every normalised fp32 value is written as v = h + m + l with h = bf16(v),
// m = bf16(v - h), l = bf16(v - h - m) (3 x 8 bits: the 24-bit significand exactly), and
//   a . b  =  sum over (hh, hm, mh, hl, lh, mm) products  +  terms below 2^-24 |a||b|,
// each bf16 x bf16 product exact in the fp32 accumulator.  metric_split64_kernel writes every row as the three 64-wide chunks
// [h | m | l] (384 bytes per token; fp32 would be 256), and the score tile is six chunk products accumulated into ONE TMEM
// tile -- 24 tcgen05.mma 128 x 128 x 16 steps -- double-buffered so the epilogue warps (thread = a row) take the running row
// max / first arg max of tile j from tensor memory while tile j + 1 is being computed.  (A first version stored the six
// operand chunks per row explicitly, 768 B per token: its 295 MB of L2 -> SM traffic per call, not the tensor pipe, set
// its 93 us -- profiles/r02_sim_argmax_tc.md.)
//   warp 4  TMA: the a tile's three chunks once (48 KB, resident), then the b tiles chunk by chunk through a 3-slot ring
//   warp 5  MMA issuer: per b chunk h: a_h, a_m, a_l;  m: a_h, a_m;  l: a_h        warps 0..3  epilogue
constexpr int SIMT_BM = 128, SIMT_BN = 128, SIMT_CHUNKS = 3, SIMT_SLOTS = 3, SIMT_ROW = 192;
constexpr int SIMT_CHUNK_BYTES = 128 * 64 * 2;   // 16 KB: 128 rows x 64 bf16, 128B-swizzled
constexpr int SIMT_SMEM = (SIMT_CHUNKS + SIMT_SLOTS) * SIMT_CHUNK_BYTES + 256 + 1024;
constexpr int SIMT_THREADS = 192;

// bf16, dim == 64, 16-byte aligned rows: 8 lanes per token row; head mean, L2 norm (no epsilon), three-way bf16 split
__global__ void __launch_bounds__(256)
metric_split64_kernel(const tome_metric_desc_t d, const __grid_constant__ SetTable tab, const __nv_bfloat16* __restrict__ src,
                      __nv_bfloat16* __restrict__ plane_a, __nv_bfloat16* __restrict__ plane_b) {
  const long long tok = ((long long)blockIdx.x * 256 + threadIdx.x) >> 3;   // b * T + t
  const int sub = threadIdx.x & 7;
  const bool valid = tok < (long long)d.batch * d.tokens;   // every lane stays for the shuffles
  const long long tk = valid ? tok : 0;
  const int b = (int)(tk / d.tokens), t = (int)(tk % d.tokens);
  const int ta = tab.a_off[tab.n], tb = tab.b_off[tab.n];
  const __nv_bfloat16* base = src + (long long)b * d.batch_stride + (long long)t * d.token_stride + sub * 8;
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int h = 0; h < d.heads; ++h) {
    const uint4 v = ld_nc_v4(base + (long long)h * d.head_stride);
    acc[0] += bf16_lo(v.x); acc[1] += bf16_hi(v.x); acc[2] += bf16_lo(v.y); acc[3] += bf16_hi(v.y);
    acc[4] += bf16_lo(v.z); acc[5] += bf16_hi(v.z); acc[6] += bf16_lo(v.w); acc[7] += bf16_hi(v.w);
  }
  float ss = 0.f;
  const float inv_h = 1.0f / (float)d.heads;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (d.heads > 1) acc[i] *= inv_h;
    ss += acc[i] * acc[i];
  }
  ss += __shfl_xor_sync(0xffffffffu, ss, 1);
  ss += __shfl_xor_sync(0xffffffffu, ss, 2);
  ss += __shfl_xor_sync(0xffffffffu, ss, 4);
  const float nrm = sqrtf(ss);
  if (!valid) return;
  float hi[8], mi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float v = acc[i] / nrm;
    hi[i] = __bfloat162float(__float2bfloat16_rn(v));
    const float r1 = v - hi[i];                       // exact: v and hi agree in their leading bits
    mi[i] = __bfloat162float(__float2bfloat16_rn(r1));
    lo[i] = __bfloat162float(__float2bfloat16_rn(r1 - mi[i]));
  }
  const uint4 wh = pack8(hi), wm = pack8(mi), wl = pack8(lo);
  bool odd;
  const int pr = set_plane_row(tab, t, odd);
  uint4* out = reinterpret_cast<uint4*>((odd ? plane_b + ((long long)b * tb + pr) * SIMT_ROW : plane_a + ((long long)b * ta + pr) * SIMT_ROW)) + sub;
  out[0] = wh;    // chunk c starts 64 elements = 8 uint4 further
  out[8] = wm;
  out[16] = wl;
}

// any dtype / even strides, dim == 64: one warp per token row, two columns per lane (the fp32 `metric` argument of
// bipartite_soft_matching takes this one)
template <typename T>
__global__ void __launch_bounds__(256)
metric_split_kernel(const tome_metric_desc_t d, const __grid_constant__ SetTable tab, const T* __restrict__ src,
                    __nv_bfloat16* __restrict__ plane_a, __nv_bfloat16* __restrict__ plane_b) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tok = (long long)blockIdx.x * 8 + warp;   // b * T + t
  if (tok >= (long long)d.batch * d.tokens) return;
  const int b = (int)(tok / d.tokens), t = (int)(tok % d.tokens);
  const int ta = tab.a_off[tab.n], tb = tab.b_off[tab.n];
  const T* base = src + (long long)b * d.batch_stride + (long long)t * d.token_stride + 2 * lane;
  float2 acc = make_float2(0.f, 0.f);
  for (int h = 0; h < d.heads; ++h) {
    const float2 v = load2<T>(base + (long long)h * d.head_stride);
    acc.x += v.x;
    acc.y += v.y;
  }
  if (d.heads > 1) {
    const float inv_h = 1.0f / (float)d.heads;
    acc.x *= inv_h;
    acc.y *= inv_h;
  }
  const float nrm = sqrtf(warp_sum(acc.x * acc.x + acc.y * acc.y));
  float v[2] = {acc.x / nrm, acc.y / nrm}, hi[2], mi[2], lo[2];
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    hi[i] = __bfloat162float(__float2bfloat16_rn(v[i]));
    const float r1 = v[i] - hi[i];
    mi[i] = __bfloat162float(__float2bfloat16_rn(r1));
    lo[i] = __bfloat162float(__float2bfloat16_rn(r1 - mi[i]));
  }
  const uint32_t wh = pack_bf16(hi[0], hi[1]), wm = pack_bf16(mi[0], mi[1]), wl = pack_bf16(lo[0], lo[1]);
  bool odd;
  const int pr = set_plane_row(tab, t, odd);
  uint32_t* out = reinterpret_cast<uint32_t*>(odd ? plane_b + ((long long)b * tb + pr) * SIMT_ROW : plane_a + ((long long)b * ta + pr) * SIMT_ROW) + lane;
  out[0] = wh;            // chunk c starts 64 elements = 32 words further
  out[32] = wm;
  out[64] = wl;
}

__global__ void __launch_bounds__(SIMT_THREADS, 2)
sim_argmax_tc_kernel(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_b, const tome_metric_desc_t d,
                     const __grid_constant__ SetTable tab, float* __restrict__ node_max, int32_t* __restrict__ node_idx,
                     float* __restrict__ scores_out) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_a = smem;                                   // chunk c at c * 16 KB
  uint8_t* s_b = s_a + SIMT_CHUNKS * SIMT_CHUNK_BYTES;   // ring slot i at i * 16 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_b + SIMT_SLOTS * SIMT_CHUNK_BYTES);
  uint64_t* a_full = bars;            // 1
  uint64_t* b_full = bars + 1;        // [SIMT_SLOTS] (room for 4)
  uint64_t* b_empty = bars + 5;       // [SIMT_SLOTS] (room for 4)
  uint64_t* s_full = bars + 9;        // [2] score tile in TMEM buffer jt & 1
  uint64_t* s_free = bars + 11;       // [2] 128 arrivals: the epilogue has read it
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA = (a-row tile of a token set, batch row).  The tiles are read at the set's rows of the planes: a rows past the set's
  // end (the next set's, or TMA zero fill) are never stored, b columns past it are skipped in the epilogue (j < tb).
  const int b = blockIdx.y;
  const int set = set_of(tab.tile_off, tab.n, blockIdx.x);
  const int at = blockIdx.x - tab.tile_off[set];
  const int ta = (tab.len[set] + 1) / 2, tb = tab.len[set] / 2;
  const int n_bt = (tb + SIMT_BN - 1) / SIMT_BN;

  if (threadIdx.x == 0) {
    mbar_init(a_full, 1);
    for (int i = 0; i < SIMT_SLOTS; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], SIMT_BM);
    }
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_b);
  }
  if (warp == 5) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    if (lane == 0) {
      mbar_expect_tx(a_full, SIMT_CHUNKS * SIMT_CHUNK_BYTES);
      for (int c = 0; c < SIMT_CHUNKS; ++c)
        tma_load_3d(s_a + c * SIMT_CHUNK_BYTES, &tm_a, a_full, c * 64, tab.a_off[set] + at * SIMT_BM, b);
      int item = 0;
      for (int jt = 0; jt < n_bt; ++jt)
        for (int c = 0; c < SIMT_CHUNKS; ++c, ++item) {
          const int slot = item % SIMT_SLOTS;
          mbar_wait(&b_empty[slot], ((item / SIMT_SLOTS) & 1) ^ 1);
          mbar_expect_tx(&b_full[slot], SIMT_CHUNK_BYTES);
          tma_load_3d(s_b + slot * SIMT_CHUNK_BYTES, &tm_b, &b_full[slot], c * 64, tab.b_off[set] + jt * SIMT_BN, b);
        }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(SIMT_BM, SIMT_BN, false, false);
      mbar_wait(a_full, 0);
      int item = 0;
      for (int jt = 0; jt < n_bt; ++jt) {
        if (jt >= 2) {
          mbar_wait(&s_free[jt & 1], ((jt - 2) >> 1) & 1);
          tc_fence_after();
        }
        const uint32_t td = tmem_base + (jt & 1) * SIMT_BN;
        for (int c = 0; c < SIMT_CHUNKS; ++c, ++item) {   // b chunk c (h, m, l) meets the a chunks 0 .. 2 - c: hh mh lh | hm mm | hl
          const int slot = item % SIMT_SLOTS;
          mbar_wait(&b_full[slot], (item / SIMT_SLOTS) & 1);
          tc_fence_after();
          const uint32_t ab = smem_u32(s_b + slot * SIMT_CHUNK_BYTES);
          for (int ca = 0; ca < SIMT_CHUNKS - c; ++ca) {
            const uint32_t aa = smem_u32(s_a + ca * SIMT_CHUNK_BYTES);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma_bf16(td, make_smem_desc(aa + k * 32, 16, 1024), make_smem_desc(ab + k * 32, 16, 1024), idesc,
                        (c > 0 || ca > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&b_empty[slot]);
        }
        umma_commit(&s_full[jt & 1]);
      }
    }
  } else {
    const int row = threadIdx.x;  // TMEM lane
    const int ai = at * SIMT_BM + row;
    const uint32_t lane_sel = ((uint32_t)(warp * 32)) << 16;
    const bool row_ok = ai < ta;
    const bool row_protected = d.class_token && ai == 0;   // :77-78
    float bv = -INFINITY;
    int bj = 0x7fffffff;
    const long long arow = (long long)b * tab.a_off[tab.n] + tab.a_off[set] + ai;
    float* dump = (scores_out && row_ok) ? scores_out + (long long)b * tab.sc_off[tab.n] + tab.sc_off[set] + (long long)ai * tb : nullptr;
    for (int jt = 0; jt < n_bt; ++jt) {
      mbar_wait(&s_full[jt & 1], (jt >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < SIMT_BN; c0 += 32) {
        float v[32];
        tmem_ld_f32x32(tmem_base + (jt & 1) * SIMT_BN + lane_sel + c0, v);
        tmem_ld_wait();
        const int j0 = jt * SIMT_BN + c0;
        if (j0 < tb) {   // uniform
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int j = j0 + i;
            float sc = v[i];
            if (row_protected || (d.distill_token && j == 0)) sc = -INFINITY;  // :77-80
            if (j < tb) {
              if (dump) dump[j] = sc;
              // first maximum; NaN is the greatest and the first NaN stays (numpy / jax argmax)
              if (sc > bv || (sc != sc && bv == bv)) {
                bv = sc;
                bj = j;
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&s_free[jt & 1]);
    }
    if (row_ok) {
      node_max[arow] = bv;
      node_idx[arow] = bj == 0x7fffffff ? 0 : bj;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

// ------------------------------------------------------------------------------------------------ K2
// Rank order of jnp.argsort(node_max)[:, ::-1] (token_compression.py:84): value descending with NaN greatest, ties by
// index DEscending.  One CTA per batch row sorts 64-bit keys (order-preserving image of the float in the high word, index in
// the low word) with a bitonic network in shared memory -- O(n log^2 n) compare-exchanges instead of the round-1 rank-by-
// count (n^2 comparisons: 1.2 ms per call at T = 8192) -- and a second sort of (destination, rank) pairs gives every merged
// source its slot in the CSR lists, keeping the rank order inside a destination that the reference's sequential adds need.
__device__ __forceinline__ unsigned long long rank_key(float v, int i) {
  uint32_t u = __float_as_uint(v);
  if (v != v) u = 0xFFFFFFFFu;                 // NaN sorts above every number (numpy / jax argsort order)
  else if (v == 0.f) u = 0x80000000u;          // -0 == +0
  else u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (uint32_t)i;
}

// in-place bitonic sort of n (a power of two) keys, DEscending; every thread of the CTA takes part
__device__ __forceinline__ void bitonic_sort_desc(unsigned long long* keys, int n, int tid, int nt) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n; i += nt) {
        const int l = i ^ j;
        if (l > i) {
          const unsigned long long a = keys[i], b = keys[l];
          const bool desc = (i & k) == 0;
          if (desc ? a < b : a > b) {
            keys[i] = b;
            keys[l] = a;
          }
        }
      }
      __syncthreads();
    }
  }
}

constexpr int SEL_THREADS = 1024;
__host__ __device__ inline int sel_pow2(int n) { int p = 1; while (p < n) p <<= 1; return p; }

__global__ void __launch_bounds__(SEL_THREADS)
select_topr_kernel(const tome_plan_shape_t s, const __grid_constant__ SetTable tab, const float* __restrict__ node_max,
                   const int32_t* __restrict__ node_idx, const tome_plan_t p) {
  extern __shared__ __align__(8) unsigned char sel_raw[];
  // CTA = (token set, batch row); every index below is local to the set, the arrays are concatenated set by set
  const int set = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
  const int T = tab.len[set], r = tab.r[set];
  const int ta = (T + 1) / 2, tb = T / 2;
  const long long arow = (long long)b * tab.a_off[tab.n] + tab.a_off[set];    // node_max / node_idx / edge_idx
  const long long rrow = (long long)b * tab.r_off[tab.n] + tab.r_off[set];    // dst_idx / dst_src
  const long long orow = (long long)b * tab.off_off[tab.n] + tab.off_off[set];  // dst_off
  int32_t* row_map = p.row_map + (long long)b * s.tokens + tab.start[set];
  const int out0 = tab.out_off[set];   // global output row of the set's first row
  if (r == 0) {   // the set is copied unchanged: identity ranking and row map, no sources
    for (int i = tid; i < ta; i += nt) p.edge_idx[arow + i] = i;
    for (int j = tid; j <= tb; j += nt) p.dst_off[orow + j] = 0;
    for (int t = tid; t < T; t += nt) row_map[t] = out0 + t;
    return;
  }
  const int n2 = sel_pow2(ta);
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(sel_raw);  // [n2]
  int* nidx = reinterpret_cast<int*>(keys + n2);   // [ta]
  int* rnk = nidx + ta;                            // [ta]   rank of even token i
  int* cnt = rnk + ta;                             // [tb+1] counts then exclusive offsets
  int* part = cnt + tb + 1;                        // [SEL_THREADS] scan partials

  for (int i = tid; i < n2; i += nt) {
    if (i < ta) {
      keys[i] = rank_key(node_max[arow + i], i);
      nidx[i] = node_idx[arow + i];
    } else {
      keys[i] = 0ull;   // below every real key (the smallest real high word is that of -inf, 0x007FFFFF)
    }
  }
  for (int j = tid; j <= tb; j += nt) cnt[j] = 0;
  __syncthreads();
  bitonic_sort_desc(keys, n2, tid, nt);
  for (int rk = tid; rk < ta; rk += nt) {
    const int i = (int)(uint32_t)keys[rk];
    rnk[i] = rk;
    p.edge_idx[arow + rk] = i;
  }
  __syncthreads();
  for (int i = tid; i < r; i += nt) {
    const int d = nidx[(int)(uint32_t)keys[i]];
    p.dst_idx[rrow + i] = d;
    atomicAdd(&cnt[d], 1);
  }
  __syncthreads();
  // exclusive scan of cnt[0..tb) -> offsets; cnt[tb] = r
  {
    const int per = (tb + nt - 1) / nt;
    const int lo = tid * per, hi = min(lo + per, tb);
    int sum = 0;
    for (int j = lo; j < hi; ++j) sum += cnt[j];
    part[tid] = sum;
    __syncthreads();
    for (int o = 1; o < nt; o <<= 1) {
      const int add = tid >= o ? part[tid - o] : 0;
      __syncthreads();
      part[tid] += add;
      __syncthreads();
    }
    int run = part[tid] - sum;  // exclusive prefix of this thread's chunk
    for (int j = lo; j < hi; ++j) {
      const int c = cnt[j];
      cnt[j] = run;
      run += c;
    }
    if (tid == 0) cnt[tb] = r;
    __syncthreads();
  }
  for (int j = tid; j <= tb; j += nt) p.dst_off[orow + j] = cnt[j];
  // placement: the merged sources sorted by (destination, rank) are the CSR lists in order -- sources of one destination
  // keep their rank order (the reference adds them in that order, :100-101).  Descending sort of the complemented key.
  {
    const int r2 = sel_pow2(r);
    // entry i is rebuilt in place from the ranking key at the same index (read and written by the same thread only)
    for (int i = tid; i < r2; i += nt) {
      unsigned long long k = 0ull;
      if (i < r) {
        const int src = (int)(uint32_t)keys[i];
        const int d = nidx[src];
        // (d, rank i) ascending == ~(d, i) descending; the even-token index rides along through part of the key: 20 bits of
        // destination, 20 bits of rank, 24 bits of source index (T <= 2^20 is far beyond the shared-memory limit anyway)
        k = ~(((unsigned long long)d << 44) | ((unsigned long long)i << 24)) & ~0xFFFFFFull;
        k |= (unsigned long long)src;
      }
      keys[i] = k;
    }
    __syncthreads();
    bitonic_sort_desc(keys, r2, tid, nt);
    for (int q = tid; q < r; q += nt) p.dst_src[rrow + q] = (int)(keys[q] & 0xFFFFFFull);
  }
  // row map: where every input token lands in the concatenation [unm | dst] (:103-108)
  const int n_unm = ta - r;
  for (int t = tid; t < T; t += nt) {
    int row;
    const int h = t >> 1;
    if (t & 1) {
      row = s.distill_token ? (h == 0 ? 1 : n_unm + h) : n_unm + h;
    } else {
      const int rk = rnk[h];
      if (rk >= r) {
        const int u = rk - r;
        row = s.distill_token ? (u == 0 ? 0 : u + 1) : u;
      } else {
        const int j = nidx[h];
        row = s.distill_token ? (j == 0 ? 1 : n_unm + j) : n_unm + j;
      }
    }
    row_map[t] = out0 + row;
  }
}

}  // namespace tome

using namespace tome;

extern "C" int tome_clamp_r(int tokens, int r, int class_token, int distill_token) {
  const int prot = (class_token ? 1 : 0) + (distill_token ? 1 : 0);
  int m = (tokens - prot) / 2;
  if (r > m) r = m;
  return r > 0 ? r : 0;
}

// the tensor-core path (split-bf16 K = 384 contraction) whenever the input allows it, else fp32 CUDA-core planes
static bool sim_tc_eligible(const tome_metric_desc_t* d) { return d->dim == 64; }
static bool sim_fast64(const tome_metric_desc_t* d, const void* src) {   // 128-bit loads, 8 lanes per row
  return d->dtype == TOME_BF16 && d->dim == 64 && d->token_stride % 8 == 0 && d->batch_stride % 8 == 0 &&
         d->head_stride % 8 == 0 && ((uintptr_t)src & 15) == 0;
}

// The normalised metric in the workspace: plane A (the ta even tokens of every batch row, set after set), then plane B (the tb
// odd ones), packed.  A token's row is three bf16 chunks of 64 (SIMT_ROW) on the tensor-core path, else dim floats padded to a
// multiple of 4.  ta + tb = tokens whatever the sets, so the size does not depend on them.
struct SimPlanes { uint8_t *a, *b; size_t total; };
static SimPlanes sim_planes(const tome_metric_desc_t* d, size_t ta, void* base) {
  const size_t row = sim_tc_eligible(d) ? SIMT_ROW * sizeof(__nv_bfloat16) : ((d->dim + 3) & ~3) * sizeof(float);
  uint8_t* a = reinterpret_cast<uint8_t*>(base);
  return {a, a ? a + d->batch * ta * row : nullptr, (size_t)d->batch * d->tokens * row};
}

extern "C" size_t tome_sim_argmax_workspace_bytes(const tome_metric_desc_t* d) {
  if (!d || d->batch <= 0 || d->tokens <= 0 || d->dim <= 0) return 0;
  return sim_planes(d, (d->tokens + 1) / 2, nullptr).total;
}

extern "C" int tome_sim_argmax(const tome_metric_desc_t* d, const void* src, float* node_max, int32_t* node_idx,
                               float* scores_out, void* workspace, size_t workspace_bytes, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(d && src && node_max && node_idx, TOME_ERR_INVALID, "sim_argmax: null argument");
  TOME_CHECK(d->batch > 0 && d->tokens >= 2 && d->heads >= 1, TOME_ERR_INVALID,
             "sim_argmax: need batch > 0, tokens >= 2, heads >= 1 (got %d, %d, %d)", d->batch, d->tokens, d->heads);
  TOME_CHECK(d->dim >= 2 && d->dim % 2 == 0 && d->dim <= SIM_MAX_DIM, TOME_ERR_INVALID,
             "sim_argmax: metric dim must be even and in [2, %d] (got %d)", SIM_MAX_DIM, d->dim);
  TOME_CHECK(d->dtype == TOME_BF16 || d->dtype == TOME_F32, TOME_ERR_INVALID, "sim_argmax: dtype must be bf16 or f32");
  TOME_CHECK(d->token_stride % 2 == 0 && d->batch_stride % 2 == 0 && d->head_stride % 2 == 0, TOME_ERR_INVALID,
             "sim_argmax: strides must be even (vector loads)");
  TOME_CHECK(d->batch <= 65535, TOME_ERR_INVALID, "sim_argmax: batch too large for one launch");
  SetTable tab;
  if (int rc = make_set_table(d->sets, d->tokens, -1, d->class_token, d->distill_token, &tab, "sim_argmax")) return rc;
  const int ta = tab.a_off[tab.n], tb = tab.b_off[tab.n];   // even / odd tokens of a batch row, over all sets
  const SimPlanes planes = sim_planes(d, ta, workspace);
  TOME_CHECK(workspace != nullptr && workspace_bytes >= planes.total && ((uintptr_t)workspace & 15) == 0, TOME_ERR_INVALID,
             "sim_argmax: workspace must be 16-byte aligned and hold tome_sim_argmax_workspace_bytes = %zu bytes (got %p, %zu bytes)",
             planes.total, workspace, workspace_bytes);
  const long long toks = (long long)d->batch * d->tokens;
  ProfScope prof(PROF_SIM, 2.0 * d->batch * (double)tab.sc_off[tab.n] * d->dim, 2, stream);
  if (sim_tc_eligible(d)) {
    __nv_bfloat16* pa = reinterpret_cast<__nv_bfloat16*>(planes.a);
    __nv_bfloat16* pb = reinterpret_cast<__nv_bfloat16*>(planes.b);
    if (sim_fast64(d, src))
      launch_k(metric_split64_kernel, (unsigned)((toks * 8 + 255) / 256), 256, 0, stream, *d, tab, reinterpret_cast<const __nv_bfloat16*>(src), pa, pb);
    else if (d->dtype == TOME_BF16)
      launch_k(metric_split_kernel<__nv_bfloat16>, (unsigned)((toks + 7) / 8), 256, 0, stream, *d, tab, reinterpret_cast<const __nv_bfloat16*>(src), pa, pb);
    else
      launch_k(metric_split_kernel<float>, (unsigned)((toks + 7) / 8), 256, 0, stream, *d, tab, reinterpret_cast<const float*>(src), pa, pb);
    TOME_CUDA(cudaGetLastError());
    CUtensorMap tma_a, tma_b;
    if (int rc = make_tmap_3d_bf16(&tma_a, pa, SIMT_ROW, ta, d->batch, SIMT_ROW, (uint64_t)ta * SIMT_ROW, SIMT_BM)) return rc;
    // tb == 0 (every set a single token): no b tile is ever loaded, the map only has to be well-formed
    const int tbm = tb > 0 ? tb : 1;
    if (int rc = make_tmap_3d_bf16(&tma_b, pb, SIMT_ROW, tbm, d->batch, SIMT_ROW, (uint64_t)tbm * SIMT_ROW, SIMT_BN)) return rc;
    static DynSmemOnce once;
    TOME_CUDA(ensure_dyn_smem(sim_argmax_tc_kernel, SIMT_SMEM, once));
    const int tiles = set_tiles(&tab, SIMT_BM);
    TOME_CUDA(launch_k(sim_argmax_tc_kernel, dim3(tiles, d->batch), SIMT_THREADS, SIMT_SMEM, stream, tma_a, tma_b, *d, tab,
                       node_max, node_idx, scores_out));
    return TOME_OK;
  }
  float* plane_a = reinterpret_cast<float*>(planes.a);
  float* plane_b = reinterpret_cast<float*>(planes.b);
  const unsigned nblk = (unsigned)((toks + 7) / 8);
  if (sim_fast64(d, src))
    launch_k(metric_norm64_kernel, (unsigned)((toks * 8 + 255) / 256), 256, 0, stream, *d, tab, reinterpret_cast<const __nv_bfloat16*>(src), plane_a, plane_b);
  else if (d->dtype == TOME_BF16)
    launch_k(metric_norm_kernel<__nv_bfloat16>, nblk, 256, 0, stream, *d, tab, reinterpret_cast<const __nv_bfloat16*>(src), plane_a, plane_b);
  else
    launch_k(metric_norm_kernel<float>, nblk, 256, 0, stream, *d, tab, reinterpret_cast<const float*>(src), plane_a, plane_b);
  TOME_CUDA(cudaGetLastError());
  const size_t smem = sim_planes_smem(d->dim);
  TOME_CUDA(cudaFuncSetAttribute(sim_argmax_planes_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles = set_tiles(&tab, SIM_TILE);
  launch_k(sim_argmax_planes_kernel, dim3(tiles, d->batch), SIM_THREADS, smem, stream, *d, tab, plane_a, plane_b,
           node_max, node_idx, scores_out);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_select_topr(const tome_plan_shape_t* s, const float* node_max, const int32_t* node_idx,
                                const tome_plan_t* plan, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(s && node_max && node_idx && plan, TOME_ERR_INVALID, "select_topr: null argument");
  TOME_CHECK(plan->edge_idx && plan->dst_idx && plan->row_map && plan->dst_off && plan->dst_src, TOME_ERR_INVALID,
             "select_topr: every plan buffer must be provided");
  TOME_CHECK(s->batch > 0 && s->batch <= 65535 && s->tokens >= 2, TOME_ERR_INVALID,
             "select_topr: need 0 < batch <= 65535 and tokens >= 2");
  TOME_CHECK(s->r >= 1 && s->r <= s->tokens / 2, TOME_ERR_INVALID,
             "select_topr: r (%d) must be clamped to [1, %d] first (tome_clamp_r; r == 0 is the identity, no plan needed)",
             s->r, s->tokens / 2);
  SetTable tab;
  if (int rc = make_set_table(s->sets, s->tokens, s->r, 0, s->distill_token, &tab, "select_topr")) return rc;
  const int ta = tab.max_ta, tb = tab.max_tb;   // shared memory for the largest set
  const size_t smem = sizeof(unsigned long long) * (size_t)sel_pow2(ta) + sizeof(int) * ((size_t)2 * ta + tb + 1 + SEL_THREADS);
  TOME_CHECK(smem <= 220 * 1024 && s->tokens < (1 << 20), TOME_ERR_UNSUPPORTED,
             "select_topr: tokens (%d) too large for the shared-memory ranking", s->tokens);
  TOME_CUDA(cudaFuncSetAttribute(select_topr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ProfScope prof(PROF_SELECT, 0.0, 1, stream);
  launch_k(select_topr_kernel, dim3(tab.n, s->batch), SEL_THREADS, smem, stream, *s, tab, node_max, node_idx, *plan);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
