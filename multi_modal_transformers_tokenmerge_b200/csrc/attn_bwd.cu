// K6: attention backward on tcgen05 (autodiff of flax dot_product_attention as used at tome_attention.py:259-285,
// with the group-table mask and log(size) bias of the forward kernel).  No atomics, no fp32 dQ buffer: two
// kernels, each owning its outputs.
//
//   prep      delta[b,h,q] = sum_d dO*O and lse2 = lse*log2(e), both padded to 64-token tiles ([B,H,Tp]) so a tile is
//             one aligned 256-byte bulk copy; attn_meta_kernel (attn_meta.cuh) builds the per-tile mask words
//   dkdv      CTA = (128-key tile, head, batch), thread = key row, loop over 64-query tiles:
//               S^T = K Q^T, dP^T = V dO^T (TMEM) -> P^T, dS^T (bf16, written over dP^T in TMEM) -> dV += P^T dO,
//               dK += dS^T Q (TMEM)
//   dq        CTA = (128-query tile, head, batch), thread = query row, loop over 64-key tiles:
//               S = Q K^T, dP = dO V^T (TMEM) -> dS (bf16, shared, double-buffered) -> dQ += dS K (TMEM)
// P is recomputed from the saved log-sum-exp: P = exp2(s2 - lse2), s2 = q.k*scale*log2e + log2(size_k);
// dS = P * (dP - delta) * scale.  Each kernel uses 256 TMEM columns, so two CTAs share an SM.
// Everything a tile needs besides Q/K/V/dO (lse2, delta, positions, mask words, bias) arrives through a small ring of
// bulk copies issued by the producer warp: the softmax threads run no global loads, ballots or CTA barriers per tile
// (the first version did, and that dependent-load chain paced the kernels).
#include <float.h>

#include "attn_meta.cuh"
#include "common.cuh"
#include "host_util.h"

namespace tome {

int check_attn_desc(const tome_attn_desc_t* d, const char* who);  // attn_fwd.cu
int attn_generic_bwd(const tome_attn_desc_t* d, const tome_attn_grad_strides_t* gs, const void* q, const void* k, const void* v,
                     const void* out, const float* lse, const void* dout, void* dq, void* dk, void* dv, cudaStream_t stream);  // attn_generic.cu

constexpr int AB_D = 64;
constexpr int AB_THREADS = 192;
constexpr int DKT_SOFTMAX_WARPS = 8;
constexpr int DKT_THREADS = 320;   // attn_bwd_dkdv_ts_kernel: eight softmax warps + producer + MMA issuer
constexpr uint32_t AB_TMEM_COLS = 256;
constexpr int AB_MSLOTS = 3;  // metadata ring

struct AttnBwdParams {
  int batch, tokens, heads, tp;  // tp = tokens padded to a multiple of 64
  float scale, scale_log2;
  const uint8_t* gid;   // null: no mask
  const int32_t* pos;
  const uint8_t* meta;  // [B][tp/64][ATTN_META_BYTES]
  int store_ds;         // dK/dV kernel: also store every dS^T tile (the dQ GEMM kernel consumes them)

  const float* size;
  const float* lse2;    // [B,H,tp]  lse * log2(e), +inf past T
  const float* delta;   // [B,H,tp]  0 past T
  const uint8_t* keep_q;  // attention dropout keep words in the dQ tiling [n_q128][n_k64][128][2], or null
  const uint8_t* keep_k;  // ... in the dK/dV tiling [n_k128][n_q64][128][2]
  float inv_keep;         // 1 / (1 - rate)
  __nv_bfloat16* dq; long long dq_bs, dq_ts;
  __nv_bfloat16* dk; long long dk_bs, dk_ts;
  __nv_bfloat16* dv; long long dv_bs, dv_ts;
  // bias-gradient partials (or null): row (b * n_tiles128 + tile) of an f32 matrix with leading dimension cs_ld receives the
  // column sums of that 128-token tile of dq / dk / dv at columns cs_q / cs_k / cs_v + h * 64
  float* cs;
  long long cs_ld;
  int cs_q, cs_k, cs_v, n_t128;
};

// one mbarrier arrival for the whole warp, after every lane has got here (the lanes' tensor-memory accesses are warp-collective
// and already waited for; their shared-memory stores are ordered by the __syncwarp)
__device__ __forceinline__ void warp_arrive(uint64_t* bar, int lane) {
  __syncwarp();
  if (lane == 0) mbar_arrive(bar);
}

// Epilogue shared by the three kernels below.  The 128 threads of warps 0-3 each own one row of a [128 x 64] fp32 accumulator in
// tensor memory.  The rows are rounded to bf16 and staged in shared memory (16 KB, 128-byte swizzled rows), then written out
// by whole 128-byte lines (8 lanes per row, 4 rows per store instruction; a thread storing its own row scatters 32 partial
// sectors per instruction) and, when asked, summed per column over the valid rows -- the Dense bias gradient of the q/k/v
// projection -- without a second pass over dq/dk/dv in HBM.  `part`: 1 KB of shared memory.  Named barrier `bar`, 128 threads.
__device__ __forceinline__ void ab_store_tile(uint8_t* stage, float* part, uint32_t tm_row, int rows_valid, __nv_bfloat16* gtile,
                                              long long row_stride, float* colsum_out, int bar) {
  const int tid = threadIdx.x & 127, row = tid, warp = tid >> 5, lane = tid & 31;   // callers: one or two groups of 128 threads
  {
    float a[32], c[32];
    tmem_ld_f32x32(tm_row, a);
    tmem_ld_f32x32(tm_row + 32, c);
    tmem_ld_wait();
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
      *reinterpret_cast<uint4*>(stage + row * 128 + ((ch ^ (row & 7)) << 4)) =
          make_uint4(pack_bf16(a[8 * ch], a[8 * ch + 1]), pack_bf16(a[8 * ch + 2], a[8 * ch + 3]),
                     pack_bf16(a[8 * ch + 4], a[8 * ch + 5]), pack_bf16(a[8 * ch + 6], a[8 * ch + 7]));
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
      *reinterpret_cast<uint4*>(stage + row * 128 + (((ch + 4) ^ (row & 7)) << 4)) =
          make_uint4(pack_bf16(c[8 * ch], c[8 * ch + 1]), pack_bf16(c[8 * ch + 2], c[8 * ch + 3]),
                     pack_bf16(c[8 * ch + 4], c[8 * ch + 5]), pack_bf16(c[8 * ch + 6], c[8 * ch + 7]));
  }
  asm volatile("bar.sync %0, 128;" ::"r"(bar) : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int pce = tid + 128 * i, r = pce >> 3, ch = pce & 7;
    const uint4 w = *reinterpret_cast<const uint4*>(stage + r * 128 + ((ch ^ (r & 7)) << 4));
    if (r < rows_valid) *reinterpret_cast<uint4*>(gtile + (long long)r * row_stride + ch * 8) = w;
  }
  if (colsum_out != nullptr) {   // CTA-uniform
    float s0 = 0.f, s1 = 0.f;   // lane = column pair, warp = 32-row group; a warp reads one row per step: no bank conflict
#pragma unroll 8
    for (int i = 0; i < 32; ++i) {
      const int r = warp * 32 + i;
      const uint32_t w = *reinterpret_cast<const uint32_t*>(stage + r * 128 + (((lane >> 2) ^ (r & 7)) << 4) + (lane & 3) * 4);
      if (r < rows_valid) { s0 += bf16_lo(w); s1 += bf16_hi(w); }
    }
    *reinterpret_cast<float2*>(part + warp * 64 + 2 * lane) = make_float2(s0, s1);
    asm volatile("bar.sync %0, 128;" ::"r"(bar) : "memory");
    if (tid < 64) colsum_out[tid] = (part[tid] + part[64 + tid]) + (part[128 + tid] + part[192 + tid]);
  }
}

// w[i] holds the bf16 pair of columns 2i, 2i + 1; the columns whose bit is set in `cols` (all 0 so far) become bf16(fill)
__device__ __forceinline__ void or_bf16_lanes(uint32_t (&w)[16], uint32_t cols, float fill) {
  const uint32_t f = pack_bf16(fill, fill);
#pragma unroll
  for (int i = 0; i < 16; ++i)
    w[i] |= f & ((((cols >> (2 * i)) & 1u) ? 0x0000ffffu : 0u) | (((cols >> (2 * i + 1)) & 1u) ? 0xffff0000u : 0u));
}

// ------------------------------------------------------------------------------------------------ prep
__global__ void attn_bwd_prep_kernel(int B, int T, int Tp, int H, const __nv_bfloat16* __restrict__ o, long long o_bs,
                                     long long o_ts, const __nv_bfloat16* __restrict__ dout, long long do_bs, long long do_ts,
                                     const float* __restrict__ lse, float* __restrict__ delta, float* __restrict__ lse2) {
  const long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x;  // (b, t, h, chunk of 8)
  const long long total = (long long)B * Tp * H * 8;
  if (idx < total) {  // total is a multiple of 8: the 8 lanes of a (b,t,h) group leave together
    const int ch = (int)(idx & 7);
    const long long r = idx >> 3;
    const int h = (int)(r % H);
    const long long bt = r / H;
    const int t = (int)(bt % Tp), b = (int)(bt / Tp);
    float s = 0.f;
    if (t < T) {
      const uint4 ov = __ldg(reinterpret_cast<const uint4*>(o + b * o_bs + t * o_ts + h * AB_D + ch * 8));
      const uint4 dv = __ldg(reinterpret_cast<const uint4*>(dout + b * do_bs + t * do_ts + h * AB_D + ch * 8));
      s = bf16_lo(ov.x) * bf16_lo(dv.x) + bf16_hi(ov.x) * bf16_hi(dv.x) + bf16_lo(ov.y) * bf16_lo(dv.y) +
          bf16_hi(ov.y) * bf16_hi(dv.y) + bf16_lo(ov.z) * bf16_lo(dv.z) + bf16_hi(ov.z) * bf16_hi(dv.z) +
          bf16_lo(ov.w) * bf16_lo(dv.w) + bf16_hi(ov.w) * bf16_hi(dv.w);
    }
    s += __shfl_xor_sync(0xffffffffu, s, 1);
    s += __shfl_xor_sync(0xffffffffu, s, 2);
    s += __shfl_xor_sync(0xffffffffu, s, 4);
    if (ch == 0) {
      const long long w = ((long long)b * H + h) * Tp + t;
      delta[w] = s;
      lse2[w] = t < T ? lse[((long long)b * H + h) * T + t] * 1.4426950408889634f : INFINITY;  // queries past T: exp2(s - inf) = 0
    }
  }
}

// ------------------------------------------------------------------------------------------------ dK / dV
constexpr int DKV_BK = 128;  // keys per CTA
constexpr int DKV_BQ = 64;   // queries per tile
static_assert(DKV_BQ == ATTN_META_TILE, "query tiles and metadata tiles must coincide");
constexpr int DKV_KV_BYTES = DKV_BK * AB_D * 2;  // 16 KB
constexpr int DKV_Q_BYTES = DKV_BQ * AB_D * 2;   // 8 KB
constexpr int DKV_PT_BYTES = DKV_BK * DKV_BQ * 2;  // 16 KB
constexpr int DKV_META_SLOT = 1280 + ATTN_DROP_TILE_BYTES;  // lse2[64] | delta[64] | pos[64] | qvis[32][2] | qvisc[32][2] | dropout keep words [128 keys][2]

// The two products that consume what the softmax threads produce take their A operand from TENSOR MEMORY (tcgen05.mma
// with [tmem] A): once a thread has read its row of dP^T_i, it writes dS^T_i (two bf16 per column) over columns [64, 96)
// and P^T_i over [96, 128) of that very accumulator, and dV += P^T dO / dK += dS^T Q read them from there.  Nothing the
// threads produce passes through shared memory on its way to the tensor core: staging P^T / dS^T there doubled the
// shared-memory traffic per 128 x 64 tile, the largest single term of the kernel at two CTAs per SM
// (profiles/r02_attention_bwd.md).  dS^T for the dQ GEMM is staged in shared memory for one TMA store per tile.
// S^T lives in columns [0, 64) and is free again as soon as every thread has read it (s_free), so S^T_{i+1} is computed
// while the threads are still busy with dP^T_i; the order on the tensor pipe is S^T_{i+1}, dV_i, dK_i, dP^T_{i+1}.
constexpr int DKT_SMEM = 2 * DKV_KV_BYTES + 2 * 2 * DKV_Q_BYTES + 2 * DKV_PT_BYTES + AB_MSLOTS * DKV_META_SLOT + 256 + 1024;

template <bool DROP>
__global__ void __launch_bounds__(DKT_THREADS, 2)
attn_bwd_dkdv_ts_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                        const __grid_constant__ CUtensorMap tm_v, const __grid_constant__ CUtensorMap tm_do,
                        const __grid_constant__ CUtensorMap tm_ds, const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_k = smem;
  uint8_t* s_v = s_k + DKV_KV_BYTES;
  uint8_t* s_qdo = s_v + DKV_KV_BYTES;            // stage s: Q at s*16K, dO at s*16K + 8K
  uint8_t* s_dst = s_qdo + 2 * 2 * DKV_Q_BYTES;   // dS^T [128 keys][64 queries] bf16, 128B-swizzled rows: staging of the TMA store, tile i in buffer i & 1
  uint8_t* s_meta = s_dst + 2 * DKV_PT_BYTES;     // slot i at i * DKV_META_SLOT
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_meta + AB_MSLOTS * DKV_META_SLOT);
  uint64_t* kv_full = bars;        // 1
  uint64_t* q_full = bars + 1;     // [2]
  uint64_t* q_empty = bars + 3;    // [2]
  uint64_t* s_full = bars + 5;     // S^T_i in TMEM
  uint64_t* dp_full = bars + 6;    // dP^T_i in TMEM
  uint64_t* s_free = bars + 7;     // every thread has read its row of S^T_i (128 arrivals)
  uint64_t* ps_ready = bars + 8;   // P^T_i, dS^T_i written over dP^T_i (128 arrivals)
  uint64_t* pd_free = bars + 9;    // dV/dK MMAs of a tile retired (accumulators final after the last one)
  uint64_t* meta_full = bars + 10;   // [3]
  uint64_t* meta_empty = bars + 13;  // [3]  128 arrivals
  uint64_t* ds_stored = bars + 16;   // [2] store_ds: the TMA store of dS^T_i has read buffer i & 1 out of shared memory
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 18);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int T = p.tokens;
  const int n_q = (T + DKV_BQ - 1) / DKV_BQ;
  const bool has_mask = p.gid != nullptr;

  if (threadIdx.x == 0) {
    mbar_init(kv_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(dp_full, 1);
    mbar_init(s_free, DKT_SOFTMAX_WARPS);       // one arrival per softmax warp (elected lane) instead of one per thread
    mbar_init(ps_ready, DKT_SOFTMAX_WARPS);     // (fewer barrier transactions; measured neutral on the kernel's duration)
    mbar_init(pd_free, 1);
    mbar_init(&ds_stored[0], 1);
    mbar_init(&ds_stored[1], 1);
    for (int i = 0; i < AB_MSLOTS; ++i) {
      mbar_init(&meta_full[i], 1);
      mbar_init(&meta_empty[i], DKT_SOFTMAX_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 8 && lane == 0) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_k);
    tma_prefetch_desc(&tm_v);
    tma_prefetch_desc(&tm_do);
  }
  if (warp == 9) tmem_alloc(tmem_slot, AB_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tm_st = tmem_base, tm_dpt = tmem_base + 64, tm_dk = tmem_base + 128, tm_dv = tmem_base + 192;
  // A operands, written by each thread over the 32 columns of dP^T it has just read: the thread of query half g leaves dS^T
  // (16 columns = 32 bf16) at dP^T[32 g, 32 g + 16) and P^T at dP^T[32 g + 16, 32 g + 32); k-step k of the two products reads
  // its 8 columns at tm_dsa(k) / tm_pa(k)
  auto tm_dsa = [&](int k) { return tm_dpt + (uint32_t)((k >> 1) * 32 + (k & 1) * 8); };
  auto tm_pa = [&](int k) { return tm_dpt + (uint32_t)((k >> 1) * 32 + 16 + (k & 1) * 8); };

  if (warp == 8) {
    if (lane == 0) {
      mbar_expect_tx(kv_full, 2 * DKV_KV_BYTES);
      tma_load_3d(s_k, &tm_k, kv_full, h * AB_D, kt * DKV_BK, b);
      tma_load_3d(s_v, &tm_v, kv_full, h * AB_D, kt * DKV_BK, b);
      const float* lse_row = p.lse2 + ((size_t)b * p.heads + h) * p.tp;
      const float* del_row = p.delta + ((size_t)b * p.heads + h) * p.tp;
      const uint8_t* meta_b = p.meta + (size_t)b * n_q * ATTN_META_BYTES;
      for (int i = 0; i < n_q; ++i) {
        const int ms = i % AB_MSLOTS;
        uint8_t* slot = s_meta + ms * DKV_META_SLOT;
        mbar_wait(&meta_empty[ms], ((i / AB_MSLOTS) & 1) ^ 1);
        mbar_expect_tx(&meta_full[ms], (has_mask ? 1280u : 512u) + (DROP ? ATTN_DROP_TILE_BYTES : 0));
        if constexpr (DROP) bulk_g2s(slot + 1280, p.keep_k + ((size_t)kt * n_q + i) * ATTN_DROP_TILE_BYTES, ATTN_DROP_TILE_BYTES, &meta_full[ms]);
        bulk_g2s(slot, lse_row + i * DKV_BQ, 256, &meta_full[ms]);
        bulk_g2s(slot + 256, del_row + i * DKV_BQ, 256, &meta_full[ms]);
        if (has_mask) bulk_g2s(slot + 512, meta_b + (size_t)i * ATTN_META_BYTES + ATTN_META_OFF_POS, 768, &meta_full[ms]);  // pos | qvis | qvisc
        const int st = i & 1;
        mbar_wait(&q_empty[st], ((i >> 1) & 1) ^ 1);
        mbar_expect_tx(&q_full[st], 2 * DKV_Q_BYTES);
        tma_load_3d(s_qdo + st * 2 * DKV_Q_BYTES, &tm_q, &q_full[st], h * AB_D, i * DKV_BQ, b);
        tma_load_3d(s_qdo + st * 2 * DKV_Q_BYTES + DKV_Q_BYTES, &tm_do, &q_full[st], h * AB_D, i * DKV_BQ, b);
      }
    }
  } else if (warp == 9) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(DKV_BK, DKV_BQ, false, false);  // K/V K-major, Q/dO K-major
      constexpr uint32_t idesc_g = make_idesc_bf16(DKV_BK, AB_D, false, true);     // P^T/dS^T from TMEM (K-major), dO/Q MN-major
      const uint32_t ak = smem_u32(s_k), av = smem_u32(s_v);
      mbar_wait(kv_full, 0);
      for (int i = 0; i <= n_q; ++i) {
        if (i < n_q) {
          const int st = i & 1;
          if (i >= 1) {
            mbar_wait(s_free, (i - 1) & 1);   // S^T_{i-1} has been read by every thread
            tc_fence_after();
          }
          mbar_wait(&q_full[st], (i >> 1) & 1);
          tc_fence_after();
          const uint32_t aq = smem_u32(s_qdo + st * 2 * DKV_Q_BYTES);
#pragma unroll
          for (int k = 0; k < AB_D / 16; ++k)
            umma_bf16(tm_st, make_smem_desc(ak + k * 32, 16, 1024), make_smem_desc(aq + k * 32, 16, 1024), idesc_s, k > 0);
          umma_commit(s_full);
        }
        if (i >= 1) {
          mbar_wait(ps_ready, (i - 1) & 1);
          tc_fence_after();
          const int st = (i - 1) & 1;
          const uint32_t aq = smem_u32(s_qdo + st * 2 * DKV_Q_BYTES), ado = aq + DKV_Q_BYTES;
          if (p.store_ds) {  // dS^T tile (keys kt*128.., queries (i-1)*64..) -> global, in the layout it has in shared memory
            asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
                         ::"l"(&tm_ds), "r"(smem_u32(s_dst + ((i - 1) & 1) * DKV_PT_BYTES)), "r"((i - 1) * DKV_BQ), "r"(kt * DKV_BK), "r"(b * p.heads + h) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
#pragma unroll
          for (int k = 0; k < DKV_BQ / 16; ++k)  // dV += P^T dO
            umma_bf16_ts(tm_dv, tm_pa(k), make_smem_desc(ado + k * 2048, 8192, 1024), idesc_g, (i > 1 || k > 0) ? 1u : 0u);
#pragma unroll
          for (int k = 0; k < DKV_BQ / 16; ++k)  // dK += dS^T Q
            umma_bf16_ts(tm_dk, tm_dsa(k), make_smem_desc(aq + k * 2048, 8192, 1024), idesc_g, (i > 1 || k > 0) ? 1u : 0u);
          umma_commit(pd_free);
          umma_commit(&q_empty[st]);
        }
        if (i < n_q) {  // dP^T_i = V dO_i^T, behind the products that read P^T_{i-1} / dS^T_{i-1} out of the same columns
          const int st = i & 1;
          const uint32_t ado = smem_u32(s_qdo + st * 2 * DKV_Q_BYTES) + DKV_Q_BYTES;
#pragma unroll
          for (int k = 0; k < AB_D / 16; ++k)
            umma_bf16(tm_dpt, make_smem_desc(av + k * 32, 16, 1024), make_smem_desc(ado + k * 32, 16, 1024), idesc_s, k > 0);
          umma_commit(dp_full);
        }
        if (i >= 2 && p.store_ds) {  // all but the newest store have left shared memory: buffer i & 1 (tile i - 2) is free again
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
          mbar_arrive(&ds_stored[i & 1]);
        }
      }
      if (p.store_ds) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // stores complete before the CTA exits
    }
  } else {
    // warps 0-7: thread = (key row, query half): warp w owns TMEM lanes 32 (w & 3) .. + 31 and the 32 queries of half w >> 2 of
    // every tile.  Nothing is reduced along a row here (lse and delta arrive precomputed), so the two halves of a row never
    // talk to each other.  Measured (profiles/r02_attention_bwd.md): eight warps at 96 registers run exactly as fast as four
    // at 168 (857 vs 865 us for the whole backward at the bench shape) -- the kernel is paced by the hand-offs between the
    // softmax threads and the single MMA thread (two dependent hops per tile), not by issue slots or latency hiding; kept
    // because the smaller register footprint leaves room for the dK / dV epilogues to run side by side.
    const int row = (warp & 3) * 32 + lane;  // key row == TMEM lane
    const int hq = warp >> 2;                // query half
    const int kk = kt * DKV_BK + row;
    const uint32_t lane_sel = ((uint32_t)((warp & 3) * 32)) << 16;
    const bool k_valid = kk < T;
    float bias2 = 0.f;
    int gk = 0, pk = 0;
    if (k_valid) {
      if (p.size) bias2 = log2f(p.size[(long long)b * T + kk]);
      if (has_mask) {
        gk = p.gid[(long long)b * T + kk];
        pk = p.pos[(long long)b * T + kk];
      }
    }
    const float2 scale2 = make_float2(p.scale_log2, p.scale_log2), bias22 = make_float2(bias2, bias2);
    const float2 sc2 = make_float2(p.scale, p.scale), ik2 = make_float2(p.inv_keep, p.inv_keep);
    // a warp whose 32 key rows are all past T (three of the four quadrants in the last tile when T mod 128 <= 32) only keeps the
    // barriers moving: its rows of the A operands stay whatever tensor memory holds (row i of A reaches row i of dK / dV only,
    // and those rows are never stored), its rows of the stored dS^T tile are zeros (the dQ GEMM sums over them)
    const bool warp_active = kt * DKV_BK + (warp & 3) * 32 < T;
    uint8_t* dst_row0 = s_dst + row * 128;
    for (int i = 0; i < n_q; ++i) {
      const int ms = i % AB_MSLOTS;
      const uint8_t* slot = s_meta + ms * DKV_META_SLOT;
      mbar_wait(&meta_full[ms], (i / AB_MSLOTS) & 1);
      if (!warp_active) {
        mbar_wait(s_full, i & 1);
        tc_fence_before();
        warp_arrive(s_free, lane);
        mbar_wait(dp_full, i & 1);
        if (p.store_ds) {
          uint8_t* dst_row = dst_row0 + (i & 1) * DKV_PT_BYTES;
          if (i >= 2) mbar_wait(&ds_stored[i & 1], ((i - 2) >> 1) & 1);
#pragma unroll
          for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(dst_row + ((hq * 4 + ch) << 4)) = make_uint4(0u, 0u, 0u, 0u);
          fence_proxy_async_smem();
        }
        warp_arrive(&meta_empty[ms], lane);
        tc_fence_before();
        warp_arrive(ps_ready, lane);
        continue;
      }
      uint32_t vw = 0xffffffffu;
      if (has_mask) {
        vw = *reinterpret_cast<const uint32_t*>(slot + 768 + gk * 8 + hq * 4);
        const uint32_t c = *reinterpret_cast<const uint32_t*>(slot + 1024 + gk * 8 + hq * 4);
        if (c) {  // rare (Text sets): fold the causal rule into the visibility word
          const int* posq = reinterpret_cast<const int*>(slot + 512) + hq * 32;
          for (int q = 0; q < 32; ++q)
            if (((c >> q) & 1u) && pk <= posq[q]) vw |= 1u << q;
        }
      }
      if (!k_valid) vw = 0u;  // rows past T contribute nothing (and store zeros into dS^T)
      uint32_t kb = 0xffffffffu;  // dropout keep bits of this key against this half's 32 queries
      if constexpr (DROP) kb = *reinterpret_cast<const uint32_t*>(slot + 1280 + row * 8 + hq * 4);
      const float4* lse4 = reinterpret_cast<const float4*>(slot) + hq * 8;
      const float4* del4 = reinterpret_cast<const float4*>(slot + 256) + hq * 8;
      // ---- phase 1: P = exp2(s2 - lse2) from S^T_i, kept as packed bf16 (what the dV product consumes, before dropout)
      uint32_t pe[16];
      mbar_wait(s_full, i & 1);
      tc_fence_after();
      {
        float sv[32];
        tmem_ld_f32x32(tm_st + lane_sel + hq * 32, sv);
        tmem_ld_wait();
        tc_fence_before();
        warp_arrive(s_free, lane);   // this thread's part of S^T_i is in registers: the next S^T may overwrite it
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 l4 = lse4[c4];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int c = c4 * 4 + 2 * u;
            const float2 lv = u ? make_float2(l4.z, l4.w) : make_float2(l4.x, l4.y);
            float2 t = __ffma2_rn(make_float2(sv[c], sv[c + 1]), scale2, bias22);
            t = __fadd2_rn(t, make_float2(-lv.x, -lv.y));
            float2 e = make_float2(fast_exp2(t.x), fast_exp2(t.y));
            e.x = ((vw >> c) & 1u) ? e.x : 0.f;
            e.y = ((vw >> (c + 1)) & 1u) ? e.y : 0.f;
            pe[c >> 1] = pack_bf16(e.x, e.y);
          }
        }
      }
      // ---- phase 2: dS = P (dP' - delta) scale from dP^T_i
      uint32_t dw[16], pw[DROP ? 16 : 1];
      mbar_wait(dp_full, i & 1);
      tc_fence_after();
      {
        float dv[32];
        tmem_ld_f32x32(tm_dpt + lane_sel + hq * 32, dv);
        tmem_ld_wait();
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 d4 = del4[c4];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int c = c4 * 4 + 2 * u;
            const float2 dl = u ? make_float2(d4.z, d4.w) : make_float2(d4.x, d4.y);
            const uint32_t pwv = pe[c >> 1];
            const float2 pf = make_float2(bf16_lo(pwv), bf16_hi(pwv));
            float2 dp = make_float2(dv[c], dv[c + 1]);
            if constexpr (DROP) {  // weights' = weights keep / (1 - rate): dP' = dP keep / (1 - rate) enters dS, P' enters dV
              const bool k0 = (kb >> c) & 1u, k1 = (kb >> (c + 1)) & 1u;
              dp = __fmul2_rn(dp, ik2);
              float2 pd = __fmul2_rn(pf, ik2);
              dp.x = k0 ? dp.x : 0.f; dp.y = k1 ? dp.y : 0.f;
              pd.x = k0 ? pd.x : 0.f; pd.y = k1 ? pd.y : 0.f;
              pw[c >> 1] = pack_bf16(pd.x, pd.y);
            }
            float2 g = __fadd2_rn(dp, make_float2(-dl.x, -dl.y));
            g = __fmul2_rn(g, sc2);
            g = __fmul2_rn(g, pf);
            dw[c >> 1] = pack_bf16(g.x, g.y);
          }
        }
      }
      if (has_mask) {  // query rows with no visible key (attn_meta.cuh): 1/T of their dO reaches every key's dV; dS stays 0
        const float lq = reinterpret_cast<const float*>(slot)[hq * 32 + lane];
        const uint32_t fw = __ballot_sync(0xffffffffu, lq < ATTN_MASKED_ROW_LSE2) & kb;   // warp-uniform, rarely non-zero
        if (fw) {
          if constexpr (DROP) or_bf16_lanes(pw, fw, p.inv_keep / (float)T);
          else or_bf16_lanes(pe, fw, 1.0f / (float)T);
        }
      }
      tmem_st_x16(tm_dpt + lane_sel + hq * 32, dw);
      if constexpr (DROP) tmem_st_x16(tm_dpt + lane_sel + hq * 32 + 16, pw);
      else tmem_st_x16(tm_dpt + lane_sel + hq * 32 + 16, pe);
      if (p.store_ds) {  // the dS^T tile the dQ GEMM consumes, staged for one TMA store (a direct 16-byte-per-lane global
                         // store of these rows cost 330 us per call: 32 partial sectors per instruction)
        uint8_t* dst_row = dst_row0 + (i & 1) * DKV_PT_BYTES;
        if (i >= 2) mbar_wait(&ds_stored[i & 1], ((i - 2) >> 1) & 1);   // the store of tile i - 2 has read this buffer
#pragma unroll
        for (int ch = 0; ch < 4; ++ch)
          *reinterpret_cast<uint4*>(dst_row + (((hq * 4 + ch) ^ (row & 7)) << 4)) = make_uint4(dw[4 * ch], dw[4 * ch + 1], dw[4 * ch + 2], dw[4 * ch + 3]);
        fence_proxy_async_smem();
      }
      tmem_st_wait();
      warp_arrive(&meta_empty[ms], lane);
      tc_fence_before();
      warp_arrive(ps_ready, lane);
    }
    mbar_wait(pd_free, (n_q - 1) & 1);  // accumulators final
    tc_fence_after();
    {
      // every MMA has retired: the K and V tiles serve as staging for dK and dV, the Q/dO ring for the column-sum scratch;
      // warps 0-3 write dK while warps 4-7 write dV (own staging tile, scratch and named barrier each)
      const int rows_valid = min(DKV_BK, T - kt * DKV_BK);
      float* cs_row = p.cs ? p.cs + ((long long)b * p.n_t128 + kt) * p.cs_ld + h * AB_D : nullptr;
      if (hq == 0)
        ab_store_tile(s_k, reinterpret_cast<float*>(s_qdo), tm_dk + lane_sel, rows_valid,
                      p.dk + (long long)b * p.dk_bs + (long long)kt * DKV_BK * p.dk_ts + h * AB_D, p.dk_ts, cs_row ? cs_row + p.cs_k : nullptr, 1);
      else
        ab_store_tile(s_v, reinterpret_cast<float*>(s_qdo) + 256, tm_dv + lane_sel, rows_valid,
                      p.dv + (long long)b * p.dv_bs + (long long)kt * DKV_BK * p.dv_ts + h * AB_D, p.dv_ts, cs_row ? cs_row + p.cs_v : nullptr, 2);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 9) {
    tc_fence_after();
    tmem_dealloc(tmem_base, AB_TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ dQ
constexpr int DQ_BQ = 128;  // queries per CTA
constexpr int DQ_BK = 64;   // keys per tile
static_assert(DQ_BK == ATTN_META_TILE, "key tiles and metadata tiles must coincide");
constexpr int DQ_Q_BYTES = DQ_BQ * AB_D * 2;   // 16 KB
constexpr int DQ_K_BYTES = DQ_BK * AB_D * 2;   // 8 KB
constexpr int DQ_DS_BYTES = DQ_BQ * DQ_BK * 2;  // 16 KB, x2 buffers
constexpr int DQ_META_SLOT = ATTN_META_KEY_BYTES + ATTN_DROP_TILE_BYTES;  // bias2 | vis | visc | pos | dropout keep words [128 queries][2]
constexpr int DQ_SMEM = 2 * DQ_Q_BYTES + 2 * 2 * DQ_K_BYTES + 2 * DQ_DS_BYTES + AB_MSLOTS * DQ_META_SLOT + 256 + 1024;

template <bool DROP>
__global__ void __launch_bounds__(AB_THREADS, 2)
attn_bwd_dq_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                   const __grid_constant__ CUtensorMap tm_v, const __grid_constant__ CUtensorMap tm_do,
                   const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_q = smem;
  uint8_t* s_do = s_q + DQ_Q_BYTES;
  uint8_t* s_kv = s_do + DQ_Q_BYTES;             // stage s: K at s*16K, V at s*16K + 8K
  uint8_t* s_ds = s_kv + 2 * 2 * DQ_K_BYTES;     // dS [128 queries][64 keys] bf16 K-major swizzled, buffer i at i * 16 KB
  uint8_t* s_meta = s_ds + 2 * DQ_DS_BYTES;      // slot i at i * DQ_META_SLOT
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_meta + AB_MSLOTS * DQ_META_SLOT);
  uint64_t* q_full = bars;          // Q and dO
  uint64_t* kv_full = bars + 1;     // [2]
  uint64_t* kv_empty = bars + 3;    // [2]
  uint64_t* s_full = bars + 5;      // S_j, dP_j in TMEM
  uint64_t* ds_ready = bars + 6;    // dS_j in smem, S_j/dP_j consumed (128 arrivals)
  uint64_t* ds_free = bars + 7;     // [2] dQ MMA of tile j done reading dS buffer j&1
  uint64_t* meta_full = bars + 9;   // [3]
  uint64_t* meta_empty = bars + 12; // [3] 128 arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 15);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int T = p.tokens;
  const int n_k = (T + DQ_BK - 1) / DQ_BK;
  const bool has_mask = p.gid != nullptr;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
      mbar_init(&ds_free[i], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(ds_ready, DQ_BQ);
    for (int i = 0; i < AB_MSLOTS; ++i) {
      mbar_init(&meta_full[i], 1);
      mbar_init(&meta_empty[i], DQ_BQ);
    }
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_k);
    tma_prefetch_desc(&tm_v);
    tma_prefetch_desc(&tm_do);
  }
  if (warp == 5) tmem_alloc(tmem_slot, AB_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tm_s = tmem_base, tm_dp = tmem_base + 64, tm_dq = tmem_base + 128;

  if (warp == 4) {
    if (lane == 0) {
      mbar_expect_tx(q_full, 2 * DQ_Q_BYTES);
      tma_load_3d(s_q, &tm_q, q_full, h * AB_D, qt * DQ_BQ, b);
      tma_load_3d(s_do, &tm_do, q_full, h * AB_D, qt * DQ_BQ, b);
      const uint32_t meta_bytes = has_mask ? ATTN_META_KEY_BYTES : 256u;
      const uint8_t* meta_b = p.meta + (size_t)b * n_k * ATTN_META_BYTES;
      for (int j = 0; j < n_k; ++j) {
        const int ms = j % AB_MSLOTS;
        mbar_wait(&meta_empty[ms], ((j / AB_MSLOTS) & 1) ^ 1);
        mbar_expect_tx(&meta_full[ms], meta_bytes + (DROP ? ATTN_DROP_TILE_BYTES : 0));
        bulk_g2s(s_meta + ms * DQ_META_SLOT, meta_b + (size_t)j * ATTN_META_BYTES, meta_bytes, &meta_full[ms]);
        if constexpr (DROP)
          bulk_g2s(s_meta + ms * DQ_META_SLOT + ATTN_META_KEY_BYTES, p.keep_q + ((size_t)qt * n_k + j) * ATTN_DROP_TILE_BYTES,
                   ATTN_DROP_TILE_BYTES, &meta_full[ms]);
        const int st = j & 1;
        mbar_wait(&kv_empty[st], ((j >> 1) & 1) ^ 1);
        mbar_expect_tx(&kv_full[st], 2 * DQ_K_BYTES);
        tma_load_3d(s_kv + st * 2 * DQ_K_BYTES, &tm_k, &kv_full[st], h * AB_D, j * DQ_BK, b);
        tma_load_3d(s_kv + st * 2 * DQ_K_BYTES + DQ_K_BYTES, &tm_v, &kv_full[st], h * AB_D, j * DQ_BK, b);
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(DQ_BQ, DQ_BK, false, false);  // Q/dO K-major, K/V K-major
      constexpr uint32_t idesc_g = make_idesc_bf16(DQ_BQ, AB_D, false, true);    // dS K-major, K MN-major
      const uint32_t aq = smem_u32(s_q), ado = smem_u32(s_do), ads = smem_u32(s_ds);
      mbar_wait(q_full, 0);
      for (int j = 0; j <= n_k; ++j) {
        if (j >= 1) {
          mbar_wait(ds_ready, (j - 1) & 1);
          tc_fence_after();
        }
        if (j < n_k) {
          const int st = j & 1;
          mbar_wait(&kv_full[st], (j >> 1) & 1);
          tc_fence_after();
          const uint32_t ak = smem_u32(s_kv + st * 2 * DQ_K_BYTES), av = ak + DQ_K_BYTES;
#pragma unroll
          for (int k = 0; k < AB_D / 16; ++k)
            umma_bf16(tm_s, make_smem_desc(aq + k * 32, 16, 1024), make_smem_desc(ak + k * 32, 16, 1024), idesc_s, k > 0);
#pragma unroll
          for (int k = 0; k < AB_D / 16; ++k)
            umma_bf16(tm_dp, make_smem_desc(ado + k * 32, 16, 1024), make_smem_desc(av + k * 32, 16, 1024), idesc_s, k > 0);
          umma_commit(s_full);
        }
        if (j >= 1) {
          const int st = (j - 1) & 1;
          const uint32_t ak = smem_u32(s_kv + st * 2 * DQ_K_BYTES), adsj = ads + ((j - 1) & 1) * DQ_DS_BYTES;
#pragma unroll
          for (int k = 0; k < DQ_BK / 16; ++k)  // dQ += dS K
            umma_bf16(tm_dq, make_smem_desc(adsj + k * 32, 16, 1024), make_smem_desc(ak + k * 2048, 8192, 1024), idesc_g,
                      (j > 1 || k > 0) ? 1u : 0u);
          umma_commit(&ds_free[(j - 1) & 1]);
          umma_commit(&kv_empty[st]);
        }
      }
    }
  } else {
    const int row = threadIdx.x;
    const int q = qt * DQ_BQ + row;
    const uint32_t lane_sel = ((uint32_t)(warp * 32)) << 16;
    const bool q_valid = q < T;
    const long long lrow = ((long long)b * p.heads + h) * p.tp + (q_valid ? q : 0);
    const float lse2 = q_valid ? p.lse2[lrow] : INFINITY;   // rows past T: exp2(s - inf) = 0
    const float dl = q_valid ? p.delta[lrow] : 0.f;
    int gq = 0, pos_q = 0;
    if (has_mask && q_valid) {
      gq = p.gid[(long long)b * T + q];
      pos_q = p.pos[(long long)b * T + q];
    }
    const float2 scale2 = make_float2(p.scale_log2, p.scale_log2);
    const float2 nl2 = make_float2(-lse2, -lse2);
    const float2 sc2 = make_float2(p.scale, p.scale);
    const float2 ik2 = make_float2(p.inv_keep, p.inv_keep);
    for (int j = 0; j < n_k; ++j) {
      const int ms = j % AB_MSLOTS;
      const uint8_t* slot = s_meta + ms * DQ_META_SLOT;
      mbar_wait(&meta_full[ms], (j / AB_MSLOTS) & 1);
      uint32_t vw[2] = {0xffffffffu, 0xffffffffu};
      if (has_mask) {
        const uint2 a = *reinterpret_cast<const uint2*>(slot + ATTN_META_OFF_VIS + gq * 8);
        const uint2 c = *reinterpret_cast<const uint2*>(slot + ATTN_META_OFF_VISC + gq * 8);
        vw[0] = a.x; vw[1] = a.y;
        if (c.x | c.y) {
          const int* m_pos = reinterpret_cast<const int*>(slot + ATTN_META_OFF_POS);
          for (int i = 0; i < 32; ++i) {
            if (((c.x >> i) & 1u) && m_pos[i] <= pos_q) vw[0] |= 1u << i;
            if (((c.y >> i) & 1u) && m_pos[32 + i] <= pos_q) vw[1] |= 1u << i;
          }
        }
      }
      uint32_t kb[2] = {0xffffffffu, 0xffffffffu};  // dropout keep bits of this query against the tile's 64 keys
      if constexpr (DROP) {
        const uint2 t = *reinterpret_cast<const uint2*>(slot + ATTN_META_KEY_BYTES + row * 8);
        kb[0] = t.x; kb[1] = t.y;
      }
      const float4* bias4 = reinterpret_cast<const float4*>(slot);
      uint8_t* dsb = s_ds + (j & 1) * DQ_DS_BYTES + row * 128;
      mbar_wait(s_full, j & 1);
      tc_fence_after();
#pragma unroll
      for (int cq = 0; cq < DQ_BK / 32; ++cq) {
        const int c0 = cq * 32;
        float sv[32], dv[32];
        tmem_ld_f32x32(tm_s + lane_sel + c0, sv);
        tmem_ld_f32x32(tm_dp + lane_sel + c0, dv);
        tmem_ld_wait();
        const uint32_t word = vw[cq];
        uint32_t dw[16];
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 b4 = bias4[cq * 8 + c4];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int c = c4 * 4 + 2 * u;
            const float2 bv = u ? make_float2(b4.z, b4.w) : make_float2(b4.x, b4.y);
            float2 t = __ffma2_rn(make_float2(sv[c], sv[c + 1]), scale2, bv);
            t = __fadd2_rn(t, nl2);
            float2 pe = make_float2(fast_exp2(t.x), fast_exp2(t.y));
            pe.x = ((word >> c) & 1u) ? pe.x : 0.f;
            pe.y = ((word >> (c + 1)) & 1u) ? pe.y : 0.f;
            float2 dp = make_float2(dv[c], dv[c + 1]);
            if constexpr (DROP) {  // dP' = dP * keep / (1 - rate)
              dp = __fmul2_rn(dp, ik2);
              dp.x = ((kb[cq] >> c) & 1u) ? dp.x : 0.f;
              dp.y = ((kb[cq] >> (c + 1)) & 1u) ? dp.y : 0.f;
            }
            // the dK/dV kernel forms dS from the bf16-rounded P it feeds to the dV product (and so does the forward's P V):
            // the same rounding and the same operation order here keep the two dQ paths bit-identical
            const uint32_t pr = pack_bf16(pe.x, pe.y);
            float2 g = __fadd2_rn(dp, make_float2(-dl, -dl));
            g = __fmul2_rn(g, sc2);
            g = __fmul2_rn(g, make_float2(bf16_lo(pr), bf16_hi(pr)));
            dw[c >> 1] = pack_bf16(g.x, g.y);
          }
        }
        if (cq == 0 && j >= 2) mbar_wait(&ds_free[j & 1], ((j - 2) >> 1) & 1);  // dQ MMA of tile j-2 has read this buffer
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int chunk = (c0 >> 3) + ch;
          *reinterpret_cast<uint4*>(dsb + ((chunk ^ (row & 7)) << 4)) = make_uint4(dw[4 * ch], dw[4 * ch + 1], dw[4 * ch + 2], dw[4 * ch + 3]);
        }
      }
      mbar_arrive(&meta_empty[ms]);
      fence_proxy_async_smem();
      tc_fence_before();
      mbar_arrive(ds_ready);
    }
    mbar_wait(&ds_free[(n_k - 1) & 1], ((n_k - 1) >> 1) & 1);
    tc_fence_after();
    ab_store_tile(s_q, reinterpret_cast<float*>(s_do), tm_dq + lane_sel, min(DQ_BQ, T - qt * DQ_BQ),
                  p.dq + (long long)b * p.dq_bs + (long long)qt * DQ_BQ * p.dq_ts + h * AB_D, p.dq_ts,
                  p.cs ? p.cs + ((long long)b * p.n_t128 + qt) * p.cs_ld + h * AB_D + p.cs_q : nullptr, 1);   // Q / dO tiles: free now
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, AB_TMEM_COLS);
  }
}

}  // namespace tome

using namespace tome;

static size_t bwd_pad_elems(const tome_attn_desc_t* d) {
  return (size_t)d->batch * d->heads * (size_t)(((d->tokens + 63) / 64) * 64);
}

// ------------------------------------------------------------------------------------------------ dQ from stored dS^T
// dQ[q, :] = sum_k dS[q, k] K[k, :] as a batched GEMM over the dS^T tiles the dK/dV kernel stored ([B*H][keys][queries] bf16):
// the alternative to attn_bwd_dq_kernel, which recomputes S, dP and the softmax.  CTA = (128-query tile, head, batch);
// per 64-key step the A operand is the dS^T block read MN-major (two 64-query atoms), the B operand the K tile read
// MN-major (as V is in the forward P V product); the accumulator sits in 64 TMEM columns.
// 3 stages x 3 CTAs per SM: the kernel is a short stream of dS^T tiles (9 k-steps at T = 536), so more resident CTAs to
// overlap one CTA's prologue / epilogue with another's loads beat a deeper ring (4 x 2: 892 us for the whole backward at the
// bench shape, 2 x 4: 870, 3 x 3: 865)
constexpr int DQG_BQ = 128, DQG_BK = 64, DQG_STAGES = 3, DQG_CTAS = 3;
constexpr int DQG_A_BYTES = 2 * DQG_BK * 128;   // 16 KB: two [64 keys][64 queries] atoms
constexpr int DQG_B_BYTES = DQG_BK * AB_D * 2;  // 8 KB
constexpr int DQG_STAGE = DQG_A_BYTES + DQG_B_BYTES;
constexpr int DQG_SMEM = DQG_STAGES * DQG_STAGE + 256 + 1024;

__global__ void __launch_bounds__(AB_THREADS, DQG_CTAS)
attn_bwd_dq_gemm_kernel(const __grid_constant__ CUtensorMap tm_ds, const __grid_constant__ CUtensorMap tm_k,
                        const AttnBwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + DQG_STAGES * DQG_STAGE);
  uint64_t* full = bars;                 // [4]
  uint64_t* empty = bars + DQG_STAGES;   // [4]
  uint64_t* acc_full = bars + 2 * DQG_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * DQG_STAGES + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int T = p.tokens;
  const int n_k = (T + DQG_BK - 1) / DQG_BK;
  if (threadIdx.x == 0) {
    for (int i = 0; i < DQG_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tm_ds);
    tma_prefetch_desc(&tm_k);
  }
  if (warp == 5) tmem_alloc(tmem_slot, 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 4) {
    if (lane == 0) {
      for (int j = 0; j < n_k; ++j) {
        const int st = j % DQG_STAGES;
        mbar_wait(&empty[st], ((j / DQG_STAGES) & 1) ^ 1);
        uint8_t* sa = smem + st * DQG_STAGE;
        mbar_expect_tx(&full[st], DQG_STAGE);
        tma_load_3d(sa, &tm_ds, &full[st], qt * DQG_BQ, j * DQG_BK, b * p.heads + h);
        tma_load_3d(sa + DQG_BK * 128, &tm_ds, &full[st], qt * DQG_BQ + 64, j * DQG_BK, b * p.heads + h);
        tma_load_3d(sa + DQG_A_BYTES, &tm_k, &full[st], h * AB_D, j * DQG_BK, b);
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(DQG_BQ, AB_D, true, true);  // dS^T read MN-major, K read MN-major
      for (int j = 0; j < n_k; ++j) {
        const int st = j % DQG_STAGES;
        mbar_wait(&full[st], (j / DQG_STAGES) & 1);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + st * DQG_STAGE), sb = sa + DQG_A_BYTES;
#pragma unroll
        for (int k = 0; k < DQG_BK / 16; ++k)
          umma_bf16(tmem_base, make_smem_desc(sa + k * 2048, DQG_BK * 128, 1024), make_smem_desc(sb + k * 2048, 8192, 1024), idesc,
                    (j > 0 || k > 0) ? 1u : 0u);
        umma_commit(&empty[st]);
      }
      umma_commit(acc_full);
    }
  } else {
    const int row = threadIdx.x;
    const int q = qt * DQG_BQ + row;
    const uint32_t lane_sel = ((uint32_t)(warp * 32)) << 16;
    mbar_wait(acc_full, 0);
    tc_fence_after();
    // every stage has been consumed: stage 0 (24 KB) holds the staging tile and the column-sum scratch
    ab_store_tile(smem, reinterpret_cast<float*>(smem + DQG_BQ * 128), tmem_base + lane_sel, min(DQG_BQ, T - qt * DQG_BQ),
                  p.dq + (long long)b * p.dq_bs + (long long)qt * DQG_BQ * p.dq_ts + h * AB_D, p.dq_ts,
                  p.cs ? p.cs + ((long long)b * p.n_t128 + qt) * p.cs_ld + h * AB_D + p.cs_q : nullptr, 1);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 64);
  }
}

// dQ from the dS^T tiles the dK/dV kernel stores (a batched GEMM: 884 vs 1 023 us at B=256 T=536 H=6, 2 383 vs 2 575 at
// T=2080, 4 340 vs 4 433 at T=4096, 4 912 vs 4 977 at T=6144) or the recomputing dQ kernel, which needs no B*H*T^2 buffer.
// -1 (default): the GEMM path while that buffer stays under 8 GiB; 0 / 1: force.  Process-wide tuning aid, not part of
// the public header.
static int g_attn_dq_from_ds = -1;
static inline size_t ds_buffer_bytes(const tome_attn_desc_t* d) {
  // [B*H][T keys][T queries, rows pitched to 16 bytes]: the TMA stores clip the tiles' rows / columns past T and the loads
  // zero-fill them, so no padding is written or read (T = 536: 575 KB per head instead of the 737 KB of whole 128 x 64 tiles)
  const size_t tq = ((size_t)d->tokens + 7) / 8 * 8, tk = (size_t)d->tokens;
  return (size_t)d->batch * d->heads * tq * tk * 2;
}
static inline bool dq_from_ds(const tome_attn_desc_t* d) {
  if (d->head_dim != AB_D) return false;
  return g_attn_dq_from_ds < 0 ? ds_buffer_bytes(d) <= ((size_t)8 << 30) : g_attn_dq_from_ds != 0;
}

extern "C" void tome_attention_set_dq_from_ds(int mode) { g_attn_dq_from_ds = mode < 0 ? -1 : (mode ? 1 : 0); }

struct BwdWs {
  uint8_t* meta;        // per-tile metadata (launch_attn_meta)
  float *delta, *lse2;  // [B, H, ceil64(T)] each (attn_bwd_prep_kernel)
  uint8_t* bits;        // dropout keep bits, both tilings (launch_attn_dropbits), only with dropout
  uint8_t* ds;          // dS^T (ds_buffer_bytes), only when dQ is the GEMM over it
  size_t total;
};
static BwdWs bwd_ws(const tome_attn_desc_t* d, void* base) {
  Bump b{reinterpret_cast<uint8_t*>(base)};
  BwdWs w;
  w.meta = b.take<uint8_t>(attn_meta_bytes(d->batch, d->tokens));
  w.delta = b.take<float>(bwd_pad_elems(d));
  w.lse2 = b.take<float>(bwd_pad_elems(d));
  w.bits = b.take<uint8_t>(d->dropout_rate > 0.f ? attn_dropbits_bytes(d->tokens) : 0);
  w.ds = b.take<uint8_t>(dq_from_ds(d) ? ds_buffer_bytes(d) : 0);
  w.total = b.total();
  return w;
}

extern "C" size_t tome_attention_bwd_workspace_bytes(const tome_attn_desc_t* d) {
  if (!d || d->batch <= 0 || d->tokens <= 0 || d->heads <= 0) return 0;
  return bwd_ws(d, nullptr).total;
}

extern "C" int tome_attention_bwd(const tome_attn_desc_t* d, const tome_attn_grad_strides_t* gs, const void* q, const void* k,
                                  const void* v, const void* out, const float* lse, const void* dout, void* dq, void* dk,
                                  void* dv, void* workspace, size_t workspace_bytes, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int rc = check_attn_desc(d, "attention_bwd")) return rc;
  TOME_CHECK(gs && q && k && v && out && lse && dout && dq && dk && dv, TOME_ERR_INVALID, "attention_bwd: null argument");
  TOME_CHECK(d->dropout_rate >= 0.f && d->dropout_rate < 1.f, TOME_ERR_INVALID, "attention_bwd: dropout_rate must be in [0, 1)");
  TOME_CHECK(!gs->bias_partial || d->head_dim == AB_D, TOME_ERR_INVALID, "attention_bwd: bias_partial needs head_dim 64");
  TOME_CHECK(!gs->bias_partial || gs->bias_partial_ld >= 0, TOME_ERR_INVALID, "attention_bwd: bad bias_partial_ld");
  if (d->head_dim != AB_D) {
    ProfScope prof(PROF_ATTN_BWD, 10.0 * d->batch * d->heads * (double)d->tokens * d->tokens * d->head_dim, 2, stream);
    return attn_generic_bwd(d, gs, q, k, v, out, lse, dout, dq, dk, dv, stream);
  }
  TOME_CHECK(workspace != nullptr, TOME_ERR_INVALID, "attention_bwd: null workspace");
  TOME_CHECK(((uintptr_t)workspace & 255) == 0, TOME_ERR_INVALID, "attention_bwd: workspace must be 256-byte aligned");
  const BwdWs ws = bwd_ws(d, workspace);
  TOME_CHECK(workspace_bytes >= ws.total, TOME_ERR_INVALID,
             "attention_bwd: workspace too small (%zu < %zu, see tome_attention_bwd_workspace_bytes)", workspace_bytes, ws.total);
  const long long st[8] = {gs->dq_batch_stride, gs->dq_token_stride, gs->dk_batch_stride, gs->dk_token_stride,
                           gs->dv_batch_stride, gs->dv_token_stride, gs->do_batch_stride, gs->do_token_stride};
  for (int i = 0; i < 8; ++i) TOME_CHECK(st[i] % 8 == 0, TOME_ERR_INVALID, "attention_bwd: strides must be multiples of 8");
  const int B = d->batch, T = d->tokens, H = d->heads;
  ProfScope prof(PROF_ATTN_BWD, 10.0 * d->batch * d->heads * (double)d->tokens * d->tokens * d->head_dim, 4, stream);
  const int Tp = ((T + 63) / 64) * 64;
  if (int rc = launch_attn_meta(B, T, d->gid, d->pos, d->allow, d->num_groups, d->size, ws.meta, stream)) return rc;
  TOME_CHECK(d->dropout_rate >= 0.f && d->dropout_rate < 1.f, TOME_ERR_INVALID, "attention_bwd: dropout_rate must be in [0, 1)");
  const uint8_t *keep_q = nullptr, *keep_k = nullptr;
  float inv_keep = 1.0f;
  if (d->dropout_rate > 0.f) {  // the same (seed, site) as the forward call regenerates the same mask
    if (int rc = launch_attn_dropbits(T, d->dropout_rate, d->dropout_seed, d->dropout_site, ws.bits, stream)) return rc;
    keep_q = ws.bits;
    keep_k = ws.bits + attn_dropbits_bytes(T) / 2;
    inv_keep = make_dropout(d->dropout_rate, d->dropout_seed, d->dropout_site).inv_keep;
  }
  {
    const long long total = (long long)B * Tp * H * 8;
    launch_k(attn_bwd_prep_kernel, (unsigned)((total + 255) / 256), 256, 0, stream, 
        B, T, Tp, H, reinterpret_cast<const __nv_bfloat16*>(out), d->o_batch_stride, d->o_token_stride,
        reinterpret_cast<const __nv_bfloat16*>(dout), gs->do_batch_stride, gs->do_token_stride, lse, ws.delta, ws.lse2);
    TOME_CUDA(cudaGetLastError());
  }
  const uint64_t hd = (uint64_t)H * d->head_dim;
  AttnBwdParams p;
  p.batch = B; p.tokens = T; p.heads = H; p.tp = Tp;
  p.scale = d->scale; p.scale_log2 = d->scale * 1.4426950408889634f;
  p.gid = d->gid; p.pos = d->pos; p.meta = ws.meta; p.size = d->size; p.lse2 = ws.lse2; p.delta = ws.delta;
  p.keep_q = keep_q; p.keep_k = keep_k; p.inv_keep = inv_keep;
  const bool from_ds = dq_from_ds(d);
  p.store_ds = from_ds ? 1 : 0;
  p.cs = gs->bias_partial; p.cs_ld = gs->bias_partial_ld;
  p.cs_q = gs->bias_q_col; p.cs_k = gs->bias_k_col; p.cs_v = gs->bias_v_col;
  p.n_t128 = ceil_div(T, 128);

  const uint64_t ds_tq = ((uint64_t)T + 7) / 8 * 8, ds_tk = (uint64_t)T;   // row pitch, rows (see ds_buffer_bytes)
  CUtensorMap tds_store, tds_load;
  if (from_ds) {
    if (int rc = make_tmap_3d_bf16(&tds_store, ws.ds, (uint64_t)T, ds_tk, (uint64_t)B * H, ds_tq, ds_tq * ds_tk, DKV_BK)) return rc;
    if (int rc = make_tmap_3d_bf16(&tds_load, ws.ds, (uint64_t)T, ds_tk, (uint64_t)B * H, ds_tq, ds_tq * ds_tk, DQG_BK)) return rc;
  } else {
    memset(&tds_store, 0, sizeof(tds_store));
  }
  p.dq = reinterpret_cast<__nv_bfloat16*>(dq); p.dq_bs = gs->dq_batch_stride; p.dq_ts = gs->dq_token_stride;
  p.dk = reinterpret_cast<__nv_bfloat16*>(dk); p.dk_bs = gs->dk_batch_stride; p.dk_ts = gs->dk_token_stride;
  p.dv = reinterpret_cast<__nv_bfloat16*>(dv); p.dv_bs = gs->dv_batch_stride; p.dv_ts = gs->dv_token_stride;
  static DynSmemOnce once[5];
  TOME_CUDA(ensure_dyn_smem(attn_bwd_dkdv_ts_kernel<false>, DKT_SMEM, once[0]));
  TOME_CUDA(ensure_dyn_smem(attn_bwd_dkdv_ts_kernel<true>, DKT_SMEM, once[1]));
  TOME_CUDA(ensure_dyn_smem(attn_bwd_dq_kernel<false>, DQ_SMEM, once[2]));
  TOME_CUDA(ensure_dyn_smem(attn_bwd_dq_kernel<true>, DQ_SMEM, once[3]));
  TOME_CUDA(ensure_dyn_smem(attn_bwd_dq_gemm_kernel, DQG_SMEM, once[4]));
  {
    CUtensorMap tq, tk, tv, tdo;
    if (int rc = make_tmap_3d_bf16(&tq, q, hd, T, B, d->q_token_stride, d->q_batch_stride, DKV_BQ)) return rc;
    if (int rc = make_tmap_3d_bf16(&tk, k, hd, T, B, d->k_token_stride, d->k_batch_stride, DKV_BK)) return rc;
    if (int rc = make_tmap_3d_bf16(&tv, v, hd, T, B, d->v_token_stride, d->v_batch_stride, DKV_BK)) return rc;
    if (int rc = make_tmap_3d_bf16(&tdo, dout, hd, T, B, gs->do_token_stride, gs->do_batch_stride, DKV_BQ)) return rc;
    dim3 grid(ceil_div(T, DKV_BK), H, B);
    if (keep_k) launch_k(attn_bwd_dkdv_ts_kernel<true>, grid, DKT_THREADS, DKT_SMEM, stream, tq, tk, tv, tdo, tds_store, p);
    else launch_k(attn_bwd_dkdv_ts_kernel<false>, grid, DKT_THREADS, DKT_SMEM, stream, tq, tk, tv, tdo, tds_store, p);
    TOME_CUDA(cudaGetLastError());
  }
  if (from_ds) {
    CUtensorMap tk;
    if (int rc = make_tmap_3d_bf16(&tk, k, hd, T, B, d->k_token_stride, d->k_batch_stride, DQG_BK)) return rc;
    dim3 grid(ceil_div(T, DQG_BQ), H, B);
    launch_k(attn_bwd_dq_gemm_kernel, grid, AB_THREADS, DQG_SMEM, stream, tds_load, tk, p);
    TOME_CUDA(cudaGetLastError());
  } else {
    CUtensorMap tq, tk, tv, tdo;
    if (int rc = make_tmap_3d_bf16(&tq, q, hd, T, B, d->q_token_stride, d->q_batch_stride, DQ_BQ)) return rc;
    if (int rc = make_tmap_3d_bf16(&tk, k, hd, T, B, d->k_token_stride, d->k_batch_stride, DQ_BK)) return rc;
    if (int rc = make_tmap_3d_bf16(&tv, v, hd, T, B, d->v_token_stride, d->v_batch_stride, DQ_BK)) return rc;
    if (int rc = make_tmap_3d_bf16(&tdo, dout, hd, T, B, gs->do_token_stride, gs->do_batch_stride, DQ_BQ)) return rc;
    dim3 grid(ceil_div(T, DQ_BQ), H, B);
    if (keep_q) launch_k(attn_bwd_dq_kernel<true>, grid, AB_THREADS, DQ_SMEM, stream, tq, tk, tv, tdo, p);
    else launch_k(attn_bwd_dq_kernel<false>, grid, AB_THREADS, DQ_SMEM, stream, tq, tk, tv, tdo, p);
    TOME_CUDA(cudaGetLastError());
  }
  return TOME_OK;
}
