// K5: attention forward (flash style) on tcgen05 with the block-causal GROUP-TABLE mask and the proportional
// log(size) key bias.  Replaces flax dot_product_attention as reached from tome_attention.py:259-285 with the mask of
// token_sequencer.py:313-321 -- without ever materialising [B,H,T,T] logits, weights or booleans.
//
// One CTA = one (batch, head, 128-query tile); 2 CTAs per SM (256 TMEM columns each).  Key tiles are 64 wide, so a
// softmax thread holds one whole row of a tile (64 fp32 logits) in registers and touches every logit exactly once:
//   warp 4      TMA producer: Q once, then K_0 K_1 V_0 K_2 V_1 ... (64 keys x 64 each) through a 6-slot ring, 128B
//               swizzle; and, through a 4-slot ring, each key tile's METADATA block (attn_meta.cuh: log2(size) bias,
//               positions, one 64-bit "visible keys" word per QUERY GROUP -- the mask depends on a query only through
//               its group, so it costs the softmax one bit test per logit), one cp.async.bulk per tile
//   warp 5      UMMA issuer:  S_j = Q K_j^T (128x64x64) into a DOUBLE-BUFFERED TMEM accumulator (S_{j+1} is computed
//               while the softmax warps work on S_j); O += P_j V_j (128x64x64) accumulates IN TMEM across key tiles
//   warps 0..3  softmax, thread = query row: S_j (TMEM) -> registers, scale + bias (packed f32x2 FMA), mask, row max,
//               exp2, row sum, P_j -> bf16 written over the first 32 columns of S_j in TMEM.
//               The running maximum is LAZY: O and l are rescaled only when a row's maximum grows by more than 2^8,
//               which after the first tile is rare, so the usual tile needs no TMEM correction pass at all; when a
//               warp does need one it multiplies its 32 rows of O in TMEM by alpha (tcgen05.ld / st) before it
//               publishes P_j -- the PV MMA that reads O next is only issued after that.
// Both MMAs take their A operand from tensor memory: the softmax warps copy Q there once per CTA, and P_j overwrites S_j,
// so P never passes through shared memory.
// Logits are kept in the log2 domain: s2 = (q.k) * scale * log2(e) + log2(size_k); masked -> -FLT_MAX (finite, as
// flax's finfo.min), keys past T -> -inf.
#include <float.h>

#include "attn_meta.cuh"
#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int ATT_BM = 128;   // queries per CTA
constexpr int ATT_BN = 64;    // keys per tile
constexpr int ATT_D = 64;
constexpr int ATT_THREADS = 192;
constexpr int ATT_Q_BYTES = ATT_BM * ATT_D * 2;         // 16 KB
constexpr int ATT_KV_BYTES = ATT_BN * ATT_D * 2;        // 8 KB each for K and V
constexpr int ATT_SLOTS = 5;  // ring of 8 KB slots; items are loaded in the order K_0 K_1 V_0 K_2 V_1 ...
constexpr int ATT_MSLOTS = 4; // metadata ring
constexpr int ATT_QAUG_BYTES = ATT_BM * ATTN_AUG_K * 2;   // 4 KB: mask augmentation operand of the query tile (attn_meta.cuh)
constexpr int ATT_KAUG_BYTES = ATT_BN * ATTN_AUG_K * 2;   // 2 KB per key tile, one per ring slot
constexpr int ATT_META_SLOT = ATTN_META_KEY_BYTES + ATTN_DROP_TILE_BYTES;  // bias2 | vis[32][2] | visc[32][2] | pos | dropout keep words [128][2]
static_assert(ATT_BN == ATTN_META_TILE, "key tiles and metadata tiles must coincide");
constexpr int ATT_SMEM = ATT_Q_BYTES + ATT_SLOTS * ATT_KV_BYTES + ATT_QAUG_BYTES + ATT_SLOTS * ATT_KAUG_BYTES +
                         ATT_MSLOTS * ATT_META_SLOT + 512 + 1024;
constexpr uint32_t ATT_TMEM_COLS = 256;  // S0 [0,64) S1 [64,128) O [128,192) Q [192,224)
constexpr float ATT_LAZY_LOG2 = 8.0f;    // rescale O only when the row maximum grows by more than 2^8

struct AttnFwdParams {
  int batch, tokens, heads;
  float scale_log2;  // scale * log2(e)
  const uint8_t* gid;   // null: no mask
  const int32_t* pos;
  const uint8_t* meta;  // [B][n_kv][ATTN_META_BYTES]
  const uint32_t* aug_flag;  // != 0: the mask is folded into S by one extra K = 16 MMA step (attn_meta.cuh)
  const uint8_t* keep_q;  // attention dropout keep words [n_q128][n_kv][128][2] or null
  float inv_keep;         // 1 / (1 - rate)
  __nv_bfloat16* out;
  long long o_batch_stride, o_token_stride;
  float* lse;
};

// TMEM -> 32 consecutive fp32 registers of a larger per-thread array (indices are compile-time after unrolling)
template <int OFF, int N>
__device__ __forceinline__ void tmem_ld_f32x32(uint32_t taddr, float (&r)[N]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=f"(r[OFF + 0]), "=f"(r[OFF + 1]), "=f"(r[OFF + 2]), "=f"(r[OFF + 3]), "=f"(r[OFF + 4]), "=f"(r[OFF + 5]),
        "=f"(r[OFF + 6]), "=f"(r[OFF + 7]), "=f"(r[OFF + 8]), "=f"(r[OFF + 9]), "=f"(r[OFF + 10]), "=f"(r[OFF + 11]),
        "=f"(r[OFF + 12]), "=f"(r[OFF + 13]), "=f"(r[OFF + 14]), "=f"(r[OFF + 15]), "=f"(r[OFF + 16]), "=f"(r[OFF + 17]),
        "=f"(r[OFF + 18]), "=f"(r[OFF + 19]), "=f"(r[OFF + 20]), "=f"(r[OFF + 21]), "=f"(r[OFF + 22]), "=f"(r[OFF + 23]),
        "=f"(r[OFF + 24]), "=f"(r[OFF + 25]), "=f"(r[OFF + 26]), "=f"(r[OFF + 27]), "=f"(r[OFF + 28]), "=f"(r[OFF + 29]),
        "=f"(r[OFF + 30]), "=f"(r[OFF + 31])
      : "r"(taddr)
      : "memory");
}

// DROP: attention-weight dropout compiled in (the keep words ride in the metadata ring); the rate-0 instantiation carries none of it
template <bool DROP>
__global__ void __launch_bounds__(ATT_THREADS, 2)
attn_fwd_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k,
                const __grid_constant__ CUtensorMap tm_v, const __grid_constant__ CUtensorMap tm_qaug,
                const __grid_constant__ CUtensorMap tm_kaug, const AttnFwdParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1 KB alignment by pointer arithmetic on the __shared__ array itself, so every access below stays LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_q = smem;
  uint8_t* s_kv = s_q + ATT_Q_BYTES;                        // slot i at i * 8 KB
  uint8_t* s_qaug = s_kv + ATT_SLOTS * ATT_KV_BYTES;        // [128 rows][16] bf16, 32-byte swizzle
  uint8_t* s_kaug = s_qaug + ATT_QAUG_BYTES;                // slot i at i * 2 KB (only K slots use theirs)
  uint8_t* s_meta = s_kaug + ATT_SLOTS * ATT_KAUG_BYTES;    // metadata slot i at i * ATT_META_SLOT
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_meta + ATT_MSLOTS * ATT_META_SLOT);
  uint64_t* q_full = bars;                 // 1
  uint64_t* kv_full = bars + 1;            // [ATT_SLOTS] (room for 6)
  uint64_t* kv_empty = bars + 7;           // [ATT_SLOTS] (room for 6)
  uint64_t* s_full = bars + 13;            // [2]  S_j ready in TMEM buffer j&1
  uint64_t* p_ready = bars + 15;           // [2]  P_j in TMEM buffer j&1, S_j consumed, O corrected (128 arrivals)
  uint64_t* pv_done = bars + 17;           // [2]  O += P_j V_j retired: O readable
  uint64_t* meta_full = bars + 19;         // [ATT_MSLOTS]  bulk copy of the tile's metadata block landed
  uint64_t* meta_empty = bars + 23;        // [ATT_MSLOTS]  128 arrivals (softmax threads), after the P stores of the tile
  uint64_t* q_ready = bars + 27;           // the query tile has been copied into tensor memory (128 arrivals)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 28);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qt = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int T = p.tokens;
  const int n_kv = (T + ATT_BN - 1) / ATT_BN;

  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    mbar_init(q_ready, ATT_BM);
    for (int i = 0; i < ATT_SLOTS; ++i) {
      mbar_init(&kv_full[i], 1);
      mbar_init(&kv_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], ATT_BM);
      mbar_init(&pv_done[i], 1);
    }
    for (int i = 0; i < ATT_MSLOTS; ++i) {
      mbar_init(&meta_full[i], 1);
      mbar_init(&meta_empty[i], ATT_BM);
    }
    fence_barrier_init();
  }
  if (warp == 4 && lane == 0) {
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_k);
    tma_prefetch_desc(&tm_v);
  }
  if (warp == 5) tmem_alloc(tmem_slot, ATT_TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_o = tmem_base + 128;   // 64 columns; S buffers at +0 and +64
  const uint32_t tmem_q = tmem_base + 192;   // 32 columns = 128 x 64 bf16
  const bool has_mask = p.gid != nullptr;
  // the mask rides in the QK^T contraction (attn_meta.cuh) when the table allows it; CTA-uniform
  const bool use_aug = has_mask && *p.aug_flag != 0u;

  if (warp == 4) {
    // ================================================================= TMA producer: K/V ring + metadata ring
    if (lane == 0) {
      int item = 0;
      auto load_item = [&](bool is_v, int tile) {  // ring order K_0 K_1 V_0 K_2 V_1 ... K_{n-1} V_{n-2} V_{n-1}
        const int slot = item % ATT_SLOTS, use = item / ATT_SLOTS;
        mbar_wait(&kv_empty[slot], (use & 1) ^ 1);
        const bool aug = use_aug && !is_v;   // a K tile brings its 2 KB one-hot group operand along
        mbar_expect_tx(&kv_full[slot], ATT_KV_BYTES + (aug ? ATT_KAUG_BYTES : 0));
        tma_load_3d(s_kv + slot * ATT_KV_BYTES, is_v ? &tm_v : &tm_k, &kv_full[slot], h * ATT_D, tile * ATT_BN, b);
        if (aug) tma_load_3d(s_kaug + slot * ATT_KAUG_BYTES, &tm_kaug, &kv_full[slot], 0, tile * ATT_BN, b);
        ++item;
      };
      // with the mask folded into S only the bias (and the dropout words) are read from the metadata block
      const uint32_t meta_bytes = (has_mask && !use_aug) ? ATTN_META_KEY_BYTES : 256u;
      const uint8_t* meta_b = p.meta + (size_t)b * n_kv * ATTN_META_BYTES;
      mbar_expect_tx(q_full, ATT_Q_BYTES + (use_aug ? ATT_QAUG_BYTES : 0));
      tma_load_3d(s_q, &tm_q, q_full, h * ATT_D, qt * ATT_BM, b);
      if (use_aug) tma_load_3d(s_qaug, &tm_qaug, q_full, 0, qt * ATT_BM, b);
      load_item(false, 0);
      for (int j = 0; j < n_kv; ++j) {
        const int ms = j % ATT_MSLOTS;
        mbar_wait(&meta_empty[ms], ((j / ATT_MSLOTS) & 1) ^ 1);
        mbar_expect_tx(&meta_full[ms], meta_bytes + (DROP ? ATTN_DROP_TILE_BYTES : 0));
        bulk_g2s(s_meta + ms * ATT_META_SLOT, meta_b + (size_t)j * ATTN_META_BYTES, meta_bytes, &meta_full[ms]);
        if constexpr (DROP)
          bulk_g2s(s_meta + ms * ATT_META_SLOT + ATTN_META_KEY_BYTES, p.keep_q + ((size_t)qt * n_kv + j) * ATTN_DROP_TILE_BYTES,
                   ATTN_DROP_TILE_BYTES, &meta_full[ms]);
        if (j + 1 < n_kv) load_item(false, j + 1);
        load_item(true, j);
      }
    }
  } else if (warp == 5) {
    // ================================================================= UMMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_bf16(ATT_BM, ATT_BN, false, false);  // Q K-major, K K-major
      constexpr uint32_t idesc_o = make_idesc_bf16(ATT_BM, ATT_D, false, true);    // P K-major, V MN-major
      const int n_items = 2 * n_kv;
      auto issue_s = [&](int t) {  // S_t = Q K_t^T into TMEM buffer t&1
        const int item = t == 0 ? 0 : 2 * t - 1, slot = item % ATT_SLOTS;
        mbar_wait(&kv_full[slot], (item / ATT_SLOTS) & 1);
        tc_fence_after();
        const uint32_t ak = smem_u32(s_kv + slot * ATT_KV_BYTES);
#pragma unroll
        for (int k = 0; k < ATT_D / 16; ++k)
          umma_bf16_ts(tmem_base + (t & 1) * ATT_BN, tmem_q + k * 8, make_smem_desc(ak + k * 32, 16, 1024), idesc_s, k > 0 ? 1u : 0u);
        if (use_aug)  // S += Mq Ek^T: 0 where the query's group sees the key's group, -2^100 (absorbing) where it does not
          umma_bf16(tmem_base + (t & 1) * ATT_BN, make_smem_desc_sw32(smem_u32(s_qaug)),
                    make_smem_desc_sw32(smem_u32(s_kaug + slot * ATT_KAUG_BYTES)), idesc_s, 1u);
        umma_commit(&s_full[t & 1]);
        umma_commit(&kv_empty[slot]);
      };
      mbar_wait(q_ready, 0);
      tc_fence_after();
      issue_s(0);
      if (n_kv > 1) issue_s(1);
      for (int j = 0; j < n_kv; ++j) {
        mbar_wait(&p_ready[j & 1], (j >> 1) & 1);  // P_j in TMEM, S_j consumed, O corrected
        tc_fence_after();
        const int item = j == n_kv - 1 ? n_items - 1 : 2 * j + 2, slot = item % ATT_SLOTS;
        mbar_wait(&kv_full[slot], (item / ATT_SLOTS) & 1);
        tc_fence_after();
        const uint32_t av = smem_u32(s_kv + slot * ATT_KV_BYTES);
#pragma unroll
        for (int k = 0; k < ATT_BN / 16; ++k)  // O += P_j V_j
          umma_bf16_ts(tmem_o, tmem_base + (j & 1) * ATT_BN + k * 8, make_smem_desc(av + k * 2048, 8192, 1024), idesc_o,
                       (j > 0 || k > 0) ? 1u : 0u);
        umma_commit(&pv_done[j & 1]);
        umma_commit(&kv_empty[slot]);
        if (j + 2 < n_kv) issue_s(j + 2);
      }
    }
  } else {
    // ================================================================= softmax warps (thread = query row)
    const int row = threadIdx.x;                 // 0..127 == TMEM lane
    const int q = qt * ATT_BM + row;
    const uint32_t lane_sel = ((uint32_t)(warp * 32)) << 16;
    const bool warp_active = qt * ATT_BM + warp * 32 < T;  // a warp whose 32 rows are all past T only keeps the barriers moving
    int gq = 0, pos_q = 0;
    if (has_mask && q < T) {
      gq = p.gid[(long long)b * T + q];
      pos_q = p.pos[(long long)b * T + q];
    }
    float m_run = -INFINITY, l_run = 0.f;
    const float2 scale2 = make_float2(p.scale_log2, p.scale_log2);
    {  // this thread's query row: shared memory (128B-swizzled, as TMA wrote it) -> 32 TMEM columns
      mbar_wait(q_full, 0);
      uint32_t qw[32];
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        const uint4 t = *reinterpret_cast<const uint4*>(s_q + row * 128 + ((ch ^ (row & 7)) << 4));
        qw[4 * ch] = t.x; qw[4 * ch + 1] = t.y; qw[4 * ch + 2] = t.z; qw[4 * ch + 3] = t.w;
      }
      tmem_st_x32(tmem_q + lane_sel, qw);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(q_ready);
    }

    for (int j = 0; j < n_kv; ++j) {
      const int ms = j % ATT_MSLOTS;
      const uint8_t* mb = s_meta + ms * ATT_META_SLOT;
      mbar_wait(&meta_full[ms], (j / ATT_MSLOTS) & 1);
      if (!warp_active) {
        mbar_wait(&s_full[j & 1], (j >> 1) & 1);   // pacing only: S_{j+2} is not issued before p_ready(j) completes
        mbar_arrive(&meta_empty[ms]);
        mbar_arrive(&p_ready[j & 1]);
        continue;
      }
      const float4* bias4 = reinterpret_cast<const float4*>(mb);
      uint32_t vw0 = 0xffffffffu, vw1 = 0xffffffffu;
      bool masked_tile = false;
      if (has_mask && !use_aug) {
        const uint2 vv = *reinterpret_cast<const uint2*>(mb + ATTN_META_OFF_VIS + gq * 8);
        const uint2 vc = *reinterpret_cast<const uint2*>(mb + ATTN_META_OFF_VISC + gq * 8);
        vw0 = vv.x; vw1 = vv.y;
        if (vc.x | vc.y) {  // rare (Text sets): fold the causal rule into the visibility words
          const int* m_pos = reinterpret_cast<const int*>(mb + ATTN_META_OFF_POS);
          for (int i = 0; i < 32; ++i) {
            if (((vc.x >> i) & 1u) && m_pos[i] <= pos_q) vw0 |= 1u << i;
            if (((vc.y >> i) & 1u) && m_pos[32 + i] <= pos_q) vw1 |= 1u << i;
          }
        }
        masked_tile = !__all_sync(0xffffffffu, (vw0 & vw1) == 0xffffffffu);  // warp-uniform: skip the selects when nothing is masked
      }

      uint2 kb = make_uint2(0xffffffffu, 0xffffffffu);  // dropout keep bits of this row's 64 keys
      if constexpr (DROP) kb = *reinterpret_cast<const uint2*>(mb + ATTN_META_KEY_BYTES + row * 8);

      mbar_wait(&s_full[j & 1], (j >> 1) & 1);
      tc_fence_after();
      float s[ATT_BN];
      const uint32_t ts = tmem_base + (j & 1) * ATT_BN + lane_sel;
      tmem_ld_f32x32<0>(ts, s);
      tmem_ld_f32x32<32>(ts + 32, s);
      tmem_ld_wait();

      // s2 = s * scale*log2e + log2(size_k)     (packed f32x2 FMA: two logits per instruction)
#pragma unroll
      for (int i4 = 0; i4 < ATT_BN / 4; ++i4) {
        const float4 bb = bias4[i4];
        const float2 t0 = __ffma2_rn(make_float2(s[4 * i4], s[4 * i4 + 1]), scale2, make_float2(bb.x, bb.y));
        const float2 t1 = __ffma2_rn(make_float2(s[4 * i4 + 2], s[4 * i4 + 3]), scale2, make_float2(bb.z, bb.w));
        s[4 * i4] = t0.x; s[4 * i4 + 1] = t0.y; s[4 * i4 + 2] = t1.x; s[4 * i4 + 3] = t1.y;
      }
      if (masked_tile) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
          s[i] = ((vw0 >> i) & 1u) ? s[i] : -FLT_MAX;
          s[32 + i] = ((vw1 >> i) & 1u) ? s[32 + i] : -FLT_MAX;
        }
      }
      float mt[4];  // four independent maxima: a single 31-deep dependent chain would serialise on the ALU latency
#pragma unroll
      for (int c = 0; c < 4; ++c) mt[c] = fmaxf(s[16 * c], s[16 * c + 1]);
#pragma unroll
      for (int i = 2; i < 16; i += 2)
#pragma unroll
        for (int c = 0; c < 4; ++c) mt[c] = fmaxf(mt[c], fmaxf(s[16 * c + i], s[16 * c + i + 1]));
      float m_tile = fmaxf(fmaxf(mt[0], mt[1]), fmaxf(mt[2], mt[3]));
      // m_tile >= -FLT_MAX: every tile holds at least one key < T, whose logit is finite or -FLT_MAX

      if (j == 0) {
        m_run = m_tile;
      } else {
        const float m_new = fmaxf(m_run, m_tile);
        const bool need = (m_new - m_run) > ATT_LAZY_LOG2;
        if (__any_sync(0xffffffffu, need)) {  // rare after the first tiles: correct this warp's 32 rows of O in TMEM
          const float alpha = need ? fast_exp2(m_run - m_new) : 1.0f;
          if (need) m_run = m_new;
          l_run *= alpha;
          mbar_wait(&pv_done[(j - 1) & 1], ((j - 1) >> 1) & 1);  // O holds tiles 0..j-1
          tc_fence_after();
#pragma unroll
          for (int c0 = 0; c0 < ATT_D; c0 += 32) {
            uint32_t v[32];
            tmem_ld_x32(tmem_o + lane_sel + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
            tmem_st_x32(tmem_o + lane_sel + c0, v);
          }
          tmem_st_wait();
        }
      }

      // P = exp2(s2 - m_run) -> bf16: the A operand of the PV product, written over the first 32 columns of S_j in tensor
      // memory (every logit of this row is already in registers; S_{j+2}, which reuses the buffer, is issued behind P_j V_j)
      const float2 nm2 = make_float2(-m_run, -m_run);
      float2 l2[4];  // four independent partial row sums (same reason as the maxima)
#pragma unroll
      for (int u = 0; u < 4; ++u) l2[u] = make_float2(0.f, 0.f);
      uint32_t pw[32];
#pragma unroll
      for (int ch = 0; ch < ATT_BN / 8; ++ch) {  // 8 chunks of 8 keys = 16 bytes
        uint32_t w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float2 d = __fadd2_rn(make_float2(s[ch * 8 + 2 * u], s[ch * 8 + 2 * u + 1]), nm2);
          float2 e = make_float2(fast_exp2(d.x), fast_exp2(d.y));
          l2[u] = __fadd2_rn(l2[u], e);   // the row sum is that of the UNdropped weights (dropout follows the softmax)
          if constexpr (DROP) {
            const uint32_t kw = ch < 4 ? kb.x : kb.y;
            const int bit = (ch & 3) * 8 + 2 * u;
            e.x = ((kw >> bit) & 1u) ? e.x : 0.f;
            e.y = ((kw >> (bit + 1)) & 1u) ? e.y : 0.f;
          }
          w[u] = pack_bf16(e.x, e.y);
        }
        pw[4 * ch] = w[0]; pw[4 * ch + 1] = w[1]; pw[4 * ch + 2] = w[2]; pw[4 * ch + 3] = w[3];
      }
      tmem_st_x32(ts, pw);
      tmem_st_wait();
      const float2 lsum = __fadd2_rn(__fadd2_rn(l2[0], l2[1]), __fadd2_rn(l2[2], l2[3]));
      l_run += lsum.x + lsum.y;
      // Release the metadata slot only HERE, after the P stores above: they consume every value loaded from the slot (bias,
      // visibility words, keep bits), so all those shared-memory loads have returned.  An arrive placed right after the
      // loads were merely ISSUED let the producer's next bulk copy overwrite the slot under loads still queued behind the
      // MUFU / tcgen05.ld traffic: rows then saw the bias of the tile three ahead (-inf past T) -- wrong, and different
      // from run to run.  Found by the full-size reproducibility test; invisible at small batch.
      mbar_arrive(&meta_empty[ms]);
      tc_fence_before();         // our TMEM reads of S_j / writes of O (and P_j) are ordered before the MMAs that follow
      mbar_arrive(&p_ready[j & 1]);
    }
    // O is final once the last P V retires
    mbar_wait(&pv_done[(n_kv - 1) & 1], ((n_kv - 1) >> 1) & 1);
    tc_fence_after();
    if (warp_active) {
      const float inv_l = p.inv_keep / l_run;   // 1 / (1 - rate) of the dropout folded into the normalisation
      __nv_bfloat16* orow = p.out + (long long)b * p.o_batch_stride + (long long)(q < T ? q : 0) * p.o_token_stride + h * ATT_D;
#pragma unroll
      for (int c0 = 0; c0 < ATT_D; c0 += 32) {
        uint32_t v[32];
        tmem_ld_x32(tmem_o + lane_sel + c0, v);   // warp-collective: rows past T take part and only skip the stores
        tmem_ld_wait();
        if (q < T) {
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            const uint4 w = make_uint4(pack_bf16(__uint_as_float(v[i]) * inv_l, __uint_as_float(v[i + 1]) * inv_l),
                                       pack_bf16(__uint_as_float(v[i + 2]) * inv_l, __uint_as_float(v[i + 3]) * inv_l),
                                       pack_bf16(__uint_as_float(v[i + 4]) * inv_l, __uint_as_float(v[i + 5]) * inv_l),
                                       pack_bf16(__uint_as_float(v[i + 6]) * inv_l, __uint_as_float(v[i + 7]) * inv_l));
            *reinterpret_cast<uint4*>(orow + c0 + i) = w;
          }
        }
      }
      if (q < T && p.lse) p.lse[((long long)b * p.heads + h) * T + q] = (m_run + log2f(l_run)) * 0.6931471805599453f;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 5) {
    tc_fence_after();
    tmem_dealloc(tmem_base, ATT_TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------ metadata (attn_meta.cuh)
__global__ void __launch_bounds__(ATTN_META_TILE)
attn_meta_kernel(int T, const uint8_t* __restrict__ gid, const int32_t* __restrict__ pos, const uint8_t* __restrict__ allow,
                 int G, const float* __restrict__ size, uint8_t* __restrict__ meta, uint32_t* __restrict__ aug_flag,
                 uint4* __restrict__ aug_q, uint4* __restrict__ aug_k) {
  const int tile = blockIdx.x, b = blockIdx.y, t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const int idx = tile * ATTN_META_TILE + t;
  const bool valid = idx < T;
  uint8_t* m = meta + ((size_t)b * gridDim.x + tile) * ATTN_META_BYTES;
  if (tile == 0 && b == 0 && t == 0) {  // does the augmentation apply?  a mask, at most 16 groups, no positional rule
    uint32_t ok = (gid != nullptr && G <= ATTN_AUG_K) ? 1u : 0u;
    for (int i = 0; ok && i < G * G; ++i)
      if (allow[i] == 2) ok = 0u;
    *aug_flag = ok;
  }
  {  // augmentation operands of this token: 16 bf16 each (two 16-byte stores); zeros past T or without a mask
    uint32_t qw[8] = {0, 0, 0, 0, 0, 0, 0, 0}, kw[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (gid != nullptr && valid && G <= ATTN_AUG_K) {
      const int g = gid[(long long)b * T + idx];
      for (int o = 0; o < G; ++o) {
        const uint32_t mq = allow[g * G + o] == 1 ? 0u : 0xF180u;   // bf16(-2^100)
        qw[o >> 1] |= mq << ((o & 1) * 16);
      }
      kw[g >> 1] |= 0x3F80u << ((g & 1) * 16);                       // bf16(1)
    }
    const size_t row = ((size_t)b * gridDim.x + tile) * ATTN_META_TILE + t;
    aug_q[row * 2] = make_uint4(qw[0], qw[1], qw[2], qw[3]);
    aug_q[row * 2 + 1] = make_uint4(qw[4], qw[5], qw[6], qw[7]);
    aug_k[row * 2] = make_uint4(kw[0], kw[1], kw[2], kw[3]);
    aug_k[row * 2 + 1] = make_uint4(kw[4], kw[5], kw[6], kw[7]);
  }
  reinterpret_cast<float*>(m)[t] = valid ? (size ? log2f(size[(long long)b * T + idx]) : 0.f) : -INFINITY;
  uint32_t cw = 0xffffffffu, cc = 0u, rw = 0xffffffffu, rc = 0u;  // tokens past T: "visible" (the -inf bias / +inf lse removes them)
  int ps = 0;
  if (gid != nullptr && valid) {
    const int g = gid[(long long)b * T + idx];
    ps = pos[(long long)b * T + idx];
    cw = cc = rw = rc = 0u;
    for (int o = 0; o < G; ++o) {
      const int a_col = allow[o * G + g];  // query group o looking at this token as a KEY
      const int a_row = allow[g * G + o];  // this token as a QUERY looking at key group o
      cw |= (a_col == 1 ? 1u : 0u) << o;
      cc |= (a_col == 2 ? 1u : 0u) << o;
      rw |= (a_row == 1 ? 1u : 0u) << o;
      rc |= (a_row == 2 ? 1u : 0u) << o;
    }
  }
  reinterpret_cast<int*>(m + ATTN_META_OFF_POS)[t] = ps;
  uint32_t* vis = reinterpret_cast<uint32_t*>(m + ATTN_META_OFF_VIS);
  uint32_t* visc = reinterpret_cast<uint32_t*>(m + ATTN_META_OFF_VISC);
  uint32_t* qvis = reinterpret_cast<uint32_t*>(m + ATTN_META_OFF_QVIS);
  uint32_t* qvisc = reinterpret_cast<uint32_t*>(m + ATTN_META_OFF_QVISC);
  for (int g = 0; g < 32; ++g) {
    const uint32_t w0 = __ballot_sync(0xffffffffu, (cw >> g) & 1u), w1 = __ballot_sync(0xffffffffu, (cc >> g) & 1u);
    const uint32_t w2 = __ballot_sync(0xffffffffu, (rw >> g) & 1u), w3 = __ballot_sync(0xffffffffu, (rc >> g) & 1u);
    if (lane == 0) {
      vis[g * 2 + warp] = w0;
      visc[g * 2 + warp] = w1;
      qvis[g * 2 + warp] = w2;
      qvisc[g * 2 + warp] = w3;
    }
  }
}

int launch_attn_meta(int B, int T, const uint8_t* gid, const int32_t* pos, const uint8_t* allow, int G, const float* size,
                     uint8_t* meta, cudaStream_t stream) {
  TOME_CHECK(meta != nullptr && ((uintptr_t)meta & 15) == 0, TOME_ERR_INVALID, "attention: workspace must be non-null and 16-byte aligned");
  dim3 grid((T + ATTN_META_TILE - 1) / ATTN_META_TILE, B);
  launch_k(attn_meta_kernel, grid, ATTN_META_TILE, 0, stream, 
      T, gid, pos, allow, G, size, meta, const_cast<uint32_t*>(attn_aug_flag(meta, B, T)),
      reinterpret_cast<uint4*>(const_cast<uint8_t*>(attn_aug_q(meta, B, T))),
      reinterpret_cast<uint4*>(const_cast<uint8_t*>(attn_aug_k(meta, B, T))));
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

// ------------------------------------------------------------------------------------------------ dropout keep bits (attn_meta.cuh)
// thread = (query q, 32-key word w), q fastest: a warp holds 32 consecutive queries of one word, so the transposed words
// come from 32 ballots
__global__ void __launch_bounds__(256)
attn_dropbits_kernel(int n128, int n64, DropoutCfg d, uint32_t* __restrict__ keep_q, uint32_t* __restrict__ keep_k) {
  const int Tq = n128 * 128;                       // padded query / key range: both arrays are written completely
  const long long t = blockIdx.x * 256ll + threadIdx.x;
  const int q = (int)(t % Tq), w = (int)(t / Tq);  // w < n128 * 4
  if (w >= n128 * 4) return;                        // whole warps leave together (Tq % 32 == 0)
  DropStream st = drop_stream(d, (uint32_t)q, (uint32_t)w);
  const uint32_t thr = d.thresh16 << 16;
  uint32_t word = 0;
#pragma unroll
  for (int e = 0; e < 32; ++e) word |= (st.next() >= thr ? 1u : 0u) << e;
  if ((w >> 1) < n64)  // key tile w/2 exists in the 64-wide tiling
    keep_q[(((long long)(q >> 7) * n64 + (w >> 1)) * 128 + (q & 127)) * 2 + (w & 1)] = word;
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int e = 0; e < 32; ++e) {
    const uint32_t col = __ballot_sync(0xffffffffu, (word >> e) & 1u);  // bit l: keep(q_base + l, 32 w + e)
    if (lane == e) {
      const int kk = 32 * w + e, q0 = q & ~31;   // this lane's q is q0 + e; the word covers queries q0 .. q0 + 31
      if ((q0 >> 6) < n64)
        keep_k[(((long long)(kk >> 7) * n64 + (q0 >> 6)) * 128 + (kk & 127)) * 2 + ((q0 >> 5) & 1)] = col;
    }
  }
}

int launch_attn_dropbits(int T, float rate, uint64_t seed, uint32_t site, uint8_t* bits, cudaStream_t stream) {
  TOME_CHECK(bits != nullptr && ((uintptr_t)bits & 15) == 0, TOME_ERR_INVALID, "attention: dropout workspace must be 16-byte aligned");
  TOME_CHECK(rate > 0.f && rate < 1.f, TOME_ERR_INVALID, "attention: dropout_rate must be in [0, 1)");
  const int n128 = (T + 127) / 128, n64 = (T + 63) / 64;
  const DropoutCfg d = make_dropout(rate, seed, site);
  uint32_t* kq = reinterpret_cast<uint32_t*>(bits);
  uint32_t* kk = kq + (size_t)n128 * n64 * (ATTN_DROP_TILE_BYTES / 4);
  const long long threads = (long long)n128 * 128 * n128 * 4;
  launch_k(attn_dropbits_kernel, (unsigned)((threads + 255) / 256), 256, 0, stream, n128, n64, d, kq, kk);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

}  // namespace tome

using namespace tome;

namespace tome {
int attn_generic_fwd(const tome_attn_desc_t* d, const void* q, const void* k, const void* v, void* out, float* lse,
                     cudaStream_t stream);  // attn_generic.cu
int check_attn_desc(const tome_attn_desc_t* d, const char* who) {
  TOME_CHECK(d != nullptr, TOME_ERR_INVALID, "%s: null descriptor", who);
  TOME_CHECK(d->batch > 0 && d->tokens > 0 && d->heads > 0, TOME_ERR_INVALID, "%s: bad shape", who);
  TOME_CHECK(d->head_dim >= 8 && d->head_dim <= 256 && d->head_dim % 8 == 0, TOME_ERR_UNSUPPORTED,
             "%s: head_dim %d not supported (64 runs on tensor cores; other multiples of 8 up to 256 on the generic path)", who,
             d->head_dim);
  TOME_CHECK(d->batch <= 65535 && d->heads <= 65535, TOME_ERR_INVALID, "%s: batch/heads exceed grid limits", who);
  TOME_CHECK(!d->gid || (d->pos && d->allow && d->num_groups >= 1 && d->num_groups <= 32), TOME_ERR_INVALID,
             "%s: a group mask needs pos, allow and 1 <= num_groups <= 32 (got %d)", who, d->num_groups);
  const long long strides[8] = {d->q_batch_stride, d->q_token_stride, d->k_batch_stride, d->k_token_stride,
                                d->v_batch_stride, d->v_token_stride, d->o_batch_stride, d->o_token_stride};
  for (int i = 0; i < 8; ++i)
    TOME_CHECK(strides[i] % 8 == 0, TOME_ERR_INVALID, "%s: strides must be multiples of 8 elements (16 bytes)", who);
  return TOME_OK;
}
}  // namespace tome

struct FwdWs {
  uint8_t* meta;  // per-tile metadata (launch_attn_meta)
  uint8_t* bits;  // dropout keep bits (launch_attn_dropbits), only with dropout
  size_t total;
};
static FwdWs fwd_ws(const tome_attn_desc_t* d, void* base) {
  Bump b{reinterpret_cast<uint8_t*>(base)};
  FwdWs w;
  w.meta = b.take<uint8_t>(attn_meta_bytes(d->batch, d->tokens));
  w.bits = b.take<uint8_t>(d->dropout_rate > 0.f ? attn_dropbits_bytes(d->tokens) : 0);
  w.total = b.total();
  return w;
}

extern "C" size_t tome_attention_workspace_bytes(const tome_attn_desc_t* d) {
  if (!d || d->batch <= 0 || d->tokens <= 0) return 0;
  return fwd_ws(d, nullptr).total;
}

extern "C" int tome_attention_fwd(const tome_attn_desc_t* d, const void* q, const void* k, const void* v, void* out,
                                  float* lse, void* workspace, size_t workspace_bytes, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int rc = check_attn_desc(d, "attention_fwd")) return rc;
  TOME_CHECK(q && k && v && out, TOME_ERR_INVALID, "attention_fwd: null tensor");
  TOME_CHECK(((uintptr_t)out & 15) == 0, TOME_ERR_INVALID, "attention_fwd: out must be 16-byte aligned");
  TOME_CHECK(d->dropout_rate >= 0.f && d->dropout_rate < 1.f, TOME_ERR_INVALID, "attention_fwd: dropout_rate must be in [0, 1)");
  if (d->head_dim != ATT_D) {  // e.g. the literal reference config (3 heads x 256): fp32 CUDA-core path, same semantics
    ProfScope prof(PROF_ATTN_FWD, 4.0 * d->batch * d->heads * (double)d->tokens * d->tokens * d->head_dim, 1, stream);
    return attn_generic_fwd(d, q, k, v, out, lse, stream);
  }
  const FwdWs ws = fwd_ws(d, workspace);
  TOME_CHECK(workspace && workspace_bytes >= ws.total, TOME_ERR_INVALID,
             "attention_fwd: workspace too small (%zu < %zu, see tome_attention_workspace_bytes)", workspace_bytes, ws.total);
  TOME_CHECK(((uintptr_t)workspace & 255) == 0, TOME_ERR_INVALID, "attention_fwd: workspace must be 256-byte aligned");
  TOME_CHECK(d->dropout_rate >= 0.f && d->dropout_rate < 1.f, TOME_ERR_INVALID, "attention_fwd: dropout_rate must be in [0, 1)");
  CUtensorMap tq, tk, tv;
  const uint64_t hd = (uint64_t)d->heads * d->head_dim;
  ProfScope prof(PROF_ATTN_FWD, 4.0 * d->batch * d->heads * (double)d->tokens * d->tokens * d->head_dim, 2, stream);
  if (int rc = launch_attn_meta(d->batch, d->tokens, d->gid, d->pos, d->allow, d->num_groups, d->size, ws.meta, stream)) return rc;
  if (int rc = make_tmap_3d_bf16(&tq, q, hd, d->tokens, d->batch, d->q_token_stride, d->q_batch_stride, ATT_BM)) return rc;
  if (int rc = make_tmap_3d_bf16(&tk, k, hd, d->tokens, d->batch, d->k_token_stride, d->k_batch_stride, ATT_BN)) return rc;
  if (int rc = make_tmap_3d_bf16(&tv, v, hd, d->tokens, d->batch, d->v_token_stride, d->v_batch_stride, ATT_BN)) return rc;
  AttnFwdParams p;
  p.batch = d->batch; p.tokens = d->tokens; p.heads = d->heads;
  p.scale_log2 = d->scale * 1.4426950408889634f;
  p.gid = d->gid; p.pos = d->pos; p.meta = ws.meta;
  p.aug_flag = attn_aug_flag(p.meta, d->batch, d->tokens);
  CUtensorMap tqa, tka;
  {
    const uint64_t tp = attn_tiles(d->tokens) * ATTN_META_TILE;
    if (int rc = make_tmap_3d_bf16_sw32(&tqa, attn_aug_q(p.meta, d->batch, d->tokens), tp, d->batch, ATT_BM)) return rc;
    if (int rc = make_tmap_3d_bf16_sw32(&tka, attn_aug_k(p.meta, d->batch, d->tokens), tp, d->batch, ATT_BN)) return rc;
  }
  p.keep_q = nullptr;
  p.inv_keep = 1.0f;
  if (d->dropout_rate > 0.f) {
    if (int rc = launch_attn_dropbits(d->tokens, d->dropout_rate, d->dropout_seed, d->dropout_site, ws.bits, stream)) return rc;
    p.keep_q = ws.bits;
    p.inv_keep = make_dropout(d->dropout_rate, d->dropout_seed, d->dropout_site).inv_keep;
  }
  p.out = reinterpret_cast<__nv_bfloat16*>(out);
  p.o_batch_stride = d->o_batch_stride; p.o_token_stride = d->o_token_stride;
  p.lse = lse;
  dim3 grid(ceil_div(d->tokens, ATT_BM), d->heads, d->batch);
#define TOME_ATT_LAUNCH(DROP_)                                                                     \
  do {                                                                                             \
    static DynSmemOnce once;                                                                       \
    TOME_CUDA(ensure_dyn_smem(attn_fwd_kernel<DROP_>, ATT_SMEM, once));                            \
    launch_k(attn_fwd_kernel<DROP_>, grid, ATT_THREADS, ATT_SMEM, stream, tq, tk, tv, tqa, tka, p); \
  } while (0)
  if (p.keep_q) TOME_ATT_LAUNCH(true);
  else TOME_ATT_LAUNCH(false);
#undef TOME_ATT_LAUNCH
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
