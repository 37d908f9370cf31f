// K7: persistent warp-specialised tcgen05 GEMM with fused epilogues (projections, MLP, dgrad, wgrad).
//
//   C[M,N] = epilogue( A (M x K)  *  B (N x K)^T )       bf16 operands, fp32 accumulation in TMEM
//
// Either operand may be stored K-major (row = M/N index, K contiguous) or MN-major (row = K index, M/N
// contiguous), so the Flax parameter layout kernel[in, out] serves forward (B MN-major), dgrad (B K-major) and
// wgrad (A and B MN-major, reduction over the B*T rows) without any transposed copies in HBM.
//
// Replaces (reference, via XLA): DenseGeneral query/key/value tome_attention.py:145-164, out :287-299,
// MLPBlock Dense layers attention.py:32-37, and their autodiff.
//
// Roles (192 threads, 1 CTA per SM, persistent over a static round-robin tile schedule):
//   warp 0      TMA producer        global -> smem ring (STAGES x {A 16 KB, B BN*128 B}), 128B swizzle
//   warp 1      UMMA issuer         one thread issues tcgen05.mma 128 x BN x 16, accumulators double-buffered in TMEM
//   warps 2..9  epilogue            two warps per TMEM lane quadrant, each owning half of the tile's columns:
//                                   tcgen05.ld (thread = row, 32 columns at a time) -> bias/ReLU/gate/dropout/residual
//                                   -> 128-bit global stores; overlaps the next tile's main loop.  Everything the
//                                   epilogue reads from memory (bias tile -> shared memory, residual / gate rows ->
//                                   registers) is fetched BEFORE it waits for the accumulator, so no global-load
//                                   latency sits between the MMA's completion and the stores.
#include <string.h>

#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_EPI_WARPS = 8;   // 4 per TMEM lane quadrant x NSPLIT column groups
constexpr int GEMM_NSPLIT = GEMM_EPI_WARPS / 4;
static_assert(GEMM_EPI_WARPS % 4 == 0 && GEMM_NSPLIT >= 1 && GEMM_NSPLIT <= 4, "epilogue warps come in groups of four (one per lane quadrant)");
constexpr int GEMM_THREADS = 64 + 32 * GEMM_EPI_WARPS;


struct GemmEpilogue {
  void* c;             // [M, ldc] bf16 or fp32
  const float* bias;   // [N] or null
  const void* residual;  // bf16 [M, ldr] or null (added last)
  const void* gate;    // bf16 [M, ldg] or null:  acc *= (gate > 0 ? gate_scale : 0)   (ReLU / dropout backward)
  long long ldc, ldr, ldg;
  float gate_scale;
  int relu;
  int c_is_f32;
  DropoutCfg drop;     // applied after ReLU, before residual
  long long split_stride;  // elements between split-K partial outputs (c_is_f32 only)
  int accumulate;          // c_is_f32 only: C += result
  // one bit per output element, [M, ldw] u32 words of 32 columns: written by a ReLU epilogue (bit = output > 0), read by a
  // gate epilogue in place of the bf16 gate rows (16x less traffic for the ReLU backward)
  uint32_t* bits_out;
  const uint32_t* bits_in;
  long long ldw;
  float* colsum_part;      // [m_tiles, n] column sums of each 128-row tile of the bf16 output (specialised epilogues), or null
};

struct GemmShape {
  int m, n, k;
  int m_tiles, n_tiles, k_splits, kb_per_split, kb_total;
  int m_items;  // m_tiles, or ceil(m_tiles / 2) when CTA pairs share the B operand
  // Row-shifted A windows (tome_gemm_args_t.a_row_shift): K is a_groups groups of a_group_kb k-blocks; group g reads columns
  // [0, a_group_kb * 64) of A at rows m0 + a_shift[g] (TMA zero-fills rows outside the matrix).  a_groups == 0: plain GEMM.
  int a_groups, a_group_kb;
  int a_shift[TOME_GEMM_MAX_SHIFTS];
};

constexpr int GEMM_BRES_KB = 6;   // k-blocks (of 64) a resident B operand may have: K <= 384

// BRES (pair MMA only): the CTA's half of the B operand -- all of K, up to GEMM_BRES_KB k-blocks -- stays in shared memory for
// the whole kernel (a cluster works on ONE column tile), and the ring carries A alone.
template <int BN, bool PAIR = false, bool BRES = false>
struct GemmSmem {
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;
  // pair MMA: this CTA holds half of the tile's columns, as whole 64-column atoms (BN = 192: 96 columns in two atoms)
  static constexpr int B_ATOMS = PAIR ? (BN / 2 + 63) / 64 : BN / 64;
  static constexpr int B_BYTES = B_ATOMS * 64 * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = BRES ? A_BYTES : A_BYTES + B_BYTES;
  static constexpr int RES_BYTES = BRES ? GEMM_BRES_KB * B_BYTES : 0;
  static constexpr int STAGES = BRES ? 6                        // 6 x 16 KB of A (one whole K = 384 tile ahead) + 96 KB of B
                              : PAIR ? ((BN <= 128) ? 8 : 6)   // 8 x 24 KB, 6 x 32 KB (BN = 192 and 256)
                                     : (BN <= 128) ? 6 : (BN <= 192) ? 5 : 4;   // 6 x 32 KB, 5 x 40 KB, 4 x 48 KB
  static constexpr int STORE_BYTES = GEMM_EPI_WARPS * 2048;  // per epilogue warp: 32 rows x 64 B staging tile for TMA stores
  static constexpr int BAR_BYTES = 256 + 2 * BN * 4;  // barriers + double-buffered bias tile
  static constexpr int COL_BYTES = 2 * 4 * BN * 4;    // column sums: [accumulator stage][lane quadrant][BN] f32
  static constexpr int TOTAL = STAGES * STAGE_BYTES + RES_BYTES + STORE_BYTES + BAR_BYTES + COL_BYTES + 1024;  // +1024: manual 1 KB alignment
  static_assert(TOTAL <= 232448, "shared memory per CTA");
};

// MC: clusters of two CTAs work on vertically adjacent tiles (same n_blk); each CTA fetches half of the shared B tile
// and TMA-multicasts it into both CTAs, halving the L2 -> SM traffic of B (the K = C = 384 projections are bound by
// that traffic, not by the tensor pipe).  A stage is reusable once BOTH CTAs' MMAs have drained it.
// EPI < 0: every epilogue option is a run-time flag (any combination, fp32 or bf16 output, split-K).
// EPI >= 0: bit set of EPI_* -- the options are compile-time, the output is bf16 through TMA stores, and the inner loops
// carry no flag tests or per-8-column edge tests.  The stack's own GEMMs all take one of these paths.
constexpr int EPI_GENERIC = -1, EPI_BIAS = 1, EPI_RELU = 2, EPI_GATE = 4, EPI_DROP = 8, EPI_RESID = 16;

template <int BN, bool A_MN, bool B_MN, int MC, int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                 const __grid_constant__ CUtensorMap tma_c, const GemmShape s, const GemmEpilogue e) {
  constexpr bool PAIR = MC >= 2;   // one 256-row cta_group::2 MMA per cluster pair (MC == 1: two 128-row MMAs sharing a multicast B)
  constexpr bool BRES = MC == 3;   // ... with the B operand resident in shared memory (K <= 384)
  using L = GemmSmem<BN, PAIR, BRES>;
  constexpr int STAGES = L::STAGES;
  constexpr uint32_t TMEM_COLS = BN <= 64 ? 128 : BN <= 128 ? 256 : 512;  // two accumulator stages of BN columns
  static_assert(2 * BN <= 512 && BN % 64 == 0, "two BN-column accumulators must fit the 512 TMEM columns");

  extern __shared__ uint8_t smem_raw[];
  // 1 KB alignment by pointer arithmetic on the __shared__ array itself, so the epilogue's accesses stay LDS/STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* s_bres = smem + STAGES * L::STAGE_BYTES;   // resident B: k-block kb at kb * B_BYTES (BRES only)
  uint8_t* s_store = s_bres + L::RES_BYTES;           // 1 KB aligned (stage sizes are multiples of 1 KB)
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_store + L::STORE_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* tmem_full = empty_bar + STAGES;
  uint64_t* tmem_empty = tmem_full + 2;
  uint64_t* bres_full = tmem_empty + 2;                // BRES: the resident B operand has landed (both CTAs', at the leader)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bres_full + 1);
  float* s_bias = reinterpret_cast<float*>(s_store + L::STORE_BYTES + 256);  // [2][BN]
  float* s_col = s_bias + 2 * BN;                                             // [2][4][BN]

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t crank = MC ? cluster_ctarank() : 0u;
  const bool leader = crank == 0;
  // Work items (tile, or vertical tile pair), dealt round-robin to the CTAs / clusters.  BRES: cluster c keeps column tile
  // c % n_tiles and walks the row-tile pairs c / n_tiles, + clusters / n_tiles, ... (the host launches a multiple of n_tiles
  // clusters), so the n_tiles clusters working on one row-tile pair read its A tile at the same time (one HBM read, L2 hits
  // for the rest); an item is then just the row-tile pair.
  const int bres_groups = BRES ? (int)(gridDim.x >> 1) / s.n_tiles : 1;
  const int bres_nblk = BRES ? (int)(blockIdx.x >> 1) % s.n_tiles : 0;
  const int num_tiles = BRES ? s.m_items : s.m_items * s.n_tiles * s.k_splits;
  const int first_item = BRES ? (int)(blockIdx.x >> 1) / s.n_tiles : MC ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int item_step = BRES ? bres_groups : MC ? (int)(gridDim.x >> 1) : (int)gridDim.x;
#define TOME_ITEM_NBLK(tile) (BRES ? bres_nblk : ((tile) / s.k_splits) % s.n_tiles)
#define TOME_ITEM_MROW(tile) (BRES ? (tile) : (tile) / (s.k_splits * s.n_tiles))

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    if (!e.c_is_f32) tma_prefetch_desc(&tma_c);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], MC == 1 ? 2 : 1);   // MC == 1: both CTAs' MMAs drain a multicast stage; pair: one commit
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], PAIR ? 2 * GEMM_EPI_WARPS : GEMM_EPI_WARPS);  // one arrive per epilogue warp (pair: of both CTAs, at the leader)
    }
    mbar_init(bres_full, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    if constexpr (PAIR) tmem_alloc2(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if (MC) cluster_sync_all();  // the peer's barriers exist before anything is multicast at them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================================================================= TMA producer
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      if constexpr (BRES) {   // this CTA's half of the column tile, every k-block, once
        constexpr uint32_t kResTx = 2 * (B_MN ? L::B_BYTES : (BN / 2) * GEMM_BK * 2);
        const uint32_t rb = map_to_cta(bres_full, 0);
        if (leader) mbar_expect_tx(bres_full, kResTx * (uint32_t)s.kb_total);
        const int nh = bres_nblk * BN + (int)crank * (BN / 2);
        for (int kb = 0; kb < s.kb_total; ++kb) {
          uint8_t* sb = s_bres + kb * L::B_BYTES;
          if (!B_MN) {
            tma_load_2d_pair(sb, &tma_b, rb, kb * GEMM_BK, nh);
          } else {
#pragma unroll
            for (int j = 0; j < L::B_ATOMS; ++j) tma_load_2d_pair(sb + j * 8192, &tma_b, rb, nh + 64 * j, kb * GEMM_BK);
          }
        }
      }
      for (int tile = first_item; tile < num_tiles; tile += item_step) {
        const int split = BRES ? 0 : tile % s.k_splits;
        const int n_blk = TOME_ITEM_NBLK(tile);
        const int m_blk = TOME_ITEM_MROW(tile) * (MC ? 2 : 1) + (int)crank;
        const int m0 = m_blk * GEMM_BM, n0 = n_blk * BN;
        const int kb0 = split * s.kb_per_split;
        const int kb1 = min(kb0 + s.kb_per_split, s.kb_total);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          uint8_t* sa = smem + stage * L::STAGE_BYTES;
          uint8_t* sb = sa + L::A_BYTES;
          const int k0 = kb * GEMM_BK;
          int ka = k0, ma = m0;   // coordinates of the A tile (K-major A): shifted windows re-read the same columns at other rows
          if (s.a_groups) {
            const int g = kb / s.a_group_kb;
            ka = (kb - g * s.a_group_kb) * GEMM_BK;
            ma = m0 + s.a_shift[g];
          }
          if constexpr (BRES) {   // the ring carries A alone
            const uint32_t fb = map_to_cta(&full_bar[stage], 0);
            if (leader) mbar_expect_tx(&full_bar[stage], 2 * L::A_BYTES);
            if (!A_MN) tma_load_2d_pair(sa, &tma_a, fb, ka, ma);
            else tma_load_2d_pair(sa, &tma_a, fb, k0, m0);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
            continue;
          }
          if constexpr (PAIR) {
            // both CTAs' loads are counted on the LEADER's barrier: its MMA thread is the only consumer
            const uint32_t fb = map_to_cta(&full_bar[stage], 0);
            // bytes both CTAs' boxes deliver (a K-major half of BN = 192 is one 96-row box: 12 KB of the 16 KB slot)
            constexpr uint32_t kPairTx = 2 * (L::A_BYTES + (B_MN ? L::B_BYTES : (BN / 2) * GEMM_BK * 2));
            if (leader) mbar_expect_tx(&full_bar[stage], kPairTx);
            if (!A_MN) {
              tma_load_2d_pair(sa, &tma_a, fb, ka, ma);
            } else {
#pragma unroll
              for (int j = 0; j < GEMM_BM / 64; ++j) tma_load_2d_pair(sa + j * 8192, &tma_a, fb, m0 + 64 * j, k0);
            }
            const int nh = n0 + (int)crank * (BN / 2);   // this CTA's half of the tile's columns
            if (!B_MN) {
              tma_load_2d_pair(sb, &tma_b, fb, k0, nh);  // box {64 k, BN/2 n}
            } else {
#pragma unroll
              for (int j = 0; j < L::B_ATOMS; ++j) tma_load_2d_pair(sb + j * 8192, &tma_b, fb, nh + 64 * j, k0);   // BN = 192: the second atom is half used
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
            continue;
          }
          mbar_expect_tx(&full_bar[stage], L::STAGE_BYTES);
          if (!A_MN) {
            tma_load_2d(sa, &tma_a, &full_bar[stage], ka, ma);  // box {64 k, 128 m}
          } else {
#pragma unroll
            for (int j = 0; j < GEMM_BM / 64; ++j)  // box {64 m, 64 k} per 64-wide M atom
              tma_load_2d(sa + j * 8192, &tma_a, &full_bar[stage], m0 + 64 * j, k0);
          }
          if (!MC) {
            if (!B_MN) {
              tma_load_2d(sb, &tma_b, &full_bar[stage], k0, n0);  // box {64 k, BN n}
            } else {
#pragma unroll
              for (int j = 0; j < BN / 64; ++j) tma_load_2d(sb + j * 8192, &tma_b, &full_bar[stage], n0 + 64 * j, k0);
            }
          } else {  // this CTA's share of B, multicast to both CTAs of the pair
            if (!B_MN) {
              tma_load_2d_mc(sb + crank * (BN / 2) * 128, &tma_b, &full_bar[stage], k0, n0 + (int)crank * (BN / 2), (uint16_t)3);  // box {64 k, BN/2 n}
            } else {
#pragma unroll
              for (int j = 0; j < BN / 64; ++j)
                if ((j & 1) == (int)crank) tma_load_2d_mc(sb + j * 8192, &tma_b, &full_bar[stage], n0 + 64 * j, k0, (uint16_t)3);
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================================================= UMMA issuer
    if (lane == 0 && (!PAIR || leader)) {
      constexpr uint32_t idesc = make_idesc_bf16(PAIR ? 2 * GEMM_BM : GEMM_BM, BN, A_MN, B_MN);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      if constexpr (BRES) {
        mbar_wait(bres_full, 0);
        tc_fence_after();
      }
      for (int tile = first_item; tile < num_tiles; tile += item_step) {
        const int split = BRES ? 0 : tile % s.k_splits;
        const int kb0 = split * s.kb_per_split;
        const int kb1 = min(kb0 + s.kb_per_split, s.kb_total);
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * L::STAGE_BYTES);
          const uint32_t sb = BRES ? smem_u32(s_bres + kb * L::B_BYTES) : sa + L::A_BYTES;
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            const uint64_t da = A_MN ? make_smem_desc(sa + k * 2048, 8192, 1024) : make_smem_desc(sa + k * 32, 16, 1024);
            const uint64_t db = B_MN ? make_smem_desc(sb + k * 2048, 8192, 1024) : make_smem_desc(sb + k * 32, 16, 1024);
            if constexpr (PAIR) umma2_bf16(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
            else umma_bf16(d_tmem, da, db, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          if constexpr (PAIR) umma2_commit_mc(&empty_bar[stage], (uint16_t)3);   // both producers may refill their halves
          else if (MC) umma_commit_mc(&empty_bar[stage], (uint16_t)3);  // both CTAs' producers may refill this stage
          else umma_commit(&empty_bar[stage]);                     // smem slot reusable once these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if constexpr (PAIR) umma2_commit_mc(&tmem_full[acc], (uint16_t)3);  // both CTAs' epilogues read their 128 rows
        else umma_commit(&tmem_full[acc]);  // accumulator complete -> epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ================================================================= epilogue (warps 2..9)
    // the tile's BN / 32 column chunks are dealt round-robin to the GEMM_NSPLIT warps of a lane quadrant: warp `part` owns
    // chunks part, part + NSPLIT, ... (chunk index = column / 32 inside the tile)
    constexpr int NCHUNKS = BN / 32;
    constexpr int NCH = (NCHUNKS + GEMM_NSPLIT - 1) / GEMM_NSPLIT;   // most chunks one warp owns
    const int ew = warp - 2;
    const int quad = warp & 3;                   // TMEM lane quadrant this warp may access
    const int part = ew >> 2;                    // which column group of the tile
#define TOME_CHUNK(c) (part + (c) * GEMM_NSPLIT)
#define TOME_CHUNK_OK(c) (NCHUNKS % GEMM_NSPLIT == 0 || TOME_CHUNK(c) < NCHUNKS)
    const int row_in_tile = quad * 32 + lane;
    const int etid = threadIdx.x - 64;           // 0..255
    const __nv_bfloat16* resid = reinterpret_cast<const __nv_bfloat16*>(e.residual);
    const __nv_bfloat16* gate = reinterpret_cast<const __nv_bfloat16*>(e.gate);
    int acc = 0;
    uint32_t acc_phase = 0;
    if constexpr (EPI >= 0) {
      // ============================================================= specialised epilogues (bf16 out, k_splits == 1)
      constexpr bool kBias = (EPI & EPI_BIAS) != 0, kRelu = (EPI & EPI_RELU) != 0, kGate = (EPI & EPI_GATE) != 0,
                     kDrop = (EPI & EPI_DROP) != 0, kResid = (EPI & EPI_RESID) != 0;
      static_assert(!(kGate && kResid) && !(kGate && kDrop), "gate is the backward of relu/dropout: it never meets them");
      const bool drop_on = kDrop && e.drop.thresh16 != 0;   // warp-uniform: rate 0 (parity / eval) skips the RNG
      const uint32_t thr32 = e.drop.thresh16 << 16;
      const float2 gs2 = make_float2(e.gate_scale, e.gate_scale);
      for (int tile = first_item; tile < num_tiles; tile += item_step) {
        const int n_blk = TOME_ITEM_NBLK(tile);   // k_splits == 1 here
        const int m_blk = TOME_ITEM_MROW(tile) * (MC ? 2 : 1) + (int)crank;
        const long long row = (long long)m_blk * GEMM_BM + row_in_tile;
        const int n0 = n_blk * BN;
        const bool row_ok = row < s.m;
        // ---- everything the epilogue reads from memory is fetched while the tensor core still works on this tile
        if (kBias && etid < BN) s_bias[acc * BN + etid] = (n0 + etid < s.n) ? __ldg(e.bias + n0 + etid) : 0.f;
        uint4 pre[kResid ? NCH : 1][4];
        uint32_t gw[kGate ? NCH : 1];
        if constexpr (kGate) {   // the gate arrives as one bit per element (a bf16 gate tensor takes the generic epilogue)
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            const int col = n0 + TOME_CHUNK(c) * 32;
            gw[c] = (TOME_CHUNK_OK(c) && row_ok && col < s.n) ? __ldg(e.bits_in + row * e.ldw + (col >> 5)) : 0u;
          }
        }
        if constexpr (kResid) {
#pragma unroll
          for (int c = 0; c < NCH; ++c)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int col = n0 + TOME_CHUNK(c) * 32 + i * 8;
              pre[c][i] = (TOME_CHUNK_OK(c) && row_ok && col < s.n) ? __ldg(reinterpret_cast<const uint4*>(resid + row * e.ldr + col)) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
        if (kBias) asm volatile("bar.sync 1, %0;" ::"r"(32 * GEMM_EPI_WARPS) : "memory");  // bias tile visible to all epilogue warps
        mbar_wait(&tmem_full[acc], acc_phase);
        tc_fence_after();
        const uint32_t t_addr = tmem_base + acc * BN + ((uint32_t)(quad * 32) << 16);
        // the TMEM read of chunk c + 1 is in flight while chunk c is processed (two register sets, compile-time ping-pong)
        float va[32], vb[32];
        tmem_ld_f32x32(t_addr + TOME_CHUNK(0) * 32, va);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          if (!TOME_CHUNK_OK(c)) break;   // warp-uniform: this warp owns one chunk fewer
          float (&v)[32] = (c & 1) ? vb : va;
          tmem_ld_wait();
          if (c + 1 < NCH && TOME_CHUNK_OK(c + 1)) tmem_ld_f32x32(t_addr + TOME_CHUNK(c + 1) * 32, (c & 1) ? va : vb);
          const int col = n0 + TOME_CHUNK(c) * 32;
          if constexpr (kBias) {
            const float4* b4p = reinterpret_cast<const float4*>(s_bias + acc * BN + TOME_CHUNK(c) * 32);
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
              const float4 b4 = b4p[i / 4];
              const float2 t0 = __fadd2_rn(make_float2(v[i], v[i + 1]), make_float2(b4.x, b4.y));
              const float2 t1 = __fadd2_rn(make_float2(v[i + 2], v[i + 3]), make_float2(b4.z, b4.w));
              v[i] = t0.x; v[i + 1] = t0.y; v[i + 2] = t1.x; v[i + 3] = t1.y;
            }
          }
          if constexpr (kGate) {  // acc *= (bit ? gate_scale : 0)
            const uint32_t w = gw[c];
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              const float2 t = __fmul2_rn(make_float2(v[i], v[i + 1]), gs2);
              v[i] = ((w >> i) & 1u) ? t.x : 0.f;
              v[i + 1] = ((w >> (i + 1)) & 1u) ? t.y : 0.f;
            }
          }
          if (drop_on) {
            DropStream ds = drop_stream(e.drop, (uint32_t)row, (uint32_t)col >> 5);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float mult = ds.next() >= thr32 ? e.drop.inv_keep : 0.f;
              if constexpr (kResid) {
                const uint32_t w = reinterpret_cast<const uint32_t*>(&pre[c][i / 8])[(i / 2) & 3];
                v[i] = fmaf(v[i], mult, (i & 1) ? bf16_hi(w) : bf16_lo(w));
              } else {
                v[i] *= mult;
              }
            }
          } else if constexpr (kResid) {
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              const uint32_t w = reinterpret_cast<const uint32_t*>(&pre[c][i / 8])[(i / 2) & 3];
              const float2 t = __fadd2_rn(make_float2(v[i], v[i + 1]), make_float2(bf16_lo(w), bf16_hi(w)));
              v[i] = t.x; v[i + 1] = t.y;
            }
          }
          if constexpr (kRelu) {
            if (e.bits_out != nullptr) {  // the ReLU (and dropout) gate of this chunk, one bit per column, for the backward GEMM
              uint32_t word = 0u;
#pragma unroll
              for (int i = 0; i < 32; ++i) word |= (v[i] > 0.f) ? (1u << i) : 0u;
              if (row_ok && col < s.n) e.bits_out[row * e.ldw + (col >> 5)] = word;
            }
          }
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            pk[i] = pack_bf16(v[2 * i], v[2 * i + 1]);
            if constexpr (kRelu) {  // relu commutes with the (non-negative) dropout factor and with rounding: apply it packed
              __nv_bfloat162 h = *reinterpret_cast<__nv_bfloat162*>(&pk[i]);
              h = __hmax2(h, __floats2bfloat162_rn(0.f, 0.f));
              pk[i] = *reinterpret_cast<uint32_t*>(&h);
            }
          }
          // stage this warp's 32 rows x 32 columns in shared memory (64-byte swizzled rows) and hand the box to TMA,
          // which writes whole lines and clips rows >= M / columns >= N.  (Reading the tile back and storing it with
          // 128-bit LSU stores, 8 rows x 64 B per instruction, was measured slower: 108 vs 78 us for the stores of the
          // 133120 x 1536 output alone, 154 vs 142 us for the whole GEMM without CTA pairs.)
          uint8_t* stg = s_store + ew * 2048;
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // previous box has left smem
          __syncwarp();
#pragma unroll
          for (int ch = 0; ch < 4; ++ch)
            *reinterpret_cast<uint4*>(stg + lane * 64 + ((ch ^ ((lane >> 1) & 3)) << 4)) =
                make_uint4(pk[4 * ch], pk[4 * ch + 1], pk[4 * ch + 2], pk[4 * ch + 3]);
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            const int row0 = m_blk * GEMM_BM + quad * 32;
            if (col < s.n && row0 < s.m) {
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                           ::"l"(&tma_c), "r"(smem_u32(stg)), "r"(col), "r"(row0) : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
          if (e.colsum_part != nullptr) {
            // column sums of what was just staged (the bf16-rounded outputs, like a separate pass over C would read):
            // lane = (half h, column pair j) adds 16 rows; the halves walk rows of opposite parity (no bank conflict)
            const int j = lane & 15, h = lane >> 4;
            const int rlim = s.m - (m_blk * GEMM_BM + quad * 32);   // rows of this warp's slab that exist
            float2 sum = make_float2(0.f, 0.f);
            const uint8_t* sp = stg + (j & 3) * 4;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int r = h * 16 + (i ^ h);
              uint32_t w = *reinterpret_cast<const uint32_t*>(sp + r * 64 + (((j >> 2) ^ ((r >> 1) & 3)) << 4));
              if (r >= rlim) w = 0u;
              sum = __fadd2_rn(sum, make_float2(bf16_lo(w), bf16_hi(w)));
            }
            sum.x += __shfl_xor_sync(0xffffffffu, sum.x, 16);
            sum.y += __shfl_xor_sync(0xffffffffu, sum.y, 16);
            if (h == 0) *reinterpret_cast<float2*>(s_col + (acc * 4 + quad) * BN + TOME_CHUNK(c) * 32 + 2 * j) = sum;
          }
        }
        tc_fence_before();
        __syncwarp();
        if (e.colsum_part != nullptr) {   // CTA-uniform
          // The four lane quadrants' sums of this tile -> one row of partials, by the first epilogue warp; the other seven only
          // signal (bar.arrive) and go on to their next tile.  One barrier per accumulator stage: no warp can be two tiles
          // ahead of another (the MMA of tile i + 2 waits for every warp's release of tile i), and warp 2 releases its
          // accumulator only after it has read the sums, so a stage's slots are never rewritten under it.
          if (ew == 0) {
            asm volatile("bar.sync %0, %1;" ::"r"(2 + acc), "r"(32 * GEMM_EPI_WARPS) : "memory");
            if (m_blk < s.m_tiles) {
#pragma unroll
              for (int cidx = lane * 2; cidx < BN; cidx += 64) {
                if (n0 + cidx < s.n) {
                  const float* sc = s_col + acc * 4 * BN + cidx;
                  const float2 q0 = *reinterpret_cast<const float2*>(sc), q1 = *reinterpret_cast<const float2*>(sc + BN),
                               q2 = *reinterpret_cast<const float2*>(sc + 2 * BN), q3 = *reinterpret_cast<const float2*>(sc + 3 * BN);
                  *reinterpret_cast<float2*>(e.colsum_part + (long long)m_blk * s.n + n0 + cidx) =
                      make_float2((q0.x + q1.x) + (q2.x + q3.x), (q0.y + q1.y) + (q2.y + q3.y));
                }
              }
            }
            __syncwarp();
          } else {
            asm volatile("bar.arrive %0, %1;" ::"r"(2 + acc), "r"(32 * GEMM_EPI_WARPS) : "memory");
          }
        }
        if (lane == 0) {
          if constexpr (PAIR) mbar_arrive_cluster(map_to_cta(&tmem_empty[acc], 0));   // the leader's MMA thread waits for both CTAs
          else mbar_arrive(&tmem_empty[acc]);
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    } else
    for (int tile = first_item; tile < num_tiles; tile += item_step) {
      const int split = tile % s.k_splits;
      const int n_blk = (tile / s.k_splits) % s.n_tiles;
      const int m_blk = (tile / (s.k_splits * s.n_tiles)) * (MC ? 2 : 1) + (int)crank;
      const long long row = (long long)m_blk * GEMM_BM + row_in_tile;
      const int n0 = n_blk * BN;
      const bool row_ok = row < s.m;
      // ---- prefetch everything the epilogue reads, while the tensor core is still working on this tile
      if (e.bias && etid < BN) s_bias[acc * BN + etid] = (n0 + etid < s.n) ? __ldg(e.bias + n0 + etid) : 0.f;
      // one prefetch array serves the residual or, when there is no residual, the gate (the library's own callers
      // never pass both; if both are given the gate is read inside the loop)
      const __nv_bfloat16* pre_src = resid ? resid : gate;
      const long long pre_ld = resid ? e.ldr : e.ldg;
      uint4 pre[NCH][4];
#pragma unroll
      for (int c = 0; c < NCH; ++c)
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int col = n0 + TOME_CHUNK(c) * 32 + i * 8;
          pre[c][i] = (TOME_CHUNK_OK(c) && pre_src && row_ok && col < s.n) ? __ldg(reinterpret_cast<const uint4*>(pre_src + row * pre_ld + col))
                                                                            : make_uint4(0u, 0u, 0u, 0u);
        }
      asm volatile("bar.sync 1, %0;" ::"r"(32 * GEMM_EPI_WARPS) : "memory");  // bias tile visible to all epilogue warps
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t t_addr = tmem_base + acc * BN + ((uint32_t)(quad * 32) << 16);
#pragma unroll
      for (int c = 0; c < NCH; ++c) {
        if (!TOME_CHUNK_OK(c)) break;   // warp-uniform
        uint32_t v[32];
        tmem_ld_x32(t_addr + TOME_CHUNK(c) * 32, v);
        tmem_ld_wait();
        const int col = n0 + TOME_CHUNK(c) * 32;
        const bool active = row_ok && col < s.n;  // rows / columns past the edge are computed but never stored
        float acc_f[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) acc_f[i] = __uint_as_float(v[i]);
        const int ncols = min(32, s.n - col);  // multiple of 8 (host checks n % 8 == 0); <= 0 past the edge
        if (e.bias) {
          const float4* b4p = reinterpret_cast<const float4*>(s_bias + acc * BN + TOME_CHUNK(c) * 32);
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            const float4 b4 = b4p[i / 4];
            acc_f[i] += b4.x; acc_f[i + 1] += b4.y; acc_f[i + 2] += b4.z; acc_f[i + 3] += b4.w;
          }
        }
        if (e.relu) {
#pragma unroll
          for (int i = 0; i < 32; ++i) acc_f[i] = fmaxf(acc_f[i], 0.f);
        }
        if (e.bits_in) {
          const uint32_t w = active ? __ldg(e.bits_in + row * e.ldw + (col >> 5)) : 0u;
#pragma unroll
          for (int i = 0; i < 32; ++i) acc_f[i] *= ((w >> i) & 1u) ? e.gate_scale : 0.f;
        } else if (gate) {
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            uint4 gq = pre[c][i / 8];
            if (resid && active && i < ncols) gq = __ldg(reinterpret_cast<const uint4*>(gate + row * e.ldg + col + i));
            const uint32_t w[4] = {gq.x, gq.y, gq.z, gq.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              acc_f[i + 2 * j] *= (bf16_lo(w[j]) > 0.f) ? e.gate_scale : 0.f;
              acc_f[i + 2 * j + 1] *= (bf16_hi(w[j]) > 0.f) ? e.gate_scale : 0.f;
            }
          }
        }
        if (e.drop.thresh16 && active) {
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            if (i < ncols) {
              const uint32_t keep = dropout_keep8(e.drop, (uint32_t)row, (uint32_t)(col + i));
#pragma unroll
              for (int j = 0; j < 8; ++j) acc_f[i + j] = ((keep >> j) & 1u) ? acc_f[i + j] * e.drop.inv_keep : 0.f;
            }
          }
        }
        if (e.bits_out && active) {  // after ReLU and dropout: bit = the element survives (columns past N read as 0)
          uint32_t word = 0u;
#pragma unroll
          for (int i = 0; i < 32; ++i) word |= (i < ncols && acc_f[i] > 0.f) ? (1u << i) : 0u;
          e.bits_out[row * e.ldw + (col >> 5)] = word;
        }
        if (resid) {
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            const uint32_t w[4] = {pre[c][i / 8].x, pre[c][i / 8].y, pre[c][i / 8].z, pre[c][i / 8].w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              acc_f[i + 2 * j] += bf16_lo(w[j]);
              acc_f[i + 2 * j + 1] += bf16_hi(w[j]);
            }
          }
        }
        if (e.c_is_f32) {
          if (active) {
            float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(e.c) + (long long)split * e.split_stride + row * e.ldc + col);
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              if (i < ncols) {
                float4 ov = make_float4(acc_f[i], acc_f[i + 1], acc_f[i + 2], acc_f[i + 3]);
                if (e.accumulate) {
                  const float4 old = o[i / 4];
                  ov.x += old.x; ov.y += old.y; ov.z += old.z; ov.w += old.w;
                }
                o[i / 4] = ov;
              }
          }
        } else {
          // bf16: stage this warp's 32 rows x 32 columns in shared memory (64-byte swizzled rows) and hand the box to
          // TMA, which writes whole lines and clips rows >= M / columns >= N.
          uint8_t* stg = s_store + ew * 2048;
          if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // previous box has left smem
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 32; i += 8) {
            const int chunk = i / 8;
            *reinterpret_cast<uint4*>(stg + lane * 64 + ((chunk ^ ((lane >> 1) & 3)) << 4)) =
                make_uint4(pack_bf16(acc_f[i], acc_f[i + 1]), pack_bf16(acc_f[i + 2], acc_f[i + 3]),
                           pack_bf16(acc_f[i + 4], acc_f[i + 5]), pack_bf16(acc_f[i + 6], acc_f[i + 7]));
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            const int row0 = m_blk * GEMM_BM + quad * 32;
            if (col < s.n && row0 < s.m) {
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                           ::"l"(&tma_c), "r"(smem_u32(stg)), "r"(col), "r"(row0) : "memory");
            }
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_cluster(map_to_cta(&tmem_empty[acc], 0));
        else mbar_arrive(&tmem_empty[acc]);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // all of this warp's TMA stores are complete
#undef TOME_CHUNK
#undef TOME_CHUNK_OK
  }
#undef TOME_ITEM_NBLK
#undef TOME_ITEM_MROW

  tc_fence_before();
  __syncthreads();
  if (MC) cluster_sync_all();  // the peer may still multicast into this CTA's smem / arrive on its barriers
  if (warp == 2) {
    tc_fence_after();
    if constexpr (PAIR) tmem_dealloc2(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// sum split-K partials: out[i] = sum_s part[s*stride + i]      (fp32, deterministic order)
__global__ void splitk_reduce_kernel(const float* __restrict__ part, float* __restrict__ out, long long n4,
                                     long long stride4, int splits, int accumulate) {
  const float4* p = reinterpret_cast<const float4*>(part);
  float4* o = reinterpret_cast<float4*>(out);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 a = p[i];
    for (int s = 1; s < splits; ++s) {
      const float4 b = p[i + s * stride4];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    if (accumulate) {
      const float4 b = o[i];
      a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    }
    o[i] = a;
  }
}

// SMs the persistent grid may occupy (0 = all).  The data-parallel trainer lowers it during backward so that the NCCL
// all-reduce kernels running beside it own their SMs: a persistent CTA that cannot be scheduled until a long collective
// kernel leaves its SM would hold back the whole GEMM (tiles are assigned statically).
static int g_gemm_sm_limit = 0;
static inline int gemm_sms() { return g_gemm_sm_limit > 0 && g_gemm_sm_limit < kNumSMs ? g_gemm_sm_limit : kNumSMs; }

// B-resident launches: groups of n_tiles clusters (one per column tile), as many groups as fit and have work
static inline int bres_clusters(int n_tiles, int m_items) {
  int groups = (gemm_sms() / 2) / n_tiles;
  if (groups > m_items) groups = m_items;
  return groups * n_tiles;
}

template <int BN, bool A_MN, bool B_MN, int MC, int EPI>
static int launch_gemm(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tc, const GemmShape& s, const GemmEpilogue& e,
                       cudaStream_t stream) {
  auto kern = gemm_bf16_kernel<BN, A_MN, B_MN, MC, EPI>;
  using SM = GemmSmem<BN, MC >= 2, MC == 3>;
  static DynSmemOnce once;  // per instantiation, per device
  TOME_CUDA(ensure_dyn_smem(kern, SM::TOTAL, once));
  const int items = s.m_items * s.n_tiles * s.k_splits;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = SM::TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  if (MC) {
    int clusters = items < gemm_sms() / 2 ? items : gemm_sms() / 2;
    if (MC == 3) clusters = bres_clusters(s.n_tiles, s.m_items);   // a multiple of the column tiles
    cfg.gridDim = dim3(2 * clusters);
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  } else {
    cfg.gridDim = dim3(items < gemm_sms() ? items : gemm_sms());
  }
  TOME_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, tc, s, e));
  return TOME_OK;
}

}  // namespace tome

using namespace tome;

static int pick_bn(int n) {  // least padded MMA work (tiles x width), then the wider tile
  const int w128 = ceil_div(n, 128) * 128, w192 = ceil_div(n, 192) * 192, w256 = ceil_div(n, 256) * 256;
  if (w256 <= w192 && w256 <= w128) return 256;
  if (w192 <= w128) return 192;
  return 128;
}

static int g_gemm_force_mode = -1, g_gemm_force_bn = 0;
// tuning aid: force the CTA mode (0 single, 1 multicast pairs, 2 pair MMA; -1 = automatic) and the tile width (0 = automatic)
extern "C" void tome_gemm_force_tile(int mode, int bn) { g_gemm_force_mode = mode; g_gemm_force_bn = bn; }

struct TileChoice { int bn, mode; };   // mode 0: one CTA per tile; 1: CTA pairs, multicast B; 2: CTA pairs, one 256-row MMA
static TileChoice pick_tile(const tome_gemm_args_t* a) {
  const int m_tiles = ceil_div(a->m, GEMM_BM);
  // CTA pairs: worth it unless an odd, small tile count would leave a large share of dummy tiles
  const bool pairs_ok = m_tiles >= 2 && (m_tiles % 2 == 0 || m_tiles >= 16);
  TileChoice t;
  t.bn = pick_bn(a->n);
  t.mode = pairs_ok ? 1 : 0;
  // The pair MMA halves each SM's B traffic (L2 -> shared memory and shared memory -> tensor core).  Measured on B200 over
  // every GEMM of an octo-small / octo-base layer with the stack's epilogues (scripts/sweep_gemm_tiles.py,
  // profiles/r02_gemm_tile_sweep.md): with the tile width below it is the fastest or within 2 % of the fastest mode at every
  // shape that can form pairs (octo-base: 1.46 - 1.56 PF/s against 1.31 - 1.41 for multicast pairs, above cuBLAS).  A pair
  // MMA narrower than 192 columns is not: 256 x 128 x 16 occupies the tensor pipe as long as 256 x 256 x 16 does.
  if (pairs_ok) {
    t.mode = 2;
    // activations x weights with a wide output: the 256-wide pair tile beats the exactly fitting 192 (qkv, N = 1152: 112 vs 121 us)
    if (t.bn == 192 && a->n >= 1024 && a->a_major == TOME_MAJOR_K) t.bn = 256;
    if (t.bn == 128) t.mode = 1;
  }
  // K <= 384 with a specialised epilogue: keep B in shared memory (mode 3; the caller checks the epilogue)
  // (with two column tiles the epilogue, not the operand stream, paces the kernel and the fixed column assignment only costs
  // balance: out projection 137216 x 384 x 384, 78 vs 76 us)
  if (t.mode == 2 && a->k <= GEMM_BRES_KB * GEMM_BK && a->a_major == TOME_MAJOR_K && ceil_div(a->n, t.bn) >= 3 &&
      ceil_div(a->n, t.bn) <= gemm_sms() / 2)
    t.mode = 3;
  if (g_gemm_force_bn == 128 || g_gemm_force_bn == 192 || g_gemm_force_bn == 256) t.bn = g_gemm_force_bn;
  if (g_gemm_force_mode == 0 || (g_gemm_force_mode > 0 && g_gemm_force_mode <= 2 && pairs_ok)) t.mode = g_gemm_force_mode;
  if (g_gemm_force_mode == 3 && pairs_ok && t.bn >= 192 && a->k <= GEMM_BRES_KB * GEMM_BK && a->a_major == TOME_MAJOR_K) t.mode = 3;
  return t;
}

static int pick_splits(const tome_gemm_args_t* a, int bn) {
  if (a->k_splits > 0) return a->k_splits;
  if (a->a_row_shift) return 1;
  if (a->c_dtype != TOME_F32 || a->ldc != a->n) return 1;  // split-K only for dense fp32 outputs (weight gradients)
  if (a->bias || a->residual || a->gate || a->gate_bits || a->relu || a->dropout_rate > 0.f) return 1;
  const int tiles = ceil_div(a->m, GEMM_BM) * ceil_div(a->n, bn);
  const int kb = ceil_div(a->k, GEMM_BK);
  int s = kNumSMs / (tiles > 0 ? tiles : 1);
  if (s < 1) s = 1;
  if (s > kb / 8) s = kb / 8 > 0 ? kb / 8 : 1;  // keep >= 8 k-blocks per split
  if (s > 64) s = 64;
  return s;
}

extern "C" int tome_gemm_set_sm_limit(int sms) {
  clear_error();
  TOME_CHECK(sms >= 0, TOME_ERR_INVALID, "gemm_set_sm_limit: sms must be >= 0 (0 = all)");
  g_gemm_sm_limit = sms >= 2 || sms == 0 ? sms : 2;
  return TOME_OK;
}

extern "C" int tome_num_sms(void) { return kNumSMs; }

extern "C" size_t tome_gemm_workspace_bytes(const tome_gemm_args_t* a) {
  if (!a) return 0;
  const int splits = pick_splits(a, pick_tile(a).bn);
  if (splits <= 1) return 0;
  return (size_t)splits * (size_t)a->m * (size_t)a->ldc * sizeof(float);
}

extern "C" int tome_gemm_bf16(const tome_gemm_args_t* a, void* workspace, size_t workspace_bytes, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(a != nullptr, TOME_ERR_INVALID, "gemm: null args");
  TOME_CHECK(a->m > 0 && a->n > 0 && a->k > 0, TOME_ERR_INVALID, "gemm: m,n,k must be positive (%d,%d,%d)", a->m, a->n, a->k);
  TOME_CHECK(a->a && a->b && a->c, TOME_ERR_INVALID, "gemm: null operand pointer");
  TOME_CHECK(a->n % 8 == 0, TOME_ERR_INVALID, "gemm: n (%d) must be a multiple of 8", a->n);
  TOME_CHECK(a->lda % 8 == 0 && a->ldb % 8 == 0, TOME_ERR_INVALID, "gemm: lda/ldb must be multiples of 8 elements (16 B)");
  TOME_CHECK(a->c_dtype == TOME_BF16 || a->c_dtype == TOME_F32, TOME_ERR_INVALID, "gemm: c_dtype must be bf16 or f32");
  TOME_CHECK(a->ldc % (a->c_dtype == TOME_F32 ? 4 : 8) == 0, TOME_ERR_INVALID, "gemm: ldc must keep rows 16-byte aligned");
  TOME_CHECK(!a->residual || a->ldr % 8 == 0, TOME_ERR_INVALID, "gemm: ldr must be a multiple of 8");
  TOME_CHECK(!a->gate || a->ldg % 8 == 0, TOME_ERR_INVALID, "gemm: ldg must be a multiple of 8");
  TOME_CHECK(!(a->gate && a->gate_bits), TOME_ERR_INVALID, "gemm: pass the gate as bf16 rows or as bits, not both");
  TOME_CHECK(!(a->gate_bits || a->relu_bits_out) || a->ld_bits * 32 >= a->n, TOME_ERR_INVALID,
             "gemm: ld_bits (%lld words) does not cover n = %d columns", a->ld_bits, a->n);
  TOME_CHECK(!a->relu_bits_out || a->relu, TOME_ERR_INVALID, "gemm: relu_bits_out needs the ReLU epilogue");
  TOME_CHECK(a->dropout_rate >= 0.f && a->dropout_rate < 1.f, TOME_ERR_INVALID, "gemm: dropout_rate must be in [0,1)");

  const TileChoice tile = pick_tile(a);
  const int bn = tile.bn;
  int mode = tile.mode;
  const bool mc = mode != 0;
  GemmShape s;
  s.m = a->m; s.n = a->n; s.k = a->k;
  s.m_tiles = ceil_div(a->m, GEMM_BM);
  s.n_tiles = ceil_div(a->n, bn);
  s.kb_total = ceil_div(a->k, GEMM_BK);
  s.k_splits = pick_splits(a, bn);
  s.kb_per_split = ceil_div(s.kb_total, s.k_splits);
  s.k_splits = ceil_div(s.kb_total, s.kb_per_split);  // drop empty splits
  s.m_items = mc ? ceil_div(s.m_tiles, 2) : s.m_tiles;
  s.a_groups = 0; s.a_group_kb = 1;
  if (a->a_row_shift) {
    TOME_CHECK(a->a_shift_groups >= 1 && a->a_shift_groups <= TOME_GEMM_MAX_SHIFTS && a->k % a->a_shift_groups == 0 &&
               (a->k / a->a_shift_groups) % GEMM_BK == 0, TOME_ERR_INVALID,
               "gemm: a_row_shift needs 1 <= a_shift_groups <= %d and k / a_shift_groups a multiple of %d", TOME_GEMM_MAX_SHIFTS, GEMM_BK);
    TOME_CHECK(a->a_major == TOME_MAJOR_K && s.k_splits == 1, TOME_ERR_INVALID, "gemm: a_row_shift needs a K-major A and no split-K");
    s.a_groups = a->a_shift_groups;
    s.a_group_kb = a->k / a->a_shift_groups / GEMM_BK;
    for (int g = 0; g < a->a_shift_groups; ++g) s.a_shift[g] = a->a_row_shift[g];
  }

  GemmEpilogue e;
  e.c = a->c; e.bias = a->bias; e.residual = a->residual; e.gate = a->gate;
  e.bits_out = reinterpret_cast<uint32_t*>(a->relu_bits_out); e.bits_in = reinterpret_cast<const uint32_t*>(a->gate_bits);
  e.ldw = a->ld_bits;
  e.colsum_part = a->colsum_partial;
  e.ldc = a->ldc; e.ldr = a->ldr; e.ldg = a->ldg;
  e.gate_scale = a->gate_scale; e.relu = a->relu; e.c_is_f32 = (a->c_dtype == TOME_F32);
  e.drop = make_dropout(a->dropout_rate, a->dropout_seed, a->dropout_site);
  e.split_stride = 0;
  e.accumulate = a->accumulate;
  TOME_CHECK(!a->accumulate || e.c_is_f32, TOME_ERR_INVALID, "gemm: accumulate requires an fp32 output");
  if (s.k_splits > 1) {
    TOME_CHECK(e.c_is_f32, TOME_ERR_INVALID, "gemm: split-K requires an fp32 output");
    TOME_CHECK(a->ldc == a->n, TOME_ERR_INVALID, "gemm: split-K requires a dense output (ldc == n)");
    TOME_CHECK(!a->bias && !a->residual && !a->gate && !a->gate_bits && !a->relu && e.drop.thresh16 == 0, TOME_ERR_INVALID,
               "gemm: split-K supports a plain epilogue only");
    const size_t need = (size_t)s.k_splits * (size_t)a->m * (size_t)a->ldc * sizeof(float);
    TOME_CHECK(workspace && workspace_bytes >= need, TOME_ERR_INVALID, "gemm: split-K workspace too small (%zu < %zu)",
               workspace_bytes, need);
    e.c = workspace;
    e.split_stride = (long long)a->m * a->ldc;
    e.accumulate = 0;  // partials are plain; the reduce kernel adds into C
  }

  CUtensorMap ta, tb;
  int rc;
  if (a->a_major == TOME_MAJOR_K) rc = make_tmap_2d_bf16(&ta, a->a, a->m, s.a_groups ? a->k / s.a_groups : a->k, a->lda, GEMM_BM);
  else rc = make_tmap_2d_bf16(&ta, a->a, a->k, a->m, a->lda, GEMM_BK);
  if (rc) return rc;
  if (a->b_major == TOME_MAJOR_K) rc = make_tmap_2d_bf16(&tb, a->b, a->n, a->k, a->ldb, mc ? bn / 2 : bn);
  else rc = make_tmap_2d_bf16(&tb, a->b, a->k, a->n, a->ldb, GEMM_BK);
  if (rc) return rc;

  CUtensorMap tc;
  memset(&tc, 0, sizeof(tc));
  if (!e.c_is_f32) {  // bf16 outputs leave through TMA stores: box {32 columns, 32 rows}, 64-byte swizzle
    rc = make_tmap_2d_bf16_store32(&tc, a->c, a->m, a->n, a->ldc);
    if (rc) return rc;
  }
  const bool amn = a->a_major == TOME_MAJOR_MN, bmn = a->b_major == TOME_MAJOR_MN;
  ProfScope prof(PROF_GEMM, 2.0 * a->m * (double)a->n * a->k, s.k_splits > 1 ? 2 : 1, stream);
  // which epilogue: a compile-time specialisation when the combination is one the stack uses, else the generic one
  int epi = EPI_GENERIC;
  if (!e.c_is_f32 && s.k_splits == 1 && !a->accumulate) {
    const int flags = (a->bias ? EPI_BIAS : 0) | (a->relu ? EPI_RELU : 0) | ((a->gate || a->gate_bits) ? EPI_GATE : 0) |
                      (e.drop.thresh16 ? EPI_DROP : 0) | (a->residual ? EPI_RESID : 0);
    if (!amn && bmn) {  // forward layers: A = activations (K-major), B = Flax kernel [in, out] (MN-major)
      if (flags == EPI_BIAS) epi = EPI_BIAS;
      else if (flags == (EPI_BIAS | EPI_RESID) || flags == (EPI_BIAS | EPI_DROP | EPI_RESID)) epi = EPI_BIAS | EPI_DROP | EPI_RESID;
      else if (flags == (EPI_BIAS | EPI_RELU) || flags == (EPI_BIAS | EPI_RELU | EPI_DROP)) epi = EPI_BIAS | EPI_RELU | EPI_DROP;
    } else if (!amn && !bmn) {  // data gradients: B = the same kernel read K-major
      if (flags == 0) epi = 0;
      else if (flags == EPI_GATE && a->gate_bits) epi = EPI_GATE;   // bf16 gate rows: generic epilogue
    }
  }
  if (mode == 3 && (epi == EPI_GENERIC || bn == 128)) mode = 2;   // the resident-B kernels exist for the specialised epilogues only
  TOME_CHECK(!a->colsum_partial || epi != EPI_GENERIC, TOME_ERR_INVALID,
             "gemm: colsum_partial needs a bf16 output without split-K and one of the stack's epilogues (plain or gated data "
             "gradient, bias / bias+ReLU(+dropout) / bias(+dropout)+residual forward)");
#define TOME_GEMM_MODE(BN_, AMN_, BMN_, EPI_)                                                        \
  do {                                                                                              \
    if (mode == 3) {                                                                                \
      if constexpr (!(AMN_) && (EPI_) >= 0 && (BN_) >= 192) rc = launch_gemm<BN_, AMN_, BMN_, 3, EPI_>(ta, tb, tc, s, e, stream); \
      else rc = TOME_ERR_INVALID;                                                                   \
    } else if (mode == 2) rc = launch_gemm<BN_, AMN_, BMN_, 2, EPI_>(ta, tb, tc, s, e, stream);     \
    else if (mode == 1) rc = launch_gemm<BN_, AMN_, BMN_, 1, EPI_>(ta, tb, tc, s, e, stream);     \
    else rc = launch_gemm<BN_, AMN_, BMN_, 0, EPI_>(ta, tb, tc, s, e, stream);                      \
  } while (0)
#define TOME_GEMM_LAYOUTS(BN_, EPI_)                                                                \
  do {                                                                                              \
    if (!amn && !bmn) TOME_GEMM_MODE(BN_, false, false, EPI_);                                      \
    else if (!amn && bmn) TOME_GEMM_MODE(BN_, false, true, EPI_);                                   \
    else if (amn && !bmn) TOME_GEMM_MODE(BN_, true, false, EPI_);                                   \
    else TOME_GEMM_MODE(BN_, true, true, EPI_);                                                     \
  } while (0)
#define TOME_GEMM_FWD(BN_, EPI_) TOME_GEMM_MODE(BN_, false, true, EPI_)
#define TOME_GEMM_DGRAD(BN_, EPI_) TOME_GEMM_MODE(BN_, false, false, EPI_)
#define TOME_GEMM_DISPATCH(BN_)                                                                     \
  do {                                                                                              \
    switch (epi) {                                                                                  \
      case EPI_BIAS: TOME_GEMM_FWD(BN_, EPI_BIAS); break;                                           \
      case EPI_BIAS | EPI_DROP | EPI_RESID: TOME_GEMM_FWD(BN_, EPI_BIAS | EPI_DROP | EPI_RESID); break; \
      case EPI_BIAS | EPI_RELU | EPI_DROP: TOME_GEMM_FWD(BN_, EPI_BIAS | EPI_RELU | EPI_DROP); break; \
      case 0: TOME_GEMM_DGRAD(BN_, 0); break;                                                       \
      case EPI_GATE: TOME_GEMM_DGRAD(BN_, EPI_GATE); break;                                         \
      default: TOME_GEMM_LAYOUTS(BN_, EPI_GENERIC); break;                                          \
    }                                                                                               \
  } while (0)
  if (bn == 128) TOME_GEMM_DISPATCH(128);
  else if (bn == 192) TOME_GEMM_DISPATCH(192);
  else TOME_GEMM_DISPATCH(256);
#undef TOME_GEMM_MODE
#undef TOME_GEMM_LAYOUTS
#undef TOME_GEMM_FWD
#undef TOME_GEMM_DGRAD
#undef TOME_GEMM_DISPATCH
  if (rc) return rc;

  if (s.k_splits > 1) {
    const long long n4 = (long long)a->m * a->ldc / 4;
    int blocks = (int)((n4 + 255) / 256);
    if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
    launch_k(splitk_reduce_kernel, blocks, 256, 0, stream, reinterpret_cast<const float*>(workspace),
                                                     reinterpret_cast<float*>(a->c), n4, n4, s.k_splits, a->accumulate);
    TOME_CUDA(cudaGetLastError());
  }
  return TOME_OK;
}
