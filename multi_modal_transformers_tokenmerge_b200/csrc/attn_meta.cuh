// Per-token-tile attention metadata, computed ONCE per (batch, 64-token tile) by attn_meta_kernel and then streamed
// into shared memory by cp.async.bulk (1 copy per tile, completion on an mbarrier) in the forward, dQ and dK/dV
// kernels.  Before this existed every CTA -- one per (batch, head, 128-row tile), i.e. 30x redundantly at the bench
// shape -- rebuilt the same words from gid / pos / size / allow with dependent global loads on its critical path,
// and that latency chain, not the tensor pipe or MUFU, paced the kernels (profiles/r01c_attn_fwd_v2_meta_bound.txt).
//
// Block layout (ATTN_META_BYTES per (b, tile); token t of the tile is bit t&31 of word t>>5):
//   +0     bias2[64]    f32   log2(size_k), 0 when size == NULL, -inf for tokens past T
//   +256   vis[32][2]   u32   vis[g]  : KEYS of this tile visible to QUERY group g          (allow == 1)
//   +512   visc[32][2]  u32   visc[g] : keys visible to query group g iff pos_k <= pos_q    (allow == 2)
//   +768   pos[64]      i32
//   +1024  qvis[32][2]  u32   qvis[g] : QUERIES of this tile that see KEY group g           (allow == 1)
//   +1280  qvisc[32][2] u32   ... iff pos_k <= pos_q                                        (allow == 2)
// Tokens past T are "visible" everywhere: the -inf bias (keys) or +inf lse (queries) removes them.
#pragma once
#include "common.cuh"

namespace tome {

constexpr int ATTN_META_TILE = 64;
constexpr int ATTN_META_BYTES = 1536;
constexpr int ATTN_META_KEY_BYTES = 1024;   // bias2 | vis | visc | pos : what a query-row kernel needs per key tile
constexpr int ATTN_META_OFF_VIS = 256, ATTN_META_OFF_VISC = 512, ATTN_META_OFF_POS = 768, ATTN_META_OFF_QVIS = 1024,
              ATTN_META_OFF_QVISC = 1280;

// ---- the mask as part of the QK^T contraction ("augmentation") ----
// mask[q,k] depends only on (group of q, group of k), i.e. it has rank <= G.  With G <= 16 and no positional (code 2)
// rule, S' = [Q | Mq] [K | Ek]^T where Ek[k] = one-hot(group of k) and Mq[q][g] = 0 if group(q) sees group g else -2^100
// adds exactly 0 to visible logits and -2^100 (which absorbs any q.k in fp32) to masked ones: ONE extra K = 16 MMA step per
// S tile and the softmax threads do no mask work at all.  attn_meta_kernel writes the two [B, Tp, 16] bf16 operand arrays
// (32-byte rows, loaded by TMA with the 32-byte swizzle) and a flag word saying whether the trick applies to this table.
constexpr int ATTN_AUG_K = 16;
constexpr float ATTN_AUG_BIG = 1.2676506002282294e30f;   // 2^100, exact in bf16
// ---- query rows with no visible key ----
// The forward gives such a row the uniform distribution over its T keys (masked logits are one finite constant, as flax's
// finfo.min), and leaves its lse at that constant: about -FLT_MAX * ln 2 on the select path, -2^100 * scale on the
// augmentation path.  A row with a visible key has an lse of the order of its logits.  The backward and the importance
// kernel therefore recognise the row by lse * log2(e) < ATTN_MASKED_ROW_LSE2, with no pass of their own, and give it the
// forward's weights: 1/T on every key for dV and importance, and no gradient into the logits.  Holds for scale >= 2^-9.
constexpr float ATTN_MASKED_ROW_LSE2 = -1.2379400392853803e27f;   // -2^90
inline size_t attn_tiles(int tokens) { return (size_t)(tokens + ATTN_META_TILE - 1) / ATTN_META_TILE; }
inline size_t attn_blocks_bytes(int batch, int tokens) { return (size_t)batch * attn_tiles(tokens) * ATTN_META_BYTES; }
inline size_t attn_aug_array_bytes(int batch, int tokens) { return (size_t)batch * attn_tiles(tokens) * ATTN_META_TILE * ATTN_AUG_K * 2; }
// workspace of launch_attn_meta: [per-tile blocks][flag, 256 B][q operand][k operand]
inline size_t attn_meta_bytes(int batch, int tokens) { return attn_blocks_bytes(batch, tokens) + 256 + 2 * attn_aug_array_bytes(batch, tokens); }
inline const uint32_t* attn_aug_flag(const uint8_t* meta, int batch, int tokens) {
  return reinterpret_cast<const uint32_t*>(meta + attn_blocks_bytes(batch, tokens));
}
inline const uint8_t* attn_aug_q(const uint8_t* meta, int batch, int tokens) { return meta + attn_blocks_bytes(batch, tokens) + 256; }
inline const uint8_t* attn_aug_k(const uint8_t* meta, int batch, int tokens) {
  return attn_aug_q(meta, batch, tokens) + attn_aug_array_bytes(batch, tokens);
}
// launches attn_meta_kernel (attn_fwd.cu); meta must be 16-byte aligned
int launch_attn_meta(int B, int T, const uint8_t* gid, const int32_t* pos, const uint8_t* allow, int G, const float* size,
                     uint8_t* meta, cudaStream_t stream);

// ---- attention-weight dropout (flax broadcast_dropout=True: ONE [Tq, Tk] mask for every batch row and head) ----
// keep(q, k) = element k % 32 of the LCG stream (seed, site, row = q, chunk = k / 32) of common.cuh -- the generator the GEMM
// epilogues use.  Because the mask is shared by all (batch, head) pairs it is tiny (T^2 bits = 36 KB at T = 536), so
// attn_dropbits_kernel materialises it ONCE per call as bit words in the two tilings the kernels stream with one 1 KB
// bulk copy per tile:
//   keep_q[q128 tile][k64 tile][128 query rows][2 words]   bit k % 64 of a row: keep(q, k)   (forward, dQ: thread = query row)
//   keep_k[k128 tile][q64 tile][128 key rows][2 words]     bit q % 64 of a row: keep(q, k)   (dK/dV:    thread = key row)
constexpr int ATTN_DROP_TILE_BYTES = 128 * 2 * 4;
inline size_t attn_dropbits_bytes(int tokens) {  // both tilings
  const size_t n128 = (tokens + 127) / 128, n64 = (tokens + 63) / 64;
  return 2 * n128 * n64 * ATTN_DROP_TILE_BYTES;
}
// keep_q at `bits`, keep_k right after it (n128 * n64 tiles each)
int launch_attn_dropbits(int T, float rate, uint64_t seed, uint32_t site, uint8_t* bits, cudaStream_t stream);

// global -> shared bulk copy completing on an mbarrier (bytes % 16 == 0, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst_smem)), "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

}  // namespace tome
