// Blackwell (sm_100a) device-side building blocks shared by every kernel in this library:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (UMMA + TMEM), 128-bit global access, counter RNG.
// Raw PTX on purpose: no CUTLASS/CuTe dependency, descriptors laid out bit by bit (layouts follow the
// PTX ISA "tcgen05 matrix/instruction descriptor" tables).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace tome {

constexpr int kNumSMs = 148;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// ------------------------------------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Bounded wait: a protocol bug must fault (trap) instead of hanging the GPU box.  try_wait carries a suspend-time
// hint, so a waiting thread sleeps in hardware until the phase completes (or ~8 us pass) instead of spinning on the
// issue port its CTA's working warps need; the spin bound is therefore counted in units of that time-out.
#ifndef TOME_MBAR_SPIN_LIMIT
#define TOME_MBAR_SPIN_LIMIT (1 << 22)
#endif
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  int spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(8192u)
        : "memory");
    if (done) break;
    if (++spins > TOME_MBAR_SPIN_LIMIT) __trap();
  }
}

// ------------------------------------------------------------------------------------------------ TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// multicast: the box lands at the same shared-memory offset, and completes on the barrier at the same offset, in every
// CTA of the cluster named in cta_mask
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1, uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {  // every thread of every CTA in the cluster
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------ tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc];   bf16 x bf16 -> fp32, issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Same with the A operand read from TENSOR MEMORY (K-major, lane = row, one 32-bit column = two consecutive bf16 of K, so a
// K = 16 step is 8 columns): the operand costs no shared-memory bandwidth.  128 x N x 16 with both operands in shared
// memory reads (128 + N) * 32 B per step, which at N = 64 is more than the 128 B/clk the SM's shared memory delivers in
// the 32 cycles the step takes on the tensor pipe.
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// ---- cta_group::2: the two CTAs of a cluster pair run ONE 256-row MMA.  A: each CTA supplies its own 128 rows; B: each CTA
// supplies N/2 of the N columns; D: each CTA's tensor memory receives its 128 rows x N columns.  Issued by the leader
// (cluster rank 0) only; shared-memory descriptors name the same offsets in both CTAs.
__device__ __forceinline__ void umma2_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this offset in every CTA of cta_mask once the pair's previously issued MMAs have completed
__device__ __forceinline__ void umma2_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* dst_smem, uint32_t ncols) {  // one full warp, in EACH CTA of the pair
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// shared::cluster address of `p` (a shared-memory location of THIS CTA) as seen in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// arrive on a barrier that may live in the peer CTA.  Relaxed: the only data the waiter depends on is tensor memory already
// read by tcgen05.ld (ordered by tcgen05.wait::ld + tcgen05.fence::before_thread_sync); a .release here costs a
// MEMBAR + ERRBAR per arrive that waits for every store of the epilogue warp still in flight (22 % of all stall samples)
__device__ __forceinline__ float ld_shared_cluster_f32(uint32_t cluster_addr) {   // distributed shared memory read (address from map_to_cta)
  float v;
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(cluster_addr) : "memory");
  return v;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load whose completion is counted on a barrier given by its shared::cluster address (the leader CTA's, for a pair MMA)
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* tm, uint32_t bar_cluster_addr, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
      : "memory");
}
// mbarrier arrives once every previously issued UMMA of this thread has completed (implies fence::before).
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// same, arriving on the barrier at this offset in every CTA of cta_mask
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(cta_mask)
               : "memory");
}

// Shared-memory matrix descriptor, 128-byte swizzle (layout_type = 2), version 1 (Blackwell).
//   bits [0,14)  start address >> 4      bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4 bits [46,48) version = 1     bits [61,64) swizzle mode
// K-major  tile (rows = M/N, 64 bf16 = 128 B of K per row):  SBO = 1024 (8 rows * 128 B), LBO unused (=16 B)
// MN-major tile (rows = K, 64 bf16 = 128 B of M/N per row):   SBO = 1024 (8 k-rows),  LBO = bytes between
//                                                             consecutive 64-wide M/N atoms
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// K-major operand of ONE K = 16 step stored as dense 32-byte rows with the 32-byte swizzle (layout_type = 6): 8-row atoms of
// 256 bytes stacked along M/N (SBO = 256); what TMA writes for a {16 x rows} bf16 box with CU_TENSOR_MAP_SWIZZLE_32B.
__device__ __forceinline__ uint64_t make_smem_desc_sw32(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;            // LBO: unused for a swizzled K-major operand that is one atom wide
  d |= (uint64_t)(256 >> 4) << 32;   // SBO
  d |= (uint64_t)1 << 46;            // version 1 (Blackwell)
  d |= (uint64_t)6 << 61;            // SWIZZLE_32B
  return d;
}
// Instruction descriptor for kind::f16, bf16 inputs, fp32 accumulator.
//   [4,6) c_format=1(F32)  [7,10) a_format=1(BF16)  [10,13) b_format=1(BF16)  [15] a_major  [16] b_major
//   [17,23) N>>3   [24,29) M>>4
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N, bool a_mn_major, bool b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) |
         ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// TMEM -> registers: warp w reads lanes [32*(w%4), +32); thread i gets lane i, N consecutive 32-bit columns.
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// same load, straight into fp32 registers
__device__ __forceinline__ void tmem_ld_f32x32(uint32_t taddr, float (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7]), "=f"(r[8]),
        "=f"(r[9]), "=f"(r[10]), "=f"(r[11]), "=f"(r[12]), "=f"(r[13]), "=f"(r[14]), "=f"(r[15]), "=f"(r[16]),
        "=f"(r[17]), "=f"(r[18]), "=f"(r[19]), "=f"(r[20]), "=f"(r[21]), "=f"(r[22]), "=f"(r[23]), "=f"(r[24]),
        "=f"(r[25]), "=f"(r[26]), "=f"(r[27]), "=f"(r[28]), "=f"(r[29]), "=f"(r[30]), "=f"(r[31])
      : "r"(taddr)
      : "memory");
}

// ------------------------------------------------------------------------------------------------ 128-bit access
__device__ __forceinline__ uint4 ld_nc_v4(const void* p) {  // streaming read, do not allocate in L1
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_na_v4(void* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z),
               "r"(v.w)
               : "memory");
}
__device__ __forceinline__ float bf16_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// ------------------------------------------------------------------------------------------------ dropout RNG
// Counter-based and stateless, so forward and backward regenerate the same mask and no mask tensor is ever stored.
// An element (row, col) of a row-major [M, N] tensor belongs to the STREAM (row, col / 32): two independent 32-bit
// hashes of (seed, site, row, chunk) give the start state x0 and an odd increment c of a 32-bit LCG, and element
// e = col % 32 of the chunk is kept iff the top 16 bits of x_{e+1} (x_{k+1} = A x_k + c) are >= thresh16.
// One multiply-add and one compare per element: this runs in the GEMM epilogue, thread = row, 32 columns at a time,
// where the previous Philox4x32-10 (~10 integer ops per element) made the epilogue, not the tensor pipe, the
// bottleneck of every dropout GEMM (profiles/r01b_gemm_ncu_summary.txt).  Jump-ahead constants let a consumer that
// owns 8 elements start in the middle of a chunk.  (Flax's threefry stream cannot be reproduced either way.)
struct DropoutCfg {
  uint32_t thresh16;  // 0 => dropout disabled; keep iff u16 >= thresh16, thresh16 = round(rate * 65536)
  float inv_keep;     // 1 / (1 - thresh16/65536)
  uint32_t seed_lo, seed_hi;
  uint32_t site;  // distinguishes call sites / layers
};
// The one rate -> threshold conversion: forward and backward regenerate the same mask only if every call site rounds
// `rate` the same way (and a dgrad's gate_scale must equal the forward epilogue's inv_keep).
inline DropoutCfg make_dropout(float rate, uint64_t seed, uint32_t site) {
  DropoutCfg d;
  d.thresh16 = (uint32_t)(rate * 65536.0f + 0.5f);
  d.inv_keep = 1.0f / (1.0f - (float)d.thresh16 / 65536.0f);
  d.seed_lo = (uint32_t)seed; d.seed_hi = (uint32_t)(seed >> 32);
  d.site = site;
  return d;
}
constexpr uint32_t DROP_A = 0x915F77F5u;  // LCG multiplier (A % 8 == 5: full period for any odd increment)
__host__ __device__ constexpr uint32_t drop_pow(int n) { uint32_t r = 1; for (int i = 0; i < n; ++i) r *= DROP_A; return r; }
__host__ __device__ constexpr uint32_t drop_geo(int n) { uint32_t r = 0, a = 1; for (int i = 0; i < n; ++i) { r += a; a *= DROP_A; } return r; }  // 1 + A + ... + A^(n-1)
__device__ __forceinline__ uint32_t lowbias32(uint32_t x) {
  x ^= x >> 16; x *= 0x21f0aaadu; x ^= x >> 15; x *= 0x735a2d97u; x ^= x >> 15;
  return x;
}
struct DropStream {
  uint32_t x, c;
  __device__ __forceinline__ uint32_t next() { x = x * DROP_A + c; return x; }   // word of the next element; top 16 bits are the uniform
  __device__ __forceinline__ void skip8(int n8) {  // jump over 8 * n8 elements (n8 in 0..3)
    const uint32_t pa = n8 == 0 ? 1u : n8 == 1 ? drop_pow(8) : n8 == 2 ? drop_pow(16) : drop_pow(24);
    const uint32_t ge = n8 == 0 ? 0u : n8 == 1 ? drop_geo(8) : n8 == 2 ? drop_geo(16) : drop_geo(24);
    x = x * pa + c * ge;
  }
};
__device__ __forceinline__ DropStream drop_stream(const DropoutCfg& d, uint32_t row, uint32_t chunk) {
  const uint32_t k = d.seed_lo ^ (d.site * 0x9E3779B9u);
  DropStream s;
  s.x = lowbias32(row * 0x9E3779B1u + chunk * 0x85EBCA77u + k);
  s.c = lowbias32((row ^ d.seed_hi) * 0xC2B2AE35u + chunk * 0x27D4EB2Fu + (k ^ 0x5bd1e995u)) | 1u;
  return s;
}
// 8 bits: bit j set => element (row, col + j) is KEPT; col % 8 == 0
__device__ __forceinline__ uint32_t dropout_keep8(const DropoutCfg& d, uint32_t row, uint32_t col) {
  DropStream s = drop_stream(d, row, col >> 5);
  s.skip8((col >> 3) & 3);
  const uint32_t thr = d.thresh16 << 16;
  uint32_t m = 0;
#pragma unroll
  for (int j = 0; j < 8; ++j) m |= (s.next() >= thr ? 1u : 0u) << j;
  return m;
}

// MUFU.EX2 without the denormal fix-up code exp2f() drags in: ex2(-inf) = +0, ex2(x < -126) flushes to 0.
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ------------------------------------------------------------------------------------------------ warp helpers
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace tome
