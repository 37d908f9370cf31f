// K3 + K4: size-weighted merge and its transpose (unmerge / merge backward).   token_compression.py:90-129
//
// HBM-bound by construction: every input row is read once and every output row written once with 128-bit
// accesses; a thread owns one 16-byte vector of one output row, consecutive threads own consecutive vectors of
// the same row, so every warp-level request is a run of full 128-byte lines.  No atomics: an output row GATHERS
// its sources through the CSR lists K2 built (dst_off / dst_src), adding them in rank order -- the same fp32
// association as the reference's sequential `dst.at[...].add(src[:, i])` loop (:100-101), hence bit-exact.
//
// algorithmic bytes / sample (merge fwd, SURVEY.md 8d):  T*C*e + 4T + 4(Ta + r) + (T-r)*C*e + 4(T-r)
#include "common.cuh"
#include "host_util.h"
#include "token_sets.cuh"

namespace tome {

template <typename T>
struct Vec;  // 16-byte vector of T <-> fp32 lanes
template <>
struct Vec<float> {
  static constexpr int N = 4;
  __device__ static void load(const float* p, float (&f)[4]) {
    const uint4 v = ld_nc_v4(p);
    f[0] = __uint_as_float(v.x); f[1] = __uint_as_float(v.y); f[2] = __uint_as_float(v.z); f[3] = __uint_as_float(v.w);
  }
  __device__ static void store(float* p, const float (&f)[4]) {
    st_na_v4(p, make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]), __float_as_uint(f[2]), __float_as_uint(f[3])));
  }
};
template <>
struct Vec<__nv_bfloat16> {
  static constexpr int N = 8;
  __device__ static void load(const __nv_bfloat16* p, float (&f)[8]) {
    const uint4 v = ld_nc_v4(p);
    f[0] = bf16_lo(v.x); f[1] = bf16_hi(v.x); f[2] = bf16_lo(v.y); f[3] = bf16_hi(v.y);
    f[4] = bf16_lo(v.z); f[5] = bf16_hi(v.z); f[6] = bf16_lo(v.w); f[7] = bf16_hi(v.w);
  }
  __device__ static void store(__nv_bfloat16* p, const float (&f)[8]) {
    st_na_v4(p, make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7])));
  }
};

constexpr int MERGE_THREADS = 256;

// Output row prow of batch row b, inverted through the concatenation order (:103-108) of its token set: the input token it
// keeps (an unmerged even token or a destination), its CSR source range, and where the set's sources are listed: source e is
// input token tok0 + 2 * dst_src[src_base + e].  Rows of a set with r == 0 are plain copies (copy = true).
struct RowPlan {
  int keep_tok, e0, e1, tok0;
  long long src_base;
  bool copy;
};
__device__ __forceinline__ RowPlan resolve_row(const SetTable& tab, bool distill, const tome_plan_t& p, int b, int prow) {
  const int set = set_of(tab.out_off, tab.n, prow);
  const int lrow = prow - tab.out_off[set], r = tab.r[set];
  RowPlan m;
  m.e0 = m.e1 = 0;
  m.tok0 = tab.start[set];
  m.src_base = (long long)b * tab.r_off[tab.n] + tab.r_off[set];
  m.copy = r == 0;
  if (m.copy) {
    m.keep_tok = m.tok0 + lrow;
    return m;
  }
  const int n_unm = (tab.len[set] + 1) / 2 - r;
  int u = -1, j = -1;
  if (!distill) {
    if (lrow < n_unm) u = lrow; else j = lrow - n_unm;
  } else {
    if (lrow == 0) u = 0;
    else if (lrow == 1) j = 0;
    else if (lrow <= n_unm) u = lrow - 1;
    else j = lrow - n_unm;
  }
  if (u >= 0) {
    m.keep_tok = m.tok0 + 2 * p.edge_idx[(long long)b * tab.a_off[tab.n] + tab.a_off[set] + r + u];
  } else {
    m.keep_tok = m.tok0 + 2 * j + 1;
    const long long o = (long long)b * tab.off_off[tab.n] + tab.off_off[set] + j;
    m.e0 = p.dst_off[o];
    m.e1 = p.dst_off[o + 1];
  }
  return m;
}

template <typename T, bool WAVG>
__global__ void __launch_bounds__(MERGE_THREADS)
merge_fwd_kernel(const tome_merge_shape_t s, const __grid_constant__ SetTable tab, const tome_plan_t p, const T* __restrict__ x,
                 const float* __restrict__ size, T* __restrict__ x_out, float* __restrict__ size_out,
                 const uint8_t* __restrict__ gid, const int32_t* __restrict__ pos, uint8_t* __restrict__ gid_out,
                 int32_t* __restrict__ pos_out) {
  constexpr int N = Vec<T>::N;
  const int Tn = s.tokens, r = s.r, C = s.channels;
  const int To = Tn - r;
  const int vpr = C / N;  // vectors per row
  const long long total = (long long)s.batch * To * vpr;
  for (long long item = blockIdx.x * (long long)MERGE_THREADS + threadIdx.x; item < total;
       item += (long long)gridDim.x * MERGE_THREADS) {
    const int v = (int)(item % vpr);
    const long long rowg = item / vpr;
    const int prow = (int)(rowg % To);
    const int b = (int)(rowg / To);
    const RowPlan m = resolve_row(tab, s.distill_token, p, b, prow);
    const T* xb = x + (long long)b * Tn * C;
    const float* sb = size ? size + (long long)b * Tn : nullptr;
    float acc[N];
    const int keep_tok = m.keep_tok;
    Vec<T>::load(xb + (long long)keep_tok * C + v * N, acc);
    float sacc = sb ? sb[keep_tok] : 1.0f;
    // merge(x*size)/merge(size), literally: an unmerged token or a destination without sources also becomes (x*s)/s
    if (!m.copy) {
      if (WAVG) {
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i] = __fmul_rn(acc[i], sacc);
      }
      for (int e = m.e0; e < m.e1; ++e) {
        const int tok = m.tok0 + 2 * p.dst_src[m.src_base + e];
        float f[N];
        Vec<T>::load(xb + (long long)tok * C + v * N, f);
        const float sz = sb ? sb[tok] : 1.0f;
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i] = __fadd_rn(acc[i], WAVG ? __fmul_rn(f[i], sz) : f[i]);  // no FMA contraction
        sacc = __fadd_rn(sacc, sz);
      }
      if (WAVG) {
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i] = __fdiv_rn(acc[i], sacc);
      }
    }
    Vec<T>::store(x_out + ((long long)b * To + prow) * C + v * N, acc);
    if (v == 0) {
      if (size_out) size_out[(long long)b * To + prow] = sacc;
      if (gid_out) gid_out[(long long)b * To + prow] = gid[(long long)b * Tn + keep_tok];
      if (pos_out) pos_out[(long long)b * To + prow] = pos[(long long)b * Tn + keep_tok];
    }
  }
}

// ------------------------------------------------------------------------------------------------ K3, bulk-copy version
// A CTA owns `rows` consecutive output rows of one batch element.
//   1. threads < rows: resolve which input token each output row keeps (edge_idx / odd position), its size, its CSR
//      source range; produce size_out / gid_out / pos_out for the row.
//   2. one cp.async.bulk (global -> shared) per kept row, all completing on one mbarrier: the gather runs in the copy
//      engine with rows * row_bytes in flight per CTA and no register staging.
//   3. rows that need arithmetic (size != 1, or sources merged into them) are patched in shared memory; their source
//      rows are read straight from global (r of T rows).
//   4. the run of output rows is contiguous in x_out: ONE cp.async.bulk (shared -> global) writes it.
struct MergeRowMeta {
  int keep_tok;
  int e0, e1;
  int tok0, src0;   // the row's token set: first token, first dst_src entry in the batch row (RowPlan)
  float size_keep;  // size of the kept token
  float size_sum;   // size_out of the row
};

template <typename T, bool WAVG>
__global__ void __launch_bounds__(MERGE_THREADS)
merge_fwd_bulk_kernel(const tome_merge_shape_t s, const __grid_constant__ SetTable tab, const tome_plan_t p, const T* __restrict__ x,
                      const float* __restrict__ size, T* __restrict__ x_out, float* __restrict__ size_out,
                      const uint8_t* __restrict__ gid, const int32_t* __restrict__ pos, uint8_t* __restrict__ gid_out,
                      int32_t* __restrict__ pos_out, int rows_per_cta) {
  constexpr int N = Vec<T>::N;
  extern __shared__ __align__(128) uint8_t smem_merge[];
  const int Tn = s.tokens, r = s.r, C = s.channels;
  const int To = Tn - r;
  const int row_bytes = C * (int)sizeof(T);
  const int b = blockIdx.y;
  const int row0 = blockIdx.x * rows_per_cta;
  const int nrows = min(rows_per_cta, To - row0);
  uint8_t* s_rows = smem_merge;
  MergeRowMeta* s_meta = reinterpret_cast<MergeRowMeta*>(smem_merge + (size_t)rows_per_cta * row_bytes);
  int* s_fix = reinterpret_cast<int*>(s_meta + rows_per_cta);  // [rows_per_cta] rows that need arithmetic
  int* s_nfix = s_fix + rows_per_cta;
  uint64_t* bar = reinterpret_cast<uint64_t*>((reinterpret_cast<uintptr_t>(s_nfix + 1) + 7) & ~uintptr_t(7));

  const T* xb = x + (long long)b * Tn * C;
  const float* sb = size ? size + (long long)b * Tn : nullptr;
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(bar, 1);
    fence_barrier_init();
    *s_nfix = 0;
  }
  __syncthreads();
  if (tid == 0) mbar_expect_tx(bar, (uint32_t)(nrows * row_bytes));
  if (tid < nrows) {
    const int prow = row0 + tid;
    const RowPlan rp = resolve_row(tab, s.distill_token, p, b, prow);
    MergeRowMeta m;
    m.keep_tok = rp.keep_tok;
    m.e0 = rp.e0;
    m.e1 = rp.e1;
    m.tok0 = rp.tok0;
    m.src0 = (int)(rp.src_base - (long long)b * tab.r_off[tab.n]);
    // the copy first: everything below overlaps it
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(s_rows + (size_t)tid * row_bytes)), "l"(xb + (long long)m.keep_tok * C), "r"(row_bytes),
                   "r"(smem_u32(bar))
                 : "memory");
    m.size_keep = sb ? sb[m.keep_tok] : 1.0f;
    float sacc = m.size_keep;
    for (int e = m.e0; e < m.e1; ++e) sacc = __fadd_rn(sacc, sb ? sb[m.tok0 + 2 * p.dst_src[rp.src_base + e]] : 1.0f);
    m.size_sum = sacc;
    s_meta[tid] = m;
    // rows of an r == 0 set stay the bit copies the bulk load made
    if (!rp.copy && ((WAVG && m.size_keep != 1.0f) || m.e1 > m.e0)) s_fix[atomicAdd(s_nfix, 1)] = tid;
    if (size_out) size_out[(long long)b * To + prow] = sacc;
    if (gid_out) gid_out[(long long)b * To + prow] = gid[(long long)b * Tn + m.keep_tok];
    if (pos_out) pos_out[(long long)b * To + prow] = pos[(long long)b * Tn + m.keep_tok];
  }
  __syncthreads();  // s_meta / s_fix visible; (thread 0's expect_tx preceded every copy: it is first in program order of warp 0, and the phase cannot complete before its arrival)
  mbar_wait(bar, 0);

  const int nfix = *s_nfix;
  if (nfix > 0) {
    const int vpr = C / N;
    for (int item = tid; item < nfix * vpr; item += MERGE_THREADS) {
      const int fr = s_fix[item / vpr], v = item % vpr;
      const MergeRowMeta m = s_meta[fr];
      T* srow = reinterpret_cast<T*>(s_rows + (size_t)fr * row_bytes) + v * N;
      float acc[N];
      {
        const uint4 q = *reinterpret_cast<const uint4*>(srow);
        if constexpr (N == 8) {
          acc[0] = bf16_lo(q.x); acc[1] = bf16_hi(q.x); acc[2] = bf16_lo(q.y); acc[3] = bf16_hi(q.y);
          acc[4] = bf16_lo(q.z); acc[5] = bf16_hi(q.z); acc[6] = bf16_lo(q.w); acc[7] = bf16_hi(q.w);
        } else {
          acc[0] = __uint_as_float(q.x); acc[1] = __uint_as_float(q.y); acc[2] = __uint_as_float(q.z); acc[3] = __uint_as_float(q.w);
        }
      }
      if (WAVG) {
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i] = __fmul_rn(acc[i], m.size_keep);
      }
      for (int e = m.e0; e < m.e1; ++e) {
        const int tok = m.tok0 + 2 * p.dst_src[(long long)b * tab.r_off[tab.n] + m.src0 + e];
        float f[N];
        Vec<T>::load(xb + (long long)tok * C + v * N, f);
        const float sz = sb ? sb[tok] : 1.0f;
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i] = __fadd_rn(acc[i], WAVG ? __fmul_rn(f[i], sz) : f[i]);  // no FMA contraction
      }
      if (WAVG) {
#pragma unroll
        for (int i = 0; i < N; ++i) acc[i] = __fdiv_rn(acc[i], m.size_sum);
      }
      uint4 o;
      if constexpr (N == 8) {
        o = make_uint4(pack_bf16(acc[0], acc[1]), pack_bf16(acc[2], acc[3]), pack_bf16(acc[4], acc[5]), pack_bf16(acc[6], acc[7]));
      } else {
        o = make_uint4(__float_as_uint(acc[0]), __float_as_uint(acc[1]), __float_as_uint(acc[2]), __float_as_uint(acc[3]));
      }
      *reinterpret_cast<uint4*>(srow) = o;
    }
    fence_proxy_async_smem();  // patched rows visible to the bulk store (async proxy)
    __syncthreads();
  }
  if (tid == 0) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                 ::"l"(x_out + ((long long)b * To + row0) * C), "r"(smem_u32(s_rows)), "r"(nrows * row_bytes)
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // shared memory must outlive the store's reads
  }
}

template <typename T, bool WAVG>
__global__ void __launch_bounds__(MERGE_THREADS)
merge_bwd_kernel(const tome_merge_shape_t s, const int32_t* __restrict__ row_map, const float* __restrict__ size,
                 const float* __restrict__ size_out, const T* __restrict__ dy, T* __restrict__ dx) {
  constexpr int N = Vec<T>::N;
  const int Tn = s.tokens, C = s.channels, To = Tn - s.r;
  const int vpr = C / N;
  const long long total = (long long)s.batch * Tn * vpr;
  for (long long item = blockIdx.x * (long long)MERGE_THREADS + threadIdx.x; item < total;
       item += (long long)gridDim.x * MERGE_THREADS) {
    const int v = (int)(item % vpr);
    const long long rowg = item / vpr;  // b * T + t
    const int b = (int)(rowg / Tn);
    const int row = row_map[rowg];
    float f[N];
    Vec<T>::load(dy + ((long long)b * To + row) * C + v * N, f);
    if (WAVG) {
      const float w = (size ? size[rowg] : 1.0f) / size_out[(long long)b * To + row];
#pragma unroll
      for (int i = 0; i < N; ++i) f[i] = __fmul_rn(f[i], w);
    }
    Vec<T>::store(dx + rowg * C + v * N, f);
  }
}

static inline int merge_grid(long long items) {
  long long blocks = (items + MERGE_THREADS - 1) / MERGE_THREADS;
  const long long cap = (long long)kNumSMs * 16;  // 8 resident CTAs/SM x 2 waves, grid-stride beyond that
  if (blocks > cap) blocks = cap;
  return (int)(blocks > 0 ? blocks : 1);
}

static int check_merge_shape(const tome_merge_shape_t* s, const tome_plan_t* plan, SetTable* tab, const char* who) {
  TOME_CHECK(s && plan, TOME_ERR_INVALID, "%s: null shape/plan", who);
  TOME_CHECK(s->batch > 0 && s->tokens >= 2 && s->channels > 0, TOME_ERR_INVALID, "%s: bad shape", who);
  TOME_CHECK(s->dtype == TOME_BF16 || s->dtype == TOME_F32, TOME_ERR_INVALID, "%s: dtype must be bf16 or f32", who);
  const int n = s->dtype == TOME_BF16 ? 8 : 4;
  TOME_CHECK(s->channels % n == 0, TOME_ERR_INVALID, "%s: channels (%d) must be a multiple of %d (16-byte vectors)", who,
             s->channels, n);
  TOME_CHECK(s->r >= 1 && s->r <= s->tokens / 2, TOME_ERR_INVALID, "%s: r (%d) out of range [1, %d]", who, s->r,
             s->tokens / 2);
  TOME_CHECK(s->mode == TOME_MERGE_SUM || s->mode == TOME_MERGE_WAVG, TOME_ERR_INVALID,
             "%s: unknown merge mode %d (the reference only implements \"sum\", token_compression.py:99)", who, s->mode);
  return make_set_table(s->sets, s->tokens, s->r, 0, s->distill_token, tab, who);
}

}  // namespace tome

using namespace tome;

extern "C" int tome_merge_fwd(const tome_merge_shape_t* s, const tome_plan_t* plan, const void* x, const float* size,
                              void* x_out, float* size_out, const uint8_t* gid, const int32_t* pos, uint8_t* gid_out,
                              int32_t* pos_out, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  SetTable tab;
  if (int rc = check_merge_shape(s, plan, &tab, "merge_fwd")) return rc;
  TOME_CHECK(x && x_out, TOME_ERR_INVALID, "merge_fwd: null x / x_out");
  TOME_CHECK(plan->edge_idx && plan->dst_off && plan->dst_src, TOME_ERR_INVALID, "merge_fwd: incomplete plan");
  TOME_CHECK((!gid_out || gid) && (!pos_out || pos), TOME_ERR_INVALID, "merge_fwd: gid_out/pos_out need gid/pos");
  TOME_CHECK((((uintptr_t)x | (uintptr_t)x_out) & 15) == 0, TOME_ERR_INVALID, "merge_fwd: x / x_out must be 16-byte aligned");
  const int n = s->dtype == TOME_BF16 ? 8 : 4;
  const long long items = (long long)s->batch * (s->tokens - s->r) * (s->channels / n);
  const double esz = s->dtype == TOME_BF16 ? 2.0 : 4.0;
  ProfScope prof(PROF_MERGE_FWD, (double)s->batch * ((double)s->tokens * s->channels * esz + 4.0 * s->tokens +
                 4.0 * ((s->tokens + 1) / 2 + s->r) + (double)(s->tokens - s->r) * s->channels * esz + 4.0 * (s->tokens - s->r)), 1, stream);
  const bool wavg = s->mode == TOME_MERGE_WAVG;
  const int row_bytes = s->channels * (int)esz;
  if (row_bytes <= 32768 && s->batch <= 65535) {
    // bulk-copy path: rows * row_bytes ~ 24 KB per CTA, so 8 CTAs (~190 KB in flight) fit one SM
    int rows = 24576 / row_bytes;
    if (rows < 1) rows = 1;
    if (rows > 128) rows = 128;
    if (rows > s->tokens - s->r) rows = s->tokens - s->r;
    const size_t smem = (size_t)rows * row_bytes + (size_t)rows * (sizeof(MergeRowMeta) + sizeof(int)) + sizeof(int) + 24;
    dim3 grid2(ceil_div(s->tokens - s->r, rows), s->batch);
#define LAUNCHB(TT, W)                                                                                                  \
  do {                                                                                                                  \
    static DynSmemOnce once;                                                                                            \
    if (smem > 48 * 1024) TOME_CUDA(ensure_dyn_smem(merge_fwd_bulk_kernel<TT, W>, (int)smem, once));                   \
    launch_k(merge_fwd_bulk_kernel<TT, W>, grid2, MERGE_THREADS, smem, stream, *s, tab, *plan, reinterpret_cast<const TT*>(x), size, \
                                                                         reinterpret_cast<TT*>(x_out), size_out, gid, pos, \
                                                                         gid_out, pos_out, rows);                       \
  } while (0)
    if (s->dtype == TOME_BF16) { if (wavg) LAUNCHB(__nv_bfloat16, true); else LAUNCHB(__nv_bfloat16, false); }
    else { if (wavg) LAUNCHB(float, true); else LAUNCHB(float, false); }
#undef LAUNCHB
    TOME_CUDA(cudaGetLastError());
    return TOME_OK;
  }
  const int grid = merge_grid(items);  // rows wider than 32 KB: thread-per-vector kernel
#define LAUNCH(TT, W)                                                                                              \
  launch_k(merge_fwd_kernel<TT, W>, grid, MERGE_THREADS, 0, stream, *s, tab, *plan, reinterpret_cast<const TT*>(x), size, \
                                                              reinterpret_cast<TT*>(x_out), size_out, gid, pos,   \
                                                              gid_out, pos_out)
  if (s->dtype == TOME_BF16) { if (wavg) LAUNCH(__nv_bfloat16, true); else LAUNCH(__nv_bfloat16, false); }
  else { if (wavg) LAUNCH(float, true); else LAUNCH(float, false); }
#undef LAUNCH
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_merge_bwd(const tome_merge_shape_t* s, const tome_plan_t* plan, const float* size,
                              const float* size_out, const void* dy, void* dx, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  SetTable tab;   // merge_bwd reads the global row map only; the table is validated so that both directions accept the same shapes
  if (int rc = check_merge_shape(s, plan, &tab, "merge_bwd")) return rc;
  TOME_CHECK(dy && dx && plan->row_map, TOME_ERR_INVALID, "merge_bwd: null dy / dx / row_map");
  const bool wavg = s->mode == TOME_MERGE_WAVG;
  TOME_CHECK(!wavg || size_out, TOME_ERR_INVALID, "merge_bwd: WAVG needs size_out");
  TOME_CHECK((((uintptr_t)dy | (uintptr_t)dx) & 15) == 0, TOME_ERR_INVALID, "merge_bwd: dy / dx must be 16-byte aligned");
  const int n = s->dtype == TOME_BF16 ? 8 : 4;
  const long long items = (long long)s->batch * s->tokens * (s->channels / n);
  const double esz = s->dtype == TOME_BF16 ? 2.0 : 4.0;
  ProfScope prof(PROF_MERGE_BWD, (double)s->batch * ((double)(s->tokens - s->r) * s->channels * esz + (double)s->tokens * s->channels * esz + 4.0 * s->tokens), 1, stream);
  const int grid = merge_grid(items);
#define LAUNCH(TT, W)                                                                                               \
  launch_k(merge_bwd_kernel<TT, W>, grid, MERGE_THREADS, 0, stream, *s, plan->row_map, size, size_out,                    \
                                                              reinterpret_cast<const TT*>(dy), reinterpret_cast<TT*>(dx))
  if (s->dtype == TOME_BF16) { if (wavg) LAUNCH(__nv_bfloat16, true); else LAUNCH(__nv_bfloat16, false); }
  else { if (wavg) LAUNCH(float, true); else LAUNCH(float, false); }
#undef LAUNCH
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
