// K9: per-modality top-k token pruning.   tokenizers/token_compression.py:15-46 (compute_top_k_tokens)
//
// For every token set (a contiguous slice [start, start + n) of the sequence) keep the k tokens with the largest
// importance score, in DESCENDING score order (jax.lax.top_k: equal scores keep the lower index first), concatenate
// the sets in the order given, and gather those rows of the embeddings.  The reference is written for one sequence
// and vmapped by its caller; here the batch is a grid dimension.
//
// One CTA per (token set, batch row): the set's scores go to shared memory, every token counts how many tokens of its
// set beat it (its rank; for n up to a few hundred the n^2 comparisons are cheaper than a sort and exact by
// construction), ranks < k publish their index, and the CTA then copies the k selected rows with 128-bit accesses.
// Token sets of 384 tokens or more take a bitonic sort of (score, index) keys and a grid-wide gather instead (below).
// Index arithmetic only: the gathered rows are bit-identical to the source rows.
#include "common.cuh"
#include "host_util.h"

namespace tome {

constexpr int PRUNE_THREADS = 256;

// "j ranks before i" in top_k order: larger score first, NaN above every number, equal scores by lower index
__device__ __forceinline__ bool topk_before(float vj, int j, float vi, int i) {
  const bool nj = vj != vj, ni = vi != vi;
  if (nj || ni) return nj && (!ni || j < i);
  return vj > vi || (vj == vi && j < i);
}

__global__ void __launch_bounds__(PRUNE_THREADS)
topk_prune_kernel(const tome_prune_desc_t d, const uint8_t* __restrict__ emb, const float* __restrict__ score,
                  uint8_t* __restrict__ out, int32_t* __restrict__ ids) {
  extern __shared__ float prune_sm[];
  const int s = blockIdx.x, b = blockIdx.y;
  const int start = d.set_start[s], n = d.set_n[s], k = d.set_k[s];
  int off = 0;
  for (int i = 0; i < s; ++i) off += d.set_k[i];
  int ktot = off;
  for (int i = s; i < d.n_sets; ++i) ktot += d.set_k[i];
  float* vals = prune_sm;                                   // [n]
  int* sel = reinterpret_cast<int*>(prune_sm + n);          // [k] token index of rank r
  // importance may arrive as `score_planes` partial planes [P][B][T] (e.g. one per attention head): summed in plane
  // order, so the ranking does not depend on how the caller reduced them
  for (int i = threadIdx.x; i < n; i += PRUNE_THREADS) {
    float v = 0.f;
    for (int p = 0; p < d.score_planes; ++p) v += score[((long long)p * d.batch + b) * d.tokens + start + i];
    vals[i] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += PRUNE_THREADS) {
    const float vi = vals[i];
    int rk = 0;
    for (int j = 0; j < n; ++j) rk += topk_before(vals[j], j, vi, i) ? 1 : 0;
    if (rk < k) {
      sel[rk] = start + i;
      ids[(long long)b * ktot + off + rk] = start + i;
    }
  }
  __syncthreads();
  const int row_bytes = d.channels * (d.dtype == TOME_BF16 ? 2 : 4);
  const int vpr = row_bytes >> 4;  // 16-byte vectors per row
  const uint8_t* eb = emb + (long long)b * d.tokens * row_bytes;
  uint8_t* ob = out + ((long long)b * ktot + off) * row_bytes;
  for (int i = threadIdx.x; i < k * vpr; i += PRUNE_THREADS) {
    const int r = i / vpr, v = i - r * vpr;
    st_na_v4(ob + (long long)r * row_bytes + v * 16, ld_nc_v4(eb + (long long)sel[r] * row_bytes + v * 16));
  }
}

// ---- long token sets: sort instead of rank-by-count (n^2 comparisons: 3.8 ms per call at n = 4076 against 0.1 ms at 500) ----
// 64-bit keys (orderable score bits, complemented index) sorted DEscending in shared memory reproduce top_k's order: larger
// score first, NaN above every number, -0 == +0, equal scores by LOWER index.  One CTA per (token set, batch row) writes the
// ids; the rows are then gathered by a grid-wide kernel (one CTA per set would copy megabytes alone).
constexpr int PRUNE_SORT_THREADS = 1024;
constexpr int PRUNE_SORT_MIN_N = 384;     // token sets at least this long take the sort path (measured: n = 488 -> 125 us by counting)

__device__ __forceinline__ unsigned long long prune_key(float v, int i) {
  uint32_t u = __float_as_uint(v);
  if (v != v) u = 0xFFFFFFFFu;
  else if (v == 0.f) u = 0x80000000u;
  else u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (uint32_t)(0x7FFFFFFF - i);
}

__global__ void __launch_bounds__(PRUNE_SORT_THREADS)
topk_sort_kernel(const tome_prune_desc_t d, const float* __restrict__ score, int32_t* __restrict__ ids) {
  extern __shared__ __align__(8) unsigned char prune_sort_raw[];
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(prune_sort_raw);
  const int s = blockIdx.x, b = blockIdx.y, tid = threadIdx.x, nt = blockDim.x;
  const int start = d.set_start[s], n = d.set_n[s], k = d.set_k[s];
  int off = 0;
  for (int i = 0; i < s; ++i) off += d.set_k[i];
  int ktot = off;
  for (int i = s; i < d.n_sets; ++i) ktot += d.set_k[i];
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  for (int i = tid; i < n2; i += nt) {
    unsigned long long key = 0ull;   // below every real key
    if (i < n) {
      float v = 0.f;
      for (int p = 0; p < d.score_planes; ++p) v += score[((long long)p * d.batch + b) * d.tokens + start + i];
      key = prune_key(v, i);
    }
    keys[i] = key;
  }
  __syncthreads();
  for (int kk = 2; kk <= n2; kk <<= 1)
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n2; i += nt) {
        const int l = i ^ j;
        if (l > i) {
          const unsigned long long a = keys[i], c = keys[l];
          const bool desc = (i & kk) == 0;
          if (desc ? a < c : a > c) { keys[i] = c; keys[l] = a; }
        }
      }
      __syncthreads();
    }
  for (int rk = tid; rk < k; rk += nt) ids[(long long)b * ktot + off + rk] = start + (0x7FFFFFFF - (int)(uint32_t)keys[rk]);
}

// out[b, j] = emb[b, ids[b, j]] (bit copies), thread = 16 bytes
__global__ void __launch_bounds__(256)
prune_gather_kernel(long long n_vec, int T, int K, int vpr, const int32_t* __restrict__ ids, const uint4* __restrict__ emb,
                    uint4* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n_vec; i += (long long)gridDim.x * 256) {
    const long long rowg = i / vpr;           // b * K + j
    const int v = (int)(i - rowg * vpr);
    const int b = (int)(rowg / K);
    st_na_v4(out + i, ld_nc_v4(emb + ((long long)b * T + ids[rowg]) * vpr + v));
  }
}

// row_map[b, t] = output row of token t, -1 when it was pruned; gid / pos follow the kept tokens.  row_map is pre-filled with
// -1 by the caller (cudaMemsetAsync 0xFF); ids are distinct per batch row, so the scatter has no collisions.
__global__ void prune_row_map_kernel(int B, int T, int K, const int32_t* __restrict__ ids, const uint8_t* __restrict__ gid,
                                     const int32_t* __restrict__ pos, int32_t* __restrict__ row_map, uint8_t* __restrict__ gid_out,
                                     int32_t* __restrict__ pos_out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)B * K) return;
  const int b = (int)(i / K), j = (int)(i - (long long)b * K);
  const int t = ids[i];
  row_map[(long long)b * T + t] = j;
  if (gid_out) gid_out[i] = gid[(long long)b * T + t];
  if (pos_out) pos_out[i] = pos[(long long)b * T + t];
}

// backward of the gather: dx[b, t] = dy[b, row_map[b, t]], zero for a pruned token.  Thread = 16 bytes.
__global__ void __launch_bounds__(256)
prune_bwd_kernel(long long n_vec, int T, int K, int vpr, const int32_t* __restrict__ row_map, const uint4* __restrict__ dy,
                 uint4* __restrict__ dx) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n_vec; i += (long long)gridDim.x * 256) {
    const long long rowg = i / vpr;
    const int v = (int)(i - rowg * vpr);
    const int b = (int)(rowg / T);
    const int r = row_map[rowg];
    dx[i] = r >= 0 ? ld_nc_v4(dy + ((long long)b * K + r) * vpr + v) : make_uint4(0u, 0u, 0u, 0u);
  }
}

}  // namespace tome

using namespace tome;

extern "C" int tome_prune_row_map(int batch, int tokens, int kept, const int32_t* ids, const uint8_t* gid, const int32_t* pos,
                                  int32_t* row_map, uint8_t* gid_out, int32_t* pos_out, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && kept >= 0 && kept <= tokens && ids && row_map, TOME_ERR_INVALID, "prune_row_map: bad argument");
  TOME_CHECK((!gid_out || gid) && (!pos_out || pos), TOME_ERR_INVALID, "prune_row_map: gid_out / pos_out need gid / pos");
  ProfScope prof(PROF_OTHER, 0.0, 2, stream);
  TOME_CUDA(cudaMemsetAsync(row_map, 0xFF, (size_t)batch * tokens * sizeof(int32_t), stream));
  if (kept == 0) return TOME_OK;
  const long long n = (long long)batch * kept;
  launch_k(prune_row_map_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, batch, tokens, kept, ids, gid, pos, row_map, gid_out, pos_out);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_prune_bwd(int batch, int tokens, int kept, int channels, int dtype, const int32_t* row_map, const void* dy,
                              void* dx, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(batch > 0 && tokens > 0 && kept > 0 && kept <= tokens && channels > 0 && row_map && dy && dx, TOME_ERR_INVALID,
             "prune_bwd: bad argument");
  TOME_CHECK(dtype == TOME_BF16 || dtype == TOME_F32, TOME_ERR_INVALID, "prune_bwd: dtype must be bf16 or f32");
  const int row_bytes = channels * (dtype == TOME_BF16 ? 2 : 4);
  TOME_CHECK(row_bytes % 16 == 0 && ((((uintptr_t)dy | (uintptr_t)dx) & 15) == 0), TOME_ERR_INVALID,
             "prune_bwd: rows must be multiples of 16 bytes, 16-byte aligned");
  const int vpr = row_bytes / 16;
  const long long n_vec = (long long)batch * tokens * vpr;
  long long blocks = (n_vec + 255) / 256;
  if (blocks > (long long)kNumSMs * 16) blocks = (long long)kNumSMs * 16;
  ProfScope prof(PROF_PRUNE, (double)batch * ((double)tokens + kept) * row_bytes, 1, stream);
  launch_k(prune_bwd_kernel, (unsigned)blocks, 256, 0, stream, n_vec, tokens, kept, vpr, row_map, reinterpret_cast<const uint4*>(dy),
           reinterpret_cast<uint4*>(dx));
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}

extern "C" int tome_topk_prune(const tome_prune_desc_t* d, const void* embeddings, const float* importance, void* out,
                               int32_t* ids, void* stream_) {
  clear_error();
  cudaStream_t stream = (cudaStream_t)stream_;
  TOME_CHECK(d && embeddings && importance && out && ids, TOME_ERR_INVALID, "topk_prune: null argument");
  TOME_CHECK(d->batch > 0 && d->batch <= 65535 && d->tokens > 0 && d->channels > 0, TOME_ERR_INVALID, "topk_prune: bad shape");
  TOME_CHECK(d->dtype == TOME_BF16 || d->dtype == TOME_F32, TOME_ERR_INVALID, "topk_prune: dtype must be bf16 or f32");
  TOME_CHECK((d->channels * (d->dtype == TOME_BF16 ? 2 : 4)) % 16 == 0, TOME_ERR_INVALID,
             "topk_prune: rows must be a multiple of 16 bytes (channels = %d)", d->channels);
  TOME_CHECK((((uintptr_t)embeddings | (uintptr_t)out) & 15) == 0, TOME_ERR_INVALID, "topk_prune: embeddings / out must be 16-byte aligned");
  TOME_CHECK(d->n_sets >= 1 && d->n_sets <= TOME_MAX_TOKEN_SETS, TOME_ERR_INVALID, "topk_prune: 1 <= n_sets <= %d (got %d)",
             TOME_MAX_TOKEN_SETS, d->n_sets);
  TOME_CHECK(d->score_planes >= 1, TOME_ERR_INVALID, "topk_prune: score_planes must be >= 1");
  int nmax = 0;
  for (int s = 0; s < d->n_sets; ++s) {
    TOME_CHECK(d->set_start[s] >= 0 && d->set_n[s] >= 1 && d->set_start[s] + d->set_n[s] <= d->tokens, TOME_ERR_INVALID,
               "topk_prune: token set %d = [%d, +%d) leaves the sequence of %d tokens", s, d->set_start[s], d->set_n[s], d->tokens);
    // jax.lax.top_k raises for k > n (token_compression.py:31)
    TOME_CHECK(d->set_k[s] >= 0 && d->set_k[s] <= d->set_n[s], TOME_ERR_INVALID,
               "topk_prune: token set %d keeps k = %d of %d tokens (top_k needs 0 <= k <= n)", s, d->set_k[s], d->set_n[s]);
    if (d->set_n[s] > nmax) nmax = d->set_n[s];
  }
  int ktot_host = 0;
  for (int s = 0; s < d->n_sets; ++s) ktot_host += d->set_k[s];
  const double row_bytes_host = d->channels * (d->dtype == TOME_BF16 ? 2.0 : 4.0);
  const size_t smem = (size_t)2 * nmax * sizeof(float);
  TOME_CHECK(nmax >= PRUNE_SORT_MIN_N || smem <= 200 * 1024, TOME_ERR_UNSUPPORTED, "topk_prune: token set of %d tokens is too large for the shared-memory ranking", nmax);
  dim3 grid(d->n_sets, d->batch);
  if (nmax >= PRUNE_SORT_MIN_N) {   // long token sets: sort + grid-wide gather
    int n2 = 1;
    while (n2 < nmax) n2 <<= 1;
    const size_t smem_sort = (size_t)n2 * sizeof(unsigned long long);
    TOME_CHECK(smem_sort <= 200 * 1024, TOME_ERR_UNSUPPORTED, "topk_prune: token set of %d tokens is too large for the shared-memory sort", nmax);
    ProfScope prof(PROF_PRUNE, (double)d->batch * ((double)d->tokens * 4 + 2.0 * ktot_host * row_bytes_host), 2, stream);
    TOME_CUDA(cudaFuncSetAttribute(topk_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_sort));
    launch_k(topk_sort_kernel, grid, PRUNE_SORT_THREADS, smem_sort, stream, *d, importance, ids);
    TOME_CUDA(cudaGetLastError());
    if (ktot_host > 0) {
      const int vpr = (int)row_bytes_host / 16;
      const long long n_vec = (long long)d->batch * ktot_host * vpr;
      long long blocks = (n_vec + 255) / 256;
      if (blocks > (long long)kNumSMs * 16) blocks = (long long)kNumSMs * 16;
      launch_k(prune_gather_kernel, (unsigned)blocks, 256, 0, stream, n_vec, d->tokens, ktot_host, vpr, ids,
               reinterpret_cast<const uint4*>(embeddings), reinterpret_cast<uint4*>(out));
      TOME_CUDA(cudaGetLastError());
    }
    return TOME_OK;
  }
  ProfScope prof(PROF_PRUNE, (double)d->batch * ((double)d->tokens * 4 + 2.0 * ktot_host * row_bytes_host), 1, stream);
  TOME_CUDA(cudaFuncSetAttribute(topk_prune_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  launch_k(topk_prune_kernel, grid, PRUNE_THREADS, smem, stream, *d, reinterpret_cast<const uint8_t*>(embeddings), importance,
                                                          reinterpret_cast<uint8_t*>(out), ids);
  TOME_CUDA(cudaGetLastError());
  return TOME_OK;
}
