// Error string + TMA tensor-map encoding (driver entry point fetched at run time; the library links only cudart).
#include "host_util.h"

#include <string.h>

#include <vector>

namespace tome {

static thread_local char g_err[512] = {0};

int set_error(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
void clear_error() { g_err[0] = 0; }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

static int encode(CUtensorMap* out, const void* base, int rank, const cuuint64_t* dims, const cuuint64_t* strides_b,
                  const cuuint32_t* box, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  EncodeTiledFn fn = get_encode();
  TOME_CHECK(fn != nullptr, TOME_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
  TOME_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, TOME_ERR_INVALID, "TMA base pointer must be 16-byte aligned");
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), dims, strides_b, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  TOME_CHECK(r == CUDA_SUCCESS, TOME_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu x %llu)",
             (int)r, rank, (unsigned long long)dims[0], (unsigned long long)dims[1]);
  return TOME_OK;
}

int make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
  TOME_CHECK((ld * 2) % 16 == 0, TOME_ERR_INVALID, "TMA row pitch must be a multiple of 16 bytes (ld=%llu)", (unsigned long long)ld);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64, box_rows};
  return encode(out, base, 2, dims, strides, box);
}

int make_tmap_2d_bf16_store32(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld) {
  TOME_CHECK((ld * 2) % 16 == 0, TOME_ERR_INVALID, "TMA row pitch must be a multiple of 16 bytes (ld=%llu)", (unsigned long long)ld);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {32, 32};
  return encode(out, base, 2, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_64B);
}

int make_tmap_3d_bf16(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                      uint64_t stride2, uint32_t box_d1) {
  TOME_CHECK((stride1 * 2) % 16 == 0 && (stride2 * 2) % 16 == 0, TOME_ERR_INVALID, "TMA strides must be multiples of 16 bytes");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1 * 2, stride2 * 2};
  cuuint32_t box[3] = {64, box_d1, 1};
  return encode(out, base, 3, dims, strides, box);
}

int make_tmap_3d_bf16_plain(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                            uint64_t stride2, uint32_t box_d0, uint32_t box_d1) {
  TOME_CHECK((stride1 * 2) % 16 == 0 && (stride2 * 2) % 16 == 0 && (box_d0 * 2) % 16 == 0, TOME_ERR_INVALID,
             "TMA strides / box width must be multiples of 16 bytes");
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1 * 2, stride2 * 2};
  cuuint32_t box[3] = {box_d0, box_d1, 1};
  return encode(out, base, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
}

int make_tmap_3d_bf16_sw32(CUtensorMap* out, const void* base, uint64_t d1, uint64_t d2, uint32_t box_d1) {
  cuuint64_t dims[3] = {16, d1, d2};
  cuuint64_t strides[2] = {32, d1 * 32};
  cuuint32_t box[3] = {16, box_d1, 1};
  return encode(out, base, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_32B);
}

}  // namespace tome

namespace tome {
struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> ev;  // ev[0] = start of the recording, ev[i + 1] = end of op i
  std::vector<int> tag;
  std::vector<double> work;
  int n = 0, cap = 0;
  long long launches = 0;
};
static Profiler g_prof;  // one process drives one GPU (one rank per process); not thread-safe by design

// ONE event per op (at its end): op i lasted from the end of op i-1 to its own end.  A pair of events per op puts two
// timestamp markers around every ~30-100 us launch and showed up as 5-8 us per op (a 37 us merge launch read as 41 us);
// with one marker the gap to the previous op is charged to the op, which is what it costs the step anyway.
ProfScope::ProfScope(int tag, double work, int kernels, cudaStream_t stream) : st(stream), rec(false) {
  g_prof.launches += kernels;
  if (g_prof.on && g_prof.n < g_prof.cap) {
    g_prof.tag[g_prof.n] = tag;
    g_prof.work[g_prof.n] = work;
    if (g_prof.n == 0) cudaEventRecord(g_prof.ev[0], st);
    rec = true;
  }
}
ProfScope::~ProfScope() {
  if (rec) {
    cudaEventRecord(g_prof.ev[g_prof.n + 1], st);
    ++g_prof.n;
  }
}
}  // namespace tome

extern "C" long long tome_launch_count(int reset) {
  const long long v = tome::g_prof.launches;
  if (reset) tome::g_prof.launches = 0;
  return v;
}
extern "C" int tome_profile_enable(int max_records) {
  using namespace tome;
  clear_error();
  TOME_CHECK(max_records > 0, TOME_ERR_INVALID, "profile_enable: max_records must be positive");
  while ((int)g_prof.ev.size() < max_records + 1) {
    cudaEvent_t e;
    TOME_CUDA(cudaEventCreate(&e));
    g_prof.ev.push_back(e);
  }
  g_prof.tag.assign(max_records, 0);
  g_prof.work.assign(max_records, 0.0);
  g_prof.cap = max_records;
  g_prof.n = 0;
  g_prof.on = true;
  return TOME_OK;
}
extern "C" int tome_profile_disable(void) {
  tome::g_prof.on = false;
  return TOME_OK;
}
// Synchronises the recorded events; per tag: total milliseconds, total algorithmic work, number of ops.
extern "C" int tome_profile_collect(int n_tags, float* ms, double* work, int* count) {
  using namespace tome;
  clear_error();
  TOME_CHECK(n_tags >= PROF_NTAGS && ms && work && count, TOME_ERR_INVALID, "profile_collect: need %d tag slots", (int)PROF_NTAGS);
  for (int i = 0; i < n_tags; ++i) { ms[i] = 0.f; work[i] = 0.0; count[i] = 0; }
  for (int i = 0; i < g_prof.n; ++i) {
    float t = 0.f;
    TOME_CUDA(cudaEventSynchronize(g_prof.ev[i + 1]));
    TOME_CUDA(cudaEventElapsedTime(&t, g_prof.ev[i], g_prof.ev[i + 1]));
    ms[g_prof.tag[i]] += t;
    work[g_prof.tag[i]] += g_prof.work[i];
    count[g_prof.tag[i]] += 1;
  }
  g_prof.n = 0;
  return TOME_OK;
}

extern "C" const char* tome_last_error(void) { return tome::g_err; }

extern "C" int tome_abi_version(void) { return TOME_ABI_VERSION; }
