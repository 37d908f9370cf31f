// Host-side helpers shared by the C-ABI translation units: error reporting (thread-local string, never throws
// across the ABI) and TMA tensor-map encoding through the driver entry point (no link-time libcuda dependency).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <atomic>

#include "../../include/tome_b200.h"

namespace tome {

int set_error(int code, const char* fmt, ...);  // returns code
void clear_error();

#define TOME_CHECK(cond, code, ...)                        \
  do {                                                     \
    if (!(cond)) return ::tome::set_error(code, __VA_ARGS__); \
  } while (0)

#define TOME_CUDA(expr)                                                                                   \
  do {                                                                                                    \
    cudaError_t _e = (expr);                                                                              \
    if (_e != cudaSuccess)                                                                                \
      return ::tome::set_error(TOME_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                               __LINE__);                                                                 \
  } while (0)

// Row-major bf16 matrix [rows, cols] with leading dimension ld (elements), described as a 2-D TMA tensor with a
// {64 x box_rows} box and 128-byte swizzle.  cols*2 and ld*2 must be multiples of 16 bytes.
int make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows);
// Same matrix as a TMA STORE target: box {32 columns, 32 rows}, 64-byte swizzle (one epilogue warp's chunk).
int make_tmap_2d_bf16_store32(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld);
// [d2, d1, d0] bf16 tensor (d0 contiguous; strides in elements), box {64, box_d1, 1}, 128-byte swizzle.
int make_tmap_3d_bf16(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                      uint64_t stride2, uint32_t box_d1);

// same tensor with a {box_d0, box_d1, 1} box and no swizzle (box_d0 * 2 bytes must be a multiple of 16)
int make_tmap_3d_bf16_plain(CUtensorMap* out, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1,
                            uint64_t stride2, uint32_t box_d0, uint32_t box_d1);

// [d2, d1, 16] bf16 tensor of 32-byte rows (dense), box {16, box_d1, 1}, 32-byte swizzle: the K = 16 "mask augmentation" operand
int make_tmap_3d_bf16_sw32(CUtensorMap* out, const void* base, uint64_t d1, uint64_t d2, uint32_t box_d1);

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Carves a workspace into 256-byte aligned buffers, in call order.  A module's `*_workspace_bytes` and its launch run
// the same carving function, the query with base == nullptr (every pointer comes back null), so the size it reports is
// the size the launch uses.
struct Bump {
  uint8_t* base;
  size_t off = 0;
  size_t reserve(size_t bytes) {  // returns the new buffer's offset from base
    off = (off + 255) & ~size_t(255);
    const size_t at = off;
    off += bytes;
    return at;
  }
  template <typename T>
  T* take(size_t count) {
    const size_t at = reserve(count * sizeof(T));
    return base ? reinterpret_cast<T*>(base + at) : nullptr;
  }
  size_t total() const { return (off + 255) & ~size_t(255); }
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is a PER-DEVICE attribute: a process that drives several GPUs (JAX's
// default) must set it on each one.  One DynSmemOnce per call site remembers, per device, the largest size already set.
struct DynSmemOnce {
  std::atomic<int> set[64];
};
template <typename Kernel>
inline cudaError_t ensure_dyn_smem(Kernel kernel, int bytes, DynSmemOnce& once) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  if (dev < 0 || dev >= 64) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (once.set[dev].load(std::memory_order_acquire) >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) once.set[dev].store(bytes, std::memory_order_release);
  return e;
}

// ---- kernel launches: the arguments are converted to the kernel's parameter types ----
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- launch accounting + optional per-op CUDA-event timing (bench.py's roofline pass; off by default) ----
enum ProfTag { PROF_GEMM = 0, PROF_ATTN_FWD, PROF_ATTN_BWD, PROF_MERGE_FWD, PROF_MERGE_BWD, PROF_SIM, PROF_SELECT,
               PROF_LN, PROF_COLSUM, PROF_OTHER, PROF_IMPORTANCE, PROF_PRUNE, PROF_NTAGS };
struct ProfScope {  // RAII around one C-ABI op: `kernels` launches doing `work` algorithmic FLOPs or bytes
  cudaStream_t st;
  bool rec;
  ProfScope(int tag, double work, int kernels, cudaStream_t stream);
  ~ProfScope();
};

}  // namespace tome
