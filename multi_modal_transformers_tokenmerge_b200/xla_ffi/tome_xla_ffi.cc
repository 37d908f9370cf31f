// XLA FFI custom-call handlers over the C ABI of include/tome_b200.h  --  the "thin jax.ffi layer" of the north star.
//
// NOT BUILT IN THIS IMAGE: jaxlib (and with it xla/ffi/api/ffi.h) is not installed and cannot be (no wheels, no
// network; SURVEY.md 0.4), so this file has never been compiled.  It is kept logic-free on purpose: every handler
// unpacks buffers and attributes, fills the matching struct of tome_b200.h and forwards to the extern "C" entry
// point on XLA's stream.  Build where jaxlib exists:
//
//   g++ -O2 -std=c++17 -fPIC -shared tome_xla_ffi.cc -o libtome_xla_ffi.so \
//       -I$(python -c "import jax.ffi; print(jax.ffi.include_dir())") -I../../include -I/usr/local/cuda/include \
//       -L.. -ltome_b200 -Wl,-rpath,'$ORIGIN/..'
//
// and register from Python with tome_jax.py (same directory).  INTEGRATION.md shows the Flax-side wiring.
#include <cstdint>
#include <cstring>
#include <optional>

#include <cuda_runtime_api.h>

#include "tome_b200.h"
#include "xla/ffi/api/ffi.h"

namespace ffi = xla::ffi;

static ffi::Error Status(int rc) {
  if (rc == TOME_OK) return ffi::Error::Success();
  return ffi::Error(rc == TOME_ERR_INVALID ? ffi::ErrorCode::kInvalidArgument : ffi::ErrorCode::kInternal, tome_last_error());
}
static int DType(ffi::DataType t) { return t == ffi::DataType::BF16 ? TOME_BF16 : TOME_F32; }

// ---- tome_sim_argmax: metric [B,T,Dm] -> node_max f32 [B,Ta], node_idx s32 [B,Ta]        token_compression.py:72-83
// workspace: tome_sim_argmax_workspace_bytes(desc) bytes from XLA's scratch allocator
static ffi::Error SimArgmax(cudaStream_t s, ffi::ScratchAllocator scratch, ffi::AnyBuffer metric,
                            ffi::Result<ffi::Buffer<ffi::F32>> node_max, ffi::Result<ffi::Buffer<ffi::S32>> node_idx,
                            int32_t class_token, int32_t distill_token) {
  auto d = metric.dimensions();
  tome_metric_desc_t m{(int)d[0], (int)d[1], (int)d[2], 1, DType(metric.element_type()), (long long)(d[1] * d[2]), (long long)d[2], 0,
                       class_token, distill_token, /*sets: one set (the FFI handlers take no token-set table)*/ nullptr};
  const size_t ws_bytes = tome_sim_argmax_workspace_bytes(&m);
  std::optional<void*> ws = scratch.Allocate(ws_bytes, 256);
  if (!ws.has_value()) return ffi::Error(ffi::ErrorCode::kResourceExhausted, "tome_sim_argmax: scratch allocation failed");
  return Status(tome_sim_argmax(&m, metric.untyped_data(), node_max->typed_data(), node_idx->typed_data(), nullptr, *ws, ws_bytes, s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeSimArgmax, SimArgmax,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Ctx<ffi::ScratchAllocator>().Arg<ffi::AnyBuffer>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::S32>>()
                                  .Attr<int32_t>("class_token").Attr<int32_t>("distill_token"));

// ---- tome_select_topr: -> edge_idx [B,Ta], dst_idx [B,r], row_map [B,T], dst_off [B,Tb+1], dst_src [B,r]    :84-88
static ffi::Error SelectTopR(cudaStream_t s, ffi::Buffer<ffi::F32> node_max, ffi::Buffer<ffi::S32> node_idx,
                             ffi::Result<ffi::Buffer<ffi::S32>> edge, ffi::Result<ffi::Buffer<ffi::S32>> dst,
                             ffi::Result<ffi::Buffer<ffi::S32>> row_map, ffi::Result<ffi::Buffer<ffi::S32>> dst_off,
                             ffi::Result<ffi::Buffer<ffi::S32>> dst_src, int32_t tokens, int32_t r, int32_t distill_token) {
  tome_plan_shape_t ps{(int)node_max.dimensions()[0], tokens, r, distill_token, /*sets=*/nullptr};
  tome_plan_t p{edge->typed_data(), dst->typed_data(), row_map->typed_data(), dst_off->typed_data(), dst_src->typed_data()};
  return Status(tome_select_topr(&ps, node_max.typed_data(), node_idx.typed_data(), &p, s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeSelectTopR, SelectTopR,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Arg<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::S32>>()
                                  .Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::S32>>().Ret<ffi::Buffer<ffi::S32>>()
                                  .Attr<int32_t>("tokens").Attr<int32_t>("r").Attr<int32_t>("distill_token"));

// ---- tome_merge_fwd (mode = attribute): x [B,T,C], size f32 [B,T] -> x_out [B,T-r,C], size_out f32 [B,T-r]   :90-129
static ffi::Error MergeFwd(cudaStream_t s, ffi::AnyBuffer x, ffi::Buffer<ffi::F32> size, ffi::Buffer<ffi::S32> edge,
                           ffi::Buffer<ffi::S32> dst_off, ffi::Buffer<ffi::S32> dst_src, ffi::Result<ffi::AnyBuffer> x_out,
                           ffi::Result<ffi::Buffer<ffi::F32>> size_out, int32_t r, int32_t mode, int32_t distill_token) {
  auto d = x.dimensions();
  tome_merge_shape_t ms{(int)d[0], (int)d[1], (int)d[2], r, distill_token, DType(x.element_type()), mode, /*sets=*/nullptr};
  tome_plan_t p{};
  p.edge_idx = edge.typed_data(); p.dst_off = dst_off.typed_data(); p.dst_src = dst_src.typed_data();
  return Status(tome_merge_fwd(&ms, &p, x.untyped_data(), size.typed_data(), x_out->untyped_data(), size_out->typed_data(),
                               nullptr, nullptr, nullptr, nullptr, s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeMergeFwd, MergeFwd,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::S32>>().Arg<ffi::Buffer<ffi::S32>>()
                                  .Arg<ffi::Buffer<ffi::S32>>().Ret<ffi::AnyBuffer>().Ret<ffi::Buffer<ffi::F32>>()
                                  .Attr<int32_t>("r").Attr<int32_t>("mode").Attr<int32_t>("distill_token"));

// ---- tome_merge_bwd (custom_vjp of merge_wavg; mode SUM == unmerge): dy [B,T-r,C] -> dx [B,T,C]
static ffi::Error MergeBwd(cudaStream_t s, ffi::AnyBuffer dy, ffi::Buffer<ffi::F32> size, ffi::Buffer<ffi::F32> size_out,
                           ffi::Buffer<ffi::S32> row_map, ffi::Result<ffi::AnyBuffer> dx, int32_t r, int32_t mode) {
  auto d = dx->dimensions();
  tome_merge_shape_t ms{(int)d[0], (int)d[1], (int)d[2], r, 0, DType(dy.element_type()), mode, /*sets=*/nullptr};
  tome_plan_t p{};
  p.row_map = row_map.typed_data();
  return Status(tome_merge_bwd(&ms, &p, size.typed_data(), size_out.typed_data(), dy.untyped_data(), dx->untyped_data(), s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeMergeBwd, MergeBwd,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::S32>>()
                                  .Ret<ffi::AnyBuffer>().Attr<int32_t>("r").Attr<int32_t>("mode"));

// ---- tome_attention_fwd: packed qkv bf16 [B,T,3,H,D], gid u8 [B,T], pos s32 [B,T], allow u8 [G,G], size f32 [B,T]
static tome_attn_desc_t AttnDesc(const ffi::AnyBuffer& qkv, const ffi::Buffer<ffi::U8>& gid, const ffi::Buffer<ffi::S32>& pos,
                                 const ffi::Buffer<ffi::U8>& allow, const ffi::Buffer<ffi::F32>& size, float scale) {
  auto d = qkv.dimensions();  // B, T, 3, H, D
  tome_attn_desc_t a;
  memset(&a, 0, sizeof(a));
  a.batch = (int)d[0]; a.tokens = (int)d[1]; a.heads = (int)d[3]; a.head_dim = (int)d[4];
  const long long tok = 3ll * d[3] * d[4];
  a.q_batch_stride = a.k_batch_stride = a.v_batch_stride = tok * d[1];
  a.q_token_stride = a.k_token_stride = a.v_token_stride = tok;
  a.o_batch_stride = (long long)d[1] * d[3] * d[4]; a.o_token_stride = (long long)d[3] * d[4];
  a.scale = scale;
  a.gid = gid.typed_data(); a.pos = pos.typed_data(); a.allow = allow.typed_data(); a.num_groups = (int)allow.dimensions()[0];
  a.size = size.typed_data();
  return a;
}
// workspace: a u8 Result buffer of tome_attention_workspace_bytes(desc) bytes that XLA allocates (tome_jax.py sizes it)
static ffi::Error AttnFwd(cudaStream_t s, ffi::AnyBuffer qkv, ffi::Buffer<ffi::U8> gid, ffi::Buffer<ffi::S32> pos,
                          ffi::Buffer<ffi::U8> allow, ffi::Buffer<ffi::F32> size, ffi::Result<ffi::AnyBuffer> out,
                          ffi::Result<ffi::Buffer<ffi::F32>> lse, ffi::Result<ffi::Buffer<ffi::U8>> workspace, float scale) {
  tome_attn_desc_t a = AttnDesc(qkv, gid, pos, allow, size, scale);
  const uint16_t* base = reinterpret_cast<const uint16_t*>(qkv.untyped_data());
  const long long hd = (long long)a.heads * a.head_dim;
  return Status(tome_attention_fwd(&a, base, base + hd, base + 2 * hd, out->untyped_data(), lse->typed_data(),
                                   workspace->typed_data(), workspace->element_count(), s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeAttentionFwd, AttnFwd,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::Buffer<ffi::U8>>().Arg<ffi::Buffer<ffi::S32>>().Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Ret<ffi::AnyBuffer>().Ret<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>().Attr<float>("scale"));

// ---- tome_attention_bwd: -> dqkv bf16 [B,T,3,H,D]; the workspace is a Result buffer XLA allocates for us
static ffi::Error AttnBwd(cudaStream_t s, ffi::AnyBuffer qkv, ffi::AnyBuffer out, ffi::Buffer<ffi::F32> lse, ffi::AnyBuffer dout,
                          ffi::Buffer<ffi::U8> gid, ffi::Buffer<ffi::S32> pos, ffi::Buffer<ffi::U8> allow, ffi::Buffer<ffi::F32> size,
                          ffi::Result<ffi::AnyBuffer> dqkv, ffi::Result<ffi::Buffer<ffi::U8>> workspace, float scale) {
  tome_attn_desc_t a = AttnDesc(qkv, gid, pos, allow, size, scale);
  tome_attn_grad_strides_t g{a.q_batch_stride, a.q_token_stride, a.q_batch_stride, a.q_token_stride, a.q_batch_stride, a.q_token_stride,
                             a.o_batch_stride, a.o_token_stride};
  const uint16_t* base = reinterpret_cast<const uint16_t*>(qkv.untyped_data());
  uint16_t* dbase = reinterpret_cast<uint16_t*>(dqkv->untyped_data());
  const long long hd = (long long)a.heads * a.head_dim;
  return Status(tome_attention_bwd(&a, &g, base, base + hd, base + 2 * hd, out.untyped_data(), lse.typed_data(), dout.untyped_data(),
                                   dbase, dbase + hd, dbase + 2 * hd, workspace->typed_data(), workspace->element_count(), s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeAttentionBwd, AttnBwd,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::AnyBuffer>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::AnyBuffer>().Arg<ffi::Buffer<ffi::U8>>()
                                  .Arg<ffi::Buffer<ffi::S32>>().Arg<ffi::Buffer<ffi::U8>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::AnyBuffer>().Ret<ffi::Buffer<ffi::U8>>().Attr<float>("scale"));

// ---- tome_gemm_bf16 as a Dense layer: y = epilogue(x [M,K] * kernel [K,N] + bias)       attention.py:32-37
static ffi::Error Dense(cudaStream_t s, ffi::AnyBuffer x, ffi::AnyBuffer kernel, ffi::Buffer<ffi::F32> bias, ffi::AnyBuffer residual,
                        ffi::Result<ffi::AnyBuffer> y, int32_t relu, int32_t has_residual, float dropout_rate, int64_t seed, int32_t site) {
  tome_gemm_args_t g;
  memset(&g, 0, sizeof(g));
  g.m = (int)x.dimensions()[0]; g.k = (int)x.dimensions()[1]; g.n = (int)kernel.dimensions()[1];
  g.a = x.untyped_data(); g.lda = g.k; g.a_major = TOME_MAJOR_K;
  g.b = kernel.untyped_data(); g.ldb = g.n; g.b_major = TOME_MAJOR_MN;   // Flax layout [in, out] used as is
  g.c = y->untyped_data(); g.ldc = g.n; g.c_dtype = TOME_BF16;
  g.bias = bias.typed_data(); g.relu = relu; g.gate_scale = 1.f;
  if (has_residual) { g.residual = residual.untyped_data(); g.ldr = g.n; }
  g.dropout_rate = dropout_rate; g.dropout_seed = (uint64_t)seed; g.dropout_site = (uint32_t)site;
  return Status(tome_gemm_bf16(&g, nullptr, 0, s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeDense, Dense,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::AnyBuffer>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::AnyBuffer>().Ret<ffi::AnyBuffer>().Attr<int32_t>("relu")
                                  .Attr<int32_t>("has_residual").Attr<float>("dropout_rate").Attr<int64_t>("seed").Attr<int32_t>("site"));

// ---- LayerNorm as configured (axis attribute: 1 tokens / 2 features)                     vanilla_decoder.yaml:7-13
static ffi::Error LayerNormFwd(cudaStream_t s, ffi::AnyBuffer x, ffi::Buffer<ffi::F32> gamma, ffi::Buffer<ffi::F32> beta,
                               ffi::Result<ffi::AnyBuffer> y, ffi::Result<ffi::Buffer<ffi::F32>> mean,
                               ffi::Result<ffi::Buffer<ffi::F32>> rstd, int32_t axis, float eps) {
  auto d = x.dimensions();
  return Status(tome_layernorm_fwd((int)d[0], (int)d[1], (int)d[2], axis, eps, x.untyped_data(), gamma.typed_data(), beta.typed_data(),
                                   y->untyped_data(), mean->typed_data(), rstd->typed_data(), s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeLayerNormFwd, LayerNormFwd,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::Buffer<ffi::F32>>().Ret<ffi::AnyBuffer>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Attr<int32_t>("axis").Attr<float>("eps"));

// ---- the whole stack as ONE custom call (forward; backward is symmetric over tome_stack_backward).  The flat parameter
// vectors, the activation workspace (a Result buffer sized by tome_stack_workspace_bytes at trace time) and the config
// (passed as a byte-string attribute holding tome_stack_cfg_t) map one to one onto tome_stack_io_t.
static ffi::Error StackFwd(cudaStream_t s, ffi::Buffer<ffi::F32> params_f32, ffi::AnyBuffer params_bf16, ffi::AnyBuffer x,
                           ffi::Buffer<ffi::U8> gid, ffi::Buffer<ffi::S32> pos, ffi::Buffer<ffi::U8> allow,
                           ffi::Buffer<ffi::S32> readout_idx, ffi::Buffer<ffi::F32> target, ffi::Result<ffi::Buffer<ffi::U8>> workspace,
                           ffi::Result<ffi::AnyBuffer> x_final, ffi::Result<ffi::Buffer<ffi::F32>> readout,
                           ffi::Result<ffi::Buffer<ffi::F32>> loss, ffi::Result<ffi::Buffer<ffi::F32>> head_out,
                           std::string_view cfg_bytes) {
  if (cfg_bytes.size() != sizeof(tome_stack_cfg_t)) return ffi::Error(ffi::ErrorCode::kInvalidArgument, "bad tome_stack_cfg_t attribute");
  tome_stack_cfg_t cfg;
  memcpy(&cfg, cfg_bytes.data(), sizeof(cfg));
  tome_stack_io_t io;
  memset(&io, 0, sizeof(io));
  io.params_f32 = params_f32.typed_data(); io.params_bf16 = params_bf16.untyped_data();
  io.x = x.untyped_data(); io.x_dtype = DType(x.element_type());
  io.gid = gid.typed_data(); io.pos = pos.typed_data(); io.allow = allow.typed_data();
  io.readout_idx = readout_idx.typed_data(); io.target = target.typed_data();
  io.workspace = workspace->typed_data(); io.workspace_bytes = workspace->element_count();
  io.x_final = x_final->untyped_data(); io.readout = readout->typed_data(); io.loss = loss->typed_data();
  io.head_out = cfg.head > 0 ? head_out->typed_data() : nullptr;   // actions / logits of the action head ([1] dummy without one)
  return Status(tome_stack_forward(&cfg, &io, s));
}
XLA_FFI_DEFINE_HANDLER_SYMBOL(TomeStackFwd, StackFwd,
                              ffi::Ffi::Bind().Ctx<ffi::PlatformStream<cudaStream_t>>().Arg<ffi::Buffer<ffi::F32>>().Arg<ffi::AnyBuffer>()
                                  .Arg<ffi::AnyBuffer>().Arg<ffi::Buffer<ffi::U8>>().Arg<ffi::Buffer<ffi::S32>>()
                                  .Arg<ffi::Buffer<ffi::U8>>().Arg<ffi::Buffer<ffi::S32>>().Arg<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::U8>>().Ret<ffi::AnyBuffer>().Ret<ffi::Buffer<ffi::F32>>()
                                  .Ret<ffi::Buffer<ffi::F32>>().Ret<ffi::Buffer<ffi::F32>>().Attr<std::string_view>("cfg"));
