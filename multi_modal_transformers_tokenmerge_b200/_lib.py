"""ctypes binding of include/tome_b200.h (the C-ABI drop-in boundary).

There is NO fallback: if libtome_b200.so is missing or a call fails, this raises.  The structures below mirror the
header field for field; `tests/test_abi.py` checks that every symbol the header declares is exported.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libtome_b200.so")

TOME_OK, TOME_ERR_INVALID, TOME_ERR_CUDA, TOME_ERR_UNSUPPORTED = 0, 1, 2, 3
TOME_BF16, TOME_F32, TOME_U8 = 0, 1, 2
TOME_MAJOR_K, TOME_MAJOR_MN = 0, 1
TOME_MERGE_SUM, TOME_MERGE_WAVG = 0, 1
ABI_VERSION = 15

vp, ll, i32, f32, u64, u32 = C.c_void_p, C.c_longlong, C.c_int, C.c_float, C.c_uint64, C.c_uint32


class TomeError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"tome_b200 error {code}: {msg}")
        self.code = code


MAX_TOKEN_SETS = 16


class TokenSets(C.Structure):
    """tome_token_sets_t: consecutive token sets covering the sequence; set s loses set_r[s] tokens to merging inside it."""
    _fields_ = [("n_sets", i32), ("set_start", i32 * MAX_TOKEN_SETS), ("set_n", i32 * MAX_TOKEN_SETS),
                ("set_r", i32 * MAX_TOKEN_SETS)]


class MetricDesc(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("dim", i32), ("heads", i32), ("dtype", i32),
                ("batch_stride", ll), ("token_stride", ll), ("head_stride", ll),
                ("class_token", i32), ("distill_token", i32), ("sets", vp)]


class Plan(C.Structure):
    _fields_ = [("edge_idx", vp), ("dst_idx", vp), ("row_map", vp), ("dst_off", vp), ("dst_src", vp)]


class PlanShape(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("r", i32), ("distill_token", i32), ("sets", vp)]


class PruneDesc(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("channels", i32), ("dtype", i32), ("n_sets", i32),
                ("set_start", i32 * 16), ("set_n", i32 * 16), ("set_k", i32 * 16), ("score_planes", i32)]


class MergeShape(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("channels", i32), ("r", i32), ("distill_token", i32),
                ("dtype", i32), ("mode", i32), ("sets", vp)]


class GemmArgs(C.Structure):
    _fields_ = [("m", i32), ("n", i32), ("k", i32),
                ("a", vp), ("lda", ll), ("a_major", i32),
                ("b", vp), ("ldb", ll), ("b_major", i32),
                ("c", vp), ("ldc", ll), ("c_dtype", i32),
                ("bias", vp),
                ("residual", vp), ("ldr", ll),
                ("gate", vp), ("ldg", ll),
                ("gate_scale", f32), ("relu", i32),
                ("dropout_rate", f32), ("dropout_seed", u64), ("dropout_site", u32),
                ("k_splits", i32), ("accumulate", i32),
                ("gate_bits", vp), ("relu_bits_out", vp), ("ld_bits", ll), ("colsum_partial", vp),
                ("a_row_shift", vp), ("a_shift_groups", i32)]


class AttnDesc(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("heads", i32), ("head_dim", i32),
                ("q_batch_stride", ll), ("q_token_stride", ll), ("k_batch_stride", ll), ("k_token_stride", ll),
                ("v_batch_stride", ll), ("v_token_stride", ll), ("o_batch_stride", ll), ("o_token_stride", ll),
                ("scale", f32),
                ("gid", vp), ("pos", vp), ("allow", vp), ("num_groups", i32),
                ("size", vp), ("dropout_rate", f32), ("dropout_seed", u64), ("dropout_site", C.c_uint32)]


class AttnGradStrides(C.Structure):
    _fields_ = [("dq_batch_stride", ll), ("dq_token_stride", ll), ("dk_batch_stride", ll), ("dk_token_stride", ll),
                ("dv_batch_stride", ll), ("dv_token_stride", ll), ("do_batch_stride", ll), ("do_token_stride", ll),
                ("bias_partial", vp), ("bias_partial_ld", ll), ("bias_q_col", i32), ("bias_k_col", i32), ("bias_v_col", i32)]


class StackCfg(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("channels", i32), ("heads", i32), ("head_dim", i32),
                ("mlp_dim", i32), ("layers", i32), ("r", i32), ("ln_axis", i32), ("ln_eps", f32),
                ("prop_attn", i32), ("class_token", i32), ("distill_token", i32), ("num_groups", i32),
                ("n_readout", i32), ("dropout_rate", f32), ("dropout_seed", u64), ("attn_dropout_rate", f32),
                ("head", i32), ("head_groups", i32), ("head_features", i32), ("max_action", f32),
                ("head_fourier_dim", i32), ("head_time_hidden", i32), ("head_time_out", i32), ("head_hidden", i32),
                ("diffusion_steps", i32),
                ("prune_sets", i32), ("prune_set_n", i32 * 16), ("prune_set_c", i32 * 16), ("prune_importance", i32),
                ("set_merge", i32)]


IMPORTANCE_ROW_MEAN, IMPORTANCE_RECEIVED = 0, 1


class DiffusionDesc(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("channels", i32), ("n_readout", i32), ("action_dim", i32),
                ("fourier_dim", i32), ("time_hidden", i32), ("time_out", i32), ("hidden", i32), ("diffusion_steps", i32)]


DIFFUSION_PARAMS = ["fourier_kernel", "tw1", "tb1", "tw2", "tb2", "w1", "b1", "w2", "b2"]


HEAD_CONTINUOUS_L2, HEAD_CATEGORICAL_CE = 0, 1


class ImageTokenizerDesc(C.Structure):
    _fields_ = [("batch", i32), ("n_images", i32), ("image_size", i32), ("channels_in", i32), ("image_dtype", i32),
                ("normalize", i32), ("patch_size", i32), ("conv_kernel", i32), ("conv_stride", i32), ("features", i32),
                ("pool_window", i32), ("num_blocks", i32), ("num_groups", i32), ("gn_eps", f32), ("embed_dim", i32),
                ("position_interval", i32), ("token_rows", i32), ("out_dtype", i32), ("chunk_rows", i32)]


IT_CONV0_KERNEL, IT_CONV0_BIAS, IT_DENSE_KERNEL, IT_DENSE_BIAS, IT_ROW_EMBED, IT_COL_EMBED, IT_BLOCK0 = 0, 1, 2, 3, 4, 5, 16


class HeadDesc(C.Structure):
    _fields_ = [("batch", i32), ("tokens", i32), ("channels", i32), ("x_dtype", i32), ("n_readout", i32),
                ("groups", i32), ("features", i32), ("kind", i32), ("max_action", f32)]


class StackIO(C.Structure):
    _fields_ = [("params_f32", vp), ("params_bf16", vp), ("x", vp), ("x_dtype", i32),
                ("gid", vp), ("pos", vp), ("allow", vp), ("readout_idx", vp), ("target", vp),
                ("workspace", vp), ("workspace_bytes", C.c_size_t),
                ("x_final", vp), ("readout", vp), ("loss", vp), ("grads_f32", vp),
                ("layer_done_events", C.POINTER(vp)), ("head_out", vp), ("head_time", vp), ("head_alpha_hats", vp),
                ("grad_trace", vp), ("layer_gid", vp), ("layer_pos", vp)]


_lib = None


def lib() -> C.CDLL:
    """The loaded shared library.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -m multi_modal_transformers_tokenmerge_b200.build` "
                "(or __graft_entry__.build()).  There is no CPU or PyTorch fallback for this package.")
        L = C.CDLL(LIB_PATH)
        L.tome_last_error.restype = C.c_char_p
        L.tome_abi_version.restype = i32
        if L.tome_abi_version() != ABI_VERSION:
            raise ImportError(f"libtome_b200.so has ABI {L.tome_abi_version()}, python binding expects {ABI_VERSION}: rebuild")
        for name in ("tome_gemm_workspace_bytes", "tome_stack_workspace_bytes", "tome_attention_workspace_bytes", "tome_sim_argmax_workspace_bytes",
                     "tome_attention_bwd_workspace_bytes", "tome_action_head_workspace_bytes", "tome_diffusion_head_workspace_bytes",
                     "tome_image_tokenizer_workspace_bytes"):
            getattr(L, name).restype = C.c_size_t
        for name in ("tome_stack_param_count", "tome_stack_layer_offset", "tome_stack_head_offset", "tome_launch_count",
                     "tome_diffusion_head_param_count", "tome_diffusion_head_param_offset",
                     "tome_image_tokenizer_param_count", "tome_image_tokenizer_param_offset"):
            getattr(L, name).restype = ll
        for name in ("tome_stack_final_x", "tome_stack_final_size", "tome_stack_layer_edge_idx", "tome_stack_layer_dst_idx",
                     "tome_stack_layer_node_max", "tome_stack_layer_node_idx", "tome_stack_layer_relu_bits",
                     "tome_stack_layer_x_in", "tome_stack_layer_size_in", "tome_stack_layer_importance", "tome_stack_layer_prune_ids"):
            getattr(L, name).restype = vp
        P = C.POINTER
        sig = {
            "tome_clamp_r": [i32, i32, i32, i32],
            "tome_sim_argmax_workspace_bytes": [P(MetricDesc)],
            "tome_sim_argmax": [P(MetricDesc), vp, vp, vp, vp, vp, C.c_size_t, vp],
            "tome_select_topr": [P(PlanShape), vp, vp, P(Plan), vp],
            "tome_merge_fwd": [P(MergeShape), P(Plan), vp, vp, vp, vp, vp, vp, vp, vp, vp],
            "tome_merge_bwd": [P(MergeShape), P(Plan), vp, vp, vp, vp, vp],
            "tome_topk_prune": [P(PruneDesc), vp, vp, vp, vp, vp],
            "tome_prune_row_map": [i32, i32, i32, vp, vp, vp, vp, vp, vp, vp],
            "tome_prune_bwd": [i32, i32, i32, i32, i32, vp, vp, vp, vp],
            "tome_attention_importance": [P(AttnDesc), vp, vp, vp, i32, vp, vp],
            "tome_stack_layer_importance": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_prune_ids": [P(StackCfg), P(StackIO), i32],
            "tome_gemm_workspace_bytes": [P(GemmArgs)],
            "tome_gemm_bf16": [P(GemmArgs), vp, C.c_size_t, vp],
            "tome_gemm_set_sm_limit": [i32],
            "tome_gemm_force_tile": [i32, i32],          # test hook, not in the header
            "tome_colsum_workspace_rows": [i32],
            "tome_reduce_rows_f32": [i32, i32, vp, vp, i32, vp],
            "tome_colsum_bf16": [i32, i32, vp, ll, vp, i32, vp, vp],
            "tome_dropout_colsum_bf16": [i32, i32, vp, vp, f32, C.c_uint64, C.c_uint32, vp, i32, vp, vp],
            "tome_layernorm_fwd": [i32, i32, i32, i32, f32, vp, vp, vp, vp, vp, vp, vp],
            "tome_layernorm_bwd": [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
            "tome_ln_force_cluster": [i32],              # test hook, not in the header
            "tome_attention_workspace_bytes": [P(AttnDesc)],
            "tome_attention_bwd_workspace_bytes": [P(AttnDesc)],
            "tome_attention_fwd": [P(AttnDesc), vp, vp, vp, vp, vp, vp, C.c_size_t, vp],
            "tome_attention_bwd": [P(AttnDesc), P(AttnGradStrides), vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp],
            "tome_attention_set_dq_from_ds": [i32],      # test hook, not in the header
            "tome_add_pos_embedding": [i32, i32, i32, vp, i32, vp, vp, vp],
            "tome_pos_embedding_bwd": [i32, i32, i32, vp, vp, vp],
            "tome_chain_row_maps": [i32, i32, P(vp), P(i32), vp, i32, vp, vp],
            "tome_readout_mse": [i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp],
            "tome_action_head_workspace_bytes": [P(HeadDesc)],
            "tome_action_head_fwd": [P(HeadDesc), vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp],
            "tome_action_head_bwd": [P(HeadDesc), vp, vp, vp, vp, vp, vp, vp],
            "tome_attention_pool_fwd": [i32, i32, i32, i32, i32, vp, vp, vp, vp, ll, i32, vp, vp, vp],
            "tome_stack_head_offset": [P(StackCfg)],
            "tome_diffusion_head_param_count": [P(DiffusionDesc)],
            "tome_diffusion_head_param_offset": [P(DiffusionDesc), i32],
            "tome_diffusion_head_workspace_bytes": [P(DiffusionDesc)],
            "tome_diffusion_head_fwd": [P(DiffusionDesc), vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp],
            "tome_diffusion_head_bwd": [P(DiffusionDesc), vp, vp, vp, vp, vp, vp, vp, vp],
            "tome_image_tokenizer_param_count": [P(ImageTokenizerDesc)],
            "tome_image_tokenizer_param_offset": [P(ImageTokenizerDesc), i32],
            "tome_image_tokenizer_workspace_bytes": [P(ImageTokenizerDesc)],
            "tome_image_tokenizer_fwd": [P(ImageTokenizerDesc), vp, vp, vp, vp, vp, vp, vp, C.c_size_t, vp],
            "tome_ddpm_step": [ll, vp, vp, vp, f32, f32, f32, f32, vp, vp],
            "tome_adamw_step": [ll, vp, vp, vp, vp, vp, f32, f32, f32, f32, f32, f32, i32, vp],
            "tome_cast_f32_to_bf16": [ll, vp, vp, vp],
            "tome_launch_count": [i32],
            "tome_profile_enable": [i32],
            "tome_profile_disable": [],
            "tome_profile_collect": [i32, P(f32), P(C.c_double), P(i32)],
            "tome_stack_param_count": [P(StackCfg)],
            "tome_stack_layer_offset": [P(StackCfg), i32],
            "tome_stack_workspace_bytes": [P(StackCfg)],
            "tome_stack_forward": [P(StackCfg), P(StackIO), vp],
            "tome_stack_backward": [P(StackCfg), P(StackIO), vp],
            "tome_stack_tokens_at": [P(StackCfg), i32],
            "tome_stack_final_x": [P(StackCfg), P(StackIO)],
            "tome_stack_final_size": [P(StackCfg), P(StackIO)],
            "tome_stack_layer_edge_idx": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_dst_idx": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_node_max": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_node_idx": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_relu_bits": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_x_in": [P(StackCfg), P(StackIO), i32],
            "tome_stack_layer_size_in": [P(StackCfg), P(StackIO), i32],
            "tome_num_sms": [],
        }
        for name, args in sig.items():
            getattr(L, name).argtypes = args
        for name in ("tome_gemm_force_tile", "tome_ln_force_cluster", "tome_attention_set_dq_from_ds"):
            getattr(L, name).restype = None
        _lib = L
    return _lib


PROF_TAGS = ["gemm", "attn_fwd", "attn_bwd", "merge_fwd", "merge_bwd", "sim_argmax", "select_topr", "layernorm", "colsum",
             "other", "importance", "prune"]


def profile_collect() -> dict:
    """{tag: (ms, work, count)} of the ops recorded since tome_profile_enable / the last collect."""
    n = len(PROF_TAGS)
    ms, work, cnt = (f32 * n)(), (C.c_double * n)(), (i32 * n)()
    check(lib().tome_profile_collect(n, ms, work, cnt))
    return {PROF_TAGS[i]: (float(ms[i]), float(work[i]), int(cnt[i])) for i in range(n)}


def check(rc: int) -> None:
    if rc != TOME_OK:
        raise TomeError(rc, lib().tome_last_error().decode())
