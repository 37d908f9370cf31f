"""Thin torch-tensor wrappers over the C ABI (include/tome_b200.h).

torch is plumbing only here: device memory, the current stream, dtype bookkeeping.  Every function launches the
hand-written sm_100a kernels through `libtome_b200.so`; nothing falls back to torch ops or to the CPU.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib as L


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dt(t: torch.Tensor) -> int:
    if t.dtype == torch.bfloat16:
        return L.TOME_BF16
    if t.dtype == torch.float32:
        return L.TOME_F32
    raise TypeError(f"unsupported dtype {t.dtype} (bf16 or fp32)")


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("multi_modal_transformers_tokenmerge_b200 runs on CUDA (sm_100a) only: got a CPU tensor. "
                               "There is no CPU fallback.")


def clamp_r(tokens: int, r: int, class_token: bool = False, distill_token: bool = False) -> int:
    """token_compression.py:60-67 (pure host arithmetic; does not need the GPU)."""
    return int(L.lib().tome_clamp_r(int(tokens), int(r), int(bool(class_token)), int(bool(distill_token))))


# ------------------------------------------------------------------------------------------------ matching
def token_sets(sets) -> Optional[L.TokenSets]:
    """tome_token_sets_t of `sets`, a sequence of (start, n, r) per token set (matching and merging stay inside each set; set s
    loses r tokens), or None: one set spanning the sequence."""
    if sets is None:
        return None
    sets = [tuple(int(v) for v in s_) for s_ in sets]
    if not 1 <= len(sets) <= L.MAX_TOKEN_SETS:
        raise ValueError(f"between 1 and {L.MAX_TOKEN_SETS} token sets are supported, got {len(sets)}")
    pad = lambda xs: (C.c_int32 * L.MAX_TOKEN_SETS)(*xs)  # noqa: E731
    return L.TokenSets(len(sets), pad([s_[0] for s_ in sets]), pad([s_[1] for s_ in sets]), pad([s_[2] for s_ in sets]))


def _sets_ptr(ts: Optional[L.TokenSets]):
    return None if ts is None else C.cast(C.pointer(ts), C.c_void_p)


@dataclass
class MatchPlan:
    """Device-resident index set of one bipartite matching (token_compression.py:84-88).  With token sets every array is
    concatenated set by set and its indices are local to the set (include/tome_b200.h); row_map holds global output rows."""

    batch: int
    tokens: int
    r: int
    distill_token: bool
    node_max: torch.Tensor  # [B,Ta] f32
    node_idx: torch.Tensor  # [B,Ta] i32
    edge_idx: torch.Tensor  # [B,Ta] i32
    dst_idx: torch.Tensor   # [B,r] i32
    row_map: torch.Tensor   # [B,T] i32
    dst_off: torch.Tensor   # [B,Tb+1] i32
    dst_src: torch.Tensor   # [B,r] i32
    scores: Optional[torch.Tensor] = None
    sets: Optional[tuple] = None   # ((start, n, r), ...) or None: one set

    @property
    def src_idx(self):
        return self.edge_idx[:, : self.r]

    @property
    def unm_idx(self):
        return self.edge_idx[:, self.r:]

    def c_plan(self) -> L.Plan:
        return L.Plan(self.edge_idx.data_ptr(), self.dst_idx.data_ptr(), self.row_map.data_ptr(),
                      self.dst_off.data_ptr(), self.dst_src.data_ptr())


def _scratch(nbytes: int, device, buf: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 device view of at least `nbytes` bytes whose data pointer is 256-byte aligned (the library's workspaces): a
    slice of `buf` (uint8, nbytes + 256 bytes or more) or of a new allocation of that size, so it keeps the storage alive."""
    if buf is None:
        buf = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
    assert buf.numel() >= nbytes + 256, (buf.numel(), nbytes)
    return buf[(-buf.data_ptr()) % 256:]


def sim_argmax(src: torch.Tensor, *, heads: int = 1, dim: Optional[int] = None, batch_stride=None, token_stride=None,
               head_stride=None, tokens=None, batch=None, class_token=False, distill_token=False, dump_scores=False,
               offset_elems: int = 0, sets=None):
    """K1.  `src` is either a [B,T,Dm] metric (heads=1) or a packed buffer addressed by the given strides.
    sets: ((start, n, r), ...) to match inside each token set; node_max / node_idx are then [B, sum ceil(n/2)] (indices local
    to the set) and the scores dump [B, sum ceil(n/2) * floor(n/2)], each set's block row-major in turn."""
    _need_cuda(src)
    if heads == 1 and dim is None:
        assert src.dim() == 3 and src.is_contiguous()
        batch, tokens, dim = src.shape
        batch_stride, token_stride, head_stride = tokens * dim, dim, 0
    ts = token_sets(sets)
    if ts is None:
        ta, tb = (tokens + 1) // 2, tokens // 2
        score_shape = (batch, ta, tb)
    else:
        ta = sum((int(n) + 1) // 2 for _, n, _ in sets)
        score_shape = (batch, sum(((int(n) + 1) // 2) * (int(n) // 2) for _, n, _ in sets))
    node_max = torch.empty(batch, ta, dtype=torch.float32, device=src.device)
    node_idx = torch.empty(batch, ta, dtype=torch.int32, device=src.device)
    scores = torch.empty(score_shape, dtype=torch.float32, device=src.device) if dump_scores else None
    d = L.MetricDesc(batch, tokens, dim, heads, _dt(src), batch_stride, token_stride, head_stride,
                     int(bool(class_token)), int(bool(distill_token)), _sets_ptr(ts))
    base = C.c_void_p(src.data_ptr() + offset_elems * src.element_size())
    ws = _scratch(L.lib().tome_sim_argmax_workspace_bytes(C.byref(d)), src.device)
    L.check(L.lib().tome_sim_argmax(C.byref(d), base, _ptr(node_max), _ptr(node_idx), _ptr(scores), _ptr(ws), ws.numel(),
                                    _stream()))
    return node_max, node_idx, scores


def select_topr(node_max: torch.Tensor, node_idx: torch.Tensor, tokens: int, r: Optional[int] = None, distill_token=False,
                sets=None) -> MatchPlan:
    """K2.  `r` must already be clamped and >= 1.  sets: ((start, n, r), ...) as for sim_argmax, whose node_max / node_idx
    this takes; r defaults to (and must equal) the sum of the sets' r."""
    _need_cuda(node_max, node_idx)
    b = node_max.shape[0]
    ts = token_sets(sets)
    if ts is None:
        ta, n_off = (tokens + 1) // 2, tokens // 2 + 1
    else:
        sets = tuple(tuple(int(v) for v in s_) for s_ in sets)
        r = sum(s_[2] for s_ in sets) if r is None else r
        ta, n_off = sum((n + 1) // 2 for _, n, _ in sets), sum(n // 2 + 1 for _, n, _ in sets)
    dev = node_max.device
    i32 = torch.int32
    plan = MatchPlan(b, tokens, r, bool(distill_token), node_max, node_idx,
                     torch.empty(b, ta, dtype=i32, device=dev), torch.empty(b, r, dtype=i32, device=dev),
                     torch.empty(b, tokens, dtype=i32, device=dev), torch.empty(b, n_off, dtype=i32, device=dev),
                     torch.empty(b, r, dtype=i32, device=dev), sets=sets)
    shp = L.PlanShape(b, tokens, r, int(bool(distill_token)), _sets_ptr(ts))
    cp = plan.c_plan()
    L.check(L.lib().tome_select_topr(C.byref(shp), _ptr(node_max), _ptr(node_idx), C.byref(cp), _stream()))
    return plan


def merge_fwd(plan: MatchPlan, x: torch.Tensor, size: Optional[torch.Tensor], mode: int, gid=None, pos=None):
    """K3.  x [B,T,C] (bf16/fp32, contiguous); size f32 [B,T] or None.  Returns (x_out, size_out, gid_out, pos_out).
    A plan of select_topr(sets=...) merges inside each token set (its sets travel with the plan)."""
    _need_cuda(x, size)
    assert x.is_contiguous() and x.dim() == 3
    b, t, c = x.shape
    assert t == plan.tokens and b == plan.batch
    to = t - plan.r
    x_out = torch.empty(b, to, c, dtype=x.dtype, device=x.device)
    size_out = torch.empty(b, to, dtype=torch.float32, device=x.device) if mode == L.TOME_MERGE_WAVG else None
    gid_out = torch.empty(b, to, dtype=torch.uint8, device=x.device) if gid is not None else None
    pos_out = torch.empty(b, to, dtype=torch.int32, device=x.device) if pos is not None else None
    ts = token_sets(plan.sets)
    shp = L.MergeShape(b, t, c, plan.r, int(plan.distill_token), _dt(x), mode, _sets_ptr(ts))
    cp = plan.c_plan()
    L.check(L.lib().tome_merge_fwd(C.byref(shp), C.byref(cp), _ptr(x), _ptr(size), _ptr(x_out), _ptr(size_out),
                                   _ptr(gid), _ptr(pos), _ptr(gid_out), _ptr(pos_out), _stream()))
    return x_out, size_out, gid_out, pos_out


def merge_bwd(plan: MatchPlan, dy: torch.Tensor, size: Optional[torch.Tensor], size_out: Optional[torch.Tensor], mode: int):
    """K4.  dy [B,T-r,C] -> dx [B,T,C].  mode SUM == ToMe `unmerge`."""
    _need_cuda(dy)
    assert dy.is_contiguous()
    b, to, c = dy.shape
    t = plan.tokens
    dx = torch.empty(b, t, c, dtype=dy.dtype, device=dy.device)
    ts = token_sets(plan.sets)
    shp = L.MergeShape(b, t, c, plan.r, int(plan.distill_token), _dt(dy), mode, _sets_ptr(ts))
    cp = plan.c_plan()
    L.check(L.lib().tome_merge_bwd(C.byref(shp), C.byref(cp), _ptr(size), _ptr(size_out), _ptr(dy), _ptr(dx), _stream()))
    return dx


# ------------------------------------------------------------------------------------------------ dense
def topk_prune(emb: torch.Tensor, importance: torch.Tensor, set_start, set_n, set_k):
    """K9.  emb [B,T,C] (bf16 / fp32), importance fp32 [B,T] or [P,B,T] (planes summed in order).
    Returns (out [B, sum k, C], ids int32 [B, sum k])."""
    _need_cuda(emb, importance)
    assert emb.dim() == 3 and emb.is_contiguous() and importance.is_contiguous() and importance.dtype == torch.float32
    b, t, c = emb.shape
    planes = 1 if importance.dim() == 2 else importance.shape[0]
    assert tuple(importance.shape[-2:]) == (b, t), (importance.shape, emb.shape)
    ns = len(set_k)
    if not (1 <= ns <= 16):
        raise ValueError(f"between 1 and 16 token sets are supported, got {ns}")
    d = L.PruneDesc(b, t, c, _dt(emb), ns, (C.c_int32 * 16)(*set_start), (C.c_int32 * 16)(*set_n), (C.c_int32 * 16)(*set_k), planes)
    ktot = int(sum(set_k))
    out = torch.empty(b, ktot, c, dtype=emb.dtype, device=emb.device)
    ids = torch.empty(b, ktot, dtype=torch.int32, device=emb.device)
    L.check(L.lib().tome_topk_prune(C.byref(d), _ptr(emb), _ptr(importance), _ptr(out), _ptr(ids), _stream()))
    return out, ids


def gemm(a: torch.Tensor, b: torch.Tensor, *, m: int, n: int, k: int, a_major=L.TOME_MAJOR_K, b_major=L.TOME_MAJOR_K,
         lda=None, ldb=None, out: Optional[torch.Tensor] = None, out_dtype=torch.bfloat16, bias=None, residual=None,
         gate=None, gate_scale=1.0, relu=False, dropout_rate=0.0, dropout_seed=0, dropout_site=0, k_splits=0,
         accumulate=False, gate_bits: Optional[torch.Tensor] = None,
         relu_bits_out: Optional[torch.Tensor] = None, colsum_partial: Optional[torch.Tensor] = None,
         a_row_shift=None) -> torch.Tensor:
    """C[M,N] = epilogue(A * B^T) on tcgen05.  a/b are 2-D bf16 tensors whose rows are M/N (K-major) or K (MN-major).
    gate_bits / relu_bits_out: int32 [M, ceil(N/32)] one-bit-per-element ReLU gates (see include/tome_b200.h).
    a_row_shift: list of row shifts, one per group of k / len(a_row_shift) reduction columns (row-shifted A windows: a
    convolution over a flattened, zero-bordered grid without im2col rows; a is [M, k / groups])."""
    _need_cuda(a, b)
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16
    lda = a.stride(0) if lda is None else lda
    ldb = b.stride(0) if ldb is None else ldb
    if out is None:
        out = torch.empty(m, n, dtype=out_dtype, device=a.device)
    args = L.GemmArgs(m, n, k, a.data_ptr(), lda, a_major, b.data_ptr(), ldb, b_major, out.data_ptr(), out.stride(0),
                      _dt(out), None if bias is None else bias.data_ptr(),
                      None if residual is None else residual.data_ptr(), 0 if residual is None else residual.stride(0),
                      None if gate is None else gate.data_ptr(), 0 if gate is None else gate.stride(0),
                      float(gate_scale), int(relu), float(dropout_rate), int(dropout_seed), int(dropout_site),
                      int(k_splits), int(accumulate),
                      None if gate_bits is None else gate_bits.data_ptr(),
                      None if relu_bits_out is None else relu_bits_out.data_ptr(),
                      0 if (gate_bits is None and relu_bits_out is None) else (gate_bits if gate_bits is not None else relu_bits_out).stride(0),
                      None if colsum_partial is None else colsum_partial.data_ptr())
    if a_row_shift is not None:
        shifts = (C.c_int * len(a_row_shift))(*[int(v) for v in a_row_shift])
        args.a_row_shift, args.a_shift_groups = C.cast(shifts, C.c_void_p), len(a_row_shift)
    ws_bytes = L.lib().tome_gemm_workspace_bytes(C.byref(args))
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=a.device) if ws_bytes else None
    L.check(L.lib().tome_gemm_bf16(C.byref(args), _ptr(ws), ws_bytes, _stream()))
    return out


def reduce_rows(partial: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate=False) -> torch.Tensor:
    """out[n] (+)= sum_r partial[r, n] (f32, fixed order): second stage of the column sums a GEMM epilogue leaves."""
    _need_cuda(partial)
    assert partial.dtype == torch.float32 and partial.is_contiguous() and partial.dim() == 2
    rows, n = partial.shape
    if out is None:
        out = torch.zeros(n, dtype=torch.float32, device=partial.device)
    L.check(L.lib().tome_reduce_rows_f32(rows, n, _ptr(partial), _ptr(out), int(accumulate), _stream()))
    return out


def colsum(x: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate=False) -> torch.Tensor:
    _need_cuda(x)
    m, n = x.shape
    rows = L.lib().tome_colsum_workspace_rows(m)
    ws = torch.empty(rows, n, dtype=torch.float32, device=x.device)
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=x.device)
    L.check(L.lib().tome_colsum_bf16(m, n, _ptr(x), x.stride(0), _ptr(out), int(accumulate), _ptr(ws), _stream()))
    return out


def dropout_colsum(x: torch.Tensor, rate: float, seed: int, site: int, out: Optional[torch.Tensor] = None, accumulate=False):
    """y = dropout(x) with the GEMM epilogue's mask for (seed, site, element) and the column sums of y, in one pass.
    x bf16 [M, N] contiguous.  Returns (y, colsum fp32 [N])."""
    _need_cuda(x)
    assert x.dim() == 2 and x.is_contiguous() and x.dtype == torch.bfloat16
    m, n = x.shape
    y = torch.empty_like(x)
    if out is None:
        out = torch.zeros(n, dtype=torch.float32, device=x.device)
    ws = torch.empty(L.lib().tome_colsum_workspace_rows(m), n, dtype=torch.float32, device=x.device)
    L.check(L.lib().tome_dropout_colsum_bf16(m, n, _ptr(x), _ptr(y), float(rate), int(seed), int(site), _ptr(out), int(accumulate),
                                             _ptr(ws), _stream()))
    return y, out


def layernorm_fwd(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float = 1e-6, axis: int = 1):
    _need_cuda(x)
    assert x.dtype == torch.bfloat16 and x.is_contiguous()
    b, t, c = x.shape
    y = torch.empty_like(x)
    stat_shape = (b, c) if axis == 1 else (b, t)
    mean = torch.empty(stat_shape, dtype=torch.float32, device=x.device)
    rstd = torch.empty(stat_shape, dtype=torch.float32, device=x.device)
    L.check(L.lib().tome_layernorm_fwd(b, t, c, axis, eps, _ptr(x), _ptr(gamma), _ptr(beta), _ptr(y), _ptr(mean),
                                       _ptr(rstd), _stream()))
    return y, mean, rstd


def layernorm_bwd(x, dy, gamma, mean, rstd, dgamma, dbeta, dres=None, axis: int = 1):
    _need_cuda(x, dy)
    b, t, c = x.shape
    dx = torch.empty_like(x)
    rows = b if axis == 1 else L.lib().tome_colsum_workspace_rows(b * t)
    partial = torch.empty(2, rows, c, dtype=torch.float32, device=x.device)
    L.check(L.lib().tome_layernorm_bwd(b, t, c, axis, _ptr(x), _ptr(dy), _ptr(gamma), _ptr(mean), _ptr(rstd), _ptr(dres),
                                       _ptr(dx), _ptr(dgamma), _ptr(dbeta), _ptr(partial), _stream()))
    return dx


# ------------------------------------------------------------------------------------------------ attention
def _attn_desc(q, k, v, out, scale, gid, pos, allow, size, dropout=(0.0, 0, 0)):
    b, t, h, d = q.shape
    for x in (q, k, v, out):
        assert x.dtype == torch.bfloat16 and x.stride(3) == 1 and x.stride(2) == d, "heads must be packed [.., H, D]"
    g = 0 if allow is None else allow.shape[0]
    return L.AttnDesc(b, t, h, d, q.stride(0), q.stride(1), k.stride(0), k.stride(1), v.stride(0), v.stride(1),
                      out.stride(0), out.stride(1), float(scale),
                      None if gid is None else gid.data_ptr(), None if pos is None else pos.data_ptr(),
                      None if allow is None else allow.data_ptr(), g, None if size is None else size.data_ptr(),
                      float(dropout[0]), int(dropout[1]), int(dropout[2]))


def attention_fwd(q, k, v, *, gid=None, pos=None, allow=None, size=None, scale=None, dropout_rate=0.0, dropout_seed=0,
                  dropout_site=0):
    """q,k,v: [B,T,H,D] bf16 views (may be slices of a packed qkv buffer).  Returns (out [B,T,H,D], lse [B,H,T]).
    dropout_*: attention-weight dropout, one mask for all batch rows and heads (flax broadcast_dropout=True)."""
    _need_cuda(q, k, v)
    b, t, h, d = q.shape
    scale = 1.0 / math.sqrt(d) if scale is None else scale
    out = torch.empty(b, t, h, d, dtype=torch.bfloat16, device=q.device)
    lse = torch.empty(b, h, t, dtype=torch.float32, device=q.device)
    desc = _attn_desc(q, k, v, out, scale, gid, pos, allow, size, (dropout_rate, dropout_seed, dropout_site))
    ws = _scratch(L.lib().tome_attention_workspace_bytes(C.byref(desc)), q.device)
    L.check(L.lib().tome_attention_fwd(C.byref(desc), _ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(lse), _ptr(ws), ws.numel(),
                                       _stream()))
    return out, lse


def attention_bwd(q, k, v, out, lse, dout, *, gid=None, pos=None, allow=None, size=None, scale=None, dqkv=None,
                  dropout_rate=0.0, dropout_seed=0, dropout_site=0, bias_partial: Optional[torch.Tensor] = None):
    """Returns (dq, dk, dv) [B,T,H,D] bf16 (views of one packed [B,T,3,H,D] buffer unless dqkv views are given).
    bias_partial: optional f32 [B * ceil(T / 128), 3 * H * D]; receives per-128-token-tile column sums of dq | dk | dv (the
    packed projection's bias gradient once reduced over rows with reduce_rows)."""
    _need_cuda(q, k, v, out, dout)
    b, t, h, d = q.shape
    scale = 1.0 / math.sqrt(d) if scale is None else scale
    if dqkv is None:
        buf = torch.empty(b, t, 3, h, d, dtype=torch.bfloat16, device=q.device)
        dq, dk, dv = buf[:, :, 0], buf[:, :, 1], buf[:, :, 2]
    else:
        dq, dk, dv = dqkv
    desc = _attn_desc(q, k, v, out, scale, gid, pos, allow, size, (dropout_rate, dropout_seed, dropout_site))
    gs = L.AttnGradStrides(dq.stride(0), dq.stride(1), dk.stride(0), dk.stride(1), dv.stride(0), dv.stride(1),
                           dout.stride(0), dout.stride(1))
    if bias_partial is not None:
        assert bias_partial.dtype == torch.float32 and bias_partial.is_contiguous()
        assert bias_partial.shape == (b * ((t + 127) // 128), 3 * h * d)
        gs.bias_partial, gs.bias_partial_ld = bias_partial.data_ptr(), 3 * h * d
        gs.bias_q_col, gs.bias_k_col, gs.bias_v_col = 0, h * d, 2 * h * d
    ws = _scratch(L.lib().tome_attention_bwd_workspace_bytes(C.byref(desc)), q.device)
    L.check(L.lib().tome_attention_bwd(C.byref(desc), C.byref(gs), _ptr(q), _ptr(k), _ptr(v), _ptr(out), _ptr(lse),
                                       _ptr(dout), _ptr(dq), _ptr(dk), _ptr(dv), _ptr(ws), ws.numel(), _stream()))
    return dq, dk, dv


# ------------------------------------------------------------------------------------------------ action heads
@dataclass
class HeadState:
    """What tome_action_head_fwd leaves behind for the backward call."""

    desc: "L.HeadDesc"
    origin: torch.Tensor
    w: torch.Tensor
    workspace: torch.Tensor


def action_head_fwd(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], *, kind: int, max_action: float,
                    groups: int = 1, origin: Optional[torch.Tensor] = None, actions: Optional[torch.Tensor] = None,
                    keep_for_backward: bool = False):
    """Pooled-readout action head + loss (continuous.py:16-25 / categorical.py:30-40, octo.py:157-190).

    x [B, tokens, C] bf16 / f32; origin i32 [B, n_readout] = rows of x holding the readouts (default: every row).
    Returns (out f32 [B, groups, features], loss f32 [1 + B] or None, HeadState or None)."""
    _need_cuda(x, w, bias, origin, actions)
    B, T, Cc = x.shape
    assert x.is_contiguous() and w.dtype == torch.float32 and w.is_contiguous() and w.shape[0] == Cc
    if origin is None:
        origin = torch.arange(T, dtype=torch.int32, device=x.device).repeat(B, 1)
    assert origin.dtype == torch.int32 and origin.is_contiguous() and origin.shape[0] == B
    feats = int(w.shape[1])
    d = L.HeadDesc(B, T, Cc, _dt(x), int(origin.shape[1]), int(groups), feats, int(kind), float(max_action))
    out = torch.empty(B, groups, feats, dtype=torch.float32, device=x.device)
    loss = None
    if actions is not None:
        assert actions.dtype == torch.float32 and actions.is_contiguous()
        want = (B, feats) if kind == L.HEAD_CONTINUOUS_L2 else (B, groups)
        assert tuple(actions.shape) == want, (actions.shape, want)
        loss = torch.zeros(1 + B, dtype=torch.float32, device=x.device)
    ws, nbytes = None, 0
    if keep_for_backward:
        nbytes = int(L.lib().tome_action_head_workspace_bytes(C.byref(d)))
        if nbytes == 0:
            L.check(1)
        ws = _scratch(nbytes, x.device)
    L.check(L.lib().tome_action_head_fwd(C.byref(d), _ptr(x), _ptr(origin), _ptr(w), _ptr(bias), _ptr(actions), _ptr(out),
                                         _ptr(loss), _ptr(ws), nbytes, _stream()))
    return out, loss, (HeadState(d, origin, w, ws) if keep_for_backward else None)


def action_head_bwd(state: HeadState, dw: torch.Tensor, dbias: Optional[torch.Tensor], want_dx: bool = True):
    """Accumulates into dw [C, features] / dbias [features]; returns dx (x's dtype and shape) or None."""
    d = state.desc
    dx = None
    if want_dx:
        dx = torch.empty(d.batch, d.tokens, d.channels, dtype=torch.bfloat16 if d.x_dtype == L.TOME_BF16 else torch.float32,
                         device=dw.device)
    L.check(L.lib().tome_action_head_bwd(C.byref(d), _ptr(state.origin), _ptr(state.w), _ptr(state.workspace), _ptr(dw),
                                         _ptr(dbias), _ptr(dx), _stream()))
    return dx


@dataclass
class DiffusionState:
    desc: "L.DiffusionDesc"
    params: torch.Tensor
    params_bf16: torch.Tensor
    origin: torch.Tensor
    time: torch.Tensor
    workspace: torch.Tensor


def diffusion_head_fwd(x: torch.Tensor, params: torch.Tensor, desc: "L.DiffusionDesc", actions: torch.Tensor, noise: torch.Tensor,
                       time: torch.Tensor, alpha_hats: torch.Tensor, origin: Optional[torch.Tensor] = None):
    """DiffusionActionHead.denoise_loss (diffusion.py:114-143) on the final sequence x bf16 [B, tokens, C].
    params: flat fp32 vector in the layout of include/tome_b200.h.  Returns (pred [B, A], loss [1 + B], state)."""
    _need_cuda(x, params, actions, noise, time, alpha_hats, origin)
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and params.dtype == torch.float32
    B, T, _ = x.shape
    if origin is None:
        origin = torch.arange(T, dtype=torch.int32, device=x.device).repeat(B, 1)
    n = int(L.lib().tome_diffusion_head_param_count(C.byref(desc)))
    if n < 0:
        L.check(1)
    assert params.numel() == n, (params.numel(), n)
    p16 = params.to(torch.bfloat16)
    nbytes = int(L.lib().tome_diffusion_head_workspace_bytes(C.byref(desc)))
    ws = _scratch(nbytes, x.device)
    pred = torch.empty(B, desc.action_dim, dtype=torch.float32, device=x.device)
    loss = torch.zeros(1 + B, dtype=torch.float32, device=x.device)
    for t, dt in ((actions, torch.float32), (noise, torch.float32), (time, torch.int32), (alpha_hats, torch.float32)):
        assert t.dtype == dt and t.is_contiguous()
    L.check(L.lib().tome_diffusion_head_fwd(C.byref(desc), _ptr(params), _ptr(p16), _ptr(x), _ptr(origin), _ptr(actions), _ptr(noise),
                                            _ptr(time), _ptr(alpha_hats), _ptr(pred), _ptr(loss), _ptr(ws), nbytes, _stream()))
    return pred, loss, DiffusionState(desc, params, p16, origin, time, ws)


def diffusion_head_bwd(state: DiffusionState, grads: torch.Tensor, want_dx: bool = True):
    d = state.desc
    dx = torch.empty(d.batch, d.tokens, d.channels, dtype=torch.bfloat16, device=grads.device) if want_dx else None
    L.check(L.lib().tome_diffusion_head_bwd(C.byref(d), _ptr(state.params), _ptr(state.params_bf16), _ptr(state.origin),
                                            _ptr(state.time), _ptr(state.workspace), _ptr(grads), _ptr(dx), _stream()))
    return dx


# ------------------------------------------------------------------------------------------------ image front end
def image_tokenizer_fwd(image: torch.Tensor, params: torch.Tensor, desc: "L.ImageTokenizerDesc", row_tokens: torch.Tensor,
                        col_tokens: torch.Tensor, params_bf16: Optional[torch.Tensor] = None, workspace: Optional[torch.Tensor] = None):
    """ImageTokenizer.__call__ (tokenizers/images/image_tokenizer.py:216-309) on image [B, N, H, W, C] (uint8 or fp32 pixels).
    params: flat fp32 vector in the layout of include/tome_b200.h section 7b; row_tokens / col_tokens i32 [token_rows, n_patches].
    Returns tokens [B, N, n_patches, E] in desc.out_dtype."""
    _need_cuda(image, params, row_tokens, col_tokens, params_bf16)
    assert image.is_contiguous() and image.dim() == 5 and params.dtype == torch.float32
    assert image.dtype == (torch.uint8 if desc.image_dtype == L.TOME_U8 else torch.float32)
    n = int(L.lib().tome_image_tokenizer_param_count(C.byref(desc)))
    if n < 0:
        L.check(1)
    assert params.numel() == n, (params.numel(), n)
    p16 = params.to(torch.bfloat16) if params_bf16 is None else params_bf16
    nbytes = int(L.lib().tome_image_tokenizer_workspace_bytes(C.byref(desc)))
    ws = _scratch(nbytes, image.device, workspace)
    n_patches = (desc.image_size // desc.patch_size) ** 2
    for t in (row_tokens, col_tokens):
        assert t.dtype == torch.int32 and t.is_contiguous() and t.numel() == desc.token_rows * n_patches
    out = torch.empty(desc.batch, desc.n_images, n_patches, desc.embed_dim, device=image.device,
                      dtype=torch.bfloat16 if desc.out_dtype == L.TOME_BF16 else torch.float32)
    L.check(L.lib().tome_image_tokenizer_fwd(C.byref(desc), _ptr(image), _ptr(params), _ptr(p16), _ptr(row_tokens), _ptr(col_tokens),
                                             _ptr(out), _ptr(ws), nbytes, _stream()))
    return out


# ------------------------------------------------------------------------------------------------ pruning path
def attention_importance(q: torch.Tensor, k: torch.Tensor, lse: torch.Tensor, mode: str = "received", size: Optional[torch.Tensor] = None,
                         gid: Optional[torch.Tensor] = None, pos: Optional[torch.Tensor] = None, allow: Optional[torch.Tensor] = None,
                         scale: Optional[float] = None) -> torch.Tensor:
    """compressed_attention.py:303-306 on q, k bf16 [B, T, H, D] (views into a packed qkv are fine) and the lse [B, H, T] of
    attention_fwd: importance f32 [B, T] = mean over heads of the mean over keys ("row_mean", as written) or over queries
    ("received") of the softmax weights.  gid / pos are per batch row [B, T]."""
    _need_cuda(q, k, lse, size, gid, pos, allow)
    B, T, H, D = q.shape
    assert q.dtype == k.dtype == torch.bfloat16 and q.stride(3) == 1 and k.stride(3) == 1 and q.stride(2) == D and k.stride(2) == D
    assert lse.dtype == torch.float32 and lse.is_contiguous() and tuple(lse.shape) == (B, H, T)
    d = L.AttnDesc(batch=B, tokens=T, heads=H, head_dim=D, q_batch_stride=q.stride(0), q_token_stride=q.stride(1),
                   k_batch_stride=k.stride(0), k_token_stride=k.stride(1), scale=float(scale if scale is not None else D ** -0.5))
    if gid is not None:
        assert gid.dtype == torch.uint8 and pos.dtype == torch.int32 and allow.dtype == torch.uint8
        assert tuple(gid.shape) == (B, T) and tuple(pos.shape) == (B, T) and gid.is_contiguous() and pos.is_contiguous()
        d.gid, d.pos, d.allow, d.num_groups = gid.data_ptr(), pos.data_ptr(), allow.data_ptr(), int(allow.shape[0])
    if size is not None:
        assert size.dtype == torch.float32 and size.is_contiguous() and tuple(size.shape) == (B, T)
        d.size = size.data_ptr()
    out = torch.empty(B, T, dtype=torch.float32, device=q.device)
    L.check(L.lib().tome_attention_importance(C.byref(d), _ptr(q), _ptr(k), _ptr(lse),
                                              {"row_mean": L.IMPORTANCE_ROW_MEAN, "received": L.IMPORTANCE_RECEIVED}[mode], _ptr(out), _stream()))
    return out


def prune_row_map(ids: torch.Tensor, tokens: int, gid: Optional[torch.Tensor] = None, pos: Optional[torch.Tensor] = None):
    """ids i32 [B, kept] -> (row_map i32 [B, tokens] with -1 for pruned tokens, gid_out, pos_out of the kept tokens)."""
    _need_cuda(ids, gid, pos)
    B, K = ids.shape
    rm = torch.empty(B, tokens, dtype=torch.int32, device=ids.device)
    go = None if gid is None else torch.empty(B, K, dtype=torch.uint8, device=ids.device)
    po = None if pos is None else torch.empty(B, K, dtype=torch.int32, device=ids.device)
    L.check(L.lib().tome_prune_row_map(B, tokens, K, _ptr(ids), _ptr(gid), _ptr(pos), _ptr(rm), _ptr(go), _ptr(po), _stream()))
    return rm, go, po


def prune_bwd(row_map: torch.Tensor, dy: torch.Tensor) -> torch.Tensor:
    """Backward of the top-k gather: dx [B, T, C] from dy [B, kept, C] (zero rows for pruned tokens)."""
    _need_cuda(row_map, dy)
    B, T = row_map.shape
    assert dy.is_contiguous() and dy.shape[0] == B
    dx = torch.empty(B, T, dy.shape[2], dtype=dy.dtype, device=dy.device)
    L.check(L.lib().tome_prune_bwd(B, T, dy.shape[1], dy.shape[2], _dt(dy), _ptr(row_map), _ptr(dy), _ptr(dx), _stream()))
    return dx
