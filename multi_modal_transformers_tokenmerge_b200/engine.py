"""Host-side owner of the buffers the native stack executor (csrc/stack.cu, `tome_stack_*`) works on.

`ToMeStackEngine` holds the flat fp32 master parameters, their bf16 working copy, the flat fp32 gradient vector, Adam
moments and the activation workspace, and drives forward / backward / optimiser step through the C ABI.  The
reference's counterpart is the Flax `TrainState` + `apply_fn` pair (models/octo/octo.py:326-386) around
`StackedEncoder1DBlock` (attention_blocks/attention.py:87-119); the drop-in modules in `attention_blocks/` sit on top
of this class.  torch is used for device memory, streams and (in `parallel.py`) NCCL only.
"""
from __future__ import annotations

import ctypes as C
import dataclasses
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import _lib as L
from .ops import _scratch

PARAM_ORDER = ["ln1_scale", "ln1_bias", "wqkv", "bqkv", "wo", "bo", "ln2_scale", "ln2_bias", "w1", "b1", "w2", "b2"]


@dataclass
class StackConfig:
    batch: int
    tokens: int
    channels: int
    heads: int
    head_dim: int
    mlp_dim: int
    layers: int
    r: int = 0
    ln_axis: int = 1            # 1 = tokens (what vanilla_decoder.yaml:10 says), 2 = features (conventional)
    ln_eps: float = 1e-6
    prop_attn: bool = True
    class_token: bool = False
    distill_token: bool = False
    num_groups: int = 0
    n_readout: int = 0
    dropout_rate: float = 0.0
    dropout_seed: int = 0
    attn_dropout_rate: float = 0.0   # attention-weight dropout (self_attention.dropout_rate, vanilla_decoder.yaml:23)
    head: str = "none"          # loss on the readouts: "none" = synthetic MSE, "continuous" (continuous.py + l2 loss,
                                # octo.py:157-165), "categorical" (categorical.py + cross-entropy, octo.py:178-190) or
                                # "diffusion" (diffusion.py:94-143 denoise loss)
    head_groups: int = 1        # categorical: action_space_dim
    head_features: int = 0      # continuous / diffusion: action dimensions; categorical: num_bins
    max_action: float = 1.0
    head_fourier_dim: int = 0   # diffusion: FourierFeatures.output_dim, time-encoder MLP widths, denoiser hidden width
    head_time_hidden: int = 0
    head_time_out: int = 0
    head_hidden: int = 0
    diffusion_steps: int = 0
    # per-modality top-k pruning per layer instead of merging (include/tome_b200.h: tome_stack_cfg_t.prune_*): token sets as
    # (tokens at layer 0, tokens dropped by every layer), in sequence order; importance: "row_mean" (compressed_attention.py:303-306
    # as written) or "received"
    prune_sets: tuple = ()
    prune_importance: str = "received"
    # with prune_sets: every layer MERGES its c tokens inside each set instead of pruning them (bipartite soft matching per
    # token set, merge_wavg; include/tome_b200.h tome_stack_cfg_t.set_merge), so no token merges across a set boundary
    set_merge: bool = False

    def c(self) -> L.StackCfg:
        return L.StackCfg(self.batch, self.tokens, self.channels, self.heads, self.head_dim, self.mlp_dim, self.layers,
                          self.r, self.ln_axis, self.ln_eps, int(self.prop_attn), int(self.class_token),
                          int(self.distill_token), self.num_groups, self.n_readout, self.dropout_rate, self.dropout_seed,
                          self.attn_dropout_rate, {"none": 0, "continuous": 1, "categorical": 2, "diffusion": 3}[self.head],
                          self.head_groups, self.head_features, self.max_action, self.head_fourier_dim, self.head_time_hidden,
                          self.head_time_out, self.head_hidden, self.diffusion_steps, len(self.prune_sets),
                          (C.c_int * 16)(*[int(n) for n, _ in self.prune_sets]), (C.c_int * 16)(*[int(c) for _, c in self.prune_sets]),
                          {"row_mean": L.IMPORTANCE_ROW_MEAN, "received": L.IMPORTANCE_RECEIVED}[self.prune_importance],
                          int(self.set_merge))

    def layer_sets(self, layer: int):
        """((start, n, r), ...) of the token sets entering `layer` of a set-merging stack, None for any other stack."""
        if not (self.set_merge and self.prune_sets):
            return None
        out, start = [], 0
        for n0, c in self.prune_sets:
            n = int(n0) - layer * int(c)
            out.append((start, n, int(c)))
            start += n
        return tuple(out)

    def diffusion_desc(self, tokens: int = 1) -> L.DiffusionDesc:
        return L.DiffusionDesc(self.batch, tokens, self.channels, self.n_readout, self.head_features, self.head_fourier_dim,
                               self.head_time_hidden, self.head_time_out, self.head_hidden, self.diffusion_steps)

    def diffusion_param_shapes(self) -> Dict[str, tuple]:
        a, f, ht, to, h = self.head_features, self.head_fourier_dim, self.head_time_hidden, self.head_time_out, self.head_hidden
        return dict(fourier_kernel=(f // 2, 1), tw1=(f, ht), tb1=(ht,), tw2=(ht, to), tb2=(to,),
                    w1=(a + to + self.channels, h), b1=(h,), w2=(h, a), b2=(a,))

    def param_shapes(self) -> Dict[str, tuple]:
        c, hd, f = self.channels, self.heads * self.head_dim, self.mlp_dim
        return dict(ln1_scale=(c,), ln1_bias=(c,), wqkv=(c, 3 * hd), bqkv=(3 * hd,), wo=(hd, c), bo=(c,),
                    ln2_scale=(c,), ln2_bias=(c,), w1=(c, f), b1=(f,), w2=(f, c), b2=(c,))


class ToMeStackEngine:
    """predict_only=True: a forward-only engine (tome_stack_predict) -- the predict workspace, no gradients, no Adam moments;
    `predict` runs it, and forward / backward / the optimiser and the per-layer accessors raise.  `predictor()` builds one
    from a training engine that shares its parameters."""

    def __init__(self, cfg: StackConfig, device="cuda", gid=None, pos=None, allow=None, readout_idx=None,
                 training: bool = True, layer_gid=None, layer_pos=None, predict_only: bool = False, _params=None):
        if not torch.cuda.is_available():
            raise RuntimeError("ToMeStackEngine needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = L.lib()
        self.cfg = cfg
        self.dev = torch.device(device)
        self.ccfg = cfg.c()
        self.predict_only = bool(predict_only)
        n = self.lib.tome_stack_param_count(C.byref(self.ccfg))
        if n < 0:
            L.check(1)
        self.n_params = int(n)
        if _params is not None:   # predictor(): the training engine's storage, not a copy
            self.params, self.params_bf16 = _params
            assert self.params.numel() == self.n_params and self.params_bf16.numel() == self.n_params
        else:
            self.params = torch.zeros(self.n_params, dtype=torch.float32, device=self.dev)
            self.params_bf16 = torch.zeros(self.n_params, dtype=torch.bfloat16, device=self.dev)
        self.grads = (torch.zeros(self.n_params, dtype=torch.float32, device=self.dev)
                      if training and not self.predict_only else None)
        self.adam_m = self.adam_v = None
        self.step_count = 0
        # adamw_step options: the gradient norm (device f32 [1]), {applied, skipped} counters, the decay mask, the norm scratch
        self.grad_norm = (torch.zeros(1, dtype=torch.float32, device=self.dev) if self.grads is not None else None)
        self._opt_steps = self._decay_ranges = self._adam_ws = None
        if self.predict_only:
            ws = self.lib.tome_stack_predict_workspace_bytes(C.byref(self.ccfg))
            if ws == 0:
                L.check(L.TOME_ERR_UNSUPPORTED)
        else:
            ws = self.lib.tome_stack_workspace_bytes(C.byref(self.ccfg))
        self.workspace = _scratch(ws, self.dev)
        self._ws_bytes = ws
        self.gid = None if gid is None else torch.as_tensor(np.asarray(gid, np.uint8)).to(self.dev)
        self.pos = None if pos is None else torch.as_tensor(np.asarray(pos, np.int32)).to(self.dev)
        self.allow = None if allow is None else torch.as_tensor(np.asarray(allow, np.uint8)).contiguous().to(self.dev)
        self.readout_idx = None if readout_idx is None else torch.as_tensor(np.asarray(readout_idx, np.int32)).to(self.dev)
        # pruning stacks: the compression grammar's per-layer masks, layer after layer (token_sequencer.py:222-238)
        self.layer_gid = None if layer_gid is None else torch.as_tensor(np.concatenate([np.asarray(g, np.uint8) for g in layer_gid])).to(self.dev)
        self.layer_pos = None if layer_pos is None else torch.as_tensor(np.concatenate([np.asarray(g, np.int32) for g in layer_pos])).to(self.dev)
        self.loss = torch.zeros(1 + cfg.batch, dtype=torch.float32, device=self.dev)
        self.readout = (torch.empty(cfg.batch, cfg.n_readout, cfg.channels, dtype=torch.float32, device=self.dev)
                        if cfg.n_readout else None)
        self.head_out = (torch.empty(cfg.batch, cfg.head_groups, cfg.head_features, dtype=torch.float32, device=self.dev)
                         if cfg.head != "none" else None)
        self.head_time = self.alpha_hats = None     # diffusion head: set_diffusion_draws()
        self._x = self._target = None
        self._events = None
        self._base_seed = int(cfg.dropout_seed)
        self._grad_trace = None

    # ------------------------------------------------------------------ parameters
    def layer_offset(self, layer: int) -> int:
        return int(self.lib.tome_stack_layer_offset(C.byref(self.ccfg), layer))

    def param_views(self, flat: torch.Tensor) -> Dict[str, object]:
        """Named views into a flat vector with the executor's layout: pos_embedding + per-layer dicts."""
        cfg = self.cfg
        out = {"pos_embedding": flat[: cfg.tokens * cfg.channels].view(cfg.tokens, cfg.channels), "layers": []}
        shapes = cfg.param_shapes()
        for l in range(cfg.layers):
            off = self.layer_offset(l)
            d = {}
            for name in PARAM_ORDER:
                n = int(np.prod(shapes[name]))
                d[name] = flat[off: off + n].view(*shapes[name])
                off += n
            out["layers"].append(d)
        if cfg.head == "diffusion":   # the diffusion head's own vector (include/tome_b200.h), after the last layer
            off = int(self.lib.tome_stack_head_offset(C.byref(self.ccfg)))
            dd = cfg.diffusion_desc()
            shapes_d = cfg.diffusion_param_shapes()
            out["head"] = {}
            for i, name in enumerate(L.DIFFUSION_PARAMS):
                o = off + int(self.lib.tome_diffusion_head_param_offset(C.byref(dd), i))
                out["head"][name] = flat[o: o + int(np.prod(shapes_d[name]))].view(*shapes_d[name])
        elif cfg.head != "none":  # Dense kernel [C, features] + bias [features] of the action head, after the last layer
            off = int(self.lib.tome_stack_head_offset(C.byref(self.ccfg)))
            n = cfg.channels * cfg.head_features
            out["head"] = {"kernel": flat[off: off + n].view(cfg.channels, cfg.head_features),
                           "bias": flat[off + n: off + n + cfg.head_features]}
        return out

    def load_params(self, pos_embedding, layers: Sequence[dict], head: Optional[dict] = None) -> None:
        """`layers[l]` uses the oracle / Flax names: ln1_scale, ln1_bias, wq, bq, wk, bk, wv, bv, wo, bo, ln2_*, w1, b1, w2, b2
        (kernels [in, out]); or already-fused wqkv / bqkv."""
        v = self.param_views(self.params)
        v["pos_embedding"].copy_(torch.as_tensor(np.asarray(pos_embedding, np.float32)).reshape(self.cfg.tokens, -1))
        for l, src in enumerate(layers):
            src = {k: torch.as_tensor(np.asarray(t, np.float32)) for k, t in src.items()}
            if "wqkv" not in src:
                src["wqkv"] = torch.cat([src["wq"], src["wk"], src["wv"]], dim=1)
                src["bqkv"] = torch.cat([src["bq"], src["bk"], src["bv"]], dim=0)
            for name in PARAM_ORDER:
                v["layers"][l][name].copy_(src[name])
        if head is not None:
            for name, t in v["head"].items():
                t.copy_(torch.as_tensor(np.asarray(head[name], np.float32)).reshape(t.shape))
        self.sync_bf16()

    def init_params(self, seed: int = 1) -> None:
        """he_normal kernels, N(0, 0.01) biases (vanilla_decoder.yaml:25-29,38-42), pos-embedding N(0, 0.02)
        (attention.py:98); generated on the device."""
        g = torch.Generator(device=self.dev)
        g.manual_seed(seed)
        v = self.param_views(self.params)
        v["pos_embedding"].normal_(0.0, 0.02, generator=g)
        for d in v["layers"]:
            for name, t in d.items():
                if name.startswith("w"):
                    t.normal_(0.0, (2.0 / t.shape[0]) ** 0.5, generator=g)
                elif name.endswith("scale"):
                    t.fill_(1.0)
                elif name.startswith("ln"):
                    t.zero_()
                else:
                    t.normal_(0.0, 0.01, generator=g)
        for name, t in v.get("head", {}).items():   # he_normal kernels / normal(0.01) biases (diffusion.yaml, vanilla_decoder.yaml)
            if t.dim() == 2:
                t.normal_(0.0, (2.0 / t.shape[0]) ** 0.5, generator=g)
            else:
                t.normal_(0.0, 0.01, generator=g)
        self.sync_bf16()

    def sync_bf16(self) -> None:
        L.check(self.lib.tome_cast_f32_to_bf16(self.n_params, self.params.data_ptr(), self.params_bf16.data_ptr(), self._stream()))

    # ------------------------------------------------------------------ execution
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def _io(self, x, target) -> L.StackIO:
        ev = None
        if self._events is not None:
            ev = (C.c_void_p * len(self._events))(*[e.cuda_event for e in self._events])
            self._ev_keepalive = ev
        return L.StackIO(self.params.data_ptr(), self.params_bf16.data_ptr(), x.data_ptr(),
                         L.TOME_BF16 if x.dtype == torch.bfloat16 else L.TOME_F32,
                         None if self.gid is None else self.gid.data_ptr(), None if self.pos is None else self.pos.data_ptr(),
                         None if self.allow is None else self.allow.data_ptr(),
                         None if self.readout_idx is None else self.readout_idx.data_ptr(),
                         None if target is None else target.data_ptr(),
                         self.workspace.data_ptr(), self._ws_bytes, None,
                         None if self.readout is None else self.readout.data_ptr(), self.loss.data_ptr(),
                         None if self.grads is None else self.grads.data_ptr(),
                         None if ev is None else C.cast(ev, C.POINTER(C.c_void_p)),
                         None if self.head_out is None else self.head_out.data_ptr(),
                         None if self.head_time is None else self.head_time.data_ptr(),
                         None if self.alpha_hats is None else self.alpha_hats.data_ptr(),
                         None if self._grad_trace is None else self._grad_trace.data_ptr(),
                         None if self.layer_gid is None else self.layer_gid.data_ptr(),
                         None if self.layer_pos is None else self.layer_pos.data_ptr())

    def set_diffusion_draws(self, time: torch.Tensor, alpha_hats) -> None:
        """Diffusion head: the sampled time steps (i32 [B], diffusion.py:125) and the alpha_hat table (:88-92)."""
        assert time.dtype == torch.int32 and tuple(time.shape) == (self.cfg.batch,) and time.is_cuda
        self.head_time = time.contiguous()
        self.alpha_hats = torch.as_tensor(np.asarray(alpha_hats, np.float32)).to(self.dev)
        assert self.alpha_hats.numel() == self.cfg.diffusion_steps

    def set_dropout_step(self, step: int) -> int:
        """Fold the training step into the dropout seed, as the reference does with `jax.random.fold_in(rngs['dropout'],
        train_state.step)` (models/octo/octo.py): every kernel derives its masks from (seed, site, row, column) only, so
        without this every step would draw the same masks.  Call before `forward`; `backward` of the same step reuses the
        value (it regenerates the masks from the same seed).  Returns the mixed 64-bit seed."""
        z = (self._base_seed + 0x9E3779B97F4A7C15 * (int(step) + 1)) & 0xFFFFFFFFFFFFFFFF   # splitmix64 finaliser
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        z ^= z >> 31
        self.ccfg.dropout_seed = z
        return z

    def set_dropout_seed(self, seed: int) -> None:
        """Replace the base dropout seed in place (no reallocation); takes effect at the next forward."""
        self._base_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.ccfg.dropout_seed = self._base_seed

    def _training_workspace(self, what: str) -> None:
        if self.predict_only:
            raise RuntimeError(f"{what} needs the training workspace: this engine is predict-only (use predict())")

    def forward(self, x: torch.Tensor, target: Optional[torch.Tensor] = None):
        self._training_workspace("forward")
        cfg = self.cfg
        assert x.is_cuda and x.is_contiguous() and tuple(x.shape) == (cfg.batch, cfg.tokens, cfg.channels), x.shape
        assert x.dtype in (torch.float32, torch.bfloat16)
        if target is not None:
            want = {"none": (cfg.batch, cfg.n_readout, cfg.channels), "continuous": (cfg.batch, cfg.head_features),
                    "categorical": (cfg.batch, cfg.head_groups), "diffusion": (2, cfg.batch, cfg.head_features)}[cfg.head]
            if cfg.head == "diffusion":
                assert self.head_time is not None, "set_diffusion_draws(time, alpha_hats) first"
            assert target.dtype == torch.float32 and tuple(target.shape) == want, (target.shape, want)
        self._x, self._target = x, target
        io = self._io(x, target)
        L.check(self.lib.tome_stack_forward(C.byref(self.ccfg), C.byref(io), self._stream()))
        return self

    def backward(self, events: Optional[List[torch.cuda.Event]] = None):
        """Loss gradient + full backward into `self.grads` (accumulating: call zero_grad() first)."""
        self._training_workspace("backward")
        assert self._x is not None and self._target is not None, "forward(x, target) first"
        self._events = events
        io = self._io(self._x, self._target)
        self._events = None
        L.check(self.lib.tome_stack_backward(C.byref(self.ccfg), C.byref(io), self._stream()))
        return self

    def zero_grad(self):
        self.grads.zero_()

    def decay_ranges(self, decay: str = "dense_kernels") -> List[tuple]:
        """Sorted [lo, hi) element ranges of the weight matrices that get weight decay under `decay="dense_kernels"`: every
        layer's wqkv, wo, w1, w2, the continuous / categorical head kernel and the diffusion head's tw1, tw2, w1, w2 (the
        Dense / DenseGeneral kernels).  LayerNorm parameters, biases, pos_embedding and the Fourier kernel get none."""
        assert decay == "dense_kernels", decay
        v = self.param_views(self.params)
        mats = [d[k] for d in v["layers"] for k in ("wqkv", "wo", "w1", "w2")]
        head = v.get("head", {})
        mats += [head[k] for k in (("tw1", "tw2", "w1", "w2") if self.cfg.head == "diffusion" else ("kernel",)) if k in head]
        return sorted((t.storage_offset(), t.storage_offset() + t.numel()) for t in mats)

    def adamw_step(self, lr=1e-4, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.0, grad_scale=1.0,
                   max_grad_norm: Optional[float] = None, skip_nonfinite: bool = False, decay: str = "all"):
        """One AdamW step on the flat vectors (tome_adamw_step).  max_grad_norm: clip grad_scale * grads to this global L2
        norm first (optax.clip_by_global_norm).  skip_nonfinite: a gradient holding a NaN / Inf changes nothing and counts
        as skipped (optax.apply_if_finite); from the first such call on, bias correction counts applied steps only.
        decay: "all" or "dense_kernels" (weight decay on the Dense kernels only, `decay_ranges`).  Steps that clip or skip
        leave the norm of grad_scale * grads in `grad_norm` (device f32 [1]).  With none of these the step is the plain one."""
        self._training_workspace("adamw_step")
        assert decay in ("all", "dense_kernels"), decay
        if self.adam_m is None:
            self.adam_m = torch.zeros_like(self.params)
            self.adam_v = torch.zeros_like(self.params)
        if skip_nonfinite and self._opt_steps is None:   # {applied, skipped}: every earlier step was applied
            self._opt_steps = torch.tensor([self.step_count, 0], dtype=torch.int32, device=self.dev)
        self.step_count += 1
        opts = None
        if max_grad_norm is not None or skip_nonfinite or decay != "all" or self._opt_steps is not None:
            ranges = None
            if decay != "all":
                if self._decay_ranges is None:
                    flat = [x for r in self.decay_ranges(decay) for x in r]
                    self._decay_ranges = ((C.c_longlong * len(flat))(*flat), len(flat) // 2)
                ranges = self._decay_ranges
            norm = max_grad_norm is not None or skip_nonfinite
            if self._adam_ws is None:
                self._adam_ws = _scratch(self.lib.tome_adamw_workspace_bytes(self.n_params), self.dev)
            opts = L.AdamwOpts(0.0 if max_grad_norm is None else float(max_grad_norm), int(bool(skip_nonfinite)),
                               None if ranges is None else ranges[0], 0 if ranges is None else ranges[1],
                               self.grad_norm.data_ptr() if norm else None,
                               None if self._opt_steps is None else self._opt_steps.data_ptr(),
                               self._adam_ws.data_ptr(), self._adam_ws.numel())
        L.check(self.lib.tome_adamw_step(self.n_params, self.params.data_ptr(), self.grads.data_ptr(), self.adam_m.data_ptr(),
                                         self.adam_v.data_ptr(), self.params_bf16.data_ptr(), lr, beta1, beta2, eps,
                                         weight_decay, grad_scale, self.step_count, None if opts is None else C.byref(opts),
                                         self._stream()))

    def optimizer_steps(self) -> tuple:
        """(applied, skipped) optimiser steps so far.  Reads the device counters (a sync) once skip_nonfinite has been used."""
        if self._opt_steps is None:
            return self.step_count, 0
        a, s = self._opt_steps.tolist()
        return a, s

    # ------------------------------------------------------------------ prediction (forward only)
    def predictor(self, batch: Optional[int] = None) -> "ToMeStackEngine":
        """A predict-only engine over THIS engine's params / params_bf16 storage (no copy), optionally at another batch size:
        it sees every optimiser step without a reload.  Masks and readout indices are shared too."""
        cfg = self.cfg if batch is None else dataclasses.replace(self.cfg, batch=int(batch))
        p = ToMeStackEngine(cfg, device=self.dev, predict_only=True, _params=(self.params, self.params_bf16))
        p.gid, p.pos, p.allow, p.readout_idx = self.gid, self.pos, self.allow, self.readout_idx
        p.layer_gid, p.layer_pos = self.layer_gid, self.layer_pos
        return p

    def policy(self, tokenizer, tokenizer_variables, token_sequence, batch: Optional[int] = None, graph: bool = False):
        """Camera frames -> actions in one native call (tome_policy_predict): a `policy.PixelPolicy` over THIS engine's
        params / params_bf16 storage (it sees every optimiser step without a reload), masks and readout indices, at `batch`
        (default: the engine's).  tokenizer / tokenizer_variables: the ImageTokenizer (bf16 out_dtype) and its Flax variables,
        packed once; token_sequence: the grammar (TokenSequence or its string) the sequence is assembled by.  graph=True replays
        every call after the first from a CUDA graph."""
        from .policy import PixelPolicy
        return PixelPolicy(self, tokenizer, tokenizer_variables, token_sequence, batch=batch, graph=graph)

    def predict(self, x: torch.Tensor, init=None, noise=None, rng=0, x_final: Optional[torch.Tensor] = None):
        """Forward only, dropout off (tome_stack_predict).  Returns (head_out, readout): head_out is the action head's output
        -- tanh actions [B, A] (continuous), logits [B, groups, bins] (categorical), sampled actions [B, A] (diffusion) -- or
        None without a head; readout f32 [B, n_readout, C] or None without readout tokens.  Diffusion head: init [B, A] and
        noise [B, A] (reused by every step) or [steps, B, A] default to draws from `rng` (numpy's generator), as
        DiffusionActionHead.predict_action draws them.  x_final: optional bf16 [B, T_L, C] output.  The returned tensors are
        copies: a later predict() does not overwrite them."""
        if not self.predict_only:
            raise RuntimeError("predict() needs a predict-only engine: ToMeStackEngine(..., predict_only=True) or predictor()")
        cfg = self.cfg
        assert x.is_cuda and x.is_contiguous() and tuple(x.shape) == (cfg.batch, cfg.tokens, cfg.channels), x.shape
        assert x.dtype in (torch.float32, torch.bfloat16)
        smp = None
        if cfg.head == "diffusion":
            from .action_heads.diffusion import cosine_beta_schedule, ddpm_coefficients
            from .attention_blocks._module import as_rng
            g = as_rng(rng)
            B, A = cfg.batch, cfg.head_features
            if init is None:
                init = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32))
            if noise is None:
                noise = torch.as_tensor(g.standard_normal((B, A)).astype(np.float32))
            init = torch.as_tensor(init).to(self.dev).float().contiguous()
            noise = torch.as_tensor(noise).to(self.dev).float().contiguous()
            assert tuple(init.shape) == (B, A) and tuple(noise.shape) in ((B, A), (cfg.diffusion_steps, B, A)), (init.shape, noise.shape)
            coef = torch.as_tensor(ddpm_coefficients(cosine_beta_schedule(cfg.diffusion_steps))).to(self.dev)
            self._draws = (init, noise, coef)   # alive until the kernels that read them have run
            smp = L.DdpmSample(init.data_ptr(), noise.data_ptr(), int(noise.dim() == 3), coef.data_ptr(), 5.0)
        if x_final is not None:
            assert x_final.is_cuda and x_final.dtype == torch.bfloat16 and x_final.is_contiguous()
            assert x_final.numel() == cfg.batch * self.tokens_at(cfg.layers) * cfg.channels
        io = self._io(x, None)
        io.x_final = None if x_final is None else x_final.data_ptr()
        L.check(self.lib.tome_stack_predict(C.byref(self.ccfg), C.byref(io), None if smp is None else C.byref(smp), self._stream()))
        out = None
        if self.head_out is not None:
            out = (self.head_out if cfg.head == "categorical" else self.head_out.view(cfg.batch, cfg.head_features)).clone()
        return out, None if self.readout is None else self.readout.clone()

    # ------------------------------------------------------------------ results (views into the workspace)
    def tokens_at(self, layer: int) -> int:
        return int(self.lib.tome_stack_tokens_at(C.byref(self.ccfg), layer))

    def _view(self, ptr: int, shape, dtype) -> torch.Tensor:
        self._training_workspace("the workspace accessors")
        off = ptr - self.workspace.data_ptr()
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        return self.workspace[off: off + n].view(dtype).view(*shape)

    def final_x(self) -> torch.Tensor:
        io = self._io(self._x, self._target)
        p = self.lib.tome_stack_final_x(C.byref(self.ccfg), C.byref(io))
        return self._view(p, (self.cfg.batch, self.tokens_at(self.cfg.layers), self.cfg.channels), torch.bfloat16)

    def final_size(self) -> Optional[torch.Tensor]:
        io = self._io(self._x, self._target)
        p = self.lib.tome_stack_final_size(C.byref(self.ccfg), C.byref(io))
        if not p:
            return None
        return self._view(p, (self.cfg.batch, self.tokens_at(self.cfg.layers)), torch.float32)

    def layer_plan(self, layer: int):
        """(node_max, node_idx, edge_idx, dst_idx) of one layer's matching, or None if that layer merged nothing.  In a
        set-merging stack the arrays are concatenated set by set (cfg.layer_sets(layer)), indices local to the set."""
        io = self._io(self._x, self._target)
        t = self.tokens_at(layer)
        r = t - self.tokens_at(layer + 1)
        if r == 0:
            return None
        sets = self.cfg.layer_sets(layer)
        ta = (t + 1) // 2 if sets is None else sum((n + 1) // 2 for _, n, _ in sets)
        b = self.cfg.batch
        f = self.lib
        nm = self._view(f.tome_stack_layer_node_max(C.byref(self.ccfg), C.byref(io), layer), (b, ta), torch.float32)
        ni = self._view(f.tome_stack_layer_node_idx(C.byref(self.ccfg), C.byref(io), layer), (b, ta), torch.int32)
        ei = self._view(f.tome_stack_layer_edge_idx(C.byref(self.ccfg), C.byref(io), layer), (b, ta), torch.int32)
        di = self._view(f.tome_stack_layer_dst_idx(C.byref(self.ccfg), C.byref(io), layer), (b, r), torch.int32)
        return nm, ni, ei, di

    def layer_prune(self, layer: int):
        """Pruning stacks: (importance f32 [B, T_in], kept token indices i32 [B, T_out]) of `layer` in the last forward."""
        io = self._io(self._x, self._target)
        b, t, to = self.cfg.batch, self.tokens_at(layer), self.tokens_at(layer + 1)
        pi = self.lib.tome_stack_layer_importance(C.byref(self.ccfg), C.byref(io), layer)
        pk = self.lib.tome_stack_layer_prune_ids(C.byref(self.ccfg), C.byref(io), layer)
        if not pi or not pk:
            return None
        return self._view(pi, (b, t), torch.float32), self._view(pk, (b, to), torch.int32)

    def layer_x_in(self, layer: int) -> torch.Tensor:
        """bf16 [B, T_in(layer), C] tokens entering `layer` in the last forward (layer == layers: the final tokens)."""
        io = self._io(self._x, self._target)
        p = self.lib.tome_stack_layer_x_in(C.byref(self.ccfg), C.byref(io), layer)
        return self._view(p, (self.cfg.batch, self.tokens_at(layer), self.cfg.channels), torch.bfloat16)

    def layer_size_in(self, layer: int) -> Optional[torch.Tensor]:
        io = self._io(self._x, self._target)
        p = self.lib.tome_stack_layer_size_in(C.byref(self.ccfg), C.byref(io), layer)
        return None if not p else self._view(p, (self.cfg.batch, self.tokens_at(layer)), torch.float32)

    def enable_grad_trace(self) -> None:
        """Parity aid: keep the gradient every layer receives during backward (tome_stack_io_t.grad_trace)."""
        cfg = self.cfg
        self._grad_trace = torch.zeros(cfg.layers, cfg.batch * cfg.tokens * cfg.channels, dtype=torch.bfloat16, device=self.dev)

    def layer_grad_out(self, layer: int) -> torch.Tensor:
        """bf16 [B, T_out(layer), C]: dL/dx_out of `layer` as the last backward received it (needs enable_grad_trace())."""
        b, to, c = self.cfg.batch, self.tokens_at(layer + 1), self.cfg.channels
        return self._grad_trace[layer, : b * to * c].view(b, to, c)

    def layer_relu_gate(self, layer: int) -> torch.Tensor:
        """bool [B, T_out(layer), mlp_dim]: which elements of MLP-1's output survived ReLU (and hidden dropout) in the
        last forward -- the gate bits the MLP backward consumes (tome_stack_layer_relu_bits)."""
        io = self._io(self._x, self._target)
        b, to, f = self.cfg.batch, self.tokens_at(layer + 1), self.cfg.mlp_dim
        words = (f + 31) // 32
        p = self.lib.tome_stack_layer_relu_bits(C.byref(self.ccfg), C.byref(io), layer)
        w = self._view(p, (b * to, words), torch.int32)
        bits = (w[:, :, None] >> torch.arange(32, device=w.device, dtype=torch.int32)) & 1
        return bits.reshape(b, to, words * 32)[:, :, :f].bool()
