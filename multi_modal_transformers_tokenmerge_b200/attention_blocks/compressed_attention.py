"""The pruning variant of the block stack: the module API of multi_modal_transformers/attention_blocks/compressed_attention.py
on the native executor (csrc/stack.cu with tome_stack_cfg_t.prune_sets > 0; SURVEY.md 8(f) rank 2).

    StackedCompressedEncoder1DBlock(num_blocks, encoder_1d_block, prune_fns, merge_fns)(x, masks, train=False)        :377-404
    CompressedEncoder1DBlock / CompressedMultiHeadDotProductAttention                                                  :19-358
    AddPositionEmbedding                                                                                               :360-375

What the reference intends per layer (:396-402): attention under masks[layer_idx] (the compression grammar's mask of that
layer, token_sequencer.py:222-238), importance scores from the attention weights (:303-306), prune_fns[layer_idx] =
compute_top_k_tokens with that layer's token sets (token_compression.py:15-46), MLP.  As written it cannot run -- :340 drops
the attention result and :345 adds a pruned tensor to an unpruned one -- so the composition is the one DESIGN.md section 7
states: the token choice is applied after the residual add.

`merge_fns` fills the merge slot the reference keeps per layer (its call is commented out, :310-311): instead of pruning, every
layer merges tokens by bipartite soft matching INSIDE each token set (tokenset_soft_matching + merge_wavg after the attention
residual), so no token merges across a frame or modality boundary.  Give exactly one of prune_fns / merge_fns (both:
NotImplementedError, pruning and merging in one stack is not supported).  `merge_fns[l]` is
`functools.partial(tokenset_soft_matching, tokenset_idx=..., tokenset_r=...)` or a `(tokenset_idx, tokenset_r)` pair, checked
against the compression grammar like prune_fns (set of n tokens merging c per layer: n - l c tokens, r = c at layer l).  A
merging stack takes masks[0] only: merged rows carry the group id and position of their destination token.

`prune_fns[l]` may be the reference's `functools.partial(compute_top_k_tokens, tokenset_idx=..., tokenset_k=...)` (of the
reference's or of this package's function: only its keywords are read) or a `(tokenset_idx, tokenset_k)` pair; every layer must
drop the same number of tokens per set, as the grammar prescribes.  `masks[l]` is a GroupMask / `(gid, pos)` pair of layer l's
grammar (TokenSequence.layer_group_ids) -- with `allow` the rule table -- or None for an unmasked stack.
Parameters: the tree of StackedEncoder1DBlock (posembed_input, ScanEncoder1DBlock_0 with the stacked per-layer leaves).
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Sequence

import numpy as np
import torch

from . import _functional as F
from .attention import AddPositionEmbedding, StackedEncoder1DBlock as _VanillaStack, _np, _seed_of, flax_tree_to_layers  # noqa: F401

__all__ = ["StackedCompressedEncoder1DBlock", "AddPositionEmbedding"]


def _sets_of(fn, counts="tokenset_k"):
    kw = getattr(fn, "keywords", None)
    if kw is not None:
        return list(kw["tokenset_idx"]), list(kw[counts])
    idx, ks = fn
    return list(idx), list(ks)


def _given(fns):
    return fns is not None and any(f is not None for f in fns)


class StackedCompressedEncoder1DBlock(_VanillaStack):
    """Stacking Transformer encoder layers that prune per modality after every attention (compressed_attention.py:377-404)."""

    def __init__(self, num_blocks: int, encoder_1d_block: Dict[str, Any], prune_fns: Optional[Sequence] = None, merge_fns=None,
                 importance: str = "received", **extra):
        super().__init__(num_blocks, encoder_1d_block, **extra)
        if _given(merge_fns) and _given(prune_fns):
            raise NotImplementedError("prune_fns and merge_fns together: pruning and merging in one stack is not supported")
        self.set_merge = _given(merge_fns)
        fns, what = (merge_fns, "tokenset_soft_matching partial (or (tokenset_idx, tokenset_r) pair)") if self.set_merge else \
            (prune_fns, "compute_top_k_tokens partial (or (tokenset_idx, tokenset_k) pair)")
        if fns is None or len(fns) != num_blocks or any(f is None for f in fns):
            raise ValueError(f"{'merge_fns' if self.set_merge else 'prune_fns'} must hold one {what} per block")
        # both as (start, n, tokens kept): a merge keeps n - r
        per_layer = [_sets_of(f, "tokenset_r") for f in fns] if self.set_merge else [_sets_of(f) for f in fns]
        if self.set_merge:
            per_layer = [(idx, [int(n) - int(r) for (_, n), r in zip(idx, rs)]) for idx, rs in per_layer]
        idx0, k0 = per_layer[0]
        self.prune_sets = tuple((int(n), int(n) - int(k)) for (_, n), k in zip(idx0, k0))
        name = "merge_fns" if self.set_merge else "prune_fns"
        for l, (idx, ks) in enumerate(per_layer):      # token_sequencer.py:236: num_tokens - layer * num_compressed_tokens
            start = 0
            if len(idx) != len(self.prune_sets) or len(ks) != len(idx):
                raise ValueError(f"{name}[{l}]: token sets must follow the compression grammar ({len(self.prune_sets)} sets)")
            for (s_, n_), k_, (n0, c) in zip(idx, ks, self.prune_sets):
                if (int(s_), int(n_), int(k_)) != (start, n0 - l * c, n0 - (l + 1) * c):
                    raise ValueError(f"{name}[{l}]: token sets must follow the compression grammar (set of {n0} tokens dropping "
                                     f"{c} per layer: expected start {start}, n {n0 - l * c}, k {n0 - (l + 1) * c}; got {s_}, {n_}, {k_})")
                start += n0 - l * c
        self.importance = importance
        self.last_ids = None

    def _apply(self, params, x, masks=None, train=False, allow=None, dropout_rng=None):
        from ..engine import StackConfig, ToMeStackEngine
        if not x.is_cuda:
            raise RuntimeError("StackedCompressedEncoder1DBlock runs on CUDA (sm_100a) only; there is no CPU fallback")
        blk = self._block()
        ln, dr, at, mlp = blk._specs()
        d, _, _, _ = mlp._specs()
        B, T, C = x.shape
        if sum(n for n, _ in self.prune_sets) != T:
            raise ValueError(f"the token sets hold {sum(n for n, _ in self.prune_sets)} tokens, the sequence {T}")
        groups = None
        if masks is not None:
            if self.set_merge:   # merged rows carry their groups: only the layer-0 mask is an input
                masks = [masks[0]]
            if (len(masks) != (1 if self.set_merge else self.num_blocks)) or allow is None:
                raise ValueError("masks: one (gid, pos) pair / GroupMask per block, with `allow` the [G, G] rule table")
            groups = [((m.gid, m.pos) if isinstance(m, F.GroupMask) else m) for m in masks]
            groups = [(np.asarray(_np(g_), np.uint8), np.asarray(_np(p_), np.int32)) for g_, p_ in groups]
        hd = at.qkv_features or C
        key = (B, T, C, bool(train), None if groups is None else int(np.asarray(_np(allow)).shape[0]))
        if self._engine is None or self._engine_key != key:
            cfg = StackConfig(batch=B, tokens=T, channels=C, heads=at.num_heads, head_dim=hd // at.num_heads, mlp_dim=d.features,
                              layers=self.num_blocks, r=0, ln_axis=ln.axis, ln_eps=ln.epsilon, prop_attn=False,
                              num_groups=0 if groups is None else int(np.asarray(_np(allow)).shape[0]),
                              dropout_rate=dr.rate if train else 0.0, dropout_seed=_seed_of(dropout_rng),
                              attn_dropout_rate=at.dropout_rate if train else 0.0, prune_sets=self.prune_sets, prune_importance=self.importance,
                              set_merge=self.set_merge)
            kw = {}
            if groups is not None:
                kw = dict(gid=groups[0][0], pos=groups[0][1], allow=np.asarray(_np(allow), np.uint8))
                if not self.set_merge:
                    kw.update(layer_gid=[g_ for g_, _ in groups], layer_pos=[p_ for _, p_ in groups])
            self._engine = ToMeStackEngine(cfg, training=bool(train), **kw)
            self._engine_key, self._loaded_params = key, None
        self._engine.set_dropout_seed(_seed_of(dropout_rng))
        if self._loaded_params is not params:
            self._engine.load_params(np.asarray(_np(params["posembed_input"]["pos_embedding"])).reshape(T, C),
                                     flax_tree_to_layers(params["ScanEncoder1DBlock_0"], blk._attn_name, self.num_blocks))
            self._loaded_params = params
        self._engine.forward(x.contiguous())
        if not self.set_merge:
            self.last_ids = [self._engine.layer_prune(l)[1].clone() for l in range(self.num_blocks)]
        return self._engine.final_x().clone()
