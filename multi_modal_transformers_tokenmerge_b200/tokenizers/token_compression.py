"""ToMe bipartite soft matching + size-weighted merge: the reference's operator API over the sm_100a kernels.

Mirror of multi_modal_transformers/tokenizers/token_compression.py (same names, argument meaning and return shapes):

    x = compute_top_k_tokens(embeddings, importance_scores, tokenset_idx, tokenset_k)      # :15-46
    merge = bipartite_soft_matching(metric, r, class_token=False, distill_token=False)   # :54-112
    y = merge(x, mode="sum")                                                               # :90-109
    x, size = merge_wavg(merge, x, size=None)                                              # :114-129

and, additive (the merging counterpart of compute_top_k_tokens' per-modality sets):

    merge = tokenset_soft_matching(metric, tokenset_idx, tokenset_r)                       # matching inside each set

Arrays are CUDA torch tensors (device memory is all torch is used for); every step launches a hand-written
kernel through the C ABI (include/tome_b200.h: tome_sim_argmax, tome_select_topr, tome_merge_fwd / _bwd).  There is
no CPU path: a CPU tensor raises.

Deliberate, documented differences from the reference (SURVEY.md Appendix C):
  * r <= 0 returns an identity `merge` (the reference returns a TUPLE `(do_nothing, do_nothing)` at :70, which
    `merge_wavg` would then fail to call);
  * `merge(x, mode)` with a mode other than "sum" raises ValueError (the reference silently drops the merged
    tokens, :99-101);
  * `size` is always fp32 (the reference gives it x's dtype, :122, inexact above 256 in bf16);
  * `merge_wavg` runs merge(x*size), merge(size) and the division in ONE kernel pass; the arithmetic (fp32
    multiply, sequential adds in rank order, divide) is the reference's, so results are bit-identical to the
    oracle's restatement of :121-127;
  * additive: `merge.unmerge(y)` (ToMe-paper unmerge, not in the reference) and `merge.plan` (the index set).
"""
from __future__ import annotations

from typing import Callable, Optional, Tuple

import torch

from .. import _lib as L
from .. import ops


### token pruning methods ###

def compute_top_k_tokens(embeddings: torch.Tensor, importance_scores: torch.Tensor, tokenset_idx, tokenset_k) -> torch.Tensor:
    """token_compression.py:15-46: top-k tokens per modality by importance score.

    embeddings [T, C] and importance_scores [T] as in the reference (one sequence; its caller vmaps), or batched
    [B, T, C] / [B, T].  tokenset_idx: (start_idx, num_tokens) per modality; tokenset_k: tokens to keep per modality.
    Returns the kept embeddings, modalities concatenated in order, each in descending score order (jax.lax.top_k; equal
    scores keep the lower index first).  One kernel launch (tome_topk_prune); `compute_top_k_tokens.last_ids` holds the
    kept indices of the most recent call (additive; the reference discards them).

    Note (SURVEY.md Appendix C): the reference computes its importance scores as mean(attn_weights, axis=-1) -- a mean
    over KEYS of rows that sum to one, i.e. the constant 1/T (compressed_attention.py:303-306) -- so with the
    reference's own scores this function keeps the first k tokens of every modality.  Any score works here.
    """
    unbatched = embeddings.dim() == 2
    if unbatched:
        embeddings, importance_scores = embeddings.unsqueeze(0), importance_scores.unsqueeze(0)
    if embeddings.dim() != 3 or importance_scores.shape != embeddings.shape[:2]:
        raise ValueError(f"embeddings {tuple(embeddings.shape)} / importance_scores {tuple(importance_scores.shape)} do not match")
    if len(tokenset_idx) != len(tokenset_k):
        raise ValueError("tokenset_idx and tokenset_k must have one entry per modality")
    starts, ns = [int(s[0]) for s in tokenset_idx], [int(s[1]) for s in tokenset_idx]
    for n, k in zip(ns, tokenset_k):
        if k > n:
            raise ValueError(f"top_k: k = {k} exceeds the modality's {n} tokens")  # jax.lax.top_k raises likewise
    out, ids = ops.topk_prune(embeddings.contiguous(), importance_scores.float().contiguous(), starts, ns,
                              [int(k) for k in tokenset_k])
    compute_top_k_tokens.last_ids = ids[0] if unbatched else ids
    return out[0] if unbatched else out


### token merging methods ###

def do_nothing(x, mode=None):
    """token_compression.py:51"""
    return x


class _Merge:
    """The closure `bipartite_soft_matching` returns (:90-112): holds the device-resident index set."""

    def __init__(self, plan: Optional[ops.MatchPlan], tokens: int):
        self.plan = plan
        self.tokens = tokens

    @property
    def r(self) -> int:
        return 0 if self.plan is None else self.plan.r

    def _check(self, x: torch.Tensor):
        if x.dim() != 3:
            raise ValueError(f"merge expects x of shape [n, t, c], got {tuple(x.shape)}")  # n, t, c = x.shape (:91)
        if x.shape[1] != self.tokens:
            raise ValueError(f"merge was built for t={self.tokens} tokens, got t={x.shape[1]}")

    def __call__(self, x: torch.Tensor, mode: str = "sum") -> torch.Tensor:
        self._check(x)
        if mode != "sum":
            raise ValueError(f'merge: mode "{mode}" is not implemented (the reference only implements "sum", :99)')
        if self.plan is None:
            return x
        squeeze = False
        if x.shape[-1] == 1 and x.dtype == torch.float32:  # merge(size): one column; the kernel wants 16-byte rows
            x, squeeze = x.expand(-1, -1, 4).contiguous(), True
        y, _, _, _ = ops.merge_fwd(self.plan, x.contiguous(), None, L.TOME_MERGE_SUM)
        return y[..., :1].contiguous() if squeeze else y

    def wavg(self, x: torch.Tensor, size: Optional[torch.Tensor]) -> Tuple[torch.Tensor, torch.Tensor]:
        self._check(x)
        if size is None:
            size = torch.ones(x.shape[0], x.shape[1], 1, dtype=torch.float32, device=x.device)  # :121-122
        if self.plan is None:
            return x, size
        s2 = size.reshape(x.shape[0], x.shape[1]).float().contiguous()
        y, s_out, _, _ = ops.merge_fwd(self.plan, x.contiguous(), s2, L.TOME_MERGE_WAVG)
        return y, s_out.unsqueeze(-1)

    def unmerge(self, y: torch.Tensor) -> torch.Tensor:
        """[n, t-r, c] -> [n, t, c]: every original position receives the row it was merged into (SURVEY.md A.7)."""
        if self.plan is None:
            return y
        return ops.merge_bwd(self.plan, y.contiguous(), None, None, L.TOME_MERGE_SUM)


def bipartite_soft_matching(metric: torch.Tensor, r: int, class_token: bool = False,
                            distill_token: bool = False) -> Callable:
    """token_compression.py:54-112.  metric [n, t, d] (fp32 or bf16, CUDA)."""
    if metric.dim() != 3:
        raise ValueError(f"metric must be [batch, tokens, dim] (one batch dim, :84), got {tuple(metric.shape)}")
    t = metric.shape[1]
    r = ops.clamp_r(t, r, class_token, distill_token)  # :60-67
    if r <= 0:
        return _Merge(None, t)
    node_max, node_idx, _ = ops.sim_argmax(metric.contiguous(), class_token=class_token, distill_token=distill_token)
    plan = ops.select_topr(node_max, node_idx, t, r, distill_token=distill_token)
    return _Merge(plan, t)


def tokenset_soft_matching(metric: torch.Tensor, tokenset_idx, tokenset_r) -> Callable:
    """Bipartite soft matching inside each token set: `merge` for merge_wavg / merge(x, "sum") that never merges a token
    with one of another set.  tokenset_idx: (start_idx, num_tokens) per set as compute_top_k_tokens takes them, consecutive
    and covering the sequence; tokenset_r: tokens each set loses (0 <= r <= num_tokens // 2; r = 0 leaves the set as it is).

    The result for set s is bipartite_soft_matching(metric[:, s], r_s) + merge applied to the set's slice alone (the even /
    odd split counted from the set's first token, the same tie rules and fp32 adds); the sets' outputs are concatenated in
    order, so every set stays contiguous.  With one set per frame and modality of a block-causal sequence, a merged row keeps
    the group of every token in it.  One launch each of K1, K2 (and K3 per merge) over all sets."""
    if metric.dim() != 3:
        raise ValueError(f"metric must be [batch, tokens, dim], got {tuple(metric.shape)}")
    if len(tokenset_idx) != len(tokenset_r):
        raise ValueError("tokenset_idx and tokenset_r must have one entry per token set")
    if not 1 <= len(tokenset_r) <= L.MAX_TOKEN_SETS:
        raise ValueError(f"between 1 and {L.MAX_TOKEN_SETS} token sets are supported, got {len(tokenset_r)}")
    t = metric.shape[1]
    sets, start = [], 0
    for (s_, n), r in zip(tokenset_idx, tokenset_r):
        s_, n, r = int(s_), int(n), int(r)
        if s_ != start or n < 1:
            raise ValueError(f"token sets must be consecutive and non-empty: expected a set starting at {start}, got ({s_}, {n})")
        if not 0 <= r <= n // 2:
            raise ValueError(f"token set ({s_}, {n}): r = {r} out of range [0, {n // 2}]")
        sets.append((s_, n, r))
        start += n
    if start != t:
        raise ValueError(f"the token sets cover {start} tokens, metric has {t}")
    if sum(r for _, _, r in sets) == 0:
        return _Merge(None, t)
    node_max, node_idx, _ = ops.sim_argmax(metric.contiguous(), sets=sets)
    return _Merge(ops.select_topr(node_max, node_idx, t, sets=sets), t)


def merge_wavg(merge: Callable, x: torch.Tensor, size: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """token_compression.py:114-129.  Returns (x [n, t-r, c], size [n, t-r, 1] fp32)."""
    if isinstance(merge, _Merge):
        return merge.wavg(x, size)
    if merge is do_nothing:
        if size is None:
            size = torch.ones(x.shape[0], x.shape[1], 1, dtype=torch.float32, device=x.device)
        return x, size
    raise TypeError("merge_wavg: `merge` must come from bipartite_soft_matching or tokenset_soft_matching")
