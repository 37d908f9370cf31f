"""Checker-side restatement of matching and merging INSIDE token sets (tome_token_sets_t), built only from the oracle's own
functions applied to set slices: for a set (start, n, r), its part of the output is oracle.merge_wavg of
oracle.bipartite_soft_matching(metric[:, start:start + n], r) on the set's slice, the parts concatenated in set order, a set
with r = 0 passed through unchanged."""
from __future__ import annotations

import numpy as np

from oracle import tome_oracle as O


def set_plans(metric, sets, node_override=None):
    """One oracle MatchPlan per set (None for r = 0).  node_override = (node_max, node_idx) concatenated set by set, as the
    kernels lay them out: the oracle then ranks and splits the GPU's own row maxima."""
    plans, off = [], 0
    for start, n, r in sets:
        ta = (n + 1) // 2
        if r == 0:
            plans.append(None)
        elif node_override is not None:
            plans.append(O.plan_from_node(node_override[0][:, off:off + ta], node_override[1][:, off:off + ta], n, r))
        else:
            plans.append(O.bipartite_soft_matching(np.asarray(metric)[:, start:start + n], r))
        off += ta
    return plans


def set_row_map(plans, sets, batch):
    """Global output row of every input token [B, T]."""
    out, row0 = [], 0
    for p, (start, n, r) in zip(plans, sets):
        out.append(np.broadcast_to(np.arange(n, dtype=np.int32), (batch, n)) + row0 if p is None else O.row_map(p) + row0)
        row0 += n - r
    return np.concatenate(out, axis=1).astype(np.int32)


def set_merge_wavg(plans, sets, x, size=None):
    """numpy merge_wavg per set: (x_out [B, T-r, C], size_out [B, T-r, 1])."""
    if size is None:
        size = np.ones_like(x[..., :1])
    xs, ss = [], []
    for p, (start, n, _) in zip(plans, sets):
        xi, si = x[:, start:start + n], size[:, start:start + n]
        if p is not None:
            xi, si = O.merge_wavg(p, xi, si)
        xs.append(xi)
        ss.append(si)
    return np.concatenate(xs, axis=1), np.concatenate(ss, axis=1)


def set_merge_wavg_torch(plans, sets, x, size):
    """merge_wavg per set with autograd (torch CPU)."""
    torch = O._torch()
    xs, ss = [], []
    for p, (start, n, _) in zip(plans, sets):
        xi, si = x[:, start:start + n], size[:, start:start + n]
        if p is not None:
            xi, si = O.merge_wavg_torch(p, xi, si)
        xs.append(xi)
        ss.append(si)
    return torch.cat(xs, dim=1), torch.cat(ss, dim=1)


def kept_token_groups(plans, sets, gid, pos, row_map):
    """gid / pos after the merge: every output row keeps those of its unmerged or destination token."""
    B, T = gid.shape
    keep = np.ones((B, T), dtype=bool)
    for p, (start, n, r) in zip(plans, sets):
        if p is None:
            continue
        ta = (n + 1) // 2
        rank = np.empty((B, ta), dtype=np.int32)
        np.put_along_axis(rank, p.edge_idx, np.broadcast_to(np.arange(ta, dtype=np.int32), (B, ta)), axis=1)
        keep[:, start:start + n:2] = rank >= r
    to = int(row_map.max()) + 1
    g2, p2 = np.zeros((B, to), gid.dtype), np.zeros((B, to), pos.dtype)
    bi, ti = np.nonzero(keep)
    g2[bi, row_map[bi, ti]] = gid[bi, ti]
    p2[bi, row_map[bi, ti]] = pos[bi, ti]
    return g2, p2


def stack_sets_at(prune_sets, layer):
    """(start, n, r) of the sets entering `layer` of a set-merging stack: prune_sets = [(n at layer 0, c merged per layer)]."""
    out, start = [], 0
    for n0, c in prune_sets:
        n = n0 - layer * c
        out.append((start, n, c))
        start += n
    return out


def set_block(p, x, size, gid, pos, allow, *, num_heads, sets, ln_axis="feature", prop_attn=True, node_override=None,
              act_dtype=None, relu_gate=None):
    """oracle.tome_block with the matching and merge_wavg run inside each token set.  Returns (x, size, gid, pos, plans,
    row_map)."""
    torch = O._torch()
    B, T, C = x.shape
    rd = lambda t: O._round_st(t, act_dtype)  # noqa: E731
    h = rd(O.layer_norm(x, p.ln1_scale, p.ln1_bias, axis=ln_axis))
    q = rd(h @ p.wq + p.bq).reshape(B, T, num_heads, -1)
    k = rd(h @ p.wk + p.bk).reshape(B, T, num_heads, -1)
    v = rd(h @ p.wv + p.bv).reshape(B, T, num_heads, -1)
    mask = torch.as_tensor(O.dense_mask(gid, pos, gid, pos, allow))[:, None, :, :]
    bias = torch.log(size[:, None, None, :, 0]) if prop_attn else None
    o = rd(O.attention(q, k, v, mask=mask, bias=bias).reshape(B, T, -1))
    x = rd(x + (o @ p.wo + p.bo))
    metric = k.detach().mean(dim=2).to(torch.float32).numpy()
    plans = set_plans(metric, sets, node_override)
    rm = set_row_map(plans, sets, B)
    x, size = set_merge_wavg_torch(plans, sets, x, size)
    x = rd(x)
    gid, pos = kept_token_groups(plans, sets, gid, pos, rm)
    y = rd(O.layer_norm(x, p.ln2_scale, p.ln2_bias, axis=ln_axis))
    pre = y @ p.w1 + p.b1
    y = rd(torch.relu(pre) if relu_gate is None else torch.where(torch.as_tensor(relu_gate), pre, torch.zeros_like(pre)))
    return rd(x + (y @ p.w2 + p.b2)), size, gid, pos, plans, rm


def set_merge_stack(params, pos_embedding, x, gid, pos, allow, *, num_heads, prune_sets, ln_axis="feature", prop_attn=True,
                    node_override=None, act_dtype=None, relu_gate=None, trace=None):
    """oracle.tome_stack with every layer merging inside its token sets.  Returns (x_final, size, origin [B, T0])."""
    torch = O._torch()
    B, T0, C = x.shape
    x = O._round_st(x + pos_embedding, act_dtype)
    size = torch.ones(B, T0, 1, dtype=x.dtype)
    gid = np.broadcast_to(gid, (B, T0)).copy()
    pos = np.broadcast_to(pos, (B, T0)).copy()
    origin = np.broadcast_to(np.arange(T0, dtype=np.int32), (B, T0)).copy()
    for li, p in enumerate(params):
        sets = stack_sets_at(prune_sets, li)
        x, size, gid, pos, plans, rm = set_block(
            p, x, size, gid, pos, allow, num_heads=num_heads, sets=sets, ln_axis=ln_axis, prop_attn=prop_attn,
            node_override=None if node_override is None else node_override[li], act_dtype=act_dtype,
            relu_gate=None if relu_gate is None else relu_gate[li])
        origin = np.take_along_axis(rm, origin, axis=1)
        if trace is not None:
            trace.append((plans, rm))
    return x, size, origin
