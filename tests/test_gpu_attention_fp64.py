"""Attention forward, backward and token importance against an fp64 reference, element by element.  Needs a B200: `-m gpu`.

The reference is oracle.attention / attention_weights / attention_importance evaluated in float64 on the exact bf16 inputs
the kernels read (mask from dense_mask, bias log(size), the regenerated dropout keep mask), gradients by autograd.  Every
output element must lie within a bound derived from the arithmetic of the kernels, fixed before any run:

    out[q]  c u sum_k w_qk |v_k| + u |out|                      w = weights after dropout, u = 2^-8 (bf16), c = 4
    dV[k]   c u sum_q w_qk |dO_q| + u |dV|
    dK[k]   c u scale sum_q P_qk (|dP_qk| + |delta_q| + D_q) |q_q| + u |dK|     (dQ: the same with |k_k|)
    lse     c u (1 + |lse|), on rows that see at least one key
    importance  c u imp + u imp                                 (a mean of non-negative weights)

where every contraction takes |.| of each operand (|dP_qk| = sum |dO_q| |v_k| keep / (1 - rate), |delta_q| =
sum |dO_q| |O_q|), P is the masked softmax and D_q = sum_d |dO_qd| (out bound of (q, d)) covers delta being formed from the
rounded bf16 output.  The kernels round P and dS to bf16 once each (u / 2) and their outputs once (u / 2); c = 4 leaves a
factor of 8 over the leading term.  An aggregate norm cannot see one wrong row among thousands; these bounds can: the
sensitivity checks at the end recompute the reference with one small deliberate defect and require the kernel output to
fail it.

The cases walk the paths the attention code picks at run time: no mask, the mask folded into QK^T (at most 16 groups, no
causal entry), the per-group visibility words (17-32 groups or a causal entry), both dQ paths, the generic fp32 path for
head_dim != 64, and the importance kernel -- at sequence lengths on either side of the 32-row, 64-key and 128-query tile
edges, with query rows that see no key at all."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import tome_oracle as O  # noqa: E402

U = 2.0 ** -8   # bf16 unit roundoff
C = 4.0
MASKED_ROW_LSE2 = -2.0 ** 90   # attn_meta.cuh: lse * log2(e) of a row with no visible key lies below this


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from multi_modal_transformers_tokenmerge_b200 import _lib, ops
    _lib.lib()
    return ops, _lib


# ------------------------------------------------------------------------------------------------ group tables
def _grammar_allow(W: int, causal: bool):
    """allow of [TaskDescriptionPrefix] [(Text;) Image; Readout]*W: 2W + 1 groups (3W + 1 with the causal Text sets)."""
    body = "Text{1};Image{1};Readout{1}" if causal else "Image{1};Readout{1}"
    _, _, allow, _ = O.sequence_groups(f"[TaskDescriptionPrefix{{1}}] [{body}]*{W}")
    return allow


def _rows(G, T, B, rng, row0_gid, row0_pos):
    """Batch row 0 as given; row 1 the same tokens permuted (as after a merge); row 2 random groups and positions."""
    gid, pos = [row0_gid], [row0_pos]
    perm = rng.permutation(T)
    gid.append(row0_gid[perm])
    pos.append(row0_pos[perm])
    gid.append(rng.integers(0, G, size=T).astype(np.uint8))
    pos.append(rng.integers(0, 64, size=T).astype(np.int32))
    return np.stack(gid[:B]).astype(np.uint8), np.stack(pos[:B]).astype(np.int32)


def _table(kind: str, B: int, T: int, rng):
    """-> (gid [B, T] u8, pos [B, T] i32, allow [G, G] u8), or Nones for "none"."""
    if kind == "none":
        return None, None, None
    if kind in ("g5", "g17", "g31", "causal"):
        allow = {"g5": lambda: _grammar_allow(2, False), "g17": lambda: _grammar_allow(8, False),
                 "g31": lambda: _grammar_allow(15, False), "causal": lambda: _grammar_allow(3, True)}[kind]()
        G = allow.shape[0]
        g0 = (np.arange(T) * G // T).astype(np.uint8)         # the grammar's groups in order, as even as T allows
        p0 = np.zeros(T, np.int32)
        for g in range(G):
            p0[g0 == g] = np.arange(int((g0 == g).sum()))
        gid, pos = _rows(G, T, B, rng, g0, p0)
        return gid, pos, allow
    # random tables: "r16" (folded into QK^T), "r32" / "r32c" (visibility words, r32c with causal entries)
    G = 16 if kind == "r16" else 32
    codes, pr = ((0, 1, 2), (0.4, 0.4, 0.2)) if kind == "r32c" else ((0, 1), (0.5, 0.5))
    allow = rng.choice(codes, size=(G, G), p=pr).astype(np.uint8)
    # rows that see no key, or see keys in only some tiles:
    allow[0] = 0                      # group 0 sees nothing
    allow[1] = 0; allow[1, 2] = 1     # group 1 sees only group 2, whose tokens sit in the last key tile: masked first, visible later
    allow[3] = 0; allow[3, 4] = 1     # group 3 sees only group 4, whose tokens sit in the first key tile
    if kind == "r32c":
        allow[5] = 0; allow[5, 6] = 2  # group 5 sees group 6 causally; group 6 positions start at 8: pos_q < 8 sees nothing
    g0 = rng.integers(7, G, size=T).astype(np.uint8)   # groups 7.. (bits 16-31 of the visibility words for G = 32)
    p0 = rng.integers(0, 24, size=T).astype(np.int32)
    idx, n = rng.permutation(T), max(1, T // 16)
    for j, g in enumerate((0, 1, 3, 5, 6) if kind == "r32c" else (0, 1, 3)):
        g0[idx[j * n:(j + 1) * n]] = g
    p0[g0 == 6] += 8
    if T >= 4:
        g0[:2] = 4        # group 4's keys: the first two tokens
        g0[-2:] = 2       # group 2's keys: the last two tokens
    gid, pos = _rows(G, T, B, rng, g0, p0)
    return gid, pos, allow


def _sizes(kind: str, B: int, T: int, rng):
    if kind == "none":
        return None
    if kind == "int":
        return rng.integers(1, 7, size=(B, T)).astype(np.float32)
    return np.where(rng.random((B, T)) < 0.5, 1.0, 4096.0).astype(np.float32)   # "mix"


# ------------------------------------------------------------------------------------------------ fp64 reference and bounds
def _reference(q, k, v, dout, gid, pos, allow, size, rate, seed, site, causal_le=True):
    """fp64 outputs, gradients and bounds.  q, k, v, dout: the kernels' bf16 inputs [B, T, H, D] (torch, CPU)."""
    B, T, H, D = q.shape
    qd, kd, vd, dod = (t.double() for t in (q, k, v, dout))
    mask = None
    if gid is not None:
        if causal_le:
            mask = O.dense_mask(gid, pos, gid, pos, allow)
        else:   # a deliberate defect for the sensitivity check: pos_k < pos_q instead of <=
            a = allow[gid[:, :, None], gid[:, None, :]]
            mask = (a == 1) | ((a == 2) & (pos[:, None, :] < pos[:, :, None]))
        mask = torch.as_tensor(mask)[:, None]
    bias = None if size is None else torch.log(torch.as_tensor(size, dtype=torch.float64))[:, None, None, :]
    keep = None
    if rate > 0:
        kb, p_eff = O.dropout_keep_mask(T, T, rate, seed, site)
        keep = torch.as_tensor(kb.astype(np.float64) / (1.0 - p_eff))[None, None]
    qr, kr, vr = (t.clone().requires_grad_(True) for t in (qd, kd, vd))
    out = O.attention(qr, kr, vr, mask=mask, bias=bias, drop_keep=keep)
    out.backward(dod)
    P = O.attention_weights(qd, kd, mask=mask, bias=bias)          # [B, H, Tq, Tk]
    w = P if keep is None else P * keep
    Pm = P if mask is None else P * mask                           # what reaches dS: masked logits get no gradient
    scale = 1.0 / math.sqrt(D)
    out = out.detach()
    aq, ak, av, ado, aout = (t.abs() for t in (qd, kd, vd, dod, out))
    b_out = C * U * torch.einsum("bhqk,bkhd->bqhd", w, av) + U * aout
    dv_ref, dk_ref, dq_ref = vr.grad, kr.grad, qr.grad
    b_dv = C * U * torch.einsum("bhqk,bqhd->bkhd", w, ado) + U * dv_ref.abs()
    adp = torch.einsum("bqhd,bkhd->bhqk", ado, av)
    if keep is not None:
        adp = adp * keep
    adelta = (ado * aout).sum(-1).permute(0, 2, 1)[..., None]      # [B, H, Tq, 1]
    Dq = (ado * b_out).sum(-1).permute(0, 2, 1)[..., None]
    g = Pm * (adp + adelta + Dq)
    b_dk = C * U * scale * torch.einsum("bhqk,bqhd->bkhd", g, aq) + U * dk_ref.abs()
    b_dq = C * U * scale * torch.einsum("bhqk,bkhd->bqhd", g, ak) + U * dq_ref.abs()
    logits = torch.einsum("bqhd,bkhd->bhqk", qd * scale, kd) + (0.0 if bias is None else bias)
    seen = torch.ones(B, 1, T, dtype=torch.bool) if mask is None else mask.any(-1)   # [B, 1, Tq]
    if mask is not None:
        logits = torch.where(mask, logits, torch.full_like(logits, -math.inf))
    lse = torch.logsumexp(logits, -1)
    return dict(out=(out, b_out), dq=(dq_ref, b_dq), dk=(dk_ref, b_dk), dv=(dv_ref, b_dv), lse=lse, seen=seen.expand(B, H, T),
                P=P, mask=mask, bias=bias)


def _ratio(got, want, bound):
    """largest |got - want| / bound (got: a kernel output, any device / dtype); an exact zero error counts 0 where the bound is 0."""
    err = (got.double().cpu() - want).abs()
    return torch.where(err == 0, torch.zeros_like(err), err / bound).max().item()


class _Checks:
    """Compares every output of a case and records its largest err / bound ratio; fails once, listing every output over."""

    def __init__(self, record_property):
        self.record, self.over = record_property, []

    def ratio(self, tag, r):
        self.record(f"ratio_{tag}", round(r, 4))
        if not r <= 1.0:
            self.over.append(f"{tag}: largest |err| / bound = {r:.3f}")

    def element(self, tag, got, want, bound):
        self.ratio(tag, _ratio(got, want, bound))

    def lse(self, lse, ref):
        lse, seen, want = lse.double().cpu(), ref["seen"], ref["lse"]
        if seen.any():
            self.ratio("lse", ((lse - want).abs() / (C * U * (1 + want.abs())))[seen].max().item())
        # a row that sees no key is marked by its lse (attn_meta.cuh, tome_b200.h)
        if not (lse[~seen] * math.log2(math.e) < MASKED_ROW_LSE2).all():
            self.over.append("lse of a row with no visible key is not below the mark")

    def done(self):
        assert not self.over, "; ".join(self.over)


def _dev(a):
    return None if a is None else torch.as_tensor(np.ascontiguousarray(a)).cuda()


def _inputs(B, T, H, D, rng):
    qkv = torch.tensor(rng.standard_normal((B, T, 3, H, D)).astype(np.float32)).cuda().bfloat16()
    dout = torch.tensor(rng.standard_normal((B, T, H, D)).astype(np.float32)).cuda().bfloat16()
    return qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2], dout


def _run(pkg, record_property, *, B, T, H, D, mask, size_kind, rate, bias_partials=False, importance=True, seed=0):
    ops, L = pkg
    rng = np.random.default_rng(seed)
    q, k, v, dout = _inputs(B, T, H, D, rng)
    gid, pos, allow = _table(mask, B, T, rng)
    size = _sizes(size_kind, B, T, rng)
    dseed, dsite = 977 + T, 0x40000003
    kw = dict(gid=_dev(gid), pos=_dev(pos), allow=_dev(allow), size=_dev(size), dropout_rate=rate, dropout_seed=dseed,
              dropout_site=dsite)
    out, lse = ops.attention_fwd(q, k, v, **kw)
    grads = {}
    for mode in ((0, 1) if D == 64 else (-1,)):   # D = 64: recomputing dQ kernel, dQ as a GEMM over the stored dS^T tiles
        part = None
        if bias_partials:
            part = torch.full((B * ((T + 127) // 128), 3 * H * D), float("nan"), device="cuda")
        L.lib().tome_attention_set_dq_from_ds(mode)
        try:
            g = ops.attention_bwd(q, k, v, out, lse, dout, bias_partial=part, **kw)
            torch.cuda.synchronize()
        finally:
            L.lib().tome_attention_set_dq_from_ds(-1)
        grads[mode] = (g, part)
    host = tuple(t.cpu() for t in (q, k, v, dout))
    ref = _reference(*host, gid, pos, allow, size, rate, dseed, dsite)
    ck = _Checks(record_property)
    ck.element("out", out, *ref["out"])
    ck.lse(lse, ref)
    for mode, ((dq, dk, dv), part) in grads.items():
        path = {0: "dq_kernel", 1: "dq_gemm", -1: "generic"}[mode]
        for name, got in (("dq", dq), ("dk", dk), ("dv", dv)):
            ck.element(f"{name}_{path}", got, *ref[name])
        if part is not None:   # column sums of the gradients per 128-token tile, reduced: within the summed element bounds
            sums = ops.reduce_rows(part).double().cpu()
            want = torch.cat([ref[n][0].sum((0, 1)).reshape(-1) for n in ("dq", "dk", "dv")])
            bound = torch.cat([ref[n][1].sum((0, 1)).reshape(-1) for n in ("dq", "dk", "dv")])
            ck.element(f"bias_partial_{path}", sums, want, bound)
    if importance and D in (64, 128, 256):
        for mode in ("row_mean", "received"):
            got = ops.attention_importance(q, k, lse, mode, **{n: kw[n] for n in ("gid", "pos", "allow", "size")})
            want = O.attention_importance(ref["P"], mode)
            ck.element(f"importance_{mode}", got, want, (C + 1) * U * want)
    ck.done()
    return out, ref, host, (gid, pos, allow, size)


# ------------------------------------------------------------------------------------------------ cases
TS = [1, 2, 31, 63, 64, 65, 127, 128, 129, 191, 193, 255, 257, 520, 536]
MASKS = ["none", "g5", "r16", "causal", "g17", "g31", "r32", "r32c"]
SIZES = ["none", "int", "mix"]
DROPOUT_TS = (65, 257, 520)
BIAS_PARTIAL_TS = (1, 129, 257)


@pytest.mark.parametrize("mask", MASKS)
@pytest.mark.parametrize("T", TS)
def test_attention_fp64(pkg, record_property, T, mask):
    """tcgen05 forward, both dQ paths of the backward, bias partials and importance at head_dim 64, element by element."""
    i = TS.index(T) * len(MASKS) + MASKS.index(mask)
    _run(pkg, record_property, B=3 if T <= 257 else 2, T=T, H=2, D=64, mask=mask, size_kind=SIZES[i % 3],
         rate=0.1 if T in DROPOUT_TS else 0.0, bias_partials=T in BIAS_PARTIAL_TS, seed=i)


@pytest.mark.parametrize("mask", ["r16", "g17", "r32c"])
def test_attention_fp64_many_heads(pkg, record_property, mask):
    """octo-base's 12 heads at a merged-sequence length."""
    _run(pkg, record_property, B=2, T=536, H=12, D=64, mask=mask, size_kind="int", rate=0.0, seed=1000 + MASKS.index(mask))


@pytest.mark.parametrize("mask", ["g17", "r32c"])
@pytest.mark.parametrize("T", [1, 65, 129])
@pytest.mark.parametrize("D", [32, 128, 256])
def test_attention_generic_fp64(pkg, record_property, D, T, mask):
    """head_dim != 64 runs the generic fp32 path: forward, dQ and dK/dV kernels (and importance at 128 / 256)."""
    _run(pkg, record_property, B=2, T=T, H=2, D=D, mask=mask, size_kind="int", rate=0.1 if T == 129 else 0.0,
         seed=2000 + D + T + len(mask))


# ------------------------------------------------------------------------------------------------ sensitivity of the bounds
@pytest.mark.parametrize("defect", ["key_tile", "group_id_plus_16", "causal_lt", "size", "partial_tile"])
def test_bound_sees_small_defects(pkg, record_property, defect):
    """The kernel output passes its bound, and fails the bound of a reference with one deliberate defect of the size a
    kernel bug would have: so the bound is tight enough to catch that bug."""
    T, mask, size_kind = {"key_tile": (257, "r32", "none"), "group_id_plus_16": (257, "r32", "none"), "causal_lt": (129, "causal", "none"),
                          "size": (65, "none", "int"), "partial_tile": (191, "g5", "none")}[defect]
    out, ref, (q, k, v, dout), (gid, pos, allow, size) = _run(pkg, record_property, B=2, T=T, H=2, D=64, mask=mask,
                                                              size_kind=size_kind, rate=0.0, importance=False, seed=3000 + T)
    args = dict(gid=gid, pos=pos, allow=allow, size=size, rate=0.0, seed=0, site=0)
    if defect == "key_tile":        # keys 64..127 skipped for queries 32..63 (one warp) of batch row 0
        ref2 = _masked_reference(q, k, v, ref, b=0, rows=slice(32, 64), cols=slice(64, 128))
    elif defect == "group_id_plus_16":    # group id g + 16 read as g (bit 4 of the group lost), for queries and keys
        args["gid"] = gid & 15
        ref2 = _reference(q, k, v, dout, **args)
    elif defect == "causal_lt":     # pos_k <= pos_q read as pos_k < pos_q
        ref2 = _reference(q, k, v, dout, causal_le=False, **args)
    elif defect == "size":          # one key's size off by one: the key whose logit shift moves its weight most
        w = ref["P"].amax(dim=(1, 2))                                     # [B, Tk]
        b, kk = np.unravel_index(int(torch.argmax(w * torch.log1p(1.0 / torch.as_tensor(size, dtype=torch.float64)))), w.shape)
        size2 = size.copy()
        size2[b, kk] += 1
        args["size"] = size2
        ref2 = _reference(q, k, v, dout, **args)
    else:                           # the last, partial key tile dropped from every row
        ref2 = _masked_reference(q, k, v, ref, b=slice(None), rows=slice(None), cols=slice(T // 64 * 64, T))
    r = _ratio(out, *ref2["out"])
    record_property("ratio_out_against_defect", round(r, 4))
    assert r > 1.0, f"the bound does not see defect {defect}: largest |err| / bound = {r:.3f}"


def _masked_reference(q, k, v, ref, b, rows, cols):
    """The forward reference (out and its bound) with keys `cols` hidden from queries `rows` of batch row(s) b."""
    B, T, H, D = q.shape
    mask = torch.ones(B, 1, T, T, dtype=torch.bool) if ref["mask"] is None else ref["mask"].clone()
    mask[b, :, rows, cols] = False
    qd, kd, vd = (t.double() for t in (q, k, v))
    out = O.attention(qd, kd, vd, mask=mask, bias=ref["bias"])
    w = O.attention_weights(qd, kd, mask=mask, bias=ref["bias"])
    bound = C * U * torch.einsum("bhqk,bkhd->bqhd", w, vd.abs()) + U * out.abs()
    return dict(out=(out, bound))
