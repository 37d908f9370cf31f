"""Parity of every CUDA kernel against the CPU oracle, through the C ABI (ctypes).  Needs a B200: `-m gpu`.

Bars (north star): indices and token sizes BIT-EXACT given the same fp32 scores; merged rows bit-exact in fp32 (same
association as the reference's sequential scatter); dense / attention / LayerNorm outputs within the bf16 tolerance
stated in each test."""
import math
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import tome_oracle as O  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from multi_modal_transformers_tokenmerge_b200 import _lib, ops as _ops
    _lib.lib()  # raises if the CUDA library is missing: no silent fallback
    return _ops


def dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


def gpu_match(ops, metric_t, r, cls=False, dis=False, **kw):
    T = kw.get("tokens", metric_t.shape[1])
    r = ops.clamp_r(T, r, cls, dis)
    nm, ni, sc = ops.sim_argmax(metric_t, class_token=cls, distill_token=dis, dump_scores=True, **kw)
    plan = ops.select_topr(nm, ni, T, r, dis) if r > 0 else None
    return r, nm, ni, sc, plan


def check_plan_exact(plan, oplan):
    np.testing.assert_array_equal(plan.node_idx.cpu().numpy(), oplan.node_idx)
    np.testing.assert_array_equal(plan.node_max.cpu().numpy(), oplan.node_max)
    np.testing.assert_array_equal(plan.edge_idx.cpu().numpy(), oplan.edge_idx)
    np.testing.assert_array_equal(plan.dst_idx.cpu().numpy(), oplan.dst_idx)
    np.testing.assert_array_equal(plan.row_map.cpu().numpy(), O.row_map(oplan))


TC = np.load(os.path.join(GOLD, "token_compression.npz"))


@pytest.mark.parametrize("name", [str(n) for n in TC["names"]])
def test_matching_and_merge_golden(ops, name):
    """GPU matching + merge on the inputs of the reference-generated goldens.  Indices are compared with the oracle
    run on the GPU's own fp32 scores (bit-exact), the scores with the golden-producing arithmetic (1e-5), and, when
    the GPU indices equal the golden ones, merged rows / sizes with the reference's outputs bit for bit."""
    B, T, Dm, C, r, cls, dis = [int(v) for v in TC[f"{name}/cfg"]]
    metric, x = TC[f"{name}/metric"], TC[f"{name}/x"]
    rc, nm, ni, sc, plan = gpu_match(ops, dev(metric), r, bool(cls), bool(dis))
    assert rc == O.clamp_r(T, r, cls, dis)
    ref_scores = O.similarity_scores(metric, cls, dis)
    got = sc.cpu().numpy()
    fin = np.isfinite(ref_scores)
    np.testing.assert_array_equal(np.isfinite(got), fin)
    np.testing.assert_allclose(got[fin], ref_scores[fin], atol=1e-5, rtol=0)
    oplan = O.plan_from_scores(got, T, rc, bool(dis))
    check_plan_exact(plan, oplan)
    # merge (fp32): bit-exact against the oracle on the same indices
    x1, s1, _, _ = ops.merge_fwd(plan, dev(x), None, 1)
    ox1, os1 = O.merge_wavg(oplan, x)
    np.testing.assert_array_equal(x1.cpu().numpy(), ox1)
    np.testing.assert_array_equal(s1.cpu().numpy(), os1[..., 0])
    xs, _, _, _ = ops.merge_fwd(plan, dev(x), None, 0)
    np.testing.assert_array_equal(xs.cpu().numpy(), O.merge(oplan, x, "sum"))
    same_idx = np.array_equal(oplan.src_idx, TC[f"{name}/src_idx"]) and np.array_equal(oplan.dst_idx, TC[f"{name}/dst_idx"])
    if name not in ("ties",):  # exact ties can legitimately resolve differently when scores differ in the last ulp
        assert same_idx, "GPU scores led to different merge indices than the reference run"
    if same_idx:
        np.testing.assert_array_equal(x1.cpu().numpy(), TC[f"{name}/x1"])
        np.testing.assert_array_equal(s1.cpu().numpy(), TC[f"{name}/s1"][..., 0])
        np.testing.assert_array_equal(xs.cpu().numpy(), TC[f"{name}/xsum"])
    # second round with non-trivial sizes
    metric2 = TC[f"{name}/metric2"]
    T1 = T - rc
    rc2, _, _, sc2, plan2 = gpu_match(ops, dev(metric2), r, bool(cls), bool(dis))
    oplan2 = O.plan_from_scores(sc2.cpu().numpy(), T1, rc2, bool(dis))
    check_plan_exact(plan2, oplan2)
    x2, s2, _, _ = ops.merge_fwd(plan2, x1, s1, 1)
    ox2, os2 = O.merge_wavg(oplan2, ox1, os1)
    np.testing.assert_array_equal(x2.cpu().numpy(), ox2)
    np.testing.assert_array_equal(s2.cpu().numpy(), os2[..., 0])
    assert np.all(s2.sum(dim=1).cpu().numpy() == T)
    # unmerge == gather through row_map; merge backward == size-weighted gather
    um = ops.merge_bwd(plan2, x2, None, None, 0)
    np.testing.assert_array_equal(um.cpu().numpy(), O.unmerge(oplan2, ox2))


# last three: BASELINE configs[3] (T0 = 2080, wrist + primary camera, 4 frames) and configs[4] (block microbench: 4096 x 1024
# at merge ratios T/2 and T/16)
@pytest.mark.parametrize("T,r,H,D,C", [(536, 16, 6, 64, 384), (75, 10, 2, 32, 64), (1024, 256, 12, 64, 768),
                                       (2080, 64, 12, 64, 768), (4096, 2048, 2, 64, 1024), (4096, 256, 2, 64, 1024)])
def test_matching_from_packed_keys_and_bf16_merge(ops, T, r, H, D, C):
    """metric = keys averaged over heads, read in place from a packed bf16 qkv buffer (the block's call site);
    bf16 merge vs oracle on the bf16-rounded inputs (fp32 arithmetic, one final rounding): bit-exact."""
    rng = np.random.default_rng(7)
    B = 3 if T <= 1024 else 2
    qkv = torch.tensor(rng.standard_normal((B, T, 3, H, D)).astype(np.float32)).cuda().bfloat16()
    nm, ni, sc = ops.sim_argmax(qkv, heads=H, dim=D, batch=B, tokens=T, batch_stride=T * 3 * H * D,
                                token_stride=3 * H * D, head_stride=D, dump_scores=True, offset_elems=H * D)
    kmean = qkv[:, :, 1].float().mean(dim=2).cpu().numpy()
    np.testing.assert_allclose(sc.cpu().numpy(), O.similarity_scores(kmean), atol=2e-5, rtol=0)
    plan = ops.select_topr(nm, ni, T, r)
    oplan = O.plan_from_scores(sc.cpu().numpy(), T, r)
    check_plan_exact(plan, oplan)
    x = torch.tensor(rng.standard_normal((B, T, C)).astype(np.float32)).cuda().bfloat16()
    size = torch.tensor(rng.integers(1, 5, size=(B, T)).astype(np.float32)).cuda()
    gid = torch.tensor(rng.integers(0, 5, size=(B, T)).astype(np.uint8)).cuda()
    pos = torch.tensor(rng.integers(0, 99, size=(B, T)).astype(np.int32)).cuda()
    x1, s1, g1, p1 = ops.merge_fwd(plan, x, size, 1, gid, pos)
    ox1, os1 = O.merge_wavg(oplan, x.float().cpu().numpy(), size.cpu().numpy()[..., None])
    np.testing.assert_array_equal(x1.float().cpu().numpy(), torch.tensor(ox1).bfloat16().float().numpy())
    np.testing.assert_array_equal(s1.cpu().numpy(), os1[..., 0])
    # group / position carried: a row keeps the metadata of its unmerged or destination token
    rm = O.row_map(oplan)
    keep = np.ones((B, T), bool)
    rank = np.empty((B, (T + 1) // 2), np.int32)
    np.put_along_axis(rank, oplan.edge_idx, np.broadcast_to(np.arange((T + 1) // 2, dtype=np.int32), rank.shape), axis=1)
    keep[:, ::2] = rank >= r
    bi, ti = np.nonzero(keep)
    g_ref = np.zeros((B, T - r), np.uint8)
    p_ref = np.zeros((B, T - r), np.int32)
    g_ref[bi, rm[bi, ti]] = gid.cpu().numpy()[bi, ti]
    p_ref[bi, rm[bi, ti]] = pos.cpu().numpy()[bi, ti]
    np.testing.assert_array_equal(g1.cpu().numpy(), g_ref)
    np.testing.assert_array_equal(p1.cpu().numpy(), p_ref)
    # backward: dx = size_t / size'_row * dy[row]
    dy = torch.tensor(rng.standard_normal((B, T - r, C)).astype(np.float32)).cuda()
    dx = ops.merge_bwd(plan, dy, size, s1, 1)
    w = size.cpu().numpy() / np.take_along_axis(s1.cpu().numpy(), rm, axis=1)
    ref = np.take_along_axis(dy.cpu().numpy(), rm[..., None], axis=1) * w[..., None]
    np.testing.assert_array_equal(dx.cpu().numpy(), ref.astype(np.float32))


def test_matching_edge_cases(ops):
    """NaN rows (zero metric rows: no epsilon in the reference normalisation), all-equal scores, r = T//2."""
    T, Dm = 12, 4
    metric = np.ones((2, T, Dm), np.float32)
    metric[1, 4] = 0.0  # zero row -> NaN scores for that even token
    rc, nm, ni, sc, plan = gpu_match(ops, dev(metric), T // 2)
    oplan = O.plan_from_scores(sc.cpu().numpy(), T, rc)
    got_nan = np.isnan(sc.cpu().numpy())
    np.testing.assert_array_equal(got_nan, np.isnan(O.similarity_scores(metric)))
    np.testing.assert_array_equal(plan.node_idx.cpu().numpy(), oplan.node_idx)
    np.testing.assert_array_equal(plan.edge_idx.cpu().numpy(), oplan.edge_idx)
    np.testing.assert_array_equal(plan.dst_idx.cpu().numpy(), oplan.dst_idx)


# ------------------------------------------------------------------------------------------------ dense
# the last five rows are the octo-base (BASELINE.json configs[2]) projections: K = 768 / 3072 at N = 2304 / 3072 / 768,
# plus the K = 2304 out-gradient and an M that is not a multiple of the 128-row tile
@pytest.mark.parametrize("m,n,k", [(256, 128, 64), (1000, 384, 384), (130, 1152, 384), (4096, 1536, 384), (384, 1536, 2000),
                                   (1072, 2304, 768), (1072, 3072, 768), (1008, 768, 3072), (1072, 768, 768), (904, 768, 2304)])
@pytest.mark.parametrize("a_mn,b_mn", [(False, True), (False, False), (True, True)])
def test_gemm_tcgen05(ops, m, n, k, a_mn, b_mn):
    """bf16 x bf16 -> fp32 accumulate.  Tolerance: |err| <= 2e-2 * sqrt(k)/16 absolute on N(0,1) operands (bf16 output
    rounding 2^-8 relative + accumulation order)."""
    if a_mn and m % 8:
        pytest.skip("MN-major A needs m % 8 == 0")
    rng = np.random.default_rng(m + n + k)
    A = torch.tensor(rng.standard_normal((m, k)).astype(np.float32)).cuda().bfloat16()
    Bm = torch.tensor(rng.standard_normal((n, k)).astype(np.float32)).cuda().bfloat16()
    a_t = A.t().contiguous() if a_mn else A
    b_t = Bm.t().contiguous() if b_mn else Bm
    ref = A.float() @ Bm.float().t()
    out = ops.gemm(a_t, b_t, m=m, n=n, k=k, a_major=int(a_mn), b_major=int(b_mn), out_dtype=torch.float32)
    torch.cuda.synchronize()
    err = (out - ref).abs().max().item()
    assert err <= 1e-3 * math.sqrt(k), f"fp32-out gemm err {err}"
    out16 = ops.gemm(a_t, b_t, m=m, n=n, k=k, a_major=int(a_mn), b_major=int(b_mn))
    rel = ((out16.float() - ref).abs() / (ref.abs() + math.sqrt(k))).max().item()
    assert rel <= 1e-2, f"bf16-out gemm rel err {rel}"


def test_gemm_epilogues_and_splitk(ops):
    rng = np.random.default_rng(3)
    m, n, k = 700, 384, 192
    A = torch.tensor(rng.standard_normal((m, k)).astype(np.float32)).cuda().bfloat16()
    W = torch.tensor(rng.standard_normal((k, n)).astype(np.float32) * 0.1).cuda().bfloat16()  # flax [in, out]
    bias = torch.tensor(rng.standard_normal(n).astype(np.float32)).cuda()
    res = torch.tensor(rng.standard_normal((m, n)).astype(np.float32)).cuda().bfloat16()
    gate = torch.tensor(rng.standard_normal((m, n)).astype(np.float32)).cuda().bfloat16()
    base = A.float() @ W.float()
    out = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, bias=bias, relu=True, residual=res)
    ref = torch.relu(base + bias) + res.float()
    assert ((out.float() - ref).abs() / (ref.abs() + 1)).max().item() <= 1e-2
    out = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, gate=gate, gate_scale=0.5)
    ref = base * (gate.float() > 0) * 0.5
    assert ((out.float() - ref).abs() / (ref.abs() + 1)).max().item() <= 1e-2
    # wgrad shape: dW[k, n] = A^T[k, m] * G[m, n], both operands MN-major, split-K, accumulate into fp32
    G = res
    dW = torch.ones(k, n, dtype=torch.float32, device="cuda")
    ops.gemm(A, G, m=k, n=n, k=m, a_major=1, b_major=1, out=dW, k_splits=3, accumulate=True)
    ref = 1.0 + A.float().t() @ G.float()
    assert (dW - ref).abs().max().item() <= 2e-3 * math.sqrt(m)
    dW2 = ops.gemm(A, G, m=k, n=n, k=m, a_major=1, b_major=1, out_dtype=torch.float32, k_splits=0)
    assert (dW2 - (ref - 1.0)).abs().max().item() <= 2e-3 * math.sqrt(m)
    # dropout: kept fraction and scaling; identical mask for identical (seed, site)
    o1 = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, dropout_rate=0.25, dropout_seed=11, dropout_site=2)
    o2 = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, dropout_rate=0.25, dropout_seed=11, dropout_site=2)
    assert torch.equal(o1, o2)
    kept = (o1 != 0).float().mean().item()
    assert abs(kept - 0.75) < 0.01
    sel = o1 != 0
    assert ((o1.float()[sel] * 0.75 - base[sel]).abs() / (base[sel].abs() + 1)).max().item() <= 2e-2
    # bias gradient: column sums
    cs = ops.colsum(res)
    assert (cs - res.float().sum(0)).abs().max().item() <= 1e-2


# ------------------------------------------------------------------------------------------------ LayerNorm
@pytest.mark.parametrize("axis", [1, 2])
# T <= 576: one CTA per (batch, slab); 700 / 1600 / 2080 / 4100: the tokens split over a cluster of 2 / 3 / 4 / 8 CTAs whose
# partial sums meet in distributed shared memory; 6000: forward cluster of 8, backward the two-pass L2 kernel (> 10 boxes / CTA)
@pytest.mark.parametrize("B,T,C", [(3, 74, 768), (4, 536, 384), (2, 33, 40), (2, 700, 72), (1, 1600, 64), (2, 2080, 96),
                                   (1, 4100, 64), (1, 6000, 40)])
def test_layernorm_fwd_bwd(ops, axis, B, T, C):
    """vs oracle.layer_norm (flax LayerNorm as configured; axis 1 = tokens) + autograd.  bf16 I/O: forward 3e-2 abs,
    dx / dgamma / dbeta within 1e-2 relative L2."""
    rng = np.random.default_rng(B * T + C)
    x = torch.tensor((rng.standard_normal((B, T, C)) * 2 + 0.5).astype(np.float32)).cuda().bfloat16()
    g = torch.tensor((1 + 0.1 * rng.standard_normal(C)).astype(np.float32)).cuda()
    bta = torch.tensor((0.1 * rng.standard_normal(C)).astype(np.float32)).cuda()
    y, mean, rstd = ops.layernorm_fwd(x, g, bta, 1e-6, axis)
    xr = x.float().cpu().requires_grad_(True)
    gr = g.cpu().requires_grad_(True)
    br = bta.cpu().requires_grad_(True)
    yr = O.layer_norm(xr, gr, br, 1e-6, "seq" if axis == 1 else "feature")
    assert (y.float().cpu() - yr).abs().max().item() <= 3e-2
    dy = torch.tensor(rng.standard_normal((B, T, C)).astype(np.float32)).cuda().bfloat16()
    dres = torch.tensor(rng.standard_normal((B, T, C)).astype(np.float32)).cuda().bfloat16()
    yr.backward(dy.float().cpu())
    dgamma = torch.zeros(C, device="cuda")
    dbeta = torch.zeros(C, device="cuda")
    dx = ops.layernorm_bwd(x, dy, g, mean, rstd, dgamma, dbeta, dres, axis)
    ref_dx = xr.grad + dres.float().cpu()
    rel = lambda a, b: ((a.double() - b.double()).norm() / b.double().norm()).item()  # noqa: E731
    assert rel(dx.float().cpu(), ref_dx) <= 1e-2
    assert rel(dgamma.cpu(), gr.grad) <= 1e-2
    assert rel(dbeta.cpu(), br.grad) <= 1e-2


@pytest.mark.parametrize("split", [1, 2, 3, 5])
def test_layernorm_token_split_matches_single_cta(ops, split):
    """The cluster kernels (tokens of a slab split over `split` CTAs, statistics exchanged through distributed shared memory)
    against the one-CTA-per-slab kernels on a shape both can run: y and dx bit-identical up to the summation order of the
    statistics (<= 1 bf16 ulp on y), saved statistics and parameter gradients to 1e-5, and the run is reproducible."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    rng = np.random.default_rng(split)
    B, T, C = 3, 536, 200
    x = dev((rng.standard_normal((B, T, C)) * 2 + 0.5).astype(np.float32), torch.bfloat16)
    g = dev((1 + 0.1 * rng.standard_normal(C)).astype(np.float32))
    bta = dev((0.1 * rng.standard_normal(C)).astype(np.float32))
    dy = dev(rng.standard_normal((B, T, C)).astype(np.float32), torch.bfloat16)
    dres = dev(rng.standard_normal((B, T, C)).astype(np.float32), torch.bfloat16)

    def run():
        y, mean, rstd = ops.layernorm_fwd(x, g, bta, 1e-6, 1)
        dgamma, dbeta = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
        dx = ops.layernorm_bwd(x, dy, g, mean, rstd, dgamma, dbeta, dres, 1)
        return y, mean, rstd, dx, dgamma, dbeta

    ref = run()
    try:
        L.lib().tome_ln_force_cluster(split)
        got = run()
        again = run()
    finally:
        L.lib().tome_ln_force_cluster(0)
    for a, b_ in zip(got, again):
        assert torch.equal(a, b_)
    rel = lambda a, b_: ((a.double() - b_.double()).norm() / b_.double().norm()).item()  # noqa: E731
    assert rel(got[1], ref[1]) <= 1e-5 and rel(got[2], ref[2]) <= 1e-5
    assert (got[0].float() - ref[0].float()).abs().max().item() <= 2 ** -5      # one bf16 ulp at |y| < 8
    assert rel(got[3].float(), ref[3].float()) <= 2e-3
    assert rel(got[4], ref[4]) <= 1e-5 and rel(got[5], ref[5]) <= 1e-5


# ------------------------------------------------------------------------------------------------ attention
def _attn_ref(q, k, v, gid, pos, allow, size):
    mask = None if gid is None else torch.as_tensor(O.dense_mask(gid, pos, gid, pos, allow))[:, None]
    bias = None if size is None else torch.log(torch.as_tensor(size))[:, None, None, :]
    return O.attention(q, k, v, mask=mask, bias=bias)


# (536, 12): octo-base heads; (2080, 12) = BASELINE.json configs[3] (two cameras, 4-frame history); (4096, 2) = configs[4]
@pytest.mark.parametrize("T,H,masked,sized", [(74, 3, True, True), (536, 6, True, True), (128, 2, False, False),
                                              (300, 4, True, False), (1000, 2, False, True), (536, 12, True, True),
                                              (2080, 12, True, True), (4096, 2, True, True)])
def test_attention_fwd(ops, T, H, masked, sized):
    """tcgen05 flash attention with group-table mask and log(size) bias vs oracle.attention (flax semantics) in fp32
    on the same bf16-rounded inputs.  Tolerance 2e-2 abs on outputs of O(1) (bf16 P and bf16 output rounding)."""
    rng = np.random.default_rng(T + H)
    B, D = (2, 64) if T < 2000 else (1, 64)
    qkv = torch.tensor(rng.standard_normal((B, T, 3, H, D)).astype(np.float32)).cuda().bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    gid = pos = allow = size = None
    if masked:
        n_img = (T - 16) // 2 - 4
        seq = f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2"
        g1, p1, allow, _ = O.sequence_groups(seq)
        pad = T - g1.shape[0]
        g1 = np.concatenate([g1, np.full(pad, g1[-1], np.uint8)])
        p1 = np.concatenate([p1, np.arange(pad, dtype=np.int32)])
        gid = np.stack([g1, rng.permutation(g1)])[:B]  # batch row 1: scrambled order, as after a merge
        pos = np.stack([p1, rng.integers(0, 50, size=T).astype(np.int32)])[:B]
        if B == 1:   # the long-sequence rows keep the scrambled (post-merge) order, the harder case
            gid, pos = np.stack([rng.permutation(g1)]), np.stack([rng.integers(0, 50, size=T).astype(np.int32)])
    if sized:
        size = rng.integers(1, 6, size=(B, T)).astype(np.float32)
    out, lse = ops.attention_fwd(q, k, v, gid=None if gid is None else dev(gid), pos=None if pos is None else dev(pos),
                                 allow=None if allow is None else dev(allow), size=None if size is None else dev(size))
    torch.cuda.synchronize()
    ref = _attn_ref(q.float().cpu(), k.float().cpu(), v.float().cpu(), gid, pos, allow, size)
    err = (out.float().cpu() - ref).abs().max().item()
    assert err <= 2e-2, f"attention fwd err {err}"
    # lse against a direct computation
    logits = torch.einsum("bqhd,bkhd->bhqk", q.float().cpu() / 8.0, k.float().cpu())
    if size is not None:
        logits = logits + torch.log(torch.as_tensor(size))[:, None, None, :]
    if gid is not None:
        m = torch.as_tensor(O.dense_mask(gid, pos, gid, pos, allow))[:, None]
        logits = torch.where(m, logits, torch.full_like(logits, -1e30))
    assert (lse.cpu() - torch.logsumexp(logits, -1)).abs().max().item() <= 2e-2


@pytest.mark.gpu
@pytest.mark.parametrize("T,growth", [(536, 6.0), (200, 20.0), (1000, -4.0)])
def test_attention_fwd_lazy_rescale(ops, T, growth):
    """The forward kernel keeps O in TMEM and rescales it only when a row maximum grows by more than 2^8.  Keys whose
    magnitude grows (or shrinks) tile by tile force that correction path on every tile (or on none); both must match
    the oracle.  Also covers a causal (code 2) group table, where visibility depends on positions."""
    rng = np.random.default_rng(7)
    B, H, D = 2, 2, 64
    qkv = rng.standard_normal((B, T, 3, H, D)).astype(np.float32)
    ramp = 1.0 + np.maximum(0.0, growth * (np.arange(T) // 64)) if growth > 0 else 1.0 + (-growth) * ((T - 1 - np.arange(T)) // 64)
    qkv[:, :, 1] *= ramp[None, :, None, None]
    qkv = torch.tensor(qkv).cuda().bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    gid = rng.integers(0, 3, size=(B, T)).astype(np.uint8)
    pos = rng.integers(0, 40, size=(B, T)).astype(np.int32)
    allow = np.array([[1, 0, 2], [1, 1, 0], [2, 1, 2]], np.uint8)   # code 2: visible iff pos_k <= pos_q
    gid[:, 0] = 0   # every group sees group-0 keys (directly or causally at pos 0): no fully masked row
    pos[:, 0] = 0
    out, lse = ops.attention_fwd(q, k, v, gid=dev(gid), pos=dev(pos), allow=dev(allow))
    torch.cuda.synchronize()
    ref = _attn_ref(q.float().cpu(), k.float().cpu(), v.float().cpu(), gid, pos, allow, None)
    err = (out.float().cpu() - ref).abs().max().item()
    assert err <= 3e-2, f"attention fwd (rescale path) err {err}"
    logits = torch.einsum("bqhd,bkhd->bhqk", q.float().cpu() / 8.0, k.float().cpu())
    m = torch.as_tensor(O.dense_mask(gid, pos, gid, pos, allow))[:, None]
    logits = torch.where(m, logits, torch.full_like(logits, -1e30))
    ref_lse = torch.logsumexp(logits, -1)
    assert ((lse.cpu() - ref_lse).abs() / ref_lse.abs().clamp_min(1.0)).max().item() <= 2e-2


@pytest.mark.gpu
@pytest.mark.parametrize("B,T,H,D", [(3, 536, 6, 64), (2, 75, 1, 30), (2, 300, 3, 128), (2, 64, 1, 296)])
def test_sim_argmax_scores_match_reference(ops, B, T, H, D):
    """tome_sim_argmax on both of its paths (tcgen05 for dim 64, fp32 planes otherwise, up to the widest accepted dim 296):
    the dumped scores match the reference's fp32 similarity of the head-mean metric, and the arg max is the exact first
    maximum of the kernel's own dumped scores."""
    rng = np.random.default_rng(B * T + D)
    src = torch.tensor(rng.standard_normal((B, T, H, D)).astype(np.float32)).cuda().bfloat16()
    nm, ni, sc = ops.sim_argmax(src, heads=H, dim=D, batch=B, tokens=T, batch_stride=T * H * D, token_stride=H * D, head_stride=D,
                                dump_scores=True)
    s = sc.cpu().numpy()
    np.testing.assert_allclose(s, O.similarity_scores(src.float().mean(dim=2).cpu().numpy()), atol=2e-5, rtol=0)
    np.testing.assert_array_equal(ni.cpu().numpy(), s.argmax(-1).astype(np.int32))
    np.testing.assert_array_equal(nm.cpu().numpy(), s.max(-1))


# ------------------------------------------------------------------------------------------------ top-k pruning
TP = np.load(os.path.join(GOLD, "token_pruning.npz"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", [str(n) for n in TP["names"]])
def test_topk_prune_golden(ops, name):
    """tome_topk_prune vs the goldens made by the reference's compute_top_k_tokens: kept rows and indices bit-exact, through
    the reference-shaped Python function (unbatched call) and batched with per-row scores, in fp32 and bf16."""
    from multi_modal_transformers_tokenmerge_b200.tokenizers import token_compression as TCm
    emb, imp = TP[f"{name}/emb"], TP[f"{name}/imp"]
    sets = [tuple(int(v) for v in s) for s in TP[f"{name}/sets"]]
    ks = [int(k) for k in TP[f"{name}/ks"]]
    kept = TCm.compute_top_k_tokens(dev(emb), dev(imp), sets, ks)
    np.testing.assert_array_equal(kept.cpu().numpy(), TP[f"{name}/kept"])
    _, oid = O.compute_top_k_tokens(emb, imp, sets, ks)
    np.testing.assert_array_equal(TCm.compute_top_k_tokens.last_ids.cpu().numpy(), oid)
    # batched, different scores per row, bf16 embeddings (16-byte rows need C % 8 == 0), scores split into two planes
    if emb.shape[1] % 8 == 0:
        rng = np.random.default_rng(3)
        B = 3
        embb = torch.tensor(rng.standard_normal((B,) + emb.shape).astype(np.float32)).cuda().bfloat16()
        p0 = rng.integers(0, 3, size=(B, emb.shape[0])).astype(np.float32)
        p1 = rng.integers(0, 3, size=(B, emb.shape[0])).astype(np.float32)
        out, ids = ops.topk_prune(embb, dev(np.stack([p0, p1])), [s[0] for s in sets], [s[1] for s in sets], ks)
        for b in range(B):
            okept, oid = O.compute_top_k_tokens(embb[b].float().cpu().numpy(), p0[b] + p1[b], sets, ks)
            np.testing.assert_array_equal(ids[b].cpu().numpy(), oid)
            np.testing.assert_array_equal(out[b].float().cpu().numpy(), okept)


@pytest.mark.gpu
def test_topk_prune_errors_and_nan(ops):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    emb = torch.zeros(1, 8, 4, device="cuda")
    imp = torch.tensor([[0.5, float("nan"), 0.1, 0.9, 0.9, 0.2, 0.3, 0.0]], device="cuda")
    _, ids = ops.topk_prune(emb, imp, [0], [8], [4])
    assert ids[0].tolist() == [1, 3, 4, 0]            # NaN ranks above every number; equal scores keep the lower index first
    with pytest.raises(L.TomeError):
        ops.topk_prune(emb, imp, [0], [8], [9])       # k > n, as jax.lax.top_k
    with pytest.raises(L.TomeError):
        ops.topk_prune(emb, imp, [4], [8], [2])       # set leaves the sequence


@pytest.mark.gpu
@pytest.mark.parametrize("m,n", [(1000, 384), (4097, 1536), (130, 40)])
@pytest.mark.parametrize("epilogue", ["specialised", "generic"])
def test_dropout_mask_identical_in_forward_epilogue_and_backward_pass(ops, m, n, epilogue):
    """Hidden dropout is never stored: the forward GEMM epilogue and the backward pass (tome_dropout_colsum_bf16) each
    regenerate the mask from (seed, site, row, column).  A GEMM whose every output is exactly 1 exposes the epilogue's mask;
    the backward pass over a tensor of ones must reproduce it bit for bit, and its column sums must be those of its output.
    `generic` adds a ReLU-free, bias-free combination that takes the run-time-flag epilogue instead of a specialised one."""
    k = 8
    A = torch.full((m, k), 0.125, device="cuda").bfloat16()
    W = torch.ones(k, n, device="cuda").bfloat16()
    bias = torch.zeros(n, device="cuda")
    resid = torch.zeros(m, n, device="cuda").bfloat16()
    rate, seed, site = 0.1, 1234567, 17
    if epilogue == "specialised":   # bias + dropout + residual: the out-projection / MLP-2 forward epilogue
        fwd = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, bias=bias, residual=resid, dropout_rate=rate, dropout_seed=seed, dropout_site=site)
    else:                            # dropout alone: no specialisation exists, the generic epilogue runs
        fwd = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, dropout_rate=rate, dropout_seed=seed, dropout_site=site)
    bwd, cs = ops.dropout_colsum(torch.ones(m, n, device="cuda").bfloat16(), rate, seed, site)
    torch.cuda.synchronize()
    assert torch.equal(fwd, bwd)
    kept = (fwd != 0).float().mean().item()
    assert abs(kept - 0.9) < 0.01
    vals = fwd[fwd != 0].float().unique()
    assert vals.numel() == 1 and abs(vals.item() - 1.0 / 0.9) < 1e-2      # inverted dropout scaling, rounded to bf16
    assert (cs - bwd.float().sum(0)).abs().max().item() <= 1e-3 * m
    other, _ = ops.dropout_colsum(torch.ones(m, n, device="cuda").bfloat16(), rate, seed, site + 1)
    assert not torch.equal(other, bwd)                                       # another site draws another mask


@pytest.mark.gpu
@pytest.mark.parametrize("T,H,D,rate", [(74, 3, 256, 0.0), (74, 3, 256, 0.1), (130, 2, 32, 0.0), (90, 2, 40, 0.25)])
def test_attention_generic_head_dims(ops, T, H, D, rate):
    """head_dim != 64 (the literal reference config has 3 heads x 256) runs on the generic attention path: forward, lse and
    dq / dk / dv vs the oracle with mask, log(size) bias and -- handed the exact regenerated mask -- weight dropout."""
    rng = np.random.default_rng(T * D + H)
    B = 2
    qkv = torch.tensor(rng.standard_normal((B, T, 3, H, D)).astype(np.float32)).cuda().bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    n_img = (T - 16) // 2 - 4
    g1, p1, allow, _ = O.sequence_groups(f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2")
    pad = T - g1.shape[0]
    g1 = np.concatenate([g1, np.full(pad, g1[-1], np.uint8)])
    p1 = np.concatenate([p1, np.arange(pad, dtype=np.int32)])
    gid, pos = np.stack([g1, rng.permutation(g1)]), np.stack([p1, rng.integers(0, 50, size=T).astype(np.int32)])
    size = rng.integers(1, 4, size=(B, T)).astype(np.float32)
    seed, site = 4242, 0x40000001
    kw = dict(gid=dev(gid), pos=dev(pos), allow=dev(allow), size=dev(size), dropout_rate=rate, dropout_seed=seed, dropout_site=site)
    out, lse = ops.attention_fwd(q, k, v, **kw)
    dout = torch.tensor(rng.standard_normal((B, T, H, D)).astype(np.float32)).cuda().bfloat16()
    dq, dk, dvv = ops.attention_bwd(q, k, v, out, lse, dout, **kw)
    torch.cuda.synchronize()
    drop_keep = None
    if rate > 0:
        keep, p_eff = O.dropout_keep_mask(T, T, rate, seed, site)
        drop_keep = torch.as_tensor(keep.astype(np.float32) / (1.0 - p_eff))[None, None]
    qr, kr, vr = (t.float().cpu().requires_grad_(True) for t in (q, k, v))
    mask = torch.as_tensor(O.dense_mask(gid, pos, gid, pos, allow))[:, None]
    bias = torch.log(torch.as_tensor(size))[:, None, None, :]
    ref = O.attention(qr, kr, vr, mask=mask, bias=bias, drop_keep=drop_keep)
    rel = lambda a, b: ((a.double() - b.double()).norm() / (b.double().norm() + 1e-12)).item()  # noqa: E731
    assert rel(out.float().cpu(), ref.detach()) <= 1e-2
    logits = torch.einsum("bqhd,bkhd->bhqk", q.float().cpu() / math.sqrt(D), k.float().cpu()) + bias
    logits = torch.where(mask, logits, torch.full_like(logits, -1e30))
    assert (lse.cpu() - torch.logsumexp(logits, -1)).abs().max().item() <= 2e-2
    ref.backward(dout.float().cpu())
    for name, got, want in (("dq", dq, qr.grad), ("dk", dk, kr.grad), ("dv", dvv, vr.grad)):
        assert rel(got.float().cpu(), want) <= 1.5e-2, name


# ------------------------------------------------------------------------------------------------ action heads
def rel_err(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def _head_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "action_heads.npz"))


@pytest.mark.parametrize("name", ["cont_small", "cont_octo", "cont_saturated"])
def test_continuous_head_matches_reference_goldens(ops, name):
    """tome_action_head_fwd (continuous) against outputs of the reference's own ContinuousActionHead.__call__
    (continuous.py:16-25, executed under the numpy shim) and the l2 loss of octo.py:163-165: fp32, 1e-5."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    g = _head_golden()
    ro = torch.tensor(g[f"{name}/readouts"]).cuda()
    w, b = torch.tensor(g[f"{name}/kernel"]).cuda(), torch.tensor(g[f"{name}/bias"]).cuda()
    act = torch.tensor(g[f"{name}/actions"]).cuda()
    out, loss, _ = ops.action_head_fwd(ro, w, b, kind=L.HEAD_CONTINUOUS_L2, max_action=float(g[f"{name}/max_action"]), actions=act)
    np.testing.assert_allclose(out.cpu().numpy(), g[f"{name}/pred"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(loss[1:].cpu().numpy(), g[f"{name}/loss"], rtol=1e-4, atol=1e-6)
    np.testing.assert_allclose(loss[0].item(), g[f"{name}/loss"].mean(), rtol=1e-4)


@pytest.mark.parametrize("name", ["cat_small", "cat_octo", "cat_edges"])
def test_categorical_head_matches_reference_goldens(ops, name):
    """tome_action_head_fwd (categorical) against the reference's CategoricalActionHead.__call__ and assign_bins
    (categorical.py:12-40, executed) + the cross-entropy of octo.py:183-187; cat_edges sits on bin edges and outside the
    range, where the reference's 1-based digitize gives all-zero labels (loss 0) or class 0."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    g = _head_golden()
    A, bins = (int(v) for v in g[f"{name}/cfg"])
    ro = torch.tensor(g[f"{name}/readouts"]).cuda()
    w, b = torch.tensor(g[f"{name}/kernel"]).cuda(), torch.tensor(g[f"{name}/bias"]).cuda()
    act = torch.tensor(g[f"{name}/actions"]).cuda()
    out, loss, _ = ops.action_head_fwd(ro, w, b, kind=L.HEAD_CATEGORICAL_CE, max_action=float(g[f"{name}/max_action"]), groups=A,
                                       actions=act)
    np.testing.assert_allclose(out.cpu().numpy(), g[f"{name}/logits"], rtol=1e-5, atol=2e-6)
    np.testing.assert_allclose(loss[1:].cpu().numpy(), g[f"{name}/loss"].sum(-1), rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(loss[0].item(), g[f"{name}/loss"].mean(), rtol=1e-4)


@pytest.mark.parametrize("kind,dtype", [("continuous", torch.float32), ("categorical", torch.float32), ("continuous", torch.bfloat16),
                                        ("categorical", torch.bfloat16)])
def test_action_head_backward_vs_oracle_autograd(ops, kind, dtype):
    """dW, db and dx of the head + loss against autograd of the oracle, with the readouts scattered over a longer sequence
    through `origin` -- including two readouts that share a row (merged tokens), whose gradients must add."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    rng = np.random.default_rng(5)
    B, T, C, n = 5, 40, 96, 8
    groups, feats = (1, 6) if kind == "continuous" else (4, 12)
    mx = 2.0
    x = torch.tensor(rng.standard_normal((B, T, C)).astype(np.float32)).to(dtype)
    origin = np.stack([rng.choice(T, size=n, replace=False) for _ in range(B)]).astype(np.int32)
    origin[1, 3] = origin[1, 2]          # two readouts merged into the same row
    origin[2, 7] = origin[2, 0]
    w = (rng.standard_normal((C, feats)) * 0.2).astype(np.float32)
    b = (rng.standard_normal(feats) * 0.1).astype(np.float32)
    if kind == "continuous":
        act = rng.uniform(-mx, mx, size=(B, feats)).astype(np.float32)
    else:
        act = rng.uniform(-mx * 1.2, mx, size=(B, groups)).astype(np.float32)
    k = L.HEAD_CONTINUOUS_L2 if kind == "continuous" else L.HEAD_CATEGORICAL_CE
    out, loss, st = ops.action_head_fwd(x.cuda(), torch.tensor(w).cuda(), torch.tensor(b).cuda(), kind=k, max_action=mx,
                                        groups=groups, origin=torch.tensor(origin).cuda(), actions=torch.tensor(act).cuda(),
                                        keep_for_backward=True)
    dw = torch.zeros(C, feats, device="cuda")
    db = torch.zeros(feats, device="cuda")
    dx = ops.action_head_bwd(st, dw, db)
    torch.cuda.synchronize()
    xr = x.float().clone().requires_grad_(True)
    wr, br = torch.tensor(w, requires_grad=True), torch.tensor(b, requires_grad=True)
    ro = torch.gather(xr, 1, torch.as_tensor(origin, dtype=torch.long)[..., None].expand(-1, -1, C))
    if kind == "continuous":
        want = O.continuous_action_head(ro, wr, br, mx)
        ref = O.l2_loss(want, torch.tensor(act)).mean()
    else:
        want = O.categorical_action_head(ro, wr, br, groups)
        ref = O.ce_loss(want, act, mx, feats).mean()
    ref.backward()
    np.testing.assert_allclose(out.cpu().numpy().reshape(want.shape), want.detach().numpy(), rtol=2e-5, atol=2e-5)
    assert abs(loss[0].item() - ref.item()) <= 1e-5 * abs(ref.item()) + 1e-7
    tol = 1e-5 if dtype == torch.float32 else 1e-2      # dx is stored in x's dtype
    assert rel_err(dw.cpu(), wr.grad) <= 1e-5 and rel_err(db.cpu(), br.grad) <= 1e-5
    assert rel_err(dx.float().cpu(), xr.grad) <= tol
    rows = torch.zeros(B, T, dtype=torch.bool)
    rows.scatter_(1, torch.as_tensor(origin, dtype=torch.long), True)
    assert torch.all(dx.float().cpu()[~rows] == 0)
    # accumulate semantics of dw / db
    ops.action_head_bwd(st, dw, db, want_dx=False)
    assert rel_err(dw.cpu(), 2 * wr.grad) <= 1e-5


def test_action_head_rejects_bad_arguments(ops):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    x = torch.zeros(2, 6, 16, device="cuda")
    w = torch.zeros(16, 4, device="cuda")
    with pytest.raises(L.TomeError, match="groups must be 1"):
        ops.action_head_fwd(x, w, None, kind=L.HEAD_CONTINUOUS_L2, max_action=1.0, groups=2)
    with pytest.raises(L.TomeError, match="do not split"):
        ops.action_head_fwd(x, w, None, kind=L.HEAD_CATEGORICAL_CE, max_action=1.0, groups=4)
    with pytest.raises(L.TomeError, match="max_action"):
        ops.action_head_fwd(x, w, None, kind=L.HEAD_CONTINUOUS_L2, max_action=0.0)


def _diffusion_flat(p):
    return np.concatenate([p[k].reshape(-1) for k in ("fourier_kernel", "tw1", "tb1", "tw2", "tb2", "w1", "b1", "w2", "b2")])


@pytest.mark.parametrize("name", ["diff_small", "diff_mid"])
def test_diffusion_head_matches_reference_goldens(ops, name):
    """tome_diffusion_head_fwd against the reference's own OctoDenoise / FourierFeatures / MLPBlock outputs
    (diffusion.py:29-64, executed under the shim) on the golden parameters and draws.  The wide Dense layers run on the
    bf16 tensor-core GEMM, so the bar is the bf16 one: relative L2 error of the prediction <= 2e-2, loss within 2e-2."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    g = _head_golden()
    p = {k: g[f"{name}/p/{k}"] for k in L.DIFFUSION_PARAMS}
    ro = torch.tensor(g[f"{name}/readouts"]).cuda().bfloat16()
    B, n, C = ro.shape
    A, steps = g[f"{name}/actions"].shape[1], int(g[f"{name}/steps"])
    desc = L.DiffusionDesc(B, n, C, n, A, p["tw1"].shape[0], p["tw1"].shape[1], p["tw2"].shape[1], p["w1"].shape[1], steps)
    pred, loss, _ = ops.diffusion_head_fwd(ro, torch.tensor(_diffusion_flat(p)).cuda(), desc, torch.tensor(g[f"{name}/actions"]).cuda(),
                                           torch.tensor(g[f"{name}/noise"]).cuda(), torch.tensor(g[f"{name}/time"].reshape(-1)).cuda(),
                                           torch.tensor(O.alpha_hats(steps)).cuda())
    assert rel_err(pred.cpu(), torch.tensor(g[f"{name}/pred"])) <= 2e-2
    assert abs(loss[0].item() - float(g[f"{name}/loss"])) <= 2e-2 * float(g[f"{name}/loss"])


def test_diffusion_head_backward_vs_oracle_autograd(ops):
    """Every parameter gradient of the diffusion head (Fourier kernel, both MLPBlocks) and the gradient reaching the
    readout rows, against autograd of oracle.denoise_loss on the same bf16-rounded weights and inputs; readouts scattered
    through `origin` with one shared row.  Both hidden biases are shifted by +12 so every ReLU gate is open and the
    comparison measures the kernels, not gates that flip when a pre-activation within bf16 rounding of zero is computed
    from bf16 instead of fp32 inputs (same protocol as the stack tests).  Relative L2 error <= 3e-2 (bf16 GEMM operands,
    bf16 intermediate gradients); the Fourier-kernel gradient, a sum over the batch of terms of both signs scaled by
    2 pi t, is allowed 0.1."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    rng = np.random.default_rng(9)
    B, T, C, n, A, F, Ht, To, H, steps = 16, 24, 64, 4, 8, 32, 48, 40, 96, 16
    desc = L.DiffusionDesc(B, T, C, n, A, F, Ht, To, H, steps)
    r_ = lambda *s: (rng.standard_normal(s) * 0.3).astype(np.float32)  # noqa: E731
    p = dict(fourier_kernel=r_(F // 2, 1) * 0.1, tw1=r_(F, Ht), tb1=r_(Ht) + 12, tw2=r_(Ht, To) * 0.3, tb2=r_(To), w1=r_(A + To + C, H) * 0.3,
             b1=r_(H) + 12, w2=r_(H, A), b2=r_(A))
    x = torch.tensor(rng.standard_normal((B, T, C)).astype(np.float32)).bfloat16()
    origin = np.stack([rng.choice(T, size=n, replace=False) for _ in range(B)]).astype(np.int32)
    origin[3, 1] = origin[3, 0]
    actions = rng.uniform(-1, 1, (B, A)).astype(np.float32)
    noise = rng.standard_normal((B, A)).astype(np.float32)
    time = rng.integers(0, steps, B).astype(np.int32)
    ah = O.alpha_hats(steps)
    flat = torch.tensor(_diffusion_flat(p)).cuda()
    pred, loss, st = ops.diffusion_head_fwd(x.cuda(), flat, desc, torch.tensor(actions).cuda(), torch.tensor(noise).cuda(),
                                            torch.tensor(time).cuda(), torch.tensor(ah).cuda(), origin=torch.tensor(origin).cuda())
    grads = torch.zeros_like(flat)
    dx = ops.diffusion_head_bwd(st, grads)
    torch.cuda.synchronize()
    # oracle on the weights the GEMMs consume: bf16-rounded kernels of the three wide layers, fp32 everything else
    pt = {k: torch.tensor(v) for k, v in p.items()}
    for k in ("tw1", "tw2", "w1"):
        pt[k] = pt[k].bfloat16().float()
    for t in pt.values():
        t.requires_grad_(True)
    xr = x.float().clone().requires_grad_(True)
    ro = torch.gather(xr, 1, torch.as_tensor(origin, dtype=torch.long)[..., None].expand(-1, -1, C))
    ref, want = O.denoise_loss(ro, torch.tensor(actions), torch.tensor(time)[:, None], torch.tensor(noise), ah, pt)
    ref.backward()
    assert rel_err(pred.cpu(), want.detach()) <= 2e-2
    assert abs(loss[0].item() - ref.item()) <= 2e-2 * abs(ref.item())
    off = 0
    for k in L.DIFFUSION_PARAMS:
        nel = p[k].size
        e = rel_err(grads[off: off + nel].cpu().reshape(p[k].shape), pt[k].grad)
        assert e <= (0.1 if k == "fourier_kernel" else 3e-2), f"grad {k}: rel err {e}"
        off += nel
    assert rel_err(dx.float().cpu(), xr.grad) <= 3e-2


# ------------------------------------------------------------------------------------------------ full-batch behaviour
@pytest.mark.parametrize("T", [536, 600])
def test_attention_full_batch_reproducible_and_accurate(ops, T):
    """At the bench batch (256 x 6 heads: 7 680 CTAs, several waves, two CTAs per SM) the forward must be bit-reproducible
    and as accurate as at small batch.  This is the test that exposes a shared-memory ring slot released before the loads
    from it have returned (profiles/r01c_attention.md): invisible at small batch and for T a multiple of 64.  The reference
    here is torch's fp32 attention on the same bf16 inputs (checker only); masked / dropout variants and the backward are
    checked for reproducibility."""
    torch.manual_seed(T)
    B, H, D = 256, 6, 64
    qkv = torch.randn(B, T, 3, H, D, device="cuda").bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    ref = torch.nn.functional.scaled_dot_product_attention(q.transpose(1, 2).float(), k.transpose(1, 2).float(),
                                                           v.transpose(1, 2).float()).transpose(1, 2)
    runs = []
    for _ in range(4):
        o, l = ops.attention_fwd(q, k, v)
        torch.cuda.synchronize()
        runs.append((o.clone(), l.clone()))
    assert (runs[0][0].float() - ref).abs().max().item() <= 0.02
    for o, l in runs[1:]:
        assert torch.equal(o, runs[0][0]) and torch.equal(l, runs[0][1])
    # masked (+ sizes, + weight dropout): reproducible forward and backward
    n_img = (T - 16) // 2 - 4
    g1, p1, allow, _ = O.sequence_groups(f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2")
    pad = T - g1.shape[0]
    gid = torch.tensor(np.concatenate([g1, np.full(pad, g1[-1], np.uint8)])).cuda().repeat(B, 1).contiguous()
    pos = torch.tensor(np.concatenate([p1, np.arange(pad, dtype=np.int32)])).cuda().repeat(B, 1).contiguous()
    size = torch.randint(1, 4, (B, T), device="cuda").float()
    kw = dict(gid=gid, pos=pos, allow=torch.tensor(allow).cuda(), size=size)
    dout = torch.randn(B, T, H, D, device="cuda").bfloat16()
    for extra in (dict(), dict(dropout_rate=0.1, dropout_seed=11, dropout_site=0x40000001)):
        outs = []
        for _ in range(3):
            o, l = ops.attention_fwd(q, k, v, **kw, **extra)
            dq, dk, dv = ops.attention_bwd(q, k, v, o, l, dout, **kw, **extra)
            torch.cuda.synchronize()
            outs.append([t.clone() for t in (o, l, dq, dk, dv)])
        for other in outs[1:]:
            for a, b in zip(outs[0], other):
                assert torch.equal(a, b)


def test_full_batch_ops_match_torch(ops):
    """The hot ops at the bench's full size (B = 256, T = 536, C = 384: 137 216 rows), against torch on the same bf16 inputs
    (checker only; far too large for the CPU oracle): attention backward, the projection / MLP GEMMs with their fused
    epilogues, token-axis LayerNorm, and merge_wavg on sampled batch rows against the oracle."""
    torch.manual_seed(1)
    B, T, C, H, D, F = 256, 536, 384, 6, 64, 1536
    M = B * T
    # attention backward vs autograd of fp32 attention
    qkv = torch.randn(B, T, 3, H, D, device="cuda").bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    o, l = ops.attention_fwd(q, k, v)
    do = torch.randn(B, T, H, D, device="cuda").bfloat16()
    dq, dk, dv = ops.attention_bwd(q, k, v, o, l, do)
    qf, kf, vf = (t.transpose(1, 2).float().detach().requires_grad_(True) for t in (q, k, v))
    ref = torch.nn.functional.scaled_dot_product_attention(qf, kf, vf)
    ref.backward(do.transpose(1, 2).float())
    for name, got, want in (("dq", dq, qf.grad), ("dk", dk, kf.grad), ("dv", dv, vf.grad)):
        e = rel_err(got.float(), want.transpose(1, 2))
        assert e <= 2e-2, f"{name}: rel err {e}"
    del qf, kf, vf, ref
    # GEMMs: bias + relu (fc1), bias + residual (fc2), gated dgrad, weight gradient over all 137 216 rows
    x = torch.randn(M, C, device="cuda").bfloat16()
    w1 = (torch.randn(C, F, device="cuda") * 0.05).bfloat16()
    b1 = torch.randn(F, device="cuda") * 0.1
    h1 = ops.gemm(x, w1, m=M, n=F, k=C, b_major=1, bias=b1, relu=True)
    want = torch.relu(x.float() @ w1.float() + b1)
    assert rel_err(h1.float(), want) <= 1e-2
    w2 = (torch.randn(F, C, device="cuda") * 0.05).bfloat16()
    b2 = torch.randn(C, device="cuda") * 0.1
    y2 = ops.gemm(h1, w2, m=M, n=C, k=F, b_major=1, bias=b2, residual=x)
    assert rel_err(y2.float(), h1.float() @ w2.float() + b2 + x.float()) <= 1e-2
    dy = torch.randn(M, C, device="cuda").bfloat16()
    dh = ops.gemm(dy, w2, m=M, n=F, k=C, gate=h1, gate_scale=1.0)
    assert rel_err(dh.float(), (dy.float() @ w2.float().t()) * (h1 > 0)) <= 1e-2
    dw = ops.gemm(x, dh, m=C, n=F, k=M, a_major=1, b_major=1, out_dtype=torch.float32)
    assert rel_err(dw, x.float().t() @ dh.float()) <= 1e-2
    del want
    # LayerNorm over tokens
    x3 = x.view(B, T, C)
    gamma, beta = torch.rand(C, device="cuda") + 0.5, torch.randn(C, device="cuda") * 0.1
    y, mean, rstd = ops.layernorm_fwd(x3, gamma, beta, axis=1)
    xf = x3.float()
    mu = xf.mean(dim=1, keepdim=True)
    var = (xf * xf).mean(dim=1, keepdim=True) - mu * mu
    assert rel_err(y.float(), (xf - mu) * torch.rsqrt(var.clamp_min(0) + 1e-6) * gamma + beta) <= 1e-2
    # matching + merge_wavg: sampled batch rows against the oracle, bit-exact given the GPU's own scores
    kk = qkv[:, :, 1].reshape(B, T, H * D).contiguous()
    nm, ni, _ = ops.sim_argmax(kk, heads=H, dim=D, batch_stride=T * H * D, token_stride=H * D, head_stride=D, tokens=T, batch=B)
    plan = ops.select_topr(nm, ni, T, 16)
    xs = torch.randn(B, T, C, device="cuda")
    size = torch.randint(1, 4, (B, T), device="cuda").float()
    x1, s1, _, _ = ops.merge_fwd(plan, xs, size, 1)
    for b_ in (0, 37, 128, 255):
        oplan = O.plan_from_node(nm[b_:b_ + 1].cpu().numpy(), ni[b_:b_ + 1].cpu().numpy(), T, 16)
        np.testing.assert_array_equal(plan.edge_idx[b_:b_ + 1].cpu().numpy(), oplan.edge_idx)
        ox1, os1 = O.merge_wavg(oplan, xs[b_:b_ + 1].cpu().numpy(), size[b_:b_ + 1].cpu().numpy()[..., None])
        np.testing.assert_array_equal(x1[b_:b_ + 1].cpu().numpy(), ox1)
        np.testing.assert_array_equal(s1[b_:b_ + 1].cpu().numpy(), os1[..., 0])


@pytest.mark.parametrize("m,n,k,rate", [(1000, 384, 256, 0.0), (4097, 1536, 384, 0.1), (130, 160, 64, 0.25)])
def test_gemm_relu_gate_bits(ops, m, n, k, rate):
    """A ReLU epilogue can emit its gate as one bit per element (after dropout, so dropped elements are gated too), and a
    later GEMM gated by those bits must equal, bit for bit, the same GEMM gated by the bf16 output itself -- for the
    specialised epilogues (K-major A, the stack's layouts) and the generic one (fp32 output)."""
    rng = np.random.default_rng(m + n)
    A = dev(rng.standard_normal((m, k)).astype(np.float32) * 0.3, torch.bfloat16)
    W = dev(rng.standard_normal((k, n)).astype(np.float32) * 0.3, torch.bfloat16)
    bias = dev(rng.standard_normal(n).astype(np.float32) * 0.1)
    words = (n + 31) // 32
    bits = torch.full((m, words), -1, dtype=torch.int32, device="cuda")
    h = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, bias=bias, relu=True, dropout_rate=rate, dropout_seed=5, dropout_site=9,
                 relu_bits_out=bits)
    h_plain = ops.gemm(A, W, m=m, n=n, k=k, b_major=1, bias=bias, relu=True, dropout_rate=rate, dropout_seed=5, dropout_site=9)
    assert torch.equal(h, h_plain)                      # asking for the bits does not change the output
    want = (h > 0).cpu().numpy()
    got = np.unpackbits(bits.cpu().numpy().view(np.uint8).reshape(m, words * 4), axis=1, bitorder="little")[:, :n].astype(bool)
    np.testing.assert_array_equal(got, want)
    if rate:
        assert 0.3 < want.mean() < 0.5                  # about half the pre-activations positive, a tenth of those dropped
    dy = dev(rng.standard_normal((m, 64)).astype(np.float32), torch.bfloat16)
    W2 = dev(rng.standard_normal((n, 64)).astype(np.float32) * 0.3, torch.bfloat16)       # [N, K] K-major: the dgrad layout
    g_rows = ops.gemm(dy, W2, m=m, n=n, k=64, gate=h, gate_scale=1.25)
    g_bits = ops.gemm(dy, W2, m=m, n=n, k=64, gate_bits=bits, gate_scale=1.25)
    assert torch.equal(g_rows, g_bits)
    f_rows = ops.gemm(dy, W2, m=m, n=n, k=64, gate=h, gate_scale=1.25, out_dtype=torch.float32)      # generic epilogue
    f_bits = ops.gemm(dy, W2, m=m, n=n, k=64, gate_bits=bits, gate_scale=1.25, out_dtype=torch.float32)
    assert torch.equal(f_rows, f_bits)
    bits2 = torch.zeros_like(bits)
    ops.gemm(A, W, m=m, n=n, k=k, b_major=1, bias=bias, relu=True, out_dtype=torch.float32, relu_bits_out=bits2)   # generic writer
    if rate == 0.0:
        assert torch.equal(bits2, bits)


@pytest.mark.parametrize("T,rate", [(536, 0.0), (300, 0.1), (74, 0.0)])
def test_attention_bwd_dq_paths_agree(ops, T, rate):
    """dQ as a batched GEMM over the dS^T tiles stored by the dK/dV kernel (the default up to 3 072 tokens) against the
    recomputing dQ kernel: same bf16 dS (both form it from the bf16-rounded P, in the same operation order), same accumulation
    order, so dq must agree bit for bit; dk / dv come from the same kernel in both modes."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    setter = L.lib().tome_attention_set_dq_from_ds
    rng = np.random.default_rng(T)
    B, H, D = 4, 3, 64
    qkv = dev(rng.standard_normal((B, T, 3, H, D)).astype(np.float32), torch.bfloat16)
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    n_img = (T - 16) // 2 - 4
    g1, p1, allow, _ = O.sequence_groups(f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2")
    pad = T - g1.shape[0]
    gid = dev(np.tile(np.concatenate([g1, np.full(pad, g1[-1], np.uint8)]), (B, 1)))
    pos = dev(np.tile(np.concatenate([p1, np.arange(pad, dtype=np.int32)]), (B, 1)))
    size = dev(rng.integers(1, 4, size=(B, T)).astype(np.float32))
    kw = dict(gid=gid, pos=pos, allow=dev(allow), size=size, dropout_rate=rate, dropout_seed=3, dropout_site=0x40000002)
    o, l = ops.attention_fwd(q, k, v, **kw)
    do = dev(rng.standard_normal((B, T, H, D)).astype(np.float32), torch.bfloat16)
    try:
        setter(0)
        a = [t.clone() for t in ops.attention_bwd(q, k, v, o, l, do, **kw)]
        setter(1)
        b = [t.clone() for t in ops.attention_bwd(q, k, v, o, l, do, **kw)]
    finally:
        setter(-1)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("m,n,k", [(4097, 1536, 384), (1000, 384, 256), (130, 160, 64), (70000, 768, 128)])
def test_gemm_epilogue_column_sums(ops, m, n, k):
    """A GEMM epilogue can leave the column sums of its bf16 output per 128-row tile (the Dense bias gradient without a second
    pass over the tensor): reduced over the tiles they must equal the column sums of the output it wrote -- rows past M
    excluded even when the epilogue adds a bias to them -- for the gated data gradient, the plain one and a forward layer, in
    every CTA mode; asking for them must not change the output; and the result is reproducible bit for bit."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    rng = np.random.default_rng(m + n + k)
    A = dev(rng.standard_normal((m, k)).astype(np.float32) * 0.5, torch.bfloat16)
    Wk = dev(rng.standard_normal((n, k)).astype(np.float32) * 0.5, torch.bfloat16)       # K-major (dgrad layout)
    Wf = dev(rng.standard_normal((k, n)).astype(np.float32) * 0.5, torch.bfloat16)       # [in, out] (forward layout)
    bias = dev(rng.standard_normal(n).astype(np.float32))
    words = (n + 31) // 32
    bits = torch.randint(-2**31, 2**31 - 1, (m, words), dtype=torch.int32, device="cuda")
    tiles = (m + 127) // 128
    cases = [dict(b=Wk, b_major=0, gate_bits=bits, gate_scale=1.25), dict(b=Wk, b_major=0), dict(b=Wf, b_major=1, bias=bias),
             dict(b=Wf, b_major=1, bias=bias, relu=True, dropout_rate=0.1, dropout_seed=3, dropout_site=2)]
    try:
        for mode in (-1, 0, 1, 2):
            L.lib().tome_gemm_force_tile(mode, 0)
            for kw in cases:
                kw = dict(kw)
                b = kw.pop("b")
                plain = ops.gemm(A, b, m=m, n=n, k=k, **kw)
                part = torch.full((tiles, n), float("nan"), device="cuda")
                out = ops.gemm(A, b, m=m, n=n, k=k, colsum_partial=part, **kw)
                assert torch.equal(out, plain)
                got = ops.reduce_rows(part)
                want = out.double().sum(0)
                scale = out.double().abs().sum(0).max().item()
                assert (got.double() - want).abs().max().item() <= 2e-6 * scale + 1e-6, (mode, list(kw))
                part2 = torch.zeros_like(part)
                ops.gemm(A, b, m=m, n=n, k=k, colsum_partial=part2, **kw)
                assert torch.equal(part, part2)
    finally:
        L.lib().tome_gemm_force_tile(-1, 0)
    with pytest.raises(Exception):   # fp32 outputs take the generic epilogue, which has no column sums
        ops.gemm(A, Wk, m=m, n=n, k=k, out_dtype=torch.float32, colsum_partial=torch.zeros(tiles, n, device="cuda"))


@pytest.mark.parametrize("T,H,rate,from_ds", [(536, 3, 0.0, 1), (300, 2, 0.1, 1), (74, 2, 0.0, 0), (257, 1, 0.1, 0)])
def test_attention_bwd_bias_partials(ops, T, H, rate, from_ds):
    """The attention-backward epilogues can leave the column sums of every 128-token tile of dq / dk / dv (the packed q/k/v
    projection's bias gradient): reduced over the tiles they equal the column sums of the gradients written, on both dQ paths,
    and asking for them changes no gradient bit."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    setter = L.lib().tome_attention_set_dq_from_ds
    rng = np.random.default_rng(T + H)
    B, D = 3, 64
    qkv = dev(rng.standard_normal((B, T, 3, H, D)).astype(np.float32), torch.bfloat16)
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    size = dev(rng.integers(1, 4, size=(B, T)).astype(np.float32))
    kw = dict(size=size, dropout_rate=rate, dropout_seed=11, dropout_site=3)
    out, lse = ops.attention_fwd(q, k, v, **kw)
    do = dev(rng.standard_normal((B, T, H, D)).astype(np.float32), torch.bfloat16)
    try:
        setter(from_ds)
        ref = [t.clone() for t in ops.attention_bwd(q, k, v, out, lse, do, **kw)]
        part = torch.full((B * ((T + 127) // 128), 3 * H * D), float("nan"), device="cuda")
        got = ops.attention_bwd(q, k, v, out, lse, do, bias_partial=part, **kw)
    finally:
        setter(-1)
    for a, b_ in zip(ref, got):
        assert torch.equal(a, b_)
    sums = ops.reduce_rows(part).double().cpu()
    want = torch.cat([g.double().sum((0, 1)).reshape(-1) for g in got]).cpu()
    scale = torch.cat([g.double().abs().sum((0, 1)).reshape(-1) for g in got]).max().item()
    assert (sums - want).abs().max().item() <= 2e-6 * scale + 1e-6


# ------------------------------------------------------------------------------------------------ image front end (SURVEY 8f rank 4)
def _it_nodes(H, P, Cin, F, G, E, PI, NB, norm):
    node = lambda t, **kw: dict(_target_=t, **kw)  # noqa: E731
    return dict(image_size=(H, H, Cin), patch_size=P, normalize=bool(norm), position_interval=PI, rng_collection="patch_encoding", embedding_dim=E,
                row_position_embedding=node("flax.linen.Embed", name="image_row_position_embedding", num_embeddings=PI, features=E),
                col_position_embedding=node("flax.linen.Embed", name="image_col_position_embedding", num_embeddings=PI, features=E),
                resnet=node("multi_modal_transformers.tokenizers.images.image_tokenizer.ResNetV2Block", num_blocks=NB,
                            input_conv=node("flax.linen.Conv", features=F, kernel_size=[12, 12], strides=[2, 2], padding="VALID", use_bias=True),
                            input_pool=dict(_partial_=True, _target_="flax.linen.max_pool", window_shape=[3, 3], strides=[1, 1], padding="VALID"),
                            resnet_norm=node("flax.linen.GroupNorm", num_groups=G, epsilon=1e-6),
                            resnet_activation=dict(_partial_=True, _target_="flax.linen.gelu"),
                            resnet_conv=node("flax.linen.Conv", features=F, kernel_size=[3, 3], strides=[1, 1], padding="SAME", use_bias=True),
                            output_dense=node("flax.linen.Dense", features=E)))


def _golden_tree(Z, prefix):
    tree = {}
    for k in Z.files:
        if k.startswith(prefix + "/"):
            node = tree
            parts = k[len(prefix) + 1:].split("/")
            for q in parts[:-1]:
                node = node.setdefault(q, {})
            node[parts[-1]] = Z[k]
    return tree


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["two_frames", "nine_patches_one_block", "group_size_one_raw_pixels"])
@pytest.mark.parametrize("pixels", ["f32", "u8"])
def test_image_tokenizer_golden(ops, name, pixels):
    """ImageTokenizer mirror (csrc/image_tokenizer.cu) against the tokens the reference's own ImageTokenizer produced under the
    shim (tests/golden/image_tokenizer.npz; image_tokenizer.py:216-309, train=False).  bf16 operands, fp32 accumulation through
    three chained contractions: |err| <= 3e-2 * max|want| (observed ~1e-2), mean |err| <= 5e-3 * max|want|."""
    from multi_modal_transformers_tokenmerge_b200.tokenizers.images import ImageTokenizer
    Z = np.load(os.path.join(GOLD, "image_tokenizer.npz"))
    B, N, H, P, Cin, F, G, E, PI, NB, norm = [int(v) for v in Z[f"{name}/meta"]]
    tok = ImageTokenizer(**_it_nodes(H, P, Cin, F, G, E, PI, NB, norm), out_dtype=torch.float32)
    img = torch.from_numpy(Z[f"{name}/image"]).cuda()
    if pixels == "f32":
        img = img.float()
    got = tok.apply({"params": _golden_tree(Z, f"{name}/params")}, img, train=False).cpu().numpy()
    want = Z[f"{name}/out"]
    assert got.shape == want.shape
    scale = np.abs(want).max()
    assert np.abs(got - want).max() <= 3e-2 * scale, (np.abs(got - want).max(), scale)
    assert np.abs(got - want).mean() <= 5e-3 * scale


@pytest.mark.gpu
def test_image_tokenizer_gato_geometry_vs_oracle(ops):
    """gato_resnet.yaml's literal geometry (280 x 280 x 3 uint8 pixels, 56-pixel patches, 64 features in 32 groups, 2 blocks,
    Dense 768, 128 position tokens), 3 batch rows x 2 images, against the oracle (pinned by the goldens above): bf16 output;
    one pass over the batch and one batch row per pass give the SAME bits (GroupNorm statistics are per batch row);
    training-mode position tokens (one row per image) select the embedding rows the host drew."""
    from multi_modal_transformers_tokenmerge_b200.tokenizers.images import ImageTokenizer, encode_patch_position
    rng = np.random.default_rng(11)
    H, P, F, G, E, PI, NB = 280, 56, 64, 32, 768, 128, 2
    nodes = _it_nodes(H, P, 3, F, G, E, PI, NB, True)
    tok = ImageTokenizer(**nodes)
    variables = tok.init(5, None)
    ef = variables["params"]["embedding_function"]
    for i in range(NB):
        ef[f"GroupNorm_{i}"]["scale"] = (1 + 0.1 * rng.standard_normal(F)).astype(np.float32)
        ef[f"GroupNorm_{i}"]["bias"] = (0.1 * rng.standard_normal(F)).astype(np.float32)
    img = rng.integers(0, 256, size=(3, 2, H, H, 3)).astype(np.uint8)
    got = tok.apply(variables, torch.from_numpy(img).cuda(), train=False)
    assert got.dtype == torch.bfloat16 and tuple(got.shape) == (3, 2, 25, E)
    p = O.image_tokenizer_params_from_flax(variables["params"], NB)
    want = O.image_tokenizer_fwd(p, img.astype(np.float32), patch_size=P, position_interval=PI, num_groups=G, normalize=True)
    scale = np.abs(want).max()
    err = np.abs(got.float().cpu().numpy() - want)
    assert err.max() <= 3e-2 * scale and err.mean() <= 5e-3 * scale, (err.max(), err.mean(), scale)
    tok1 = ImageTokenizer(**nodes, chunk_rows=1)
    got1 = tok1.apply(variables, torch.from_numpy(img).cuda(), train=False)
    assert torch.equal(got, got1)
    # training mode: tokens per (batch row, image); the embedding rows are the only thing that changes
    gt = tok.apply(variables, torch.from_numpy(img).cuda(), train=True, rngs={"patch_encoding": 9})
    row, col = encode_patch_position(H, P, PI, True, np.random.default_rng(9), images=6)
    r0, c0 = encode_patch_position(H, P, PI, False)
    re_, ce = variables["params"]["image_row_position_embedding"]["embedding"], variables["params"]["image_col_position_embedding"]["embedding"]
    delta = (re_[row] + ce[col] - re_[r0][None] - ce[c0][None]).reshape(3, 2, 25, E)
    d_got = gt.float().cpu().numpy() - got.float().cpu().numpy()
    assert np.abs(d_got - delta).max() <= 2 ** -7 * max(1.0, scale)      # two bf16 roundings


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,cols,shifts", [(1000, 64, 64, [-24, -23, -22, -1, 0, 1, 22, 23, 24]), (4096, 128, 128, [0, 5, -700]),
                                             (300, 256, 64, [-400, 400, 0, 1])])
def test_gemm_row_shifted_windows(ops, m, n, cols, shifts):
    """tome_gemm_args_t.a_row_shift: C[i] = sum_g A[i + shift_g] B_g with rows outside [0, m) reading as zero -- the 3 x 3
    convolution of the image front end as one GEMM (first case: its nine shifts on a 23-wide grid).  Against an fp32 torch sum
    over explicitly shifted, zero-filled copies of the same bf16 operands: |err| <= 2e-2 * sqrt(k) / 16."""
    rng = np.random.default_rng(m + n)
    G = len(shifts)
    A = torch.tensor(rng.standard_normal((m, cols)).astype(np.float32)).cuda().bfloat16()
    W = torch.tensor(rng.standard_normal((G * cols, n)).astype(np.float32)).cuda().bfloat16()
    bias = torch.tensor(rng.standard_normal(n).astype(np.float32)).cuda()
    out = ops.gemm(A, W, m=m, n=n, k=G * cols, b_major=1, bias=bias, out_dtype=torch.float32, a_row_shift=shifts)
    out16 = ops.gemm(A, W, m=m, n=n, k=G * cols, b_major=1, bias=bias, a_row_shift=shifts)
    Af, Wf = A.float().cpu(), W.float().cpu()
    ref = bias.cpu()[None].repeat(m, 1)
    for g_, sh in enumerate(shifts):
        sa = torch.zeros_like(Af)
        lo, hi = max(0, -sh), min(m, m - sh)
        if hi > lo:
            sa[lo:hi] = Af[lo + sh:hi + sh]
        ref = ref + sa @ Wf[g_ * cols:(g_ + 1) * cols]
    tol = 2e-2 * math.sqrt(G * cols) / 16
    assert (out.cpu() - ref).abs().max().item() <= tol
    assert (out16.float().cpu() - ref).abs().max().item() <= tol + 2 ** -7 * ref.abs().max().item()


@pytest.mark.gpu
def test_image_tokenizer_other_geometry_vs_oracle(ops):
    """A geometry none of the reference-made goldens has -- one input channel, a 4 x 4 / stride-1 input convolution, a 2 x 2 pool,
    three blocks of 64 features (the row-shifted 3 x 3 path) -- against the oracle: exercises the byte-wise pixel im2col (odd
    element offsets rule out the 32-bit path) and the general index arithmetic.  Same tolerance as the golden test."""
    from multi_modal_transformers_tokenmerge_b200.tokenizers.images import ImageTokenizer
    rng = np.random.default_rng(23)
    H, P, Cin, F, G, E, PI, NB = 36, 12, 1, 64, 8, 64, 32, 3
    nodes = _it_nodes(H, P, Cin, F, G, E, PI, NB, True)
    nodes["resnet"]["input_conv"].update(kernel_size=[4, 4], strides=[1, 1])
    nodes["resnet"]["input_pool"].update(window_shape=[2, 2])
    tok = ImageTokenizer(**nodes, out_dtype=torch.float32)
    variables = tok.init(3, None)
    img = rng.integers(0, 256, size=(2, 3, H, H, Cin)).astype(np.uint8)
    got = tok.apply(variables, torch.from_numpy(img).cuda(), train=False).cpu().numpy()
    p = O.image_tokenizer_params_from_flax(variables["params"], NB)
    want = O.image_tokenizer_fwd(p, img.astype(np.float32), patch_size=P, position_interval=PI, num_groups=G, conv_stride=1,
                                 pool_window=2, normalize=True)
    assert got.shape == want.shape == (2, 3, 9, E)
    scale = np.abs(want).max()
    err = np.abs(got - want)
    assert err.max() <= 3e-2 * scale and err.mean() <= 5e-3 * scale, (err.max(), err.mean(), scale)


@pytest.mark.gpu
def test_image_tokenizer_full_batch_properties(ops):
    """The image front end at a full batch (256 batch rows x 2 frames of 256 x 256 x 3, 16-pixel patches -> 131 072 tokens), where
    the oracle is too slow: size-independent properties.  GroupNorm statistics are per batch row, so (i) one pass and 32-row
    passes give identical bits, (ii) permuting the batch rows permutes the output rows bit for bit, (iii) a batch row computed
    alone equals its rows in the batch; and the first two batch rows agree with the oracle."""
    from multi_modal_transformers_tokenmerge_b200.tokenizers.images import ImageTokenizer
    rng = np.random.default_rng(31)
    H, P, F, G, E, PI, NB, B = 256, 16, 64, 32, 384, 128, 2, 256
    nodes = _it_nodes(H, P, 3, F, G, E, PI, NB, True)
    tok = ImageTokenizer(**nodes)
    variables = tok.init(9, None)
    img = torch.from_numpy(rng.integers(0, 256, size=(B, 2, H, H, 3)).astype(np.uint8)).cuda()
    full = tok.apply(variables, img, train=False)
    assert tuple(full.shape) == (B, 2, 256, E) and torch.isfinite(full.float()).all()
    chunked = ImageTokenizer(**nodes, chunk_rows=32).apply(variables, img, train=False)
    assert torch.equal(full, chunked)
    perm = torch.from_numpy(rng.permutation(B)).cuda()
    assert torch.equal(tok.apply(variables, img[perm].contiguous(), train=False), full[perm])
    assert torch.equal(tok.apply(variables, img[5:6].contiguous(), train=False), full[5:6])
    p = O.image_tokenizer_params_from_flax(variables["params"], NB)
    want = O.image_tokenizer_fwd(p, img[:2].cpu().numpy().astype(np.float32), patch_size=P, position_interval=PI, num_groups=G, normalize=True)
    err = np.abs(full[:2].float().cpu().numpy() - want)
    scale = np.abs(want).max()
    assert err.max() <= 3e-2 * scale and err.mean() <= 5e-3 * scale, (err.max(), err.mean(), scale)
