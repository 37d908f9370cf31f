"""Matching and merging INSIDE token sets (tome_token_sets_t) on the B200: K1 / K2 / K3 with a set table against the one-set
kernels on every set's slice and against the oracle's per-set merge_wavg (tests/set_merge_oracle.py), the set-merging stack
executor forward and backward against the oracle, block-causality end to end, and the StackedCompressedEncoder1DBlock
merge_fns path.  Needs a B200: `-m gpu`."""
import functools

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import tome_oracle as O  # noqa: E402
import set_merge_oracle as SO  # noqa: E402


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from multi_modal_transformers_tokenmerge_b200 import _lib, engine, ops
    _lib.lib()
    return ops, engine


def rel_err(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def table(lens):
    """(start, n, r) per set: odd starts and lengths, r = n / 2, r = 0 and one-token sets in the mix."""
    out, start = [], 0
    for i, n in enumerate(lens):
        r = (n // 2, 0, n // 4)[i % 3]
        out.append((start, n, r))
        start += n
    return out


# 16 sets (the most a table holds) with 300- and 257-token sets (150 / 129 even rows: more than one 128-row tcgen05 tile and
# several 64-row planes tiles), one-token sets, odd starts and lengths; and a short table
LONG16 = table([1, 5, 300, 7, 2, 3, 64, 129, 1, 2, 9, 11, 4, 33, 6, 257])
SHORT = table([37, 300, 1, 90])


@pytest.mark.parametrize("sets", [LONG16, SHORT], ids=["16sets", "4sets"])
@pytest.mark.parametrize("dim,dtype", [(64, torch.bfloat16), (64, torch.float32), (48, torch.bfloat16), (48, torch.float32)])
def test_k1_sets_equal_separate_calls_on_each_slice(pkg, sets, dim, dtype):
    """node_max / node_idx / the scores dump with a set table equal, bit for bit, tome_sim_argmax on each set's slice alone
    (dim 64: tcgen05 split-bf16 path; dim 48: fp32 planes).  A one-token set has no partner: -inf, index 0."""
    ops, _ = pkg
    B, T = 3, sum(n for _, n, _ in sets)
    m = torch.tensor(np.random.default_rng(dim).standard_normal((B, T, dim)), dtype=dtype).cuda()
    nm, ni, sc = ops.sim_argmax(m, sets=sets, dump_scores=True)
    off, soff = 0, 0
    for start, n, _ in sets:
        ta, tb = (n + 1) // 2, n // 2
        if n == 1:
            assert (nm[:, off] == -float("inf")).all() and (ni[:, off] == 0).all()
        else:
            nm1, ni1, sc1 = ops.sim_argmax(m[:, start:start + n].contiguous(), dump_scores=True)
            assert torch.equal(nm[:, off:off + ta].view(torch.int32), nm1.view(torch.int32)), (start, n)
            assert torch.equal(ni[:, off:off + ta], ni1), (start, n)
            assert torch.equal(sc[:, soff:soff + ta * tb].view(torch.int32), sc1.reshape(B, -1).view(torch.int32)), (start, n)
        off += ta
        soff += ta * tb
    assert off == nm.shape[1] and soff == sc.shape[1]


@pytest.mark.parametrize("sets", [LONG16, SHORT], ids=["16sets", "4sets"])
def test_k2_k3_sets_against_the_oracle(pkg, sets):
    """Plans bit-exact against the oracle's per-set ranking of the GPU's own node_max / node_idx; fp32 merged rows, sizes,
    group ids and positions bit-exact against the oracle's per-set merge_wavg; no token lands outside its set's output rows;
    r = 0 sets are copied unchanged; merge backward through the global row map."""
    ops, _ = pkg
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    rng = np.random.default_rng(7)
    B, T, C = 3, sum(n for _, n, _ in sets), 64
    m = torch.tensor(rng.standard_normal((B, T, 64)), dtype=torch.float32).cuda()
    x = rng.standard_normal((B, T, C)).astype(np.float32)
    size = rng.uniform(0.5, 4.0, (B, T)).astype(np.float32)
    gid = rng.integers(0, 5, (B, T)).astype(np.uint8)
    pos = rng.integers(0, 1000, (B, T)).astype(np.int32)
    nm, ni, _ = ops.sim_argmax(m, sets=sets)
    plan = ops.select_topr(nm, ni, T, sets=sets)
    plans = SO.set_plans(None, sets, (nm.cpu().numpy(), ni.cpu().numpy()))
    want_edge = np.concatenate([np.broadcast_to(np.arange((n + 1) // 2, dtype=np.int32), (B, (n + 1) // 2)) if p is None else p.edge_idx
                                for p, (_, n, _) in zip(plans, sets)], axis=1)
    want_dst = np.concatenate([p.dst_idx for p in plans if p is not None], axis=1)
    np.testing.assert_array_equal(plan.edge_idx.cpu().numpy(), want_edge)
    np.testing.assert_array_equal(plan.dst_idx.cpu().numpy(), want_dst)
    rm = SO.set_row_map(plans, sets, B)
    np.testing.assert_array_equal(plan.row_map.cpu().numpy(), rm)
    row0 = 0
    for start, n, r in sets:   # every token stays inside its set's block of output rows
        blk = rm[:, start:start + n]
        assert blk.min() >= row0 and blk.max() < row0 + n - r, (start, n, r)
        row0 += n - r
    xo, so, go, po = ops.merge_fwd(plan, torch.tensor(x).cuda(), torch.tensor(size).cuda(), L.TOME_MERGE_WAVG,
                                   torch.tensor(gid).cuda(), torch.tensor(pos).cuda())
    wx, ws = SO.set_merge_wavg(plans, sets, x, size[..., None])
    wg, wp = SO.kept_token_groups(plans, sets, gid, pos, rm)
    np.testing.assert_array_equal(xo.cpu().numpy(), wx)
    np.testing.assert_array_equal(so.cpu().numpy(), ws[..., 0])
    np.testing.assert_array_equal(go.cpu().numpy(), wg)
    np.testing.assert_array_equal(po.cpu().numpy(), wp)
    row0 = 0
    for start, n, r in sets:
        if r == 0:
            np.testing.assert_array_equal(xo[:, row0:row0 + n].cpu().numpy(), x[:, start:start + n])
            np.testing.assert_array_equal(so[:, row0:row0 + n].cpu().numpy(), size[:, start:start + n])
        row0 += n - r
    dy = torch.tensor(rng.standard_normal((B, T - plan.r, C)), dtype=torch.float32).cuda()
    dx = ops.merge_bwd(plan, dy, torch.tensor(size).cuda(), so, L.TOME_MERGE_WAVG).cpu().numpy()
    w = size / np.take_along_axis(so.cpu().numpy(), rm, axis=1)
    want = np.take_along_axis(dy.cpu().numpy(), rm[..., None].astype(np.int64), axis=1) * w[..., None]
    np.testing.assert_array_equal(dx, want.astype(np.float32))


def test_tokenset_soft_matching_is_per_set_merge_wavg(pkg):
    """The operator API: merge_wavg(tokenset_soft_matching(...)) equals the oracle's per-set merge_wavg on its own scores."""
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_compression import merge_wavg, tokenset_soft_matching
    rng = np.random.default_rng(3)
    sets = SHORT
    T = sum(n for _, n, _ in sets)
    m = rng.standard_normal((2, T, 64)).astype(np.float32)
    x = rng.standard_normal((2, T, 32)).astype(np.float32)
    merge = tokenset_soft_matching(torch.tensor(m).cuda(), [(s, n) for s, n, _ in sets], [r for _, _, r in sets])
    y, size = merge_wavg(merge, torch.tensor(x).cuda())
    plans = SO.set_plans(None, sets, (merge.plan.node_max.cpu().numpy(), merge.plan.node_idx.cpu().numpy()))
    wx, ws = SO.set_merge_wavg(plans, sets, x)
    np.testing.assert_array_equal(y.cpu().numpy(), wx)
    np.testing.assert_array_equal(size.cpu().numpy(), ws)


# ------------------------------------------------------------------------------------------------ the stack
def _build(pkg, B, W, P, C, H, Dff, Lyr, c_img, ln_axis=2, n_ro=2, n_tdp=4, seed=0):
    ops, engine = pkg
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence
    rng = np.random.default_rng(seed)
    seq = f"[TaskDescriptionPrefix{{{n_tdp}}}] [Image{{{P}}};Readout{{{n_ro}}}]*{W}"
    comp = f"[TaskDescriptionPrefix{{0}}] [Image{{{c_img}}};Readout{{0}}]*{W}"
    gid, pos, allow, ro = O.sequence_groups(seq)
    sets = tuple(TokenSequence(seq, comp).prune_sets())
    T = gid.shape[0]
    layers = [O.init_block_params(rng, C, H, 64, Dff) for _ in range(Lyr)]
    for d in layers:
        for k_ in ("ln1_scale", "ln2_scale"):
            d[k_] = (d[k_] + 0.1 * rng.standard_normal(C)).astype(np.float32)
        for k_ in ("ln1_bias", "ln2_bias"):
            d[k_] = (0.1 * rng.standard_normal(C)).astype(np.float32)
    pe = (rng.standard_normal((1, T, C)) * 0.02).astype(np.float32)
    x = rng.standard_normal((B, T, C)).astype(np.float32)
    y = rng.standard_normal((B, len(ro), C)).astype(np.float32)
    cfg = engine.StackConfig(batch=B, tokens=T, channels=C, heads=H, head_dim=64, mlp_dim=Dff, layers=Lyr, r=0, ln_axis=ln_axis,
                             num_groups=allow.shape[0], n_readout=len(ro), prune_sets=sets, set_merge=True)
    eng = engine.ToMeStackEngine(cfg, gid=gid, pos=pos, allow=allow, readout_idx=ro)
    eng.load_params(pe[0], layers)
    return eng, cfg, x, y, (gid, pos, allow, ro)


def _oracle_params(eng, cfg):
    v = eng.param_views(eng.params_bf16.float().cpu())
    vf = eng.param_views(eng.params.cpu())
    params, hd = [], cfg.heads * cfg.head_dim
    for l in range(cfg.layers):
        s_, f_ = v["layers"][l], vf["layers"][l]
        d = dict(ln1_scale=f_["ln1_scale"], ln1_bias=f_["ln1_bias"], ln2_scale=f_["ln2_scale"], ln2_bias=f_["ln2_bias"],
                 wq=s_["wqkv"][:, :hd], wk=s_["wqkv"][:, hd:2 * hd], wv=s_["wqkv"][:, 2 * hd:], bq=f_["bqkv"][:hd],
                 bk=f_["bqkv"][hd:2 * hd], bv=f_["bqkv"][2 * hd:], wo=s_["wo"], bo=f_["bo"], w1=s_["w1"], b1=f_["b1"],
                 w2=s_["w2"], b2=f_["b2"])
        params.append(O.BlockParams(**{k_: t.clone().contiguous().requires_grad_(True) for k_, t in d.items()}))
    return params, vf["pos_embedding"].clone()[None].requires_grad_(True)


def _stack_vs_oracle(pkg, shape, Lyr, c_img, tol_fwd, tol_grad):
    eng, cfg, x, y, (gid, pos, allow, ro) = _build(pkg, Lyr=Lyr, c_img=c_img, **shape)
    eng.zero_grad()
    eng.forward(torch.tensor(x).cuda(), torch.tensor(y).cuda())
    eng.backward()
    torch.cuda.synchronize()
    pls = [eng.layer_plan(l) for l in range(Lyr)]
    gates = [eng.layer_relu_gate(l).cpu().numpy() for l in range(Lyr)]
    params, pet = _oracle_params(eng, cfg)
    tr = []
    xf, size, origin = SO.set_merge_stack(params, pet, torch.tensor(x), gid, pos, allow, num_heads=cfg.heads, prune_sets=cfg.prune_sets,
                                          ln_axis="feature", prop_attn=True, act_dtype=torch.bfloat16, relu_gate=gates, trace=tr,
                                          node_override=[(p[0].cpu().numpy(), p[1].cpu().numpy()) for p in pls])
    loss, out = O.readout_loss(xf, origin, ro, torch.tensor(y))
    loss.backward()
    B = x.shape[0]
    for l, (plans, _) in enumerate(tr):   # merge indices bit-exact, set by set
        sets = cfg.layer_sets(l)
        want = np.concatenate([np.broadcast_to(np.arange((n + 1) // 2, dtype=np.int32), (B, (n + 1) // 2)) if p is None else p.edge_idx
                               for p, (_, n, _) in zip(plans, sets)], axis=1)
        np.testing.assert_array_equal(pls[l][2].cpu().numpy(), want)
        np.testing.assert_array_equal(pls[l][3].cpu().numpy(), np.concatenate([p.dst_idx for p in plans if p is not None], axis=1))
    np.testing.assert_array_equal(eng.final_size().cpu().numpy(), size.detach().numpy()[..., 0])
    e_fwd = dict(final_x=rel_err(eng.final_x().float().cpu(), xf.detach()), readout=rel_err(eng.readout.cpu(), out.detach()),
                 loss=abs(eng.loss[0].item() - loss.item()) / abs(loss.item()))
    g = eng.param_views(eng.grads.cpu())
    e_grad = {"pos_embedding": rel_err(g["pos_embedding"], pet.grad[0])}
    for l in range(Lyr):
        p, gl = params[l], g["layers"][l]
        ref = dict(ln1_scale=p.ln1_scale.grad, ln1_bias=p.ln1_bias.grad, ln2_scale=p.ln2_scale.grad, ln2_bias=p.ln2_bias.grad,
                   wqkv=torch.cat([p.wq.grad, p.wk.grad, p.wv.grad], 1), bqkv=torch.cat([p.bq.grad, p.bk.grad, p.bv.grad]),
                   wo=p.wo.grad, bo=p.bo.grad, w1=p.w1.grad, b1=p.b1.grad, w2=p.w2.grad, b2=p.b2.grad)
        for name, want in ref.items():
            e_grad[f"layer {l} grad {name}"] = rel_err(gl[name], want)
    worst = max(e_grad, key=e_grad.get)
    print(f"\n[set-merge stack parity] {shape} L={Lyr}: fwd {e_fwd}; worst grad {worst} = {e_grad[worst]:.4f}")
    for k_, v in e_fwd.items():
        assert v <= tol_fwd, f"{k_}: rel err {v}"
    for k_, v in e_grad.items():
        assert v <= tol_grad, f"{k_}: rel err {v}"


@pytest.mark.parametrize("Lyr,c_img", [(2, 4), (3, 3)])
def test_set_merge_stack_forward_backward_vs_oracle(pkg, Lyr, c_img):
    """A set-merging stack (text and readout sets keep every token, each frame's image set merges c_img per layer), prop_attn,
    block-causal mask, feature-axis LayerNorm: merge indices and sizes bit-exact, forward within 1e-2 and every parameter
    gradient within 2e-2 of the oracle, which follows the GPU's matches and ReLU gates."""
    _stack_vs_oracle(pkg, dict(B=2, W=2, P=24, C=128, H=2, Dff=256), Lyr, c_img, 1e-2, 2e-2)


def test_set_merge_stack_octo_small_widths_vs_oracle(pkg):
    """octo-small widths (C = 384, 6 heads, Dff = 1536) over 12 layers, 536 tokens, each image set merging 8 per layer (the
    16 tokens per layer of the global r = 16 configuration): forward within 2e-2, every gradient within 4e-2."""
    _stack_vs_oracle(pkg, dict(B=2, W=2, P=256, C=384, H=6, Dff=1536, n_ro=4, n_tdp=16), 12, 8, 2e-2, 4e-2)


def test_set_merge_keeps_block_causality_end_to_end(pkg):
    """With feature-axis LayerNorm (token-axis LayerNorm mixes all tokens by design) frame 1's readout rows do not depend on
    frame 2: changing every frame-2 input leaves them bit-identical, and so their part of the loss."""
    eng, cfg, x, y, (gid, pos, allow, ro) = _build(pkg, B=2, W=2, P=64, C=128, H=2, Dff=256, Lyr=4, c_img=8, n_ro=4, n_tdp=8)
    n_tdp, P, n_ro = 8, 64, 4
    frame2 = slice(n_tdp + P + n_ro, n_tdp + 2 * (P + n_ro))
    x2 = x.copy()
    x2[:, frame2] = np.random.default_rng(11).standard_normal(x2[:, frame2].shape).astype(np.float32)
    yd = torch.tensor(y).cuda()
    outs = []
    for xi in (x, x2):
        eng.forward(torch.tensor(xi).cuda(), yd)
        torch.cuda.synchronize()
        outs.append((eng.readout.clone(), eng.loss.clone()))
    (r1, l1), (r2, l2) = outs
    assert torch.equal(r1[:, :n_ro].view(torch.int32), r2[:, :n_ro].view(torch.int32)), "frame-1 readouts changed"
    assert not torch.equal(r1[:, n_ro:], r2[:, n_ro:]), "frame-2 readouts should see frame-2 inputs"
    part = lambda r: ((r[:, :n_ro] - yd[:, :n_ro]) ** 2).sum(dim=(1, 2))  # noqa: E731
    assert torch.equal(part(r1), part(r2)) and l1[0].item() != l2[0].item()


def test_compressed_stack_module_with_merge_fns_matches_the_engine(pkg):
    """StackedCompressedEncoder1DBlock(merge_fns=...) as the reference's caller would build it (partials of
    tokenset_soft_matching following the compression grammar) or as (tokenset_idx, tokenset_r) pairs: the same bits as the
    set-merging engine on the same parameters."""
    ops, engine = pkg
    from multi_modal_transformers_tokenmerge_b200 import model_configs as MC
    from multi_modal_transformers_tokenmerge_b200.attention_blocks import compressed_attention as CA
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_compression import tokenset_soft_matching
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence
    C, H, Dff, L_ = 128, 2, 256, 3
    cfg = MC.load("attention_blocks/tome_decoder_octo_small")
    e = dict(cfg["encoder_1d_block"], _target_="multi_modal_transformers.attention_blocks.compressed_attention.CompressedEncoder1DBlock")
    e["layer_norm"] = dict(e["layer_norm"], reduction_axes=[-1])
    e["self_attention"] = dict(e["self_attention"], num_heads=H, qkv_features=C)
    e["mlp_block"] = dict(e["mlp_block"], dense=dict(e["mlp_block"]["dense"], features=Dff), dense_out=dict(e["mlp_block"]["dense_out"], features=C))
    ts = TokenSequence("[TaskDescriptionPrefix{8}] [Image{40};Readout{2}]*2", "[TaskDescriptionPrefix{0}] [Image{6};Readout{0}]*2")
    fns, pairs = [], []
    for l in range(L_):
        sets = SO.stack_sets_at(ts.prune_sets(), l)
        idx, rs = [(s_, n) for s_, n, _ in sets], [r for _, _, r in sets]
        fns.append(functools.partial(tokenset_soft_matching, tokenset_idx=idx, tokenset_r=rs))
        pairs.append((idx, rs))
    with pytest.raises(ValueError, match="compression grammar"):
        CA.StackedCompressedEncoder1DBlock(L_, e, merge_fns=[fns[0]] * L_)
    B, T = 2, 92
    x = torch.tensor(np.random.default_rng(5).standard_normal((B, T, C)), dtype=torch.float32).cuda()
    masks = [ts.layer_group_ids(0)]
    ys = []
    for m_fns in (fns, pairs):
        stack = CA.StackedCompressedEncoder1DBlock(L_, e, merge_fns=m_fns)
        assert stack.set_merge and stack.prune_sets == tuple(ts.prune_sets())
        variables = stack.init(4, torch.zeros(B, T, C))
        ys.append(stack.apply(variables, x, masks=masks, allow=ts.allow_table(), train=False))
    assert tuple(ys[0].shape) == (B, T - 3 * 12, C) and torch.equal(ys[0], ys[1])
    gid, pos = ts.layer_group_ids(0)
    scfg = engine.StackConfig(batch=B, tokens=T, channels=C, heads=H, head_dim=C // H, mlp_dim=Dff, layers=L_, r=0, ln_axis=2,
                              ln_eps=stack._engine.cfg.ln_eps, prop_attn=False, num_groups=ts.allow_table().shape[0], prune_sets=tuple(ts.prune_sets()), set_merge=True)
    eng = engine.ToMeStackEngine(scfg, gid=gid, pos=pos, allow=ts.allow_table(), training=False)
    eng.params.copy_(stack._engine.params)
    eng.sync_bf16()
    eng.forward(x.contiguous())
    assert torch.equal(eng.final_x(), ys[1])
