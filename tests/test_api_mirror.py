"""The reference-facing Python API (same names / signatures / error behaviour as multi_modal_transformers/
tokenizers/token_compression.py and attention_blocks/{attention,tome_attention}.py).

CPU part: configuration, parameter-tree shape, mask conversion, argument errors (no kernel is launched).
GPU part (-m gpu): the operator API against the reference-generated goldens and the oracle; the per-block modules
chained in Python against the native stack executor (same kernels -> identical bits) and against the oracle."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from multi_modal_transformers_tokenmerge_b200 import model_configs as MC  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.attention_blocks import _functional as F  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.attention_blocks import attention as A  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.attention_blocks import tome_attention as TA  # noqa: E402
from multi_modal_transformers_tokenmerge_b200 import action_heads as AH  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers import token_compression as TCm  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence  # noqa: E402
from oracle import tome_oracle as O  # noqa: E402  (checker only)

GOLD = os.path.join(os.path.dirname(__file__), "golden")
SEQ = "[TaskDescriptionPrefix{4}] [Image{24};Readout{2}]*2"


def small_cfg(C=128, H=2, Dff=256, blocks=2, r=4, hidden_drop=0.0):
    cfg = MC.load("attention_blocks/tome_decoder_octo_small")
    cfg["num_blocks"], cfg["tome_r"] = blocks, r
    e = cfg["encoder_1d_block"]
    e["self_attention"].update(num_heads=H, qkv_features=C)
    e["mlp_block"]["dense"]["features"] = Dff
    e["mlp_block"]["dense_out"]["features"] = C
    e["dropout"]["rate"] = hidden_drop
    e["mlp_block"]["norm"]["rate"] = hidden_drop
    return cfg


# ------------------------------------------------------------------------------------------------ CPU
def test_yaml_schema_of_the_reference_is_accepted():
    cfg = MC.load("attention_blocks/tome_decoder_octo_base")
    assert set(cfg["encoder_1d_block"]) == {"_target_", "layer_norm", "dropout", "self_attention", "mlp_block"}
    st = MC.build_stack(cfg)
    assert isinstance(st, TA.StackedEncoder1DBlock) and st.r == 32 and st.num_blocks == 12
    ln, dr, at, mlp = st._block()._specs()
    assert (ln.axis, ln.epsilon, dr.rate, at.num_heads, at.qkv_features) == (1, 1e-6, 0.1, 12, 768)
    d, act, mdrop, do = mlp._specs()
    assert (d.features, act, mdrop.rate, do.features) == (3072, "relu", 0.1, 768)
    # the literal reference node kinds (SelfAttention target, vanilla block) resolve to the vanilla stack
    lit = {"num_blocks": 1, "encoder_1d_block": dict(cfg["encoder_1d_block"], _target_="multi_modal_transformers.attention_blocks.attention.Encoder1DBlock")}
    lit["encoder_1d_block"]["self_attention"] = dict(cfg["encoder_1d_block"]["self_attention"], _target_="flax.linen.SelfAttention")
    assert type(MC.build_stack(lit)) is A.StackedEncoder1DBlock
    with pytest.raises(ValueError):
        A.instantiate({"_target_": "flax.linen.Conv"})


def test_param_tree_has_flax_names_and_scan_axis():
    cfg = small_cfg(C=128, H=2, Dff=256, blocks=3)
    st = MC.build_stack(cfg)
    x = torch.zeros(2, 56, 128)
    v = st.init(0, x)
    p = v["params"]
    assert p["posembed_input"]["pos_embedding"].shape == (1, 56, 128)          # attention.py:97-100
    blk = p["ScanEncoder1DBlock_0"]                                             # nn.scan, params stacked on axis 0
    a = blk["ToMeMultiHeadDotProductAttention_0"]
    assert a["query"]["kernel"].shape == (3, 128, 2, 64) and a["query"]["bias"].shape == (3, 2, 64)
    assert a["out"]["kernel"].shape == (3, 2, 64, 128) and a["out"]["bias"].shape == (3, 128)
    assert blk["LayerNorm_0"]["scale"].shape == (3, 128) and blk["LayerNorm_1"]["bias"].shape == (3, 128)
    assert blk["MLPBlock_0"]["Dense_0"]["kernel"].shape == (3, 128, 256)
    assert blk["MLPBlock_0"]["Dense_1"]["kernel"].shape == (3, 256, 128)
    layers = A.flax_tree_to_layers(blk, "ToMeMultiHeadDotProductAttention_0", 3)
    assert layers[1]["wq"].shape == (128, 128) and layers[2]["wo"].shape == (128, 128) and layers[0]["w1"].shape == (128, 256)


def test_dense_mask_to_group_table_roundtrip():
    ts = TokenSequence("[TaskDescriptionPrefix{16}] [Image{25};Readout{4}]*2")     # octo_base.yaml:10
    dense = ts.generate_attention_mask(repeats=3)                                 # [H, T, T] as octo.py:66-68
    gm = F.group_mask_from_dense(np.broadcast_to(dense, (2,) + dense.shape), device="cpu")
    gid = gm.gid.numpy()
    allow = gm.allow.numpy()
    assert allow.shape[0] <= 5
    np.testing.assert_array_equal(allow[gid][:, gid].astype(bool), dense[0])
    bad = np.broadcast_to(dense, (2,) + dense.shape).copy()
    bad[1, 0, 0, -1] ^= True
    with pytest.raises(ValueError):
        F.group_mask_from_dense(bad, device="cpu")


def test_argument_errors_follow_the_reference():
    att = TA.ToMeMultiHeadDotProductAttention(num_heads=2, qkv_features=128)
    x = torch.zeros(1, 8, 128)
    v = att.init(0, x)
    with pytest.raises(ValueError):                      # tome_attention.py:116-121
        att.apply(v, x, None, x)
    with pytest.raises(ValueError):                      # :94-103
        att.apply(v, x, x, inputs_kv=x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        att.apply(v, x)
    with pytest.raises(ValueError):                      # :139-142
        TA.ToMeMultiHeadDotProductAttention(num_heads=3, qkv_features=128).init(0, x)
    blk = MC.build_stack(small_cfg())._block()
    with pytest.raises(ValueError):                      # merge_param('train', None, None)  attention.py:54
        blk.apply(blk.init(0, x), x.cuda() if torch.cuda.is_available() else x)
    with pytest.raises(ValueError):
        TCm.bipartite_soft_matching(torch.zeros(4, 8), 2)
    m = TCm._Merge(None, 8)
    with pytest.raises(ValueError):
        m(torch.zeros(1, 8, 4), mode="mean")


# ------------------------------------------------------------------------------------------------ GPU
gpu = pytest.mark.gpu


def _dev(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return t if dtype is None else t.to(dtype)


@gpu
def test_operator_api_against_reference_goldens():
    """bipartite_soft_matching / merge / merge_wavg called exactly as the reference is (token_compression.py:54-129) on
    the golden inputs: outputs equal the reference's own outputs bit for bit wherever the indices agree."""
    TC = np.load(os.path.join(GOLD, "token_compression.npz"))
    n_exact = 0
    for name in [str(n) for n in TC["names"]]:
        B, T, Dm, C, r, cls, dis = [int(v) for v in TC[f"{name}/cfg"]]
        metric, x = _dev(TC[f"{name}/metric"]), _dev(TC[f"{name}/x"])
        merge = TCm.bipartite_soft_matching(metric, r, class_token=bool(cls), distill_token=bool(dis))
        x1, s1 = TCm.merge_wavg(merge, x)
        assert s1.shape == (B, T - merge.r, 1) and x1.shape == (B, T - merge.r, C)
        if merge.r == 0:
            np.testing.assert_array_equal(x1.cpu().numpy(), TC[f"{name}/x"])
            continue
        same = np.array_equal(merge.plan.src_idx.cpu().numpy(), TC[f"{name}/src_idx"][..., 0] if TC[f"{name}/src_idx"].ndim == 3 else TC[f"{name}/src_idx"]) \
            and np.array_equal(merge.plan.dst_idx.cpu().numpy(), TC[f"{name}/dst_idx"][..., 0] if TC[f"{name}/dst_idx"].ndim == 3 else TC[f"{name}/dst_idx"])
        if same:
            n_exact += 1
            np.testing.assert_array_equal(x1.cpu().numpy(), TC[f"{name}/x1"])
            np.testing.assert_array_equal(s1.cpu().numpy(), TC[f"{name}/s1"])
            np.testing.assert_array_equal(merge(x, mode="sum").cpu().numpy(), TC[f"{name}/xsum"])
        # merge(size) alone, as merge_wavg's second call does (:126)
        ones = torch.ones(B, T, 1, device="cuda")
        np.testing.assert_array_equal(merge(ones).cpu().numpy(), s1.cpu().numpy())
        # unmerge(merge_wavg(x)) puts every merged row back at all of its members' positions
        um = merge.unmerge(x1)
        assert um.shape == (B, T, C)
    assert n_exact >= 3


@gpu
@pytest.mark.parametrize("r", [0, 4])
def test_blocks_chained_in_python_equal_the_native_stack_and_the_oracle(r):
    cfg = small_cfg(C=128, H=2, Dff=256, blocks=2, r=r)
    ts = TokenSequence(SEQ)
    T = ts.num_tokens
    B, C = 2, 128
    rng = np.random.default_rng(0)
    x = _dev(rng.standard_normal((B, T, C)).astype(np.float32))
    stack = MC.build_stack(cfg)
    variables = stack.init(1, x)
    gm = F.GroupMask.from_token_sequence(ts)
    # (a) the native executor through the reference-shaped call
    y_stack = stack.apply(variables, x, train=False, mask=gm)
    assert y_stack.shape == (B, T - 2 * r, C)
    # (b) the caller's own loop over ToMeEncoder1DBlock, parameters unstacked from the scan axis
    p = variables["params"]
    h = A.AddPositionEmbedding().apply({"params": p["posembed_input"]}, x)
    state = F.ToMeState()
    blk = stack._block()
    for l in range(2):
        pl = {"params": _index_tree(p["ScanEncoder1DBlock_0"], l)}
        h, none = blk.apply(pl, h, mask=gm, train=False, tome_state=state, site=3 * l)
        assert none is None
    torch.testing.assert_close(h, y_stack, rtol=0, atol=0)
    if r:
        torch.testing.assert_close(state.size, stack.last_size, rtol=0, atol=0)
        assert float(state.size.sum(dim=1)[0]) == T
    # (c) the same with the dense boolean mask of octo.py:66-68 instead of the group table
    dense = torch.as_tensor(ts.generate_attention_mask(repeats=2))[None].expand(B, -1, -1, -1)
    y_dense = stack.apply(variables, x, train=False, mask=dense)
    torch.testing.assert_close(y_dense, y_stack, rtol=0, atol=0)
    # (d) the oracle (fp32, bf16-rounded weights), tolerance 3e-2 relative L2 as in test_gpu_stack.py
    gid, pos, allow, _ = O.sequence_groups(SEQ)
    layers = A.flax_tree_to_layers(p["ScanEncoder1DBlock_0"], blk._attn_name, 2)
    rb = lambda a: torch.as_tensor(np.asarray(a)).bfloat16().float()  # noqa: E731
    params = []
    for lay in layers:
        d = {k: (rb(v) if k.startswith("w") else torch.as_tensor(np.asarray(v))) for k, v in lay.items()}
        params.append(O.BlockParams(**d))
    node_override = None
    if r:
        eng = stack._engine
        node_override = [tuple(t.cpu().numpy() for t in eng.layer_plan(l)[:2]) for l in range(2)]
    xf, size, origin = O.tome_stack(params, torch.as_tensor(p["posembed_input"]["pos_embedding"]), x.cpu(), gid, pos, allow,
                                    num_heads=2, r=r, node_override=node_override)
    err = (y_stack.float().cpu() - xf).norm() / xf.norm()
    assert err <= 3e-2, err


@gpu
def test_literal_reference_yaml_values_run_through_the_vanilla_modules():
    """The reference's own hyper-parameters (vanilla_decoder.yaml: one Encoder1DBlock, flax.linen.SelfAttention with 3 heads over
    768 features = head_dim 256, MLP 768 -> 768, LayerNorm over tokens; octo_base.yaml:10: 74 tokens) through the
    reference-shaped modules: the vanilla StackedEncoder1DBlock, eval mode, dense boolean mask as octo.py:66-68 builds it,
    against the oracle.  head_dim 256 is served by the generic attention path."""
    cfg = MC.load("attention_blocks/tome_decoder_octo_base")
    e = dict(cfg["encoder_1d_block"], _target_="multi_modal_transformers.attention_blocks.attention.Encoder1DBlock")
    e["self_attention"] = dict(e["self_attention"], _target_="flax.linen.SelfAttention", num_heads=3, qkv_features=768)
    e["mlp_block"] = dict(e["mlp_block"], dense=dict(e["mlp_block"]["dense"], features=768),
                          dense_out=dict(e["mlp_block"]["dense_out"], features=768))
    stack = MC.build_stack({"num_blocks": 1, "encoder_1d_block": e})
    assert type(stack) is A.StackedEncoder1DBlock
    seq = "[TaskDescriptionPrefix{16}] [Image{25};Readout{4}]*2"
    ts = TokenSequence(seq)
    B, T, C = 2, ts.num_tokens, 768
    assert T == 74
    rng = np.random.default_rng(5)
    x = _dev(rng.standard_normal((B, T, C)).astype(np.float32))
    variables = stack.init(3, x)
    dense = torch.as_tensor(ts.generate_attention_mask(repeats=3))[None].expand(B, -1, -1, -1)   # [B, H, T, T] booleans
    y = stack.apply(variables, x, train=False, mask=dense)
    assert y.shape == (B, T, C)
    p = variables["params"]
    gid, pos, allow, _ = O.sequence_groups(seq)
    layers = A.flax_tree_to_layers(p["ScanEncoder1DBlock_0"], stack._block()._attn_name, 1)
    rb = lambda a: torch.as_tensor(np.asarray(a)).bfloat16().float()  # noqa: E731
    params = [O.BlockParams(**{k: (rb(v) if k.startswith("w") else torch.as_tensor(np.asarray(v))) for k, v in layers[0].items()})]
    xf, _, _ = O.tome_stack(params, torch.as_tensor(p["posembed_input"]["pos_embedding"]), x.cpu(), gid, pos, allow, num_heads=3, r=0)
    err = (y.float().cpu() - xf).norm() / xf.norm()
    assert err <= 3e-2, err


def _index_tree(tree, l):
    if isinstance(tree, dict):
        return {k: _index_tree(v, l) for k, v in tree.items()}
    return tree[l]


@gpu
def test_mha_module_and_hidden_dropout_site_parity():
    """ToMeMultiHeadDotProductAttention alone (projections + masked attention + out) against the oracle's attention, and
    train=True hidden dropout: the Python-chained blocks and the native stack draw the same Philox masks."""
    ts = TokenSequence(SEQ)
    T, B, C, H = ts.num_tokens, 2, 128, 2
    rng = np.random.default_rng(3)
    x = _dev(rng.standard_normal((B, T, C)).astype(np.float32)).bfloat16()
    att = TA.ToMeMultiHeadDotProductAttention(num_heads=H, qkv_features=C, kernel_init="he_normal", bias_init="normal")
    v = att.init(5, x)
    gm = F.GroupMask.from_token_sequence(ts)
    size = _dev(rng.integers(1, 4, size=(B, T)).astype(np.float32))
    out, metric = att.apply(v, x, mask=gm, size=size, return_metric=True)
    p = v["params"]
    rb = lambda a: torch.as_tensor(a).bfloat16().float()  # noqa: E731
    xf = x.float().cpu()
    q, k, vv = [(xf @ rb(p[n]["kernel"]).reshape(C, C) + torch.as_tensor(p[n]["bias"]).reshape(-1)).bfloat16().float().reshape(B, T, H, 64)
                for n in ("query", "key", "value")]
    gid, pos, allow, _ = O.sequence_groups(SEQ)
    g2, p2 = np.broadcast_to(gid, (B, T)), np.broadcast_to(pos, (B, T))
    mask = torch.as_tensor(O.dense_mask(g2, p2, g2, p2, allow))[:, None]
    ref = O.attention(q, k, vv, mask=mask, bias=torch.log(size.cpu())[:, None, None, :]).reshape(B, T, C)
    ref = ref.bfloat16().float() @ rb(p["out"]["kernel"]).reshape(C, C) + torch.as_tensor(p["out"]["bias"])
    assert ((out.float().cpu() - ref).norm() / ref.norm()) <= 2e-2
    assert metric.shape == (B, T, 64)
    # hidden dropout: same seed + site numbering -> identical bits on both routes
    cfg = small_cfg(C=128, H=2, Dff=256, blocks=2, r=4, hidden_drop=0.1)
    stack = MC.build_stack(cfg)
    xs = x.float()
    variables = stack.init(1, xs)
    y_stack = stack.apply(variables, xs, train=True, mask=gm, dropout_rng=77)
    pz = variables["params"]
    h = A.AddPositionEmbedding().apply({"params": pz["posembed_input"]}, xs)
    state, blk = F.ToMeState(), stack._block()
    for l in range(2):
        h, _ = blk.apply({"params": _index_tree(pz["ScanEncoder1DBlock_0"], l)}, h, mask=gm, train=True, tome_state=state,
                         site=3 * l, dropout_rng=77)
    torch.testing.assert_close(h, y_stack, rtol=0, atol=0)
    y_eval = stack.apply(variables, xs, train=False, mask=gm)
    assert not torch.equal(y_eval, y_stack)


@gpu
def test_action_head_modules_against_reference_goldens():
    """ContinuousActionHead / CategoricalActionHead constructed and called as the reference's modules are
    (continuous.py:12-25, categorical.py:24-40; the Dense node is the one diffusion.yaml / vanilla_decoder.yaml use), on
    the inputs and parameters of goldens made by executing those modules: same shapes, same numbers (fp32, 1e-5), and
    the losses of octo.py:157-190 on top."""
    g = np.load(os.path.join(GOLD, "action_heads.npz"))
    dense = lambda f: {"_target_": "flax.linen.Dense", "features": f, "use_bias": True,  # noqa: E731
                       "kernel_init": {"_target_": "flax.linen.initializers.he_normal"},
                       "bias_init": {"_target_": "flax.linen.initializers.normal"}}
    for name in g["continuous"]:
        ro, act = _dev(g[f"{name}/readouts"]), _dev(g[f"{name}/actions"])
        A_ = g[f"{name}/kernel"].shape[1]
        head = AH.ContinuousActionHead(max_action=float(g[f"{name}/max_action"]), attention_pooling=None, dense=dense(A_))
        v = head.init(0, ro)
        assert v["params"]["Dense_0"]["kernel"].shape == g[f"{name}/kernel"].shape       # Flax's auto-name for the Dense
        v = {"params": {"Dense_0": {"kernel": g[f"{name}/kernel"], "bias": g[f"{name}/bias"]}}}
        pred = head.apply(v, ro)
        assert tuple(pred.shape) == g[f"{name}/pred"].shape                              # [B, 1, A] (continuous.py:22)
        np.testing.assert_allclose(pred.cpu().numpy(), g[f"{name}/pred"], rtol=1e-5, atol=1e-6)
        per_row, mean = AH.l2_loss(head, v, ro, act)
        np.testing.assert_allclose(per_row.cpu().numpy(), g[f"{name}/loss"], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(mean.item(), g[f"{name}/loss"].mean(), rtol=1e-4)
    for name in g["categorical"]:
        A_, bins = (int(x) for x in g[f"{name}/cfg"])
        ro, act = _dev(g[f"{name}/readouts"]), _dev(g[f"{name}/actions"])
        mx = float(g[f"{name}/max_action"])
        head = AH.CategoricalActionHead(num_bins=bins, max_action=mx, action_space_dim=A_, dense=dense(bins))
        v = {"params": {"Dense_0": {"kernel": g[f"{name}/kernel"], "bias": g[f"{name}/bias"]}}}
        logits = head.apply(v, ro)
        np.testing.assert_allclose(logits.cpu().numpy().reshape(g[f"{name}/logits"].shape), g[f"{name}/logits"], rtol=1e-5, atol=2e-6)
        np.testing.assert_array_equal(AH.categorical.assign_bins(act, (-mx, mx), bins), g[f"{name}/target_bin"])
        per_row, mean = AH.ce_loss(head, v, ro, act)
        np.testing.assert_allclose(per_row.cpu().numpy(), g[f"{name}/loss"].sum(-1), rtol=1e-4, atol=1e-5)
    with pytest.raises(ValueError, match="num_bins"):
        AH.CategoricalActionHead(num_bins=8, max_action=1.0, action_space_dim=2, dense=dense(7)).apply(
            {"params": {"Dense_0": {"kernel": np.zeros((16, 7), np.float32)}}}, torch.zeros(1, 4, 16, device="cuda"))


def _diffusion_node(A, F, Ht, To, H):
    dense = lambda f: {"_target_": "flax.linen.Dense", "features": f, "use_bias": True,  # noqa: E731
                       "kernel_init": {"_target_": "flax.linen.initializers.he_normal"},
                       "bias_init": {"_target_": "flax.linen.initializers.normal"}}
    mlp = lambda f0, f1: {"_target_": "multi_modal_transformers.attention_blocks.attention.MLPBlock", "dense": dense(f0),  # noqa: E731
                          "activation": {"_partial_": True, "_target_": "flax.linen.relu"},
                          "norm": {"_target_": "flax.linen.Dropout", "rate": 0.1}, "dense_out": dense(f1)}
    return {"_target_": "multi_modal_transformers.action_heads.diffusion.OctoDenoise", "num_blocks": 1,
            "time_encoder": {"_target_": "multi_modal_transformers.action_heads.diffusion.FourierFeatures", "output_dim": F,
                             "kernel_init": {"_target_": "flax.linen.initializers.he_normal"}, "mlp_block": mlp(Ht, To)},
            "mlp_block": mlp(H, A)}


def test_diffusion_head_module_schedule_and_param_tree():
    """DiffusionActionHead built from a diffusion.yaml-shaped node: the cosine schedule of :16-26 / :85-92 equals the
    reference's own (golden), and init() yields Flax's parameter tree with the yaml's literal widths."""
    g = np.load(os.path.join(GOLD, "action_heads.npz"))
    head = AH.DiffusionActionHead(diffusion_steps=32, attention_pooling=None, denoising_model=_diffusion_node(8, 768, 768, 768, 768))
    np.testing.assert_array_equal(head.betas, g["diff_schedule32/betas"])
    np.testing.assert_array_equal(head.alpha_hats, g["diff_schedule32/alpha_hats"])
    v = head.init(0, np.zeros((2, 8, 768), np.float32))["params"]["denoiser"]
    assert v["FourierFeatures_0"]["fourier_kernel"].shape == (384, 1)
    assert v["FourierFeatures_0"]["MLPBlock_0"]["Dense_1"]["kernel"].shape == (768, 768)
    assert v["MLPBlock_0"]["Dense_0"]["kernel"].shape == (8 + 768 + 768, 768)        # [noisy | time | readout] (:61)
    assert v["MLPBlock_0"]["Dense_1"]["kernel"].shape == (768, 8)
    with pytest.raises(NotImplementedError):
        AH.DiffusionActionHead(32, None, {**_diffusion_node(8, 32, 32, 32, 32), "num_blocks": 2})


@gpu
def test_diffusion_head_module_against_reference_goldens():
    """denoise_loss / predict_denoise_term of the module, on the parameters and draws of the goldens made by executing
    the reference's OctoDenoise (bf16 tensor-core GEMMs inside: 2e-2 relative)."""
    g = np.load(os.path.join(GOLD, "action_heads.npz"))
    for name in g["diffusion"]:
        p = {k: g[f"{name}/p/{k}"] for k in ("fourier_kernel", "tw1", "tb1", "tw2", "tb2", "w1", "b1", "w2", "b2")}
        A, F, Ht, To, H = p["w2"].shape[1], p["tw1"].shape[0], p["tw1"].shape[1], p["tw2"].shape[1], p["w1"].shape[1]
        head = AH.DiffusionActionHead(int(g[f"{name}/steps"]), None, _diffusion_node(A, F, Ht, To, H))
        v = {"params": {"denoiser": {
            "FourierFeatures_0": {"fourier_kernel": p["fourier_kernel"],
                                  "MLPBlock_0": {"Dense_0": {"kernel": p["tw1"], "bias": p["tb1"]}, "Dense_1": {"kernel": p["tw2"], "bias": p["tb2"]}}},
            "MLPBlock_0": {"Dense_0": {"kernel": p["w1"], "bias": p["b1"]}, "Dense_1": {"kernel": p["w2"], "bias": p["b2"]}}}}}
        ro, act = _dev(g[f"{name}/readouts"]), _dev(g[f"{name}/actions"])
        loss = head.denoise_loss(v, ro, act, time=_dev(g[f"{name}/time"]), noise=_dev(g[f"{name}/noise"]))
        assert abs(loss.item() - float(g[f"{name}/loss"])) <= 2e-2 * float(g[f"{name}/loss"])
        pred = head.predict_denoise_term(v, ro, _dev(g[f"{name}/time"]), _dev(g[f"{name}/noisy"]))
        want = torch.tensor(g[f"{name}/pred"])
        assert ((pred.cpu() - want).norm() / want.norm()).item() <= 2e-2
        # drawn internally: finite, reproducible for a seed, different for another
        l1, l2, l3 = (head.denoise_loss(v, ro, act, rng=s).item() for s in (1, 1, 2))
        assert np.isfinite(l1) and l1 == l2 and l1 != l3


def test_action_head_configs_build_the_mirror_modules():
    """model_configs.build_action_head on the reference's head schema (`_target_` strings of
    multi_modal_transformers.action_heads.*): the diffusion YAML shipped here, and continuous / categorical nodes."""
    head = MC.build_action_head(MC.load("action_heads/diffusion_octo_small"))
    assert isinstance(head, AH.DiffusionActionHead) and head.diffusion_steps == 32 and head.rng_collection == "diffusion"
    v = head.init(0, np.zeros((2, 8, 384), np.float32))["params"]["denoiser"]
    assert v["MLPBlock_0"]["Dense_0"]["kernel"].shape == (8 + 384 + 384, 384) and v["MLPBlock_0"]["Dense_1"]["kernel"].shape == (384, 8)
    dense = {"_target_": "flax.linen.Dense", "features": 7}
    c = MC.build_action_head({"_target_": "multi_modal_transformers.action_heads.continuous.ContinuousActionHead", "max_action": 2.0,
                              "attention_pooling": {"ignored": True}, "dense": dense})
    assert isinstance(c, AH.ContinuousActionHead) and c.max_action == 2.0
    k = MC.build_action_head({"_target_": "multi_modal_transformers.action_heads.categorical.CategoricalActionHead", "num_bins": 256,
                              "max_action": 1.0, "action_space_dim": 8, "dense": {**dense, "features": 256}})
    assert isinstance(k, AH.CategoricalActionHead) and k.action_space_dim == 8
    with pytest.raises(ValueError, match="unsupported action head"):
        MC.build_action_head({"_target_": "somewhere.OtherHead"})


@gpu
@pytest.mark.parametrize("name", ["lit_seq", "allones_1blk", "feature_ln"])
def test_vanilla_stack_module_against_the_executed_reference_blocks(name):
    """The drop-in StackedEncoder1DBlock (CUDA path) fed the SAME Flax parameter tree and inputs as the reference's own
    StackedEncoder1DBlock.__call__ (attention.py:87-119, executed under the shim by oracle/gen_golden.py ->
    tests/golden/encoder_blocks.npz): position embedding, scan over the stacked block parameters, pre-LN attention and MLP
    branches with their residuals, dense boolean mask as octo.py:66-68 / :119 builds it.  bf16 kernels vs the fp32 fixture:
    relative L2 error <= 2e-2."""
    EB = np.load(os.path.join(os.path.dirname(__file__), "golden", "encoder_blocks.npz"))
    B, T, C, H, Dff, N, ax = [int(v) for v in EB[f"{name}/meta"]]
    tree, pre = {}, f"{name}/params/"
    for k in EB.files:
        if k.startswith(pre):
            node, parts = tree, k[len(pre):].split("/")
            for p_ in parts[:-1]:
                node = node.setdefault(p_, {})
            node[parts[-1]] = EB[k]
    cfg = MC.load("attention_blocks/tome_decoder_octo_base")
    e = dict(cfg["encoder_1d_block"], _target_="multi_modal_transformers.attention_blocks.attention.Encoder1DBlock")
    e["layer_norm"] = dict(e["layer_norm"], reduction_axes=[ax])
    e["self_attention"] = dict(e["self_attention"], _target_="flax.linen.SelfAttention", num_heads=H, qkv_features=C)
    e["mlp_block"] = dict(e["mlp_block"], dense=dict(e["mlp_block"]["dense"], features=Dff),
                          dense_out=dict(e["mlp_block"]["dense_out"], features=C))
    stack = MC.build_stack({"num_blocks": N, "encoder_1d_block": e})
    assert type(stack) is A.StackedEncoder1DBlock
    x = _dev(EB[f"{name}/x"])
    mask = torch.as_tensor(EB[f"{name}/mask"]).expand(B, H, T, T)
    y = stack.apply({"params": tree}, x, train=False, mask=mask)
    want = torch.as_tensor(EB[f"{name}/y"])
    err = ((y.float().cpu() - want).norm() / want.norm()).item()
    assert err <= 2e-2, err


def test_image_tokenizer_config_nodes():
    """model_configs.build_image_tokenizer on the package's gato_resnet_octo.yaml: the geometry the file states, param tree
    names and shapes; unsupported nodes raise.  The reference's own gato_resnet.yaml is not part of this repository, so the
    packaged file is not compared with it here: a difference between the two would not be caught by this test."""
    import pytest
    from multi_modal_transformers_tokenmerge_b200 import model_configs as M
    tok = M.build_image_tokenizer(M.load("tokenizers/images/gato_resnet_octo"))
    assert tok.image_size == (280, 280, 3) and tok.patch_size == 56 and tok._geometry() == (23, 21)
    assert (tok.resnet.num_blocks, tok.resnet.num_groups, tok.resnet.pool_window, tok.resnet.dense_features) == (2, 32, 3, 768)
    node = M.load("tokenizers/images/gato_resnet_octo")["encoder"]
    bad = dict(node, resnet=dict(node["resnet"], input_pool=dict(node["resnet"]["input_pool"], strides=[2, 2])))
    with pytest.raises(NotImplementedError):
        M.build_image_tokenizer(bad)
    v = tok.init(0, None)["params"]
    assert v["embedding_function"]["Conv_0"]["kernel"].shape == (12, 12, 3, 64) and v["embedding_function"]["Dense_0"]["kernel"].shape == (21 * 21 * 64, 768)
    assert set(v) == {"embedding_function", "image_row_position_embedding", "image_col_position_embedding"}


def test_image_tokenizer_config_resolves_hydra_interpolations():
    """build_image_tokenizer resolves the hydra forms its docstring accepts: embedding sizes written as
    `${tokenizers.images.encoder.position_interval}` take the node's position_interval, and `dtype` / `param_dtype` keys are
    dropped.  The node is the packaged one rewritten in those forms with position_interval 64; it checks the resolver, not
    the reference's file."""
    import copy
    from multi_modal_transformers_tokenmerge_b200 import model_configs as M
    node = M.load("tokenizers/images/gato_resnet_octo")["encoder"]
    tok = M.build_image_tokenizer(node)
    hydra = copy.deepcopy(node)
    hydra["position_interval"] = 64
    dt = {"dtype": "${dtype}", "param_dtype": "${param_dtype}"}
    for k in ("row_position_embedding", "col_position_embedding"):
        hydra[k].update(num_embeddings="${tokenizers.images.encoder.position_interval}", **dt)
    for k in ("input_conv", "resnet_conv", "output_dense"):
        hydra["resnet"][k].update(dt)
    t2 = M.build_image_tokenizer({"encoder": hydra})
    assert (t2.image_size, t2.patch_size, t2.position_interval, t2.embedding_dim) == (tok.image_size, tok.patch_size, 64, 768)
    assert t2.resnet.input_conv == tok.resnet.input_conv and t2.resnet.resnet_conv == tok.resnet.resnet_conv
    v = t2.init(0, None)["params"]
    assert v["image_row_position_embedding"]["embedding"].shape == v["image_col_position_embedding"]["embedding"].shape == (64, 768)


def _pool_nodes(H, Dff, E, ax):
    he = {"_target_": "flax.linen.initializers.he_normal"}
    dense = lambda f: {"_target_": "flax.linen.Dense", "features": f, "use_bias": True, "kernel_init": he,  # noqa: E731
                       "bias_init": {"_target_": "flax.linen.initializers.normal"}}
    return dict(query_map_input={"kernel_init": he},
                dot_product_attention={"_target_": "flax.linen.MultiHeadDotProductAttention", "num_heads": H, "kernel_init": he},
                layer_norm={"_target_": "flax.linen.LayerNorm", "epsilon": 1e-6, "reduction_axes": [ax], "feature_axes": [-1]},
                mlp_block={"_target_": "multi_modal_transformers.attention_blocks.attention.MLPBlock", "dense": dense(Dff),
                           "activation": {"_partial_": True, "_target_": "flax.linen.relu"},
                           "norm": {"_target_": "flax.linen.Dropout", "rate": 0.1}, "dense_out": dense(E)})


def test_attention_pooling_param_tree():
    """MultiHeadAttentionPooling.init: Flax's names and shapes (attention.py:139-149), config nodes of diffusion.yaml:6-51."""
    pool = A.MultiHeadAttentionPooling(**_pool_nodes(3, 768, 768, 1))
    v = pool.init(0, np.zeros((2, 4, 768), np.float32))["params"]
    assert set(v) == {"learnt_q_input", "MultiHeadDotProductAttention_0", "LayerNorm_0", "MLPBlock_0"}
    assert v["learnt_q_input"].shape == (1, 1, 768)
    a = v["MultiHeadDotProductAttention_0"]
    assert a["query"]["kernel"].shape == (768, 3, 256) and a["key"]["bias"].shape == (3, 256) and a["out"]["kernel"].shape == (3, 256, 768)
    assert v["MLPBlock_0"]["Dense_0"]["kernel"].shape == (768, 768)


@gpu
@pytest.mark.parametrize("name", ["yaml_axes", "feature_ln", "one_readout"])
def test_attention_pooling_module_against_the_executed_reference(name):
    """MultiHeadAttentionPooling (CUDA path: key | value GEMM, csrc/attn_pool.cu, out GEMM, LayerNorm, MLP GEMMs) fed the SAME Flax
    parameter tree and tokens as the reference's own module (attention.py:122-150, executed under the shim ->
    tests/golden/attention_pooling.npz).  bf16 kernels vs the fp32 fixture: relative L2 error <= 2e-2."""
    Z = np.load(os.path.join(GOLD, "attention_pooling.npz"))
    B, n, E, H, Dff, ax = [int(v) for v in Z[f"{name}/meta"]]
    tree, pre = {}, f"{name}/params/"
    for k in Z.files:
        if k.startswith(pre):
            node, parts = tree, k[len(pre):].split("/")
            for p_ in parts[:-1]:
                node = node.setdefault(p_, {})
            node[parts[-1]] = Z[k]
    pool = A.MultiHeadAttentionPooling(**_pool_nodes(H, Dff, E, ax))
    y = pool.apply({"params": tree}, _dev(Z[f"{name}/x"]), train=False)
    want = torch.as_tensor(Z[f"{name}/y"])
    assert tuple(y.shape) == (B, 1, E)
    err = ((y.float().cpu() - want).norm() / want.norm()).item()
    assert err <= 2e-2, err


@gpu
def test_diffusion_head_sampler_against_the_oracle():
    """DiffusionActionHead.predict_action (diffusion.py:146-213, the inference loop) on the golden denoiser parameters with the
    start sample and the step noise supplied: vs oracle.diffusion_predict_action (fp32 restatement over the reference-pinned
    OctoDenoise).  bf16 GEMMs inside every one of the steps, each step scaling the running error by 1 / sqrt(alpha_t) >= 1:
    |err| <= 5e-2 of the clip range; results stay inside [-5, 5] and are reproducible."""
    g = np.load(os.path.join(GOLD, "action_heads.npz"))
    for name in g["diffusion"]:
        p = {k: g[f"{name}/p/{k}"] for k in ("fourier_kernel", "tw1", "tb1", "tw2", "tb2", "w1", "b1", "w2", "b2")}
        A, F, Ht, To, H = p["w2"].shape[1], p["tw1"].shape[0], p["tw1"].shape[1], p["tw2"].shape[1], p["w1"].shape[1]
        steps = int(g[f"{name}/steps"])
        head = AH.DiffusionActionHead(steps, None, _diffusion_node(A, F, Ht, To, H))
        v = {"params": {"denoiser": {
            "FourierFeatures_0": {"fourier_kernel": p["fourier_kernel"],
                                  "MLPBlock_0": {"Dense_0": {"kernel": p["tw1"], "bias": p["tb1"]}, "Dense_1": {"kernel": p["tw2"], "bias": p["tb2"]}}},
            "MLPBlock_0": {"Dense_0": {"kernel": p["w1"], "bias": p["b1"]}, "Dense_1": {"kernel": p["w2"], "bias": p["b2"]}}}}}
        ro = g[f"{name}/readouts"]
        rng = np.random.default_rng(5)
        B = ro.shape[0]
        init = rng.standard_normal((B, A)).astype(np.float32)
        noise = rng.standard_normal((B, A)).astype(np.float32)
        got = head.predict_action(v, _dev(ro), init=torch.tensor(init), noise=torch.tensor(noise))
        again = head.predict_action(v, _dev(ro), init=torch.tensor(init), noise=torch.tensor(noise))
        assert torch.equal(got, again) and got.abs().max().item() <= 5.0
        pt = {k: torch.tensor(a) for k, a in p.items()}
        want = O.diffusion_predict_action(torch.tensor(ro).to(torch.bfloat16).float(), torch.tensor(init), torch.tensor(noise), head.betas, pt)
        err = (got.cpu() - want).abs().max().item()
        assert err <= 5e-2 * 5.0, (name, err)
        drawn = head.predict_action(v, _dev(ro), rng=3)
        assert tuple(drawn.shape) == (B, A) and torch.isfinite(drawn).all()


def _compressed_stack(num_blocks=3, C=128, H=2, Dff=256, ln_axis=-1):
    import functools
    from multi_modal_transformers_tokenmerge_b200.attention_blocks import compressed_attention as CA
    cfg = MC.load("attention_blocks/tome_decoder_octo_small")
    e = dict(cfg["encoder_1d_block"], _target_="multi_modal_transformers.attention_blocks.compressed_attention.CompressedEncoder1DBlock")
    e["layer_norm"] = dict(e["layer_norm"], reduction_axes=[ln_axis])
    e["self_attention"] = dict(e["self_attention"], num_heads=H, qkv_features=C)
    e["mlp_block"] = dict(e["mlp_block"], dense=dict(e["mlp_block"]["dense"], features=Dff), dense_out=dict(e["mlp_block"]["dense_out"], features=C))
    ts = TokenSequence("[TaskDescriptionPrefix{8}] [Image{40};Readout{2}]*2", "[TaskDescriptionPrefix{0}] [Image{6};Readout{0}]*2")
    fns = []
    for l in range(num_blocks):     # what the reference's caller builds: partial(compute_top_k_tokens, tokenset_idx=..., tokenset_k=...)
        idx, ks = O.prune_sets_at(ts.prune_sets(), l)
        fns.append(functools.partial(TCm.compute_top_k_tokens, tokenset_idx=idx, tokenset_k=ks))
    return CA.StackedCompressedEncoder1DBlock(num_blocks, e, prune_fns=fns, merge_fns=[None] * num_blocks), ts, fns


def test_compressed_stack_module_arguments():
    """StackedCompressedEncoder1DBlock (compressed_attention.py:377-404): prune_fns as the reference builds them, token sets
    that must follow the compression grammar, merge_fns rejected (commented out in the reference, :310-311)."""
    from multi_modal_transformers_tokenmerge_b200.attention_blocks import compressed_attention as CA
    stack, ts, fns = _compressed_stack()
    assert stack.prune_sets == ((8, 0), (40, 6), (2, 0), (40, 6), (2, 0)) == tuple(ts.prune_sets())
    e = stack.encoder_1d_block
    with pytest.raises(ValueError, match="compression grammar"):
        CA.StackedCompressedEncoder1DBlock(3, e, prune_fns=[fns[0], fns[0], fns[2]])
    with pytest.raises(ValueError, match="one compute_top_k_tokens"):
        CA.StackedCompressedEncoder1DBlock(3, e, prune_fns=fns[:2])
    with pytest.raises(NotImplementedError):
        CA.StackedCompressedEncoder1DBlock(3, e, prune_fns=fns, merge_fns=[object()] * 3)
    v = stack.init(0, torch.zeros(2, 92, 128))["params"]
    assert set(v) == {"posembed_input", "ScanEncoder1DBlock_0"} and v["posembed_input"]["pos_embedding"].shape == (1, 92, 128)


@gpu
def test_compressed_stack_module_against_the_oracle():
    """The drop-in StackedCompressedEncoder1DBlock: masks[layer] from the compression grammar, one per-set top-k per layer
    (92 -> 80 -> 68 -> 56 tokens), against oracle.prune_stack following the module's keep decisions and ReLU gates: <= 2e-2."""
    stack, ts, _ = _compressed_stack()
    rng = np.random.default_rng(2)
    B, T, C = 2, 92, 128
    variables = stack.init(4, torch.zeros(B, T, C))
    x = rng.standard_normal((B, T, C)).astype(np.float32)
    masks = [ts.layer_group_ids(l) for l in range(3)]
    y = stack.apply(variables, _dev(x), masks=masks, allow=ts.allow_table(), train=False)
    assert tuple(y.shape) == (B, 56, C) and [tuple(i.shape) for i in stack.last_ids] == [(B, 80), (B, 68), (B, 56)]
    eng = stack._engine
    v, vf = eng.param_views(eng.params_bf16.float().cpu()), eng.param_views(eng.params.cpu())
    params, hd = [], 128
    for l in range(3):
        s_, f_ = v["layers"][l], vf["layers"][l]
        d = dict(ln1_scale=f_["ln1_scale"], ln1_bias=f_["ln1_bias"], ln2_scale=f_["ln2_scale"], ln2_bias=f_["ln2_bias"],
                 wq=s_["wqkv"][:, :hd], wk=s_["wqkv"][:, hd:2 * hd], wv=s_["wqkv"][:, 2 * hd:], bq=f_["bqkv"][:hd], bk=f_["bqkv"][hd:2 * hd],
                 bv=f_["bqkv"][2 * hd:], wo=s_["wo"], bo=f_["bo"], w1=s_["w1"], b1=f_["b1"], w2=s_["w2"], b2=f_["b2"])
        params.append(O.BlockParams(**{k_: t.clone().contiguous() for k_, t in d.items()}))
    gid, pos = ts.group_ids()
    want, _ = O.prune_stack(params, vf["pos_embedding"].clone()[None], torch.tensor(x), gid, pos, ts.allow_table(), num_heads=2,
                            sets=ts.prune_sets(), importance="received", ln_axis="feature", act_dtype=torch.bfloat16,
                            relu_gate=[eng.layer_relu_gate(l).cpu().numpy() for l in range(3)],
                            ids_override=[i.cpu().numpy() for i in stack.last_ids], layer_groups=masks)
    err = ((y.float().cpu() - want).norm() / want.norm()).item()
    assert err <= 2e-2, err
