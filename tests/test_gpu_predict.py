"""The forward-only executor (tome_stack_predict) and the one-kernel diffusion sampler (tome_diffusion_head_sample) on the GPU.
Needs a B200: `-m gpu`.

Parity protocol: with dropout 0 the predict path runs the training forward's kernels on the same shapes, so x_final, the
readout rows and the continuous / categorical head output must equal tome_stack_forward's bit for bit (after checking that
two training forwards do)."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from oracle import tome_oracle as O  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence  # noqa: E402

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SEQ = "[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2"
COMP = "[TaskDescriptionPrefix{0}] [Image{8};Readout{0}]*2"


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from multi_modal_transformers_tokenmerge_b200 import _lib, engine, ops
    _lib.lib()
    return ops, engine


def _stack(engine, kind, B=4, **over):
    """A training engine (dropout 0) of one stack kind at octo-small widths (12 layers) unless the kind says otherwise."""
    ts = TokenSequence(SEQ, COMP)
    gid, pos = ts.group_ids()
    allow, ro = ts.allow_table(), ts.get_modality_idx("readouts")
    cfg = dict(batch=B, tokens=536, channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, r=16, ln_axis=1,
               num_groups=allow.shape[0], n_readout=len(ro), head="continuous", head_features=7, max_action=1.0)
    extra = {}
    if kind == "set_merge":
        cfg.update(r=0, prune_sets=tuple(ts.prune_sets()), set_merge=True, ln_axis=2, head="categorical", head_groups=4, head_features=16)
    elif kind in ("prune", "prune_grammar"):
        cfg.update(r=0, prune_sets=tuple(ts.prune_sets()), prop_attn=False)
        if kind == "prune_grammar":
            lg = [ts.layer_group_ids(l) for l in range(12)]
            extra = dict(layer_gid=[g for g, _ in lg], layer_pos=[p for _, p in lg])
    elif kind == "feature_ln":
        cfg.update(ln_axis=2, head="categorical", head_groups=8, head_features=32)
    elif kind == "head_dim_32":
        cfg.update(channels=256, heads=4, head_dim=32, mlp_dim=512, layers=4)
    elif kind == "class_token":
        cfg.update(class_token=True, num_groups=0, head="none")
        gid = pos = allow = None
    elif kind == "diffusion":
        cfg.update(head="diffusion", head_features=8, head_fourier_dim=64, head_time_hidden=64, head_time_out=64, head_hidden=256,
                   diffusion_steps=32, layers=4)
    cfg.update(over)
    eng = engine.ToMeStackEngine(engine.StackConfig(**cfg), gid=gid, pos=pos, allow=allow, readout_idx=ro, **extra)
    eng.init_params(seed=3)
    return eng


def _input(eng, dtype, seed=1):
    c = eng.cfg
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(c.batch, c.tokens, c.channels, device="cuda", generator=g).to(dtype)


def _train_outputs(eng, x):
    eng.forward(x)
    torch.cuda.synchronize()
    head = None if eng.head_out is None else eng.head_out.clone()
    return eng.final_x().clone(), None if eng.readout is None else eng.readout.clone(), head


@pytest.mark.parametrize("kind,dtype", [("global", torch.bfloat16), ("set_merge", torch.bfloat16), ("prune", torch.bfloat16),
                                        ("prune_grammar", torch.float32), ("feature_ln", torch.float32),
                                        ("head_dim_32", torch.bfloat16), ("class_token", torch.float32)])
def test_predict_equals_training_forward_bitwise(pkg, kind, dtype):
    _, engine = pkg
    eng = _stack(engine, kind)
    x = _input(eng, dtype)
    xf0, ro0, h0 = _train_outputs(eng, x)
    xf1, ro1, h1 = _train_outputs(eng, x)
    assert torch.equal(xf0, xf1) and (ro0 is None or torch.equal(ro0, ro1)) and (h0 is None or torch.equal(h0, h1))
    p = eng.predictor()
    xf = torch.empty_like(xf0)
    out, ro = p.predict(x, x_final=xf)
    torch.cuda.synchronize()
    assert torch.equal(xf, xf0), kind
    assert ro0 is None or torch.equal(ro, ro0), kind
    if h0 is not None:
        assert torch.equal(out.reshape(h0.shape), h0), kind
    # dropout in the config is not applied by the predictor
    drop = engine.ToMeStackEngine(engine.StackConfig(**{**eng.cfg.__dict__, "dropout_rate": 0.1, "attn_dropout_rate": 0.1}),
                                  predict_only=True, _params=(eng.params, eng.params_bf16))
    drop.gid, drop.pos, drop.allow, drop.readout_idx, drop.layer_gid, drop.layer_pos = p.gid, p.pos, p.allow, p.readout_idx, p.layer_gid, p.layer_pos
    drop.predict(x, x_final=xf)
    torch.cuda.synchronize()
    assert torch.equal(xf, xf0), kind


def _diffusion_node(A, F, Ht, To, H):
    """OctoDenoise config node of diffusion.yaml's shape (time encoder MLPBlock Ht -> To, denoiser MLPBlock H -> A)."""
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


def _golden_head(AH, name, g):
    p = {k: g[f"{name}/p/{k}"] for k in ("fourier_kernel", "tw1", "tb1", "tw2", "tb2", "w1", "b1", "w2", "b2")}
    A, F, Ht, To, H = p["w2"].shape[1], p["tw1"].shape[0], p["tw1"].shape[1], p["tw2"].shape[1], p["w1"].shape[1]
    head = AH.DiffusionActionHead(int(g[f"{name}/steps"]), None, _diffusion_node(A, F, Ht, To, H))
    v = {"params": {"denoiser": {
        "FourierFeatures_0": {"fourier_kernel": p["fourier_kernel"],
                              "MLPBlock_0": {"Dense_0": {"kernel": p["tw1"], "bias": p["tb1"]}, "Dense_1": {"kernel": p["tw2"], "bias": p["tb2"]}}},
        "MLPBlock_0": {"Dense_0": {"kernel": p["w1"], "bias": p["b1"]}, "Dense_1": {"kernel": p["w2"], "bias": p["b2"]}}}}}
    return head, v, p, A


@pytest.mark.parametrize("per_step", [False, True])
def test_sampler_against_the_oracle(pkg, per_step):
    """The whole reverse process in one call vs oracle.diffusion_predict_action on the golden denoiser parameters, the step
    noise given as [B, A] (reused by every step) or [steps, B, A]: |err| <= 5e-2 of the clip range, as the per-step loop's test
    allows; bitwise reproducible; inside [-5, 5]; predict_action(rng=3) finite and [B, A]."""
    from multi_modal_transformers_tokenmerge_b200 import action_heads as AH
    g = np.load(os.path.join(GOLD, "action_heads.npz"))
    for name in g["diffusion"]:
        head, v, p, A = _golden_head(AH, name, g)
        ro = g[f"{name}/readouts"]
        B, steps = ro.shape[0], head.diffusion_steps
        rng = np.random.default_rng(7)
        init = rng.standard_normal((B, A)).astype(np.float32)
        noise = rng.standard_normal((steps, B, A) if per_step else (B, A)).astype(np.float32)
        x = torch.tensor(ro).cuda()
        got = head.predict_action(v, x, init=torch.tensor(init), noise=torch.tensor(noise))
        again = head.predict_action(v, x, init=torch.tensor(init), noise=torch.tensor(noise))
        assert torch.equal(got, again) and got.abs().max().item() <= 5.0
        want = O.diffusion_predict_action(torch.tensor(ro).to(torch.bfloat16).float(), torch.tensor(init), torch.tensor(noise), head.betas,
                                          {k: torch.tensor(a) for k, a in p.items()})
        err = (got.cpu() - want).abs().max().item()
        assert err <= 5e-2 * 5.0, (name, err)
        drawn = head.predict_action(v, x, rng=3)
        assert tuple(drawn.shape) == (B, A) and torch.isfinite(drawn).all()


def test_stack_diffusion_prediction_equals_the_sampler_on_training_readouts(pkg):
    """head 3: tome_stack_predict == tome_diffusion_head_sample on the readout rows of a dropout-0 training forward, bitwise."""
    ops, engine = pkg
    from multi_modal_transformers_tokenmerge_b200.action_heads.diffusion import cosine_beta_schedule, ddpm_coefficients
    eng = _stack(engine, "diffusion", B=8)
    c = eng.cfg
    x = _input(eng, torch.bfloat16)
    B, A = c.batch, c.head_features
    eng.set_diffusion_draws(torch.zeros(B, dtype=torch.int32, device="cuda"), np.ones(c.diffusion_steps, np.float32))
    eng.forward(x, torch.zeros(2, B, A, device="cuda"))
    readouts = eng.readout.to(torch.bfloat16).contiguous()
    rng = np.random.default_rng(11)
    init = torch.tensor(rng.standard_normal((B, A)).astype(np.float32)).cuda()
    for noise in (torch.tensor(rng.standard_normal((B, A)).astype(np.float32)).cuda(),
                  torch.tensor(rng.standard_normal((c.diffusion_steps, B, A)).astype(np.float32)).cuda()):
        coef = torch.tensor(ddpm_coefficients(cosine_beta_schedule(c.diffusion_steps))).cuda()
        off = eng.layer_offset(c.layers)
        want = ops.diffusion_head_sample(readouts, eng.params[off:], c.diffusion_desc(c.n_readout), init, noise, coef,
                                         params_bf16=eng.params_bf16[off:])
        got, _ = eng.predictor().predict(x, init=init, noise=noise)
        torch.cuda.synchronize()
        assert torch.equal(got, want)
        assert got.abs().max().item() <= 5.0


def test_large_batch_beyond_the_training_workspace(pkg, record_property):
    """octo-small at B = 4096: the training workspace does not fit the card, the predict one does; the first 256 rows match a
    B = 256 prediction within bf16 tolerance (the GEMMs take no split-K and every other kernel works row by row, so they are
    expected to match bit for bit; the assertion is the tolerance)."""
    _, engine = pkg
    import ctypes as C
    eng = _stack(engine, "global", B=256)
    big = eng.predictor(4096)
    total = torch.cuda.get_device_properties(0).total_memory
    assert eng.lib.tome_stack_workspace_bytes(C.byref(big.ccfg)) > total
    x = _input(big, torch.bfloat16, seed=5)
    out_big, ro_big = big.predict(x)
    out_big, ro_big = out_big[:256].clone(), ro_big[:256].clone()
    del big
    out, ro = eng.predictor().predict(x[:256].contiguous())
    torch.cuda.synchronize()
    assert torch.isfinite(out_big).all()
    assert torch.allclose(out_big, out, atol=2e-2, rtol=0) and torch.allclose(ro_big, ro, atol=3e-2, rtol=2e-2)
    bitwise = torch.equal(out_big, out) and torch.equal(ro_big, ro)
    record_property("first_256_rows_bitwise", bitwise)
    print(f"B = 4096 vs B = 256, first 256 rows bitwise equal: {bitwise}")


@pytest.mark.parametrize("kind", ["global", "diffusion"])
def test_predictor_sees_optimiser_steps_without_reload(pkg, kind):
    """A predictor built before an AdamW step predicts with the stepped parameters: equal, bit for bit, to a freshly loaded
    predict-only engine's output, and different from its own output before the step."""
    _, engine = pkg
    eng = _stack(engine, kind, B=4)
    c = eng.cfg
    p = eng.predictor()
    x = _input(eng, torch.bfloat16)
    init = torch.zeros(c.batch, c.head_features, device="cuda")
    before, _ = p.predict(x, init=init, noise=init)
    before = before.clone()
    if kind == "diffusion":
        eng.set_diffusion_draws(torch.full((c.batch,), 3, dtype=torch.int32, device="cuda"),
                                np.linspace(0.9, 0.1, c.diffusion_steps).astype(np.float32))
        y = torch.randn(2, c.batch, c.head_features, device="cuda")
    else:
        y = torch.rand(c.batch, c.head_features, device="cuda") * 2 - 1
    eng.zero_grad()
    eng.forward(x, y)
    eng.backward()
    eng.adamw_step(lr=1e-3)
    after, _ = p.predict(x, init=init, noise=init)
    after = after.clone()
    fresh = engine.ToMeStackEngine(c, predict_only=True)
    fresh.params.copy_(eng.params)
    fresh.params_bf16.copy_(eng.params_bf16)
    fresh.gid, fresh.pos, fresh.allow, fresh.readout_idx = eng.gid, eng.pos, eng.allow, eng.readout_idx
    want, _ = fresh.predict(x, init=init, noise=init)
    torch.cuda.synchronize()
    assert torch.equal(after, want)
    assert not torch.equal(after, before)
