"""AdamW options on the GPU (tome_adamw_opts_t): no-op options keep the plain step's bits, clipping and the masked decay match
an fp64 restatement of optax's clip_by_global_norm -> adamw(mask), non-finite steps are skipped without a trace, and a
data-parallel train step clips the mean gradient with the same norm bits on every rank."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

LR, B1, B2, EPS, WD = 1e-3, 0.9, 0.999, 1e-8, 0.1


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from multi_modal_transformers_tokenmerge_b200 import _lib, engine
    _lib.lib()
    return _lib, engine


def _octo_small(engine, **kw):
    base = dict(batch=2, tokens=536, channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, r=16, num_groups=5,
                n_readout=8, head="continuous", head_features=7)
    base.update(kw)
    return engine.StackConfig(**base)


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.bfloat16 else torch.int32).clone()


def _state(eng):
    return [_bits(t) for t in (eng.params, eng.adam_m, eng.adam_v, eng.params_bf16)]


def _reference(p, grads, steps, max_norm, decay_mask, gs=1.0, wd=WD, lr=LR):
    """fp64 optax.chain(clip_by_global_norm(max_norm), adamw(lr, b1, b2, eps, wd, mask)) over `grads`, one per step, with the
    hyperparameters the library receives (fp32 values: 1 - 0.999 alone differs by 1e-5 relative from 1 - fp32(0.999))."""
    b1, b2, eps, wd, lr = (float(np.float32(h)) for h in (B1, B2, EPS, wd, lr))
    p = p.double().clone()
    m = torch.zeros_like(p)
    v = torch.zeros_like(p)
    for t, g in zip(steps, grads):
        g = g.double() * gs
        norm = g.norm()
        if max_norm and norm >= max_norm:
            g = g / norm * max_norm
        m = b1 * m + (1 - b1) * g
        v = b2 * v + (1 - b2) * g * g
        upd = (m / (1 - b1 ** t)) / ((v / (1 - b2 ** t)).sqrt() + eps)
        p = p - lr * (upd + wd * p * decay_mask)
    return p, m, v


def _rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-300)).item()


def test_noop_options_give_the_plain_step_bits(pkg):
    """max_grad_norm above the norm, one decay range covering everything and no skipping: three steps through the options
    path equal three plain (opts == NULL) steps bit for bit, n not a multiple of 4."""
    L, _ = pkg
    lib = L.lib()
    n = (1 << 22) + 3
    g = torch.Generator(device="cuda").manual_seed(3)
    p0 = torch.randn(n, device="cuda", generator=g)
    grads = [torch.randn(n, device="cuda", generator=g) * 1e-2 for _ in range(3)]
    ws = torch.empty(lib.tome_adamw_workspace_bytes(n), dtype=torch.uint8, device="cuda")
    norm = torch.zeros(1, device="cuda")
    rng = (C.c_longlong * 2)(0, n)
    out = []
    for use_opts in (False, True):
        p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
        w16 = torch.empty(n, dtype=torch.bfloat16, device="cuda")
        for t, gr in enumerate(grads, 1):
            opts = L.AdamwOpts(1e6, 0, rng, 1, norm.data_ptr(), None, ws.data_ptr(), ws.numel()) if use_opts else None
            L.check(lib.tome_adamw_step(n, p.data_ptr(), gr.data_ptr(), m.data_ptr(), v.data_ptr(), w16.data_ptr(), LR, B1, B2,
                                        EPS, WD, 0.5, t, None if opts is None else C.byref(opts), None))
        torch.cuda.synchronize()
        out.append([_bits(x) for x in (p, m, v, w16)])
    for a, b in zip(*out):
        assert torch.equal(a, b)
    assert abs(norm.item() - (grads[-1].double() * 0.5).norm().item()) <= 1e-6 * norm.item()


def test_clipping_and_masked_decay_match_fp64_optax(pkg):
    """Octo-small parameter count, gradients 10-1000x over max_grad_norm: three clipped steps with weight decay on the Dense
    kernels only match the fp64 restatement per tensor within 1e-6 relative; the norm equals the fp64 norm within 1e-6 and
    is the same bits every time the same gradient comes back."""
    _, engine = pkg
    eng = engine.ToMeStackEngine(_octo_small(engine))
    eng.init_params(seed=2)
    p0 = eng.params.clone()
    g = torch.Generator(device="cuda").manual_seed(5)
    scales = [10.0, 1000.0, 10.0]
    base = torch.randn(eng.n_params, device="cuda", generator=g)
    grads = [base * (s / base.norm()) for s in scales]   # steps 1 and 3 see the same gradient
    mask = torch.zeros(eng.n_params, dtype=torch.float64, device="cuda")
    for a, b in eng.decay_ranges("dense_kernels"):
        mask[a:b] = 1.0
    norms = []
    for gr in grads:
        eng.grads.copy_(gr)
        eng.adamw_step(lr=LR, beta1=B1, beta2=B2, eps=EPS, weight_decay=WD, max_grad_norm=1.0, decay="dense_kernels")
        norms.append(eng.grad_norm.clone())
    torch.cuda.synchronize()
    p, m, v = _reference(p0, grads, [1, 2, 3], 1.0, mask)
    for got, want, name in ((eng.params, p, "param"), (eng.adam_m, m, "m"), (eng.adam_v, v, "v")):
        gv, wv = eng.param_views(got), eng.param_views(want)
        pairs = [(gv["pos_embedding"], wv["pos_embedding"], "pos_embedding")]
        pairs += [(gv["layers"][l][k], wv["layers"][l][k], f"{l}.{k}") for l in range(eng.cfg.layers) for k in gv["layers"][l]]
        pairs += [(gv["head"][k], wv["head"][k], f"head.{k}") for k in gv["head"]]
        for a, b, k in pairs:
            e = _rel(a, b)
            assert e <= 1e-6, f"{name} {k}: rel err {e}"
    for gr, nrm in zip(grads, norms):
        want = gr.double().norm().item()
        assert abs(nrm.item() - want) <= 1e-6 * want
    assert torch.equal(_bits(norms[0]), _bits(norms[2]))
    assert torch.equal(eng.params_bf16, eng.params.bfloat16())


@pytest.mark.parametrize("bad", [float("nan"), float("inf")], ids=["nan", "inf"])
def test_nonfinite_step_is_skipped_without_a_trace(pkg, bad):
    """One NaN / +Inf in layer 0's w1 gradient: params, moments, bf16 copy and the applied counter stay bit-unchanged and the
    skipped counter becomes 1; the next finite step equals the fp64 reference that never saw the bad step, bias correction
    included."""
    _, engine = pkg
    eng = engine.ToMeStackEngine(_octo_small(engine, layers=2))
    eng.init_params(seed=4)
    p0 = eng.params.clone()
    g = torch.Generator(device="cuda").manual_seed(6)
    g1, g3 = (torch.randn(eng.n_params, device="cuda", generator=g) * 1e-3 for _ in range(2))
    kw = dict(lr=LR, beta1=B1, beta2=B2, eps=EPS, weight_decay=WD, max_grad_norm=1.0, skip_nonfinite=True)
    eng.grads.copy_(g1)
    eng.adamw_step(**kw)
    before = _state(eng)
    assert eng.optimizer_steps() == (1, 0)
    eng.grads.copy_(g3)
    eng.param_views(eng.grads)["layers"][0]["w1"][5, 17] = bad
    eng.adamw_step(**kw)
    torch.cuda.synchronize()
    for a, b in zip(before, _state(eng)):
        assert torch.equal(a, b)
    assert eng.optimizer_steps() == (1, 1)
    if bad != bad:
        assert eng.grad_norm.isnan().item()
    eng.grads.copy_(g3)
    eng.adamw_step(**kw)
    assert eng.optimizer_steps() == (2, 1)
    p, m, v = _reference(p0, [g1, g3], [1, 2], 1.0, torch.ones(eng.n_params, dtype=torch.float64, device="cuda"))
    for got, want in ((eng.params, p), (eng.adam_m, m), (eng.adam_v, v)):
        gv, wv = eng.param_views(got), eng.param_views(want)
        for l in range(eng.cfg.layers):
            for k in gv["layers"][l]:
                assert _rel(gv["layers"][l][k], wv["layers"][l][k]) <= 1e-6, (l, k)
        assert _rel(gv["head"]["kernel"], wv["head"]["kernel"]) <= 1e-6


def test_decay_mask_leaves_the_unmasked_parameters_alone(pkg):
    """Zero gradient, lr and wd > 0, decay="dense_kernels" on a diffusion-head stack: LayerNorm parameters, all biases,
    pos_embedding and the Fourier kernel keep their bits; every Dense kernel becomes p - lr * (wd * p) in fp32 (the kernel
    fuses the last multiply-subtract, so within one ulp)."""
    _, engine = pkg
    cfg = _octo_small(engine, layers=2, head="diffusion", head_features=8, head_fourier_dim=64, head_time_hidden=64,
                      head_time_out=64, head_hidden=256, diffusion_steps=32)
    eng = engine.ToMeStackEngine(cfg)
    eng.init_params(seed=8)
    eng.param_views(eng.params)["head"]["fourier_kernel"].normal_()
    for d in eng.param_views(eng.params)["layers"]:
        d["ln1_bias"].normal_()
        d["ln2_scale"].normal_()
    p0 = eng.params.clone()
    eng.zero_grad()
    lr, wd = 1e-2, 0.1
    eng.adamw_step(lr=lr, weight_decay=wd, decay="dense_kernels")
    torch.cuda.synchronize()
    got, was = eng.param_views(eng.params), eng.param_views(p0)
    fixed = [(got["pos_embedding"], was["pos_embedding"])]
    decayed = []
    for l in range(cfg.layers):
        for k in got["layers"][l]:
            (decayed if k in ("wqkv", "wo", "w1", "w2") else fixed).append((got["layers"][l][k], was["layers"][l][k]))
    for k in got["head"]:
        (decayed if k in ("tw1", "tw2", "w1", "w2") else fixed).append((got["head"][k], was["head"][k]))
    for a, b in fixed:
        assert torch.equal(_bits(a), _bits(b))
    lr32, wd32 = torch.tensor(lr, dtype=torch.float32), torch.tensor(wd, dtype=torch.float32)
    for a, b in decayed:
        want = b - lr32.cuda() * (wd32.cuda() * b)
        ulps = (_bits(a).long() - _bits(want).long()).abs().max().item()
        assert ulps <= 1, ulps
        assert not torch.equal(a, b)


def test_data_parallel_step_clips_the_mean_gradient(pkg):
    """Octo-small widths, two layers, continuous head, through DataParallelTrainer (one rank): the norm the step clipped with
    is the fp64 norm of grads / world within 1e-6, and the loss falls over a few clipped steps."""
    _, engine = pkg
    from multi_modal_transformers_tokenmerge_b200.parallel import DataParallelTrainer
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import sequence_groups
    gid, pos, allow, ro = sequence_groups("[TaskDescriptionPrefix{16}] [Image{64};Readout{4}]*2")
    B, A = 16, 7
    cfg = engine.StackConfig(batch=B, tokens=len(gid), channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=2, r=8,
                             num_groups=allow.shape[0], n_readout=len(ro), head="continuous", head_features=A)
    eng = engine.ToMeStackEngine(cfg, gid=gid, pos=pos, allow=allow, readout_idx=ro)
    eng.init_params(seed=1)
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(B, len(gid), 384, device="cuda", generator=g).bfloat16()
    y = torch.rand(B, A, device="cuda", generator=g) * 2 - 1
    tr = DataParallelTrainer(eng)
    losses = []
    for _ in range(8):
        tr.train_step(x, y, lr=1e-4, max_grad_norm=1.0, skip_nonfinite=True, decay="dense_kernels", weight_decay=1e-4)
        torch.cuda.synchronize()
        want = (eng.grads / tr.world).double().norm().item()
        assert abs(eng.grad_norm.item() - want) <= 1e-6 * want
        losses.append(eng.loss[0].item())
    assert eng.optimizer_steps() == (8, 0)
    assert losses[-1] < losses[0], losses


@pytest.mark.parametrize("overlap", ["layer", "none"])
def test_two_ranks_clip_with_the_same_norm_bits(overlap):
    """Two GPUs, different shards, clipping that triggers: both ranks report the same grad_norm bits at every step and the
    replicas' parameters stay bit-identical."""
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29534", os.path.join(here, "dp_clip_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env={**os.environ, "TOME_DP_OVERLAP": overlap})
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("DPCLIP ")][-1]
    res = json.loads(line[len("DPCLIP "):])
    print(res)
    assert res["world"] == 2 and res["overlap"] == overlap
    assert res["clipped_steps"] == res["steps"] > 0, res
    assert res["norm_bits_equal"] and res["params_in_sync"], res
