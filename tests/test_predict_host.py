"""CPU-only: the forward-only executor's C ABI (tome_stack_predict, tome_diffusion_head_sample) -- struct layout, workspace
sizes and argument checks, all before any CUDA call -- and predictor()'s parameter sharing."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = C.c_void_p(1 << 20)   # a device pointer the validation must refuse before touching


@pytest.fixture(scope="module")
def lib():
    from multi_modal_transformers_tokenmerge_b200 import _lib, build
    build.build()
    return _lib.lib()


def _octo_small(**kw):
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    base = dict(batch=256, tokens=536, channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, r=16, num_groups=5, n_readout=8,
                head="continuous", head_features=7)
    base.update(kw)
    return StackConfig(**base)


def _diffusion(**kw):
    d = dict(head="diffusion", head_features=8, head_fourier_dim=64, head_time_hidden=64, head_time_out=64, head_hidden=256,
             diffusion_steps=32)
    d.update(kw)
    return _octo_small(**d)


def test_ddpm_sample_struct_matches_header(tmp_path):
    """tome_ddpm_sample_t as gcc lays it out in C99 equals the ctypes mirror, field by field."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lines = ['printf("size %zu\\n", sizeof(tome_ddpm_sample_t));']
    want = [f"size {C.sizeof(L.DdpmSample)}"]
    for f, _ in L.DdpmSample._fields_:
        lines.append(f'printf("{f} %zu %zu\\n", offsetof(tome_ddpm_sample_t, {f}), sizeof(((tome_ddpm_sample_t*)0)->{f}));')
        want.append(f"{f} {getattr(L.DdpmSample, f).offset} {getattr(L.DdpmSample, f).size}")
    src = tmp_path / "s.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "include/tome_b200.h"\nint main(void) {\n' + "\n".join(lines) +
                   "\nreturn 0;\n}\n")
    exe = tmp_path / "s"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", f"-I{ROOT}", str(src), "-o", str(exe)], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    assert subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines() == want


def test_predict_workspace_is_a_fraction_of_training(lib):
    """octo-small, B = 256, 12 layers, r = 16: the predict workspace is under a sixth of the training one."""
    c = _octo_small().c()
    train, pred = lib.tome_stack_workspace_bytes(C.byref(c)), lib.tome_stack_predict_workspace_bytes(C.byref(c))
    assert 0 < pred < train / 6, (pred, train)
    d = _diffusion().c()
    assert 0 < lib.tome_stack_predict_workspace_bytes(C.byref(d)) < lib.tome_stack_workspace_bytes(C.byref(d)) / 6


@pytest.mark.parametrize("kind", ["global", "set_merge", "prune"])
def test_predict_workspace_grows_by_the_row_maps_only(lib, kind):
    """12 layers minus 1 layer = the row maps of layers 1 .. 11 (i32 [B, T_in(l)], each rounded up to 256 bytes)."""
    sets = ((16, 0), (256, 8), (4, 0), (256, 8), (4, 0))
    kw = {"global": {}, "set_merge": dict(r=0, prune_sets=sets, set_merge=True),
          "prune": dict(r=0, prune_sets=sets, prop_attn=False)}[kind]
    c12, c1 = _octo_small(**kw).c(), _octo_small(layers=1, **kw).c()
    b12, b1 = lib.tome_stack_predict_workspace_bytes(C.byref(c12)), lib.tome_stack_predict_workspace_bytes(C.byref(c1))
    maps = sum((4 * 256 * lib.tome_stack_tokens_at(C.byref(c12), l) + 255) // 256 * 256 for l in range(1, 12))
    assert b12 - b1 == maps


def _io(ws_bytes, head_out=True):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    io = L.StackIO()
    io.params_f32 = io.params_bf16 = io.x = io.workspace = FAKE
    io.gid = io.pos = io.allow = io.readout_idx = FAKE
    io.workspace_bytes = ws_bytes
    io.head_out = FAKE if head_out else None
    return io


def test_predict_arguments_are_checked_on_the_host(lib):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    d = _diffusion().c()
    ws = lib.tome_stack_predict_workspace_bytes(C.byref(d))
    smp = L.DdpmSample(FAKE, FAKE, 0, FAKE, 5.0)
    assert lib.tome_stack_predict(C.byref(d), C.byref(_io(ws)), None, None) == L.TOME_ERR_INVALID
    assert b"sample" in lib.tome_last_error()
    cont = _octo_small().c()
    ws_c = lib.tome_stack_predict_workspace_bytes(C.byref(cont))
    assert lib.tome_stack_predict(C.byref(cont), C.byref(_io(ws_c)), C.byref(smp), None) == L.TOME_ERR_INVALID
    for field, value, msg in (("noise_per_step", 2, b"noise_per_step"), ("clip", 0.0, b"clip"), ("clip", -1.0, b"clip")):
        bad = L.DdpmSample.from_buffer_copy(smp)
        setattr(bad, field, value)
        assert lib.tome_stack_predict(C.byref(d), C.byref(_io(ws)), C.byref(bad), None) == L.TOME_ERR_INVALID, field
        assert msg in lib.tome_last_error(), (field, lib.tome_last_error())
    assert lib.tome_stack_predict(C.byref(d), C.byref(_io(ws - 256)), C.byref(smp), None) == L.TOME_ERR_INVALID
    assert b"workspace too small" in lib.tome_last_error()
    assert lib.tome_stack_predict(C.byref(cont), C.byref(_io(ws_c - 1)), None, None) == L.TOME_ERR_INVALID
    assert lib.tome_stack_predict(C.byref(cont), C.byref(_io(ws_c, head_out=False)), None, None) == L.TOME_ERR_INVALID
    assert b"head_out" in lib.tome_last_error()


def test_sampler_arguments_and_limits(lib):
    """The sampling kernel keeps W1[:A] and W2 in fp32 shared memory: wider shapes are refused as unsupported."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    smp = L.DdpmSample(FAKE, FAKE, 0, FAKE, 5.0)
    ok = L.DiffusionDesc(4, 10, 64, 4, 8, 64, 64, 64, 768, 32)
    n = lib.tome_diffusion_head_sample_workspace_bytes(C.byref(ok))
    assert n > 0
    call = lambda d, s, nb: lib.tome_diffusion_head_sample(C.byref(d), FAKE, FAKE, FAKE, FAKE, s, FAKE, FAKE, nb, None)  # noqa: E731
    for field, value in (("noise_per_step", -1), ("clip", 0.0)):
        bad = L.DdpmSample.from_buffer_copy(smp)
        setattr(bad, field, value)
        assert call(ok, C.byref(bad), n) == L.TOME_ERR_INVALID, field
    assert call(ok, None, n) == L.TOME_ERR_INVALID
    assert call(ok, C.byref(smp), n - 256) == L.TOME_ERR_INVALID and b"workspace" in lib.tome_last_error()
    for a, h in ((72, 256), (8, 4096), (64, 2048)):
        wide = L.DiffusionDesc(4, 10, 64, 4, a, 64, 64, 64, h, 32)
        assert lib.tome_diffusion_head_sample_workspace_bytes(C.byref(wide)) == 0
        assert call(wide, C.byref(smp), 1 << 30) == L.TOME_ERR_UNSUPPORTED, (a, h)
        assert b"limits" in lib.tome_last_error()
    d = _diffusion(head_hidden=4096).c()
    assert lib.tome_stack_predict_workspace_bytes(C.byref(d)) == 0
    assert lib.tome_stack_predict(C.byref(d), C.byref(_io(1 << 40)), C.byref(smp), None) == L.TOME_ERR_UNSUPPORTED


def test_predictor_shares_the_parameter_storage(lib, monkeypatch):
    """predictor() wraps the training engine's params / params_bf16, at its batch or another one (no device work: built on
    CPU tensors here)."""
    import torch
    from multi_modal_transformers_tokenmerge_b200 import engine
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    cfg = _octo_small(batch=2, layers=2)
    eng = engine.ToMeStackEngine(cfg, device="cpu")
    for batch in (None, 64):
        p = eng.predictor(batch)
        assert p.params.data_ptr() == eng.params.data_ptr() and p.params_bf16.data_ptr() == eng.params_bf16.data_ptr()
        assert p.predict_only and p.grads is None and p.cfg.batch == (batch or 2)
        assert p._ws_bytes == lib.tome_stack_predict_workspace_bytes(C.byref(p.ccfg))
        with pytest.raises(RuntimeError, match="predict-only"):
            p.forward(torch.zeros(p.cfg.batch, cfg.tokens, cfg.channels))
        with pytest.raises(RuntimeError, match="predict-only"):
            p.adamw_step()
    with pytest.raises(RuntimeError, match="predict-only engine"):
        eng.predict(torch.zeros(2, cfg.tokens, cfg.channels))
