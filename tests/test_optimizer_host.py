"""CPU-only: the AdamW options of the C ABI (tome_adamw_opts_t) -- struct layout against the header, malformed options refused
before any CUDA call -- and the engine's weight-decay mask built from its parameter layout."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = C.c_void_p(1 << 20)   # a device pointer the validation must refuse before touching
N = 1000


@pytest.fixture(scope="module")
def lib():
    from multi_modal_transformers_tokenmerge_b200 import _lib, build
    build.build()
    return _lib.lib()


def test_adamw_opts_struct_matches_header(tmp_path):
    """tome_adamw_opts_t as gcc lays it out in C99 equals the ctypes mirror, field by field."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lines = ['printf("size %zu\\n", sizeof(tome_adamw_opts_t));', 'printf("max %d\\n", TOME_ADAMW_MAX_DECAY_RANGES);']
    want = [f"size {C.sizeof(L.AdamwOpts)}", f"max {L.ADAMW_MAX_DECAY_RANGES}"]
    for f, _ in L.AdamwOpts._fields_:
        lines.append(f'printf("{f} %zu %zu\\n", offsetof(tome_adamw_opts_t, {f}), sizeof(((tome_adamw_opts_t*)0)->{f}));')
        want.append(f"{f} {getattr(L.AdamwOpts, f).offset} {getattr(L.AdamwOpts, f).size}")
    src = tmp_path / "s.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "include/tome_b200.h"\nint main(void) {\n' + "\n".join(lines) +
                   "\nreturn 0;\n}\n")
    exe = tmp_path / "s"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", f"-I{ROOT}", str(src), "-o", str(exe)], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    assert subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines() == want


def _opts(lib, **kw):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    ws = lib.tome_adamw_workspace_bytes(N)
    o = L.AdamwOpts(1.0, 1, None, 0, FAKE, FAKE, FAKE, ws)
    ranges = kw.pop("ranges", None)
    if ranges is not None:
        flat = [x for r in ranges for x in r]
        o.decay_ranges = (C.c_longlong * max(1, len(flat)))(*flat)
        o.n_decay_ranges = len(ranges)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


def _step(lib, opts, grad=FAKE):
    return lib.tome_adamw_step(N, FAKE, grad, FAKE, FAKE, FAKE, 1e-3, 0.9, 0.999, 1e-8, 0.1, 1.0, 1,
                               None if opts is None else C.byref(opts), None)


BAD_OPTS = [
    (dict(max_grad_norm=-1.0), b"max_grad_norm"),
    (dict(max_grad_norm=float("nan")), b"max_grad_norm"),
    (dict(max_grad_norm=float("inf")), b"max_grad_norm"),
    (dict(skip_nonfinite=2), b"skip_nonfinite must be"),
    (dict(steps=None), b"needs the steps"),                              # skipping without the counters
    (dict(ranges=[(10, 20), (5, 30)]), b"unsorted or overlaps"),
    (dict(ranges=[(10, 20), (19, 30)]), b"unsorted or overlaps"),
    (dict(ranges=[(-1, 20)]), b"unsorted or overlaps"),                  # below 0
    (dict(ranges=[(10, N + 1)]), b"outside"),
    (dict(ranges=[(10, 10)]), b"empty"),
    (dict(n_decay_ranges=-1), b"n_decay_ranges"),
    (dict(n_decay_ranges=513), b"n_decay_ranges"),
    (dict(n_decay_ranges=2), b"NULL decay_ranges"),
    (dict(workspace=None), b"workspace"),
    (dict(workspace_bytes=0), b"workspace"),
    (dict(workspace=C.c_void_p((1 << 20) + 4)), b"workspace"),           # misaligned
]


@pytest.mark.parametrize("kw,msg", BAD_OPTS)
def test_malformed_options_are_refused_before_any_cuda_call(lib, kw, msg):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    o = _opts(lib, **kw)
    assert _step(lib, o) == L.TOME_ERR_INVALID
    assert msg in lib.tome_last_error(), lib.tome_last_error()


def test_short_workspace_and_misaligned_grad_are_refused(lib):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    ws = lib.tome_adamw_workspace_bytes(N)
    assert ws >= 1024 * 4 and lib.tome_adamw_workspace_bytes(0) == 0
    assert _step(lib, _opts(lib, workspace_bytes=ws - 1)) == L.TOME_ERR_INVALID
    assert b"tome_adamw_workspace_bytes" in lib.tome_last_error()
    assert _step(lib, _opts(lib), grad=C.c_void_p((1 << 20) + 4)) == L.TOME_ERR_INVALID
    assert b"16-byte aligned" in lib.tome_last_error()
    # clipping alone needs the workspace too (the norm); a decay mask alone needs none
    assert _step(lib, _opts(lib, skip_nonfinite=0, steps=None, grad_norm=None, workspace=None)) == L.TOME_ERR_INVALID
    assert b"workspace" in lib.tome_last_error()
    # the legacy arguments are still checked with options
    assert lib.tome_adamw_step(N, FAKE, FAKE, FAKE, FAKE, FAKE, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1.0, 0, C.byref(_opts(lib)), None) \
        == L.TOME_ERR_INVALID


def _engine(monkeypatch, **kw):
    import torch
    from multi_modal_transformers_tokenmerge_b200 import engine
    monkeypatch.setattr(torch.cuda, "is_available", lambda: True)
    base = dict(batch=2, tokens=40, channels=64, heads=2, head_dim=32, mlp_dim=128, layers=3, r=2, num_groups=1, n_readout=2)
    base.update(kw)
    return engine.ToMeStackEngine(engine.StackConfig(**base), device="cpu")


HEADS = [dict(), dict(head="continuous", head_features=7), dict(head="categorical", head_groups=2, head_features=32),
         dict(head="diffusion", head_features=8, head_fourier_dim=32, head_time_hidden=64, head_time_out=32, head_hidden=128,
              diffusion_steps=20)]


@pytest.mark.parametrize("head", HEADS, ids=["none", "continuous", "categorical", "diffusion"])
def test_dense_kernel_ranges_cover_exactly_the_weight_matrices(lib, monkeypatch, head):
    """The mask marks every element of the named Dense kernels in param_views and nothing else: not LayerNorm, biases,
    pos_embedding or the diffusion Fourier kernel."""
    import torch
    eng = _engine(monkeypatch, **head)
    ranges = eng.decay_ranges("dense_kernels")
    assert all(a < b for a, b in ranges) and all(b <= c for (_, b), (c, _) in zip(ranges, ranges[1:]))
    assert len(ranges) <= 512
    mask = np.zeros(eng.n_params, bool)
    for a, b in ranges:
        mask[a:b] = True
    want = np.zeros(eng.n_params, bool)
    idx = torch.arange(eng.n_params, dtype=torch.float64)
    v = eng.param_views(idx)
    names = {"none": [], "continuous": ["kernel"], "categorical": ["kernel"], "diffusion": ["tw1", "tw2", "w1", "w2"]}[eng.cfg.head]
    for d in v["layers"]:
        for k in ("wqkv", "wo", "w1", "w2"):
            want[d[k].reshape(-1).long().numpy()] = True
    for k in names:
        want[v["head"][k].reshape(-1).long().numpy()] = True
    assert np.array_equal(mask, want)
    # what must never decay
    never = [v["pos_embedding"]] + [d[k] for d in v["layers"] for k in d if not k.startswith("w")]
    never += [t for k, t in v.get("head", {}).items() if k not in names]
    for t in never:
        assert not mask[t.reshape(-1).long().numpy()].any()
    assert eng.optimizer_steps() == (0, 0)
