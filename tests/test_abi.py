"""CPU-only: the C-ABI library builds for sm_100a, loads, and exports every symbol include/tome_b200.h declares.
No compute call is made (there is no GPU here); host-only entry points (shape arithmetic, validation) are exercised."""
import ctypes as C
import os
import re

import numpy as np

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "tome_b200.h")


@pytest.fixture(scope="module")
def lib():
    from multi_modal_transformers_tokenmerge_b200 import _lib, build
    build.build()
    return _lib.lib()


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(tome_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(lib):
    names = declared_symbols()
    assert len(names) >= 35, names
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in tome_b200.h but not exported: {missing}"


def test_abi_version_and_struct_sizes(lib):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    assert lib.tome_abi_version() == L.ABI_VERSION
    # field-by-field layout agreement with the C structs: test_ctypes_mirrors_match_header_layout; sizes are sane
    assert C.sizeof(L.GemmArgs) % 8 == 0 and C.sizeof(L.AttnDesc) % 8 == 0 and C.sizeof(L.StackCfg) % 8 == 0


def test_clamp_r_matches_reference_arithmetic(lib):
    # token_compression.py:60-67: r = min(r, (t - protected) // 2); r <= 0 -> nothing to merge
    for t in (2, 3, 10, 74, 75, 536):
        for r in (0, 1, 5, 16, 999):
            for cls in (0, 1):
                for dis in (0, 1):
                    assert lib.tome_clamp_r(t, r, cls, dis) == max(0, min(r, (t - cls - dis) // 2))


def test_stack_shape_arithmetic_on_host(lib):
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    cfg = StackConfig(batch=256, tokens=536, channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, r=16,
                      num_groups=5, n_readout=8).c()
    toks = [lib.tome_stack_tokens_at(C.byref(cfg), l) for l in range(13)]
    assert toks == [536 - 16 * l for l in range(13)]  # SURVEY 8d: 536, 520, ..., 360 -> 344
    n = lib.tome_stack_param_count(C.byref(cfg))
    c, hd, f = 384, 384, 1536
    per = 2 * c + c * 3 * hd + 3 * hd + hd * c + c + 2 * c + c * f + f + f * c + c
    assert n == 536 * c + 12 * per
    assert lib.tome_stack_layer_offset(C.byref(cfg), 0) == 536 * c
    assert lib.tome_stack_workspace_bytes(C.byref(cfg)) > 10 * 2**30  # saved activations of 12 layers at B=256
    bad = StackConfig(batch=1, tokens=8, channels=100, heads=1, head_dim=64, mlp_dim=64, layers=1).c()
    assert lib.tome_stack_param_count(C.byref(bad)) == -1
    assert b"multiples of 8" in lib.tome_last_error()


def test_action_head_shapes_on_host(lib):
    """Head descriptors are validated on the host, and a stack with a head carries the head's Dense kernel + bias at the
    end of the flat parameter vector (continuous.py:21 / categorical.py:38)."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    d = L.HeadDesc(256, 344, 384, L.TOME_BF16, 8, 1, 7, L.HEAD_CONTINUOUS_L2, 1.0)
    assert lib.tome_action_head_workspace_bytes(C.byref(d)) >= 256 * (384 + 7) * 4
    d = L.HeadDesc(4, 10, 32, L.TOME_BF16, 8, 3, 16, L.HEAD_CATEGORICAL_CE, 1.0)   # 8 readouts / 3 actions
    assert lib.tome_action_head_workspace_bytes(C.byref(d)) == 0 and b"do not split" in lib.tome_last_error()
    d = L.HeadDesc(4, 10, 32, L.TOME_BF16, 8, 2, 16, L.HEAD_CONTINUOUS_L2, 1.0)
    assert lib.tome_action_head_workspace_bytes(C.byref(d)) == 0 and b"groups must be 1" in lib.tome_last_error()
    base = dict(batch=8, tokens=74, channels=768, heads=12, head_dim=64, mlp_dim=3072, layers=2, r=4, num_groups=5, n_readout=8)
    n0 = lib.tome_stack_param_count(C.byref(StackConfig(**base).c()))
    assert lib.tome_stack_head_offset(C.byref(StackConfig(**base).c())) == -1
    cfg = StackConfig(**base, head="categorical", head_groups=8, head_features=256, max_action=1.0).c()
    assert lib.tome_stack_param_count(C.byref(cfg)) == n0 + 768 * 256 + 256
    assert lib.tome_stack_head_offset(C.byref(cfg)) == n0
    bad = StackConfig(**base, head="continuous", head_groups=2, head_features=7).c()
    assert lib.tome_stack_param_count(C.byref(bad)) == -1 and b"groups must be 1" in lib.tome_last_error()


def test_diffusion_head_shapes_on_host(lib):
    """diffusion.yaml's literal widths: parameter layout and its place at the end of the stack's flat vector."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    d = L.DiffusionDesc(8, 74, 768, 8, 8, 768, 768, 768, 768, 32)
    n = 384 + (768 * 768 + 768) * 2 + (8 + 768 + 768) * 768 + 768 + 768 * 8 + 8
    assert lib.tome_diffusion_head_param_count(C.byref(d)) == n
    assert lib.tome_diffusion_head_param_offset(C.byref(d), 0) == 0 and lib.tome_diffusion_head_param_offset(C.byref(d), 1) == 384
    assert lib.tome_diffusion_head_param_offset(C.byref(d), 9) == n
    assert lib.tome_diffusion_head_workspace_bytes(C.byref(d)) > 0
    bad = L.DiffusionDesc(8, 74, 768, 8, 7, 768, 768, 768, 768, 32)      # action_dim 7: rows of the concatenated input unaligned
    assert lib.tome_diffusion_head_param_count(C.byref(bad)) == -1 and b"action_dim" in lib.tome_last_error()
    base = dict(batch=8, tokens=74, channels=768, heads=12, head_dim=64, mlp_dim=3072, layers=1, num_groups=5, n_readout=8)
    n0 = lib.tome_stack_param_count(C.byref(StackConfig(**base).c()))
    cfg = StackConfig(**base, head="diffusion", head_features=8, head_fourier_dim=768, head_time_hidden=768, head_time_out=768,
                      head_hidden=768, diffusion_steps=32).c()
    assert lib.tome_stack_param_count(C.byref(cfg)) == n0 + n and lib.tome_stack_head_offset(C.byref(cfg)) == n0


def test_validation_errors_are_reported_not_thrown(lib):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    assert lib.tome_gemm_bf16(None, None, 0, None) == L.TOME_ERR_INVALID
    assert b"null args" in lib.tome_last_error()
    shp = L.MergeShape(1, 8, 6, 2, 0, L.TOME_BF16, L.TOME_MERGE_WAVG)  # channels not a multiple of 8
    plan = L.Plan(None, None, None, None, None)
    assert lib.tome_merge_fwd(C.byref(shp), C.byref(plan), None, None, None, None, None, None, None, None, None) == L.TOME_ERR_INVALID
    shp = L.MergeShape(1, 8, 8, 2, 0, L.TOME_BF16, 7)  # unknown mode (the reference only implements "sum")
    assert lib.tome_merge_fwd(C.byref(shp), C.byref(plan), None, None, None, None, None, None, None, None, None) == L.TOME_ERR_INVALID
    assert b"mode" in lib.tome_last_error()
    d = L.AttnDesc(1, 8, 1, 260, 0, 0, 0, 0, 0, 0, 0, 0, 1.0, None, None, None, 0, None)  # head_dim 260: not a multiple of 8
    assert lib.tome_attention_fwd(C.byref(d), None, None, None, None, None, None, 0, None) == L.TOME_ERR_UNSUPPORTED
    # tome_sim_argmax refuses these before any CUDA call, so the (16-byte aligned) fake device pointers are never touched
    fake = C.c_void_p(1 << 20)
    for dim, ws, ws_delta, msg in ((64, None, 0, b"tome_sim_argmax_workspace_bytes"),   # the workspace is required
                                   (64, fake, -1, b"tome_sim_argmax_workspace_bytes"),   # one byte short
                                   (48, fake, -1, b"tome_sim_argmax_workspace_bytes"),
                                   (298, fake, 0, b"metric dim")):                       # planes tiles exceed 227 KB of smem
        d = L.MetricDesc(2, 64, dim, 1, L.TOME_BF16, 64 * dim, dim, 0, 0, 0)
        ws_bytes = lib.tome_sim_argmax_workspace_bytes(C.byref(d)) + ws_delta
        assert lib.tome_sim_argmax(C.byref(d), fake, fake, fake, None, ws, ws_bytes, None) == L.TOME_ERR_INVALID, (dim, ws_delta)
        assert msg in lib.tome_last_error(), (dim, ws_delta, lib.tome_last_error())


def test_product_path_has_no_cpu_fallback():
    """The package must refuse CPU tensors loudly instead of computing on the host, and must not import oracle/."""
    import torch

    from multi_modal_transformers_tokenmerge_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.sim_argmax(torch.zeros(1, 4, 2))
    pkg = os.path.join(ROOT, "multi_modal_transformers_tokenmerge_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f"{f} imports the oracle"


def test_image_tokenizer_shapes_on_host(lib):
    """gato_resnet.yaml's literal geometry (280 x 280 x 3, 56-pixel patches, 12 x 12 / 2 convolution, 3 x 3 pool, 2 blocks of
    64 features, Dense 768, 128 position tokens): parameter layout, workspace, argument checks -- no GPU."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    d = L.ImageTokenizerDesc(batch=4, n_images=2, image_size=280, channels_in=3, image_dtype=L.TOME_U8, normalize=1, patch_size=56,
                             conv_kernel=12, conv_stride=2, features=64, pool_window=3, num_blocks=2, num_groups=32, gn_eps=1e-6,
                             embed_dim=768, position_interval=128, token_rows=1, out_dtype=L.TOME_BF16)
    conv0 = 12 * 12 * 3 * 64 + 64
    block = 64 + 64 + 9 * 64 * 64 + 64
    kd = 21 * 21 * 64                                   # (56 - 12) / 2 + 1 = 23 -> pool -> 21
    n = conv0 + 2 * block + kd * 768 + 768 + 2 * 128 * 768
    assert lib.tome_image_tokenizer_param_count(C.byref(d)) == n
    off = lambda w: lib.tome_image_tokenizer_param_offset(C.byref(d), w)  # noqa: E731
    assert off(L.IT_CONV0_KERNEL) == 0 and off(L.IT_CONV0_BIAS) == conv0 - 64
    assert off(L.IT_BLOCK0) == conv0 and off(L.IT_BLOCK0 + 2) == conv0 + 128 and off(L.IT_BLOCK0 + 4) == conv0 + block
    assert off(L.IT_DENSE_KERNEL) == conv0 + 2 * block and off(L.IT_COL_EMBED) == n - 128 * 768
    assert off(L.IT_BLOCK0 + 8) == -1 and b"no parameter" in lib.tome_last_error()
    ws = lib.tome_image_tokenizer_workspace_bytes(C.byref(d))
    assert ws >= 2 * 4 * 2 * 25 * 23 * 23 * 432          # at least the input convolution's im2col rows of the 4 batch rows
    # every buffer of a pass at its size: im2col rows and output of the input convolution, four bordered (23 x 23) activation
    # buffers, the Dense output (an undersized one here once let a kernel write into its neighbour)
    n_patch = 4 * 2 * 25
    assert ws >= n_patch * (529 * 432 * 2 + 529 * 64 * 2 + 4 * 529 * 64 * 2 + 768 * 4)
    d.batch = 4096                                       # the workspace is per chunk of batch rows, not per batch
    assert lib.tome_image_tokenizer_workspace_bytes(C.byref(d)) < (3 << 30)
    for field, value, msg in (("patch_size", 57, b"multiple of patch_size"), ("features", 60, b"multiple of 8"),
                              ("num_groups", 7, b"num_groups"), ("token_rows", 3, b"token_rows"), ("pool_window", 30, b"pool")):
        bad = L.ImageTokenizerDesc.from_buffer_copy(d)
        setattr(bad, field, value)
        assert lib.tome_image_tokenizer_param_count(C.byref(bad)) == -1 and msg in lib.tome_last_error(), field


def test_pruning_stack_shapes_on_host(lib):
    """tome_stack_cfg_t.prune_*: token counts per layer follow the compression grammar (n - layer * c), the argument checks
    name what is wrong -- no GPU."""
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence
    ts = TokenSequence("[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2", "[TaskDescriptionPrefix{0}] [Image{8};Readout{0}]*2")
    sets = ts.prune_sets()
    assert sets == [(16, 0), (256, 8), (4, 0), (256, 8), (4, 0)]
    g3, p3 = ts.layer_group_ids(3)
    assert g3.shape == (536 - 48,) and list(np.bincount(g3)) == [16, 232, 4, 232, 4] and p3[16 + 231] == 231
    base = dict(batch=2, tokens=536, channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, prop_attn=False, num_groups=5, n_readout=8)
    cfg = StackConfig(**base, prune_sets=tuple(sets)).c()
    assert [lib.tome_stack_tokens_at(C.byref(cfg), l) for l in (0, 1, 12)] == [536, 520, 344]
    assert lib.tome_stack_workspace_bytes(C.byref(cfg)) > 0
    for kw, msg in ((dict(prune_sets=tuple(sets), r=4), b"r = 0"), (dict(prune_sets=((16, 0), (256, 30), (4, 0), (256, 8), (4, 0))), b"cannot drop"),
                    (dict(prune_sets=((16, 0), (256, 8))), b"token sets hold")):
        b2 = dict(base)
        b2.update(kw)
        bad = StackConfig(**b2).c()
        assert lib.tome_stack_param_count(C.byref(bad)) == -1 and msg in lib.tome_last_error(), kw


def test_header_is_plain_c(tmp_path):
    """include/tome_b200.h is the drop-in boundary: it must compile as C99 on its own (no C++, no CUDA, no torch types)."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = tmp_path / "h.c"
    src.write_text('#include "include/tome_b200.h"\nint main(void) { tome_gemm_args_t g; tome_stack_cfg_t c; tome_image_tokenizer_desc_t d; '
                   '(void)g; (void)c; (void)d; return TOME_ABI_VERSION > 0 ? 0 : 1; }\n')
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", f"-I{root}", str(src)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_ctypes_mirrors_match_header_layout(tmp_path):
    """Every struct _lib.py mirrors has the header's size, and every mirrored field the header's offset and size, as gcc
    lays them out (a field that moves into or out of padding changes no size, so behaviour alone would not show it)."""
    import shutil
    import subprocess
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    mirrors = {"tome_metric_desc_t": L.MetricDesc, "tome_plan_t": L.Plan, "tome_plan_shape_t": L.PlanShape,
               "tome_prune_desc_t": L.PruneDesc, "tome_merge_shape_t": L.MergeShape, "tome_gemm_args_t": L.GemmArgs,
               "tome_attn_desc_t": L.AttnDesc, "tome_attn_grad_strides_t": L.AttnGradStrides, "tome_stack_cfg_t": L.StackCfg,
               "tome_diffusion_desc_t": L.DiffusionDesc, "tome_image_tokenizer_desc_t": L.ImageTokenizerDesc,
               "tome_head_desc_t": L.HeadDesc, "tome_stack_io_t": L.StackIO}
    lines, want = [], []
    for cname, cls in mirrors.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        want.append(f"{cname} {C.sizeof(cls)}")
        for fname, _ in cls._fields_:
            lines.append(f'printf("{cname}.{fname} %zu %zu\\n", offsetof({cname}, {fname}), sizeof((({cname}*)0)->{fname}));')
            f = getattr(cls, fname)
            want.append(f"{cname}.{fname} {f.offset} {f.size}")
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "include/tome_b200.h"\nint main(void) {\n' + "\n".join(lines) +
                   "\nreturn 0;\n}\n")
    exe = tmp_path / "layout"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", f"-I{ROOT}", str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines()
    assert got == want
