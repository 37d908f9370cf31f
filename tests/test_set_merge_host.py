"""Matching inside token sets, host side (no GPU): the C ABI refuses malformed set tables before any CUDA call, the stack's
set-merging configuration is checked, tokenset_soft_matching checks its arguments, and the ctypes mirror of
tome_token_sets_t matches the header."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from multi_modal_transformers_tokenmerge_b200 import _lib
    return _lib.lib()


def _sets(rows):
    from multi_modal_transformers_tokenmerge_b200 import ops
    return ops.token_sets(rows)


BAD_TABLES = [
    ([(0, 10, 2), (9, 10, 2)], b"starts at 9"),            # overlap
    ([(0, 10, 2), (11, 9, 2)], b"starts at 11"),           # gap
    ([(0, 10, 6), (10, 10, 0)], b"out of range"),          # r > n / 2
    ([(0, 10, -1), (10, 10, 1)], b"out of range"),         # r < 0
    ([(0, 10, 2), (10, 8, 2)], b"cover 18 tokens"),        # does not cover the sequence
    ([(0, 0, 0), (0, 20, 2)], b"empty"),
]


@pytest.mark.parametrize("rows,msg", BAD_TABLES)
def test_bad_set_tables_are_refused_before_any_cuda_call(lib, rows, msg):
    """T = 20 tokens.  The fake (16-byte aligned) device pointers are never touched: every entry point returns
    TOME_ERR_INVALID while validating."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    ts = _sets(rows)
    sp = C.cast(C.pointer(ts), C.c_void_p)
    fake = C.c_void_p(1 << 20)
    d = L.MetricDesc(2, 20, 64, 1, L.TOME_BF16, 20 * 64, 64, 0, 0, 0, sp)
    ws = lib.tome_sim_argmax_workspace_bytes(C.byref(d))
    assert lib.tome_sim_argmax(C.byref(d), fake, fake, fake, None, fake, ws, None) == L.TOME_ERR_INVALID
    assert msg in lib.tome_last_error(), lib.tome_last_error()
    r = sum(max(v[2], 0) for v in rows) or 1
    plan = L.Plan(fake, fake, fake, fake, fake)
    ps = L.PlanShape(2, 20, r, 0, sp)
    assert lib.tome_select_topr(C.byref(ps), fake, fake, C.byref(plan), None) == L.TOME_ERR_INVALID
    assert msg in lib.tome_last_error(), lib.tome_last_error()
    ms = L.MergeShape(2, 20, 64, r, 0, L.TOME_BF16, L.TOME_MERGE_WAVG, sp)
    assert lib.tome_merge_fwd(C.byref(ms), C.byref(plan), fake, None, fake, fake, None, None, None, None, None) == L.TOME_ERR_INVALID
    assert msg in lib.tome_last_error(), lib.tome_last_error()
    assert lib.tome_merge_bwd(C.byref(ms), C.byref(plan), None, fake, fake, fake, None) == L.TOME_ERR_INVALID
    assert msg in lib.tome_last_error(), lib.tome_last_error()


def test_sets_with_class_or_distill_token_or_wrong_r_total_are_refused(lib):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    ts = _sets([(0, 10, 2), (10, 10, 3)])
    sp = C.cast(C.pointer(ts), C.c_void_p)
    fake = C.c_void_p(1 << 20)
    for cls, dist in ((1, 0), (0, 1)):
        d = L.MetricDesc(2, 20, 48, 1, L.TOME_F32, 20 * 48, 48, 0, cls, dist, sp)
        ws = lib.tome_sim_argmax_workspace_bytes(C.byref(d))
        assert lib.tome_sim_argmax(C.byref(d), fake, fake, fake, None, fake, ws, None) == L.TOME_ERR_INVALID
        assert b"class or distill" in lib.tome_last_error()
    plan = L.Plan(fake, fake, fake, fake, fake)
    ps = L.PlanShape(2, 20, 5, 1, sp)
    assert lib.tome_select_topr(C.byref(ps), fake, fake, C.byref(plan), None) == L.TOME_ERR_INVALID
    assert b"class or distill" in lib.tome_last_error()
    ps = L.PlanShape(2, 20, 4, 0, sp)                  # r must be the sum of the sets' r (5)
    assert lib.tome_select_topr(C.byref(ps), fake, fake, C.byref(plan), None) == L.TOME_ERR_INVALID
    assert b"sum of the sets" in lib.tome_last_error()
    # the workspace does not depend on the sets: even + odd tokens are the sequence either way
    d0 = L.MetricDesc(2, 20, 64, 1, L.TOME_BF16, 20 * 64, 64, 0, 0, 0, None)
    d1 = L.MetricDesc(2, 20, 64, 1, L.TOME_BF16, 20 * 64, 64, 0, 0, 0, sp)
    assert lib.tome_sim_argmax_workspace_bytes(C.byref(d0)) == lib.tome_sim_argmax_workspace_bytes(C.byref(d1)) > 0


def test_set_merging_stack_config(lib):
    """tome_stack_cfg_t.set_merge: token counts follow n - l c like the pruning path; r != 0, c > floor(n(l) / 2) at some
    layer, a class token and layer_gid / layer_pos are refused."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    sets = ((16, 0), (256, 8), (4, 0), (256, 8), (4, 0))
    base = dict(batch=2, tokens=536, channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, num_groups=5, n_readout=8)
    cfg = StackConfig(**base, prune_sets=sets, set_merge=True)
    c = cfg.c()
    assert [lib.tome_stack_tokens_at(C.byref(c), l) for l in (0, 1, 12)] == [536, 520, 344]
    assert lib.tome_stack_workspace_bytes(C.byref(c)) > 0
    assert cfg.layer_sets(2) == ((0, 16, 0), (16, 240, 8), (256, 4, 0), (260, 240, 8), (500, 4, 0))
    for kw, msg in ((dict(r=4), b"r = 0"), (dict(class_token=True), b"class / distill"),
                    (dict(prune_sets=((16, 0), (40, 8), (4, 0), (472, 8), (4, 0)), layers=5), b"cannot merge"),   # 8 tokens at layer 4
                    (dict(prune_sets=()), b"set_merge needs")):
        b2 = dict(base, prune_sets=sets, set_merge=True)
        b2.update(kw)
        bad = StackConfig(**b2).c()
        assert lib.tome_stack_param_count(C.byref(bad)) == -1 and msg in lib.tome_last_error(), kw
    # c = floor(n / 2) at the last layer is allowed: 40 - 3 * 8 = 16 tokens merge 8
    ok = StackConfig(**dict(base, prune_sets=((16, 0), (40, 8), (4, 0), (472, 8), (4, 0)), layers=4, set_merge=True)).c()
    assert lib.tome_stack_param_count(C.byref(ok)) > 0
    # layer_gid / layer_pos stay pruning-only: refused before anything is launched (fake, aligned workspace)
    ws = lib.tome_stack_workspace_bytes(C.byref(c))
    fake = 1 << 20
    io = L.StackIO(params_f32=fake, params_bf16=fake, x=fake, x_dtype=L.TOME_BF16, gid=fake, pos=fake, allow=fake, readout_idx=fake,
                   workspace=fake, workspace_bytes=ws, loss=fake, layer_gid=fake, layer_pos=fake)
    c.num_groups = 5
    assert lib.tome_stack_forward(C.byref(c), C.byref(io), None) == L.TOME_ERR_INVALID
    assert b"layer_gid" in lib.tome_last_error()


def test_tokenset_soft_matching_argument_checks():
    import torch

    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_compression import tokenset_soft_matching
    m = torch.zeros(2, 20, 8)
    for idx, rs, msg in (([(0, 10), (10, 10)], [1], "one entry per token set"),
                         ([(0, 10), (9, 11)], [1, 1], "consecutive"),
                         ([(0, 10), (10, 10)], [6, 1], "out of range"),
                         ([(0, 10), (10, 8)], [1, 1], "cover 18 tokens"),
                         ([(i, 1) for i in range(17)], [0] * 17, "between 1 and 16")):
        with pytest.raises(ValueError, match=msg):
            tokenset_soft_matching(m, idx, rs)
    with pytest.raises(ValueError, match="batch, tokens, dim"):
        tokenset_soft_matching(torch.zeros(20, 8), [(0, 20)], [2])
    with pytest.raises(RuntimeError, match="no CPU fallback"):       # valid arguments reach the kernels: CUDA only
        tokenset_soft_matching(m, [(0, 10), (10, 10)], [2, 0])
    # all r = 0: the identity merge, as bipartite_soft_matching with r = 0
    assert tokenset_soft_matching(m, [(0, 10), (10, 10)], [0, 0]).r == 0


def test_token_sets_mirror_matches_header_layout(tmp_path):
    """tome_token_sets_t and the `sets` fields it adds to the metric / plan / merge descriptors, as gcc lays them out."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    mirrors = {"tome_token_sets_t": L.TokenSets, "tome_metric_desc_t": L.MetricDesc, "tome_plan_shape_t": L.PlanShape,
               "tome_merge_shape_t": L.MergeShape, "tome_stack_cfg_t": L.StackCfg}
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
    assert "sets" in dict(L.MetricDesc._fields_) and "set_merge" in dict(L.StackCfg._fields_)


def test_oracle_set_merge_is_per_set_merge_wavg():
    """The checker restatement: a set table of one set is oracle.merge_wavg itself; r = 0 sets are copied."""
    from oracle import tome_oracle as O
    from set_merge_oracle import set_merge_wavg, set_plans, set_row_map
    rng = np.random.default_rng(0)
    m, x = rng.standard_normal((2, 30, 8)).astype(np.float32), rng.standard_normal((2, 30, 4)).astype(np.float32)
    one = [(0, 30, 6)]
    xo, so = set_merge_wavg(set_plans(m, one), one, x)
    want = O.merge_wavg(O.bipartite_soft_matching(m, 6), x)
    assert np.array_equal(xo, want[0]) and np.array_equal(so, want[1])
    sets = [(0, 11, 3), (11, 4, 0), (15, 15, 7)]
    plans = set_plans(m, sets)
    xo, _ = set_merge_wavg(plans, sets, x)
    rm = set_row_map(plans, sets, 2)
    assert xo.shape == (2, 20, 4) and np.array_equal(xo[:, 8:12], x[:, 11:15])
    assert rm[:, :11].max() < 8 and (rm[:, 15:] >= 12).all() and np.array_equal(rm[:, 11:15], np.broadcast_to(np.arange(8, 12), (2, 4)))
