"""CPU-only: the pixels-to-actions call of the C ABI (tome_policy_predict) -- struct layout against the header, workspace
arithmetic, malformed inputs refused before any CUDA call with a message naming the fault, and the sequence placement built
from the grammars."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAKE = 1 << 20   # a 256-byte aligned device pointer the validation must refuse before touching
OCTO_BASE_SEQ = "[TaskDescriptionPrefix{16}] [Image{25};Readout{4}]*2"    # octo_base.yaml:10, T = 74
NAMED_SEQ = "[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2"       # the named shape: 256 x 256 frames, T0 = 536


@pytest.fixture(scope="module")
def lib():
    from multi_modal_transformers_tokenmerge_b200 import _lib, build
    build.build()
    return _lib.lib()


def _struct_lines(name, cls):
    lines = [f'printf("{name} size %zu\\n", sizeof({name}));']
    want = [f"{name} size {C.sizeof(cls)}"]
    for f, _ in cls._fields_:
        lines.append(f'printf("{name}.{f} %zu %zu\\n", offsetof({name}, {f}), sizeof((({name}*)0)->{f}));')
        want.append(f"{name}.{f} {getattr(cls, f).offset} {getattr(cls, f).size}")
    return lines, want


def test_policy_structs_match_header(tmp_path):
    """tome_policy_rows_t / tome_policy_inputs_t as gcc lays them out in C99 equal the ctypes mirrors, field by field."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    lines, want = [], []
    for name, cls in (("tome_policy_rows_t", L.PolicyRows), ("tome_policy_inputs_t", L.PolicyInputs),
                      ("tome_image_tokenizer_desc_t", L.ImageTokenizerDesc)):
        a, b = _struct_lines(name, cls)
        lines += a
        want += b
    lines.append('printf("abi %d\\n", TOME_ABI_VERSION);')
    want.append(f"abi {L.ABI_VERSION}")
    src = tmp_path / "s.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "include/tome_b200.h"\nint main(void) {\n' + "\n".join(lines) +
                   "\nreturn 0;\n}\n")
    exe = tmp_path / "s"
    r = subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", f"-I{ROOT}", str(src), "-o", str(exe)], capture_output=True,
                       text=True)
    assert r.returncode == 0, r.stderr
    assert subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines() == want
    assert L.ABI_VERSION == 18


def _geometry(named: bool):
    """(grammar, image_size, patch_size): the named shape's or the gato geometry with octo_base.yaml's grammar."""
    return (NAMED_SEQ, 256, 16) if named else (OCTO_BASE_SEQ, 280, 56)


def _setup(B=4, named=False, head="continuous", layers=12, C_=768):
    """(cfg, inputs) of a well-formed call: octo-base widths, the gato geometry (or the named shape), uint8 frames, evaluation
    position tokens; every device pointer FAKE."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig
    from multi_modal_transformers_tokenmerge_b200.policy import placement
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence
    seq, image, patch = _geometry(named)
    ts = TokenSequence(seq)
    gid, _ = ts.group_ids()
    n_ro = ts.get_modality_idx("readouts").size
    kw = dict(head="continuous", head_features=7) if head == "continuous" else dict(
        head="diffusion", head_features=8, head_fourier_dim=64, head_time_hidden=64, head_time_out=64, head_hidden=256, diffusion_steps=32)
    cfg = StackConfig(batch=B, tokens=len(gid), channels=C_, heads=C_ // 64, head_dim=64, mlp_dim=4 * C_, layers=layers, r=4,
                      num_groups=int(gid.max()) + 1, n_readout=n_ro, **kw).c()
    np_ = (image // patch) ** 2
    rows, sets = placement(ts, 2 * np_)
    inp = L.PolicyInputs()
    inp.image = L.ImageTokenizerDesc(batch=B, n_images=2, image_size=image, channels_in=3, image_dtype=L.TOME_U8, normalize=1,
                                     patch_size=patch, conv_kernel=12, conv_stride=2, features=64, pool_window=3, num_blocks=2,
                                     num_groups=32, gn_eps=1e-6, embed_dim=C_, position_interval=128, token_rows=1,
                                     out_dtype=L.TOME_BF16, chunk_rows=0)
    inp.image_params_f32 = inp.image_params_bf16 = inp.pixels = inp.row_tokens = inp.col_tokens = FAKE
    inp._rows = (C.c_int * len(rows))(*[int(r) for r in rows])
    inp.image_rows = inp._rows
    inp.n_sets = len(sets)
    for i, (_, _, n, row) in enumerate(sets):
        inp.sets[i].rows, inp.sets[i].batch_stride, inp.sets[i].n, inp.sets[i].first_row = FAKE, 0, n, row
    return cfg, inp


def _call(lib, cfg, inp, ws_bytes=None):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    n = lib.tome_policy_predict_workspace_bytes(C.byref(cfg), C.byref(inp))
    io = L.StackIO()
    io.params_f32 = io.params_bf16 = io.gid = io.pos = io.allow = io.readout_idx = io.head_out = FAKE
    io.workspace = FAKE
    io.workspace_bytes = n if ws_bytes is None else ws_bytes
    return lib.tome_policy_predict(C.byref(cfg), C.byref(inp), C.byref(io), None, None)


@pytest.mark.parametrize("named", [False, True])
def test_workspace_overlaps_front_end_and_stack(lib, named):
    """sequence + max(front end, stack) <= workspace <= sequence + front end + stack, >= the larger of the two, and it grows with
    the sequence buffer (batch)."""
    last = 0
    for B in (1, 8, 64, 256):
        cfg, inp = _setup(B, named)
        ws = lib.tome_policy_predict_workspace_bytes(C.byref(cfg), C.byref(inp))
        it = lib.tome_image_tokenizer_workspace_bytes(C.byref(inp.image))
        st = lib.tome_stack_predict_workspace_bytes(C.byref(cfg))
        seq = B * cfg.tokens * cfg.channels * 2
        assert ws > 0 and it > 0 and st > 0, lib.tome_last_error()
        assert max(it, st) <= ws <= it + st + seq + 512, (ws, it, st, seq)
        assert ws >= seq + max(it, st)
        assert ws > last
        last = ws


BAD = [
    ("batch", lambda cfg, inp: setattr(inp.image, "batch", cfg.batch + 1), b"batch"),
    ("embed_dim", lambda cfg, inp: setattr(inp.image, "embed_dim", 512), b"embed_dim 512"),
    ("out_dtype", lambda cfg, inp: setattr(inp.image, "out_dtype", 1), b"out_dtype must be bf16"),
    ("row_high", lambda cfg, inp: inp.image_rows.__setitem__(3, cfg.tokens), b"outside the sequence"),
    ("row_negative", lambda cfg, inp: inp.image_rows.__setitem__(0, -1), b"outside the sequence"),
    ("row_twice", lambda cfg, inp: inp.image_rows.__setitem__(1, inp.image_rows[0]), b"covered twice"),
    ("set_overlaps_image", lambda cfg, inp: setattr(inp.sets[0], "n", inp.sets[0].n + 1), b"covered twice"),
    ("row_uncovered", lambda cfg, inp: setattr(inp, "n_sets", inp.n_sets - 1), b"covered by no image token and no set"),
    ("set_outside", lambda cfg, inp: setattr(inp.sets[inp.n_sets - 1], "first_row", cfg.tokens - 1), b"outside the sequence"),
    ("set_stride", lambda cfg, inp: setattr(inp.sets[0], "batch_stride", 8), b"batch_stride"),
    ("n_sets", lambda cfg, inp: setattr(inp, "n_sets", 17), b"n_sets"),
    ("no_rows", lambda cfg, inp: setattr(inp, "image_rows", None), b"image_rows missing"),
    ("front_end_shape", lambda cfg, inp: setattr(inp.image, "patch_size", 48), b"multiple of patch_size"),
]


@pytest.mark.parametrize("what,mutate,msg", BAD, ids=[b[0] for b in BAD])
def test_malformed_inputs_refused_before_any_cuda_call(lib, what, mutate, msg):
    """Every malformed input gives TOME_ERR_INVALID and a message naming the fault, from the size query and from the call.
    The pointers are fake and the machine may have no GPU: any CUDA call would fail with TOME_ERR_CUDA instead."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    cfg, inp = _setup()
    mutate(cfg, inp)
    assert lib.tome_policy_predict_workspace_bytes(C.byref(cfg), C.byref(inp)) == 0
    assert msg in lib.tome_last_error(), lib.tome_last_error()
    assert _call(lib, cfg, inp, ws_bytes=1 << 40) == L.TOME_ERR_INVALID
    assert msg in lib.tome_last_error(), lib.tome_last_error()


def test_workspace_and_pointer_checks(lib):
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    cfg, inp = _setup()
    n = lib.tome_policy_predict_workspace_bytes(C.byref(cfg), C.byref(inp))
    assert _call(lib, cfg, inp, ws_bytes=n - 1) == L.TOME_ERR_INVALID and b"workspace too small" in lib.tome_last_error()
    inp.sets[0].rows = FAKE + 8
    assert _call(lib, cfg, inp) == L.TOME_ERR_INVALID and b"16-byte aligned" in lib.tome_last_error()
    cfg, inp = _setup(head="diffusion")   # the diffusion head without the sampler's draws: the stack's own error
    assert _call(lib, cfg, inp) == L.TOME_ERR_INVALID and b"sampler's draws" in lib.tome_last_error()


@pytest.mark.parametrize("named", [False, True])
def test_placement_covers_every_row_once(named):
    """The tables built from octo_base.yaml's grammar (T = 74) and from the named shape's (T0 = 536) cover every row once, and
    put each token where TokenSequence.assemble_embeddings puts it."""
    import numpy as np

    from multi_modal_transformers_tokenmerge_b200.policy import placement
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenEmbeddings, TokenSequence
    seq, image, patch = _geometry(named)
    ts = TokenSequence(seq)
    T = ts.num_tokens
    assert T == (536 if named else 74)
    n_img = 2 * (image // patch) ** 2
    rows, sets = placement(ts, n_img)
    owner = np.zeros(T, np.int64)
    np.add.at(owner, rows, 1)
    for _, _, n, r0 in sets:
        owner[r0: r0 + n] += 1
    assert (owner == 1).all()
    # tag every input token with a distinct value and assemble both ways
    text = np.arange(16)[None, :, None] + 1000
    imgs = np.arange(n_img)[None, :, None] + 2000
    ro = np.arange(8)[None, :, None] + 3000
    want = ts.assemble_embeddings(TokenEmbeddings(text=text, images=imgs, readouts=ro))[0, :, 0]
    got = np.full(T, -1)
    got[rows] = imgs[0, :, 0]
    for m, a, n, r0 in sets:
        got[r0: r0 + n] = (text if m == "text" else ro)[0, a: a + n, 0]
    assert np.array_equal(got, want)
    with pytest.raises(ValueError):
        placement(ts, n_img + 1)
