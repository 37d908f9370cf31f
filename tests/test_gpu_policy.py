"""Pixels to actions in one native call (tome_policy_predict via ToMeStackEngine.policy / PixelPolicy) on the GPU.  Needs a
B200: `-m gpu`.

Parity protocol: the fused call runs the front end's kernels with its last stage writing into the sequence rows, a bit copy of
the text / readout rows, then the forward-only stack; so its outputs must equal the composed Python path
(ImageTokenizer.apply -> TokenSequence.assemble_embeddings -> predictor().predict) bit for bit."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenEmbeddings, TokenSequence  # noqa: E402

GEOMETRY = {   # grammar, compression grammar (pruning / set-merging stacks), frame side, patch side, width
    "gato": ("[TaskDescriptionPrefix{16}] [Image{25};Readout{4}]*2", "[TaskDescriptionPrefix{0}] [Image{2};Readout{0}]*2", 280, 56, 768),
    "named": ("[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2", "[TaskDescriptionPrefix{0}] [Image{8};Readout{0}]*2", 256, 16, 384),
}


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from multi_modal_transformers_tokenmerge_b200 import _lib, engine
    _lib.lib()
    return engine


def _tokenizer(geo, chunk_rows=0):
    from multi_modal_transformers_tokenmerge_b200 import model_configs
    _, _, image, patch, C = GEOMETRY[geo]
    node = dict(model_configs.load("tokenizers/images/gato_resnet_octo")["encoder"])
    node.update(image_size=[image, image, 3], patch_size=patch, embedding_dim=C)
    for k in ("row_position_embedding", "col_position_embedding"):
        node[k] = dict(node[k], features=C)
    node["resnet"] = dict(node["resnet"], output_dense=dict(node["resnet"]["output_dense"], features=C))
    tok = model_configs.build_image_tokenizer(node, chunk_rows=chunk_rows)
    return tok, tok.init(5, None)


def _engine(engine, geo, kind, head, B=4, layers=4):
    seq, comp, _, _, C = GEOMETRY[geo]
    ts = TokenSequence(seq, comp)
    gid, pos = ts.group_ids()
    allow, ro = ts.allow_table(), ts.get_modality_idx("readouts")
    cfg = dict(batch=B, tokens=ts.num_tokens, channels=C, heads=C // 64, head_dim=64, mlp_dim=4 * C, layers=layers, r=4, ln_axis=1,
               num_groups=allow.shape[0], n_readout=len(ro))
    if kind == "set_merge":
        cfg.update(r=0, prune_sets=tuple(ts.prune_sets()), set_merge=True)
    elif kind == "prune":
        cfg.update(r=0, prune_sets=tuple(ts.prune_sets()), prop_attn=False)
    cfg.update({"continuous": dict(head="continuous", head_features=7, max_action=1.0),
                "categorical": dict(head="categorical", head_groups=4, head_features=16, max_action=1.0),
                "diffusion": dict(head="diffusion", head_features=8, head_fourier_dim=64, head_time_hidden=64, head_time_out=64,
                                  head_hidden=256, diffusion_steps=32)}[head])
    eng = engine.ToMeStackEngine(engine.StackConfig(**cfg), gid=gid, pos=pos, allow=allow, readout_idx=ro)
    eng.init_params(seed=3)
    return eng, TokenSequence(seq)


def _inputs(geo, B, pixels, seed, bcast=False):
    _, _, image, _, C = GEOMETRY[geo]
    g = torch.Generator(device="cuda").manual_seed(seed)
    if pixels == "u8":
        frames = torch.randint(0, 256, (B, 2, image, image, 3), dtype=torch.uint8, device="cuda", generator=g)
    else:
        frames = torch.rand(B, 2, image, image, 3, device="cuda", generator=g) * 255.0
    text = torch.randn(B, 16, C, device="cuda", generator=g).bfloat16()
    readouts = torch.randn(1 if bcast else B, 8, C, device="cuda", generator=g).bfloat16()
    return frames, text, readouts


def _composed(eng, B, tok, tvars, ts, frames, text, readouts, rng):
    """ImageTokenizer.apply -> assemble_embeddings -> predictor().predict: the path the fused call replaces."""
    C = eng.cfg.channels
    img = tok.apply(tvars, frames, train=False).reshape(B, -1, C)
    x = ts.assemble_embeddings(TokenEmbeddings(text=text, images=img, readouts=readouts.expand(B, -1, -1))).contiguous()
    return eng.predictor(B).predict(x, rng=rng)


def _equal(a, b):
    return (a is None and b is None) or (a is not None and b is not None and torch.equal(a, b))


@pytest.mark.parametrize("geo,B,head,pixels,kind,bcast,chunk_rows", [
    ("gato", 1, "continuous", "u8", "merge", False, 0),
    ("gato", 256, "categorical", "f32", "merge", True, 0),       # 256 rows: the front end runs six chunks of whole rows
    ("gato", 8, "diffusion", "u8", "prune", False, 0),
    ("gato", 8, "continuous", "f32", "set_merge", True, 3),      # three chunks at a small batch
    ("named", 1, "diffusion", "f32", "set_merge", True, 0),
    ("named", 256, "continuous", "u8", "merge", False, 0),
    ("named", 4, "categorical", "u8", "prune", True, 0),
])
def test_policy_equals_composed_path_bitwise(pkg, geo, B, head, pixels, kind, bcast, chunk_rows):
    engine = pkg
    tok, tvars = _tokenizer(geo, chunk_rows)
    eng, ts = _engine(engine, geo, kind, head)
    pol = eng.policy(tok, tvars, ts, batch=B)
    frames, text, readouts = _inputs(geo, B, pixels, seed=B)
    out, ro = pol.predict(frames, text, readouts, rng=9)
    want_out, want_ro = _composed(eng, B, tok, tvars, ts, frames, text, readouts, rng=9)
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
    assert torch.equal(out, want_out), (geo, B, head, (out - want_out).abs().max().item())
    assert _equal(ro, want_ro)


def test_broadcast_readouts_equal_expanded(pkg):
    """Readout rows given once (batch stride 0) equal the same rows expanded to [B, n, C]."""
    engine = pkg
    tok, tvars = _tokenizer("gato")
    eng, ts = _engine(engine, "gato", "merge", "continuous")
    pol = eng.policy(tok, tvars, ts, batch=6)
    frames, text, readouts = _inputs("gato", 6, "u8", seed=4, bcast=True)
    a = pol.predict(frames, text, readouts)
    b = pol.predict(frames, text, readouts.expand(6, -1, -1).contiguous())
    c = pol.predict(frames, text, readouts[0])
    torch.cuda.synchronize()
    assert all(torch.equal(x, y) and torch.equal(x, z) for x, y, z in zip(a, b, c))


@pytest.mark.parametrize("geo,head", [("gato", "diffusion"), ("named", "continuous")])
def test_graph_replay_equals_eager(pkg, geo, head):
    """graph=True: the first call eager, the rest replayed; over several calls with new frames, text, readouts and sampler draws
    each equals an eager policy's output bit for bit."""
    engine = pkg
    tok, tvars = _tokenizer(geo)
    eng, ts = _engine(engine, geo, "merge", head)
    B = 2
    eager = eng.policy(tok, tvars, ts, batch=B)
    graphed = eng.policy(tok, tvars, ts, batch=B, graph=True)
    outs = []
    for i in range(4):
        frames, text, readouts = _inputs(geo, B, "u8", seed=20 + i)
        got = graphed.predict(frames, text, readouts, rng=i)
        want = eager.predict(frames, text, readouts, rng=i)
        outs.append(got[0])
        torch.cuda.synchronize()
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), i
    assert graphed._graph is not None
    assert not torch.equal(outs[0], outs[1])


def test_policy_sees_adamw_step(pkg):
    """A policy built before an AdamW step of the training engine predicts with the stepped parameters: equal to the composed
    path after the step, and different from its own output before it."""
    engine = pkg
    tok, tvars = _tokenizer("gato")
    eng, ts = _engine(engine, "gato", "merge", "continuous", B=4)
    pol = eng.policy(tok, tvars, ts)
    frames, text, readouts = _inputs("gato", 4, "u8", seed=7)
    before = pol.predict(frames, text, readouts)[0]
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(4, eng.cfg.tokens, eng.cfg.channels, device="cuda", generator=g).bfloat16()
    eng.zero_grad()
    eng.forward(x, torch.rand(4, 7, device="cuda", generator=g) * 2 - 1)
    eng.backward()
    eng.adamw_step(lr=1e-3)
    after, ro = pol.predict(frames, text, readouts)
    want, want_ro = _composed(eng, 4, tok, tvars, ts, frames, text, readouts, rng=0)
    torch.cuda.synchronize()
    assert torch.equal(after, want) and torch.equal(ro, want_ro)
    assert not torch.equal(after, before)
