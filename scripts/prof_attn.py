"""One attention forward + backward at the bench's layer-0 shape, for ncu captures.  python scripts/prof_attn.py [T] [H] [B]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200 import ops  # noqa: E402
from bench_kernels import attn_inputs as inputs  # noqa: E402

T = int(sys.argv[1]) if len(sys.argv) > 1 else 536
H = int(sys.argv[2]) if len(sys.argv) > 2 else 6
B = int(sys.argv[3]) if len(sys.argv) > 3 else 256
q, k, v, kw = inputs(B, T, H)
drop = dict(dropout_rate=0.1, dropout_seed=3, dropout_site=5)
for _ in range(3):
    out, lse = ops.attention_fwd(q, k, v, **kw, **drop)
    do = torch.randn_like(out)
    g = ops.attention_bwd(q, k, v, out, lse, do, **kw, **drop)
torch.cuda.synchronize()
print("ok", float(out.float().abs().mean()), float(g[0].float().abs().mean()))
