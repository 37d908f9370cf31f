"""Attention backward at the bench shapes (masked + weight dropout), CUDA events, L2 flushed.  python scripts/bench_attn_bwd.py"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200 import ops
from bench_kernels import attn_inputs as inputs, timeit
drop = dict(dropout_rate=0.1, dropout_seed=3, dropout_site=5)
for (B, T, H) in [(256, 536, 6), (256, 440, 6), (256, 392, 6), (256, 536, 12)]:
    q, k, v, kw = inputs(B, T, H)
    out, lse = ops.attention_fwd(q, k, v, **kw, **drop)
    do = torch.randn_like(out)
    part = torch.empty(B * ((T + 127) // 128), 3 * H * 64, device="cuda")
    tf = timeit(lambda: ops.attention_fwd(q, k, v, **kw, **drop), iters=5)
    tb = timeit(lambda: ops.attention_bwd(q, k, v, out, lse, do, bias_partial=part, **kw, **drop), iters=5)
    print(f"B{B} T{T} H{H}: fwd {tf*1e6:7.1f} us  bwd {tb*1e6:7.1f} us")
