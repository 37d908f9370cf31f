"""Attention backward at the bench shape with the dS^T store on / off (for ncu --metrics gpu__time_duration.sum)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200 import ops, _lib
from bench_kernels import attn_inputs as inputs
q, k, v, kw = inputs(256, 536, 6)
drop = dict(dropout_rate=0.1, dropout_seed=3, dropout_site=5)
out, lse = ops.attention_fwd(q, k, v, **kw, **drop)
do = torch.randn_like(out)
setter = _lib.lib().tome_attention_set_dq_from_ds
for mode in (1, 0, 1, 0):
    setter(mode)
    ops.attention_bwd(q, k, v, out, lse, do, **kw, **drop)
torch.cuda.synchronize()
print("ok")
