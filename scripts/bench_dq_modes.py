"""Backward attention with dQ from stored dS^T tiles (mode 1) against the recomputing dQ kernel (mode 0) at several lengths."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200 import _lib, ops  # noqa: E402

setter = _lib.lib().tome_attention_set_dq_from_ds
for B, T, H in ((256, 536, 6), (32, 2080, 12), (20, 3072, 12), (16, 4096, 12), (8, 6144, 12)):
    qkv = torch.randn(B, T, 3, H, 64, device="cuda").bfloat16()
    q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
    o, l = ops.attention_fwd(q, k, v)
    do = torch.randn(B, T, H, 64, device="cuda").bfloat16()
    res = []
    for mode in (0, 1):
        setter(mode)
        for _ in range(3):
            ops.attention_bwd(q, k, v, o, l, do)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            ops.attention_bwd(q, k, v, o, l, do)
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) * 100)
    setter(-1)
    print(f"B{B} T{T} H{H}: recompute {res[0]:.0f} us, from dS^T {res[1]:.0f} us")
