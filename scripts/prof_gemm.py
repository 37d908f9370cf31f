"""One GEMM shape, a few launches, for ncu:  python scripts/prof_gemm.py M N K B_MN [bias]"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200 import ops
m, n, k, bmn = [int(v) for v in sys.argv[1:5]]
a = torch.randn(m, k, device="cuda").bfloat16()
b = (torch.randn(k, n, device="cuda") if bmn else torch.randn(n, k, device="cuda")).bfloat16()
out = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
kw = {}
if len(sys.argv) > 5:
    kw["bias"] = torch.randn(n, device="cuda")
for _ in range(3):
    ops.gemm(a, b, m=m, n=n, k=k, b_major=bmn, out=out, **kw)
torch.cuda.synchronize()
print("ok")
