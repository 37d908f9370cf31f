"""Per-kernel microbenchmarks (CUDA events, L2 flushed between timed launches).  Development tool; the contract
benchmark is bench.py.   python scripts/bench_kernels.py [merge|gemm|attn|ln|match ...]"""
import json
import math
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200 import ops  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import sequence_groups  # noqa: E402

PEAKS = json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json"))) if os.path.exists(
    os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}
_flush = None


def timeit(fn, iters=10, warmup=3, flush=True):
    global _flush
    if _flush is None:
        _flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        if flush:
            _flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        torch.cuda.synchronize()
        tot += s.elapsed_time(e)
    return tot / iters * 1e-3


def attn_inputs(B, T, H):
    """q, k, v of B x T x H heads of 64 and the stack's block-causal group mask in a scrambled token order (as after a merge)."""
    qkv = torch.randn(B, T, 3, H, 64, device="cuda").bfloat16()
    n_img = (T - 16) // 2 - 4
    g1, p1, allow, _ = sequence_groups(f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2")
    rng = np.random.default_rng(0)
    kw = dict(size=torch.ones(B, T, device="cuda"), gid=torch.tensor(np.stack([rng.permutation(g1) for _ in range(B)])).cuda(),
              pos=torch.tensor(np.broadcast_to(p1, (B, len(g1))).copy()).cuda(), allow=torch.tensor(allow).cuda())
    return qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2], kw


def bench_merge():
    for (B, T, C, r) in [(256, 536, 384, 16), (256, 536, 768, 32), (32, 4096, 1024, 1024), (16, 8192, 768, 2048), (128, 1024, 768, 128)]:
        x = torch.randn(B, T, C, device="cuda").bfloat16()
        metric = torch.randn(B, T, 64, device="cuda")
        nm, ni, _ = ops.sim_argmax(metric)
        plan = ops.select_topr(nm, ni, T, r)
        size = torch.ones(B, T, device="cuda")
        ta = (T + 1) // 2
        by = B * (T * C * 2 + 4 * T + 4 * (ta + r) + (T - r) * C * 2 + 4 * (T - r))
        t = timeit(lambda: ops.merge_fwd(plan, x, size, 1))
        print(f"merge_fwd  B{B} T{T} C{C} r{r}: {t*1e6:8.1f} us  {by/t/1e9:7.1f} GB/s  frac {by/t/1e9/PEAKS['hbm_gbs']:.3f}")
        size2 = torch.randint(1, 4, (B, T), device="cuda").float()   # sizes != 1: every row takes the arithmetic path
        t = timeit(lambda: ops.merge_fwd(plan, x, size2, 1))
        print(f"merge_fwd  (all rows patched) : {t*1e6:8.1f} us  {by/t/1e9:7.1f} GB/s  frac {by/t/1e9/PEAKS['hbm_gbs']:.3f}")
        x1, s1, _, _ = ops.merge_fwd(plan, x, size, 1)
        dy = torch.randn_like(x1)
        by2 = B * ((T - r) * C * 2 + T * C * 2 + 4 * T)
        t = timeit(lambda: ops.merge_bwd(plan, dy, size, s1, 1))
        print(f"merge_bwd  B{B} T{T} C{C} r{r}: {t*1e6:8.1f} us  {by2/t/1e9:7.1f} GB/s  frac {by2/t/1e9/PEAKS['hbm_gbs']:.3f}")
        t = timeit(lambda: ops.sim_argmax(metric))
        t2 = timeit(lambda: ops.select_topr(nm, ni, T, r))
        print(f"   sim_argmax {t*1e6:8.1f} us   select_topr {t2*1e6:8.1f} us")
        H = C // 64   # the stack's call: keys read in place from the packed bf16 qkv buffer, mean over heads
        qkv = torch.randn(B, T, 3, H, 64, device="cuda").bfloat16()
        kwm = dict(heads=H, dim=64, batch=B, tokens=T, batch_stride=T * 3 * H * 64, token_stride=3 * H * 64, head_stride=64, offset_elems=H * 64)
        t = timeit(lambda: ops.sim_argmax(qkv, **kwm))
        print(f"   sim_argmax from packed bf16 keys, {H} heads: {t*1e6:8.1f} us")


def bench_gemm():
    for (m, n, k, bmn) in [(137216, 1152, 384, 1), (137216, 384, 384, 1), (133120, 1536, 384, 1), (133120, 384, 1536, 1),
                           (137216, 2304, 768, 1), (129024, 3072, 768, 1), (129024, 768, 3072, 1), (8192, 8192, 8192, 0)]:
        a = torch.randn(m, k, device="cuda").bfloat16()
        b = (torch.randn(k, n, device="cuda") if bmn else torch.randn(n, k, device="cuda")).bfloat16()
        out = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
        t = timeit(lambda: ops.gemm(a, b, m=m, n=n, k=k, b_major=bmn, out=out), iters=5)
        fl = 2.0 * m * n * k
        by = 2.0 * (m * k + n * k + m * n)
        tt = timeit(lambda: torch.matmul(a, b if bmn else b.t(), out=out), iters=5)
        print(f"gemm {m}x{n}x{k}: {t*1e6:9.1f} us {fl/t/1e12:7.1f} TF/s (frac {fl/t/1e12/PEAKS['bf16_tflops']:.3f}) "
              f"{by/t/1e9:7.1f} GB/s | cuBLAS {tt*1e6:9.1f} us {fl/tt/1e12:7.1f} TF/s")
    # wgrad
    for (m, n, k) in [(384, 1152, 137216), (1536, 384, 133120), (768, 3072, 129024)]:
        a = torch.randn(k, m, device="cuda").bfloat16()
        b = torch.randn(k, n, device="cuda").bfloat16()
        out = torch.zeros(m, n, device="cuda")
        t = timeit(lambda: ops.gemm(a, b, m=m, n=n, k=k, a_major=1, b_major=1, out=out, accumulate=True), iters=5)
        fl = 2.0 * m * n * k
        print(f"wgrad {m}x{n}x{k}: {t*1e6:9.1f} us {fl/t/1e12:7.1f} TF/s")


def bench_attn():
    for (B, T, H) in [(256, 536, 6), (256, 536, 12), (32, 2080, 12), (16, 4096, 12)]:
        qkv = torch.randn(B, T, 3, H, 64, device="cuda").bfloat16()
        q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
        size = torch.ones(B, T, device="cuda")
        t = timeit(lambda: ops.attention_fwd(q, k, v, size=size), iters=5)
        fl = 4.0 * B * H * T * T * 64
        print(f"attn_fwd B{B} T{T} H{H}: {t*1e6:9.1f} us {fl/t/1e12:7.1f} TF/s")
        # block-causal group mask in a scrambled token order (as after a merge)
        from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import sequence_groups
        import numpy as np
        n_img = (T - 16) // 2 - 4
        g1, p1, allow, _ = sequence_groups(f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2")
        rng = np.random.default_rng(0)
        gm = torch.tensor(np.stack([rng.permutation(g1) for _ in range(B)])).cuda()
        pm = torch.tensor(np.broadcast_to(p1, (B, len(g1))).copy()).cuda()
        am = torch.tensor(allow).cuda()
        if gm.shape[1] == T:
            t = timeit(lambda: ops.attention_fwd(q, k, v, size=size, gid=gm, pos=pm, allow=am), iters=5)
            print(f"attn_fwd B{B} T{T} H{H} masked: {t*1e6:9.1f} us {fl/t/1e12:7.1f} TF/s")
            t = timeit(lambda: ops.attention_fwd(q, k, v, size=size, gid=gm, pos=pm, allow=am, dropout_rate=0.1, dropout_seed=3, dropout_site=5), iters=5)
            print(f"attn_fwd B{B} T{T} H{H} masked + weight dropout 0.1: {t*1e6:9.1f} us {fl/t/1e12:7.1f} TF/s")
        if hasattr(ops, "attention_bwd"):
            try:
                out, lse = ops.attention_fwd(q, k, v, size=size)
                do = torch.randn_like(out)
                t = timeit(lambda: ops.attention_bwd(q, k, v, out, lse, do, size=size), iters=5)
                print(f"attn_bwd B{B} T{T} H{H}: {t*1e6:9.1f} us {2.5*fl/t/1e12:7.1f} TF/s")
                if gm.shape[1] == T:
                    t = timeit(lambda: ops.attention_bwd(q, k, v, out, lse, do, size=size, gid=gm, pos=pm, allow=am), iters=5)
                    print(f"attn_bwd B{B} T{T} H{H} masked: {t*1e6:9.1f} us {2.5*fl/t/1e12:7.1f} TF/s")
                    t = timeit(lambda: ops.attention_bwd(q, k, v, out, lse, do, size=size, gid=gm, pos=pm, allow=am, dropout_rate=0.1, dropout_seed=3, dropout_site=5), iters=5)
                    print(f"attn_bwd B{B} T{T} H{H} masked + weight dropout 0.1: {t*1e6:9.1f} us {2.5*fl/t/1e12:7.1f} TF/s")
            except Exception as ex:  # not built yet
                print("attn_bwd unavailable:", ex)


def bench_ln():
    for (B, T, C) in [(256, 536, 384), (256, 536, 768)]:
        x = torch.randn(B, T, C, device="cuda").bfloat16()
        g = torch.ones(C, device="cuda")
        b = torch.zeros(C, device="cuda")
        for axis in (1, 2):
            t = timeit(lambda: ops.layernorm_fwd(x, g, b, 1e-6, axis))
            by = 2.0 * B * T * C * 2
            print(f"ln_fwd axis{axis} B{B} T{T} C{C}: {t*1e6:8.1f} us {by/t/1e9:7.1f} GB/s")
            y, mean, rstd = ops.layernorm_fwd(x, g, b, 1e-6, axis)
            dg, db = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
            dres = torch.randn_like(x)
            t = timeit(lambda: ops.layernorm_bwd(x, y, g, mean, rstd, dg, db, dres, axis))
            print(f"ln_bwd axis{axis} B{B} T{T} C{C}: {t*1e6:8.1f} us {2.0*by/t/1e9:7.1f} GB/s")


if __name__ == "__main__":
    which = sys.argv[1:] or ["merge", "gemm", "attn", "ln"]
    for w in which:
        globals()["bench_" + w]()
