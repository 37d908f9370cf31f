"""Inference on the native executor: tome_stack_predict against tome_stack_forward (dropout 0, same inputs), the largest batch
each path can allocate, and the one-kernel diffusion sampler against the per-step loop it replaces.

    python scripts/bench_predict.py --out profiles/r03_predict.json

Stacks: octo-small (C 384, 6 heads, MLP 1536) and octo-base (C 768, 12 heads, MLP 3072) widths, 12 layers, r = 16, the
[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2 sequence (T0 = 536), continuous head (7 actions) or diffusion head
(diffusion_octo_small.yaml's form: A = 8, every other width = C, 32 steps).  Every shape is warmed up first, the two arms of a
comparison alternate inside one loop, times are CUDA-event medians.  Inputs are a few MB to a few GB; no L2 flush between
runs (an inference server sees the same weights every call)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from multi_modal_transformers_tokenmerge_b200 import _lib as L  # noqa: E402
from multi_modal_transformers_tokenmerge_b200 import engine, ops  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.action_heads.diffusion import cosine_beta_schedule, ddpm_coefficients  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence  # noqa: E402

SEQ = "[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2"
WIDTHS = {"octo_small": dict(channels=384, heads=6, mlp_dim=1536), "octo_base": dict(channels=768, heads=12, mlp_dim=3072)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def stack_cfg(width, head, batch):
    ts = TokenSequence(SEQ)
    gid, pos = ts.group_ids()
    allow, ro = ts.allow_table(), ts.get_modality_idx("readouts")
    w = WIDTHS[width]
    kw = dict(batch=batch, tokens=len(gid), head_dim=64, layers=12, r=16, ln_axis=1, num_groups=allow.shape[0], n_readout=len(ro), **w)
    if head == "continuous":
        kw.update(head="continuous", head_features=7)
    else:
        c = w["channels"]
        kw.update(head="diffusion", head_features=8, head_fourier_dim=c, head_time_hidden=c, head_time_out=c, head_hidden=c,
                  diffusion_steps=32)
    return engine.StackConfig(**kw), dict(gid=gid, pos=pos, allow=allow, readout_idx=ro)


def median_ms(fns, iters):
    """Alternate the arms; per arm the median of `iters` CUDA-event timings."""
    times = [[] for _ in fns]
    for _ in range(iters):
        for i, f in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            times[i].append(a.elapsed_time(b))
    return [float(np.median(t)) for t in times]


def launches(fn):
    lib = L.lib()
    torch.cuda.synchronize()
    lib.tome_launch_count(1)
    fn()
    torch.cuda.synchronize()
    return int(lib.tome_launch_count(1))


def kernels(fn):
    """(kernels, memcpy / memset operations) on the device during one call of fn, counted by torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    copies = sum(1 for e in ev if e.name.startswith(("Memcpy", "Memset")))
    return len(ev) - copies, copies


def bench_stacks(iters):
    rows = []
    for width in WIDTHS:
        for head in ("continuous", "diffusion"):
            for batch in (1, 8, 256):
                cfg, masks = stack_cfg(width, head, batch)
                eng = engine.ToMeStackEngine(cfg, training=False, **masks)
                eng.init_params(seed=1)
                pred = eng.predictor()
                x = torch.randn(batch, cfg.tokens, cfg.channels, device="cuda").bfloat16()
                A = cfg.head_features
                if head == "diffusion":
                    eng.set_diffusion_draws(torch.zeros(batch, dtype=torch.int32, device="cuda"),
                                            torch.ones(cfg.diffusion_steps).numpy())
                    target = torch.zeros(2, batch, A, device="cuda")
                    init = torch.randn(batch, A, device="cuda")
                    train = lambda: eng.forward(x, target)  # noqa: E731
                    predict = lambda: pred.predict(x, init=init, noise=init)  # noqa: E731
                else:
                    train = lambda: eng.forward(x)  # noqa: E731
                    predict = lambda: pred.predict(x)  # noqa: E731
                for _ in range(3):
                    train()
                    predict()
                t_train, t_pred = median_ms([train, predict], iters)
                rows.append(dict(width=width, head=head, batch=batch, train_forward_ms=t_train, predict_ms=t_pred,
                                 predict_samples_per_s=batch / (t_pred / 1e3), train_forward_samples_per_s=batch / (t_train / 1e3),
                                 launches_train_forward=launches(train), launches_predict=launches(predict),
                                 workspace_train_bytes=int(eng._ws_bytes), workspace_predict_bytes=int(pred._ws_bytes)))
                print(json.dumps(rows[-1]), flush=True)
                del eng, pred
                torch.cuda.empty_cache()
    return rows


def bench_capacity():
    lib = L.lib()
    total = torch.cuda.get_device_properties(0).total_memory
    out = {"device_memory_bytes": int(total), "workspace_bytes": []}
    for width in WIDTHS:
        for batch in (256, 1024, 4096):
            cfg, _ = stack_cfg(width, "continuous", batch)
            c = cfg.c()
            out["workspace_bytes"].append(dict(width=width, batch=batch, train=int(lib.tome_stack_workspace_bytes(C.byref(c))),
                                               predict=int(lib.tome_stack_predict_workspace_bytes(C.byref(c)))))
    # one predict run at B = 4096 (octo-small), whose training workspace does not fit the card; its first 256 rows vs B = 256
    cfg, masks = stack_cfg("octo_small", "continuous", 256)
    eng = engine.ToMeStackEngine(cfg, training=False, **masks)
    eng.init_params(seed=1)
    big = eng.predictor(4096)
    x = torch.randn(4096, cfg.tokens, cfg.channels, device="cuda").bfloat16()
    big.predict(x)
    t_big = median_ms([lambda: big.predict(x)], 5)[0]
    a_big, r_big = [t[:256].clone() for t in big.predict(x)]
    del big
    torch.cuda.empty_cache()
    small = eng.predictor()
    a, r = small.predict(x[:256].contiguous())
    torch.cuda.synchronize()
    out["large_batch"] = dict(width="octo_small", batch=4096, train_workspace_fits=bool(
        lib.tome_stack_workspace_bytes(C.byref(engine.dataclasses.replace(cfg, batch=4096).c())) < total),
        predict_ms=t_big, samples_per_s=4096 / (t_big / 1e3), first_256_rows_bitwise_equal_to_b256=bool(torch.equal(a_big, a) and torch.equal(r_big, r)),
        first_256_rows_max_abs_diff_actions=float((a_big - a).abs().max()), first_256_rows_max_abs_diff_readout=float((r_big - r).abs().max()))
    print(json.dumps(out["large_batch"]), flush=True)
    return out


def bench_sampler(iters):
    rows = []
    for width, c in (("octo_small", 384), ("octo_base", 768)):
        A, steps, n = 8, 32, 8
        desc_args = (c, n, A, c, c, c, c, steps)
        betas = cosine_beta_schedule(steps)
        alphas = np.float32(1) - betas
        ah = np.array([np.prod(alphas[: i + 1]) for i in range(steps)], np.float32)
        coef_np = ddpm_coefficients(betas)
        for batch in (1, 8, 256):
            g = torch.Generator(device="cuda").manual_seed(batch)
            desc = L.DiffusionDesc(batch, n, *desc_args)
            npar = int(L.lib().tome_diffusion_head_param_count(C.byref(desc)))
            params = torch.randn(npar, device="cuda", generator=g) * 0.05
            p16 = params.bfloat16()
            x = torch.randn(batch, n, c, device="cuda", generator=g).bfloat16()
            init = torch.randn(batch, A, device="cuda", generator=g)
            noise = torch.randn(batch, A, device="cuda", generator=g)
            coef = torch.tensor(coef_np).cuda()
            ones = torch.ones(steps, device="cuda")
            zeros = torch.zeros(batch, A, device="cuda")
            times = [torch.full((batch,), t, dtype=torch.int32, device="cuda") for t in range(steps)]

            def one_call():
                return ops.diffusion_head_sample(x, params, desc, init, noise, coef, 5.0, params_bf16=p16)

            def per_step():   # the loop predict_action ran before: denoiser forward + the update, step by step
                s = init
                for t in range(steps - 1, -1, -1):
                    eps, _, _ = ops.diffusion_head_fwd(x, params, desc, s, zeros, times[t], ones)
                    c1, c2, c3 = (float(v) for v in coef_np[t])
                    s = torch.clamp(c1 * (s - c2 * eps) + c3 * noise, -5.0, 5.0)
                return s

            for _ in range(3):
                one_call()
                per_step()
            t_one, t_loop = median_ms([one_call, per_step], iters)
            a, b = one_call(), per_step()
            torch.cuda.synchronize()
            rows.append(dict(width=width, batch=batch, A=A, hidden=c, steps=steps, one_call_ms=t_one, per_step_loop_ms=t_loop,
                             library_launches_one_call=launches(one_call), library_launches_per_step_loop=launches(per_step),
                             profiled_kernels_and_copies_one_call=kernels(one_call),
                             profiled_kernels_and_copies_per_step_loop=kernels(per_step),
                             max_abs_diff=float((a - b).abs().max())))
            print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_predict.py measures on the GPU; there is none")
    L.lib()
    res = {"card": card(), "sampler": bench_sampler(args.iters), "capacity": bench_capacity(), "stacks": bench_stacks(args.iters)}
    res["card_after"] = card()
    txt = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
