"""The AdamW step and its options: the plain step, the step with weight decay on the Dense kernels only, and the step with
global-norm clipping, non-finite skipping and the norm, at the octo-small and octo-base parameter counts; then an
octo-small train step through DataParallelTrainer with and without clipping.

    python scripts/bench_optimizer.py --out profiles/r03_optimizer.json

Optimizer rows: the flat vectors of a real StackConfig (12 layers, continuous head).  Each arm rotates over enough copies
of (param, grad, m, v, bf16) that one pass moves more than four times the 126 MB L2, so every step reads from HBM; the
three arms alternate, each timed with CUDA events over a window of at least one second.  Bytes are what the step must move:
30 B / parameter (read p, g, m, v; write p, m, v and the bf16 copy) plus 4 B / parameter for the norm pass.  The share of
HBM peak is those bytes over the time against 7.7 TB/s (the data sheet's figure for a 1000 W B200).

Train-step rows: octo-small, batch 256, hidden and attention dropout 0.1 (bench.py's workload) on one GPU, clipping at 1.0
with non-finite skipping and masked decay against the plain step, alternated in blocks of steps inside one run."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from multi_modal_transformers_tokenmerge_b200 import _lib as L  # noqa: E402
from multi_modal_transformers_tokenmerge_b200 import engine  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.ops import _scratch  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.parallel import DataParallelTrainer  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence  # noqa: E402

SEQ = "[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2"
WIDTHS = {"octo_small": dict(channels=384, heads=6, mlp_dim=1536, r=16), "octo_base": dict(channels=768, heads=12, mlp_dim=3072, r=32)}
HBM_PEAK = 7.7e12
L2_BYTES = 126e6


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def stack_cfg(width, batch):
    ts = TokenSequence(SEQ)
    gid, pos = ts.group_ids()
    allow, ro = ts.allow_table(), ts.get_modality_idx("readouts")
    cfg = engine.StackConfig(batch=batch, tokens=len(gid), head_dim=64, layers=12, ln_axis=1, num_groups=allow.shape[0],
                             n_readout=len(ro), head="continuous", head_features=7, **WIDTHS[width])
    return cfg, dict(gid=gid, pos=pos, allow=allow, readout_idx=ro)


def optimizer_rows(width, min_window_s):
    lib = L.lib()
    cfg, _ = stack_cfg(width, batch=2)
    eng = engine.ToMeStackEngine(cfg)   # only for n and the layout of the decay ranges
    n = eng.n_params
    flat = [x for r in eng.decay_ranges("dense_kernels") for x in r]
    ranges = (C.c_longlong * len(flat))(*flat)
    del eng
    torch.cuda.empty_cache()
    copies = max(2, int(4 * L2_BYTES / (30 * n)) + 1)
    g = torch.Generator(device="cuda").manual_seed(0)
    sets = [dict(p=torch.randn(n, device="cuda", generator=g), g=torch.randn(n, device="cuda", generator=g) * 1e-2,
                 m=torch.zeros(n, device="cuda"), v=torch.zeros(n, device="cuda"),
                 w=torch.empty(n, dtype=torch.bfloat16, device="cuda")) for _ in range(copies)]
    ws = _scratch(lib.tome_adamw_workspace_bytes(n), "cuda")
    norm = torch.zeros(1, device="cuda")
    steps = torch.zeros(2, dtype=torch.int32, device="cuda")
    arms = {
        "plain": (None, 30),
        "dense_kernels_decay": (L.AdamwOpts(0.0, 0, ranges, len(flat) // 2, None, None, None, 0), 30),
        "clip_skip_norm": (L.AdamwOpts(1.0, 1, None, 0, norm.data_ptr(), steps.data_ptr(), ws.data_ptr(), ws.numel()), 34),
    }
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run(opts, k, t):
        s = sets[k % copies]
        L.check(lib.tome_adamw_step(n, s["p"].data_ptr(), s["g"].data_ptr(), s["m"].data_ptr(), s["v"].data_ptr(), s["w"].data_ptr(),
                                    1e-4, 0.9, 0.999, 1e-8, 0.1, 1.0, t, None if opts is None else C.byref(opts), stream))

    # warm-up, then size the window: at least min_window_s per arm
    for opts, _ in arms.values():
        for k in range(2 * copies):
            run(opts, k, 1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(copies):
        run(None, k, 1)
    e1.record()
    torch.cuda.synchronize()
    per = e0.elapsed_time(e1) / 1e3 / copies
    iters = max(copies, int(1.2 * min_window_s / per) + 1)   # margin: sized on the plain arm, which is the fastest
    times = {name: [] for name in arms}
    for _ in range(3):   # three alternated windows per arm
        for name, (opts, _) in arms.items():
            e0.record()
            for k in range(iters):
                run(opts, k, 1 + k)
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / 1e3 / iters)
    rows = []
    for name, (_, bpp) in arms.items():
        t = sorted(times[name])[1]
        rows.append({"width": width, "arm": name, "n_params": n, "bytes": bpp * n, "us_per_step": t * 1e6,
                     "window_s": t * iters, "l2_rotation_copies": copies, "hbm_fraction": bpp * n / t / HBM_PEAK,
                     "us_per_step_all_windows": [x * 1e6 for x in times[name]]})
        print(json.dumps(rows[-1]), flush=True)
    del sets
    torch.cuda.empty_cache()
    return rows


def train_rows(steps, blocks):
    cfg, masks = stack_cfg("octo_small", batch=256)
    cfg = engine.StackConfig(**{**cfg.__dict__, "dropout_rate": 0.1, "attn_dropout_rate": 0.1})
    eng = engine.ToMeStackEngine(cfg, **masks)
    eng.init_params(seed=1)
    g = torch.Generator(device="cuda").manual_seed(2)
    x = torch.randn(cfg.batch, cfg.tokens, cfg.channels, device="cuda", generator=g).bfloat16()
    y = torch.rand(cfg.batch, 7, device="cuda", generator=g) * 2 - 1
    tr = DataParallelTrainer(eng)
    arms = {"plain": {}, "clip_skip_dense_decay": dict(max_grad_norm=1.0, skip_nonfinite=True, decay="dense_kernels",
                                                       weight_decay=1e-4)}
    for kw in arms.values():
        for _ in range(3):
            tr.train_step(x, y, lr=1e-4, **kw)
    torch.cuda.synchronize()
    ms = {name: [] for name in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(blocks):
        for name, kw in arms.items():
            e0.record()
            for _ in range(steps):
                tr.train_step(x, y, lr=1e-4, **kw)
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / steps)
    rows = []
    for name in arms:
        t = sorted(ms[name])[len(ms[name]) // 2]
        rows.append({"workload": "octo_small train step, batch 256, dropout 0.1, 1 GPU", "arm": name, "ms_per_step_median": t,
                     "samples_per_s": cfg.batch / t * 1e3, "ms_per_step_blocks": ms[name]})
        print(json.dumps(rows[-1]), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the JSON result here as well")
    ap.add_argument("--min-window", type=float, default=1.0, help="seconds per timed optimizer window")
    ap.add_argument("--train-steps", type=int, default=10, help="train steps per timed block")
    ap.add_argument("--train-blocks", type=int, default=5, help="alternated blocks per train-step arm")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_optimizer needs a CUDA device")
    res = {"card": card(), "optimizer": [], "train_step": []}
    print(json.dumps(res["card"]), flush=True)
    for width in WIDTHS:
        res["optimizer"] += optimizer_rows(width, args.min_window)
    res["train_step"] = train_rows(args.train_steps, args.train_blocks)
    txt = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt)
    print(txt)


if __name__ == "__main__":
    main()
