"""Global ToMe merging against merging inside token sets, at bench.py's octo-small workload (T0 = 536, B = 256, 12 layers,
C = 384, 6 heads, continuous action head, dropout 0.1, token-axis LayerNorm).

Both arms remove 16 tokens per layer, so every layer has the same shape:
  global  r = 16 over the whole sequence (bench.py's default);
  sets    "[TaskDescriptionPrefix{0}] [Image{8};Readout{0}]*2": 8 merges inside each frame's image set, text and readout sets kept.
The two arms alternate, `--reps` times, each a device-timed run of `--steps` train steps after `--warmup`; then a separate
per-op CUDA-event pass gives the matching (sim_argmax), ranking (select_topr) and merge (forward + backward) times per step.
The global arm's last step also gives the measured share of merges whose source and destination lie in different mask
groups (text, a frame's image tokens, a frame's readouts): what merging inside sets rules out.  Prints one JSON object; the
GPU name and power limit are read in the same run and stored beside the numbers.

    python scripts/bench_set_merge.py [--steps 30 --warmup 5 --reps 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEQ = "[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2"
COMP = "[TaskDescriptionPrefix{0}] [Image{8};Readout{0}]*2"
SHAPE = dict(channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12)


def gpu_info():
    import torch
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [v.strip() for v in out.split(",")]
    except Exception as e:  # noqa: BLE001 -- the numbers stay valid without it; say so in the output
        info["power_limit"] = f"unavailable ({e})"
    return info


def build(arm, batch, dropout):
    import torch

    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig, ToMeStackEngine
    from multi_modal_transformers_tokenmerge_b200.parallel import DataParallelTrainer
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence, sequence_groups
    gid, pos, allow, ro = sequence_groups(SEQ)
    kw = dict(r=16) if arm == "global" else dict(r=0, prune_sets=tuple(TokenSequence(SEQ, COMP).prune_sets()), set_merge=True)
    cfg = StackConfig(batch=batch, tokens=len(gid), ln_axis=1, num_groups=allow.shape[0], n_readout=len(ro), dropout_rate=dropout,
                      dropout_seed=1234, attn_dropout_rate=dropout, head="continuous", head_features=8, max_action=1.0, **SHAPE, **kw)
    eng = ToMeStackEngine(cfg, gid=gid, pos=pos, allow=allow, readout_idx=ro)
    eng.init_params(seed=1)
    g = torch.Generator(device="cuda").manual_seed(100)
    x = torch.randn(batch, len(gid), SHAPE["channels"], device="cuda", generator=g).bfloat16()
    y = torch.rand(batch, 8, device="cuda", generator=g) * 2 - 1
    trainer = DataParallelTrainer(eng)
    return eng, (lambda: trainer.train_step(x, y, lr=1e-4)), np.asarray(gid)


def timed(fn, steps):
    import torch
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def per_op_ms(step, steps):
    """ms per train step of the matching / ranking / merge ops (CUDA events at every op end, tome_profile_*)."""
    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    lib = L.lib()
    L.check(lib.tome_profile_enable(1 << 16))
    for _ in range(steps):
        step()
    import torch
    torch.cuda.synchronize()
    prof = L.profile_collect()
    L.check(lib.tome_profile_disable())
    return {k: round(prof[k][0] / steps, 4) for k in ("sim_argmax", "select_topr", "merge_fwd", "merge_bwd")}


def cross_group_share(eng, gid0):
    """Share of the last forward's merges (all layers, all batch rows) whose source and destination tokens carry different
    mask groups, from the per-layer plan dumps; group ids are followed through the merges (unmerged even tokens, then the
    odd tokens, which keep their own group: token_compression.py:103-108)."""
    B = eng.cfg.batch
    gid = np.broadcast_to(gid0, (B, len(gid0))).copy()
    cross = total = 0
    per_layer = []
    for l in range(eng.cfg.layers):
        pl = eng.layer_plan(l)
        ei = pl[2].cpu().numpy()
        di = pl[3].cpu().numpy()
        r = di.shape[1]
        src_g = np.take_along_axis(gid[:, ::2], ei[:, :r], axis=1)
        dst_g = np.take_along_axis(gid[:, 1::2], di, axis=1)
        c = int((src_g != dst_g).sum())
        per_layer.append(round(c / src_g.size, 4))
        cross, total = cross + c, total + src_g.size
        gid = np.concatenate([np.take_along_axis(gid[:, ::2], ei[:, r:], axis=1), gid[:, 1::2]], axis=1)
    return {"share": round(cross / total, 4), "merges": int(total), "per_layer": per_layer}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_set_merge.py measures on the GPU; no GPU is visible")
    arms = {a: build(a, args.batch, args.dropout) for a in ("global", "sets")}
    for _, step, _ in arms.values():
        for _ in range(args.warmup):
            step()
    sps = {a: [] for a in arms}
    for _ in range(args.reps):            # alternate the arms so drift in clocks or neighbours hits both alike
        for a, (_, step, _) in arms.items():
            sps[a].append(round(args.batch * args.steps / (timed(step, args.steps) * 1e-3), 1))
    res = {"workload": f"octo_small, B={args.batch}, T0=536, 12 layers, 16 tokens removed per layer, train step",
           "gpu": gpu_info(), "steps": args.steps, "reps": args.reps,
           "samples_per_s": {a: {"runs": v, "median": float(np.median(v))} for a, v in sps.items()},
           "ms_per_step": {a: per_op_ms(step, args.steps) for a, (_, step, _) in arms.items()}}
    eng, step, gid0 = arms["global"]
    step()
    torch.cuda.synchronize()
    res["global_cross_group_merges"] = cross_group_share(eng, gid0)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
