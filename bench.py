#!/usr/bin/env python
"""bench.py -- ToMe-transformer train samples/s (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus N --steps K --warmup W                  # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W # the reference's algorithm on the host CPU

A "step" is one full training step of the octo-small-style ToMe stack (BASELINE.json configs[1]: batch 256 per GPU,
T0 = 536 tokens, 12 layers, r = 16 / layer, block-causal readout mask, bf16) on synthetic embeddings: zero grads,
forward, action head + l2 loss on the readouts (or the synthetic readout MSE), full backward, (N > 1: NCCL gradient all-reduce, see --overlap), AdamW.
One JSON line is printed by rank 0.  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEQ = "[TaskDescriptionPrefix{16}] [Image{256};Readout{4}]*2"   # T0 = 536 (form of octo_base.yaml:10)
SEQ_C3 = "[TaskDescriptionPrefix{16}] [Image{256};Image{256};Readout{4}]*4"   # T0 = 2080: wrist + primary camera, 4-frame history
CONFIGS = {
    # BASELINE.json configs[1]: octo-small train step bf16, batch 256 / GPU, r = 16
    "octo_small": dict(channels=384, heads=6, head_dim=64, mlp_dim=1536, layers=12, r=16, batch=256, seq=SEQ, baseline_cfg=1),
    # BASELINE.json configs[2] per-GPU shard: octo-base, 256 / GPU (2048 on 8 GPUs), r = 32
    "octo_base": dict(channels=768, heads=12, head_dim=64, mlp_dim=3072, layers=12, r=32, batch=256, seq=SEQ, baseline_cfg=2),
    # BASELINE.json configs[3]: octo-base with wrist + primary cameras (2x image tokens), 4-frame history; sweep with --r 0..64
    "c3": dict(channels=768, heads=12, head_dim=64, mlp_dim=3072, layers=12, r=32, batch=32, seq=SEQ_C3, baseline_cfg=3),
}
METRIC = "ToMe-transformer train samples/sec"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


def flops_per_sample(c, T0):
    """Algorithmic block FLOPs (SURVEY.md 8d): forward, x3 for a train step."""
    C, Dff, D, r = c["channels"], c["mlp_dim"], c["head_dim"], c["r"]
    T, tot = T0, 0.0
    for _ in range(c["layers"]):
        rr = min(r, T // 2)
        tot += 6 * T * C * C + 4 * T * T * C + 2 * T * C * C + 2 * ((T + 1) // 2) * (T // 2) * D + 4 * (T - rr) * C * Dff
        T -= rr
    return tot


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([v.strip() for v in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        mx = max(float(r[1]) for r in self.rows if len(r) >= 7)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ reference arm / cpu baseline
ACTION_DIM, MAX_ACTION = 8, 1.0   # action_heads/diffusion.yaml dense_out features: 8; continuous.py:13 max_action


def cpu_reference_steps(cfgname, steps, warmup, sample_batch, loss_kind="continuous", r=None, dropout=0.0, attn_dropout=0.0):
    """The reference's algorithm for this path, restated (oracle/tome_oracle.py: sequential scatter loop, double merge
    call, dense [B,H,T,T] mask, fp32) as a torch-CPU train step with autograd + AdamW and the same dropout sites, all host
    threads.  JAX/Flax are not installable here (no wheels, no network), so this is the port ("kind": "port"), not the
    JAX program."""
    import numpy as np
    import torch
    from oracle import tome_oracle as O

    c = dict(CONFIGS[cfgname])
    if r is not None:
        c["r"] = r
    gid, pos, allow, ro = O.sequence_groups(c["seq"])
    T0 = gid.shape[0]
    rng = np.random.default_rng(1)
    params = [O.block_params_to_torch(O.init_block_params(rng, c["channels"], c["heads"], c["head_dim"], c["mlp_dim"]),
                                      requires_grad=True) for _ in range(c["layers"])]
    pe = torch.tensor((rng.standard_normal((1, T0, c["channels"])) * 0.02).astype(np.float32), requires_grad=True)
    x = torch.tensor(np.random.default_rng(0).standard_normal((sample_batch, T0, c["channels"])).astype(np.float32))
    y = torch.tensor(np.random.default_rng(2).standard_normal((sample_batch, len(ro), c["channels"])).astype(np.float32))
    leaves = [t for p in params for t in p.tensors()] + [pe]
    if loss_kind == "continuous":   # ContinuousActionHead + compute_l2_loss (continuous.py:16-25, octo.py:157-165, 253-263)
        hk = torch.tensor((rng.standard_normal((c["channels"], ACTION_DIM)) * (2.0 / c["channels"]) ** 0.5).astype(np.float32),
                          requires_grad=True)
        hb = torch.zeros(ACTION_DIM, requires_grad=True)
        actions = torch.tensor(np.random.default_rng(3).uniform(-1, 1, (sample_batch, ACTION_DIM)).astype(np.float32))
        leaves += [hk, hb]
    opt = torch.optim.AdamW(leaves, lr=1e-4, weight_decay=0.0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        xf, size, origin = O.tome_stack(params, pe, x, gid, pos, allow, num_heads=c["heads"], r=c["r"], dropout_rate=dropout,
                                        attn_dropout_rate=attn_dropout)
        loss, readouts = O.readout_loss(xf, origin, ro, y)
        if loss_kind == "continuous":
            loss = O.l2_loss(O.continuous_action_head(readouts, hk, hb, MAX_ACTION), actions).mean()
        loss.backward()
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return sample_batch * len(times) / sum(times), sum(times) / len(times), torch.get_num_threads(), T0


def cfg_of(args):
    c = dict(CONFIGS[args.config])
    if getattr(args, "r", None) is not None:
        c["r"] = args.r
    if getattr(args, "batch", 0):
        c["batch"] = args.batch
    return c


REF_SAMPLE_BATCH = 8   # BASELINE.md section 3: the reference's own CPU-runnable case is batch 8
DUMP_SAMPLE = 1 << 20  # --dump-outputs: larger arrays are reduced to this many elements (4 MB each in float32)


def step_outputs(eng):
    """What one train step hands its caller, copied to the host as float32: the per-sample losses with their mean
    (loss[0]), the action head's output, the pooled readout rows, and the parameters and gradients after the AdamW update.
    An array of more than DUMP_SAMPLE elements is flattened and reduced to a sample at fixed, seeded positions (the same
    positions for every run of the same shape), which keeps the five arrays under 20 MB at any batch."""
    import numpy as np
    import torch

    out, positions = {}, {}
    for name, t in (("loss", eng.loss), ("head_out", eng.head_out), ("readout", eng.readout), ("params", eng.params),
                    ("grads", eng.grads)):
        if t is None:
            continue
        if t.numel() > DUMP_SAMPLE:
            if t.numel() not in positions:
                idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
                positions[t.numel()] = torch.from_numpy(idx).to(t.device)
            t = t.reshape(-1).index_select(0, positions[t.numel()])
            name += "_sample"
        out[name] = t.float().cpu().numpy()
    return out


def workload_config(args, world, B, T0):
    """The `config` object both arms print: the workload is the same, only the implementation differs."""
    c = cfg_of(args)
    return {"workload": f"{args.config} ToMe stack train step (BASELINE.json configs[{c['baseline_cfg']}] shape)",
            "global_batch": B * world, "per_gpu_batch": B, "tokens": T0, "layers": c["layers"], "channels": c["channels"],
            "heads": c["heads"], "mlp_dim": c["mlp_dim"], "r_per_layer": c["r"], "mask": "block-causal group table",
            "compression": ("per-modality top-k pruning per layer (attention-received importance)" if getattr(args, "compress", "merge") == "prune"
                            else "ToMe bipartite merge per layer"),
            "ln_axis": "tokens",
            "loss": ("continuous action head + l2 loss on the pooled readouts (continuous_train_step, octo.py:242-280)"
                     if args.loss == "continuous" else "synthetic MSE on the readout rows"),
            "hidden_dropout": args.dropout, "attention_dropout": args.attn_dropout, "optimizer": "AdamW fp32 master",
            "parallelism": f"dp{world}", "allreduce": (args.overlap if world > 1 else None), "comm_sms": args.comm_sms if world > 1 else 0, "l2_policy": "inputs and activations (>= 1 GB/step) exceed the 126 MB L2"}


def run_reference(args, rank):
    if rank != 0:
        return
    sb = REF_SAMPLE_BATCH   # the same bounded sample whatever --steps / --warmup say
    c = cfg_of(args)
    sps, sec, cores, T0 = cpu_reference_steps(args.config, args.steps, args.warmup, sb, args.loss, r=c["r"], dropout=args.dropout,
                                              attn_dropout=args.attn_dropout)
    sample = (f"{sb} samples/step of the {args.config} workload (T0={T0}, {c['layers']} layers, r={c['r']}), fp32, train step "
              f"(forward, loss, backward, AdamW; hidden dropout {args.dropout}, attention dropout {args.attn_dropout})")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": sps, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": dict(workload_config(args, int(os.environ.get("WORLD_SIZE", "1")), c["batch"], T0),
                       reference_note=f"restated reference on the host CPU: each step is a bounded sample of {sb} of the "
                                      f"{c['batch']} samples per GPU, same loss, AdamW and dropout sites as the GPU arm"),
        "cpu_baseline": {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def tracked_traffic():
    """DRAM read + write per launch of the two roofline kernels, from the tracked summary of this round's ncu --set full
    captures (profiles/roofline_traffic.json: written by scripts/ncu_summaries.py traffic, never typed in by hand)."""
    p = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    return json.load(open(p)) if os.path.exists(p) else {}


# ------------------------------------------------------------------------------------------------ configs[4]: block microbench
def microbench(args):
    """BASELINE.json configs[4]: the kernels of one ToMe block, standalone, at 1k - 8k tokens and d = 768 / 1024, with a merge
    ratio sweep, each against the roofline that bounds it.  Every kernel is timed ALONE (CUDA events, L2 flushed by writing
    256 MB between launches, 3 warm-up + 5 timed launches), so the denominators are the burst peaks of MEASURED_PEAKS.json.
    B is chosen so that B * T = 32 768 tokens.  Algorithmic work per launch: attention 4 T^2 D / 10 T^2 D flop per (b, h);
    sim 2 Ta Tb D flop per sample; GEMM 2 M N K; merge / LayerNorm bytes as in DESIGN.md section 4."""
    import numpy as np
    import torch

    from multi_modal_transformers_tokenmerge_b200 import ops
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import sequence_groups

    P = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timeit(fn, iters=5, warmup=3):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        tot = 0.0
        for _ in range(iters):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            tot += e0.elapsed_time(e1)
        return tot / iters * 1e-3

    rows = []

    def add(kernel, T, C, r, sec, flops=None, nbytes=None):
        row = {"kernel": kernel, "tokens": T, "channels": C, "r": r, "us": sec * 1e6}
        if flops is not None:
            row.update(bound="tensor", achieved_tflops=flops / sec / 1e12, frac=flops / sec / 1e12 / P["tf_burst"])
        else:
            row.update(bound="hbm", achieved_gbs=nbytes / sec / 1e9, frac=nbytes / sec / 1e9 / P["hbm"])
        rows.append(row)

    rng = np.random.default_rng(0)
    for T in (1024, 2048, 4096, 8192):
        for C in (768, 1024):
            B, H, D = 32768 // T, C // 64, 64
            M = B * T
            x = torch.randn(B, T, C, device="cuda").bfloat16()
            qkv = torch.randn(B, T, 3, H, D, device="cuda").bfloat16()
            q, k, v = qkv[:, :, 0], qkv[:, :, 1], qkv[:, :, 2]
            n_img = (T - 16) // 2 - 4
            g1, p1, allow, _ = sequence_groups(f"[TaskDescriptionPrefix{{16}}] [Image{{{n_img}}};Readout{{4}}]*2")
            gid = torch.tensor(np.stack([rng.permutation(g1) for _ in range(B)])).cuda()   # scrambled, as after a merge
            pos = torch.tensor(np.broadcast_to(p1, (B, T)).copy()).cuda()
            kw = dict(gid=gid, pos=pos, allow=torch.tensor(allow).cuda(), size=torch.randint(1, 4, (B, T), device="cuda").float())
            # --- attention (masked, proportional bias)
            fl = 4.0 * B * H * T * T * D
            add("attn_fwd", T, C, None, timeit(lambda: ops.attention_fwd(q, k, v, **kw)), flops=fl)
            out, lse = ops.attention_fwd(q, k, v, **kw)
            do = torch.randn_like(out)
            add("attn_bwd", T, C, None, timeit(lambda: ops.attention_bwd(q, k, v, out, lse, do, **kw)), flops=2.5 * fl)
            # --- dense layers of the block (forward shapes)
            for name, n_, k_ in (("gemm_qkv", 3 * C, C), ("gemm_mlp1", 4 * C, C), ("gemm_mlp2", C, 4 * C)):
                a = torch.randn(M, k_, device="cuda").bfloat16()
                w = torch.randn(k_, n_, device="cuda").bfloat16()
                o_ = torch.empty(M, n_, device="cuda", dtype=torch.bfloat16)
                add(name, T, C, None, timeit(lambda: ops.gemm(a, w, m=M, n=n_, k=k_, b_major=1, out=o_)), flops=2.0 * M * n_ * k_)
                del a, w, o_
            # --- LayerNorm over tokens
            gm, bt = torch.ones(C, device="cuda"), torch.zeros(C, device="cuda")
            add("ln_fwd", T, C, None, timeit(lambda: ops.layernorm_fwd(x, gm, bt, 1e-6, 1)), nbytes=2.0 * M * C * 2)
            y_, mean, rstd = ops.layernorm_fwd(x, gm, bt, 1e-6, 1)
            dg, db = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
            add("ln_bwd", T, C, None, timeit(lambda: ops.layernorm_bwd(x, y_, gm, mean, rstd, dg, db, None, 1)), nbytes=3.0 * M * C * 2)
            # --- matching + merge, ratio sweep
            ta, tb = (T + 1) // 2, T // 2
            kwm = dict(heads=H, dim=D, batch=B, tokens=T, batch_stride=T * 3 * H * D, token_stride=3 * H * D, head_stride=D,
                       offset_elems=H * D)   # the keys, read in place from the packed qkv buffer
            add("sim_argmax", T, C, None, timeit(lambda: ops.sim_argmax(qkv, **kwm)), flops=2.0 * B * ta * tb * D)
            nm, ni, _ = ops.sim_argmax(qkv, **kwm)
            size = torch.ones(B, T, device="cuda")
            for r in (T // 16, T // 8, T // 4, T // 2):
                add("select_topr", T, C, r, timeit(lambda: ops.select_topr(nm, ni, T, r)), nbytes=B * (8.0 * ta + 4 * (ta + r + T + tb + 1 + r)))
                plan = ops.select_topr(nm, ni, T, r)
                add("merge_fwd", T, C, r, timeit(lambda: ops.merge_fwd(plan, x, size, 1)),
                    nbytes=B * (T * C * 2.0 + 4 * T + 4 * (ta + r) + (T - r) * C * 2 + 4 * (T - r)))
                x1, s1, _, _ = ops.merge_fwd(plan, x, size, 1)
                dy = torch.randn_like(x1)
                add("merge_bwd", T, C, r, timeit(lambda: ops.merge_bwd(plan, dy, size, s1, 1)),
                    nbytes=B * ((T - r) * C * 2.0 + T * C * 2 + 4 * T))
                del plan, x1, s1, dy
            # --- the sibling compression path: importance from the attention weights, per-set top-k + gather, its backward
            add("importance", T, C, None, timeit(lambda: ops.attention_importance(q, k, lse, "received", **kw)), flops=2.0 * B * H * T * T * D)
            imp = ops.attention_importance(q, k, lse, "received", **kw)
            for r in (T // 16, T // 4):
                c_img = r // 2
                ss, sn = [0, 16, 16 + n_img, 20 + n_img, 20 + 2 * n_img], [16, n_img, 4, n_img, 4]
                sk = [16, n_img - c_img, 4, n_img - c_img, 4]
                kept = sum(sk)
                add("topk_prune", T, C, 2 * c_img, timeit(lambda: ops.topk_prune(x, imp, ss, sn, sk)), nbytes=B * (4.0 * T + 2.0 * kept * C * 2 + 4 * kept))
                _, ids = ops.topk_prune(x, imp, ss, sn, sk)
                rm, _, _ = ops.prune_row_map(ids, T)
                dy = torch.randn(B, kept, C, device="cuda").bfloat16()
                add("prune_bwd", T, C, 2 * c_img, timeit(lambda: ops.prune_bwd(rm, dy)), nbytes=B * (kept * C * 2.0 + T * C * 2 + 4 * T))
                del ids, rm, dy
            del x, qkv, out, lse, do, imp
            torch.cuda.empty_cache()
    # --- the image patch-embed front end (forward): gato_resnet.yaml's geometry and the named shape's (256 x 256, 16-pixel patches)
    from multi_modal_transformers_tokenmerge_b200 import model_configs
    for label, image, patch, E_, nb in (("gato 280/56", 280, 56, 768, 64), ("named shape 256/16", 256, 16, 768, 256)):
        node = dict(model_configs.load("tokenizers/images/gato_resnet_octo")["encoder"])
        node.update(image_size=[image, image, 3], patch_size=patch)
        tok = model_configs.build_image_tokenizer(node)
        tv = tok.init(1, None)
        frames = torch.randint(0, 256, (nb, 2, image, image, 3), dtype=torch.uint8, device="cuda")
        o1 = (patch - 12) // 2 + 1
        o2 = o1 - 2
        npatch = (image // patch) ** 2
        fl = 2.0 * nb * 2 * npatch * (o1 * o1 * 432 * 64 + 2 * o2 * o2 * 576 * 64 + o2 * o2 * 64 * E_)
        sec = timeit(lambda: tok.apply(tv, frames, train=False))
        rows.append({"kernel": "image_front_end", "geometry": label, "frames": nb * 2, "us": sec * 1e6, "frames_per_s": nb * 2 / sec,
                     "bound": "tensor", "achieved_tflops": fl / sec / 1e12, "frac": fl / sec / 1e12 / P["tf_burst"]})
        del frames, tok, tv
        torch.cuda.empty_cache()
    return {"metric": "ToMe block microbench (BASELINE.json configs[4]): per-kernel time against its roofline",
            "unit": "us per launch; frac = achieved / measured burst peak", "n_gpus": 1, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "standalone ToMe block kernels, B * T = 32768 tokens, T in 1k..8k, d in {768, 1024}, heads = d / 64, "
                                   "r in T/16..T/2, block-causal group mask in post-merge order, log-size bias",
                       "l2_policy": "256 MB written between timed launches"},
            "peaks": {"hbm_gbs": P["hbm"], "bf16_tflops_burst": P["tf_burst"], "source": P["src"]}, "rows": rows}


# ------------------------------------------------------------------------------------------------ this repo's arm
def measure_workload(args, cfgname, rank, world, local, steps, warmup, with_extras=True, dump_dir=None):
    """One workload measured three ways on this rank's GPU (max over ranks): device-timed steps with resident inputs
    (`value`), end to end through the public trainer API with pinned-host inputs (`e2e`), and a per-op CUDA-event pass
    (`kernels`, `roofline`).  Returns the dict rank 0 prints (None on other ranks).  dump_dir: rank 0 writes what the last
    timed step computed there (step_outputs), before the later passes train on further inputs."""
    import torch
    import torch.distributed as dist

    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    from multi_modal_transformers_tokenmerge_b200.engine import StackConfig, ToMeStackEngine
    from multi_modal_transformers_tokenmerge_b200.parallel import DataParallelTrainer
    from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import sequence_groups

    lib = L.lib()
    a2 = argparse.Namespace(**{**vars(args), "config": cfgname})
    c = cfg_of(a2)
    gid, pos, allow, ro = sequence_groups(c["seq"])
    T0, B, C = len(gid), c["batch"], c["channels"]
    prune_kw, eng_kw = {}, {}
    if getattr(args, "compress", "merge") == "prune":
        # the sibling compression path (SURVEY 8f rank 2): every layer DROPS r tokens, split evenly over the image sets, by
        # attention-received importance + per-set top-k, masks from the compression grammar at each layer
        from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenSequence
        n_img = c["seq"].count("Image{")
        assert c["r"] % n_img == 0, "--compress prune: r must split evenly over the image sets"
        comp = re.sub(r"Image\{\d+\}", "Image{%d}" % (c["r"] // n_img), re.sub(r"(TaskDescriptionPrefix|Readout)\{\d+\}", r"\1{0}", c["seq"]))
        ts = TokenSequence(c["seq"], comp)
        lg = [ts.layer_group_ids(l) for l in range(c["layers"])]
        prune_kw = dict(prune_sets=tuple(ts.prune_sets()), prune_importance="received", prop_attn=False)
        eng_kw = dict(layer_gid=[g_ for g_, _ in lg], layer_pos=[p_ for _, p_ in lg])
    cfg = StackConfig(batch=B, tokens=T0, channels=C, heads=c["heads"], head_dim=c["head_dim"], mlp_dim=c["mlp_dim"],
                      layers=c["layers"], r=0 if prune_kw else c["r"], ln_axis=1, num_groups=allow.shape[0], n_readout=len(ro),
                      dropout_rate=args.dropout, dropout_seed=1234 + rank, attn_dropout_rate=args.attn_dropout, **prune_kw,
                      **(dict(head="continuous", head_features=ACTION_DIM, max_action=MAX_ACTION) if args.loss == "continuous" else {}))
    eng = ToMeStackEngine(cfg, gid=gid, pos=pos, allow=allow, readout_idx=ro, **eng_kw)
    eng.init_params(seed=1)  # same weights on every rank
    trainer = DataParallelTrainer(eng, comm_sms=args.comm_sms if world > 1 else 0, overlap=args.overlap)
    g = torch.Generator(device="cuda").manual_seed(100 + rank)
    x = torch.randn(B, T0, C, device="cuda", generator=g).bfloat16()      # synthetic block inputs (embeddings)
    tshape = (B, ACTION_DIM) if args.loss == "continuous" else (B, len(ro), C)   # target actions / synthetic readout targets
    y = torch.rand(*tshape, device="cuda", generator=g) * 2 - 1 if args.loss == "continuous" else torch.randn(*tshape, device="cuda", generator=g)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    step = lambda: trainer.train_step(x, y, lr=1e-4)  # noqa: E731
    for _ in range(warmup):
        step()
    lib.tome_launch_count(1)
    with ClockSampler(local) as clk:
        ms = timed(steps, step)
    launches = int(lib.tome_launch_count(1))
    loss_dev = float(eng.loss[0].item())
    value = world * B * steps / (ms * 1e-3)
    if dump_dir is not None and rank == 0:
        import numpy as np
        os.makedirs(dump_dir, exist_ok=True)
        for name, a in step_outputs(eng).items():
            np.save(os.path.join(dump_dir, name + ".npy"), a)

    # every rank started from the same weights and applied the same summed gradients: the parameter vectors must be
    # bit-identical (a checksum of the fp32 bit patterns, min == max over the ranks)
    in_sync = None
    if world > 1:
        chk = eng.params.view(torch.int32).to(torch.int64).sum().reshape(1)
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        in_sync = bool(lo.item() == hi.item())

    # ---- end to end through the public API: pinned host inputs -> H2D -> step -> D2H loss, every step ----
    xh = [torch.randn(B, T0, C).bfloat16().pin_memory() for _ in range(2)]
    yh = [(torch.rand(*tshape) * 2 - 1 if args.loss == "continuous" else torch.randn(*tshape)).pin_memory() for _ in range(2)]
    xd = [torch.empty_like(x) for _ in range(2)]
    yd = [torch.empty_like(y) for _ in range(2)]
    loss_h = torch.zeros(1).pin_memory()
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"i": 0}

    def prefetch(i):
        s_ = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s_])
            xd[s_].copy_(xh[s_], non_blocking=True)
            yd[s_].copy_(yh[s_], non_blocking=True)
            ready[s_].record(copy_stream)

    def e2e_step():
        i = state["i"]
        s_ = i & 1
        if i == 0:
            prefetch(0)
        prefetch(i + 1)                       # next step's inputs stream in under this step's compute
        torch.cuda.current_stream().wait_event(ready[s_])
        trainer.train_step(xd[s_], yd[s_], lr=1e-4)
        consumed[s_].record()
        loss_h.copy_(eng.loss[:1], non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the step's result is read on the host every step
        state["i"] = i + 1

    for ev in consumed:
        ev.record()
    for _ in range(2):
        e2e_step()
    ms_e2e = timed(steps, e2e_step)
    e2e_value = world * B * steps / (ms_e2e * 1e-3)
    h2d = xh[0].numel() * 2 + yh[0].numel() * 4
    d2h = 4

    # ---- from pixels (extra, N = 1 line only): the image patch-embed front end (csrc/image_tokenizer.cu, forward) produces the
    # image tokens of the step from uint8 frames -- 256 x 256 x 3 per frame, 16-pixel patches = 256 tokens per frame, the named
    # shape -- which are assembled with the language / readout token embeddings (TokenSequence.assemble_embeddings) into the
    # block's input; then the same train step.  The front end has no backward here (the reference trains it), so this is an
    # observations -> loss throughput of the block's step with its inputs computed on the device, not a second headline.
    from_pixels = None
    if with_extras and getattr(args, "from_pixels", "auto") != "off" and c["seq"] == SEQ:
        from multi_modal_transformers_tokenmerge_b200.tokenizers.images import ImageTokenizer
        from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenEmbeddings, TokenSequence
        node = lambda t_, **kw: dict(_target_=t_, **kw)  # noqa: E731
        tok = ImageTokenizer(image_size=(256, 256, 3), patch_size=16, normalize=True, position_interval=128, rng_collection="patch_encoding",
                             embedding_dim=C, out_dtype=torch.bfloat16,
                             row_position_embedding=node("flax.linen.Embed", name="image_row_position_embedding", num_embeddings=128, features=C),
                             col_position_embedding=node("flax.linen.Embed", name="image_col_position_embedding", num_embeddings=128, features=C),
                             resnet=dict(num_blocks=2,
                                         input_conv=node("flax.linen.Conv", features=64, kernel_size=[12, 12], strides=[2, 2], padding="VALID"),
                                         input_pool=node("flax.linen.max_pool", window_shape=[3, 3], strides=[1, 1], padding="VALID"),
                                         resnet_norm=node("flax.linen.GroupNorm", num_groups=32, epsilon=1e-6),
                                         resnet_activation=node("flax.linen.gelu"),
                                         resnet_conv=node("flax.linen.Conv", features=64, kernel_size=[3, 3], strides=[1, 1], padding="SAME"),
                                         output_dense=node("flax.linen.Dense", features=C)))
        tvars = tok.init(3, None)
        ts = TokenSequence(c["seq"])
        frames = torch.randint(0, 256, (B, 2, 256, 256, 3), dtype=torch.uint8, device="cuda", generator=g)
        text = torch.randn(B, 16, C, device="cuda", generator=g).bfloat16()
        readouts = torch.randn(B, 8, C, device="cuda", generator=g).bfloat16()
        state_px = {}

        def pixel_step():
            img_tok = tok.apply(tvars, frames, train=False).reshape(B, 2 * 256, C)
            xin = ts.assemble_embeddings(TokenEmbeddings(text=text, images=img_tok, readouts=readouts)).contiguous()
            state_px["x"] = xin
            trainer.train_step(xin, y, lr=1e-4)

        for _ in range(3):
            pixel_step()
        lib.tome_launch_count(1)
        ms_px = timed(steps, pixel_step)
        launches_px = int(lib.tome_launch_count(1))
        e0_, e1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0_.record()
        for _ in range(steps):
            tok.apply(tvars, frames, train=False)
        e1_.record()
        torch.cuda.synchronize()
        from_pixels = {"value": world * B * steps / (ms_px * 1e-3), "unit": "samples/s", "ms_per_step": ms_px / steps,
                       "front_end_ms": e0_.elapsed_time(e1_) / steps, "frames_per_sample": 2, "frame": "256 x 256 x 3 uint8, 16-pixel patches -> 256 tokens",
                       "pixel_bytes_per_step": int(frames.numel()), "gpu_launches": launches_px,
                       "note": "image front end forward (no backward) + token assembly + the same train step"}
        del frames, text, readouts, state_px

    # ---- roofline pass: same step, every op bracketed by CUDA events on its own stream ----
    P = peaks()
    L.check(lib.tome_profile_enable(4096))
    nprof = 2
    for _ in range(nprof):
        step()
    torch.cuda.synchronize()
    prof = L.profile_collect()
    lib.tome_profile_disable()
    tot_ms = sum(v[0] for v in prof.values())
    kernels = {}
    for k_, (kms, work, cnt) in prof.items():
        if cnt == 0:
            continue
        ent = {"ms_per_step": kms / nprof, "share": kms / tot_ms, "ops_per_step": cnt // nprof}
        if k_ in ("gemm", "attn_fwd", "attn_bwd", "sim_argmax", "importance") and kms > 0:
            ent["tflops"] = work / (kms * 1e-3) / 1e12
            ent["frac_of_sustained_bf16_peak"] = ent["tflops"] / P["tf_sust"]
        elif work > 0 and kms > 0:
            ent["gbs"] = work / (kms * 1e-3) / 1e9
            ent["frac_of_hbm_peak"] = ent["gbs"] / P["hbm"]
        kernels[k_] = ent
    gms, gwork, gcnt = prof["gemm"]
    # DRAM read + write per launch from the tracked summary of this round's ncu captures; only for the captured configuration
    tr = tracked_traffic()
    captured = cfgname == "octo_small" and B == 256 and c["r"] == 16
    gt, mt = tr.get("gemm_bf16_kernel", {}), tr.get("merge_fwd_bulk_kernel", {})
    roof = {"bound": "tensor", "kernel": "gemm_bf16_kernel (tcgen05)", "achieved": gwork / (gms * 1e-3) / 1e12,
            "peak": P["tf_sust"], "unit": "TFLOP/s", "frac": gwork / (gms * 1e-3) / 1e12 / P["tf_sust"],
            "traffic": gt.get("bytes_per_launch") if captured else None,
            "traffic_unit": "bytes per launch (ncu dram read+write, mean over the GEMM launches of layer 0)",
            "traffic_source": gt.get("source") if captured else None,
            "peak_source": f"{P['src']} bf16_tflops_sustained", "launches_per_step": gcnt // nprof,
            "avg_launch_us": gms / gcnt * 1e3, "share_of_step": gms / tot_ms}
    mms, mwork, mcnt = prof["merge_fwd"]
    merge_roof = {"bound": "hbm", "kernel": "merge_fwd_kernel", "achieved": mwork / (mms * 1e-3) / 1e9, "peak": P["hbm"],
                  "unit": "GB/s", "frac": mwork / (mms * 1e-3) / 1e9 / P["hbm"],
                  "traffic": mt.get("bytes_per_launch") if captured else None,
                  "traffic_unit": "bytes per launch (ncu dram read+write, layer 0)", "traffic_source": mt.get("source") if captured else None,
                  "peak_source": f"{P['src']} hbm_gbs", "avg_launch_us": mms / mcnt * 1e3} if mcnt else None

    # ---- the same merge kernel timed back to back (no per-launch event pair): three disjoint input/output sets of the
    # layer-0 shape (> the 126 MB L2), 30 launches between ONE pair of events.
    if with_extras and merge_roof is not None and c["r"] > 0 and not prune_kw:
        from multi_modal_transformers_tokenmerge_b200 import ops as O_
        r0 = lib.tome_clamp_r(T0, c["r"], 0, 0)
        metric = torch.randn(B, T0, c["head_dim"], device="cuda", generator=g)
        nm, ni, _ = O_.sim_argmax(metric)
        plan = O_.select_topr(nm, ni, T0, r0)
        import ctypes as CT
        sets = [(torch.randn(B, T0, C, device="cuda", generator=g).bfloat16(), torch.ones(B, T0, device="cuda"),
                 torch.empty(B, T0 - r0, C, device="cuda", dtype=torch.bfloat16), torch.empty(B, T0 - r0, device="cuda"))
                for _ in range(3)]   # inputs AND outputs rotate, so neither side is served from L2
        shp = L.MergeShape(B, T0, C, r0, 0, L.TOME_BF16, L.TOME_MERGE_WAVG)
        cp = plan.c_plan()
        strm = CT.c_void_p(torch.cuda.current_stream().cuda_stream)

        def merge_once(it=iter(range(10 ** 9))):
            xs, ss, xo, so = sets[next(it) % 3]
            L.check(lib.tome_merge_fwd(CT.byref(shp), CT.byref(cp), xs.data_ptr(), ss.data_ptr(), xo.data_ptr(), so.data_ptr(),
                                       None, None, None, None, strm))

        for _ in range(3):
            merge_once()
        n_rep = 30
        ms_m = timed(n_rep, merge_once)
        bytes_m = B * (T0 * C * 2 + 4 * T0 + 4 * ((T0 + 1) // 2 + r0) + (T0 - r0) * C * 2 + 4 * (T0 - r0))
        gbs = bytes_m / (ms_m / n_rep * 1e-3) / 1e9
        merge_roof["back_to_back"] = {"achieved": gbs, "frac": gbs / P["hbm"], "avg_launch_us": ms_m / n_rep * 1e3,
                                      "note": "layer-0 shape through the C ABI, 3 rotating input/output buffer sets (> L2), "
                                              "one event pair around 30 launches"}
        del sets

    out = None
    if rank == 0:
        fl = flops_per_sample(c, T0) * 3
        out = {
            "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": workload_config(a2, world, B, T0),
            "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / steps},
            "gpu_launches": launches, "clocks": clk.summary(), "roofline": roof, "merge_roofline": merge_roof,
            "kernels": kernels, "model_tflops": value / world * fl / 1e12,
            "model_frac_of_sustained_bf16_peak": value / world * fl / 1e12 / P["tf_sust"], "loss": loss_dev,
        }
        if from_pixels is not None:
            out["from_pixels"] = from_pixels
        if in_sync is not None:
            out["params_in_sync"] = in_sync
    del trainer, eng, x, y, xd, yd
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="tome_b200", choices=["tome_b200", "reference"])
    ap.add_argument("--config", default="octo_small", choices=list(CONFIGS),
                    help="octo_small = BASELINE.json configs[1] (the metric's configuration), octo_base = configs[2] per-GPU shard, "
                         "c3 = configs[3] (two cameras, 4-frame history, T0 = 2080; sweep it with --r)")
    ap.add_argument("--r", type=int, default=None, help="tokens merged per layer (default: the config's; configs[3] sweeps 0..64)")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override (default: the config's)")
    ap.add_argument("--dropout", type=float, default=0.1, help="hidden dropout rate (vanilla_decoder.yaml:17,50)")
    ap.add_argument("--attn-dropout", type=float, default=0.1, help="attention-weight dropout rate (vanilla_decoder.yaml:23)")
    ap.add_argument("--loss", default="continuous", choices=["continuous", "synthetic"],
                    help="continuous: ContinuousActionHead + l2 loss on the pooled readouts, the reference's "
                         "continuous_train_step; synthetic: MSE on the readout rows")
    ap.add_argument("--comm-sms", type=int, default=0,
                    help="N > 1: SMs reserved for the NCCL all-reduce kernels during backward (NCCL max_ctas = this, the "
                         "persistent GEMM grid shrinks by this); 0 = NCCL's default and the full grid")
    ap.add_argument("--overlap", default="none", choices=["layer", "none"],
                    help="gradient all-reduce: per-layer buckets overlapped with backward, or one all-reduce after backward")
    ap.add_argument("--compress", default="merge", choices=["merge", "prune"],
                    help="merge: ToMe bipartite soft matching + merge_wavg per layer (the metric's path); prune: the sibling path, "
                         "per-modality top-k pruning of r tokens per layer (compressed_attention.py / token_compression.py:15-46)")
    ap.add_argument("--from-pixels", default="auto", choices=["auto", "off"],
                    help="also time the step with its image tokens computed from uint8 frames by the image front end (sub-object "
                         "`from_pixels`; octo_small / octo_base sequences)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--octo-base", default="auto", choices=["auto", "on", "off"],
                    help="also measure the octo_base shard (BASELINE.json configs[2]) and attach it as `octo_base`; auto = at 8 GPUs")
    ap.add_argument("--microbench", action="store_true",
                    help="BASELINE.json configs[4]: standalone ToMe block kernels at 1k-8k tokens, d = 768 / 1024, merge-ratio "
                         "sweep, each against its roofline (one JSON object; N = 1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed train step computed to DIR/<name>.npy (float32): loss, head_out, readout, "
                         "and seeded samples of the updated params and of the grads; inputs are seeded, so two builds run "
                         "with the same arguments can be compared array by array")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "tome_b200" or args.microbench):
        ap.error("--dump-outputs applies to the train-step workload of --impl tome_b200")
    args.warmup = max(args.warmup, 3) if args.impl == "tome_b200" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    from multi_modal_transformers_tokenmerge_b200 import _lib as L
    from multi_modal_transformers_tokenmerge_b200.parallel import nccl_options

    L.lib()  # raises if the CUDA library is missing: the product path has no fallback
    # stdout carries exactly ONE JSON line: anything a library prints meanwhile (NCCL's version banner at N > 1) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    torch.cuda.set_device(local)
    if args.microbench:
        out = microbench(args) if rank == 0 else None
    else:
        if world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=torch.device("cuda", local), pg_options=nccl_options(args.comm_sms))
        out = measure_workload(args, args.config, rank, world, local, args.steps, args.warmup, dump_dir=args.dump_outputs)
        want_base = args.octo_base == "on" or (args.octo_base == "auto" and world == 8)
        if want_base and args.config == "octo_small":
            # BASELINE.json configs[2] (octo-base, batch 2048 over 8 GPUs) rides on the same line, so that the driver's scaling
            # run carries a measured number for it; fewer steps, same protocol
            a3 = argparse.Namespace(**{**vars(args), "r": None, "batch": 0})
            base = measure_workload(a3, "octo_base", rank, world, local, max(3, args.steps // 2), 3, with_extras=False)
            if out is not None:
                out["octo_base"] = {k_: base[k_] for k_ in ("value", "unit", "n_gpus", "steps", "ms_per_step", "config", "e2e", "roofline",
                                                            "kernels", "model_tflops", "model_frac_of_sustained_bf16_peak", "clocks")
                                    if k_ in base}
                if "params_in_sync" in base:
                    out["octo_base"]["params_in_sync"] = base["params_in_sync"]
        if out is not None and world == 1 and not args.no_cpu_baseline:
            c = cfg_of(args)
            sps, sec, cores, _ = cpu_reference_steps(args.config, 2, 1, REF_SAMPLE_BATCH if args.config != "c3" else 2, args.loss, r=c["r"],
                                                     dropout=args.dropout, attn_dropout=args.attn_dropout)
            out["cpu_baseline"] = {"value": sps, "unit": "samples/s", "cores": cores, "kind": "port",
                                   "sample": f"2 train steps (after 1 warm-up) of {REF_SAMPLE_BATCH if args.config != 'c3' else 2} samples of the "
                                             f"same workload (fp32, torch-CPU restatement of the reference, AdamW, same dropout sites), "
                                             f"{sec:.1f} s/step"}
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    if out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
