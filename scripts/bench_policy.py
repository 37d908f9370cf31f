"""Latency of one prediction from camera frames (closed-loop control: one observation per robot per tick), three arms alternated
call by call in one run:
  composed  ImageTokenizer.apply -> TokenSequence.assemble_embeddings -> predictor().predict   (the Python glue)
  fused     PixelPolicy.predict, eager                                                          (tome_policy_predict)
  graph     PixelPolicy.predict replayed from a CUDA graph
at B = 1, 8, 64, 256, octo-small and octo-base widths (12 layers, bench.py's r), continuous and diffusion heads, on the named
shape (two 256 x 256 x 3 uint8 frames per sample, 16-pixel patches, T0 = 536).  Each call is timed by CUDA events around it and
by a host clock around the call plus a synchronise; medians and the 10th / 90th percentiles over --calls calls after --warmup.
Also: predictions per second at B = 256 (B / median device latency), library launches per call (tome_launch_count, eager
arms), workspace bytes of both paths, whether the three arms' outputs are bitwise equal, and the card's name, power limit and
max SM clock read in the same run.  Usage: python scripts/bench_policy.py --out profiles/r04_policy.json"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench import CONFIGS, SEQ  # noqa: E402
from multi_modal_transformers_tokenmerge_b200 import _lib as L  # noqa: E402
from multi_modal_transformers_tokenmerge_b200 import model_configs  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.engine import StackConfig, ToMeStackEngine  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import TokenEmbeddings, TokenSequence  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def tokenizer(C):
    node = dict(model_configs.load("tokenizers/images/gato_resnet_octo")["encoder"])
    node.update(image_size=[256, 256, 3], patch_size=16, embedding_dim=C)
    for k in ("row_position_embedding", "col_position_embedding"):
        node[k] = dict(node[k], features=C)
    node["resnet"] = dict(node["resnet"], output_dense=dict(node["resnet"]["output_dense"], features=C))
    tok = model_configs.build_image_tokenizer(node)
    return tok, tok.init(3, None)


def stats(ms):
    a = np.asarray(ms)
    return {"median": float(np.median(a)), "p10": float(np.percentile(a, 10)), "p90": float(np.percentile(a, 90))}


def run(width, head, B, calls, warmup):
    c = CONFIGS[width]
    ts = TokenSequence(SEQ)
    gid, pos = ts.group_ids()
    allow, ro = ts.allow_table(), ts.get_modality_idx("readouts")
    C = c["channels"]
    hk = dict(head="continuous", head_features=7, max_action=1.0) if head == "continuous" else dict(
        head="diffusion", head_features=8, head_fourier_dim=C, head_time_hidden=C, head_time_out=C, head_hidden=2 * C, diffusion_steps=32)
    cfg = StackConfig(batch=B, tokens=ts.num_tokens, channels=C, heads=c["heads"], head_dim=c["head_dim"], mlp_dim=c["mlp_dim"],
                      layers=c["layers"], r=c["r"], ln_axis=1, num_groups=allow.shape[0], n_readout=len(ro), **hk)
    eng = ToMeStackEngine(cfg, gid=gid, pos=pos, allow=allow, readout_idx=ro, predict_only=True)
    eng.init_params(seed=1)
    tok, tv = tokenizer(C)
    pred = eng   # a predict-only engine: predict() is the composed path's last stage
    fused = eng.policy(tok, tv, ts)
    graphed = eng.policy(tok, tv, ts, graph=True)
    g = torch.Generator(device="cuda").manual_seed(B)
    frames = torch.randint(0, 256, (B, 2, 256, 256, 3), dtype=torch.uint8, device="cuda", generator=g)
    text = torch.randn(B, 16, C, device="cuda", generator=g).bfloat16()
    readouts = torch.randn(1, 8, C, device="cuda", generator=g).bfloat16()

    def composed():
        img = tok.apply(tv, frames, train=False).reshape(B, -1, C)
        x = ts.assemble_embeddings(TokenEmbeddings(text=text, images=img, readouts=readouts.expand(B, -1, -1))).contiguous()
        return pred.predict(x, rng=0)

    arms = {"composed": composed, "fused": lambda: fused.predict(frames, text, readouts, rng=0),
            "graph": lambda: graphed.predict(frames, text, readouts, rng=0)}
    first = {k: f() for k, f in arms.items()}
    torch.cuda.synchronize()
    bitwise = all(torch.equal(first["composed"][0], first[k][0]) and torch.equal(first["composed"][1], first[k][1]) for k in ("fused", "graph"))
    lib = L.lib()
    launches = {}
    for k in ("composed", "fused"):
        torch.cuda.synchronize()
        lib.tome_launch_count(1)
        arms[k]()
        launches[k] = int(lib.tome_launch_count(1))
    dev = {k: [] for k in arms}
    host = {k: [] for k in arms}
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(warmup + calls):
        for k, f in arms.items():   # the arms alternate call by call
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            if i >= warmup:
                dev[k].append(e0.elapsed_time(e1))
                host[k].append((t1 - t0) * 1e3)
    ws_composed = lib.tome_image_tokenizer_workspace_bytes(ctypes.byref(tok._desc(B, 2, torch.uint8, 1))) + pred._ws_bytes
    row = {"width": width, "head": head, "batch": B, "bitwise_equal_arms": bitwise, "launches_per_call": launches,
           "workspace_bytes": {"composed": int(ws_composed), "fused": int(fused._ws_bytes)},
           "device_ms": {k: stats(v) for k, v in dev.items()}, "host_ms": {k: stats(v) for k, v in host.items()}}
    if B == 256:
        row["predictions_per_s"] = {k: B / (row["device_ms"][k]["median"] * 1e-3) for k in arms}
    del fused, graphed, pred, eng, frames
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batches", default="1,8,64,256")
    ap.add_argument("--widths", default="octo_small,octo_base")
    ap.add_argument("--heads", default="continuous,diffusion")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_policy.py needs a GPU: latencies are not measured without one")
    out = {"metric": "latency of one prediction from pixels (two 256 x 256 x 3 uint8 frames per sample, T0 = 536)",
           "card": card(), "calls": a.calls, "warmup": a.warmup,
           "timing": "CUDA events around each call and a host clock around call + synchronise; arms alternated call by call",
           "rows": []}
    for width in a.widths.split(","):
        for head in a.heads.split(","):
            for B in [int(b) for b in a.batches.split(",")]:
                row = run(width, head, B, a.calls, a.warmup)
                d = row["device_ms"]
                print(f"{width} {head} B={B}: composed {d['composed']['median']:.3f} ms, fused {d['fused']['median']:.3f} ms, "
                      f"graph {d['graph']['median']:.3f} ms, bitwise {row['bitwise_equal_arms']}, launches {row['launches_per_call']}",
                      flush=True)
                out["rows"].append(row)
    s = json.dumps(out, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s)
    print(s[-2000:])


if __name__ == "__main__":
    main()
