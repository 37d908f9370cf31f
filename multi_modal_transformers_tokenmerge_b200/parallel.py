"""Data parallelism for the stack: batches shard across ranks (one process per GPU), parameters are replicated, and the
ONLY exchange on the path is the gradient all-reduce (the reference has no parallelism at all: SURVEY.md 2a, 8e).

The flat gradient vector is cut into one bucket per layer (plus the position embedding); the native backward records a
CUDA event as each layer's gradients become final (last layer first), and the bucket's all-reduce is issued on a side
stream behind that event, so NCCL traffic over NVLink overlaps the remaining backward kernels.
`GradBucketReducer` is device-agnostic so that the bucket logic is testable with gloo on CPU (tests/test_parallel.py).
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
import torch.distributed as dist


def layer_buckets(layer_offsets: Sequence[int], total: int) -> List[Tuple[int, int]]:
    """[(start, end)] in BACKWARD completion order: layer L-1, ..., layer 0, then the position embedding [0, off_0)."""
    L = len(layer_offsets)
    out = []
    for l in range(L - 1, -1, -1):
        end = layer_offsets[l + 1] if l + 1 < L else total
        out.append((layer_offsets[l], end))
    out.append((0, layer_offsets[0]))
    return out


class GradBucketReducer:
    def __init__(self, flat_grads: torch.Tensor, buckets: Sequence[Tuple[int, int]], group=None):
        self.flat = flat_grads
        self.buckets = list(buckets)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        covered = sorted(self.buckets)
        assert covered[0][0] == 0 and covered[-1][1] == flat_grads.numel(), "buckets must tile the gradient vector"
        for (a, b), (c, d) in zip(covered, covered[1:]):
            assert b == c, "buckets must tile the gradient vector"
        self.comm_stream = torch.cuda.Stream() if flat_grads.is_cuda else None

    def reduce(self, events: Optional[Sequence] = None) -> None:
        """Sum every bucket over the ranks.  `events[i]` (CUDA) gates bucket i; None = reduce right away."""
        if self.world == 1:
            return
        if self.comm_stream is None:
            for a, b in self.buckets:
                dist.all_reduce(self.flat[a:b], op=dist.ReduceOp.SUM, group=self.group)
            return
        main = torch.cuda.current_stream()
        with torch.cuda.stream(self.comm_stream):
            if events is None:
                self.comm_stream.wait_stream(main)
            for i, (a, b) in enumerate(self.buckets):
                if events is not None:
                    self.comm_stream.wait_event(events[i])
                dist.all_reduce(self.flat[a:b], op=dist.ReduceOp.SUM, group=self.group)
        main.wait_stream(self.comm_stream)


def nccl_options(max_ctas: int):
    """ProcessGroupNCCL options capping the CTAs (= SMs) one collective may occupy; None when max_ctas == 0."""
    if not max_ctas:
        return None
    opts = dist.ProcessGroupNCCL.Options()
    opts.config.max_ctas = int(max_ctas)
    opts.config.min_ctas = 1
    return opts


class DataParallelTrainer:
    """forward + backward + overlapped gradient all-reduce + AdamW for one rank's shard of the batch."""

    def __init__(self, engine, group=None, comm_sms: int = 0, overlap: str = "none"):
        """overlap: "none" (default) -- ONE all-reduce over the whole gradient vector after backward; "layer" -- one bucket per
        layer, reduced on a side stream as soon as backward has finished that layer.  The persistent 148-CTA GEMM grids cannot
        share an SM with an NCCL CTA, so every GEMM launched under a running collective waits for it on those SMs; the whole
        octo-small gradient vector (87 MB fp32) takes 0.35 ms over NVSwitch at N = 8 (octo-base: 0.89 ms), less than the stalls
        cost: 33.66 ms per step against 34.69 with per-layer overlap and 33.83 at N = 1 on the same box
        (profiles/r02_scaling.md).
        comm_sms > 0: SMs left to the NCCL kernels while backward runs (the persistent GEMM grid shrinks by that many;
        pair it with an NCCL CTA cap of the same size, see `nccl_options`)."""
        assert overlap in ("layer", "none")
        self.engine = engine
        self.overlap = overlap
        self.comm_sms = int(comm_sms) if overlap == "layer" else 0
        offs = [engine.layer_offset(l) for l in range(engine.cfg.layers)]
        self.reducer = GradBucketReducer(engine.grads, layer_buckets(offs, engine.n_params), group)
        self.world = self.reducer.world
        # one event per layer (recorded by the native backward in layer order L-1..0) + one for the position embedding
        self.events = [torch.cuda.Event() for _ in range(engine.cfg.layers + 1)]
        for ev in self.events:  # torch creates the CUDA event lazily; the native backward needs real handles
            ev.record()

    def train_step(self, x: torch.Tensor, target: torch.Tensor, lr: float = 1e-4, **adam) -> None:
        """`adam` goes to `engine.adamw_step` (max_grad_norm, skip_nonfinite, decay, ...).  The step runs after the
        all-reduce with grad_scale = 1/world, so its norm is the norm of the mean gradient and every rank computes the
        same bits from the same reduced vector."""
        e = self.engine
        e.zero_grad()
        e.set_dropout_step(e.step_count)   # fresh dropout masks every step (forward and backward of a step share them)
        e.forward(x, target)
        if self.world > 1 and self.overlap == "none":
            e.backward()
            dist.all_reduce(e.grads, op=dist.ReduceOp.SUM, group=self.reducer.group)
        elif self.world > 1:
            if self.comm_sms:
                e.lib.tome_gemm_set_sm_limit(int(e.lib.tome_num_sms()) - self.comm_sms)
            e.backward(events=self.events)  # events[l] <- layer l done; events[L] <- everything done
            if self.comm_sms:
                e.lib.tome_gemm_set_sm_limit(0)
            L = e.cfg.layers
            order = [self.events[l] for l in range(L - 1, -1, -1)] + [self.events[L]]
            self.reducer.reduce(order)
        else:
            e.backward()
        e.adamw_step(lr=lr, grad_scale=1.0 / self.world, **adam)
