"""Worker of tests/test_gpu_optimizer.py: one rank of a 2-GPU data-parallel run whose steps clip the gradient (launched by
torch.distributed.run).  Reports whether every rank saw the same norm bits and whether the replicas stayed identical."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_modal_transformers_tokenmerge_b200.engine import StackConfig, ToMeStackEngine  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.parallel import DataParallelTrainer  # noqa: E402
from multi_modal_transformers_tokenmerge_b200.tokenizers.token_sequencer import sequence_groups  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    gid, pos, allow, ro = sequence_groups("[TaskDescriptionPrefix{8}] [Image{40};Readout{2}]*2")
    B, T, C, A = 8, len(gid), 256, 8
    cfg = StackConfig(batch=B, tokens=T, channels=C, heads=4, head_dim=64, mlp_dim=512, layers=3, r=6, ln_axis=1,
                      num_groups=allow.shape[0], n_readout=len(ro), head="continuous", head_features=A, max_action=1.0)
    eng = ToMeStackEngine(cfg, gid=gid, pos=pos, allow=allow, readout_idx=ro)
    eng.init_params(seed=1)                                    # identical weights on every rank
    g = torch.Generator(device="cuda").manual_seed(7 + rank)   # a different shard on every rank
    x = torch.randn(B, T, C, device="cuda", generator=g).bfloat16()
    y = torch.rand(B, A, device="cuda", generator=g) * 2 - 1
    tr = DataParallelTrainer(eng, overlap=os.environ.get("TOME_DP_OVERLAP", "layer"))
    steps, clipped, equal = 4, 0, True
    max_norm = 1e-3                                            # far below the gradient's norm: every step clips
    for _ in range(steps):
        tr.train_step(x, y, lr=1e-3, max_grad_norm=max_norm, skip_nonfinite=True, decay="dense_kernels", weight_decay=0.1)
        bits = eng.grad_norm.view(torch.int32).to(torch.int64)
        lo, hi = bits.clone(), bits.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        equal &= bool(lo.item() == hi.item())
        clipped += int(eng.grad_norm.item() > max_norm)
    torch.cuda.synchronize()
    chk = eng.params.view(torch.int32).to(torch.int64).sum().reshape(1)
    lo, hi = chk.clone(), chk.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("DPCLIP " + json.dumps({"world": world, "overlap": tr.overlap, "steps": steps, "clipped_steps": clipped,
                                      "norm_bits_equal": equal, "params_in_sync": bool(lo.item() == hi.item()),
                                      "optimizer_steps": eng.optimizer_steps()}))
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
