#!/usr/bin/env python
"""Multi-rank check of the in-kernel grad_weight all-reduce through the channels-last backward
(ts_shift_backward_nhwc with a peer group) against torch.distributed's NCCL all-reduce of the plain
channels-last backward.  Run under torchrun on 2..8 GPUs:
    timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/cl_fused_probe.py
`tests/test_channels_last_float.py::test_fused_exchange_two_ranks` runs it on 2 GPUs."""
import os
import sys
from pathlib import Path

import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "activesparseshifts-pytorch_b200")]
import torchshifts  # noqa: E402,F401
from torchshifts.extension import native  # noqa: E402
from torchshifts.functional import shift2d_func  # noqa: E402
from torchshifts.sharded import FusedGradWeightAllReduce  # noqa: E402

local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
dist.init_process_group("nccl", device_id=dev)
rank, world = dist.get_rank(), dist.get_world_size()
fused = FusedGradWeightAllReduce(capacity=4096, device=dev)
CL = torch.channels_last
ok = True
for it, (shape, dtype, pad, active) in enumerate([((8, 64, 32, 32), torch.float32, 0, False), ((8, 256, 28, 28), torch.float32, 3, True),
                                                  ((4, 128, 16, 20), torch.bfloat16, 2, True)]):
    torch.manual_seed(100 * it + rank)
    x = torch.randn(shape, device=dev).to(dtype).contiguous(memory_format=CL).requires_grad_(True)
    g = torch.randn(shape, device=dev).to(dtype).contiguous(memory_format=CL)
    torch.manual_seed(it)
    w = ((torch.rand(shape[1], 2, device=dev) * 2 - 1) * 2).to(dtype).requires_grad_(True)
    shift2d_func(x, w, pad, active, memory_format=torch.preserve_format).backward(g)
    ref = w.grad.float()
    dist.all_reduce(ref)
    gi_plain = x.grad.clone()
    x.grad = None; w.grad = None
    with fused:
        shift2d_func(x, w, pad, active, memory_format=torch.preserve_format).backward(g)
    served = native().lib.ts_last_kernel_path() == 4
    err = float((w.grad.float() - ref).abs().max() / ref.abs().max().clamp_min(1e-30))
    same = [torch.empty_like(w.grad) for _ in range(world)]
    dist.all_gather(same, w.grad.contiguous())
    identical = all(torch.equal(same[0], t) for t in same)
    tol = 1e-5 if dtype is torch.float32 else 1e-2
    case_ok = served and err < tol and identical and torch.equal(x.grad, gi_plain)
    if rank == 0:
        print(f"case {it} {shape} {dtype} pad {pad} active {active}: NHWC kernel {served}, max rel err vs NCCL {err:.2e}, "
              f"identical on all ranks {identical}", flush=True)
    ok = ok and case_ok
flag = torch.tensor([1 if ok else 0], device=dev)
dist.all_reduce(flag, op=dist.ReduceOp.MIN)
if rank == 0:
    print("PROBE", "OK" if int(flag.item()) else "FAILED", flush=True)
dist.destroy_process_group()
sys.exit(0 if int(flag.item()) else 1)
