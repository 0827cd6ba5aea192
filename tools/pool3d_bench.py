#!/usr/bin/env python
"""Shift3d emulating a strided depth-wise convolution (modules/shifts.py:85-89) on the cfg4 tensor (32, 128, 16, 56, 56):
the fused operators (shift + crop + avg_pool3d in one kernel forward; the pooling adjoint applied while the gradient is staged
backward) against the two-step path (shift op + ATen avg_pool3d and their backwards), timed in the same run, alternating.

Per case: forward, backward and step (forward + backward) times of both paths from CUDA events after warm-up (median of
rounds), the traffic floor of the fused layer (forward: x + pooled y; backward: x + pooled grad + grad_input) over the run's
own measured copy_ rate, the plain 3-D shift forward / backward of the same case as context, and once the peak memory of a
training step of both layers.  Every tensor is larger than the L2 cache.  The GPU's name, power limit and SM clock are
read in the same run.  Writes one JSON file (--out)."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "activesparseshifts-pytorch_b200")]
import torchshifts  # noqa: E402
from torchshifts.functional import shift3d_func  # noqa: E402

ops = torch.ops.torchshifts
SHAPE = (32, 128, 16, 56, 56)
CASES = [("zeros", 0, False), ("zeros", 0, True), ("reflect", 3, True)]
CROPS = {"none": [[0, 0], [0, 0], [0, 0]], "crop": [[1, 1], [2, 2], [4, 4]]}     # crop: output 14 x 52 x 48


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except (OSError, IndexError, subprocess.SubprocessError):
        return {"name": torch.cuda.get_device_name(0)}


def timer(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def alternate(fns, reps, rounds):
    """fns: name -> callable; every round times each once, in turn -> name -> median ms"""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    got = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            got[k].append(timer(f, reps))
    return {k: sorted(v)[len(v) // 2] for k, v in got.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "pool3d_bench_b200.json"))
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=7)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "pool3d_bench measures on a CUDA device"
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    x = torch.randn(SHAPE, device=dev)
    with torch.no_grad():
        dst = torch.empty_like(x)
        copy_ms = alternate({"copy": lambda: dst.copy_(x)}, args.reps, args.rounds)["copy"]
    del dst
    peak = 2 * x.numel() * 4 / (copy_ms * 1e-3)
    result = {"gpu": gpu_info(), "shape": list(SHAPE), "copy_rate_GBps": peak / 1e9, "cases": []}
    print(json.dumps(result["gpu"]), f"copy_ rate {peak / 1e9:.0f} GB/s", flush=True)
    for st in ((1, 2, 2), (2, 2, 2)):
        for crop_name, cuts in CROPS.items():
            lb = [c[0] for c in cuts]
            rb = [s - c[1] for s, c in zip(SHAPE[2:], cuts)]
            std = torch.tensor([lb[0], rb[0], lb[1], rb[1], lb[2], rb[2]], dtype=torch.int32)
            new_size = list(SHAPE[:2]) + [r - l for l, r in zip(lb, rb)]
            pooled = list(SHAPE[:2]) + [-(-o // s) for o, s in zip(new_size[2:], st)]
            gp = torch.randn(pooled, device=dev)
            gfull = torch.randn(new_size, device=dev)
            like = torch.empty(new_size, device=dev)
            for pad_name, pad, active in CASES:
                w = (torch.rand(SHAPE[1], 3, device=dev) * 2 - 1) * 2

                def f_fused():
                    return ops._shift3d_avgpool_forward(x, w, std, new_size, list(st), pad, active)

                def f_two():
                    return torch.nn.functional.avg_pool3d(ops._shift3d_forward(x, w, std, new_size, pad, active), st, st, ceil_mode=True)

                def b_fused():
                    return ops._shift3d_avgpool_backward(gp, w, x, std, new_size, list(st), pad, active)

                def b_two():
                    gy = torch.ops.aten.avg_pool3d_backward(gp, like, list(st), list(st), [0, 0, 0], True, True, None)
                    return ops._shift3d_backward(gy, w, x, std, pad, active)
                with torch.no_grad():
                    assert torch.equal(f_fused(), f_two())
                    assert torch.equal(b_fused()[0], b_two()[0])
                    t = alternate({"fwd_fused": f_fused, "fwd_two_step": f_two, "bwd_fused": b_fused, "bwd_two_step": b_two,
                                   "step_fused": lambda: (f_fused(), b_fused()), "step_two_step": lambda: (f_two(), b_two()),
                                   "fwd_plain_shift": lambda: ops._shift3d_forward(x, w, std, new_size, pad, active),
                                   "bwd_plain_shift": lambda: ops._shift3d_backward(gfull, w, x, std, pad, active)},
                                  args.reps, args.rounds)
                xb, pb = x.numel() * 4, gp.numel() * 4
                floor_f, floor_b = (xb + pb) / peak * 1e3, (2 * xb + pb) / peak * 1e3     # ms at the copy_ rate
                case = {"stride": list(st), "crop": crop_name, "padding": pad_name, "active": active, "ms": t,
                        "floor_ms": {"fwd": floor_f, "bwd": floor_b},
                        "floor_share": {"fwd": floor_f / t["fwd_fused"], "bwd": floor_b / t["bwd_fused"]},
                        "speedup": {k: t[f"{k}_two_step"] / t[f"{k}_fused"] for k in ("fwd", "bwd", "step")}}
                result["cases"].append(case)
                print(f"stride {st} {crop_name:4s} {pad_name:7s} active={int(active)}: fwd {t['fwd_fused']:.3f} / {t['fwd_two_step']:.3f} ms"
                      f" (plain shift {t['fwd_plain_shift']:.3f}, floor share {case['floor_share']['fwd']:.2f})  bwd {t['bwd_fused']:.3f} /"
                      f" {t['bwd_two_step']:.3f} ms (plain shift {t['bwd_plain_shift']:.3f}, floor share {case['floor_share']['bwd']:.2f})"
                      f"  step {t['step_fused']:.3f} / {t['step_two_step']:.3f} ms", flush=True)
            del gp, gfull, like
    # peak memory of one training step: reflect active, stride (2, 2, 2)
    m = torchshifts.Shift3d(SHAPE[1], padding="reflect", active_flag=True, sparsity_term=0,
                            emulate_dw={"kernel_size": 3, "stride": 2, "padding": 1}).to(dev)
    xr = x.clone().requires_grad_(True)

    def peak_mem(step):
        xr.grad, m.weight.grad = None, None
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        step()
        torch.cuda.synchronize()
        return (torch.cuda.max_memory_allocated() - base) / 2**20

    def fused():
        m(xr)[0].sum().backward()

    def two_step():
        torch.nn.functional.avg_pool3d(shift3d_func(xr, m.weight, 3, True), 2, 2, ceil_mode=True).sum().backward()
    fused(), two_step()
    result["peak_memory_MiB"] = {"fused": peak_mem(fused), "two_step": peak_mem(two_step), "full_tensor": x.numel() * 4 / 2**20}
    print("peak memory of a training step (MiB):", json.dumps(result["peak_memory_MiB"]), flush=True)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
