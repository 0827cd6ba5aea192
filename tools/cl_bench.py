#!/usr/bin/env python
"""Channels-last float Shift2d on the GPU: the preserving path (memory_format=torch.preserve_format, native NHWC kernels)
against today's path for a channels-last network (planar kernels + layout passes), cfg3-shaped N=256 C=256 56x56.

    python tools/cl_bench.py [--out DIR]

Timed with CUDA events after warm-up; every tensor is larger than the 126 MB L2.  Algorithmic bytes: 2e for a forward
(read x, write y), 3e for a backward (read grad and x, write grad_input), 5e for a training step, e = tensor bytes.  The
copy-peak denominator is this run's own torch copy of a tensor of the same size (read + write = 2e).
  forward: no autograd.  Today = shift2d_func on the channels-last x (ts_nhwc_to_nchw, planar kernel), then
           y.contiguous(channels_last).
  step:    autograd forward + torch.autograd.grad with a channels-last grad, as in training.  Today's backward reuses the
           planar copy of x its forward made (so x is converted once per step), converts grad to planar and grad_input
           back to channels-last.  backward = step - forward (derived).
Then, for the new path only: device time per kernel from torch.profiler (kernel vs pass 2), the same kernels under the
staging knobs cl_ahead (steps of copies in flight) and cl_rows (rows per step), and with all weights 0 (every lane reads
the same pixel: the cost of the per-channel gather itself).  Writes cl_bench.json under --out (default: a temp dir)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT), str(ROOT / "activesparseshifts-pytorch_b200")]
from torchshifts.extension import native  # noqa: E402
from torchshifts.functional import shift2d_func  # noqa: E402

CL = torch.channels_last
ap = argparse.ArgumentParser()
ap.add_argument("--out", default=None)
ap.add_argument("--reps", type=int, default=30)
args = ap.parse_args()
assert torch.cuda.is_available(), "tools/cl_bench.py measures on the GPU"
dev = torch.device("cuda:0")
lib = native().lib


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def timed(body, reps):
    for _ in range(5):
        body()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        body()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


N, C, H, W = 256, 256, 56, 56
rows, kernels = [], []
info = gpu_info()
print(f"GPU: {info}")


def step(fn, x, w, g):
    xr = x.detach().requires_grad_(True)
    wr = w.detach().requires_grad_(True)
    return lambda: torch.autograd.grad(fn(xr, wr), (xr, wr), g)


def kernel_times(body, reps=10):
    from torch.profiler import ProfilerActivity, profile
    body()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            body()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count:
            name = ev.key.split("<")[0].split("::")[-1].split("(")[0]
            t = getattr(ev, "device_time_total", None) or ev.cuda_time_total
            out[name] = out.get(name, 0.0) + t / 1000.0 / reps
    return out


for dtype in (torch.float32, torch.bfloat16):
    torch.manual_seed(0)
    x = torch.randn(N, C, H, W, device=dev).to(dtype).contiguous(memory_format=CL)
    g = torch.randn(N, C, H, W, device=dev).to(dtype).contiguous(memory_format=CL)
    w = ((torch.rand(C, 2, device=dev) * 2 - 1) * 2).to(dtype)
    e = x.numel() * x.element_size()
    dst = torch.empty_like(x)
    t_copy = timed(lambda: dst.copy_(x), args.reps)
    peak = 2 * e / t_copy / 1e6                                   # GB/s
    rows.append(dict(dtype=str(dtype), what="torch copy (copy-peak denominator)", ms=t_copy, gbs=peak, share=1.0))
    for pad, active in ((0, False), (3, True)):
        new = lambda a, b: shift2d_func(a, b, pad, active, memory_format=torch.preserve_format)        # noqa: E731
        old = lambda a, b: shift2d_func(a, b, pad, active).contiguous(memory_format=CL)                # noqa: E731
        (gi_new, gw_new), (gi_old, gw_old) = step(new, x, w, g)(), step(old, x, w, g)()
        gi_old = gi_old.contiguous(memory_format=CL)
        same = bool(torch.equal(new(x, w), old(x, w)) and torch.equal(gi_new, gi_old))
        assert gi_new.is_contiguous(memory_format=CL) and lib.ts_last_kernel_path() != 4
        step(new, x, w, g)()
        assert lib.ts_last_kernel_path() == 4
        del gi_new, gi_old, gw_new, gw_old
        t = {}
        with torch.no_grad():
            t["fwd_new"], t["fwd_old"] = timed(lambda: new(x, w), args.reps), timed(lambda: old(x, w), args.reps)
        s_new, s_old = step(new, x, w, g), step(old, x, w, g)
        s_old_cl = lambda: s_old()[0].contiguous(memory_format=CL)                                      # noqa: E731
        t["step_new"], t["step_old"] = timed(s_new, args.reps), timed(s_old_cl, args.reps)
        for what, ms, nbytes in (("forward, preserving (NHWC kernel)", t["fwd_new"], 2 * e),
                                 ("forward, today (planar + layout passes)", t["fwd_old"], 2 * e),
                                 ("step fwd+bwd, preserving", t["step_new"], 5 * e),
                                 ("step fwd+bwd, today", t["step_old"], 5 * e),
                                 ("backward, preserving (step - forward)", t["step_new"] - t["fwd_new"], 3 * e),
                                 ("backward, today (step - forward)", t["step_old"] - t["fwd_old"], 3 * e)):
            gbs = nbytes / ms / 1e6
            rows.append(dict(dtype=str(dtype), pad=pad, active=active, what=what, ms=ms, gbs=gbs, share=gbs / peak, same_values=same))
        # the new path's kernels: profiler device times, staging knobs, zero shifts
        std = torch.tensor([0, H, 0, W, 0, 1], dtype=torch.int32)
        fwd_op = lambda ww: torch.ops.torchshifts._shift2d_forward_cl(x, ww, std, [N, C, H, W], pad, active)    # noqa: E731
        bwd_op = lambda ww: torch.ops.torchshifts._shift2d_backward_cl(g, ww, x, std, pad, active)              # noqa: E731
        for knobs in ("", "cl_ahead=1", "cl_ahead=3", "cl_ahead=4", "cl_rows=1", "cl_ahead=3,cl_rows=1", "cl_ahead=4,cl_rows=1"):
            assert lib.ts_set_tuning((knobs or "cl_ahead=0").encode()) == 0
            for ww, wname in ((w, "weights U(-2,2)"), (torch.zeros_like(w), "weights 0")):
                if wname == "weights 0" and knobs:
                    continue
                kt = kernel_times(lambda: fwd_op(ww))
                kt.update(kernel_times(lambda: bwd_op(ww)))
                if lib.ts_last_kernel_path() != 4:      # the window these knobs leave is too small for the shape
                    continue
                kernels.append(dict(dtype=str(dtype), pad=pad, active=active, knobs=knobs or "default (cl_ahead=2, cl_rows=2)",
                                    weights=wname, ms={k: round(v, 4) for k, v in kt.items()}))
        lib.ts_set_tuning(b"cl_ahead=0,cl_rows=0")
for r in rows:
    extra = f" pad={r['pad']} active={r['active']}" if "pad" in r else ""
    print(f"{r['dtype']:>15}{extra:>22}  {r['what']:<42} {r['ms']:8.4f} ms {r['gbs']:8.0f} GB/s  {100 * r['share']:5.1f} % of copy"
          + (f"  same values as today: {r['same_values']}" if "same_values" in r else ""))
for k in kernels:
    print(f"{k['dtype']:>15} pad={k['pad']} active={k['active']!s:<5} {k['knobs']:<32} {k['weights']:<16} "
          + "  ".join(f"{n} {v:.4f} ms" for n, v in sorted(k["ms"].items())))
out = Path(args.out) if args.out else Path(tempfile.mkdtemp())
out.mkdir(parents=True, exist_ok=True)
(out / "cl_bench.json").write_text(json.dumps(dict(gpu=info, shape=[N, C, H, W], rows=rows, kernels=kernels), indent=1))
print(f"wrote {out / 'cl_bench.json'}")
