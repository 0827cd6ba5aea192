"""Mixed-precision step of the cfg3 layer: Shift2d forward + backward, N=256 C=256 56x56, zeros padding.

Times, for the sparse and the active shift, one training step of the layer (forward, then backward with grad_input and
grad_weight) in three precisions:

  fp32   x, grad, weights fp32 (the project's fp32 baseline)
  mixed  x, grad bf16, weights and grad_weight fp32 (TS_WEIGHTS_F32: the 16-bit TMA kernels)
  bf16   x, grad, weights bf16 (what a user had before mixed precision: ``Shift2d(...).bfloat16()``)

against the measured copy peak: ``torch.Tensor.copy_`` of a dense bf16 tensor of the same size (one read + one write).
Algorithmic bytes of a step: forward reads x and writes y, backward reads grad and x and writes grad_input -- five
passes over the tensor at the element size (the weights and partials are negligible).  Every tensor is larger than L2.
Times are CUDA-event times over --steps steps after --warmup steps; the card's name and power limit are printed with them.

    python tools/amp_bench.py [--steps 50] [--warmup 10] [--out profiles/amp_bench_b200.json]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
for p in (str(ROOT), str(ROOT / "activesparseshifts-pytorch_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

N, C, H, W = 256, 256, 56, 56
PATHS = {0: "none", 1: "generic", 2: "staged", 3: "tma", 4: "nhwc", 5: "halo", 6: "flat"}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name()


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", type=str, default=None, help="also write the JSON result here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("amp_bench: needs a CUDA device (B200); there is no CPU measurement")
    import torchshifts  # noqa: F401  (registers torch.ops.torchshifts)
    from torchshifts.extension import native
    lib = native().lib
    lib.ts_set_kernel_path(0)
    dev = torch.device("cuda")
    torch.manual_seed(0)
    numel = N * C * H * W
    borders = torch.tensor([0, H, 0, W, 0, 1], dtype=torch.int32)
    fwd, bwd = torch.ops.torchshifts._shift2d_forward, torch.ops.torchshifts._shift2d_backward

    x32 = torch.randn(N, C, H, W, device=dev)
    g32 = torch.randn(N, C, H, W, device=dev)
    w32 = (torch.rand(C, 2, device=dev) * 6 - 3)
    xb, gb = x32.bfloat16(), g32.bfloat16()
    del x32, g32
    torch.cuda.empty_cache()
    copy_dst = torch.empty_like(xb)
    copy_ms = time_ms(lambda: copy_dst.copy_(xb), args.steps, args.warmup)
    del copy_dst
    copy_gbs = 2 * numel * 2 / copy_ms / 1e6
    result = {"config": f"cfg3 Shift2d N={N} C={C} {H}x{W} zeros padding, forward + backward", "card": card(),
              "steps": args.steps, "warmup": args.warmup,
              "copy_peak": {"ms": round(copy_ms, 4), "GBps": round(copy_gbs, 1),
                            "what": "copy_ of a dense bf16 tensor of the layer's size (read + write)"},
              "runs": []}
    for active in (False, True):
        for name in ("fp32", "mixed", "bf16"):
            if name == "fp32":
                x, g, w = xb.float(), gb.float(), w32
            else:
                x, g, w = xb, gb, (w32 if name == "mixed" else w32.bfloat16())
            es = x.element_size()
            new = [N, C, H, W]
            fwd(x, w, borders, new, 0, active)
            fpath = PATHS.get(lib.ts_last_kernel_path())
            bwd(g, w, x, borders, 0, active)
            bpath = PATHS.get(lib.ts_last_kernel_path())
            f_ms = time_ms(lambda: fwd(x, w, borders, new, 0, active), args.steps, args.warmup)
            b_ms = time_ms(lambda: bwd(g, w, x, borders, 0, active), args.steps, args.warmup)
            s_ms = time_ms(lambda: (fwd(x, w, borders, new, 0, active), bwd(g, w, x, borders, 0, active)), args.steps, args.warmup)
            gi, gw = bwd(g, w, x, borders, 0, active)
            step_bytes = 5 * numel * es
            gbs = step_bytes / s_ms / 1e6
            result["runs"].append({
                "shift": "active" if active else "sparse", "precision": name, "x": str(x.dtype), "weights": str(w.dtype),
                "grad_weight": str(gw.dtype), "forward_family": fpath, "backward_family": bpath,
                "forward_ms": round(f_ms, 4), "backward_ms": round(b_ms, 4), "step_ms": round(s_ms, 4),
                "step_GBps": round(gbs, 1), "of_copy_peak": round(gbs / copy_gbs, 3),
                "of_7.7TBps_datasheet": round(gbs / 7700.0, 3)})
            del gi, gw
            if name == "fp32":
                del x, g
                torch.cuda.empty_cache()
    line = json.dumps(result, indent=1)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
