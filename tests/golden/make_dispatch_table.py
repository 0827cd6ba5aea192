#!/usr/bin/env python
"""Generate tests/golden/dispatch_table.json.xz: which kernel family each C entry point picks, and what it returns, for
every kernel-path override and family knob, by calling the C ABI directly on torch-allocated device buffers.

    python tests/golden/make_dispatch_table.py [--out PATH]      # needs the GPU

Cases: ts_shift_forward, ts_shift_backward, ts_shift_backward_allreduce (one rank, FusedGradWeightAllReduce's buffers),
ts_qshift_forward (1- and 4-byte elements, zero point 0 and 3), both ts_shift2d_avgpool2_* and both float NHWC entries;
forced path 0/1/2/3/5/6 x the use_tma / use_halo / use_flat sets of KNOBS; dims 1-3, all paddings, sparse and active,
fp32/fp64/fp16/bf16; the GEOMETRIES below, picked so that every family both plans and declines.

Stored per case, a string of three-digit codes, one per steering (FORCED x KNOBS, in that order): the returned status, then
ts_last_kernel_path() after the call, then the ts_launch_count() delta.  ts_last_kernel_path() keeps its value over a call
that launches nothing, so the codes hold only when the cases run in the order run_table() runs them.  Per geometry and
dtype, ts_shift_backward_workspace_bytes() under each knob set.  tests/test_dispatch_table.py replays the table.  The JSON
is stored xz-compressed (about 650 KB of text, 8 KB compressed); `xz -dc` or load() prints it.
"""
import json
import lzma
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
for p in (str(ROOT), str(ROOT / "activesparseshifts-pytorch_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

SEED = 11
FORCED = (0, 1, 2, 3, 5, 6)
KNOBS = {"all": b"use_tma=1,use_halo=1,use_flat=1", "no_tma": b"use_tma=0,use_halo=1,use_flat=1",
         "no_halo": b"use_tma=1,use_halo=0,use_flat=1", "no_flat": b"use_tma=1,use_halo=1,use_flat=0",
         "none": b"use_tma=0,use_halo=0,use_flat=0"}
DTYPES = ("f32", "f64", "f16", "bf16")          # TS_F32 .. TS_BF16
QBYTES = (1, 4)
QZERO = (0, 3)                                  # the TMA family takes zero points of 0 only
PADDINGS = range(5)

# name -> (shape, borders: (lb, rb) per axis or None, x sliced out of a wider tensor along its last axis)
GEOMETRIES = {
    "1d": ((4, 8, 64), None, False),
    "1d_odd": ((3, 5, 7), None, False),                             # rows not a multiple of 16 bytes
    "1d_size1": ((2, 4, 1), None, False),
    "1d_crop": ((4, 8, 64), [(3, 60)], False),
    "1d_c520": ((1, 520, 32), None, False),                         # more channels than TABLE_MAX_C
    "1d_sliced": ((4, 8, 64), None, True),
    "1d_n0": ((0, 8, 64), None, False),
    "2d": ((4, 8, 32, 32), None, False),
    "2d_c32": ((2, 32, 8, 16), None, False),                        # the NHWC float kernels serve C % 32 == 0
    "2d_c32_crop": ((2, 32, 8, 16), [(1, 7), (2, 16)], False),
    "2d_odd": ((3, 5, 7, 9), None, False),
    "2d_size1": ((2, 4, 1, 32), None, False),
    "2d_crop": ((4, 8, 32, 32), [(1, 31), (2, 30)], False),
    "2d_c520": ((1, 520, 8, 16), None, False),
    "2d_sliced": ((4, 8, 32, 32), None, True),
    "2d_small": ((2, 4, 8, 8), None, False),                        # halo plane below 128 pairs: the unforced plan declines
    "2d_n0": ((0, 8, 32, 32), None, False),
    "3d": ((2, 4, 8, 16, 16), None, False),
    "3d_odd": ((2, 3, 3, 5, 7), None, False),
    "3d_size1": ((2, 4, 1, 8, 16), None, False),
    "3d_crop": ((2, 4, 8, 16, 16), [(1, 7), (0, 15), (2, 16)], False),
    "3d_c520": ((1, 520, 2, 4, 8), None, False),
    "3d_sliced": ((2, 4, 8, 16, 16), None, True),
    "3d_small": ((1, 2, 4, 4, 4), None, False),
    "3d_n0": ((0, 4, 8, 16, 16), None, False),
}
PLANAR_OPS = ("fwd", "bwd", "bwd_allreduce")
TWO_D_OPS = ("pool_fwd", "pool_bwd", "nhwc_fwd", "nhwc_bwd")      # 2-D only: run for other dims on one geometry each


def _geometry(shape, strides, borders):
    from torchshifts._cabi import make_geometry
    dim = len(shape) - 2
    lb = [b[0] for b in borders] if borders else [0] * dim
    rb = [b[1] for b in borders] if borders else list(shape[2:])
    return make_geometry(dim, shape, strides, lb + [0] * (3 - dim), rb + [1] * (3 - dim))


def _out_shape(shape, borders):
    return tuple(shape[:2]) + (tuple(b[1] - b[0] for b in borders) if borders else tuple(shape[2:]))


def _tensor(torch, gen, shape, dtype, sliced, dev):
    """Seeded values in [-4, 4) of `dtype`; sliced: a view of the first shape[-1] columns of a wider tensor."""
    full = list(shape[:-1]) + [shape[-1] + 3 if sliced else shape[-1]]
    t = ((torch.rand(full, generator=gen) * 8 - 4).to(dtype) if dtype.is_floating_point
         else torch.randint(0, 100, full, generator=gen).to(dtype))
    t = t.to(dev)
    return t[..., :shape[-1]] if sliced else t


class _Buffers:
    """The device buffers of one geometry and element type, and the ts_geometry of x (planar and, for dense 2-D,
    channels-last)."""

    def __init__(self, torch, lib, gen, dev, shape, borders, sliced, dtype, code):
        import ctypes as ct
        dim = len(shape) - 2
        out = _out_shape(shape, borders)
        self.x = _tensor(torch, gen, shape, dtype, sliced, dev)
        self.geo = _geometry(shape, self.x.stride(), borders)
        self.y = torch.zeros(out, dtype=dtype, device=dev)
        self.gi = torch.zeros(shape, dtype=dtype, device=dev)
        if dtype.is_floating_point:
            self.w = _tensor(torch, gen, (shape[1], dim), dtype, False, dev)
            self.grad = _tensor(torch, gen, out, dtype, False, dev)
            self.gw = torch.zeros((shape[1], dim), dtype=dtype, device=dev)
            ws = 16
            for spec in KNOBS.values():
                lib.ts_set_tuning(spec)
                ws = max(ws, int(lib.ts_shift_backward_workspace_bytes(ct.byref(self.geo), code)))
            self.ws = torch.zeros(ws, dtype=torch.uint8, device=dev)
            cl = dim == 2 and not sliced
            fmt = torch.channels_last if cl else torch.contiguous_format
            self.x_cl = self.x.contiguous(memory_format=fmt)
            self.geo_cl = _geometry(shape, self.x_cl.stride(), borders)
            self.y_cl = self.y.contiguous(memory_format=fmt)
            self.grad_cl = self.grad.contiguous(memory_format=fmt)
            self.gi_cl = self.gi.contiguous(memory_format=fmt)
            self.ws_cl = torch.zeros(max(16, int(lib.ts_shift_backward_nhwc_workspace_bytes(ct.byref(self.geo_cl), code))),
                                     dtype=torch.uint8, device=dev)
        else:
            self.w = torch.randint(-4, 5, (shape[1], dim), generator=gen, dtype=torch.int8).to(dev)


def _call(lib, op, b, code, pad, flag, peers):
    """code: the dtype, or the element bytes of qfwd; flag: active, or the zero point of qfwd."""
    import ctypes as ct
    geo, a = ct.byref(b.geo), int(flag)
    if op == "qfwd":      # int8 weights (TS_QW_I8) with zero point 0
        return lib.ts_qshift_forward(geo, code, pad, a, b.x.data_ptr(), b.w.data_ptr(), 1, 0, b.y.data_ptr(), None)
    if op == "fwd":
        return lib.ts_shift_forward(geo, code, pad, a, b.x.data_ptr(), b.w.data_ptr(), b.y.data_ptr(), None)
    if op == "pool_fwd":
        return lib.ts_shift2d_avgpool2_forward(geo, code, pad, a, b.x.data_ptr(), b.w.data_ptr(), b.y.data_ptr(), None)
    if op == "nhwc_fwd":
        return lib.ts_shift_forward_nhwc(ct.byref(b.geo_cl), code, pad, a, b.x_cl.data_ptr(), b.w.data_ptr(), b.y_cl.data_ptr(),
                                         None)
    if op == "nhwc_bwd":
        return lib.ts_shift_backward_nhwc(ct.byref(b.geo_cl), code, pad, a, b.grad_cl.data_ptr(), b.x_cl.data_ptr(), b.w.data_ptr(),
                                          b.gi_cl.data_ptr(), b.gw.data_ptr(), b.ws_cl.data_ptr(), b.ws_cl.numel(), None, None)
    args = (geo, code, pad, a, b.grad.data_ptr(), b.x.data_ptr(), b.w.data_ptr(), b.gi.data_ptr(), b.gw.data_ptr(),
            b.ws.data_ptr(), b.ws.numel())
    if op == "bwd":
        return lib.ts_shift_backward(*args, None)
    if op == "pool_bwd":
        return lib.ts_shift2d_avgpool2_backward(*args, None)
    assert op == "bwd_allreduce", op
    return lib.ts_shift_backward_allreduce(*args, ct.byref(peers), None)


def run_table():
    """Runs every case on cuda:0 -> the table as stored in dispatch_table.json.xz.  Leaves the kernel path automatic and the
    family knobs on."""
    import ctypes as ct
    import torch
    from torchshifts.extension import native
    from torchshifts.sharded import FusedGradWeightAllReduce
    lib = native().lib
    dev = torch.device("cuda:0")
    gen = torch.Generator().manual_seed(SEED)
    peers = FusedGradWeightAllReduce(capacity=4096, device=dev).peer_group()
    fdt = {"f32": torch.float32, "f64": torch.float64, "f16": torch.float16, "bf16": torch.bfloat16}
    qdt = {1: torch.uint8, 4: torch.int32}
    rows, planar = [], {}
    try:
        for name, (shape, borders, sliced) in GEOMETRIES.items():
            for code, dt in enumerate(DTYPES):
                b = _Buffers(torch, lib, gen, dev, shape, borders, sliced, fdt[dt], code)
                planar[f"{name}|{dt}"] = (b.geo, code)
                ops = PLANAR_OPS + (TWO_D_OPS if len(shape) == 4 or name in ("1d", "3d") else ())
                rows += [(f"{op}|{name}|{dt}|p{pad}|a{int(active)}", op, b, code, pad, active)
                         for op in ops for pad in PADDINGS for active in (False, True)]
            for eb in QBYTES:
                b = _Buffers(torch, lib, gen, dev, shape, borders, sliced, qdt[eb], eb)
                rows += [(f"qfwd|{name}|q{eb}|p{pad}|z{zp}", "qfwd", b, eb, pad, zp) for pad in PADDINGS for zp in QZERO]
        torch.cuda.synchronize()
        codes = {key: [] for key, *_ in rows}
        workspace = {key: [] for key in planar}
        for forced in FORCED:
            for spec in KNOBS.values():
                assert lib.ts_set_kernel_path(forced) >= 0 and lib.ts_set_tuning(spec) == 0
                if forced == 0:
                    for key, (geo, code) in planar.items():
                        workspace[key].append(int(lib.ts_shift_backward_workspace_bytes(ct.byref(geo), code)))
                for key, op, b, code, pad, flag in rows:
                    n0 = lib.ts_launch_count()
                    status = _call(lib, op, b, code, pad, flag, peers)
                    launches = lib.ts_launch_count() - n0
                    assert 0 <= status < 10 and launches < 10, (key, status, launches)
                    codes[key].append(f"{status}{lib.ts_last_kernel_path()}{launches}")
        torch.cuda.synchronize()
    finally:
        lib.ts_set_kernel_path(0)
        lib.ts_set_tuning(KNOBS["all"])
    cases = {key: "".join(c) for key, c in codes.items()}
    return {"seed": SEED, "forced": list(FORCED), "knobs": list(KNOBS), "workspace": workspace, "cases": cases}


TABLE = Path(__file__).resolve().parent / "dispatch_table.json.xz"


def load(path=TABLE):
    with lzma.open(path, "rt") as f:
        return json.load(f)


def main():
    out = Path(sys.argv[sys.argv.index("--out") + 1]) if "--out" in sys.argv else TABLE
    table = run_table()
    with lzma.open(out, "wt", preset=9 | lzma.PRESET_EXTREME) as f:
        json.dump(table, f, indent=0, separators=(",", ":"))
        f.write("\n")
    print(f"{out}: {len(table['cases'])} cases x {len(FORCED) * len(KNOBS)} steerings, {out.stat().st_size} bytes")


if __name__ == "__main__":
    main()
