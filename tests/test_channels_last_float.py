"""Channels-last float layers: ``memory_format=torch.preserve_format`` keeps dense channels-last inputs channels-last
(output and grad_input) through the ``_shift{2,3}d_forward_cl / _backward_cl`` operators and the native NHWC kernels
(ts_shift_forward_nhwc / ts_shift_backward_nhwc), with the values of the default (NCHW) path.

CPU tests: argument validation, fake-tensor strides, the ctypes declarations, the C entry points' argument checks.
GPU tests (marked): the oracle sweep, every kernel-selection mode, determinism, launch counts, full size, modules,
torch.compile and the fused grad_weight exchange.
"""
import ctypes as ct
import re
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
CL = torch.channels_last
NHWC_PATH, GENERIC = 4, 1


@pytest.fixture(scope="module")
def native():
    import torchshifts.extension as ext
    assert ext._HAS_OPS, ext.error_str
    return ext.native()


# ------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("bad", [torch.channels_last, torch.channels_last_3d, None, "preserve_format"])
def test_memory_format_rejects_other_values(native, bad):
    from torchshifts import Shift1d, Shift2d, Shift3d
    from torchshifts.functional import shift1d_func, shift2d_func, shift3d_func
    for fn, shape in ((shift1d_func, (1, 2, 5)), (shift2d_func, (1, 2, 5, 5)), (shift3d_func, (1, 2, 3, 3, 3))):
        x, w = torch.zeros(shape), torch.zeros(2, len(shape) - 2)
        with pytest.raises(ValueError, match="memory_format"):
            fn(x, w, 0, False, memory_format=bad)
    for cls in (Shift1d, Shift2d, Shift3d):
        with pytest.raises(ValueError, match="memory_format"):
            cls(4, memory_format=bad)


def test_memory_format_is_keyword_only_and_a_module_attribute(native):
    from torchshifts import Shift1d, Shift2d, Shift3d
    from torchshifts.functional import shift2d_func
    with pytest.raises(TypeError):
        shift2d_func(torch.zeros(1, 2, 3, 3), torch.zeros(2, 2), 0, False, None, None, torch.preserve_format)
    for cls in (Shift1d, Shift2d, Shift3d):
        m = cls(4, 'reflect', 1, 0, True, None, 1, torch.preserve_format)
        assert m.memory_format is torch.preserve_format
        assert list(m.state_dict()) == ["weight"]
        assert cls(4).memory_format is torch.contiguous_format
    # the emulated strided depth-wise conv keeps its fused pooled kernel only in the default mode
    m = Shift2d(8, emulate_dw={"kernel_size": 3, "stride": 2, "padding": 1}, memory_format=torch.preserve_format)
    assert m._stride_ints == [2, 2]


def test_cl_ops_have_no_cpu_kernel(native):
    x = torch.zeros(1, 32, 4, 4).contiguous(memory_format=CL)
    std = torch.tensor([0, 4, 0, 4, 0, 1], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        torch.ops.torchshifts._shift2d_forward_cl(x, torch.zeros(32, 2), std, [1, 32, 4, 4], 0, False)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        torch.ops.torchshifts._shift2d_backward_cl(x, torch.zeros(32, 2), x, std, 0, False)


@pytest.mark.parametrize("dim", [2, 3])
def test_fake_tensors_carry_channels_last_strides(native, dim):
    from torch._subclasses.fake_tensor import FakeTensorMode
    from torchshifts.functional import _resolve_borders
    fmt = {2: torch.channels_last, 3: torch.channels_last_3d}[dim]
    shape = (3, 64, 9, 7) if dim == 2 else (2, 32, 5, 6, 7)
    for cuts in ([[0, 0]] * dim, [[1, 1], [2, 1], [0, 2]][:dim]):
        lb, rb = _resolve_borders(dim, shape[2:], cuts)
        new_size = list(shape[:2]) + [rb[a] - lb[a] for a in range(dim)]
        std = torch.tensor([lb[0], rb[0], lb[1], rb[1], lb[2], rb[2]], dtype=torch.int32)
        with FakeTensorMode(allow_non_fake_inputs=True) as mode:
            x = mode.from_tensor(torch.empty(shape).contiguous(memory_format=fmt))
            w = mode.from_tensor(torch.empty(shape[1], dim))
            y = getattr(torch.ops.torchshifts, f"_shift{dim}d_forward_cl")(x, w, std, new_size, 3, True)
            g = mode.from_tensor(torch.empty(new_size))           # any layout
            gi, gw = getattr(torch.ops.torchshifts, f"_shift{dim}d_backward_cl")(g, w, x, std, 3, True)
        assert list(y.shape) == new_size and y.is_contiguous(memory_format=fmt)
        assert y.stride() == torch.empty(new_size).contiguous(memory_format=fmt).stride()
        assert gi.shape == x.shape and gi.is_contiguous(memory_format=fmt) and gi.stride() == x.stride()
        assert gw.shape == w.shape


_CTYPES = {"int": ct.c_int, "size_t": ct.c_size_t, "void*": ct.c_void_p, "const void*": ct.c_void_p}


def test_ctypes_declarations_match_the_header(native):
    from torchshifts._cabi import Geometry, PeerGroup
    header = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "torchshifts_b200.h").read_text(), flags=re.S)
    for name in ("ts_shift_forward_nhwc", "ts_shift_backward_nhwc_workspace_bytes", "ts_shift_backward_nhwc"):
        m = re.search(r"(\w+)\s+" + name + r"\s*\(([^)]*)\)\s*;", header)
        assert m, name
        ret, params = m.group(1), [re.sub(r"\s+", " ", p.strip()) for p in m.group(2).split(",")]
        fn = getattr(native.lib, name)
        assert fn.restype is _CTYPES[ret], name
        want = []
        for p in params:
            typ = p.rsplit(" ", 1)[0].replace(" *", "*")
            if typ == "const ts_geometry*":
                want.append(ct.POINTER(Geometry))
            elif typ == "const ts_peer_group*":
                want.append(ct.POINTER(PeerGroup))
            else:
                want.append(_CTYPES[typ])
        assert list(fn.argtypes) == want, (name, params)


def test_entry_points_validate_before_touching_a_device(native):
    from torchshifts._cabi import make_geometry
    lib = native.lib
    shape, strides = (2, 32, 6, 5), (32 * 30, 1, 5 * 32, 32)
    geo = make_geometry(2, shape, strides, [0, 0, 0], [6, 5, 1])
    assert lib.ts_shift_forward_nhwc(ct.byref(geo), 0, 7, 0, 16, 16, 16, None) == 1          # padding
    assert lib.ts_shift_forward_nhwc(ct.byref(geo), 9, 0, 0, 16, 16, 16, None) == 1          # dtype
    empty = make_geometry(2, (0,) + shape[1:], strides, [0, 0, 0], [6, 5, 1])
    assert lib.ts_shift_forward_nhwc(ct.byref(empty), 0, 0, 0, 16, 16, 16, None) == 2        # empty: planar path
    old = lib.ts_set_kernel_path(GENERIC)
    try:   # a forced kernel family sends both entry points to the planar path
        assert lib.ts_shift_forward_nhwc(ct.byref(geo), 0, 0, 0, 16, 16, 16, None) == 2
        assert lib.ts_shift_backward_nhwc(ct.byref(geo), 0, 0, 0, 16, 16, 16, 16, 16, 16, 1 << 20, None, None) == 2
    finally:
        lib.ts_set_kernel_path(old)
    assert lib.ts_shift_backward_nhwc_workspace_bytes(ct.byref(geo), 1) == 16                 # fp64: not served
    assert lib.ts_shift_backward_nhwc_workspace_bytes(ct.byref(geo), 0) >= 2 * 32 * 2 * 8


# ------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture()
def lib(native):
    native.lib.ts_set_kernel_path(0)
    yield native.lib
    native.lib.ts_set_kernel_path(0)


def _gw_close(gw, gw64, tol):
    return np.allclose(np.asarray(gw, np.float64), gw64, rtol=tol, atol=tol * np.abs(gw64).max() + 1e-30)


def _run_cl(dev, x, w, g, pad, active, borders, fmt=torch.preserve_format):
    from torchshifts.functional import shift2d_func
    xd = x.to(dev).contiguous(memory_format=CL).requires_grad_(True)
    wd = w.to(dev).requires_grad_(True)
    b = torch.tensor(borders, dtype=torch.long) if borders is not None else None
    y = shift2d_func(xd, wd, pad, active, b, memory_format=fmt)
    # torch.autograd.grad hands back the operator's own grad_input (AccumulateGrad would restride it like the leaf)
    gi, gw = torch.autograd.grad(y, (xd, wd), g.to(dev).contiguous(memory_format=CL))
    return y.detach(), gi, gw


SWEEP_SHAPES = [(2, 32, 9, 7), (1, 64, 5, 13), (3, 96, 1, 11), (2, 256, 8, 1), (1, 520, 6, 5), (2, 64, 17, 3)]


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["auto", "generic"])
def test_sweep_against_the_oracle(dev, lib, oracle_port, mode):
    """fp32 forward / grad_input bit-exact, 16-bit = the fp32 oracle on the upcast values rounded once, grad_weight
    against the fp64 oracle; outputs and grad_input dense channels-last; the NHWC kernels serve every fast-path shape in
    the automatic mode, the planar fallback in the generic mode (and for fp64 and C = 520)."""
    rng = np.random.default_rng(31)
    lib.ts_set_kernel_path(GENERIC if mode == "generic" else 0)
    for shape in SWEEP_SHAPES:
        for tdtype in (torch.float32, torch.float16, torch.bfloat16, torch.float64):
            for spread in (3.0, 12.0):
                x = torch.from_numpy(rng.standard_normal(shape)).to(tdtype)
                w = torch.from_numpy((rng.random((shape[1], 2)) * 2 - 1) * spread).to(tdtype)
                x64, w64 = x.double().numpy(), w.double().numpy()
                ref_t = np.float64 if tdtype is torch.float64 else np.float32
                xr, wr = x64.astype(ref_t), w64.astype(ref_t)
                for borders in (None, [[1, 1], [2, 1]]):
                    if borders is not None and (shape[2] < 4 or shape[3] < 4):
                        continue
                    for pad in range(5):
                        for active in (False, True):
                            y_ref = oracle_port.forward(xr, wr, pad, active, borders)
                            g = torch.from_numpy(rng.standard_normal(y_ref.shape)).to(tdtype)
                            gr = g.double().numpy().astype(ref_t)
                            y, gi, gw = _run_cl(dev, x, w, g, pad, active, borders)
                            fast = (mode == "auto" and tdtype is not torch.float64 and shape[1] % 32 == 0
                                    and shape[1] != 520)
                            tag = (mode, shape, str(tdtype), spread, borders, pad, active)
                            assert (lib.ts_last_kernel_path() == NHWC_PATH) == fast, tag
                            assert y.is_contiguous(memory_format=CL) and gi.is_contiguous(memory_format=CL), tag
                            gi_ref, _ = oracle_port.backward(gr, xr, wr, pad, active, borders)
                            _, gw64 = oracle_port.backward(gr.astype(np.float64), x64.astype(ref_t).astype(np.float64),
                                                           wr.astype(np.float64), pad, active, borders)
                            assert torch.equal(y.cpu(), torch.from_numpy(y_ref).to(tdtype)), ("forward",) + tag
                            assert torch.equal(gi.cpu(), torch.from_numpy(gi_ref).to(tdtype)), ("grad_input",) + tag
                            tol = 1e-5 if tdtype in (torch.float32, torch.float64) else 1e-2
                            assert _gw_close(gw.double().cpu().numpy(), gw64, tol), ("grad_weight",) + tag


@pytest.mark.gpu
def test_same_values_as_the_default_path_and_deterministic(dev, lib):
    torch.manual_seed(3)
    x = torch.randn(4, 128, 20, 19, device=dev)
    w = (torch.rand(128, 2, device=dev) * 2 - 1) * 2.5
    g = torch.randn(4, 128, 20, 19, device=dev)
    for pad in range(5):
        for active in (False, True):
            y0, gi0, gw0 = _run_cl(dev, x, w, g, pad, active, None, torch.contiguous_format)
            assert y0.is_contiguous() and gi0.is_contiguous()
            assert lib.ts_last_kernel_path() != NHWC_PATH
            y1, gi1, gw1 = _run_cl(dev, x, w, g, pad, active, None)
            _, _, gw2 = _run_cl(dev, x, w, g, pad, active, None)
            assert torch.equal(y0, y1) and torch.equal(gi0, gi1), (pad, active)
            assert torch.allclose(gw0, gw1, rtol=1e-5, atol=1e-5 * float(gw0.abs().max())), (pad, active)
            assert torch.equal(gw1, gw2), "grad_weight must be bit-identical from run to run"


@pytest.mark.gpu
def test_launch_counts_and_expanded_grad(dev, lib):
    """Forward: one launch; backward: kernel + pass 2.  No layout pass on either side; a stride-0 gradient from .sum()
    is made dense channels-last first (one more launch, ATen's copy)."""
    from torchshifts.functional import shift2d_func
    x = torch.randn(8, 256, 28, 28, device=dev).contiguous(memory_format=CL).requires_grad_(True)
    w = ((torch.rand(256, 2, device=dev) * 2 - 1) * 2).requires_grad_(True)
    g = torch.randn(8, 256, 28, 28, device=dev).contiguous(memory_format=CL)
    for active in (False, True):
        torch.cuda.synchronize()
        before = lib.ts_launch_count()
        y = shift2d_func(x, w, 3, active, memory_format=torch.preserve_format)
        assert lib.ts_launch_count() - before == 1 and lib.ts_last_kernel_path() == NHWC_PATH
        before = lib.ts_launch_count()
        y.backward(g)
        assert lib.ts_launch_count() - before == 2 and lib.ts_last_kernel_path() == NHWC_PATH
    x.grad = None
    xe = x.detach().clone().requires_grad_(True)
    shift2d_func(xe, w.detach(), 0, True, memory_format=torch.preserve_format).sum().backward()
    shift2d_func(x, w.detach(), 0, True, memory_format=torch.preserve_format).backward(torch.ones_like(g))
    assert torch.equal(xe.grad, x.grad) and xe.grad.is_contiguous(memory_format=CL)


def _sample_check(oracle_port, x, w, g, pad, active, y, gi, gw, idx, tdtype):
    xs = x[idx].float().cpu().numpy()
    ws = w.detach().float().cpu().numpy()
    gs = g[idx].float().cpu().numpy()
    y_ref = oracle_port.forward(xs, ws, pad, active)
    gi_ref, _ = oracle_port.backward(gs, xs, ws, pad, active)
    assert torch.equal(y[idx].cpu(), torch.from_numpy(y_ref).to(tdtype))
    assert torch.equal(gi[idx].cpu(), torch.from_numpy(gi_ref).to(tdtype))


@pytest.mark.gpu
@pytest.mark.parametrize("tdtype", [torch.float32, torch.bfloat16])
def test_full_size_cfg3_channels_last(dev, lib, oracle_port, tdtype):
    """cfg3-shaped N=256 C=256 56x56 channels-last: zeros sparse and reflect active, sampled images against the oracle,
    grad_weight of a sub-batch against the fp64 oracle, the whole tensor against the default path."""
    from torchshifts.functional import shift2d_func
    torch.manual_seed(0)
    N, C, H, W = 256, 256, 56, 56
    x = torch.randn(N, C, H, W, device=dev).to(tdtype).contiguous(memory_format=CL)
    g = torch.randn(N, C, H, W, device=dev).to(tdtype).contiguous(memory_format=CL)
    w0 = ((torch.rand(C, 2, device=dev) * 2 - 1) * 3).to(tdtype)
    for pad, active in ((0, False), (3, True)):
        xr, w = x.clone().requires_grad_(True), w0.clone().requires_grad_(True)
        y = shift2d_func(xr, w, pad, active, memory_format=torch.preserve_format)
        assert lib.ts_last_kernel_path() == NHWC_PATH and y.is_contiguous(memory_format=CL)
        y.backward(g)
        assert lib.ts_last_kernel_path() == NHWC_PATH and xr.grad.is_contiguous(memory_format=CL)
        _sample_check(oracle_port, x, w, g, pad, active, y.detach(), xr.grad, w.grad, [0, 17, 255], tdtype)
        wq = w0.clone().requires_grad_(True)
        shift2d_func(x[:4].contiguous(memory_format=CL), wq, pad, active, memory_format=torch.preserve_format).backward(g[:4])
        _, gw64 = oracle_port.backward(g[:4].double().cpu().numpy(), x[:4].double().cpu().numpy(), w0.double().cpu().numpy(), pad, active)
        assert _gw_close(wq.grad.double().cpu().numpy(), gw64, 1e-5 if tdtype is torch.float32 else 1e-2)
        x0, w1 = x.clone().requires_grad_(True), w0.clone().requires_grad_(True)
        y0 = shift2d_func(x0, w1, pad, active)
        y0.backward(g)
        assert torch.equal(y0, y.detach()) and torch.equal(x0.grad, xr.grad)
        del xr, y, x0, y0


class _Net(torch.nn.Module):
    def __init__(self, fmt, shift_kwargs):
        super().__init__()
        from torchshifts import Shift2d
        self.c1 = torch.nn.Conv2d(16, 64, 1)
        self.shift = Shift2d(64, memory_format=fmt, **shift_kwargs)
        self.c2 = torch.nn.Conv2d(64, 32, 1)

    def forward(self, x):
        h, _ = self.shift(self.c1(x))
        self.last_shift_out = h
        return self.c2(h)


@pytest.mark.gpu
@pytest.mark.parametrize("kwargs", [dict(padding="reflect", active_flag=True, sparsity_term=0),
                                    dict(padding="zeros", emulate_dw={"kernel_size": 3, "stride": 2, "padding": 1}),
                                    dict(padding="symmetric", active_flag=True, emulate_dw={"kernel_size": 5, "padding": 1})])
def test_module_in_a_channels_last_network(dev, lib, kwargs):
    """conv -> Shift2d(preserve) -> conv gives the default model's outputs and gradients; the shift output stays
    channels-last.  Covers the emulated stride-2 depth-wise conv (shift then avg_pool2d: the fused pooled kernels are
    NCHW-only) and a cropping layer."""
    torch.manual_seed(5)
    models = {}
    for fmt in (torch.contiguous_format, torch.preserve_format):
        torch.manual_seed(5)
        models[fmt] = _Net(fmt, dict(kwargs, emulate_dw=dict(kwargs["emulate_dw"]) if "emulate_dw" in kwargs else None)) \
            .to(dev).to(memory_format=CL)
    models[torch.preserve_format].load_state_dict(models[torch.contiguous_format].state_dict())
    x = torch.randn(4, 16, 23, 18, device=dev).contiguous(memory_format=CL)
    outs = {}
    for fmt, m in models.items():
        assert not m.shift._pool_is_fused(m.c1(x)) or fmt is torch.contiguous_format
        out = m(x)
        out.square().sum().backward()
        outs[fmt] = (out, m.last_shift_out)
    a, b = models[torch.contiguous_format], models[torch.preserve_format]
    assert outs[torch.preserve_format][1].is_contiguous(memory_format=CL)
    assert torch.allclose(outs[torch.contiguous_format][0], outs[torch.preserve_format][0], rtol=1e-5, atol=1e-5)
    assert torch.equal(outs[torch.contiguous_format][1], outs[torch.preserve_format][1])
    for (name, pa), pb in zip(a.named_parameters(), b.parameters()):
        assert torch.allclose(pa.grad, pb.grad, rtol=1e-4, atol=1e-4 * float(pa.grad.abs().max())), name


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["aot_eager", "inductor"])
def test_compile_matches_eager(dev, lib, backend, tmp_path, monkeypatch):
    monkeypatch.setenv("TORCHINDUCTOR_CACHE_DIR", str(tmp_path / "inductor"))
    monkeypatch.setenv("TRITON_CACHE_DIR", str(tmp_path / "triton"))
    from torchshifts import Shift2d
    torch.manual_seed(7)
    m = Shift2d(64, padding="border", active_flag=True, sparsity_term=0, emulate_dw={"kernel_size": 5, "padding": 1},
                memory_format=torch.preserve_format).to(dev)
    x = torch.randn(2, 64, 12, 10, device=dev).contiguous(memory_format=CL)
    xe, xc = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    ye, _ = m(xe)
    ye.square().sum().backward()
    gwe = m.weight.grad.clone()
    m.weight.grad = None
    torch._dynamo.reset()
    cm = torch.compile(m, backend=backend, fullgraph=True)
    yc, _ = cm(xc)
    assert yc.is_contiguous(memory_format=CL) and yc.stride() == ye.stride()
    yc.square().sum().backward()
    assert torch.equal(yc, ye) and torch.equal(xc.grad, xe.grad)
    assert xc.grad.is_contiguous(memory_format=CL)
    assert torch.allclose(m.weight.grad, gwe, rtol=1e-5, atol=1e-6)
    torch._dynamo.reset()


@pytest.mark.gpu
def test_fused_exchange_through_the_nhwc_backward(dev, lib):
    """The fused grad_weight exchange on one rank through the new backward equals the plain backward bit for bit, and
    fp64 / capacity raise as in the planar backward."""
    from torchshifts.functional import shift2d_func
    from torchshifts.sharded import FusedGradWeightAllReduce
    torch.manual_seed(9)
    x = torch.randn(4, 64, 14, 12, device=dev).contiguous(memory_format=CL)
    g = torch.randn(4, 64, 14, 12, device=dev).contiguous(memory_format=CL)
    w = (torch.rand(64, 2, device=dev) * 2 - 1) * 2
    wd = w.clone().requires_grad_(True)
    shift2d_func(x, wd, 0, True, memory_format=torch.preserve_format).backward(g)
    plain = wd.grad
    with FusedGradWeightAllReduce(None, device=dev, capacity=256):
        wd = w.clone().requires_grad_(True)
        shift2d_func(x, wd, 0, True, memory_format=torch.preserve_format).backward(g)
        assert lib.ts_last_kernel_path() == NHWC_PATH
        assert torch.equal(wd.grad, plain)
        with pytest.raises(RuntimeError, match="fp32 contributions"):
            shift2d_func(x.double().contiguous(memory_format=CL), w.double().requires_grad_(True), 0, True,
                         memory_format=torch.preserve_format).backward(g.double())
    with FusedGradWeightAllReduce(None, device=dev, capacity=64):
        with pytest.raises(RuntimeError, match="exceed the exchange capacity"):
            shift2d_func(x, w.clone().requires_grad_(True), 0, True, memory_format=torch.preserve_format).backward(g)


@pytest.mark.gpu
def test_fused_exchange_two_ranks():
    """The exchange through the new backward on TWO ranks against NCCL (tools/cl_fused_probe.py under torchrun)."""
    import socket
    import subprocess
    import sys
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(ROOT / "tools" / "cl_fused_probe.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "PROBE OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]


@pytest.mark.gpu
def test_taps_beyond_the_staged_window(dev, lib, oracle_port):
    """Images taller than the staged window (48 x 60 fp32: K = 14 ring rows, window 8 rows) with shifts up to |w| = 12:
    the window cap applies and the taps it leaves out are read from global memory -- still the NHWC kernels, still
    bit-exact."""
    rng = np.random.default_rng(41)
    shape = (2, 32, 48, 60)
    x = torch.from_numpy(rng.standard_normal(shape).astype(np.float32))
    w = torch.from_numpy(((rng.random((shape[1], 2)) * 2 - 1) * 12).astype(np.float32))
    for borders in (None, [[1, 1], [2, 1]]):
        for pad in range(5):
            for active in (False, True):
                y_ref = oracle_port.forward(x.numpy(), w.numpy(), pad, active, borders)
                g = torch.from_numpy(rng.standard_normal(y_ref.shape).astype(np.float32))
                y, gi, gw = _run_cl(dev, x, w, g, pad, active, borders)
                assert lib.ts_last_kernel_path() == NHWC_PATH
                gi_ref, _ = oracle_port.backward(g.numpy(), x.numpy(), w.numpy(), pad, active, borders)
                _, gw64 = oracle_port.backward(g.double().numpy(), x.double().numpy(), w.double().numpy(), pad, active, borders)
                tag = (borders, pad, active)
                assert torch.equal(y.cpu(), torch.from_numpy(y_ref)), ("forward",) + tag
                assert torch.equal(gi.cpu(), torch.from_numpy(gi_ref)), ("grad_input",) + tag
                assert _gw_close(gw.cpu().numpy(), gw64, 1e-5), ("grad_weight",) + tag


@pytest.mark.gpu
def test_staging_knobs_keep_the_values(dev, lib):
    """Every setting of the staging knobs (copies in flight, rows per step) gives the same forward and grad_input bits;
    grad_weight sums each thread's pixels in a knob-dependent order, so it agrees to rounding."""
    torch.manual_seed(13)
    x = torch.randn(3, 64, 30, 21, device=dev)
    w = (torch.rand(64, 2, device=dev) * 2 - 1) * 4
    g = torch.randn(3, 64, 28, 18, device=dev)            # the cropped output
    try:
        for active in (False, True):
            ref = _run_cl(dev, x, w, g, 4, active, [[1, 1], [2, 1]])
            for knobs in (b"cl_ahead=1,cl_rows=1", b"cl_ahead=4,cl_rows=1", b"cl_ahead=3,cl_rows=4", b"cl_ahead=1,cl_rows=4"):
                assert lib.ts_set_tuning(knobs) == 0
                got = _run_cl(dev, x, w, g, 4, active, [[1, 1], [2, 1]])
                assert lib.ts_last_kernel_path() == NHWC_PATH
                assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1]), (knobs, active)
                assert torch.allclose(ref[2], got[2], rtol=1e-5, atol=1e-5 * float(ref[2].abs().max())), (knobs, active)
    finally:
        lib.ts_set_tuning(b"cl_ahead=0,cl_rows=0")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 32, 5, 6, 7), (1, 20, 4, 3, 6)])
def test_3d_preserving_layers(dev, lib, shape):
    """Shift3d through _shift3d_forward_cl / _backward_cl (the planar path and a conversion): channels_last_3d output and
    grad_input, the default path's values."""
    from torchshifts.functional import shift3d_func
    fmt = torch.channels_last_3d
    torch.manual_seed(17)
    x = torch.randn(shape, device=dev).contiguous(memory_format=fmt)
    w = (torch.rand(shape[1], 3, device=dev) * 2 - 1) * 2.5
    g = torch.randn(shape, device=dev)
    b = torch.tensor([[1, 0], [0, 1], [1, 1]])
    for pad in range(5):
        for active in (False, True):
            outs = []
            for mf in (torch.contiguous_format, torch.preserve_format):
                xd, wd = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
                y = shift3d_func(xd, wd, pad, active, b, memory_format=mf)
                gi, gw = torch.autograd.grad(y, (xd, wd), g[:, :, :y.shape[2], :y.shape[3], :y.shape[4]].contiguous())
                outs.append((y, gi, gw))
            (y0, gi0, gw0), (y1, gi1, gw1) = outs
            assert y0.is_contiguous() and y1.is_contiguous(memory_format=fmt) and not y1.is_contiguous()
            assert gi1.is_contiguous(memory_format=fmt) and not gi1.is_contiguous()
            assert torch.equal(y0, y1) and torch.equal(gi0, gi1) and torch.equal(gw0, gw1), (pad, active)
