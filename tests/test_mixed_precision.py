"""Mixed precision: fp16 / bf16 activations with fp32 weights and an fp32 grad_weight.

Method (as for the bit-exact bf16 cfg2 test): the kernels compute in fp32 on the 16-bit values and round once at the
store, so the forward and grad_input equal the fp32 oracle run on the 16-bit-rounded x / grad and the UNROUNDED fp32
weights, rounded once to the 16-bit type -- bit for bit.  grad_weight is fp32 and within rtol 1e-5 of the fp64 oracle on
the same values.  Every kernel family serves the weights flag; the 2-D zeros-padded layer runs on the TMA family.

The CPU-side tests pin the C ABI's flag rules; everything else needs a B200.
"""
import ctypes as ct
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = Path(__file__).resolve().parents[1]
GENERIC, TMA, NHWC = 1, 3, 4
TS_F32, TS_F64, TS_F16, TS_BF16, TS_WEIGHTS_F32 = 0, 1, 2, 3, 0x100
TS_OK, TS_ERR_INVALID_ARGUMENT = 0, 1
BORDERS = {1: [[1, 2]], 2: [[1, 1], [2, 1]], 3: [[1, 0], [0, 2], [1, 1]]}
SHAPES = {1: (2, 8, 40), 2: (2, 16, 12, 24), 3: (2, 4, 5, 6, 16)}
HALF = {"fp16": torch.float16, "bf16": torch.bfloat16}
MODES = ["auto", "no_tma", "generic"]


@pytest.fixture(scope="module")
def lib():
    from torchshifts.extension import native
    return native().lib


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture()
def steering(lib):
    def set_mode(mode):
        lib.ts_set_kernel_path(GENERIC if mode == "generic" else 0)
        lib.ts_set_tuning(b"use_tma=0,use_halo=1,use_flat=1" if mode == "no_tma" else b"use_tma=1,use_halo=1,use_flat=1")
    set_mode("auto")
    yield set_mode
    set_mode("auto")


def _func(dim):
    from torchshifts import functional as F
    return {1: F.shift1d_func, 2: F.shift2d_func, 3: F.shift3d_func}[dim]


def _weights(rng, C, dim):
    """Integer parts -8..7 on the last axis (every sub-16-byte phase of an 8-element item), random fractions."""
    w = rng.uniform(-3.0, 3.0, (C, dim)).astype(np.float32)
    w[:, dim - 1] = (np.arange(C) % 16 - 8 + rng.uniform(0.05, 0.95, C)).astype(np.float32)
    return w


def _gw_close(gw, gw64):
    scale = np.abs(gw64).max()
    return np.allclose(gw.astype(np.float64), gw64, rtol=1e-5, atol=1e-5 * scale + 1e-30)


def _check_case(dev, oracle, dim, x, w, g, pad, active, borders, dtype, memory_format=torch.contiguous_format):
    """Runs the mixed layer (x, g in `dtype`, w fp32) through autograd and checks it against the oracle."""
    xd = x.to(dev).requires_grad_(True)
    wd = torch.from_numpy(w).to(dev).requires_grad_(True)
    b = torch.tensor(borders, dtype=torch.long) if borders is not None else None
    y = _func(dim)(xd, wd, pad, active, b, memory_format=memory_format)
    y.backward(g.to(dev))
    assert y.dtype == dtype and xd.grad.dtype == dtype and wd.grad.dtype == torch.float32
    xr, gr = np.ascontiguousarray(x.float().numpy()), np.ascontiguousarray(g.float().numpy())
    y_ref = torch.from_numpy(oracle.forward(xr, w, pad, active, borders)).to(dtype)
    gi_ref = torch.from_numpy(oracle.backward(gr, xr, w, pad, active, borders)[0]).to(dtype)
    _, gw64 = oracle.backward(gr.astype(np.float64), xr.astype(np.float64), w.astype(np.float64), pad, active, borders)
    case = (dim, pad, active, borders, dtype)
    assert torch.equal(y.detach().cpu(), y_ref), case
    assert torch.equal(xd.grad.cpu(), gi_ref), case
    assert _gw_close(wd.grad.cpu().numpy(), gw64), case
    return y, xd.grad


# ------------------------------------------------------------------------------------------ CPU: the C ABI's flag
def test_weights_flag_rules_of_the_c_abi(lib):
    from torchshifts._cabi import make_geometry
    geo = make_geometry(2, (2, 16, 12, 24), (16 * 288, 288, 24, 1), [0, 0, 0], [12, 24, 1])
    for bad in (TS_F32 | TS_WEIGHTS_F32, TS_F64 | TS_WEIGHTS_F32, 7 | TS_WEIGHTS_F32):
        # rejected before anything touches a device
        assert lib.ts_shift_forward(ct.byref(geo), bad, 0, 1, 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
        assert lib.ts_shift_backward(ct.byref(geo), bad, 0, 1, 16, 16, 16, 16, 16, 16, 1 << 20, None) == TS_ERR_INVALID_ARGUMENT
        assert lib.ts_shift_forward_nhwc(ct.byref(geo), bad, 0, 1, 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
        assert lib.ts_shift2d_avgpool2_forward(ct.byref(geo), bad, 0, 1, 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
        assert lib.ts_shift2d_avgpool2_backward(ct.byref(geo), bad, 0, 1, 16, 16, 16, 16, 16, 16, 1 << 20, None) \
            == TS_ERR_INVALID_ARGUMENT
        assert lib.ts_shift_backward_workspace_bytes(ct.byref(geo), bad) == 0
        assert lib.ts_shift_backward_nhwc_workspace_bytes(ct.byref(geo), bad) == 0
    for half in (TS_F16, TS_BF16):
        # the workspace query accepts the flag: at least what the same-dtype call needs (its plans plus the 16-bit TMA ones)
        mixed = lib.ts_shift_backward_workspace_bytes(ct.byref(geo), half | TS_WEIGHTS_F32)
        assert mixed >= 16 and mixed >= lib.ts_shift_backward_workspace_bytes(ct.byref(geo), half)
        assert lib.ts_shift_backward_nhwc_workspace_bytes(ct.byref(geo), half | TS_WEIGHTS_F32) >= 16


def test_type_rule_of_the_operator_layer():
    sys.path.insert(0, str(ROOT / "activesparseshifts-pytorch_b200"))
    from torchshifts import _ops
    from torchshifts._cabi import TS_WEIGHTS_F32 as flag
    assert flag == TS_WEIGHTS_F32
    w32 = torch.zeros(4, 2)
    for half, code in ((torch.float16, TS_F16), (torch.bfloat16, TS_BF16)):
        x = torch.zeros(1, 4, 8, 8, dtype=half)
        _ops._same_device_and_type("f", x, w32, x)
        assert _ops._dtype_code(x, w32) == code | TS_WEIGHTS_F32
        assert _ops._dtype_code(x, w32.to(half)) == code
        with pytest.raises(RuntimeError, match="scalar type"):           # grad must match x
            _ops._same_device_and_type("f", x, w32, x.float())
    for x, w in ((torch.zeros(1, 4, 8, 8), w32.half()), (torch.zeros(1, 4, 8, 8, dtype=torch.float64), w32),
                 (torch.zeros(1, 4, 8, 8, dtype=torch.bfloat16), w32.double()), (torch.zeros(1, 4, 8, 8), w32.double())):
        with pytest.raises(RuntimeError, match="scalar type"):
            _ops._same_device_and_type("f", x, w)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _allreduce_worker(rank, world, port, out_dir):
    for p in (str(ROOT), str(ROOT / "activesparseshifts-pytorch_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from torchshifts import Shift1d, Shift2d
        from torchshifts.sharded import allreduce_grad_weights
        mixed = Shift2d(3)                                   # fp32 master weights of a layer fed bf16 activations
        pure = Shift1d(2).bfloat16()                         # an all-bf16 layer
        wide = Shift1d(2).double()
        layers = torch.nn.ModuleList([mixed, pure, wide])
        base = [torch.arange(m.weight.numel(), dtype=torch.float64).reshape(m.weight.shape) for m in layers]
        eps = [1e-7, 0.0, 1e-12]                             # below what fp32 / fp64 of the other rank can hold alone
        for m, b, e in zip(layers, base, eps):
            m.weight.grad = ((b + 1.0) * (1.0 + e * rank)).to(m.weight.dtype)
        allreduce_grad_weights(layers)
        for m, b, e in zip(layers, base, eps):
            assert m.weight.grad.dtype == m.weight.dtype
            local = [((b + 1.0) * (1.0 + e * r)).to(m.weight.dtype).double() for r in range(world)]
            expect = sum(local)
            if m is wide:
                assert torch.equal(m.weight.grad, expect)            # an fp64 layer is reduced in fp64
            else:
                assert torch.equal(m.weight.grad, expect.float().to(m.weight.dtype))
        Path(out_dir, f"ok{rank}").write_text("ok")
    finally:
        dist.destroy_process_group()


def test_allreduce_keeps_each_layers_gradient_dtype(tmp_path):
    """Mixed (fp32 grads), all-bf16 and fp64 layers in one coalesced exchange: every gradient comes back in its own
    parameter's dtype, none is narrowed on the way (gloo, two ranks)."""
    world, port = 2, _free_port()
    mp.spawn(_allreduce_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(world))


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("half", sorted(HALF))
@pytest.mark.parametrize("dim", [1, 2, 3])
def test_mixed_sweep_vs_oracle(dev, lib, oracle_port, steering, dim, half, mode):
    """1-D / 2-D / 3-D, five paddings, sparse and active, with and without crops, under auto routing, without the TMA
    family and on the generic family alone."""
    steering(mode)
    dtype = HALF[half]
    rng = np.random.default_rng(10 * dim + len(half))
    shape = SHAPES[dim]
    w = _weights(rng, shape[1], dim)
    x = torch.from_numpy(rng.standard_normal(shape).astype(np.float32)).to(dtype)
    for pad in range(5):
        for active in (False, True):
            for borders in (None, BORDERS[dim]):
                osz = list(shape[:2]) + [shape[2 + a] - (sum(borders[a]) if borders else 0) for a in range(dim)]
                g = torch.from_numpy(rng.standard_normal(osz).astype(np.float32)).to(dtype)
                _check_case(dev, oracle_port, dim, x, w, g, pad, active, borders, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("half", sorted(HALF))
def test_zeros_padded_2d_runs_on_the_tma_family(dev, lib, oracle_port, steering, half):
    """The 16-bit TMA kernels (sparse / active forward, sparse / active backward) serve the mixed 2-D zeros-padded layer,
    with rows of several 16-byte items and every sub-item phase of the column shift."""
    from torchshifts.functional import shift2d_func
    dtype = HALF[half]
    rng = np.random.default_rng(7)
    N, C, H, W = 3, 32, 20, 56
    w = _weights(rng, C, 2)
    x = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32)).to(dtype)
    g = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32)).to(dtype)
    borders = torch.zeros(6, dtype=torch.int32)
    borders[1], borders[3], borders[5] = H, W, 1
    for active in (False, True):
        _check_case(dev, oracle_port, 2, x, w, g, 0, active, None, dtype)
        xd, wd, gd = x.to(dev), torch.from_numpy(w).to(dev), g.to(dev)
        shift2d_func(xd, wd, 0, active)
        assert lib.ts_last_kernel_path() == TMA, active
        # the backward op in this thread (autograd runs it on its own): the path is recorded per thread
        gi, gw = torch.ops.torchshifts._shift2d_backward(gd, wd, xd, borders, 0, active)
        assert lib.ts_last_kernel_path() == TMA, active
        assert gi.dtype == dtype and gw.dtype == torch.float32
        # same-dtype 16-bit layers keep their routing: the active ones never take the TMA family
        if active:
            shift2d_func(xd, wd.to(dtype), 0, True)
            assert lib.ts_last_kernel_path() != TMA


@pytest.mark.gpu
def test_weights_are_not_rounded_to_16_bits(dev, lib, oracle_port, steering):
    """Weights whose bf16 rounding changes the integer or the fractional part: the mixed layer matches the oracle with the
    fp32 weights and differs from the all-bf16 layer."""
    from torchshifts.functional import shift2d_func
    rng = np.random.default_rng(3)
    C = 8
    w = np.array([[40.3, -17.6], [10.52, -3.3], [-17.6, 40.3], [2.5039, 6.7], [-10.52, 1.3], [5.3, -2.7],
                  [0.3, 12.52], [-6.7, -0.3]], dtype=np.float32)
    assert not np.array_equal(torch.from_numpy(w).bfloat16().float().numpy(), w)
    x = torch.from_numpy(rng.standard_normal((2, C, 48, 64)).astype(np.float32)).bfloat16()
    g = torch.from_numpy(rng.standard_normal((2, C, 48, 64)).astype(np.float32)).bfloat16()
    for mode in MODES:
        steering(mode)
        for pad in (0, 2):
            for active in (False, True):
                y, gi = _check_case(dev, oracle_port, 2, x, w, g, pad, active, None, torch.bfloat16)
                y16 = shift2d_func(x.to(dev), torch.from_numpy(w).to(dev).bfloat16(), pad, active)
                assert not torch.equal(y.detach(), y16), (mode, pad, active)


@pytest.mark.gpu
@pytest.mark.parametrize("half", sorted(HALF))
def test_channels_last_mixed(dev, lib, oracle_port, steering, half):
    """memory_format=torch.preserve_format: the native NHWC kernels with fp32 weights, channels-last out."""
    from torchshifts.functional import shift2d_func
    dtype = HALF[half]
    rng = np.random.default_rng(5)
    shape = (2, 64, 10, 12)
    w = _weights(rng, shape[1], 2)
    for pad in (0, 3):
        for active in (False, True):
            x = torch.from_numpy(rng.standard_normal(shape).astype(np.float32)).to(dtype).contiguous(memory_format=torch.channels_last)
            g = torch.from_numpy(rng.standard_normal(shape).astype(np.float32)).to(dtype).contiguous(memory_format=torch.channels_last)
            y, gi = _check_case(dev, oracle_port, 2, x, w, g, pad, active, None, dtype, torch.preserve_format)
            assert y.is_contiguous(memory_format=torch.channels_last) and gi.is_contiguous(memory_format=torch.channels_last)
            shift2d_func(x.to(dev), torch.from_numpy(w).to(dev), pad, active, memory_format=torch.preserve_format)
            assert lib.ts_last_kernel_path() == NHWC


@pytest.mark.gpu
def test_pooled_layer_mixed(dev, oracle_port, steering):
    """Shift2d emulating a stride-2 depth-wise conv (shift, then avg_pool2d(2, 2, ceil_mode)) in bf16 with fp32 weights."""
    from torchshifts import Shift2d
    torch.manual_seed(4)
    layer = Shift2d(16, sparsity_term=0.0, active_flag=True, emulate_dw={'kernel_size': 3, 'stride': 2, 'padding': 1}).to(dev)
    x = torch.randn(2, 16, 14, 24, device=dev).bfloat16().requires_grad_(True)
    out, _ = layer(x)
    assert out.dtype == torch.bfloat16 and list(out.shape) == [2, 16, 7, 12]
    gp = torch.randn_like(out)
    out.backward(gp)
    assert x.grad.dtype == torch.bfloat16 and layer.weight.grad.dtype == torch.float32
    w = layer.weight.detach().cpu().numpy()
    xr = x.detach().float().cpu().numpy()
    y_ref = torch.from_numpy(oracle_port.forward(xr, w, 0, True)).bfloat16()
    pooled = torch.nn.functional.avg_pool2d(y_ref.to(dev), 2, 2, ceil_mode=True)
    assert torch.equal(out.detach(), pooled)
    gy = torch.ops.aten.avg_pool2d_backward(gp.double().cpu(), torch.empty(2, 16, 14, 24, dtype=torch.float64), [2, 2], [2, 2],
                                            [0, 0], True, True, None)
    _, gw64 = oracle_port.backward(gy.numpy(), xr.astype(np.float64), w.astype(np.float64), 0, True)
    assert _gw_close(layer.weight.grad.cpu().numpy(), gw64)


class _Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        from torchshifts import Shift2d
        self.conv1 = torch.nn.Conv2d(8, 32, 3, padding=1)
        self.shift = Shift2d(32, init_shift=3, sparsity_term=0.0, active_flag=True)
        self.conv2 = torch.nn.Conv2d(32, 8, 1)

    def forward(self, x):
        y, _ = self.shift(self.conv1(x))
        return self.conv2(y)


@pytest.mark.gpu
def test_autocast_training_step(dev, steering):
    """conv -> Shift2d -> conv under torch.autocast(bfloat16): the shift weight stays fp32, its gradient is fp32, and one
    SGD step moves weights by less than a bf16 ulp -- steps an all-bf16 layer could not take."""
    torch.manual_seed(0)
    net = _Net().to(dev)
    w0 = net.shift.weight.detach().clone()
    opt = torch.optim.SGD(net.parameters(), lr=1e-4)
    x = torch.randn(4, 8, 16, 32, device=dev)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        loss = net(x).float().square().mean()
    loss.backward()
    assert net.shift.weight.dtype == torch.float32 and net.shift.weight.grad.dtype == torch.float32
    opt.step()
    w1 = net.shift.weight.detach()
    moved = w1 != w0
    assert moved.any()
    # steps smaller than one bf16 ulp of the weight (8 significant bits): an all-bf16 parameter could not take them
    ulp = torch.exp2(torch.floor(torch.log2(w0.abs())) - 7)
    assert (moved & (torch.abs(w1 - w0) < ulp)).any()


@pytest.mark.gpu
def test_autocast_training_step_compiled(dev, steering):
    """torch.compile (aot_eager) of the same model under autocast: same fp32 weight gradient as eager."""
    torch.manual_seed(0)
    net = _Net().to(dev)
    x = torch.randn(4, 8, 16, 32, device=dev)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        net(x).float().square().mean().backward()
    eager = net.shift.weight.grad.clone()
    net.zero_grad(set_to_none=True)
    compiled = torch.compile(net, backend="aot_eager")
    with torch.autocast("cuda", dtype=torch.bfloat16):
        out = compiled(x)
        out.float().square().mean().backward()
    assert out.dtype == torch.bfloat16
    assert net.shift.weight.grad.dtype == torch.float32
    assert torch.allclose(net.shift.weight.grad, eager, rtol=1e-5, atol=1e-6 * float(eager.abs().max()))


@pytest.mark.gpu
def test_fused_exchange_takes_mixed_layers(dev, steering):
    """FusedGradWeightAllReduce (one rank: the exchange degenerates to a local copy) carries the fp32 contributions of a
    mixed layer: the same fp32 grad_weight as the plain backward, also through the channels-last kernels."""
    from torchshifts.functional import shift2d_func
    from torchshifts.sharded import FusedGradWeightAllReduce
    torch.manual_seed(1)
    fused = FusedGradWeightAllReduce(device=dev)
    w = (torch.rand(32, 2, device=dev) * 6 - 3).requires_grad_(True)
    for fmt in (torch.contiguous_format, torch.channels_last):
        x = torch.randn(2, 32, 8, 16, device=dev).bfloat16().contiguous(memory_format=fmt)
        g = torch.randn(2, 32, 8, 16, device=dev).bfloat16()
        mf = torch.preserve_format if fmt is torch.channels_last else torch.contiguous_format
        (gw,) = torch.autograd.grad(shift2d_func(x, w, 0, True, memory_format=mf), w, g)
        with fused:
            (gwf,) = torch.autograd.grad(shift2d_func(x, w, 0, True, memory_format=mf), w, g)
        assert gwf.dtype == torch.float32 and torch.equal(gwf, gw)


@pytest.mark.gpu
def test_other_type_mixes_still_raise(dev):
    from torchshifts.functional import shift2d_func
    x = torch.randn(1, 2, 8, 8, device=dev)
    w = torch.randn(2, 2, device=dev)
    with pytest.raises(RuntimeError, match="scalar type"):
        shift2d_func(x, w.half(), 0, False)
    with pytest.raises(RuntimeError, match="scalar type"):
        shift2d_func(x.double(), w, 0, False)
    with pytest.raises(RuntimeError, match="scalar type"):
        shift2d_func(x.bfloat16(), w.double(), 0, True)
