"""The strided depth-wise-conv emulation of Shift3d (stride (1, 2, 2) or (2, 2, 2)): shift, crop and avg_pool3d in one kernel,
forward and backward (``torchshifts::_shift3d_avgpool_forward/_backward``, ``ts_shift_avgpool_forward/_backward``), and the
fused 2-D pooled backward taking part in the grad_weight exchange.

CPU: schemas, fake shapes, the C ABI's argument checks.  GPU: the oracle (shift) followed by a numpy pooling in ATen's order,
the two-step path (shift op + torch's avg_pool3d) and autograd through it, cfg4 at full size, peak memory, torch.compile and
the in-kernel exchange.
"""
import ctypes as ct
import re

import numpy as np
import pytest
import torch

HALO = 5
TS_ERR_INVALID_ARGUMENT, TS_ERR_UNSUPPORTED = 1, 2
FORWARD = ("(Tensor input, Tensor weights, Tensor borders, int[] new_size, int[] stride, int padding_mode, bool active_flag)"
           " -> Tensor")
BACKWARD = ("(Tensor grad, Tensor weights, Tensor input, Tensor borders, int[] new_size, int[] stride, int padding_mode, "
            "bool active_flag) -> (Tensor, Tensor)")


@pytest.fixture(scope="module")
def lib():
    from torchshifts.extension import native
    return native().lib


def _strides(v):
    return (ct.c_int32 * len(v))(*v)


# ------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name,schema", [("_shift3d_avgpool_forward", FORWARD), ("_shift3d_avgpool_backward", BACKWARD)])
def test_schema_and_dispatch_keys(lib, name, schema):
    dump = torch._C._dispatch_dump(f"torchshifts::{name}")
    assert re.search(r"^schema: (.*)$", dump, re.M).group(1) == f"torchshifts::{name}{schema}"
    assert re.findall(r"^(\w+(?:\[alias\])?): registered at", dump, re.M) == ["debug", "CPU", "CUDA", "Meta", "Autograd[alias]"]


@pytest.mark.parametrize("stride", [(1, 2, 2), (2, 2, 2)])
def test_fake_shapes(lib, stride):
    x, w = torch.empty(2, 3, 7, 9, 12, device='meta'), torch.empty(3, 3, device='meta')
    borders = torch.tensor([1, 7, 0, 9, 2, 12], dtype=torch.int32)
    new_size = [2, 3, 6, 9, 10]
    y = torch.ops.torchshifts._shift3d_avgpool_forward(x, w, borders, new_size, list(stride), 0, True)
    assert y.device.type == 'meta' and list(y.shape) == [2, 3, -(-6 // stride[0]), 5, 5]
    gi, gw = torch.ops.torchshifts._shift3d_avgpool_backward(y, w, x, borders, new_size, list(stride), 0, True)
    assert gi.shape == x.shape and gw.shape == w.shape


def test_cpu_kernels_raise(lib):
    x, w = torch.zeros(1, 2, 4, 4, 8), torch.zeros(2, 3)
    borders = torch.tensor([0, 4, 0, 4, 0, 8], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        torch.ops.torchshifts._shift3d_avgpool_forward(x, w, borders, [1, 2, 4, 4, 8], [2, 2, 2], 0, False)


def test_ctypes_declarations_match_the_header(lib):
    from torchshifts._cabi import SIGNATURES
    _geo = SIGNATURES['ts_shift_avgpool_forward'][1][0]
    i32p = ct.POINTER(ct.c_int32)
    vp, i, sz = ct.c_void_p, ct.c_int, ct.c_size_t
    peers = SIGNATURES['ts_shift_backward_nhwc'][1][-2]
    assert SIGNATURES['ts_shift_avgpool_forward'] == (i, [_geo, i, i, i, i32p, vp, vp, vp, vp])
    assert SIGNATURES['ts_shift_avgpool_backward_workspace_bytes'] == (sz, [_geo, i])
    assert SIGNATURES['ts_shift_avgpool_backward'] == (i, [_geo, i, i, i, i32p, vp, vp, vp, vp, vp, vp, sz, peers, vp])
    for name in ('ts_shift_avgpool_forward', 'ts_shift_avgpool_backward', 'ts_shift_avgpool_backward_workspace_bytes'):
        assert hasattr(lib, name)


def test_entry_point_argument_checks(lib):
    """Rejected before any device work: this runs without a GPU."""
    from torchshifts._cabi import PeerGroup, TS_WEIGHTS_F32, make_geometry
    g3 = make_geometry(3, (2, 4, 8, 16, 16), (8192, 2048, 256, 16, 1), [0, 0, 0], [8, 16, 16])
    g2 = make_geometry(2, (2, 4, 16, 16), (1024, 256, 16, 1), [0, 0, 0], [16, 16, 1])
    g1 = make_geometry(1, (2, 4, 16), (64, 16, 1), [0, 0, 0], [16, 1, 1])
    s222 = _strides([2, 2, 2])
    fwd, bwd = lib.ts_shift_avgpool_forward, lib.ts_shift_avgpool_backward

    def b(geo, dtype=0, stride=s222, ptr=16, peers=None, pad=0):
        return bwd(ct.byref(geo), dtype, pad, 1, stride, ptr, ptr, ptr, ptr, ptr, ptr, 1 << 20, peers, None)
    # null geometry / pointers, bad dtypes and paddings
    assert fwd(None, 0, 0, 1, s222, 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
    assert fwd(ct.byref(g3), 0, 0, 1, None, 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
    assert fwd(ct.byref(g3), 0, 0, 1, s222, None, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
    assert fwd(ct.byref(g3), 0, 0, 1, s222, 16, None, 16, None) == TS_ERR_INVALID_ARGUMENT
    assert fwd(ct.byref(g3), 0, 0, 1, s222, 16, 16, None, None) == TS_ERR_INVALID_ARGUMENT
    assert b(g3, ptr=None) == TS_ERR_INVALID_ARGUMENT
    assert b(g3, stride=None) == TS_ERR_INVALID_ARGUMENT
    assert b(g3, pad=5) == TS_ERR_INVALID_ARGUMENT
    for bad in (7, 0 | TS_WEIGHTS_F32, 1 | TS_WEIGHTS_F32):
        assert fwd(ct.byref(g3), bad, 0, 1, s222, 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
        assert b(g3, dtype=bad) == TS_ERR_INVALID_ARGUMENT
    # served element types: fp32 only
    for other in (1, 2, 3, 2 | TS_WEIGHTS_F32):
        assert fwd(ct.byref(g3), other, 0, 1, s222, 16, 16, 16, None) == TS_ERR_UNSUPPORTED
        assert b(g3, dtype=other) == TS_ERR_UNSUPPORTED
    # strides: entries below 1 are invalid, unserved ones unsupported
    assert fwd(ct.byref(g3), 0, 0, 1, _strides([0, 2, 2]), 16, 16, 16, None) == TS_ERR_INVALID_ARGUMENT
    assert b(g3, stride=_strides([2, -1, 2])) == TS_ERR_INVALID_ARGUMENT
    for st in ([3, 2, 2], [2, 1, 2], [2, 2, 1], [1, 1, 1], [2, 2, 3]):
        assert fwd(ct.byref(g3), 0, 0, 1, _strides(st), 16, 16, 16, None) == TS_ERR_UNSUPPORTED, st
        assert b(g3, stride=_strides(st)) == TS_ERR_UNSUPPORTED, st
    for st in ([1, 2], [2, 1], [3, 3]):
        assert fwd(ct.byref(g2), 0, 0, 1, _strides(st), 16, 16, 16, None) == TS_ERR_UNSUPPORTED, st
    assert fwd(ct.byref(g1), 0, 0, 1, _strides([2]), 16, 16, 16, None) == TS_ERR_UNSUPPORTED
    assert b(g1, stride=_strides([2])) == TS_ERR_UNSUPPORTED
    # peers: checked like ts_shift_backward_nhwc's
    pg = PeerGroup()
    pg.world, pg.rank, pg.capacity = 1, 0, 4096
    pg.bufs[0], pg.state = 4096, None
    assert b(g3, peers=ct.byref(pg)) == TS_ERR_INVALID_ARGUMENT          # no state
    pg.state = 4096
    pg.rank = 1
    assert b(g3, peers=ct.byref(pg)) == TS_ERR_INVALID_ARGUMENT          # rank outside the world
    pg.rank, pg.capacity = 0, 8
    assert b(g3, peers=ct.byref(pg)) == TS_ERR_INVALID_ARGUMENT          # C x dim above the capacity
    pg.capacity, pg.bufs[0] = 4096, 4097
    assert b(g3, peers=ct.byref(pg)) == TS_ERR_INVALID_ARGUMENT          # misaligned buffer
    assert lib.ts_shift_avgpool_backward_workspace_bytes(None, 0) == 16
    assert lib.ts_shift_avgpool_backward_workspace_bytes(ct.byref(g3), 1) == 16
    assert lib.ts_shift_avgpool_backward_workspace_bytes(ct.byref(g1), 0) == 16


def test_functional_rejects_other_strides(lib):
    from torchshifts.functional import shift3d_avgpool_func
    x, w = torch.zeros(1, 2, 4, 4, 8), torch.zeros(2, 3)
    for st in (1, 3, (2, 2, 1), (1, 1, 2), (2, 2), (3, 2, 2), [1, 2, 2, 2]):
        with pytest.raises(ValueError, match="stride"):
            shift3d_avgpool_func(x, w, 0, False, st)
    with pytest.raises(AssertionError):
        shift3d_avgpool_func(x[0], w, 0, False, 2)
    with pytest.raises(AssertionError):
        shift3d_avgpool_func(x, w[:, :2], 0, False, 2)


# ------------------------------------------------------------------------------------------ GPU helpers
def _pool_np(y, st):
    """avg_pool3d(kernel = stride = st, ceil_mode) in ATen's order: one running fp32 sum per window over (slab, row, column),
    divided by the element count."""
    oa, ob, ol = y.shape[2:]
    out = [-(-oa // st[0]), -(-ob // 2), -(-ol // 2)]
    acc = np.zeros(y.shape[:2] + tuple(out), np.float32)
    cnt = np.zeros(out, np.int64)
    for di in range(st[0]):
        for dj in range(2):
            for dk in range(2):
                v = y[:, :, di::st[0], dj::2, dk::2]
                sl = (slice(None), slice(None), slice(0, v.shape[2]), slice(0, v.shape[3]), slice(0, v.shape[4]))
                first = cnt[sl[2:]] == 0
                acc[sl] = np.where(first, v, (acc[sl] + v).astype(np.float32))
                cnt[sl[2:]] += 1
    return (acc / cnt.astype(np.float32)).astype(np.float32)


def _expand_np(gp, st, size):
    """ATen's avg_pool3d_backward for kernel = stride: every element of a window receives grad / count."""
    oa, ob, ol = size
    ia, ib, il = np.arange(oa) // st[0], np.arange(ob) // 2, np.arange(ol) // 2
    ca = np.minimum(st[0] * ia + st[0], oa) - st[0] * ia
    cb = np.minimum(2 * ib + 2, ob) - 2 * ib
    cl = np.minimum(2 * il + 2, ol) - 2 * il
    cnt = (ca[:, None, None] * cb[None, :, None] * cl[None, None, :]).astype(np.float32)
    return (gp[:, :, ia][:, :, :, ib][:, :, :, :, il] / cnt).astype(np.float32)


def _gw_close(gw, gw64, rtol=1e-5):
    scale = np.abs(gw64).max()
    return np.allclose(gw.astype(np.float64), gw64, rtol=rtol, atol=rtol * scale + 1e-30)


def _check_case(lib, oracle_port, dev, x, w, pad, active, st, borders, fused_fwd, fused_bwd, layer=None, oracle=True):
    """Fused operator vs the numpy pooling of the oracle's shift, the two-step path and its autograd, and the oracle backward
    of the numpy-expanded gradient."""
    from torchshifts.functional import shift3d_avgpool_func, shift3d_func
    bt = torch.tensor(borders, dtype=torch.long) if borders is not None else None
    xd = torch.from_numpy(x).to(dev).requires_grad_(True)
    wd = torch.from_numpy(w).to(dev).requires_grad_(True)
    before = lib.ts_launch_count()
    if layer is not None:
        layer.weight.data.copy_(wd.detach())
        out, _ = layer(xd)
        wgrad = lambda: layer.weight.grad          # noqa: E731
    else:
        out = shift3d_avgpool_func(xd, wd, pad, active, st, bt)
        wgrad = lambda: wd.grad                    # noqa: E731
    if fused_fwd:
        assert lib.ts_last_kernel_path() == HALO and lib.ts_launch_count() - before == 1
    x2 = torch.from_numpy(x).to(dev).requires_grad_(True)
    w2 = torch.from_numpy(w).to(dev).requires_grad_(True)
    two = torch.nn.functional.avg_pool3d(shift3d_func(x2, w2, pad, active, bt), st, st, ceil_mode=True)
    assert torch.equal(out, two)
    if oracle:
        y = oracle_port.forward(x, w, pad, active, borders)
        assert np.array_equal(out.detach().cpu().numpy(), _pool_np(y, st))
    g = torch.randn(out.shape, device=dev)
    before = lib.ts_launch_count()
    out.backward(g)
    if fused_bwd:
        assert lib.ts_launch_count() - before == 2          # the shift kernel + the pass-2 reduction
    two.backward(g)
    assert torch.equal(xd.grad, x2.grad)
    assert _gw_close(wgrad().cpu().numpy(), w2.grad.double().cpu().numpy())
    if oracle:
        gy = _expand_np(g.cpu().numpy(), st, y.shape[2:])
        gi_ref, _ = oracle_port.backward(gy, x, w, pad, active, borders)
        assert np.array_equal(xd.grad.cpu().numpy(), gi_ref)
        _, gw64 = oracle_port.backward(gy.astype(np.float64), x.astype(np.float64), w.astype(np.float64), pad, active, borders)
        assert _gw_close(wgrad().cpu().numpy(), gw64)
    return out, xd.grad, wgrad()


def _fused_backward_path(lib, dev, x, w, pad, active, st, borders, g):
    """The kernel path of a direct call of the backward operator (autograd runs it on its own thread)."""
    from torchshifts import _ops
    t = torch.from_numpy(x).to(dev)
    std, new_size = _ops.check_borders(t, torch.tensor(borders) if borders is not None else None, 3)
    torch.ops.torchshifts._shift3d_avgpool_backward(g, torch.from_numpy(w).to(dev), t, std, new_size, list(st), pad, active)
    return lib.ts_last_kernel_path()


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture()
def auto_path(lib):
    lib.ts_set_kernel_path(0)
    lib.ts_set_tuning(b"use_tma=1,use_halo=1,use_flat=1,nhwc_variant=0,nhwc_ring_rows=0")
    yield
    lib.ts_set_kernel_path(0)


# ------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
@pytest.mark.parametrize("st", [(1, 2, 2), (2, 2, 2)])
@pytest.mark.parametrize("pad", range(5))
@pytest.mark.parametrize("active", [False, True])
def test_sweep_against_the_oracle(lib, oracle_port, dev, auto_path, st, pad, active):
    """Every padding, sparse and active, odd slab count (7) and row count (17): bit-exact forward and grad_input."""
    rng = np.random.default_rng(17 + pad)
    x = rng.standard_normal((2, 5, 7, 17, 24)).astype(np.float32)
    w = (rng.uniform(-3, 3, (5, 3))).astype(np.float32)
    _check_case(lib, oracle_port, dev, x, w, pad, active, st, None, True, True)
    g = torch.randn((2, 5, -(-7 // st[0]), 9, 12), device=dev)
    assert _fused_backward_path(lib, dev, x, w, pad, active, st, None, g) == HALO


@pytest.mark.gpu
def test_emulated_depthwise_layers(lib, oracle_port, dev, auto_path):
    """Shift3d(emulate_dw={kernel 3 / 5, padding 0 / 1, stride}): crops, odd extents and the shapes that keep the two-step
    path (rows that are not a multiple of 4 elements; pooled rows that are not a multiple of 16 bytes in the backward)."""
    import torchshifts
    # (shape, padding, active, conv kernel, conv padding, stride, fused forward, fused backward)
    cases = [((2, 4, 9, 20, 24), 'zeros', False, 3, 1, (2, 2, 2), True, True),
             ((2, 4, 8, 17, 36), 'reflect', True, 5, 0, (1, 2, 2), True, True),
             ((2, 3, 11, 22, 28), 'periodic', False, 5, 0, (2, 2, 2), True, True),
             ((2, 3, 7, 15, 32), 'symmetric', True, 5, 0, (2, 2, 2), True, True),
             ((2, 3, 6, 16, 20), 'border', True, 3, 0, (2, 2, 2), False, False),     # rows 20 -> 18: no fused forward
             ((2, 3, 6, 15, 22), 'border', True, 3, 1, (1, 2, 2), False, False),     # rows of 22 elements
             ((2, 3, 5, 16, 20), 'zeros', True, 3, 1, (2, 2, 2), True, False),       # pooled rows of 10: no fused backward
             ((2, 3, 5, 13, 28), 'reflect', False, 5, 1, (1, 2, 2), False, False)]   # crop 1: rows 28 -> 26
    for shape, pad_name, active, ks, cpad, st, ff, fb in cases:
        torch.manual_seed(5)
        m = torchshifts.Shift3d(shape[1], padding=pad_name, active_flag=active, sparsity_term=0,
                                emulate_dw={'kernel_size': ks, 'stride': list(st), 'padding': cpad}).to(dev)
        assert (m.cut_borders is not None) == (2 * cpad - ks + 1 < 0)
        x = np.random.default_rng(3).standard_normal(shape).astype(np.float32)
        w = m.weight.detach().cpu().numpy()
        pad = torchshifts.modules.shifts.paddings_dict[pad_name]
        borders = m.cut_borders.tolist() if m.cut_borders is not None else None
        _check_case(lib, oracle_port, dev, x, w, pad, active, st, borders, ff, fb, layer=m)


@pytest.mark.gpu
def test_scalar_stride_and_module_routing(lib, dev, auto_path):
    import torchshifts
    m = torchshifts.Shift3d(4, emulate_dw={'kernel_size': 3, 'stride': 2, 'padding': 1}).to(dev)
    x = torch.randn(2, 4, 6, 16, 16, device=dev)
    assert m._stride_ints == [2, 2, 2] and m._pool_is_fused(x)
    y, _ = m(x)
    assert y.shape == (2, 4, 3, 8, 8) and lib.ts_last_kernel_path() == HALO
    assert not m._pool_is_fused(x.double()) and not m._pool_is_fused(x.half())
    assert not torchshifts.Shift3d(4, emulate_dw={'kernel_size': 3, 'stride': [2, 1, 2]})._pool_is_fused(x)
    cl = torchshifts.Shift3d(4, emulate_dw={'kernel_size': 3, 'stride': 2, 'padding': 1}, memory_format=torch.preserve_format).to(dev)
    assert not cl._pool_is_fused(x.contiguous(memory_format=torch.channels_last_3d)) and cl._pool_is_fused(x)


@pytest.mark.gpu
def test_shifts_beyond_the_halo_many_channels_and_empty(lib, oracle_port, dev, auto_path):
    rng = np.random.default_rng(9)
    for st in ((1, 2, 2), (2, 2, 2)):
        for pad, active in ((0, True), (3, False), (2, True)):
            x = rng.standard_normal((2, 6, 5, 12, 16)).astype(np.float32)
            w = rng.uniform(-12, 12, (6, 3)).astype(np.float32)      # most channels reach beyond the 4-cell halo
            w[:2] = rng.uniform(-1, 1, (2, 3))
            _check_case(lib, oracle_port, dev, x, w, pad, active, st, None, True, True)
    # more channels than the shift table holds (C = 520): run-time window classes
    x = rng.standard_normal((1, 520, 3, 8, 16)).astype(np.float32)
    w = rng.uniform(-2, 2, (520, 3)).astype(np.float32)
    _check_case(lib, oracle_port, dev, x, w, 3, True, (2, 2, 2), None, True, True)
    # N = 0: empty output, zero grad_weight
    from torchshifts.functional import shift3d_avgpool_func
    x0 = torch.zeros(0, 4, 6, 8, 16, device=dev, requires_grad=True)
    w0 = torch.randn(4, 3, device=dev, requires_grad=True)
    y0 = shift3d_avgpool_func(x0, w0, 0, True, 2)
    assert y0.shape == (0, 4, 3, 4, 8)
    y0.sum().backward()
    assert x0.grad.shape == x0.shape and torch.equal(w0.grad, torch.zeros_like(w0))


@pytest.mark.gpu
def test_grad_weight_is_identical_from_run_to_run(dev, auto_path):
    from torchshifts.functional import shift3d_avgpool_func
    torch.manual_seed(4)
    x = torch.randn(8, 32, 9, 28, 32, device=dev)
    g = None
    for st in ((1, 2, 2), (2, 2, 2)):
        for pad, active in ((0, False), (3, True)):
            grads = []
            for _ in range(3):
                w = (torch.rand(32, 3, device=dev) * 4 - 2).requires_grad_(True) if not grads else w.detach().requires_grad_(True)
                y = shift3d_avgpool_func(x, w, pad, active, st)
                g = torch.randn_like(y) if g is None or g.shape != y.shape else g
                y.backward(g)
                grads.append(w.grad.clone())
            assert torch.equal(grads[0], grads[1]) and torch.equal(grads[0], grads[2])


@pytest.mark.gpu
@pytest.mark.parametrize("pad,active", [(3, True), (0, False)])
def test_cfg4_stride_2(lib, oracle_port, dev, auto_path, pad, active):
    """cfg4 (32, 128, 16, 56, 56), stride (2, 2, 2): the fused kernels serve both passes; sampled images against the oracle,
    the whole tensor against the two-step path."""
    from torchshifts.functional import shift3d_avgpool_func, shift3d_func
    torch.manual_seed(11)
    st = (2, 2, 2)
    x = torch.randn(32, 128, 16, 56, 56, device=dev)
    w = ((torch.rand(128, 3, device=dev) * 2 - 1) * 3).requires_grad_(True)
    xr = x.clone().requires_grad_(True)
    y = shift3d_avgpool_func(xr, w, pad, active, st)
    assert lib.ts_last_kernel_path() == HALO and y.shape == (32, 128, 8, 28, 28)
    g = torch.randn_like(y)
    before = lib.ts_launch_count()
    y.backward(g)
    assert lib.ts_launch_count() - before == 2
    std = torch.tensor([0, 16, 0, 56, 0, 56], dtype=torch.int32)
    torch.ops.torchshifts._shift3d_avgpool_backward(g, w.detach(), x, std, list(x.shape), list(st), pad, active)
    assert lib.ts_last_kernel_path() == HALO
    w2 = w.detach().clone().requires_grad_(True)
    x2 = x.clone().requires_grad_(True)
    two = torch.nn.functional.avg_pool3d(shift3d_func(x2, w2, pad, active), st, st, ceil_mode=True)
    assert torch.equal(y, two)
    two.backward(g)
    assert torch.equal(xr.grad, x2.grad)
    assert _gw_close(w.grad.cpu().numpy(), w2.grad.double().cpu().numpy())
    wn = w.detach().cpu().numpy()
    for n in (0, 31):
        xn = x[n:n + 1].cpu().numpy()
        yo = oracle_port.forward(xn, wn, pad, active)
        assert np.array_equal(y[n:n + 1].detach().cpu().numpy(), _pool_np(yo, st)), n
        gy = _expand_np(g[n:n + 1].cpu().numpy(), st, (16, 56, 56))
        gi, _ = oracle_port.backward(gy, xn, wn, pad, active)
        assert np.array_equal(xr.grad[n:n + 1].cpu().numpy(), gi), n


@pytest.mark.gpu
def test_fused_layer_saves_a_full_size_tensor_of_memory(dev, auto_path):
    """One training step of a Shift3d stride layer on a cfg4-sized tensor: the two-step path keeps the full-size shift
    output alive for avg_pool3d's backward and allocates the full-size gradient; the fused layer does neither."""
    import torchshifts
    from torchshifts.functional import shift3d_func
    m = torchshifts.Shift3d(128, padding='reflect', active_flag=True, sparsity_term=0,
                            emulate_dw={'kernel_size': 3, 'stride': 2, 'padding': 1}).to(dev)
    x = torch.randn(32, 128, 16, 56, 56, device=dev, requires_grad=True)
    full = x.numel() * x.element_size()

    def peak(step):
        x.grad = None
        m.weight.grad = None
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        step()
        torch.cuda.synchronize()
        return torch.cuda.max_memory_allocated() - base

    def fused():
        y, _ = m(x)
        y.sum().backward()

    def two_step():
        y = torch.nn.functional.avg_pool3d(shift3d_func(x, m.weight, m.padding, True), 2, 2, ceil_mode=True)
        y.sum().backward()
    fused(), two_step()                       # warm-up: allocator pools
    p_fused, p_two = peak(fused), peak(two_step)
    assert p_two - p_fused >= 0.9 * full, (p_fused / 2**20, p_two / 2**20, full / 2**20)


@pytest.mark.gpu
def test_torch_compile_cropping_stride_layer(dev, auto_path):
    import torchshifts
    torch.manual_seed(2)
    m = torchshifts.Shift3d(6, padding='symmetric', active_flag=True, sparsity_term=0,
                            emulate_dw={'kernel_size': 5, 'stride': [1, 2, 2], 'padding': 0}).to(dev)
    assert m.cut_borders is not None
    x = torch.randn(2, 6, 7, 18, 28, device=dev)

    def f(t):
        y, _ = m(t)
        return y * 2.0
    xe = x.clone().requires_grad_(True)
    want = f(xe)
    want.sum().backward()
    gx, gw = xe.grad.clone(), m.weight.grad.clone()
    m.weight.grad = None
    xc = x.clone().requires_grad_(True)
    got = torch.compile(f, dynamic=False, backend="aot_eager", fullgraph=True)(xc)
    assert torch.equal(got, want)
    got.sum().backward()
    assert torch.equal(xc.grad, gx) and torch.equal(m.weight.grad, gw)


@pytest.mark.gpu
def test_fused_exchange_of_pooled_layers(dev, auto_path):
    """Under FusedGradWeightAllReduce the fused pooled backward (2-D stride 2 and 3-D) takes part in the in-kernel exchange:
    one exchange per layer backward, weight.grad equal to the plain backward's (one rank: the sum is the local value)."""
    import torchshifts
    from torchshifts.sharded import FusedGradWeightAllReduce
    fused = FusedGradWeightAllReduce(None, device=dev)
    cases = [(torchshifts.Shift2d(16, padding='reflect', active_flag=True, sparsity_term=0,
                                  emulate_dw={'kernel_size': 3, 'stride': 2, 'padding': 1}), (4, 16, 32, 32)),
             (torchshifts.Shift3d(16, padding='zeros', active_flag=False, sparsity_term=0,
                                  emulate_dw={'kernel_size': 3, 'stride': 2, 'padding': 1}), (2, 16, 6, 16, 16))]
    for m, shape in cases:
        m = m.to(dev)
        x = torch.randn(shape, device=dev, requires_grad=True)
        y, _ = m(x)
        g = torch.randn_like(y)
        y.backward(g)
        plain_w, plain_x = m.weight.grad.clone(), x.grad.clone()
        m.weight.grad, x.grad = None, None
        with fused:
            calls = fused.calls()
            y, _ = m(x)
            y.backward(g)
            torch.cuda.synchronize()
            assert fused.calls() == calls + 1, type(m).__name__
        assert torch.equal(m.weight.grad, plain_w), type(m).__name__
        assert torch.equal(x.grad, plain_x), type(m).__name__
