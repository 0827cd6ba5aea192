"""Definition of the ``torchshifts::`` operators on top of the C ABI.

Operator names and schemas are the reference's (csrc/torchshifts.cpp:35-40, csrc/ops/shifts.cpp:168-181):

    torchshifts::_cuda_version() -> int
    torchshifts::shift{1,2,3}d(Tensor input, Tensor weights, Tensor borders, int padding_mode, bool active_flag) -> Tensor
    torchshifts::_shift{1,2,3}d_forward(Tensor input, Tensor weights, Tensor borders, int[] new_size,
                                        int padding_mode, bool active_flag) -> Tensor
    torchshifts::_shift{1,2,3}d_backward(Tensor grad, Tensor weights, Tensor input, Tensor borders,
                                         int padding_mode, bool active_flag) -> (Tensor, Tensor)

Extension over the reference (the functional layer routes channels-last inputs here under
``memory_format=torch.preserve_format``; the reference's float path always returns NCHW):

    torchshifts::_shift{2,3}d_forward_cl(Tensor input, Tensor weights, Tensor borders, int[] new_size,
                                         int padding_mode, bool active_flag) -> Tensor
    torchshifts::_shift{2,3}d_backward_cl(Tensor grad, Tensor weights, Tensor input, Tensor borders,
                                          int padding_mode, bool active_flag) -> (Tensor, Tensor)

same arguments and values as ``_shiftNd_forward/_backward``, but the output and ``grad_input`` are dense
channels-last (``channels_last`` / ``channels_last_3d``).

Dispatch keys: ``shiftNd`` is CompositeImplicitAutograd (border validation, then ``_shiftNd_forward``);
``_shiftNd_forward/_backward`` carry the autograd wiring of csrc/ops/autograd/shifts_autograd.cpp
(``torch.library.register_autograd``: saves input/weights/borders, double backward is an error),
``CUDA`` and ``QuantizedCUDA`` kernels that call the sm_100a library, fake kernels for tracing,
and ``CPU`` / ``QuantizedCPU`` kernels that raise: this build has NO CPU compute path.
"""
import collections
import contextlib
import ctypes as ct
import weakref

import torch

from ._cabi import QW_I8, QW_I32, QW_U8, make_geometry

_LIB = None            # torch.library.Library handle (kept alive)
_FUSED_ALLREDUCE = None   # torchshifts.sharded.FusedGradWeightAllReduce while enabled: grad_weight is summed over the ranks in-kernel
_NATIVE = None         # NativeLibrary
_DTYPES = {torch.float32: 0, torch.float64: 1, torch.float16: 2, torch.bfloat16: 3}
_QKINDS = {torch.quint8: QW_U8, torch.qint8: QW_I8, torch.qint32: QW_I32}
_QBYTES = {torch.quint8: 1, torch.qint8: 1, torch.qint32: 4}


def _no_cpu(*args, **kwargs):
    raise RuntimeError(
        'torchshifts-b200 has no CPU implementation of the shift operator (no CPU fallback by design): '
        'move the input and the weights to a CUDA device (B200 / sm_100a).')


def _check_mode(padding_mode):
    # the reference's switch has no default and returns an undefined tensor (cpu/shifts_cpu.cpp:267-289)
    if padding_mode not in (0, 1, 2, 3, 4):
        raise RuntimeError(f'torchshifts: padding_mode must be 0..4 (zeros, border, periodic, reflect, symmetric), got {padding_mode}')


def _borders_lists(borders, dim):
    """``borders`` is the int32[6] tensor {l0,r0,l1,r1,l2,r2} produced by check_borders."""
    b = borders.tolist() if borders.device.type == 'cpu' else borders.cpu().tolist()
    if len(b) < 6:
        raise RuntimeError('torchshifts: internal borders tensor must have 6 entries')
    return [b[0], b[2], b[4]], [b[1], b[3], b[5]]


def _same_device_and_type(fn, input, weights, grad=None):
    # checkAllSameGPU / checkAllSameType of cuda/shifts_cuda.cu:213-214, :282-283
    if weights.device != input.device or (grad is not None and grad.device != input.device):
        raise RuntimeError(f'{fn}: expected input, weights' + (', grad' if grad is not None else '') +
                           f' to be on the same GPU, but got {input.device}, {weights.device}' +
                           (f', {grad.device}' if grad is not None else ''))
    if weights.dtype != input.dtype or (grad is not None and grad.dtype != input.dtype):
        raise RuntimeError(f'{fn}: expected scalar type {input.dtype} for every tensor but found '
                           f'weights {weights.dtype}' + (f', grad {grad.dtype}' if grad is not None else ''))
    if input.dtype not in _DTYPES:
        raise RuntimeError(f'{fn}: "shiftnd_cuda" not implemented for {input.dtype}')


_COPY_THRESHOLD = 1 << 16


_CL_FORMATS = {4: torch.channels_last, 5: torch.channels_last_3d}


_PLANAR = collections.OrderedDict()     # (data_ptr, shape, strides, version) -> planar copy made by the forward, for the backward
_PLANAR_MAX = 2
_LAST_PLANAR = [None]                   # (key, copy) of the forward that just ran, until autograd claims it (or the composite returns)


def _dense(input, keep=False, take=False):
    """Channels-last / sliced inputs: the stride-aware generic kernels read them in place, but their
    per-element strided loads waste most of every 32-byte sector.  Above a few tens of thousands of
    elements one extra coalesced pass plus the bandwidth kernels is several times faster: a dense
    channels-last tensor goes through the library's own tiled transpose (``ts_nhwc_to_nchw``), anything
    else through ``.contiguous()``.

    ``keep`` (forward): park the planar copy in ``_LAST_PLANAR``; when autograd records the call,
    ``_setup_forward_context`` -- the one place that knows the call is differentiated: the CUDA kernel runs below the
    Autograd key, with grad mode off -- moves it to ``_PLANAR``, otherwise the composite drops it when the operator
    returns.  ``take`` (backward): reuse that copy instead of converting the saved input a second time (0.26 ms per step
    for cfg3) -- at most ``_PLANAR_MAX`` copies are held."""
    if input.numel() < _COPY_THRESHOLD or input.is_contiguous():
        return input
    key = _planar_key(input)
    if take:
        hit = _PLANAR.pop(key, None)
        if hit is not None:
            return hit
    fmt = _CL_FORMATS.get(input.dim())
    if fmt is not None and input.is_contiguous(memory_format=fmt) and input.element_size() in (2, 4, 8):
        out = torch.empty(input.shape, dtype=input.dtype, device=input.device)
        n, c = input.shape[0], input.shape[1]
        with _guard(input.device):
            st = _NATIVE.lib.ts_nhwc_to_nchw(input.data_ptr(), out.data_ptr(), n, c, input.numel() // max(n * c, 1),
                                             input.element_size(), _stream(input.device))
        _NATIVE.check(st, 'ts_nhwc_to_nchw')
    else:
        out = input.contiguous()
    if keep:
        _LAST_PLANAR[0] = (key, out)
    return out


def _planar_key(input):
    return (input.data_ptr(), tuple(input.shape), tuple(input.stride()), input._version, input.dtype)


def _claim_planar(input):
    """Called while autograd records a forward: keep the planar copy that forward made for its backward."""
    last, _LAST_PLANAR[0] = _LAST_PLANAR[0], None
    if last is None or isinstance(input, torch._subclasses.FakeTensor):
        return
    if last[0] == _planar_key(input):
        _PLANAR[last[0]] = last[1]
        while len(_PLANAR) > _PLANAR_MAX:
            _PLANAR.popitem(last=False)


def _stream(device):
    return ct.c_void_p(torch._C._cuda_getCurrentRawStream(device.index))


_NO_GUARD = contextlib.nullcontext()


def _guard(device):
    """CUDAGuard of cuda/shifts_cuda.cu:215, :284 -- skipped (it costs ~10 us in Python) when the tensor's device
    already is the current one."""
    return _NO_GUARD if device.index == torch._C._cuda_getDevice() else torch.cuda.device(device)


_GEO_CACHE = {}        # (dim, shape, strides, lb, rb) -> ts_geometry; shift layers see the same few shapes every step
_WS_CACHE = {}         # (geometry key, dtype code, device index) -> backward workspace bytes


def _geometry(dim, input, lb, rb):
    """-> (ts_geometry, its cache key)"""
    key = (dim, tuple(input.shape), tuple(input.stride()), tuple(lb), tuple(rb))
    geo = _GEO_CACHE.get(key)
    if geo is None:
        if len(_GEO_CACHE) > 256:
            _GEO_CACHE.clear()
            _WS_CACHE.clear()
        geo = _GEO_CACHE[key] = make_geometry(dim, input.shape, input.stride(), lb, rb)
    return geo, key


def _workspace_bytes(geo, key, code, device):
    wkey = (key, code, device.index)
    n = _WS_CACHE.get(wkey)
    if n is None:
        if len(_WS_CACHE) > 256:
            _WS_CACHE.clear()
        n = _WS_CACHE[wkey] = int(_NATIVE.lib.ts_shift_backward_workspace_bytes(ct.byref(geo), code))
    return n


# ------------------------------------------------------------------------------------------ CUDA
def _check_forward(fn, dim, input, weights, padding_mode):
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights)
    if input.dim() != dim + 2:
        raise RuntimeError(f'{fn}: expected a {dim + 2}-D input, got {input.dim()}-D')
    if weights.dim() != 2 or weights.shape[0] != input.shape[1] or weights.shape[1] != dim:
        raise RuntimeError(f'{fn}: weights must be [{input.shape[1]}, {dim}], got {list(weights.shape)}')


def _forward_cuda(dim, input, weights, borders, new_size, padding_mode, active_flag):
    fn = f'shift{dim}d_forward'
    _check_forward(fn, dim, input, weights, padding_mode)
    lb, rb = _borders_lists(borders, dim)
    out = torch.empty(list(new_size), dtype=input.dtype, device=input.device)
    w = weights.contiguous()
    input = _dense(input, keep=True)
    geo, _ = _geometry(dim, input, lb, rb)
    if list(out.shape[2:]) != [rb[a] - lb[a] for a in range(dim)]:
        raise RuntimeError(f'{fn}: new_size {list(new_size)} does not match the borders')
    with _guard(input.device):
        st = _NATIVE.lib.ts_shift_forward(ct.byref(geo), _DTYPES[input.dtype], int(padding_mode), int(bool(active_flag)),
                                          input.data_ptr(), w.data_ptr(), out.data_ptr(), _stream(input.device))
    if st:
        _NATIVE.check(st, 'ts_shift_forward')
    return out


def _pool_forward_cuda(input, weights, borders, new_size, padding_mode, active_flag):
    """Shift2d forward + avg_pool2d(kernel 2, stride 2, ceil_mode=True) in ONE kernel (ts_shift2d_avgpool2_forward): one
    read of x, one quarter-size write.  Shapes the fused kernel does not serve (non-fp32, odd row lengths, strided
    inputs, planes too large to stage) run the two steps separately -- same values."""
    fn = 'shift2d_avgpool2_forward'
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights)
    lb, rb = _borders_lists(borders, 2)
    oh, ow = rb[0] - lb[0], rb[1] - lb[1]
    if input.dtype == torch.float32 and input.is_contiguous() and ow % 4 == 0 and input.dim() == 4:
        out = torch.empty((input.shape[0], input.shape[1], (oh + 1) // 2, ow // 2), dtype=input.dtype, device=input.device)
        w = weights.contiguous()
        geo, _ = _geometry(2, input, lb, rb)
        with _guard(input.device):
            st = _NATIVE.lib.ts_shift2d_avgpool2_forward(ct.byref(geo), 0, int(padding_mode), int(bool(active_flag)), input.data_ptr(),
                                                         w.data_ptr(), out.data_ptr(), _stream(input.device))
        if st == 0:
            return out
        if st != 2:        # TS_ERR_UNSUPPORTED: fall through to the two-step path
            _NATIVE.check(st, 'ts_shift2d_avgpool2_forward')
    y = _forward_cuda(2, input, weights, borders, new_size, padding_mode, active_flag)
    return torch.nn.functional.avg_pool2d(y, kernel_size=2, stride=2, ceil_mode=True)


def _pool_forward_meta(input, weights, borders, new_size, padding_mode, active_flag):
    return input.new_empty([new_size[0], new_size[1], (new_size[2] + 1) // 2, (new_size[3] + 1) // 2])


def _pool_setup_context(ctx, inputs, output):
    input, weights, borders, new_size, padding_mode, active_flag = inputs
    ctx.save_for_backward(input, weights, borders)
    ctx.padding_mode, ctx.active_flag, ctx.new_size = padding_mode, active_flag, list(new_size)


def _pool_backward(ctx, grad_pooled):
    input, weights, borders = ctx.saved_tensors
    op = torch.ops.torchshifts._shift2d_avgpool2_backward
    grad_input, grad_weight = op(grad_pooled, weights, input, borders, ctx.new_size, ctx.padding_mode, ctx.active_flag)
    return grad_input, grad_weight, None, None, None, None


def _pool_backward_cuda(grad_pooled, weights, input, borders, new_size, padding_mode, active_flag):
    """Backward of the fused shift + avg_pool2d(2, 2, ceil_mode): ONE kernel (ts_shift2d_avgpool2_backward) that expands the
    pooled gradient while staging it -- the full-size gradient of the shift's output never exists in HBM.  Shapes the fused
    kernel does not serve take ATen's avg_pool2d_backward followed by the shift backward (same values)."""
    fn = 'shift2d_avgpool2_backward'
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights, grad_pooled)
    lb, rb = _borders_lists(borders, 2)
    oh, ow = rb[0] - lb[0], rb[1] - lb[1]
    if list(grad_pooled.shape) != [input.shape[0], input.shape[1], (oh + 1) // 2, (ow + 1) // 2]:
        raise RuntimeError(f'{fn}: grad has shape {list(grad_pooled.shape)}, the pooled output is '
                           f'{[input.shape[0], input.shape[1], (oh + 1) // 2, (ow + 1) // 2]}')
    if input.dtype == torch.float32 and input.is_contiguous() and ow % 8 == 0 and input.dim() == 4 and input.numel() > 0:
        grad = grad_pooled.contiguous()
        w = weights.contiguous()
        out_grad = torch.empty(input.shape, dtype=input.dtype, device=input.device)
        weights_grad = torch.empty(w.shape, dtype=w.dtype, device=w.device)
        geo, key = _geometry(2, input, lb, rb)
        dev = input.device
        with _guard(dev):
            for attempt in (0, 1):
                nbytes = _workspace_bytes(geo, key, 0, dev)
                workspace = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
                st = _NATIVE.lib.ts_shift2d_avgpool2_backward(ct.byref(geo), 0, int(padding_mode), int(bool(active_flag)), grad.data_ptr(),
                                                              input.data_ptr(), w.data_ptr(), out_grad.data_ptr(), weights_grad.data_ptr(),
                                                              workspace.data_ptr(), nbytes, _stream(dev))
                if st != 3:
                    break
                _WS_CACHE.clear()
        if st == 0:
            return out_grad, weights_grad
        if st != 2:        # TS_ERR_UNSUPPORTED: fall through to the two-step path
            _NATIVE.check(st, 'ts_shift2d_avgpool2_backward')
    like = torch.empty(list(new_size), dtype=grad_pooled.dtype, device=grad_pooled.device)
    grad_y = torch.ops.aten.avg_pool2d_backward(grad_pooled.contiguous(), like, [2, 2], [2, 2], [0, 0], True, True, None)
    return _backward_cuda(2, grad_y, weights, input, borders, padding_mode, active_flag)


def _pool_backward_meta(grad_pooled, weights, input, borders, new_size, padding_mode, active_flag):
    return input.new_empty(input.shape), weights.new_empty(weights.shape)


def _check_fused(fn, fused, dev, code, weight_numel):
    # Taking part in the in-kernel exchange must never depend on rank-local data (an empty shard, a ragged last
    # batch): a rank that skipped it would leave its peers waiting.  What cannot be served raises on EVERY rank
    # (dtype, weight count and device are the same everywhere for replicated layers).
    if fused.device != dev:
        raise RuntimeError(f'{fn}: FusedGradWeightAllReduce was created for {fused.device} but the tensors live on {dev}')
    if code == 1:
        raise RuntimeError(f'{fn}: the fused grad_weight all-reduce carries fp32 contributions; float64 layers must use '
                           'torchshifts.sharded.allreduce_grad_weights (disable() the fused mode around them)')
    if weight_numel > fused.capacity:
        raise RuntimeError(f'{fn}: {weight_numel} weight elements exceed the exchange capacity {fused.capacity} '
                           '(FusedGradWeightAllReduce(capacity=...), at most 4096)')


def _backward_cuda(dim, grad, weights, input, borders, padding_mode, active_flag):
    fn = f'shift{dim}d_backward'
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights, grad)
    lb, rb = _borders_lists(borders, dim)
    grad = grad.contiguous()
    w = weights.contiguous()
    out_grad = torch.empty(input.shape, dtype=input.dtype, device=input.device)
    weights_grad = torch.empty(w.shape, dtype=w.dtype, device=w.device)
    input = _dense(input, take=True)
    geo, key = _geometry(dim, input, lb, rb)
    if list(grad.shape[2:]) != [rb[a] - lb[a] for a in range(dim)] or list(grad.shape[:2]) != list(input.shape[:2]):
        raise RuntimeError(f'{fn}: grad shape {list(grad.shape)} does not match the (cropped) output of input {list(input.shape)}')
    code = _DTYPES[input.dtype]
    dev = input.device
    fused = _FUSED_ALLREDUCE
    if fused is not None:
        _check_fused(fn, fused, dev, code, w.numel())
    with _guard(dev):
        for attempt in (0, 1):
            nbytes = _workspace_bytes(geo, key, code, dev)
            workspace = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
            args = (ct.byref(geo), code, int(padding_mode), int(bool(active_flag)), grad.data_ptr(), input.data_ptr(), w.data_ptr(),
                    out_grad.data_ptr(), weights_grad.data_ptr(), workspace.data_ptr(), nbytes)
            if fused is not None:
                st = _NATIVE.lib.ts_shift_backward_allreduce(*args, ct.byref(fused.peer_group()), _stream(dev))
            else:
                st = _NATIVE.lib.ts_shift_backward(*args, _stream(dev))
            if st != 3:       # TS_ERR_WORKSPACE (nothing was launched): the tuning knobs changed since the size was cached
                break
            _WS_CACHE.clear()
    if st:
        _NATIVE.check(st, 'ts_shift_backward_allreduce' if fused is not None else 'ts_shift_backward')
    return out_grad, weights_grad


# ------------------------------------------------------------------------------------------ CUDA, channels-last
_CL_WS_CACHE = {}      # (geometry key, dtype code, device index) -> workspace bytes of ts_shift_backward_nhwc


def _cl_workspace_bytes(geo, key, code, device):
    wkey = (key, code, device.index)
    n = _CL_WS_CACHE.get(wkey)
    if n is None:
        if len(_CL_WS_CACHE) > 256:
            _CL_WS_CACHE.clear()
        with _guard(device):
            n = _CL_WS_CACHE[wkey] = int(_NATIVE.lib.ts_shift_backward_nhwc_workspace_bytes(ct.byref(geo), code))
    return n


def _forward_cl_cuda(dim, input, weights, borders, new_size, padding_mode, active_flag):
    """``_shiftNd_forward`` with a dense channels-last output.  2-D dense channels-last fp32 / fp16 / bf16 inputs run the
    native NHWC kernel (ts_shift_forward_nhwc: one read, one write, no layout pass); whatever it does not serve takes the
    planar forward and converts its output -- the same values."""
    fn = f'shift{dim}d_forward_cl'
    fmt = _CL_FORMATS[dim + 2]
    _check_forward(fn, dim, input, weights, padding_mode)
    if dim == 2 and input.dtype != torch.float64 and input.shape[1] % 32 == 0 and input.is_contiguous(memory_format=fmt):
        lb, rb = _borders_lists(borders, dim)
        if list(new_size) != list(input.shape[:2]) + [rb[a] - lb[a] for a in range(dim)]:
            raise RuntimeError(f'{fn}: new_size {list(new_size)} does not match the borders')
        out = torch.empty(list(new_size), dtype=input.dtype, device=input.device, memory_format=fmt)
        w = weights.contiguous()
        geo, _ = _geometry(dim, input, lb, rb)
        with _guard(input.device):
            st = _NATIVE.lib.ts_shift_forward_nhwc(ct.byref(geo), _DTYPES[input.dtype], int(padding_mode), int(bool(active_flag)),
                                                   input.data_ptr(), w.data_ptr(), out.data_ptr(), _stream(input.device))
        if st == 0:
            return out
        if st != 2:        # TS_ERR_UNSUPPORTED: the planar path below
            _NATIVE.check(st, 'ts_shift_forward_nhwc')
    return _forward_cuda(dim, input, weights, borders, new_size, padding_mode, active_flag).contiguous(memory_format=fmt)


def _backward_cl_cuda(dim, grad, weights, input, borders, padding_mode, active_flag):
    """``_shiftNd_backward`` with a dense channels-last ``grad_input``.  ``grad`` may arrive in any layout (an expanded
    tensor from ``.sum()``, say): the native kernel (ts_shift_backward_nhwc) reads it dense channels-last.  What the
    kernel does not serve takes the planar backward and converts ``grad_input`` -- the same values."""
    fn = f'shift{dim}d_backward_cl'
    fmt = _CL_FORMATS[dim + 2]
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights, grad)
    code = _DTYPES[input.dtype]
    dev = input.device
    fused = _FUSED_ALLREDUCE
    if fused is not None:
        _check_fused(fn, fused, dev, code, weights.numel())
    nbytes = 0
    if dim == 2 and code != 1 and input.dim() == 4 and input.shape[1] % 32 == 0 and input.is_contiguous(memory_format=fmt):
        lb, rb = _borders_lists(borders, dim)
        geo, key = _geometry(dim, input, lb, rb)
        nbytes = _cl_workspace_bytes(geo, key, code, dev)
    # 16 bytes: the kernel does not serve this geometry -- decided before grad is converted to a layout the planar path
    # would convert again
    for attempt in (0, 1):
        if nbytes <= 16:
            break
        if list(grad.shape[2:]) != [rb[a] - lb[a] for a in range(dim)] or list(grad.shape[:2]) != list(input.shape[:2]):
            raise RuntimeError(f'{fn}: grad shape {list(grad.shape)} does not match the (cropped) output of input {list(input.shape)}')
        grad_cl = grad.contiguous(memory_format=fmt)
        w = weights.contiguous()
        out_grad = torch.empty(input.shape, dtype=input.dtype, device=dev, memory_format=fmt)
        weights_grad = torch.empty(w.shape, dtype=w.dtype, device=dev)
        workspace = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        with _guard(dev):
            st = _NATIVE.lib.ts_shift_backward_nhwc(ct.byref(geo), code, int(padding_mode), int(bool(active_flag)), grad_cl.data_ptr(),
                                                    input.data_ptr(), w.data_ptr(), out_grad.data_ptr(), weights_grad.data_ptr(),
                                                    workspace.data_ptr(), nbytes,
                                                    ct.byref(fused.peer_group()) if fused is not None else None, _stream(dev))
        if st == 0:
            return out_grad, weights_grad
        if st == 2:        # TS_ERR_UNSUPPORTED (e.g. a misaligned view): the planar path below
            break
        if st != 3:
            _NATIVE.check(st, 'ts_shift_backward_nhwc')
        _CL_WS_CACHE.clear()      # TS_ERR_WORKSPACE (nothing was launched): the tuning knobs changed since the size was cached
        nbytes = _cl_workspace_bytes(geo, key, code, dev)
    else:
        _NATIVE.check(st, 'ts_shift_backward_nhwc')
    grad_input, grad_weight = _backward_cuda(dim, grad, weights, input, borders, padding_mode, active_flag)
    return grad_input.contiguous(memory_format=fmt), grad_weight


_QW_CACHE = {}         # id(quantized weight) -> (weakref, version, device, raw integer weights on that device)


def _raw_qweights(weights, device):
    """``weights.int_repr()`` on ``device``, memoised per weight tensor (a quantized layer presents the same
    tensor on every forward; int_repr + copy are two ATen launches otherwise)."""
    hit = _QW_CACHE.get(id(weights))
    if hit is not None and hit[0]() is weights and hit[1] == weights._version and hit[2] == device:
        return hit[3]
    wq = weights.int_repr().to(device).contiguous()
    if len(_QW_CACHE) > 64:
        _QW_CACHE.clear()
    _QW_CACHE[id(weights)] = (weakref.ref(weights), weights._version, device, wq)
    return wq


def _forward_qcuda(dim, input, weights, borders, new_size, padding_mode, active_flag):
    fn = f'q_shift{dim}d_cuda'
    _check_mode(padding_mode)
    if not weights.is_quantized:
        raise RuntimeError(f'{fn}: weights must be a quantized tensor (see torchshifts.quantized.modules.shifts.quantize_shift_weights)')
    if input.qscheme() not in (torch.per_tensor_affine, torch.per_tensor_symmetric):
        raise RuntimeError(f'{fn}: only per-tensor quantized inputs are supported')
    if input.dtype not in _QBYTES or weights.dtype not in _QKINDS:
        raise RuntimeError(f'{fn}: unsupported quantized dtype {input.dtype} / {weights.dtype}')
    lb, rb = _borders_lists(borders, dim)
    if list(new_size[2:]) != [rb[a] - lb[a] for a in range(dim)] or list(new_size[:2]) != list(input.shape[:2]):
        raise RuntimeError(f'{fn}: new_size {list(new_size)} does not match the borders')
    wq = _raw_qweights(weights, input.device)
    args = (_QBYTES[input.dtype], int(padding_mode), int(input.q_zero_point()))
    wargs = (wq.data_ptr(), _QKINDS[weights.dtype], int(weights.q_zero_point()))
    # the reference allocates the quantized output in the input's memory format
    # (quantized/shifts_quantized.cpp:119-122): channels-last in, channels-last out -- served by the
    # native NHWC kernel (one read + one write, no layout conversion on either side)
    fmt = {2: torch.channels_last, 3: torch.channels_last_3d}.get(dim)
    if fmt is not None and not input.is_contiguous() and input.is_contiguous(memory_format=fmt):
        to_cl = (0,) + tuple(range(2, dim + 2)) + (1,)
        to_nc = (0, dim + 1) + tuple(range(1, dim + 1))
        out_cl = torch._empty_affine_quantized([new_size[i] for i in to_cl], scale=input.q_scale(),
                                               zero_point=input.q_zero_point(), dtype=input.dtype, device=input.device)
        geo, _ = _geometry(dim, input, lb, rb)
        with _guard(input.device):
            st = _NATIVE.lib.ts_qshift_forward_nhwc(ct.byref(geo), *args, input.data_ptr(), *wargs, out_cl.data_ptr(),
                                                    _stream(input.device))
        if st not in (2, 4):      # TS_ERR_UNSUPPORTED / TOO_LARGE (row offsets beyond 32 bits): planar kernels + conversions
            _NATIVE.check(st, 'ts_qshift_forward_nhwc')
            return out_cl.permute(*to_nc)
        del out_cl
    x = input if input.is_contiguous() else input.contiguous()
    out = torch._empty_affine_quantized(list(new_size), scale=input.q_scale(), zero_point=input.q_zero_point(),
                                        dtype=input.dtype, device=input.device)
    geo, _ = _geometry(dim, x, lb, rb)
    with _guard(input.device):
        st = _NATIVE.lib.ts_qshift_forward(ct.byref(geo), *args, x.data_ptr(), *wargs, out.data_ptr(), _stream(input.device))
    _NATIVE.check(st, 'ts_qshift_forward')
    if x is not input and fmt is not None and input.is_contiguous(memory_format=fmt):
        out = out.contiguous(memory_format=fmt)
    return out


def _backward_quantized(dim, *args):
    # quantized/shifts_quantized.cpp:218-225
    raise RuntimeError(f'torchshifts::_shift{dim}d_backward: backward is not supported for quantized tensors')


# ------------------------------------------------------------------------------------------ Meta
def _forward_meta(dim, input, weights, borders, new_size, padding_mode, active_flag):
    return input.new_empty(list(new_size))


def _backward_meta(dim, grad, weights, input, borders, padding_mode, active_flag):
    return input.new_empty(input.shape), weights.new_empty(weights.shape)


def _forward_cl_meta(dim, input, weights, borders, new_size, padding_mode, active_flag):
    return torch.empty(list(new_size), dtype=input.dtype, device=input.device, memory_format=_CL_FORMATS[dim + 2])


def _backward_cl_meta(dim, grad, weights, input, borders, padding_mode, active_flag):
    return (torch.empty(input.shape, dtype=input.dtype, device=input.device, memory_format=_CL_FORMATS[dim + 2]),
            weights.new_empty(weights.shape))


# ------------------------------------------------------------------------------------------ Autograd
# csrc/ops/autograd/shifts_autograd.cpp:15-47 (and the 2d/3d twins): forward saves input, weights and
# borders; backward calls _shiftNd_backward and returns grads for input and weights only; the backward
# op itself is not differentiable (:50-72).  Registered with torch.library.register_autograd (not an
# Autograd-key kernel wrapping an autograd.Function) so that AOTAutograd / torch.compile can trace it.
def _setup_forward_context(ctx, inputs, output):
    input, weights, borders, new_size, padding_mode, active_flag = inputs
    ctx.save_for_backward(input, weights, borders)
    ctx.padding_mode, ctx.active_flag = padding_mode, active_flag
    if _LAST_PLANAR[0] is not None:
        _claim_planar(input)


def _make_forward_backward(dim, suffix=''):
    def backward(ctx, grad_output):
        input, weights, borders = ctx.saved_tensors
        op = getattr(torch.ops.torchshifts, f'_shift{dim}d_backward{suffix}')
        grad_input, grad_weight = op(grad_output, weights, input, borders, ctx.padding_mode, ctx.active_flag)
        return grad_input, grad_weight, None, None, None, None
    return backward


def _setup_backward_context(ctx, inputs, output):
    pass


def _double_backward(ctx, *grads):
    raise RuntimeError('double backwards on shiftNd not supported')


# ------------------------------------------------------------------------------------------ composite
def check_borders(input, borders, dim):
    """csrc/ops/shifts.cpp:93-135: -> (int32[6] CPU tensor {l0,r0,l1,r1,l2,r2}, new_size list).

    Unlike the reference the border tensor stays on the host (the kernels take the six integers
    by value), which removes the per-call host-to-device copy of shifts.cpp:134.
    """
    user = None
    if borders is not None and borders.numel() != 0:
        user = borders.to(torch.int32).cpu().reshape(-1).tolist()
    lb, rb = _NATIVE.check_borders(dim, list(input.shape[2:2 + dim]), user)
    std = torch.tensor([lb[0], rb[0], lb[1], rb[1], lb[2], rb[2]], dtype=torch.int32)
    new_size = list(input.shape[:2]) + [rb[a] - lb[a] for a in range(dim)]
    return std, new_size


def _shift_composite(dim, input, weights, borders, padding_mode, active_flag):
    std_borders, new_size = check_borders(input, borders, dim)
    op = getattr(torch.ops.torchshifts, f'_shift{dim}d_forward')
    out = op(input, weights, std_borders, new_size, padding_mode, active_flag)
    if not torch.compiler.is_compiling():
        _LAST_PLANAR[0] = None      # a planar copy nobody claimed (no autograd): drop it now
    return out


def _bind(fn, dim):
    def bound(*args):
        return fn(dim, *args)
    bound.__name__ = f'{fn.__name__}_{dim}d'
    return bound


def register(native):
    """Define and implement the operators (idempotent)."""
    global _LIB, _NATIVE
    _NATIVE = native
    if _LIB is not None:
        return
    lib = torch.library.Library('torchshifts', 'DEF')
    lib.define('_cuda_version() -> int')
    lib.impl('_cuda_version', lambda: int(native.lib.ts_cuda_version()), 'CompositeExplicitAutograd')
    for dim in (1, 2, 3):
        lib.define(f'shift{dim}d(Tensor input, Tensor weights, Tensor borders, int padding_mode, bool active_flag) -> Tensor')
        lib.define(f'_shift{dim}d_forward(Tensor input, Tensor weights, Tensor borders, int[] new_size, '
                   f'int padding_mode, bool active_flag) -> Tensor')
        lib.define(f'_shift{dim}d_backward(Tensor grad, Tensor weights, Tensor input, Tensor borders, '
                   f'int padding_mode, bool active_flag) -> (Tensor, Tensor)')
        lib.impl(f'shift{dim}d', _bind(_shift_composite, dim), 'CompositeImplicitAutograd')
        fwd, bwd = f'_shift{dim}d_forward', f'_shift{dim}d_backward'
        lib.impl(fwd, _bind(_forward_cuda, dim), 'CUDA')
        lib.impl(bwd, _bind(_backward_cuda, dim), 'CUDA')
        lib.impl(fwd, _bind(_forward_qcuda, dim), 'QuantizedCUDA')
        lib.impl(bwd, _bind(_backward_quantized, dim), 'QuantizedCUDA')
        # fake (meta) implementations: `borders` is a host tensor next to device tensors, so the output
        # device is stated here instead of being inferred from the arguments
        torch.library.register_fake(f'torchshifts::{fwd}', _bind(_forward_meta, dim), lib=lib)
        torch.library.register_fake(f'torchshifts::{bwd}', _bind(_backward_meta, dim), lib=lib)
        torch.library.register_autograd(f'torchshifts::{fwd}', _make_forward_backward(dim), setup_context=_setup_forward_context, lib=lib)
        torch.library.register_autograd(f'torchshifts::{bwd}', _double_backward, setup_context=_setup_backward_context, lib=lib)
        for key in ('CPU', 'QuantizedCPU'):
            lib.impl(fwd, _no_cpu, key)
            lib.impl(bwd, _no_cpu, key)
    for dim in (2, 3):
        fwd, bwd = f'_shift{dim}d_forward_cl', f'_shift{dim}d_backward_cl'
        lib.define(f'{fwd}(Tensor input, Tensor weights, Tensor borders, int[] new_size, int padding_mode, bool active_flag) -> Tensor')
        lib.define(f'{bwd}(Tensor grad, Tensor weights, Tensor input, Tensor borders, int padding_mode, bool active_flag) -> (Tensor, Tensor)')
        lib.impl(fwd, _bind(_forward_cl_cuda, dim), 'CUDA')
        lib.impl(bwd, _bind(_backward_cl_cuda, dim), 'CUDA')
        lib.impl(fwd, _no_cpu, 'CPU')
        lib.impl(bwd, _no_cpu, 'CPU')
        torch.library.register_fake(f'torchshifts::{fwd}', _bind(_forward_cl_meta, dim), lib=lib)
        torch.library.register_fake(f'torchshifts::{bwd}', _bind(_backward_cl_meta, dim), lib=lib)
        torch.library.register_autograd(f'torchshifts::{fwd}', _make_forward_backward(dim, '_cl'), setup_context=_setup_forward_context, lib=lib)
        torch.library.register_autograd(f'torchshifts::{bwd}', _double_backward, setup_context=_setup_backward_context, lib=lib)
    # fused epilogue of the strided depth-wise-conv emulation (modules/shifts.py:85-89): shift + crop + avg_pool2d(2, 2, ceil)
    pool = '_shift2d_avgpool2_forward'
    lib.define(f'{pool}(Tensor input, Tensor weights, Tensor borders, int[] new_size, int padding_mode, bool active_flag) -> Tensor')
    lib.impl(pool, _pool_forward_cuda, 'CUDA')
    lib.impl(pool, _no_cpu, 'CPU')
    torch.library.register_fake(f'torchshifts::{pool}', _pool_forward_meta, lib=lib)
    torch.library.register_autograd(f'torchshifts::{pool}', _pool_backward, setup_context=_pool_setup_context, lib=lib)
    poolb = '_shift2d_avgpool2_backward'
    lib.define(f'{poolb}(Tensor grad, Tensor weights, Tensor input, Tensor borders, int[] new_size, int padding_mode, '
               f'bool active_flag) -> (Tensor, Tensor)')
    lib.impl(poolb, _pool_backward_cuda, 'CUDA')
    lib.impl(poolb, _no_cpu, 'CPU')
    torch.library.register_fake(f'torchshifts::{poolb}', _pool_backward_meta, lib=lib)
    torch.library.register_autograd(f'torchshifts::{poolb}', _double_backward, setup_context=_setup_backward_context, lib=lib)
    _LIB = lib
