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

Mixed precision (an extension over the reference, whose type check raises): an fp16 / bf16 ``input`` (and ``grad``) may
come with fp32 ``weights``.  The output and ``grad_input`` keep the input's dtype, ``grad_weight`` is fp32 like the
weights, and the weights are split in fp32 -- never rounded to 16 bits.  No autocast kernel is registered: under
``torch.autocast`` the operators take the activation dtype they receive and never cast the weights.

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

from ._cabi import (QW_I8, QW_I32, QW_U8, TS_ERR_TOO_LARGE, TS_ERR_UNSUPPORTED, TS_ERR_WORKSPACE, TS_OK, TS_WEIGHTS_F32,
                    make_geometry)

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


_HALF = (torch.float16, torch.bfloat16)


def _mixed(input, weights):
    """fp16 / bf16 activations with fp32 (master) weights."""
    return input.dtype in _HALF and weights.dtype == torch.float32


def _same_device_and_type(fn, input, weights, grad=None):
    # checkAllSameGPU / checkAllSameType of cuda/shifts_cuda.cu:213-214, :282-283; in addition fp16 / bf16 input and grad
    # may come with fp32 weights (mixed precision)
    if weights.device != input.device or (grad is not None and grad.device != input.device):
        raise RuntimeError(f'{fn}: expected input, weights' + (', grad' if grad is not None else '') +
                           f' to be on the same GPU, but got {input.device}, {weights.device}' +
                           (f', {grad.device}' if grad is not None else ''))
    if (weights.dtype != input.dtype and not _mixed(input, weights)) or (grad is not None and grad.dtype != input.dtype):
        raise RuntimeError(f'{fn}: expected scalar type {input.dtype} for every tensor but found '
                           f'weights {weights.dtype}' + (f', grad {grad.dtype}' if grad is not None else ''))
    if input.dtype not in _DTYPES:
        raise RuntimeError(f'{fn}: "shiftnd_cuda" not implemented for {input.dtype}')


def _dtype_code(input, weights):
    """The C ABI's dtype argument: the element type, with TS_WEIGHTS_F32 for fp32 weights of a 16-bit input."""
    return _DTYPES[input.dtype] | (TS_WEIGHTS_F32 if _mixed(input, weights) else 0)


_COPY_THRESHOLD = 1 << 16
CL_FORMATS = {2: torch.channels_last, 3: torch.channels_last_3d}    # number of spatial dims -> channels-last format
_FALLBACK = (TS_ERR_UNSUPPORTED,)


def _served(status, what, fallback=()):
    """Reads a library status: True for TS_OK, False for a status in ``fallback`` (the kernel does not serve the call and
    nothing was launched: the caller runs its fallback path); any other status raises."""
    if status == TS_OK:
        return True
    if status in fallback:
        return False
    _NATIVE.check(status, what)


_PLANAR = collections.OrderedDict()     # (data_ptr, shape, strides, version) -> planar copy made by the forward, for the backward
_PLANAR_MAX = 2
_LAST_PLANAR = [None]                   # (key, copy) of the forward that just ran, until autograd claims it (or the composite returns)


def _dense(input, keep=False, take=False):
    """Channels-last / sliced inputs: the stride-aware generic kernels read them in place, but their
    per-element strided loads waste most of every 32-byte sector.  Above a few tens of thousands of
    elements one extra coalesced pass plus the bandwidth kernels is several times faster: a dense
    channels-last tensor goes through the library's own tiled transpose (``ts_nhwc_to_nchw``), anything
    else through ``.contiguous()``.

    ``keep`` (forward): park the planar copy in ``_LAST_PLANAR``; when autograd records the call, the forward's
    ``setup_context`` -- the one place that knows the call is differentiated: the CUDA kernel runs below the Autograd key,
    with grad mode off -- moves it to ``_PLANAR``, otherwise ``drop_unclaimed_planar`` drops it when the operator returns.
    ``take`` (backward): reuse that copy instead of converting the saved input a second time (0.26 ms per step for cfg3)
    -- at most ``_PLANAR_MAX`` copies are held."""
    if input.numel() < _COPY_THRESHOLD or input.is_contiguous():
        return input
    key = _planar_key(input)
    if take:
        hit = _PLANAR.pop(key, None)
        if hit is not None:
            return hit
    fmt = CL_FORMATS.get(input.dim() - 2)
    if fmt is not None and input.is_contiguous(memory_format=fmt) and input.element_size() in (2, 4, 8):
        out = torch.empty(input.shape, dtype=input.dtype, device=input.device)
        n, c = input.shape[0], input.shape[1]
        with _guard(input.device):
            st = _NATIVE.lib.ts_nhwc_to_nchw(input.data_ptr(), out.data_ptr(), n, c, input.numel() // max(n * c, 1),
                                             input.element_size(), _stream(input.device))
        _served(st, 'ts_nhwc_to_nchw')
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


def drop_unclaimed_planar():
    """Called when a shift operator returns to its caller: a planar copy no autograd record claimed is not needed."""
    if not torch.compiler.is_compiling():
        _LAST_PLANAR[0] = None


def _stream(device):
    return ct.c_void_p(torch._C._cuda_getCurrentRawStream(device.index))


_NO_GUARD = contextlib.nullcontext()


def _guard(device):
    """CUDAGuard of cuda/shifts_cuda.cu:215, :284 -- skipped (it costs ~10 us in Python) when the tensor's device
    already is the current one."""
    return _NO_GUARD if device.index == torch._C._cuda_getDevice() else torch.cuda.device(device)


_GEO_CACHE = {}        # (dim, shape, strides, lb, rb) -> ts_geometry; shift layers see the same few shapes every step
_WS_CACHE = {}         # (workspace query's name, geometry key, dtype code with its flags, device index) -> backward workspace bytes


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


def _check_size(fn, name, size, dim, input, lb, rb):
    """``size`` (a forward's ``new_size``, a backward's ``grad`` shape) must be input's N, C and the cropped extent."""
    if list(size) != list(input.shape[:2]) + [rb[a] - lb[a] for a in range(dim)]:
        raise RuntimeError(f'{fn}: {name} {list(size)} does not match the borders and input {list(input.shape)}')


def _launch_backward(entry, query, geo, key, grad, input, weights, padding_mode, active_flag, peers=(),
                     fmt=torch.contiguous_format, fallback=(), lead=()):
    """Runs the backward entry point ``entry`` -> (grad_input in ``fmt``, grad_weight).  ``query`` is its workspace-size
    function, cached per geometry; ``peers``: the trailing peer-group argument of the entry points that take one;
    ``lead``: arguments between ``active`` and ``grad`` (the pooling stride of the fused avg-pool backward).

    With a ``fallback`` (statuses as for ``_served``) returns None when the kernel does not serve the call: the launch
    returned such a status, or ``query`` answered 16 bytes (no partials), which is decided before ``grad`` is converted
    to ``fmt`` -- a conversion the caller's fallback path would do again."""
    code = _dtype_code(input, weights)
    dev = input.device
    wkey = (query.__name__, key, code, dev.index)
    with _guard(dev):
        for attempt in (0, 1):
            nbytes = _WS_CACHE.get(wkey)
            if nbytes is None:
                if len(_WS_CACHE) > 256:
                    _WS_CACHE.clear()
                nbytes = _WS_CACHE[wkey] = int(query(ct.byref(geo), code))
            if fallback and nbytes <= 16:
                return None
            grad = grad.contiguous(memory_format=fmt)
            w = weights.contiguous()
            grad_input = torch.empty(input.shape, dtype=input.dtype, device=dev, memory_format=fmt)
            grad_weight = torch.empty(w.shape, dtype=w.dtype, device=dev)
            workspace = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=dev)
            st = entry(ct.byref(geo), code, int(padding_mode), int(bool(active_flag)), *lead, grad.data_ptr(), input.data_ptr(),
                       w.data_ptr(), grad_input.data_ptr(), grad_weight.data_ptr(), workspace.data_ptr(), nbytes, *peers,
                       _stream(dev))
            if st != TS_ERR_WORKSPACE:      # (nothing was launched): the tuning knobs changed since the size was cached
                break
            _WS_CACHE.clear()
    return (grad_input, grad_weight) if _served(st, entry.__name__, fallback) else None


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
    _check_size(fn, 'new_size', new_size, dim, input, lb, rb)
    with _guard(input.device):
        st = _NATIVE.lib.ts_shift_forward(ct.byref(geo), _dtype_code(input, w), int(padding_mode), int(bool(active_flag)),
                                          input.data_ptr(), w.data_ptr(), out.data_ptr(), _stream(input.device))
    _served(st, 'ts_shift_forward')
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
        if _served(st, 'ts_shift2d_avgpool2_forward', _FALLBACK):
            return out
    y = _forward_cuda(2, input, weights, borders, new_size, padding_mode, active_flag)
    return torch.nn.functional.avg_pool2d(y, kernel_size=2, stride=2, ceil_mode=True)


def _pool_forward_meta(input, weights, borders, new_size, padding_mode, active_flag):
    return input.new_empty([new_size[0], new_size[1], (new_size[2] + 1) // 2, (new_size[3] + 1) // 2])


def _strides(values):
    return (ct.c_int32 * len(values))(*[int(v) for v in values])


def _pool_backward_fused(fn, dim, stride, grad_pooled, weights, input, lb, rb, padding_mode, active_flag):
    """The fused avg-pool backward (ts_shift_avgpool_backward) -> (grad_input, grad_weight), or None where the kernels do not
    serve the call.  Under FusedGradWeightAllReduce grad_weight is summed over the ranks in the same launch; a rank whose call
    is not served takes the caller's two-step path, whose shift backward exchanges too."""
    geo, key = _geometry(dim, input, lb, rb)
    lib, fused = _NATIVE.lib, _FUSED_ALLREDUCE
    peers = (ct.byref(fused.peer_group()) if fused is not None else None,)
    return _launch_backward(lib.ts_shift_avgpool_backward, lib.ts_shift_avgpool_backward_workspace_bytes, geo, key, grad_pooled,
                            input, weights, padding_mode, active_flag, peers, fallback=_FALLBACK, lead=(_strides(stride),))


def _pool_backward_cuda(grad_pooled, weights, input, borders, new_size, padding_mode, active_flag):
    """Backward of the fused shift + avg_pool2d(2, 2, ceil_mode): ONE kernel (ts_shift_avgpool_backward) that expands the
    pooled gradient while staging it -- the full-size gradient of the shift's output never exists in HBM.  Shapes the fused
    kernel does not serve take ATen's avg_pool2d_backward followed by the shift backward (same values)."""
    fn = 'shift2d_avgpool2_backward'
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights, grad_pooled)
    if _FUSED_ALLREDUCE is not None:
        _check_fused(fn, _FUSED_ALLREDUCE, input.device, _DTYPES[input.dtype], weights.numel())
    lb, rb = _borders_lists(borders, 2)
    oh, ow = rb[0] - lb[0], rb[1] - lb[1]
    if list(grad_pooled.shape) != [input.shape[0], input.shape[1], (oh + 1) // 2, (ow + 1) // 2]:
        raise RuntimeError(f'{fn}: grad has shape {list(grad_pooled.shape)}, the pooled output is '
                           f'{[input.shape[0], input.shape[1], (oh + 1) // 2, (ow + 1) // 2]}')
    if input.dtype == torch.float32 and input.is_contiguous() and ow % 8 == 0 and input.dim() == 4 and input.numel() > 0:
        grads = _pool_backward_fused(fn, 2, (2, 2), grad_pooled, weights, input, lb, rb, padding_mode, active_flag)
        if grads is not None:
            return grads
    like = torch.empty(list(new_size), dtype=grad_pooled.dtype, device=grad_pooled.device)
    grad_y = torch.ops.aten.avg_pool2d_backward(grad_pooled.contiguous(), like, [2, 2], [2, 2], [0, 0], True, True, None)
    return _backward_cuda(2, grad_y, weights, input, borders, padding_mode, active_flag)


def _pool_backward_meta(grad_pooled, weights, input, borders, new_size, padding_mode, active_flag):
    return input.new_empty(input.shape), weights.new_empty(weights.shape)


def _pooled_size(new_size, stride):
    return list(new_size[:2]) + [-(-int(o) // int(s)) for o, s in zip(new_size[2:], stride)]


def _pool3d_forward_cuda(input, weights, borders, new_size, stride, padding_mode, active_flag):
    """Shift3d forward + avg_pool3d(kernel = stride, ceil_mode=True) for the strides (1, 2, 2) and (2, 2, 2) in ONE kernel
    (ts_shift_avgpool_forward): one read of x, one pooled write.  Shapes the fused kernel does not serve (non-fp32, rows that
    are not a multiple of 4 elements, strided inputs, slabs too large to stage) run the two steps separately -- same values."""
    fn = 'shift3d_avgpool_forward'
    _check_forward(fn, 3, input, weights, padding_mode)
    lb, rb = _borders_lists(borders, 3)
    _check_size(fn, 'new_size', new_size, 3, input, lb, rb)
    if input.dtype == torch.float32 and weights.dtype == torch.float32 and input.is_contiguous():
        out = torch.empty(_pooled_size(new_size, stride), dtype=input.dtype, device=input.device)
        w = weights.contiguous()
        geo, _ = _geometry(3, input, lb, rb)
        with _guard(input.device):
            st = _NATIVE.lib.ts_shift_avgpool_forward(ct.byref(geo), 0, int(padding_mode), int(bool(active_flag)), _strides(stride),
                                                      input.data_ptr(), w.data_ptr(), out.data_ptr(), _stream(input.device))
        if _served(st, 'ts_shift_avgpool_forward', _FALLBACK):
            return out
    y = _forward_cuda(3, input, weights, borders, new_size, padding_mode, active_flag)
    return torch.nn.functional.avg_pool3d(y, kernel_size=list(stride), stride=list(stride), ceil_mode=True)


def _pool3d_forward_meta(input, weights, borders, new_size, stride, padding_mode, active_flag):
    return input.new_empty(_pooled_size(new_size, stride))


def _pool3d_backward_cuda(grad_pooled, weights, input, borders, new_size, stride, padding_mode, active_flag):
    """Backward of ``_shift3d_avgpool_forward``: ONE kernel (ts_shift_avgpool_backward) applies the pooling adjoint while the
    pooled gradient is staged, plus the pass-2 reduction.  What the kernel does not serve (and empty shards) takes ATen's
    avg_pool3d_backward followed by the shift backward -- same values, and the same grad_weight exchange."""
    fn = 'shift3d_avgpool_backward'
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights, grad_pooled)
    if _FUSED_ALLREDUCE is not None:
        _check_fused(fn, _FUSED_ALLREDUCE, input.device, _DTYPES[input.dtype], weights.numel())
    lb, rb = _borders_lists(borders, 3)
    _check_size(fn, 'new_size', new_size, 3, input, lb, rb)
    if list(grad_pooled.shape) != _pooled_size(new_size, stride):
        raise RuntimeError(f'{fn}: grad has shape {list(grad_pooled.shape)}, the pooled output is {_pooled_size(new_size, stride)}')
    if (input.dtype == torch.float32 and weights.dtype == torch.float32 and input.is_contiguous() and new_size[4] % 8 == 0
            and input.numel() > 0):
        grads = _pool_backward_fused(fn, 3, stride, grad_pooled, weights, input, lb, rb, padding_mode, active_flag)
        if grads is not None:
            return grads
    if grad_pooled.numel() == 0:
        grad_y = grad_pooled.new_zeros(list(new_size))
    else:
        like = torch.empty(list(new_size), dtype=grad_pooled.dtype, device=grad_pooled.device)
        grad_y = torch.ops.aten.avg_pool3d_backward(grad_pooled.contiguous(), like, list(stride), list(stride), [0, 0, 0], True, True,
                                                    None)
    return _backward_cuda(3, grad_y, weights, input, borders, padding_mode, active_flag)


def _pool3d_backward_meta(grad_pooled, weights, input, borders, new_size, stride, padding_mode, active_flag):
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
    input = _dense(input, take=True)
    geo, key = _geometry(dim, input, lb, rb)
    _check_size(fn, 'grad shape', grad.shape, dim, input, lb, rb)
    lib, fused = _NATIVE.lib, _FUSED_ALLREDUCE
    if fused is None:
        return _launch_backward(lib.ts_shift_backward, lib.ts_shift_backward_workspace_bytes, geo, key, grad, input, weights,
                                padding_mode, active_flag)
    _check_fused(fn, fused, input.device, _DTYPES[input.dtype], weights.numel())
    return _launch_backward(lib.ts_shift_backward_allreduce, lib.ts_shift_backward_workspace_bytes, geo, key, grad, input, weights,
                            padding_mode, active_flag, (ct.byref(fused.peer_group()),))


# ------------------------------------------------------------------------------------------ CUDA, channels-last
def _forward_cl_cuda(dim, input, weights, borders, new_size, padding_mode, active_flag):
    """``_shiftNd_forward`` with a dense channels-last output.  2-D dense channels-last fp32 / fp16 / bf16 inputs run the
    native NHWC kernel (ts_shift_forward_nhwc: one read, one write, no layout pass); whatever it does not serve takes the
    planar forward and converts its output -- the same values."""
    fn = f'shift{dim}d_forward_cl'
    fmt = CL_FORMATS[dim]
    _check_forward(fn, dim, input, weights, padding_mode)
    if dim == 2 and input.dtype != torch.float64 and input.shape[1] % 32 == 0 and input.is_contiguous(memory_format=fmt):
        lb, rb = _borders_lists(borders, dim)
        _check_size(fn, 'new_size', new_size, dim, input, lb, rb)
        out = torch.empty(list(new_size), dtype=input.dtype, device=input.device, memory_format=fmt)
        w = weights.contiguous()
        geo, _ = _geometry(dim, input, lb, rb)
        with _guard(input.device):
            st = _NATIVE.lib.ts_shift_forward_nhwc(ct.byref(geo), _dtype_code(input, w), int(padding_mode), int(bool(active_flag)),
                                                   input.data_ptr(), w.data_ptr(), out.data_ptr(), _stream(input.device))
        if _served(st, 'ts_shift_forward_nhwc', _FALLBACK):
            return out
    return _forward_cuda(dim, input, weights, borders, new_size, padding_mode, active_flag).contiguous(memory_format=fmt)


def _backward_cl_cuda(dim, grad, weights, input, borders, padding_mode, active_flag):
    """``_shiftNd_backward`` with a dense channels-last ``grad_input``.  ``grad`` may arrive in any layout (an expanded
    tensor from ``.sum()``, say): the native kernel (ts_shift_backward_nhwc) reads it dense channels-last.  What the
    kernel does not serve takes the planar backward and converts ``grad_input`` -- the same values."""
    fn = f'shift{dim}d_backward_cl'
    fmt = CL_FORMATS[dim]
    _check_mode(padding_mode)
    _same_device_and_type(fn, input, weights, grad)
    fused = _FUSED_ALLREDUCE
    if fused is not None:
        _check_fused(fn, fused, input.device, _DTYPES[input.dtype], weights.numel())
    if dim == 2 and input.dtype != torch.float64 and input.dim() == 4 and input.shape[1] % 32 == 0 \
            and input.is_contiguous(memory_format=fmt):
        lb, rb = _borders_lists(borders, dim)
        _check_size(fn, 'grad shape', grad.shape, dim, input, lb, rb)
        geo, key = _geometry(dim, input, lb, rb)
        lib = _NATIVE.lib
        grads = _launch_backward(lib.ts_shift_backward_nhwc, lib.ts_shift_backward_nhwc_workspace_bytes, geo, key, grad, input,
                                 weights, padding_mode, active_flag, (ct.byref(fused.peer_group()) if fused is not None else None,),
                                 fmt, _FALLBACK)
        if grads is not None:
            return grads
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
    _check_size(fn, 'new_size', new_size, dim, input, lb, rb)
    wq = _raw_qweights(weights, input.device)
    args = (_QBYTES[input.dtype], int(padding_mode), int(input.q_zero_point()))
    wargs = (wq.data_ptr(), _QKINDS[weights.dtype], int(weights.q_zero_point()))
    # the reference allocates the quantized output in the input's memory format
    # (quantized/shifts_quantized.cpp:119-122): channels-last in, channels-last out -- served by the
    # native NHWC kernel (one read + one write, no layout conversion on either side)
    fmt = CL_FORMATS.get(dim)
    if fmt is not None and not input.is_contiguous() and input.is_contiguous(memory_format=fmt):
        to_cl = (0,) + tuple(range(2, dim + 2)) + (1,)
        to_nc = (0, dim + 1) + tuple(range(1, dim + 1))
        out_cl = torch._empty_affine_quantized([new_size[i] for i in to_cl], scale=input.q_scale(),
                                               zero_point=input.q_zero_point(), dtype=input.dtype, device=input.device)
        geo, _ = _geometry(dim, input, lb, rb)
        with _guard(input.device):
            st = _NATIVE.lib.ts_qshift_forward_nhwc(ct.byref(geo), *args, input.data_ptr(), *wargs, out_cl.data_ptr(),
                                                    _stream(input.device))
        # TS_ERR_TOO_LARGE: row offsets beyond 32 bits; both take the planar kernels and conversions
        if _served(st, 'ts_qshift_forward_nhwc', (TS_ERR_UNSUPPORTED, TS_ERR_TOO_LARGE)):
            return out_cl.permute(*to_nc)
        del out_cl
    x = input if input.is_contiguous() else input.contiguous()
    out = torch._empty_affine_quantized(list(new_size), scale=input.q_scale(), zero_point=input.q_zero_point(),
                                        dtype=input.dtype, device=input.device)
    geo, _ = _geometry(dim, x, lb, rb)
    with _guard(input.device):
        st = _NATIVE.lib.ts_qshift_forward(ct.byref(geo), *args, x.data_ptr(), *wargs, out.data_ptr(), _stream(input.device))
    _served(st, 'ts_qshift_forward')
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
    return torch.empty(list(new_size), dtype=input.dtype, device=input.device, memory_format=CL_FORMATS[dim])


def _backward_cl_meta(dim, grad, weights, input, borders, padding_mode, active_flag):
    return (torch.empty(input.shape, dtype=input.dtype, device=input.device, memory_format=CL_FORMATS[dim]),
            weights.new_empty(weights.shape))


# ------------------------------------------------------------------------------------------ Autograd
# csrc/ops/autograd/shifts_autograd.cpp:15-47 (and the 2d/3d twins): forward saves input, weights and
# borders; backward calls _shiftNd_backward and returns grads for input and weights only; the backward
# op itself is not differentiable (:50-72).  Registered with torch.library.register_autograd (not an
# Autograd-key kernel wrapping an autograd.Function) so that AOTAutograd / torch.compile can trace it.
def _forward_autograd(backward_op, takes_new_size):
    """-> (backward, setup_context) of a forward op: save input, weights and borders (and new_size when ``backward_op``
    takes it), keep the planar copy the forward made, and call ``backward_op``."""
    def setup_context(ctx, inputs, output):
        input, weights, borders, new_size, *rest = inputs         # rest: (stride,) padding_mode, active_flag
        ctx.save_for_backward(input, weights, borders)
        ctx.tail = (list(new_size), *rest) if takes_new_size else tuple(rest)
        ctx.n_inputs = len(inputs)
        if _LAST_PLANAR[0] is not None:
            _claim_planar(input)

    def backward(ctx, grad_output):
        input, weights, borders = ctx.saved_tensors
        op = getattr(torch.ops.torchshifts, backward_op)
        grad_input, grad_weight = op(grad_output, weights, input, borders, *ctx.tail)
        return (grad_input, grad_weight) + (None,) * (ctx.n_inputs - 2)
    return backward, setup_context


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
    drop_unclaimed_planar()
    return out


def _bind(fn, dim):
    def bound(*args):
        return fn(dim, *args)
    bound.__name__ = f'{fn.__name__}_{dim}d'
    return bound


_FORWARD = '(Tensor input, Tensor weights, Tensor borders, int[] new_size, int padding_mode, bool active_flag) -> Tensor'
_BACKWARD = '(Tensor grad, Tensor weights, Tensor input, Tensor borders, int padding_mode, bool active_flag) -> (Tensor, Tensor)'
_POOL_BACKWARD = ('(Tensor grad, Tensor weights, Tensor input, Tensor borders, int[] new_size, int padding_mode, '
                  'bool active_flag) -> (Tensor, Tensor)')

_POOL3D_FORWARD = ('(Tensor input, Tensor weights, Tensor borders, int[] new_size, int[] stride, int padding_mode, '
                   'bool active_flag) -> Tensor')
_POOL3D_BACKWARD = ('(Tensor grad, Tensor weights, Tensor input, Tensor borders, int[] new_size, int[] stride, int padding_mode, '
                    'bool active_flag) -> (Tensor, Tensor)')


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
        lib.impl(f'shift{dim}d', _bind(_shift_composite, dim), 'CompositeImplicitAutograd')
    # name -> (schema, CUDA kernel, fake kernel, QuantizedCUDA kernel or None).  Fake kernels: `borders` is a host tensor
    # next to device tensors, so they state the output device instead of leaving it to be inferred from the arguments.
    ops = {}
    for dim in (1, 2, 3):
        ops[f'_shift{dim}d_forward'] = (_FORWARD, _bind(_forward_cuda, dim), _bind(_forward_meta, dim), _bind(_forward_qcuda, dim))
        ops[f'_shift{dim}d_backward'] = (_BACKWARD, _bind(_backward_cuda, dim), _bind(_backward_meta, dim),
                                         _bind(_backward_quantized, dim))
    for dim in (2, 3):
        ops[f'_shift{dim}d_forward_cl'] = (_FORWARD, _bind(_forward_cl_cuda, dim), _bind(_forward_cl_meta, dim), None)
        ops[f'_shift{dim}d_backward_cl'] = (_BACKWARD, _bind(_backward_cl_cuda, dim), _bind(_backward_cl_meta, dim), None)
    # fused epilogue of the strided depth-wise-conv emulation (modules/shifts.py:85-89): shift + crop + avg_pool2d(2, 2, ceil)
    ops['_shift2d_avgpool2_forward'] = (_FORWARD, _pool_forward_cuda, _pool_forward_meta, None)
    ops['_shift2d_avgpool2_backward'] = (_POOL_BACKWARD, _pool_backward_cuda, _pool_backward_meta, None)
    # 3-D: shift + crop + avg_pool3d(kernel = stride, ceil_mode) for the strides (1, 2, 2) and (2, 2, 2)
    ops['_shift3d_avgpool_forward'] = (_POOL3D_FORWARD, _pool3d_forward_cuda, _pool3d_forward_meta, None)
    ops['_shift3d_avgpool_backward'] = (_POOL3D_BACKWARD, _pool3d_backward_cuda, _pool3d_backward_meta, None)
    for name, (schema, cuda, fake, qcuda) in ops.items():
        lib.define(name + schema)
        lib.impl(name, cuda, 'CUDA')
        lib.impl(name, _no_cpu, 'CPU')
        if qcuda is not None:
            lib.impl(name, qcuda, 'QuantizedCUDA')
            lib.impl(name, _no_cpu, 'QuantizedCPU')
        torch.library.register_fake(f'torchshifts::{name}', fake, lib=lib)
        if '_forward' in name:
            backward_op = name.replace('_forward', '_backward')
            backward, setup_context = _forward_autograd(backward_op, 'new_size' in ops[backward_op][0])
        else:
            backward, setup_context = _double_backward, _setup_backward_context
        torch.library.register_autograd(f'torchshifts::{name}', backward, setup_context=setup_context, lib=lib)
    _LIB = lib
