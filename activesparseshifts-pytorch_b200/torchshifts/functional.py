"""Functional interface: ``shift{1,2,3}d_func`` -- same names, argument order, argument checks and
error behaviour as the reference's ``torchshifts/functional.py:7-99`` (bare ``assert`` with the
reference's messages, ``borders=None`` becomes an empty tensor, then the registered operator
``torch.ops.torchshifts.shift{1,2,3}d`` is called).  The compute behind the operator is the
sm_100a library; tensors must live on a CUDA device.
"""
from typing import Optional

import torch

from ._ops import CL_FORMATS, drop_unclaimed_planar
from .extension import _assert_has_ops

Tensor = torch.Tensor
_AXES = {1: 'H', 2: 'H and W', 3: 'H,W and D'}
_MODES = '0 - zeros, 1 - border, 2 - periodic, 3 - reflect, 4 - symmetric'


def _resolve_borders(dim, sizes, cuts):
    """Pure-Python twin of ``ts_check_borders`` (csrc/ops/shifts.cpp:111-127): ``cuts`` = ``dim`` pairs
    (left_cut, right_cut) -> (lb, rb) lists of 3.  Used only while ``torch.compile`` traces a layer that crops
    its output: there the border tensor is a traced (fake) tensor whose values cannot be read, while the
    module's cached Python integers can (tests pin this function against the C one)."""
    lb, rb = [0, 0, 0], [int(sizes[a]) if a < dim else 1 for a in range(3)]
    for a in range(dim):
        size = int(sizes[a])
        r, l = size - int(cuts[a][1]), int(cuts[a][0])
        if r - l < 1:
            r = l + 1
        if l == size:
            l, r = size - 1, size
        if r == 0:
            l, r = 0, 1
        l = max(l, 0)
        r = min(r, size)
        if r - l < 0:
            raise RuntimeError('torchshifts-b200: borders give a negative output dimension '
                               '(the reference fails here with "Trying to create tensor with negative dimension")')
        lb[a], rb[a] = l, r
    return lb, rb


@torch.compiler.assume_constant_result
def _std_borders(vals):
    """int32[6] host tensor {l0,r0,l1,r1,l2,r2}; a constant of the compiled graph (no CPU code is generated for it)"""
    return torch.tensor(list(vals), dtype=torch.int32)


def _crop(dim: int, input: Tensor, borders: Optional[Tensor], border_ints):
    """-> (std_borders, new_size) of the crop given by ``border_ints`` (the module's cached Python integers), else by
    ``borders``' values; no crop when ``borders`` is None."""
    if borders is None:
        cuts = [[0, 0]] * dim
    else:
        cuts = border_ints if border_ints is not None else [[int(v) for v in row] for row in borders.tolist()]
    lb, rb = _resolve_borders(dim, input.shape[2:], cuts)
    return _std_borders((lb[0], rb[0], lb[1], rb[1], lb[2], rb[2])), list(input.shape[:2]) + [rb[a] - lb[a] for a in range(dim)]


def _check_memory_format(memory_format) -> bool:
    """-> True for ``torch.preserve_format``, False for ``torch.contiguous_format``; anything else raises."""
    if memory_format is torch.contiguous_format:
        return False
    if memory_format is torch.preserve_format:
        return True
    raise ValueError(f'memory_format must be torch.contiguous_format or torch.preserve_format, got {memory_format!r}')


def _keeps_channels_last(dim: int, input: Tensor) -> bool:
    """Dense channels-last (not also NCHW-contiguous) float input of a 2-D / 3-D shift."""
    fmt = CL_FORMATS.get(dim)
    return (fmt is not None and not input.is_quantized and input.is_contiguous(memory_format=fmt)
            and not input.is_contiguous())


def _shift_cl(dim: int, input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool,
              borders: Optional[Tensor], _border_ints) -> Tensor:
    """The channels-last operator ``_shift{dim}d_forward_cl``: output (and grad_input) dense channels-last."""
    std, new_size = _crop(dim, input, borders, _border_ints)
    out = getattr(torch.ops.torchshifts, f'_shift{dim}d_forward_cl')(input, weights, std, new_size, padding_mode, active_flag)
    drop_unclaimed_planar()
    return out


def _shift_func(dim: int, input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool,
                borders: Optional[Tensor], _border_ints=None, memory_format=torch.contiguous_format) -> Tensor:
    name = f'shift{dim}d_func()'
    _assert_has_ops()
    preserve = _check_memory_format(memory_format)
    assert padding_mode in [0, 1, 2, 3, 4], f'{name} expected padding_mode can be {_MODES}'
    assert len(input.shape) == dim + 2, f'{name[:-2]}(): expected {dim + 2}D tensor as input, but it is shape is {input.shape}'
    assert weights.shape[-1] == dim, f'{name[:-2]}(): expected [n_channels,{dim}] tensor as weight, but it is shape is {weights.shape}'
    assert input.shape[1] == weights.shape[0], (f'{name[:-2]}(): expected that input and weight have equal number of channels, '
                                                f'but input have {input.shape[1]} and weight have {weights.shape[0]} channels.')
    assert input.device == weights.device, (f'{name[:-2]}(): expected input and weights to be on same device, '
                                            f'but input is  on {input.device} and weights is on {weights.device}')
    if borders is not None:
        assert (len(borders.shape) == 2) and (borders.shape[1] == 2) and (borders.shape[0] == dim), f'borders must have shape [{dim}, 2]'
    if preserve and _keeps_channels_last(dim, input):
        return _shift_cl(dim, input, weights, padding_mode, active_flag, borders, _border_ints)
    if borders is not None:
        if _border_ints is not None and torch.compiler.is_compiling():
            # torch.compile: resolve the crop from Python integers (constants of the trace) and call the inner
            # operator, which has a fake kernel and a registered autograd formula
            std, new_size = _crop(dim, input, borders, _border_ints)
            return getattr(torch.ops.torchshifts, f'_shift{dim}d_forward')(input, weights, std, new_size, padding_mode, active_flag)
    else:
        borders = torch.Tensor()
    op = getattr(torch.ops.torchshifts, f'shift{dim}d')
    return op(input, weights, borders, padding_mode, active_flag)


def shift1d_func(input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool,
                 borders: Optional[Tensor] = None, _border_ints=None, *, memory_format=torch.contiguous_format) -> Tensor:
    """Shift every channel of ``input [N, C, H]`` along H by its own learnable amount.

    ``weights [C, 1]`` holds sign and magnitude of the per-channel shift; ``padding_mode`` selects
    what is read outside the tensor (0 zeros, 1 border, 2 periodic, 3 reflect, 4 symmetric);
    ``active_flag`` switches from the rounded (sparse) shift to linear interpolation (ignored for
    quantized inputs); ``borders [1, 2]`` = (left_cut, right_cut) crops the output.
    ``memory_format`` (keyword only) is accepted for symmetry with the 2-D / 3-D layers and ignored: 3-D
    tensors have no channels-last format.

    Mixed precision: an fp16 / bf16 ``input`` may come with fp32 ``weights`` (an extension over the reference, which
    raises).  The output and ``grad_input`` keep ``input``'s dtype, ``grad_weight`` is fp32, and the shifts are taken from
    the fp32 weights without rounding them to 16 bits.  No autocast rule is registered: under ``torch.autocast`` the shift
    takes the activation dtype it receives and never casts the weights.
    """
    return _shift_func(1, input, weights, padding_mode, active_flag, borders, _border_ints, memory_format)


def shift2d_func(input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool,
                 borders: Optional[Tensor] = None, _border_ints=None, *, memory_format=torch.contiguous_format) -> Tensor:
    """2-D version: ``input [N, C, H, W]``, ``weights [C, 2]`` (H and W shifts), ``borders [2, 2]``;
    the active shift is bilinear.

    ``memory_format`` (keyword only): ``torch.contiguous_format`` (default) returns NCHW outputs and NCHW
    ``grad_input``, as the reference does; ``torch.preserve_format`` returns both dense ``channels_last`` when
    ``input`` is dense channels-last (and not also NCHW-contiguous), with the same values.  Other layouts give
    the default result.  This is an extension over the reference.

    Mixed precision (fp16 / bf16 ``input``, fp32 ``weights``, fp32 ``grad_weight``; no autocast cast of the weights) as
    for :func:`shift1d_func`."""
    return _shift_func(2, input, weights, padding_mode, active_flag, borders, _border_ints, memory_format)


def shift3d_func(input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool,
                 borders: Optional[Tensor] = None, _border_ints=None, *, memory_format=torch.contiguous_format) -> Tensor:
    """3-D version: ``input [N, C, H, W, D]``, ``weights [C, 3]``, ``borders [3, 2]``; the active
    shift is trilinear.  ``memory_format`` as for :func:`shift2d_func`, with ``channels_last_3d``.  Mixed precision
    (fp16 / bf16 ``input``, fp32 ``weights``, fp32 ``grad_weight``; no autocast cast of the weights) as for
    :func:`shift1d_func`."""
    return _shift_func(3, input, weights, padding_mode, active_flag, borders, _border_ints, memory_format)


def shift2d_avgpool2_func(input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool,
                          borders: Optional[Tensor] = None, _border_ints=None) -> Tensor:
    """``avg_pool2d(shift2d_func(...), kernel_size=2, stride=2, ceil_mode=True)`` in one kernel: what a ``Shift2d`` built
    with ``emulate_dw={..., 'stride': 2}`` computes (reference ``modules/shifts.py:85-89, 153``), with one read of the
    input and one quarter-size write.  Same argument checks as :func:`shift2d_func`."""
    name = 'shift2d_avgpool2_func'
    _assert_has_ops()
    assert padding_mode in [0, 1, 2, 3, 4], f'{name}() expected padding_mode can be {_MODES}'
    assert len(input.shape) == 4, f'{name}(): expected 4D tensor as input, but it is shape is {input.shape}'
    assert weights.shape[-1] == 2, f'{name}(): expected [n_channels,2] tensor as weight, but it is shape is {weights.shape}'
    assert input.shape[1] == weights.shape[0], f'{name}(): expected that input and weight have equal number of channels'
    assert input.device == weights.device, f'{name}(): expected input and weights to be on same device'
    if borders is not None:
        assert tuple(borders.shape) == (2, 2), 'borders must have shape [2, 2]'
    std, new_size = _crop(2, input, borders, _border_ints)
    out = torch.ops.torchshifts._shift2d_avgpool2_forward(input, weights, std, new_size, padding_mode, active_flag)
    drop_unclaimed_planar()
    return out


_POOL3D_STRIDES = ((1, 2, 2), (2, 2, 2))


def shift3d_avgpool_func(input: Tensor, weights: Tensor, padding_mode: int, active_flag: bool, stride,
                         borders: Optional[Tensor] = None, _border_ints=None) -> Tensor:
    """``avg_pool3d(shift3d_func(...), kernel_size=stride, stride=stride, ceil_mode=True)`` in one kernel, for ``stride``
    (1, 2, 2) -- the spatial downsampling of video networks -- or (2, 2, 2) (a scalar 2 is (2, 2, 2)): what a ``Shift3d``
    built with ``emulate_dw={..., 'stride': stride}`` computes (reference ``modules/shifts.py:85-89``), with one read of the
    input and one pooled write; the backward never materialises the full-size gradient.  Same values as the two steps (the
    forward and ``grad_input`` bit for bit).  Same argument checks as :func:`shift3d_func`; any other stride raises
    ``ValueError``.  fp32 CUDA tensors run the fused kernels, others the two steps inside the same operator."""
    name = 'shift3d_avgpool_func'
    _assert_has_ops()
    st = tuple(int(v) for v in stride) if isinstance(stride, (tuple, list, torch.Size)) else (int(stride),) * 3
    if st not in _POOL3D_STRIDES:
        raise ValueError(f'{name}(): stride must be (1, 2, 2) or (2, 2, 2), got {stride!r}')
    assert padding_mode in [0, 1, 2, 3, 4], f'{name}() expected padding_mode can be {_MODES}'
    assert len(input.shape) == 5, f'{name}(): expected 5D tensor as input, but it is shape is {input.shape}'
    assert weights.shape[-1] == 3, f'{name}(): expected [n_channels,3] tensor as weight, but it is shape is {weights.shape}'
    assert input.shape[1] == weights.shape[0], (f'{name}(): expected that input and weight have equal number of channels, '
                                                f'but input have {input.shape[1]} and weight have {weights.shape[0]} channels.')
    assert input.device == weights.device, (f'{name}(): expected input and weights to be on same device, '
                                            f'but input is  on {input.device} and weights is on {weights.device}')
    if borders is not None:
        assert tuple(borders.shape) == (3, 2), 'borders must have shape [3, 2]'
    std, new_size = _crop(3, input, borders, _border_ints)
    out = torch.ops.torchshifts._shift3d_avgpool_forward(input, weights, std, new_size, list(st), padding_mode, active_flag)
    drop_unclaimed_planar()
    return out


# BASELINE.json names these "functional.shift1d/2d/3d"; keep the real names and add the aliases.
shift1d, shift2d, shift3d = shift1d_func, shift2d_func, shift3d_func
