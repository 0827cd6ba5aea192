"""``Shift1d / Shift2d / Shift3d``: per-channel learnable shift layers (a zero-FLOP stand-in for a
depth-wise convolution).  Python surface of the reference's ``torchshifts/modules/shifts.py``:
same constructor arguments, attributes, ``(output, loss)`` return convention, ``extra_repr`` and
the depth-wise-convolution emulation heuristics.  The compute is ``torchshifts.functional``.

Reference behaviours kept on purpose (SURVEY.md 8b), so that a model moved over from the reference
initialises and behaves identically:
  * ``init_thumb_rule=2`` does not change the initialiser (reference ``modules/shifts.py:117-118``
    compares instead of assigning);
  * ``emulate_dw['padding_mode']`` does not change the padding (``:128-129``, same reason);
  * the padding name is validated lower-cased but looked up as given (``:107-108``): ``'Zeros'`` raises KeyError;
  * ``cut_borders`` / ``init_shift`` / ``_w_post_init_scale`` are plain attributes, the only
    parameter / state_dict entry is ``weight [C, dim]``.
"""
import random
from functools import partial

import torch
from torch import nn

from torchshifts.functional import (_check_memory_format, _keeps_channels_last, shift1d_func, shift2d_avgpool2_func,
                                    shift2d_func, shift3d_avgpool_func, shift3d_func)

paddings_dict = {'zeros': 0, 'border': 1, 'periodic': 2, 'reflect': 3, 'symmetric': 4}
_SHIFT_FUNCS = {1: shift1d_func, 2: shift2d_func, 3: shift3d_func}
_POOLS = {1: torch.nn.functional.avg_pool1d, 2: torch.nn.functional.avg_pool2d, 3: torch.nn.functional.avg_pool3d}


def _wrap_dim(val, dim, name):
    """Broadcast a scalar to ``dim`` entries; truncate (with a message) a longer sequence."""
    if isinstance(val, tuple):
        val = list(val)
    if not isinstance(val, list):
        val = [val] * dim
    if len(val) != dim:
        print(f'{name} params has different kernel sizes, but length of list do not corresponds to dim: {dim}, and was reduced')
        val = val[:dim]
    return val


def _create_dw_emulation(args, dim):
    """Translate depth-wise-conv hyper-parameters into shift-layer settings.

    Returns ``(init_shift, stride_scales, borders, padding)``: the shift initialisation range
    (kernel_size, halved for thumb rule 1), the per-axis stride used to scale the initial weights
    and to average-pool the output, the output crop that reproduces the conv's output size when
    ``2*padding - kernel_size + 1 < 0``, and the conv padding mode translated to ours (-1 if absent).
    """
    assert isinstance(args, dict), f'args must be dict'
    assert 'kernel_size' in args, f'args must contains at least the kernel_size inside'
    if 'dilation' in args:
        print('Warning! Found the dilation param which is not supported and will be ignored')
    kernel_size = torch.tensor(_wrap_dim(args['kernel_size'], dim, 'kernel_size'), requires_grad=False)
    padding = torch.tensor(_wrap_dim(args.get('padding', 0), dim, 'padding'), requires_grad=False)
    stride = _wrap_dim(args.get('stride', 1), dim, 'stride')
    halve = 2 if args['init_thumb_rule_type'] == 1 else 1

    borders = None
    shrink = 2 * padding - kernel_size + 1
    cut = shrink < 0
    if cut.any():
        borders = torch.zeros(dim, 2, dtype=torch.long, requires_grad=False)
        borders[cut, 0] = abs(shrink[cut]) // 2
        borders[cut, 1] = abs(shrink[cut]) - borders[cut, 0]

    init_shift = kernel_size // halve
    scales = torch.tensor(stride, requires_grad=False).unsqueeze(0)

    conv_modes = {'zeros': 0, 'replicate': 1, 'circular': 2, 'reflect': 3}
    mode = args.get('padding_mode', -1)
    if isinstance(mode, str):
        mode = conv_modes[mode]
    return init_shift, scales, borders, mode


class _Shiftnd(nn.Module):
    """Common base of the shift layers.

    Arguments:
        in_channels (int): number of channels of the input.
        padding (str): 'zeros' (default), 'border', 'periodic', 'reflect' or 'symmetric'.
        init_shift (float or tuple): bound of the uniform weight initialisation. Default 1.
        sparsity_term (float): strength of the L1 penalty returned as ``loss``. Default 5e-4.
        active_flag (bool): interpolate in the forward pass (active shift). Default False.
        emulate_dw (dict): parameters of the depth-wise convolution being replaced
            (kernel_size, padding, stride); output shape and initialisation follow it.
        init_thumb_rule (int): 1: uniform(-init_shift, init_shift); 2: see the module docstring.
        memory_format (torch.memory_format): ``torch.contiguous_format`` (default): NCHW outputs, as the
            reference; ``torch.preserve_format``: a dense channels-last input gives a channels-last output and
            ``grad_input`` (see :func:`torchshifts.functional.shift2d_func`).  Ignored by ``Shift1d``.

    Mixed precision: ``weight`` stays an fp32 parameter while the layer takes fp16 / bf16 inputs, e.g. under
    ``torch.autocast('cuda', dtype=torch.bfloat16)``.  The output keeps the input's dtype, ``weight.grad`` is fp32, and
    the shifts come from the fp32 weights unrounded.  No autocast rule is registered and the weights are never cast; an
    extension over the reference, which raises on the dtype mismatch.
    """

    @staticmethod
    def _identity(x):
        return x

    @staticmethod
    def _pooling(ks, dim):
        if isinstance(ks, torch.Tensor):
            ks = ks.squeeze().cpu().numpy().tolist()
        return partial(_POOLS[min(dim, 3)], kernel_size=ks, stride=ks, ceil_mode=True)

    @staticmethod
    def _init_thumb_rule_1(size, shape):
        return 2 * size * torch.rand(shape) - size

    @staticmethod
    def _init_thumb_rule_2(size, shape):
        return size * torch.rand(shape) * (1 if random.random() < 0.5 else -1)

    def __init__(self, in_channels, padding='zeros', init_shift=1, sparsity_term=5e-4, active_flag=False,
                 emulate_dw=None, init_thumb_rule=1, memory_format=torch.contiguous_format):
        super(_Shiftnd, self).__init__()
        _check_memory_format(memory_format)
        self.memory_format = memory_format
        assert padding.lower() in paddings_dict.keys(), f'incorrect padding option: {padding}'
        self.padding = paddings_dict[padding]
        self.sparsity_term = sparsity_term
        self.in_channels = in_channels
        self._active_flag = active_flag
        self._shift_func = self._init_shift_fn()
        self.cut_borders = None
        self._reduction_fn = self._identity
        self._w_init_func = self._init_thumb_rule_1        # rule 2 is inert in the reference; kept so
        self.init_shift = torch.tensor(_wrap_dim(init_shift, self.dim, 'init_shift'), requires_grad=False)
        self._w_post_init_scale = torch.ones(1, self.dim, requires_grad=False)

        if emulate_dw is not None:
            emulate_dw['init_thumb_rule_type'] = init_thumb_rule
            self.init_shift, self._w_post_init_scale, self.cut_borders, _ = _create_dw_emulation(emulate_dw, self.dim)
            if not (self._w_post_init_scale == 1).all():
                self._reduction_fn = self._pooling(self._w_post_init_scale, self.dim)
        self._cut_cache = None
        self._border_ints()
        self._stride_ints = [int(v) for v in self._w_post_init_scale.reshape(-1).tolist()]
        self._init_weights()

    def _init_shift_fn(self):
        return _SHIFT_FUNCS[self.dim]

    def _init_weights(self):
        self.weight = nn.Parameter(torch.Tensor(self.in_channels, self.dim))
        self.reset_parameters()

    def reset_parameters(self):
        for i in range(self.dim):
            self.weight.data[:, i] = self._w_init_func(self.init_shift[i], self.in_channels)
        self.weight.data *= self._w_post_init_scale

    def _compute_weight_loss(self):
        return self.sparsity_term * torch.sum(torch.abs(self.weight))

    def _border_ints(self):
        """``cut_borders`` as Python integers, read once per distinct tensor (and never while torch.compile traces,
        where the tensor's values are not available)."""
        cb = self.cut_borders
        if cb is None:
            return None
        cached = getattr(self, '_cut_cache', None)
        if cached is None or cached[0] is not cb:
            if torch.compiler.is_compiling():
                return cached[1] if cached is not None else None
            cached = self._cut_cache = (cb, [[int(v) for v in row] for row in cb.tolist()])
        return cached[1]

    def _pool_is_fused(self, input):
        """The average pooling of a depth-wise-conv emulation with stride (2, 2), or (1, 2, 2) / (2, 2, 2) in 3-D, runs inside
        the shift kernel (one read, one pooled write) for float32 CUDA tensors; everything else takes the shift followed by
        ``_reduction_fn``."""
        fused = {2: ([2, 2],), 3: ([1, 2, 2], [2, 2, 2])}.get(self.dim, ())
        return (self._reduction_fn is not self._identity and self._stride_ints in fused and input.is_cuda
                and input.dtype == torch.float32 and not input.is_quantized
                and not (self.memory_format is torch.preserve_format and _keeps_channels_last(self.dim, input)))

    def forward(self, input):
        loss = self._compute_weight_loss() if bool(self.sparsity_term) else None
        if self._pool_is_fused(input):
            if self.dim == 3:
                out = shift3d_avgpool_func(input, self.weight, self.padding, self._active_flag, self._stride_ints, self.cut_borders,
                                           _border_ints=self._border_ints())
            else:
                out = shift2d_avgpool2_func(input, self.weight, self.padding, self._active_flag, self.cut_borders,
                                            _border_ints=self._border_ints())
            return out, loss
        if self.cut_borders is None:
            out = self._shift_func(input, self.weight, self.padding, self._active_flag, None, memory_format=self.memory_format)
        else:
            out = self._shift_func(input, self.weight, self.padding, self._active_flag, self.cut_borders,
                                   _border_ints=self._border_ints(), memory_format=self.memory_format)
        return self._reduction_fn(out), loss

    def extra_repr(self):
        pad = dict(zip(paddings_dict.values(), paddings_dict.keys()))[self.padding]
        active = f'Active shift on forward pass: {"Yes" if self._active_flag else "No"}'
        sp = f'Sparse shift: {"Yes - sparsity strength: {}".format(self.sparsity_term) if bool(self.sparsity_term) else "No"}'
        return f'in_channels={self.in_channels}, padding_method={pad}, {active}, {sp}'


def _make_shift_class(dim, what):
    class _Shift(_Shiftnd):
        def __init__(self, in_channels, padding='zeros', init_shift=1, sparsity_term=5e-4, active_flag=False,
                     emulate_dw=None, init_thumb_rule=1, memory_format=torch.contiguous_format):
            self.dim = dim
            super().__init__(in_channels, padding, init_shift, sparsity_term, active_flag, emulate_dw, init_thumb_rule, memory_format)

    _Shift.__name__ = _Shift.__qualname__ = f'Shift{dim}d'
    _Shift.__doc__ = (f'Per-channel learnable shift of a {dim + 2}-D tensor ({what}).\n\n'
                      '    ``forward`` returns ``(output, loss)``; ``loss`` is ``sparsity_term * sum|weight|`` or ``None`` when\n'
                      '    ``sparsity_term`` is 0.  See :class:`_Shiftnd` for the arguments.\n\n'
                      '    Mixed precision: fp16 / bf16 inputs with the fp32 ``weight`` (e.g. under ``torch.autocast``) give an output\n'
                      '    in the input\'s dtype and an fp32 ``weight.grad``; the weights are never cast or rounded to 16 bits.')
    return _Shift


Shift1d = _make_shift_class(1, '[N, C, H], shift along H')
Shift2d = _make_shift_class(2, '[N, C, H, W], shifts along H and W')
Shift3d = _make_shift_class(3, '[N, C, H, W, D], shifts along H, W and D')
