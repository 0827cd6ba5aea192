"""The ``torchshifts::`` operators as registered by ``torchshifts/_ops.py``: schemas and dispatch keys of every op (CPU),
and the planar copy that a channels-last input's layout pass leaves behind (GPU).
"""
import re

import pytest
import torch

FORWARD = "(Tensor input, Tensor weights, Tensor borders, int[] new_size, int padding_mode, bool active_flag) -> Tensor"
BACKWARD = "(Tensor grad, Tensor weights, Tensor input, Tensor borders, int padding_mode, bool active_flag) -> (Tensor, Tensor)"
POOL_BACKWARD = ("(Tensor grad, Tensor weights, Tensor input, Tensor borders, int[] new_size, int padding_mode, "
                 "bool active_flag) -> (Tensor, Tensor)")
COMPOSITE = "(Tensor input, Tensor weights, Tensor borders, int padding_mode, bool active_flag) -> Tensor"
PLANAR_KEYS = ["CPU", "CUDA", "Meta", "QuantizedCPU", "QuantizedCUDA", "Autograd[alias]"]
FLOAT_KEYS = ["CPU", "CUDA", "Meta", "Autograd[alias]"]

OPS = {f"shift{d}d": (COMPOSITE, ["CompositeImplicitAutograd[alias]"]) for d in (1, 2, 3)}
OPS["_cuda_version"] = ("() -> int", ["CompositeExplicitAutograd[alias]"])
for d in (1, 2, 3):
    OPS[f"_shift{d}d_forward"] = (FORWARD, PLANAR_KEYS)
    OPS[f"_shift{d}d_backward"] = (BACKWARD, PLANAR_KEYS)
for d in (2, 3):
    OPS[f"_shift{d}d_forward_cl"] = (FORWARD, FLOAT_KEYS)
    OPS[f"_shift{d}d_backward_cl"] = (BACKWARD, FLOAT_KEYS)
OPS["_shift2d_avgpool2_forward"] = (FORWARD, FLOAT_KEYS)
OPS["_shift2d_avgpool2_backward"] = (POOL_BACKWARD, FLOAT_KEYS)


@pytest.fixture(scope="module")
def native():
    import torchshifts.extension as ext
    assert ext._HAS_OPS, ext.error_str
    return ext.native()


@pytest.mark.parametrize("name", sorted(OPS))
def test_schema_and_dispatch_keys(native, name):
    schema, keys = OPS[name]
    dump = torch._C._dispatch_dump(f"torchshifts::{name}")
    assert re.search(r"^schema: (.*)$", dump, re.M).group(1) == f"torchshifts::{name}{schema}"
    registered = re.findall(r"^(\w+(?:\[alias\])?): registered at", dump, re.M)
    assert registered == ["debug"] + keys


@pytest.mark.gpu
def test_pooled_layer_leaves_no_planar_copy(native):
    """A stride-2 emulated depth-wise conv on a channels-last fp32 input takes the shift + avg_pool2d path, whose layout
    pass makes a planar copy of the input: dropped when no autograd record claims it, kept for the backward and
    reused there otherwise."""
    from torchshifts import Shift2d, _ops
    layer = Shift2d(32, emulate_dw={"kernel_size": 3, "stride": 2, "padding": 1}).cuda()
    x = torch.randn(2, 32, 40, 40, device="cuda").contiguous(memory_format=torch.channels_last)
    assert x.numel() > _ops._COPY_THRESHOLD
    with torch.no_grad():
        y, _ = layer(x)
    assert y.shape == (2, 32, 20, 20)
    assert _ops._LAST_PLANAR[0] is None
    assert _ops._planar_key(x) not in _ops._PLANAR

    x.requires_grad_(True)
    y, _ = layer(x)
    assert _ops._LAST_PLANAR[0] is None
    assert _ops._planar_key(x) in _ops._PLANAR
    y.sum().backward()
    assert _ops._planar_key(x) not in _ops._PLANAR
    assert x.grad is not None and layer.weight.grad is not None
