"""ctypes binding of the C ABI in include/torchshifts_b200.h (libtorchshifts_b200.so).

This module is the only place that talks to the native library.  It has no torch dependency:
pointers, sizes and the stream handle are passed as plain integers.
"""
import ctypes as ct
import os
from pathlib import Path

LIB_NAME = 'libtorchshifts_b200.so'

TS_OK, TS_ERR_UNSUPPORTED, TS_ERR_WORKSPACE, TS_ERR_TOO_LARGE = 0, 2, 3, 4
ABI_VERSION = 2
STATUS_NAMES = {0: 'TS_OK', 1: 'TS_ERR_INVALID_ARGUMENT', 2: 'TS_ERR_UNSUPPORTED', 3: 'TS_ERR_WORKSPACE',
                4: 'TS_ERR_TOO_LARGE', 5: 'TS_ERR_BORDERS', 6: 'TS_ERR_CUDA', 7: 'TS_ERR_NO_DEVICE'}
PATH_NONE, PATH_GENERIC, PATH_STAGED, PATH_TMA, PATH_NHWC, PATH_HALO, PATH_FLAT = 0, 1, 2, 3, 4, 5, 6
QW_U8, QW_I8, QW_I32 = 0, 1, 2
TS_WEIGHTS_F32 = 0x100        # dtype flag: fp16 / bf16 x with fp32 weights and grad_weight


class Geometry(ct.Structure):
    """struct ts_geometry."""
    _fields_ = [('dim', ct.c_int32), ('reserved', ct.c_int32), ('N', ct.c_int64), ('C', ct.c_int64),
                ('size', ct.c_int64 * 3), ('x_stride', ct.c_int64 * 5), ('lb', ct.c_int64 * 3), ('rb', ct.c_int64 * 3)]


class PeerGroup(ct.Structure):
    """struct ts_peer_group."""
    _fields_ = [('world', ct.c_int32), ('rank', ct.c_int32), ('capacity', ct.c_int32), ('reserved', ct.c_int32),
                ('timeout_ns', ct.c_uint64), ('bufs', ct.c_void_p * 8), ('state', ct.c_void_p)]


_vp, _i, _i64, _sz = ct.c_void_p, ct.c_int, ct.c_int64, ct.c_size_t
_geo, _peers, _i64p, _i32p = ct.POINTER(Geometry), ct.POINTER(PeerGroup), ct.POINTER(ct.c_int64), ct.POINTER(ct.c_int32)
# restype and argtypes of every symbol include/torchshifts_b200.h declares
SIGNATURES = {
    'ts_abi_version': (_i, []), 'ts_cuda_version': (_i, []),
    'ts_error_string': (ct.c_char_p, [_i]), 'ts_last_cuda_error': (ct.c_char_p, []),
    'ts_last_kernel_path': (_i, []), 'ts_set_kernel_path': (_i, [_i]),
    'ts_launch_count': (ct.c_uint64, []), 'ts_set_tuning': (_i, [ct.c_char_p]),
    'ts_check_borders': (_i, [_i, _i64p, _i64p, _i64p, _i64p]),
    'ts_debug_remap': (_i, [_i, _i, _i]), 'ts_debug_remap_reduced': (_i, [_i, _i, _i, _i64, _i]),
    'ts_debug_split_f32': (None, [_i, _i, ct.c_float, _i64p, ct.POINTER(ct.c_float)]),
    'ts_debug_split_f64': (None, [_i, _i, ct.c_double, _i64p, ct.POINTER(ct.c_double)]),
    'ts_shift_forward': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp]),
    'ts_shift2d_avgpool2_forward': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp]),
    'ts_shift_backward_workspace_bytes': (_sz, [_geo, _i]),
    'ts_shift_backward': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'ts_shift2d_avgpool2_backward': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'ts_qshift_forward': (_i, [_geo, _i, _i, _i64, _vp, _vp, _i, _i64, _vp, _vp]),
    'ts_qshift_forward_nhwc': (_i, [_geo, _i, _i, _i64, _vp, _vp, _i, _i64, _vp, _vp]),
    'ts_debug_nhwc_emulate': (_i, [_geo, _i, _i, _i64, _vp, _vp, _i, _i64, _vp, _i, _i, _i, _i]),
    'ts_debug_route': (_i, [_geo, _i, _i, _i, _i, _i, _i64p, _i]),
    'ts_nhwc_to_nchw': (_i, [_vp, _vp, _i64, _i64, _i64, _i, _vp]),
    'ts_shift_backward_allreduce': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _peers, _vp]),
    'ts_shift_forward_nhwc': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp]),
    'ts_shift_backward_nhwc_workspace_bytes': (_sz, [_geo, _i]),
    'ts_shift_backward_nhwc': (_i, [_geo, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _peers, _vp]),
    'ts_shift_avgpool_forward': (_i, [_geo, _i, _i, _i, _i32p, _vp, _vp, _vp, _vp]),
    'ts_shift_avgpool_backward_workspace_bytes': (_sz, [_geo, _i]),
    'ts_shift_avgpool_backward': (_i, [_geo, _i, _i, _i, _i32p, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _peers, _vp]),
}
# tests check that the library exports all of them and that the header declares no others
EXPORTED_SYMBOLS = tuple(SIGNATURES)


def make_geometry(dim, shape, strides, lb, rb):
    g = Geometry()
    g.dim = dim
    g.N, g.C = int(shape[0]), int(shape[1])
    for a in range(3):
        g.size[a] = int(shape[2 + a]) if a < dim else 1
        g.lb[a] = int(lb[a]) if a < dim else 0
        g.rb[a] = int(rb[a]) if a < dim else 1
    for a in range(5):
        g.x_stride[a] = int(strides[a]) if a < 2 + dim else 0
    return g


class NativeLibrary:
    def __init__(self, path=None):
        # TORCHSHIFTS_B200_LIB: another build of the same ABI (A/B measurements of kernel changes)
        path = path or os.environ.get('TORCHSHIFTS_B200_LIB')
        self.path = Path(path) if path else Path(__file__).resolve().parent / LIB_NAME
        if not self.path.exists():
            raise ImportError(f'{self.path} not found: build it with `python __graft_entry__.py` '
                              f'(nvcc -gencode arch=compute_100a,code=sm_100a)')
        lib = ct.CDLL(str(self.path))
        self.lib = lib
        for name, (res, args) in SIGNATURES.items():
            if not hasattr(lib, name) and os.environ.get('TORCHSHIFTS_B200_LIB'):
                continue              # an older build under A/B measurement may lack the newest entry points
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        if lib.ts_abi_version() != ABI_VERSION:
            raise ImportError(f'{self.path}: ABI version {lib.ts_abi_version()} != {ABI_VERSION}')
        spec = os.environ.get('TS_TUNING')          # e.g. TS_TUNING="stages=3,use_tma=0"
        if spec and lib.ts_set_tuning(spec.encode()) != TS_OK:
            raise ImportError(f'TS_TUNING={spec!r} is not a valid tuning spec (see ts_set_tuning in include/torchshifts_b200.h)')

    def check(self, status, what):
        if status != TS_OK:
            msg = self.lib.ts_error_string(status).decode()
            extra = self.lib.ts_last_cuda_error().decode() if status in (2, 6, 7) else ''
            raise RuntimeError(f'torchshifts-b200: {what} failed with {STATUS_NAMES.get(status, status)}: {msg}'
                               + (f' [{extra}]' if extra else ''))

    def check_borders(self, dim, sizes, user):
        """csrc/ops/shifts.cpp:93-135 -> (lb, rb) lists of 3."""
        s = (ct.c_int64 * 3)(*([int(v) for v in sizes] + [1] * (3 - dim)))
        lb, rb = (ct.c_int64 * 3)(), (ct.c_int64 * 3)()
        u = None
        if user is not None:
            flat = [int(v) for v in user]
            assert len(flat) >= 2 * dim, 'borders must hold dim x (left, right)'
            u = (ct.c_int64 * (2 * dim))(*flat[:2 * dim])
        st = self.lib.ts_check_borders(dim, s, u, lb, rb)
        if st == 5:
            # the reference fails inside at::empty: "Trying to create tensor with negative dimension"
            raise RuntimeError('torchshifts-b200: borders give a negative output dimension '
                               '(the reference fails here with "Trying to create tensor with negative dimension")')
        self.check(st, 'ts_check_borders')
        return list(lb), list(rb)
