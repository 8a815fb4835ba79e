"""ctypes binding of the C-ABI library (include/octseg.h).

The product path has no CPU implementation: if ``liboctseg.so`` is missing or a call fails the
caller gets an exception, never a silent fallback.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'liboctseg.so')

MAX_SEG = 6
ACT = {'none': 0, 'relu': 1, 'swish': 2, 'sigmoid': 3}
RES = {'none': 0, 'before_act': 1, 'after_act': 2}
OUT = {'bf16_nhwc': 0, 'f32_nchw': 1, 'u8_nchw': 2}

# every symbol include/octseg.h declares; tests check the .so exports all of them
EXPORTS = [
    'octseg_last_error', 'octseg_abi_version', 'octseg_sm_count',
    'octseg_conv_plan_create', 'octseg_conv_plan_destroy', 'octseg_conv_run', 'octseg_conv_plan_info',
    'octseg_stem_pack', 'octseg_maxpool3x3s2', 'octseg_dwconv', 'octseg_se_hidden',
    'octseg_se_gate', 'octseg_se_scale_weights', 'octseg_preprocess_resize_bgr', 'octseg_postprocess',
    'octseg_radial_thickness', 'octseg_overlay', 'octseg_preprocess_resize_gray',
    'octseg_fold_average_threshold', 'octseg_contour_largest', 'octseg_dwconv_pool_slots', 'octseg_preprocess_resize_s2d',
]


class ConvSeg(C.Structure):
    _fields_ = [
        ('ptr', C.c_void_p), ('N', C.c_int32), ('H', C.c_int32), ('W', C.c_int32), ('C', C.c_int32),
        ('ldc', C.c_int32), ('kh', C.c_int32), ('kw', C.c_int32), ('mul', C.c_int32),
        ('off_h', C.c_int32 * 2), ('off_w', C.c_int32 * 2), ('c_per_tile', C.c_int32),
        ('cchunks', C.c_int32), ('kc', C.c_int32), ('wide', C.c_int32),
    ]


class ConvDesc(C.Structure):
    _fields_ = [
        ('nseg', C.c_int32), ('seg', ConvSeg * MAX_SEG), ('phases', C.c_int32),
        ('N', C.c_int32), ('Hq', C.c_int32), ('Wq', C.c_int32), ('TH', C.c_int32), ('TW', C.c_int32),
        ('BN', C.c_int32), ('n_tiles_n', C.c_int32), ('cout_per_tile', C.c_int32), ('Cout', C.c_int32),
        ('weight', C.c_void_p), ('Ktot', C.c_int32), ('per_image_weights', C.c_int32),
        ('bias', C.c_void_p), ('act', C.c_int32), ('res_mode', C.c_int32), ('res', C.c_void_p),
        ('res_ldc', C.c_int32), ('out', C.c_void_p), ('out_mode', C.c_int32), ('out_H', C.c_int32),
        ('out_W', C.c_int32), ('out_ldc', C.c_int32), ('out_c_off', C.c_int32), ('out_pack', C.c_int32),
        ('d2s', C.c_int32), ('halo', C.c_int32),
        ('head_classes', C.c_int32), ('head_cmid', C.c_int32), ('head_weight', C.c_void_p), ('head_bias', C.c_void_p),
        ('head_conv_bias', C.c_void_p),
    ]


class ConvPlanInfo(C.Structure):
    """struct octseg_conv_plan_info: what octseg_conv_plan_create decided for a plan."""
    _fields_ = [(n, C.c_int32) for n in ('grid', 'total_tiles', 'n_acc', 'nstages', 'use_tma_store', 'out_grouped',
                                         'd2s_tma', 'own_spatial', 'halo', 'wide')]


class OctsegError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load liboctseg.so (built in-tree by ``__graft_entry__.build()``); raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OctsegError(
            f'{LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"`. '
            'There is no CPU fallback for the product path.')
    lib = C.CDLL(LIB_PATH)
    lib.octseg_last_error.restype = C.c_char_p
    lib.octseg_abi_version.restype = C.c_int
    lib.octseg_sm_count.restype = C.c_int
    lib.octseg_conv_plan_create.argtypes = [C.POINTER(ConvDesc), C.POINTER(C.c_void_p)]
    lib.octseg_conv_plan_destroy.argtypes = [C.c_void_p]
    lib.octseg_conv_run.argtypes = [C.c_void_p, C.c_void_p]
    lib.octseg_conv_plan_info.argtypes = [C.c_void_p, C.POINTER(ConvPlanInfo)]
    lib.octseg_stem_pack.argtypes = [
        C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
        C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p, C.c_void_p]
    lib.octseg_maxpool3x3s2.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 6 + [C.c_void_p]
    lib.octseg_dwconv.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int32] * 11 + [
        C.c_void_p, C.c_int32, C.c_void_p]
    lib.octseg_dwconv_pool_slots.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    lib.octseg_se_hidden.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                     C.c_int32, C.c_void_p]
    lib.octseg_se_gate.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_void_p]
    lib.octseg_se_scale_weights.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                            C.c_int32, C.c_int32, C.c_void_p]
    lib.octseg_preprocess_resize_s2d.argtypes = [
        C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
        C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.octseg_preprocess_resize_bgr.argtypes = [
        C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
        C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    lib.octseg_preprocess_resize_gray.argtypes = lib.octseg_preprocess_resize_bgr.argtypes
    lib.octseg_postprocess.argtypes = [
        C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_void_p),
        C.POINTER(C.c_int32), C.c_int32,
        C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.octseg_radial_thickness.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                            C.c_void_p, C.c_void_p]
    lib.octseg_overlay.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8),
                                   C.c_int32, C.c_void_p]
    lib.octseg_fold_average_threshold.argtypes = [C.POINTER(C.c_void_p), C.c_int32, C.c_int64, C.c_void_p, C.c_void_p]
    lib.octseg_contour_largest.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_int32, C.c_void_p]
    for name in EXPORTS:
        if name not in ('octseg_last_error',):
            getattr(lib, name).restype = C.c_int
    if lib.octseg_abi_version() != 4:
        raise OctsegError('liboctseg.so ABI version mismatch')
    _lib = lib
    return lib


def check(rc: int, what: str = '') -> None:
    if rc != 0:
        msg = load().octseg_last_error().decode('utf-8', 'replace')
        raise OctsegError(f'{what} failed (code {rc}): {msg}')


def stream_ptr() -> int:
    """Raw cudaStream_t of torch's current stream (kernels are enqueued there)."""
    import torch
    return torch.cuda.current_stream().cuda_stream
