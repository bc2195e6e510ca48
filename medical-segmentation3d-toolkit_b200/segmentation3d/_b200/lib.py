"""ctypes binding of the C-ABI CUDA library (include/seg3d_b200.h).

The library is the product: there is no Python/torch fallback.  If it is missing or a call
fails, a RuntimeError is raised.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SEG3D_LIB') or os.path.abspath(os.path.join(_HERE, '..', '..', 'lib', 'libseg3d_b200.so'))   # SEG3D_LIB: a variant build (kernel experiments)

F32, F16, BF16 = 0, 1, 2
OUT_F32 = 0x100
CONV_K3, CONV_K2S2, CONV_T2S2, CONV_K1 = 0, 1, 2, 3
IMPL_AUTO, IMPL_SIMT, IMPL_TCGEN05 = 0, 1, 2
NORM_NONE, NORM_FIXED, NORM_ADAPTIVE = 0, 1, 2
CIN1_PAD, CIN1_LEFT = 16, 9           # row padding of the input block's tensor-core layout (seg3d_conv3d_cin1_fwd)

TORCH_DTYPE = {F32: torch.float32, F16: torch.float16, BF16: torch.bfloat16}
DTYPE_CODE = {v: k for k, v in TORCH_DTYPE.items()}

_vp, _i, _f, _i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_int64

_SIGNATURES = {
    'seg3d_version': (_i, []),
    'seg3d_last_error': (ctypes.c_char_p, []),
    'seg3d_device_check': (_i, [_i]),
    'seg3d_conv3d_fwd': (_i, [_i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_conv3d_cin1_fwd': (_i, [_i, _i, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _f, _vp]),
    'seg3d_conv3d_cin1_wgrad': (_i, [_i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _vp]),
    'seg3d_conv3d_cin1_dgrad': (_i, [_i, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp]),
    'seg3d_conv3d_k3_narrow_np': (_i, [_i]),
    'seg3d_conv3d_k3_narrow_fwd': (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_conv3d_k3_gnin_fwd': (_i, [_i, _vp, _i, _i, _i, _vp, _vp, _vp, _f, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_conv3d_k3_narrow_gn2_fwd': (_i, [_i, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_conv3d_k3_narrow_split_fwd': (_i, [_vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_conv3d_k3_narrow_gn_fwd': (_i, [_i, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _f, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_conv3d_gn_relu_fwd': (_i, [_i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _f, _vp]),
    'seg3d_conv3d_split_fwd': (_i, [_i, _vp, _i, _i, _i, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_gn_apply_split': (_i, [_vp, _i, _i, _vp, _vp, _vp, _f, _vp, _i, _i, _vp, _i, _i, _i, _i, _i64, _vp]),
    'seg3d_gn_apply': (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _f, _vp, _i, _vp, _i, _i, _i, _i64, _vp]),
    'seg3d_outblock_tail_stats': (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _i, _i64, _vp]),
    'seg3d_outblock_tail_probs': (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _i, _i64, _vp]),
    'seg3d_outblock_tail_wide': (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _i, _i64, _vp]),
    'seg3d_patch_stats': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _vp, _vp]),
    'seg3d_patch_gather': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _f, _f, _i, _f, _f, _vp, _i, _vp, _vp]),
    'seg3d_patch_gather_rows': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _i, _f, _f, _i, _f, _f, _vp, _i, _vp, _i, _i, _vp]),
    'seg3d_blend_accumulate': (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _vp]),
    'seg3d_blend_finalize_argmax': (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    'seg3d_blend_finalize_argmax_z': (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    'seg3d_resample': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, ctypes.c_double, ctypes.c_double, ctypes.c_double, _i, _f, _vp]),
    'seg3d_crop_resample': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, ctypes.c_double, ctypes.c_double, ctypes.c_double,
                                 ctypes.c_double, ctypes.c_double, ctypes.c_double, _i, _f, _vp]),
    'seg3d_cc_filter': (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    'seg3d_dice_terms': (_i, [_vp, _vp, _i, _i, _i64, _vp, _vp]),
    'seg3d_dice_bwd': (_i, [_vp, _vp, _i, _i, _i64, _vp, _vp, _vp]),
    'seg3d_focal_fwd': (_i, [_vp, _vp, _i, _i, _i64, _vp, _f, _vp, _vp]),
    'seg3d_focal_bwd': (_i, [_vp, _vp, _i, _i, _i64, _vp, _f, _f, _vp, _vp]),
    'seg3d_ce_fwd': (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _vp, _vp, _vp]),
    'seg3d_ce_bwd': (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _f, _vp, _vp, _vp]),
    'seg3d_gn_bwd': (_i, [_i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp, _vp, _vp, _f, _vp, _vp, _vp,
                          _vp, _i, _vp, _i, _vp, _i, _i64, _vp]),
    'seg3d_gn_bwd_noact': (_i, [_i, _i, _vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _vp, _vp, _f, _vp, _vp, _vp,
                                _vp, _i, _vp, _i, _vp, _i, _i64, _vp]),
    'seg3d_grad_to_ncdhw': (_i, [_i, _i, _vp, _i, _i, _vp, _i, _i, _vp, _i, _i, _i, _i, _i64, _vp, _vp]),
    'seg3d_grad_from_ncdhw': (_i, [_i, _vp, _i, _i, _i64, _vp, _i, _i, _vp]),
    'seg3d_conv3d_wgrad': (_i, [_i, _i, _vp, _i, _i, _vp, _i, _i, _vp, _i, _i, _i, _i, _vp]),
    'seg3d_outblock_tail_bwd': (_i, [_i, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i64, _vp]),
    'seg3d_gather_pack': (_i, [_vp, _vp, _i, _vp]),
    'seg3d_adam_step': (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f, _f, _i, _vp]),
    'seg3d_adam_step_ranges': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _f, _f, _f, _f, _f, _vp]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class PackEntry(ctypes.Structure):
    """seg3d_pack_entry of include/seg3d_b200.h"""
    _fields_ = [('src', ctypes.c_void_p), ('dst', ctypes.c_void_p), ('src_base', ctypes.c_int64), ('dst_base', ctypes.c_int64),
                ('src_stride', ctypes.c_int64 * 5), ('dst_stride', ctypes.c_int64 * 5),
                ('size', ctypes.c_int32 * 5), ('limit', ctypes.c_int32 * 5), ('dtype', ctypes.c_int32), ('kind', ctypes.c_int32)]


class AdamRange(ctypes.Structure):
    """seg3d_adam_range of include/seg3d_b200.h"""
    _fields_ = [('offset', ctypes.c_int64), ('n', ctypes.c_int64), ('step', ctypes.c_int64)]


PACK_PLAIN, PACK_SPLIT_HI, PACK_SPLIT_LO = 0, 1, 2
PACK_CHUNK = 4096

_lib = None


def load():
    """Load libseg3d_b200.so (built by medical-segmentation3d-toolkit_b200/build.py). Raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError('seg3d_b200: CUDA library not built: %s (run __graft_entry__.build())' % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _check(rc, name):
    if rc != 0:
        raise RuntimeError('%s failed (%d): %s' % (name, rc, load().seg3d_last_error().decode()))


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def ptr(t, elem_offset=0):
    """device pointer of tensor `t` advanced by `elem_offset` elements (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr() + elem_offset * t.element_size()


def call(name, *args):
    _check(getattr(load(), name)(*args), name)
