"""ctypes binding of libyolo2_b200.so (include/yolo2_b200.h).  No fallback: if the library is
missing or a call fails, this raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('Y2_LIB_PATH') or os.path.join(_HERE, 'lib', 'libyolo2_b200.so')   # override: A/B experiments

Y2_CONV_LEAKY, Y2_CONV_POOL2, Y2_CONV_OUT_F32, Y2_CONV_IN_SPLIT, Y2_CONV_OUT_SPLIT = 1, 2, 4, 8, 16


class ConvParams(C.Structure):
    _fields_ = [('x', C.c_void_p), ('w_packed', C.c_void_p), ('scale', C.c_void_p), ('shift', C.c_void_p),
                ('y', C.c_void_p), ('N', C.c_int), ('H', C.c_int), ('W', C.c_int), ('Cin', C.c_int),
                ('Cout', C.c_int), ('ksize', C.c_int), ('flags', C.c_int), ('alpha', C.c_float),
                ('ldy', C.c_int), ('lo_off', C.c_int)]


class Y2Error(RuntimeError):
    pass


_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
_SIGNATURES = {
    'y2_version': (C.c_int, []),
    'y2_last_error': (C.c_char_p, []),
    'y2_launch_count': (C.c_ulonglong, []),
    'y2_reload_env': (C.c_int, []),
    'y2_preprocess_u8': (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    'y2_pad_cast_f32_to_bf16c8': (_i, [_vp, _vp, _i, _i, _i, _vp]),
    'y2_resize_bilinear_u8': (_i, [_vp, _i, _i, _vp, _i, _i, _vp]),
    'y2_conv_fwd_f32': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    'y2_conv_cin_padded': (_i, [_i]),
    'y2_conv_packed_weight_elems': (_sz, [_i, _i, _i]),
    'y2_pack_weights_bf16': (_i, [_vp, _vp, _i, _i, _i, _vp]),
    'y2_conv_packed_weight_split_elems': (_sz, [_i, _i, _i]),
    'y2_pack_weights_bf16_split': (_i, [_vp, _vp, _i, _i, _i, _vp]),
    'y2_conv_fwd_bf16': (_i, [C.POINTER(ConvParams), _vp]),
    'y2_conv_workspace_bytes': (_sz, []),
    'y2_conv_set_workspace': (_i, [_vp, _sz]),
    'y2_conv1_u8_packed_weight_elems': (_sz, []),
    'y2_pack_weights_conv1_u8': (_i, [_vp, _vp, _vp, _vp]),
    'y2_conv1_u8_pool_fwd': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    'y2_pack_weights_conv1_u8_split': (_i, [_vp, _vp, _vp, _vp]),
    'y2_conv1_u8_pool_fwd_split': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp]),
    'y2_bn_stats_workspace_bytes': (_sz, [_i, _i]),
    'y2_bn_stats': (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'y2_bn_stats_fold': (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _sz, _vp]),
    'y2_bn_stats_fold_train': (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _f, _vp, _sz, _vp]),
    'y2_bn_fold': (_i, [_vp, _vp, _vp, _vp, _vp, _f, _vp, _vp, _i, _vp]),
    'y2_bn_update_moving': (_i, [_vp, _vp, _vp, _vp, _f, _i, _vp]),
    'y2_affine_leaky_pool': (_i, [_vp, _i, _vp, _vp, _vp, _f, _i, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    'y2_affine_leaky_pool_ex': (_i, [_vp, _i, _vp, _vp, _vp, _f, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'y2_maxpool2x2_bf16': (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    'y2_avgpool': (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp]),
    'y2_cast': (_i, [_vp, _i, _vp, _i, _sz, _vp]),
    'y2_scale_by_device_scalar': (_i, [_vp, _vp, _vp, _sz, _vp]),
    'y2_decode_ref_v1': (_i, [_vp, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _vp]),
    'y2_decode_region': (_i, [_vp, _vp, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    'y2_nms_workspace_bytes': (_sz, [_i, _i, _i]),
    'y2_nms': (_i, [_vp, _vp, _i, _i, _i, _f, _f, _vp, _vp, _i, _vp, _sz, _vp]),
    'y2_detect_fused': (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp, _vp, _vp, _vp, _i, _vp]),
    'y2_detect_workspace_bytes': (_sz, [_i, _i]),
    'y2_detect_split': (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp, _vp, _vp, _vp, _i, _vp, _sz, _vp]),
    'y2_iou': (_i, [_vp, _vp, _vp, _sz, _vp]),
    'y2_loss_v1_workspace_bytes': (_sz, [_i, _i]),
    'y2_loss_v1_fwd_bwd': (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'y2_loss_v1_box_deltas': (_i, [_vp, _vp, _i, _i, _i, _i, _f, _vp, _vp]),
    'y2_region_loss_workspace_bytes': (_sz, [_i, _i]),
    'y2_region_loss_fwd_bwd': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _f, _f, _f, _vp, _vp, _vp, _sz, _vp]),
    'y2_bn_bwd_workspace_bytes': (_sz, [_i, _i]),
    'y2_bn_leaky_pool_bwd': (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _f, _f, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i,
                                  _vp, _sz, _vp]),
    'y2_bn_leaky_pool_bwd_ex': (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _f, _i, _i, _i, _i, _i, _i, _vp, _vp,
                                     _vp, _i, _vp, _sz, _vp]),
    'y2_conv_packed_weight_dgrad_elems': (_sz, [_i, _i, _i]),
    'y2_pack_weights_dgrad_bf16': (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    'y2_conv_wgrad_bf16': (_i, [_vp, _vp, _i, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    'y2_conv_wgrad_c3': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'y2_sum_rows_bf16': (_i, [_vp, _i, _sz, _i, _vp, _vp]),
    'y2_adam_step': (_i, [_vp, _vp, _vp, _vp, _sz, _f, _f, _f, _f, _vp]),
    'y2_adam_step_ex': (_i, [_vp, _vp, _vp, _vp, _sz, _f, _vp, _f, _f, _f, _f, _i, _vp]),
    'y2_softmax_xent_fwd_bwd': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    'y2_momentum_step': (_i, [_vp, _vp, _vp, _sz, _f, _f, _f, _i, _vp]),
}

_lib = None


def load():
    """Load (building first if the .so is absent and nvcc exists).  Raises Y2Error otherwise."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        try:
            from . import build as _build
            _build.build()
        except Exception as e:  # noqa: BLE001
            raise Y2Error('libyolo2_b200.so is missing and could not be built: %s' % e)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=''):
    if rc != 0:
        msg = load().y2_last_error()
        raise Y2Error('%s failed (rc=%d): %s' % (what, rc, msg.decode() if msg else ''))


def exported_symbols():
    return sorted(_SIGNATURES.keys())
