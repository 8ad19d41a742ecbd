"""ctypes binding of libwctb200.so (include/wctb200.h).  No fallback: if the
library is missing or fails to load this module raises -- the product path never
runs on the CPU."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libwctb200.so")

RELU = 1
CLIP01 = 2
HALO_EDGE = 4
POOL2 = 8
EINVAL, ECUDA, EWS, EDEVICE = -1, -2, -3, -4       # include/wctb200.h

_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/wctb200.h one to one
SIGNATURES = {
    "wctb200_abi_version": (_i, []),
    "wctb200_last_error": (C.c_char_p, []),
    "wctb200_check_device": (_i, [_vp]),
    "wctb200_act_bytes": (_sz, [_i, _i, _i, _i]),
    "wctb200_act_from_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "wctb200_act_to_f32": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "wctb200_image_u8_to_f32": (_i, [_vp, _sz, _vp, _vp]),
    "wctb200_image_f32_to_u8": (_i, [_vp, _sz, _vp, _vp]),
    "wctb200_resize_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "wctb200_resize_bilinear_u8": (_i, [_vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "wctb200_rgb_moments_u8": (_i, [_vp, C.c_longlong, _vp, _vp]),
    "wctb200_coral_apply_u8": (_i, [_vp, C.c_longlong, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "wctb200_conv_weight_bytes": (_sz, [_i, _i, _i]),
    "wctb200_prep_conv_weights": (_i, [_vp, _i, _i, _i, _vp, _vp]),
    "wctb200_prep_conv_weights_up2": (_i, [_vp, _i, _i, _vp, _vp]),
    "wctb200_conv3x3": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "wctb200_conv3x3_up2": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "wctb200_conv3x3_ref": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "wctb200_conv_head": (_i, [_vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "wctb200_conv_tail": (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "wctb200_maxpool2": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "wctb200_upsample2": (_i, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "wctb200_wct_workspace_bytes": (_sz, [_i, _i, _i]),
    "wctb200_wct_level": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _f, _f, _f, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "wctb200_wct_style_state_bytes": (_sz, [_i, _i]),
    "wctb200_wct_style_prepare": (_i, [_vp, _i, _i, _i, _i, _f, _f, _f, _vp, _vp, _sz, _vp]),
    "wctb200_wct_apply": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _f, _f, _f, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "wctb200_adain_level": (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _f, _f, _vp, _vp, _sz, _vp]),
    "wctb200_covariance": (_i, [_vp, _i, _i, _i, _i, _f, _vp, _vp, _vp]),
    "wctb200_jacobi_eigh": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "wctb200_style_swap_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "wctb200_style_swap_level": (_i, [_vp, _i, _i, _vp, _i, _i, _i, _i, _i, _f, _f, _f, _vp, _vp, _vp, _sz, _vp]),
    "wctb200_labels_resize_nearest": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "wctb200_wct_regions_workspace_bytes": (_sz, [_i, _i, _i]),
    "wctb200_wct_apply_regions": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _f, _f, _f, _f, _i, _vp, _vp, _vp, _sz, _vp]),
    "wctb200_adain_regions": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _f, _f, _vp, _vp, _sz, _vp]),
}

# tuning / probe hooks (wct_tf_b200/csrc/wctb200_debug.h): NOT part of the ABI, bound for tools/ and tests/ only
DEBUG_SIGNATURES = {
    "wctb200_debug_set_conv_bn": (_i, [_i]),
    "wctb200_debug_set_conv_oversub": (_i, [_i]),
    "wctb200_debug_set_conv_fuse": (_i, [_i]),
    "wctb200_debug_set_jacobi": (_i, [_i, _i]),
    "wctb200_debug_set_jacobi_tolq": (_i, [_f]),
    "wctb200_debug_set_conv_products": (_i, [_i]),
    "wctb200_debug_set_conv_tail_tc": (_i, [_i]),
    "wctb200_debug_set_conv_head_tc": (_i, [_i]),
    "wctb200_debug_set_matfun": (_i, [_i, _i]),
    "wctb200_debug_matfun": (_i, [_vp, _i, _i, _i, _f, _f, _vp, _vp, _vp, _vp]),
    "wctb200_debug_set_cov_stages": (_i, [_i]),
}

_lib = None


class WctB200Error(RuntimeError):
    pass


def load():
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WctB200Error("%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for table in (SIGNATURES, DEBUG_SIGNATURES):
        for name, (res, args) in table.items():
            fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
            fn.restype = res
            fn.argtypes = args
    if lib.wctb200_abi_version() != 1:
        raise WctB200Error("libwctb200 ABI version mismatch")
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise WctB200Error("libwctb200 error %d: %s" % (rc, load().wctb200_last_error().decode()))
