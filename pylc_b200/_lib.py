"""
ctypes binding of the pylc_b200 C ABI (include/pylc_b200.h).

The shared library is built in-tree by `__graft_entry__.build()` / `make -C pylc_b200/csrc` into
pylc_b200/lib/libpylc_b200.so.  There is no CPU fallback: if the library is missing or a call
fails, this module raises.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64,
                    c_size_t, c_uint8, c_uint64, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libpylc_b200.so")

MAX_CLASSES = 32
AREA_TAPS = 6
ABI_VERSION = 6
MAX_SCALES = 8
SCORES_WS_DOUBLES = 2048      # PYLC_SCORES_WS_DOUBLES


class PylcError(RuntimeError):
    pass


class LossCfg(Structure):
    """struct pylc_loss_cfg"""
    _fields_ = [("ce_weight", c_float), ("dice_weight", c_float), ("focal_weight", c_float),
                ("dice_smooth", c_float), ("fl_gamma", c_float), ("fl_alpha", c_float),
                ("eps", c_float)]


_u8p = c_void_p      # device / host byte pointers are passed as raw addresses
_ptr = c_void_p

# name -> (restype, argtypes); must list every symbol declared in include/pylc_b200.h
SIGNATURES = {
    "pylc_abi_version": (c_int, []),
    "pylc_error_string": (c_char_p, [c_int]),
    "pylc_device_info": (c_int, [POINTER(c_int), POINTER(c_int)]),
    "pylc_launch_count": (c_int64, []),
    "pylc_tile_grid": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "pylc_tile_gather_u8": (c_int, [_u8p, c_int, c_int, c_int, c_size_t, c_int, c_int, _u8p, _ptr, _ptr]),
    "pylc_mask_gather_encode_hist": (c_int, [_u8p, c_int, c_int, c_size_t, c_int, c_int,
                                             POINTER(c_uint8), c_int, _u8p, _ptr, _ptr]),
    "pylc_tile_gather_u8_stack": (c_int, [_u8p, c_int, c_size_t, c_int, c_int, c_int, c_size_t, c_int, c_int, _u8p, _ptr, _ptr]),
    "pylc_mask_gather_encode_hist_stack": (c_int, [_u8p, c_int, c_size_t, c_int, c_int, c_size_t, c_int, c_int,
                                                   POINTER(c_uint8), c_int, _u8p, _ptr, _ptr]),
    "pylc_class_encode": (c_int, [_u8p, c_int, c_int, c_int, c_size_t, c_int, POINTER(c_uint8), c_int,
                                  _u8p, _ptr, _ptr]),
    "pylc_profile_tiles": (c_int, [_u8p, c_int, _u8p, c_int, c_int64, c_int, _ptr, _ptr, _ptr]),
    "pylc_tile_gather_norm_f32": (c_int, [_u8p, c_int, c_int, c_int, c_size_t, c_int, c_int,
                                          POINTER(c_float), POINTER(c_float), c_float, c_int, _ptr, _ptr]),
    "pylc_sample_rate_grid": (c_int, [_ptr, _ptr, c_int, c_int, _ptr, c_int, _ptr, c_int, c_int, c_int, _ptr, _ptr, _ptr]),
    "pylc_augment_tiles_u8": (c_int, [_u8p, _u8p, c_int, c_int, c_int, _ptr, _ptr, _ptr, c_int, _u8p, _u8p, _ptr]),
    "pylc_area_supported": (c_int, [c_int, c_int, c_int, c_int]),
    "pylc_area_table": (c_int, [c_int, c_int, _ptr, _ptr, _ptr]),
    "pylc_fit_resize_area_u8": (c_int, [_u8p, c_int, c_int, c_int, c_size_t, _u8p, c_int, c_int, c_size_t,
                                        _ptr, _ptr, _ptr, _ptr, _ptr, _ptr, _ptr]),
    "pylc_upload_pitched": (c_int, [_ptr, c_size_t, _ptr, c_size_t, c_size_t, c_size_t, _ptr]),
    "pylc_upsample_concat_nhwc_f32": (c_int, [_ptr, c_int, c_int, c_int, c_int, _ptr, c_int, c_int, c_int, _ptr, _ptr]),
    "pylc_maxpool3x3s2_nhwc_f32": (c_int, [_ptr, c_int, c_int, c_int, c_int, _ptr, _ptr]),
    "pylc_tap_combine_relu_f32": (c_int, [_ptr, c_int, c_int, c_int, c_int, POINTER(ctypes.c_void_p), POINTER(ctypes.c_int32),
                                          POINTER(ctypes.c_int32), POINTER(ctypes.c_int32), POINTER(ctypes.c_int32), c_int, _ptr]),
    "pylc_upsample_nhwc_to_nchw_f32": (c_int, [_ptr, c_int, c_int, c_int, c_int, _ptr, c_int, c_int, _ptr]),
    "pylc_tile_gather_norm_s2d_f32": (c_int, [_u8p, c_int, c_int, c_int, c_size_t, c_int, c_int,
                                              POINTER(c_float), POINTER(c_float), c_float, _ptr, _ptr]),
    "pylc_stitch_probs": (c_int, [_ptr, _ptr, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                  POINTER(c_uint8), _u8p, _u8p, _u8p, _ptr, c_float, _ptr]),
    "pylc_stitch_upsample_probs": (c_int, [_ptr, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                           POINTER(c_uint8), _u8p, _u8p, _u8p, _ptr, c_float, _ptr]),
    "pylc_colourise_u8": (c_int, [_u8p, c_int64, POINTER(c_uint8), c_int, _u8p, _ptr]),
    "pylc_prob_scores": (c_int, [_ptr, c_int, c_int, c_int, _ptr, _ptr, c_int, c_int, _u8p, c_int, _ptr, _ptr, _ptr]),
    "pylc_resample_encode_confusion": (c_int, [_u8p, c_int, c_int, _ptr, _ptr, c_int, c_int, _u8p, c_size_t,
                                               POINTER(c_uint8), POINTER(c_uint8), c_int, c_int, _ptr,
                                               _u8p, _u8p, _u8p, _ptr]),
    "pylc_confusion_u8": (c_int, [_u8p, _u8p, c_int64, c_int, c_int, _ptr, _ptr]),
    "pylc_confidence_resample": (c_int, [_u8p, c_int, c_int, _ptr, _ptr, c_int, c_int, _u8p, _u8p, c_int, _u8p, _ptr, _ptr]),
    "pylc_multiscale_combine": (c_int, [_ptr, _ptr, _ptr, POINTER(c_int), POINTER(c_int), c_int, c_int, c_int, c_int,
                                        POINTER(c_uint8), _u8p, _u8p, _u8p, _ptr]),
    "pylc_multiloss_reduce": (c_int, [_ptr, _ptr, c_int, c_int, c_int, c_int64, _ptr, POINTER(LossCfg),
                                      _ptr, _u8p, _ptr]),
    "pylc_multiloss_finalize": (c_int, [_ptr, c_int, c_int64, POINTER(LossCfg), _ptr, _ptr]),
    "pylc_multiloss_grad": (c_int, [_ptr, _ptr, c_int, c_int, c_int, c_int64, _ptr, POINTER(LossCfg),
                                    _ptr, c_int64, c_float, _ptr, _ptr, _ptr]),
    "pylc_multiloss_fwd_bwd": (c_int, [_ptr, _ptr, c_int, c_int, c_int, c_int64, _ptr, POINTER(LossCfg),
                                       _ptr, c_float, _ptr, _ptr, _ptr, _u8p, _ptr]),
    "pylc_multiloss_fwd_bwd_dp": (c_int, [_ptr, _ptr, c_int, c_int, c_int, c_int64, _ptr, POINTER(LossCfg),
                                          _ptr, c_float, _ptr, _ptr, _ptr, _u8p, _ptr, c_int, c_int, ctypes.c_uint64, _ptr]),
    "pylc_scale_unless_one_f32": (c_int, [_ptr, c_int64, _ptr, _ptr]),
}

_lib = None


def load():
    """Load (once) and return the ctypes handle; raises PylcError if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise PylcError(
            "pylc_b200 CUDA library not found at %s -- build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `make -C pylc_b200/csrc`. "
            "There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise PylcError("libpylc_b200.so does not export %s" % name) from exc
        fn.restype = restype
        fn.argtypes = argtypes
    ver = lib.pylc_abi_version()
    if ver != ABI_VERSION:
        raise PylcError("libpylc_b200.so ABI version %d, binding expects %d" % (ver, ABI_VERSION))
    _lib = lib
    return lib


def check(code, what):
    if code != 0:
        msg = load().pylc_error_string(code)
        raise PylcError("%s failed: %s (code %d)" % (what, msg.decode() if msg else "?", code))


def launch_count():
    return int(load().pylc_launch_count())


_PALETTES = {}


def palette_array(palette):
    """HOST [C,3] u8 array for the `palette` / `lut_rgb` arguments (cached per palette)."""
    key = tuple(int(v) for rgb in palette for v in rgb)
    hit = _PALETTES.get(key)
    if hit is None:
        if len(key) % 3 or any(v < 0 or v > 255 for v in key):
            raise PylcError("palette must be a list of [R,G,B] byte triples")
        if len(_PALETTES) > 256:
            _PALETTES.clear()
        hit = _PALETTES[key] = ((c_uint8 * len(key))(*key), len(key) // 3)
    return hit


def float3(vals):
    vals = [float(v) for v in vals]
    while len(vals) < 3:
        vals.append(vals[-1])
    return (c_float * 3)(*vals[:3])
