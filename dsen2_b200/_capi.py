"""ctypes binding of the C ABI in ``include/dsen2_b200.h`` -- fails loudly, never falls back."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_longlong, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libdsen2_b200.so")

IMG_F32, IMG_U16 = 0, 1

# name -> (restype, argtypes); must list every symbol the header declares (checked by tests)
SIGNATURES = {
    "dsen2_abi_version": (c_int, []),
    "dsen2_last_error": (c_char_p, []),
    "dsen2_patch_counts": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_int), POINTER(c_int)]),
    "dsen2_extract_patches": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                      c_void_p, c_void_p]),
    "dsen2_bilinear_mirror_up": (c_int, [c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "dsen2_recompose": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p,
                                c_void_p]),
    "dsen2_bicubic_imresize": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                       c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_down_pixel_aggr": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "dsen2_pack_conv_weights": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_conv_relu": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_s2model_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "dsen2_s2model_forward": (c_int, [POINTER(c_void_p), POINTER(c_int), c_int, c_int, c_int, c_int, c_int,
                                      POINTER(c_void_p), POINTER(c_void_p), c_void_p, c_size_t, c_void_p, c_void_p]),
    "dsen2_prep_from_patches": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                        c_void_p, c_void_p]),
    "dsen2_pack_head_weights": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_pack_tail_weights": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_pack_tail16_weights": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_conv_head": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    "dsen2_conv_res32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                 c_void_p, c_void_p]),
    "dsen2_conv_resq": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    "dsen2_prep16_from_patches": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                          c_void_p, c_void_p]),
    "dsen2_prep16_from_images": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                         c_void_p, c_void_p, c_void_p]),
    "dsen2_pack_head16_weights": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_conv_head16_q": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p]),
    "dsen2_conv_head16_relu": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                       c_void_p]),
    "dsen2_conv_tail16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_int, c_int, c_void_p, c_void_p]),
    "dsen2_conv_tail16_stitch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                         c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "dsen2_prep16_from_images_ids": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                             c_float, c_void_p, c_void_p, c_void_p]),
    "dsen2_conv_tail16_stitch_ids": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                             c_int, c_int, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "dsen2_nodata_patches": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                     c_void_p, c_void_p, c_void_p]),
    "dsen2_nodata_fill": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                  c_int, c_void_p, c_void_p]),
    "dsen2_conv_tail16_stitch_u16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                             c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p]),
    "dsen2_conv_tail16_stitch_ids_u16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                                 c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p,
                                                 c_void_p]),
    "dsen2_nodata_fill_u16": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_float, c_int, c_void_p, c_void_p]),
    "dsen2_prep16_from_images_offset": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                                c_void_p, c_int, c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "dsen2_conv_tail16_stitch_offset": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                                c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_int, c_float, c_float,
                                                c_int, c_int, c_void_p, c_void_p]),
    "dsen2_prep16_from_chips": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                        c_int, c_float, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "dsen2_conv_tail16_stitch_chips": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                               c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_int,
                                               c_float, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_conv_resq256": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                   c_void_p, c_void_p]),
    "dsen2_conv_tail": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                c_int, c_void_p, c_void_p]),
    "dsen2_pack_dgrad_weights": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p]),
    "dsen2_pack_trunk_layers": (c_int, [c_void_p, c_longlong, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "dsen2_conv_relu_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "dsen2_nchw_to_nhwc_f16": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                       c_void_p, c_void_p]),
    "dsen2_relu_mask": (c_int, [c_void_p, c_void_p, c_longlong, c_void_p, c_void_p]),
    "dsen2_wgrad_nhwc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "dsen2_mae_grad": (c_int, [c_void_p, c_void_p, c_longlong, c_float, c_void_p, c_void_p, c_void_p]),
    "dsen2_nadam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong] + [c_float] * 10 + [c_void_p]),
    "dsen2_nadam_step_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p]),
}


class DSen2Error(RuntimeError):
    pass


_lib = None


def lib():
    """Load the shared library (once).  Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DSen2Error(
                "dsen2_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or dsen2_b200/build.py).  There is no CPU fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        if handle.dsen2_abi_version() != 3:
            raise DSen2Error("dsen2_b200: ABI version mismatch")
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().dsen2_last_error()
        raise DSen2Error("%s failed (code %d): %s" % (what, rc, msg.decode("utf-8", "replace") if msg else ""))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise DSen2Error("dsen2_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
    return torch


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)
