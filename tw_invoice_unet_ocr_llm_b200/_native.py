"""ctypes binding of ``libunetb200.so`` (C ABI declared in ``include/unetb200.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``python -m
tw_invoice_unet_ocr_llm_b200.build``.  There is no fallback: if the shared object
is missing, importing :func:`lib` raises with the build command.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# UNETB200_LIB: load an alternative build of the same sources (A/B of compile-time switches); default in-tree
LIB_PATH = os.environ.get("UNETB200_LIB") or os.path.join(_HERE, "libunetb200.so")

OK, EINVAL, ECUDA, EARCH, ENOMEM = 0, 1, 2, 3, 4
STEM, CONV3X3, CONVT2X2, HEAD = 0, 1, 2, 3
X_F32_NCHW, X_U8_NHWC, X_F16_NCHW, X_BF16_NCHW, X_F32_NHWC, X_F16_NHWC, X_BF16_NHWC = range(7)
LOGITS_F32, LOGITS_F16, LOGITS_BF16 = 0, 1, 2
A_TAP, A_COL3, A_HALO = 0, 1, 2


class Arch(C.Structure):
    _fields_ = [("n_channels", C.c_int32), ("n_classes", C.c_int32), ("base_width", C.c_int32)]


class Layer(C.Structure):
    _fields_ = [
        ("name", C.c_char * 32),
        ("bn_name", C.c_char * 32),
        ("kind", C.c_int32),
        ("cin", C.c_int32),
        ("cout", C.c_int32),
        ("level", C.c_int32),
        ("w_off", C.c_uint64),
        ("w_bytes", C.c_uint64),
        ("b_off", C.c_uint64),
        ("b_bytes", C.c_uint64),
    ]


class EnhCrop(C.Structure):
    """``unetb200_enh_crop`` (include/unetb200.h): one crop of an enhancement batch."""
    _fields_ = [
        ("h", C.c_int32), ("w", C.c_int32), ("flags", C.c_int32), ("clip", C.c_float),
        ("clip_count", C.c_int32), ("tile_h", C.c_int32), ("tile_w", C.c_int32),
        ("first_block", C.c_int32), ("blocks_x", C.c_int32), ("n_blocks", C.c_int32),
        ("src_stride", C.c_int32), ("src_pixel_bytes", C.c_int32),
        ("src_off", C.c_uint64), ("out_off", C.c_uint64), ("ws_off", C.c_uint64),
    ]


class WarpCrop(C.Structure):
    """``unetb200_warp_crop`` (include/unetb200.h): one crop of an affine-crop batch."""
    _fields_ = [
        ("src", C.c_uint64), ("src_h", C.c_int32), ("src_w", C.c_int32), ("src_stride", C.c_int32),
        ("src_pixel_bytes", C.c_int32), ("m", C.c_double * 6), ("out_w", C.c_int32), ("out_h", C.c_int32),
        ("out_off", C.c_uint64),
    ]


# every symbol include/unetb200.h declares: name -> (restype, argtypes)
_VP, _I, _U64, _F = C.c_void_p, C.c_int, C.c_uint64, C.c_float
SYMBOLS = {
    "unetb200_abi_version": (_I, []),
    "unetb200_build_flags": (_I, []),
    "unetb200_last_error": (C.c_char_p, []),
    "unetb200_num_layers": (_I, [C.POINTER(Arch)]),
    "unetb200_layer_info": (_I, [C.POINTER(Arch), _I, C.POINTER(Layer)]),
    "unetb200_packed_bytes": (_U64, [C.POINTER(Arch)]),
    "unetb200_pack_layer": (_I, [C.POINTER(Arch), _I, _VP, _VP, _VP, _VP, _VP, _VP, _F, _VP, _VP]),
    "unetb200_pack_fused_up": (_I, [C.POINTER(Arch), _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _F, _VP, _VP]),
    "unetb200_fused_up_info": (_I, [C.POINTER(Arch), _I, C.POINTER(_U64), C.POINTER(_U64), C.POINTER(_U64),
                                    C.POINTER(_U64)]),
    "unetb200_create": (_I, [C.POINTER(Arch), _VP, _U64, _I, C.POINTER(_VP)]),
    "unetb200_destroy": (_I, [_VP]),
    "unetb200_set_option": (_I, [_VP, C.c_char_p, _I]),
    "unetb200_get_option": (_I, [_VP, C.c_char_p, C.POINTER(_I)]),
    "unetb200_workspace_bytes": (_U64, [_VP, _I, _I, _I]),
    "unetb200_forward": (_I, [_VP, _VP, _I, _I, _I, _I, _VP, _U64, _VP, _VP, C.POINTER(_F), _VP]),
    "unetb200_forward_bits": (_I, [_VP, _VP, _I, _I, _I, _I, _VP, _U64, _VP, _VP, C.POINTER(_F), _VP]),
    "unetb200_forward_typed": (_I, [_VP, _VP, _I, _I, _I, _I, _VP, _U64, _VP, _I, _VP, _I, C.POINTER(_F), _VP]),
    "unetb200_layer_times": (_I, [_VP, C.POINTER(_F), _I]),
    "unetb200_last_launch_count": (_I, [_VP]),
    "unetb200_conv3x3": (_I, [_VP, _I, _VP, _I, _VP, _VP, _I, _I, _I, _I, _I, _VP, _VP, _I, _I, _I, _VP]),
    "unetb200_conv3x3_head": (_I, [_VP, _I, _VP, _VP, _VP, _VP, _I, _I, _I, _I, _VP, _VP,
                                   C.POINTER(_F), _I, _I, _VP]),
    "unetb200_convt2x2": (_I, [_VP, _I, _VP, _VP, _I, _I, _I, _I, _VP, _I, _VP]),
    "unetb200_upconv3x3": (_I, [_VP, _I, _VP, _I, _VP, _VP, _I, _VP, _I, _I, _I, _I, _I, _VP, _I, _I, _VP]),
    "unetb200_stem": (_I, [_VP, _I, _I, _VP, _VP, _I, _I, _I, _VP, _VP]),
    "unetb200_stem_tc": (_I, [_VP, _I, _I, _VP, _VP, _I, _I, _I, _VP, _VP]),
    "unetb200_stem_tc_offset": (_U64, [_I]),
    "unetb200_stem_patch": (_I, [_VP, _I, _I, _VP, _VP, _I, _I, _I, _VP, _VP]),
    "unetb200_stem_patch_offset": (_U64, [_I]),
    "unetb200_resize_ksize": (_I, [_I, _I]),
    "unetb200_resize_coeffs": (_I, [_I, _I, _VP, _VP]),
    "unetb200_resize_bicubic_u8": (_I, [_VP, _I, _I, _I, _I, _VP, _VP, _I, _VP, _VP, _I, _VP, _VP, _I, _I, _VP]),
    "unetb200_resize_bicubic_u8_ps": (_I, [_VP, _I, _I, _I, _I, _I, _VP, _VP, _I, _VP, _VP, _I, _VP, _VP, _I, _I, _VP]),
    "unetb200_mask_bbox": (_I, [_VP, _I, _I, _I, _VP, _VP]),
    "unetb200_mask_bbox_bits": (_I, [_VP, _I, _I, _I, _VP, _VP]),
    "unetb200_components_workspace_bytes": (_U64, [_I, _I, _I]),
    "unetb200_mask_components": (_I, [_VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _U64, _VP]),
    "unetb200_components_oriented_workspace_bytes": (_U64, [_I, _I, _I]),
    "unetb200_mask_components_oriented": (_I, [_VP, _I, _I, _I, _I, _I, _I, _VP, _VP, _VP, _VP, _VP, _VP, _VP,
                                               _U64, _VP]),
    "unetb200_warp_crops": (_I, [C.POINTER(WarpCrop), _VP, _I, _VP, _VP, _VP]),
    "unetb200_box_sums": (_I, [_VP, _I, _I, _I, C.POINTER(C.c_int32), _I, _VP, _VP]),
    "unetb200_box_sums_ps": (_I, [_VP, _I, _I, _I, _I, C.POINTER(C.c_int32), _I, _VP, _VP]),
    "unetb200_test_fastdiv": (C.c_uint32, [C.c_uint32, C.c_uint32]),
    "unetb200_enhance_plan": (_I, [C.POINTER(EnhCrop), _I, C.POINTER(_U64), C.POINTER(_U64), C.POINTER(_U64)]),
    "unetb200_enhance_run": (_I, [C.POINTER(EnhCrop), _VP, _I, _VP, _VP, _VP, _VP]),
}

_lib = None
_lock = threading.Lock()


class UnetB200Error(RuntimeError):
    """A libunetb200 call returned a non-zero code."""

    def __init__(self, code: int, message: str):
        super().__init__(f"libunetb200 error {code}: {message}")
        self.code = code


def lib() -> C.CDLL:
    """Load the shared library (once) and attach prototypes."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no "
                    "fallback path. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(or `python -m tw_invoice_unet_ocr_llm_b200.build`) from the repository root."
                )
            handle = C.CDLL(LIB_PATH)
            for name, (res, args) in SYMBOLS.items():
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def has_test_variants() -> bool:
    """True when the library was built with -DUNETB200_TEST_VARIANTS (A_COL3 staging, patch stem)."""
    return bool(lib().unetb200_build_flags() & 1)


def last_error() -> str:
    return (lib().unetb200_last_error() or b"").decode("utf-8", "replace")


def check(code: int) -> None:
    if code != OK:
        raise UnetB200Error(code, last_error())


def layer_table(arch: Arch) -> list[Layer]:
    n = lib().unetb200_num_layers(C.byref(arch))
    if n < 0:
        raise UnetB200Error(EINVAL, last_error())
    out = []
    for i in range(n):
        l = Layer()
        check(lib().unetb200_layer_info(C.byref(arch), i, C.byref(l)))
        out.append(l)
    return out
