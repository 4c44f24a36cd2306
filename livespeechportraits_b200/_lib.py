"""ctypes binding of the C ABI in include/lspg.h.  Plain pointers and sizes only."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import build as _build

LSPG_VARIANT = {"normal": 0, "large": 1}
LSPG_MODE = {"fast": 0, "parity": 1}

SYMBOLS = [
    "lspg_create", "lspg_load_weights", "lspg_workspace_bytes", "lspg_forward", "lspg_forward_image", "lspg_draw_feature_maps", "lspg_destroy",
    "lspg_last_error",
    "lspg_num_layers", "lspg_layer_info_get", "lspg_layer_packed", "lspg_layer_affine", "lspg_num_tensors",
    "lspg_tensor_shape", "lspg_debug_read_tensor", "lspg_launches_per_forward", "lspg_flops_per_frame",
    "lspg_profile_enable", "lspg_profile_read", "lspg_debug_read_trace", "lspg_debug_fast_div", "lspg_debug_layer_geo",
    "lspg_graph_stats", "lspg_release_workspace", "lspg_debug_tensor_offset",
]

# include/lsph.h (Audio2Headpose generation loop)
SYMBOLS_H = ["lsph_create", "lsph_load_weights", "lsph_generate", "lsph_receptive_field", "lsph_debug_packed", "lsph_destroy",
             "lsph_last_error"]


class LsphConfig(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("apc_hidden", "frame_future", "layers", "blocks", "residual_ch", "dilation_ch", "skip_ch",
                                       "kernel_size", "use_bias", "cond_ch", "input_ch", "ncenter", "ndim", "loss_gmm")]


class LspgTensor(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.POINTER(C.c_float)), ("numel", C.c_int64)]


class LspgLayerInfo(C.Structure):
    _fields_ = [
        ("kind", C.c_int), ("n_src", C.c_int), ("src", C.c_int * 2), ("cin", C.c_int * 2),
        ("out", C.c_int), ("res", C.c_int), ("cout", C.c_int), ("cout_pad", C.c_int),
        ("n_phases", C.c_int), ("n_taps", C.c_int), ("k_total", C.c_int), ("relu", C.c_int), ("has_bn", C.c_int),
        ("tap_map", (C.c_int8 * 9) * 4), ("tap_dx", (C.c_int8 * 9) * 4), ("tap_dy", (C.c_int8 * 9) * 4),
        ("conv_key", C.c_char * 96), ("bn_key", C.c_char * 96),
    ]


class LspgLayerGeo(C.Structure):
    _fields_ = [("kernel", C.c_int), ("bn", C.c_int), ("tile_w", C.c_int), ("tile_h", C.c_int), ("tile_n", C.c_int),
                ("m_tiles", C.c_int), ("n_tiles", C.c_int), ("n_phases", C.c_int), ("n_split", C.c_int), ("split_len", C.c_int),
                ("k_items", C.c_int), ("ctas", C.c_int), ("partial_bytes", C.c_int64), ("cluster_split", C.c_int),
                ("cta_cluster", C.c_int)]


class LspgError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"lspg error {code}: {message}")
        self.code = code


_LIB: Optional[C.CDLL] = None


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load liblspg.so (building it with nvcc first if the in-tree copy is absent or stale).

    There is deliberately no alternative implementation: if the library cannot be built or loaded the
    error propagates.
    """
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if build_if_missing and _build.needs_build():
        try:
            _build.build_library()
        except Exception as exc:
            if not os.path.exists(path):
                raise
            # a stale library next to newer sources: usable (the GPU box has no reason to rebuild), but say so loudly
            import warnings
            warnings.warn(f"liblspg.so is older than its sources and could not be rebuilt ({exc}); using the existing binary",
                          RuntimeWarning)
    lib = C.CDLL(path)
    lib.lspg_last_error.restype = C.c_char_p
    lib.lspg_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    lib.lspg_load_weights.argtypes = [C.c_void_p, C.POINTER(LspgTensor), C.c_int]
    lib.lspg_workspace_bytes.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_size_t)]
    lib.lspg_forward.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_int,
                                 C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    lib.lspg_forward_image.argtypes = lib.lspg_forward.argtypes
    lib.lspg_debug_layer_geo.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(LspgLayerGeo)]
    lib.lspg_debug_tensor_offset.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.POINTER(C.c_size_t)]
    lib.lspg_debug_fast_div.argtypes = [C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
    lib.lspg_draw_feature_maps.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                           C.c_void_p]
    lib.lspg_destroy.argtypes = [C.c_void_p]
    lib.lspg_release_workspace.argtypes = [C.c_void_p, C.c_void_p]
    lib.lspg_graph_stats.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.lspg_num_layers.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    lib.lspg_layer_info_get.argtypes = [C.c_void_p, C.c_int, C.POINTER(LspgLayerInfo)]
    lib.lspg_layer_packed.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64]
    lib.lspg_layer_affine.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
    lib.lspg_num_tensors.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    lib.lspg_tensor_shape.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                      C.POINTER(C.c_int)]
    lib.lspg_debug_read_tensor.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64]
    lib.lspg_launches_per_forward.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    lib.lspg_debug_read_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
    lib.lspg_profile_enable.argtypes = [C.c_void_p, C.c_int]
    lib.lspg_profile_read.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    lib.lspg_flops_per_frame.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_double)]
    for name in SYMBOLS:
        if name != "lspg_last_error":
            getattr(lib, name).restype = C.c_int
    lib.lsph_last_error.restype = C.c_char_p
    lib.lsph_create.argtypes = [C.POINTER(C.c_void_p), C.POINTER(LsphConfig), C.c_int]
    lib.lsph_load_weights.argtypes = [C.c_void_p, C.POINTER(LspgTensor), C.c_int]
    lib.lsph_generate.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_float, C.c_void_p,
                                  C.c_void_p, C.c_int, C.c_void_p]
    lib.lsph_receptive_field.argtypes = [C.c_void_p, C.POINTER(C.c_int)]
    lib.lsph_destroy.argtypes = [C.c_void_p]
    lib.lsph_debug_packed.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int64]
    for name in SYMBOLS_H:
        if name != "lsph_last_error":
            getattr(lib, name).restype = C.c_int
    _LIB = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        raise LspgError(code, (load().lspg_last_error() or b"").decode("utf-8", "replace"))


def check_h(code: int) -> None:
    if code != 0:
        raise LspgError(code, (load().lsph_last_error() or b"").decode("utf-8", "replace"))
