"""ctypes binding of libcbinfer_sm100.so -- the C-ABI boundary (include/cbinfer_b200.h).

Mirrors what the reference does with cffi at import time (pycbinfer/conv2d_cg.py:40-50,
pycbinfer/conv2d_fg.py:30-32) but for ONE sm_100a library, with status codes turned into
exceptions.  There is no CPU fallback and no other backend: if the library cannot be loaded the
import fails loudly.
"""
import ctypes
import os

import torch

from . import build as _build

F32, F16, BF16 = 0, 1, 2
UPDATE_NONE, UPDATE_CHANGED, UPDATE_ALL = 0, 1, 2
GEMM_SIMT_F32, GEMM_TC, GEMM_TC_3X, GEMM_TC_BF16X3 = 0, 1, 2, 3
AUX_NONE, AUX_TF32_LO, AUX_BF16_PAIR = 0, 1, 2
RESET_FILL_ZERO, RESET_FILL_INF = 0, 1

_DTYPES = {torch.float32: F32, torch.float16: F16, torch.bfloat16: BF16}

# every symbol include/cbinfer_b200.h declares (tests check the library exports all of them)
SYMBOLS = [
    "cb_version", "cb_last_error", "cb_device_info", "cb_bitmap_row_words", "cb_bitmap_words",
    "cb_compact_ws_bytes", "cb_channel_pitch", "cb_plane_pitch16", "cb_packed_weight_bytes", "cb_change_detect", "cb_change_detect_u8",
    "cb_change_detect_streams", "cb_change_detect_u8_streams",
    "cb_dilate_compact", "cb_map_to_bits", "cb_change_detect_sparse", "cb_pool_compact", "cb_maxpool2x2_detect",
    "cb_pack_weights", "cb_conv_ws_bytes", "cb_conv_update", "cb_conv_update_masked", "cb_maxpool2x2",
    "cb_gen_xmatrix", "cb_matrix_mult", "cb_update_output", "cb_fg_update",
    "cb_fg_detect", "cb_conv_accumulate", "cb_compact_small_max_words", "cb_change_detect_sparse_compact",
    "cb_tile_ws_bytes", "cb_dilate_compact_tiles", "cb_conv_tiled_supported", "cb_conv_update_tiled",
    "cb_conv_tiled_pool_supported", "cb_conv_update_tiled_pool", "cb_dilate_tiles",
    "cb_tail_supported", "cb_tail_update", "cb_reset_streams",
    "cb_resize_ws_bytes", "cb_resize_bicubic_u8_init", "cb_resize_bicubic_u8", "cb_resize_bilinear_u8",
    "cb_dilate_compact_streams", "cb_dilate_compact_tiles_streams", "cb_dilate_tiles_streams",
    "cb_change_detect_sparse_compact_streams", "cb_conv_update_masked_streams", "cb_tail_update_streams",
    "cb_stream_bucket",
    "cb_change_detect_thr", "cb_change_detect_u8_thr", "cb_change_detect_sparse_thr",
    "cb_change_detect_sparse_compact_thr", "cb_maxpool2x2_detect_thr", "cb_conv_update_tiled_pool_thr",
    "cb_tail_update_thr",
    "cb_change_detect_zone", "cb_change_detect_u8_zone",
]


class ResetSegment(ctypes.Structure):
    """cb_reset_segment: one pixel-major buffer whose per-stream slices cb_reset_streams rewrites."""
    _fields_ = [("base", ctypes.c_void_p), ("pixels", ctypes.c_longlong), ("pitch_bytes", ctypes.c_int),
                ("channel_bytes", ctypes.c_int), ("dtype", ctypes.c_int), ("fill", ctypes.c_int)]


def _load():
    path = _build.LIB
    if _build.needs_build():
        try:
            path = _build.build()
        except Exception as e:  # no nvcc on this box and no prebuilt library: fail loudly
            if not os.path.exists(_build.LIB):
                raise ImportError(
                    "cbinfer_b200: libcbinfer_sm100.so is missing and could not be built (%s). "
                    "There is no CPU or fallback path." % (e,))
            path = _build.LIB
    path = os.environ.get("CBINFER_LIB", path)       # experiments: an alternative build of the library
    lib = ctypes.CDLL(path)
    vp, i32, i64, f32, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_size_t
    sig = {
        "cb_version": (i32, []),
        "cb_last_error": (ctypes.c_char_p, []),
        "cb_device_info": (i32, [vp, vp, vp]),
        "cb_bitmap_row_words": (i32, [i32]),
        "cb_bitmap_words": (sz, [i32, i32, i32]),
        "cb_compact_ws_bytes": (sz, [i32, i32, i32]),
        "cb_channel_pitch": (i32, [i32, i32]),
        "cb_plane_pitch16": (i32, [i32]),
        "cb_packed_weight_bytes": (sz, [i32] * 6),
        "cb_change_detect": (i32, [vp, i32, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32, vp, vp,
                                   vp, i32, i32, i32, i32, f32, i32]),
        "cb_change_detect_u8": (i32, [vp, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32, vp, vp, vp,
                                      i32, i32, i32, i32, f32, f32, f32, i32]),
        "cb_change_detect_streams": (i32, [vp, i32, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32, vp, vp,
                                           vp, i32, i32, i32, i32, f32, i32, vp]),
        "cb_change_detect_u8_streams": (i32, [vp, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32, vp, vp, vp,
                                              i32, i32, i32, i32, f32, f32, f32, i32, vp]),
        "cb_dilate_compact": (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32]),
        "cb_tile_ws_bytes": (sz, [i32, i32, i32]),
        "cb_dilate_compact_tiles": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32]),
        "cb_conv_tiled_supported": (i32, [i32] * 9),
        "cb_conv_update_tiled": (i32, [vp, i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32,
                                       i32, i32, i32, i32, i32]),
        "cb_tail_supported": (i32, [i32] * 5),
        "cb_tail_update": (i32, [vp, vp, vp, vp, vp, vp, i32, f32, vp, vp, vp, vp, i32, i32, f32, vp, vp, i32, i32, i32,
                                 i32, vp, vp, vp]),
        "cb_reset_streams": (i32, [vp, vp, i32, ctypes.POINTER(ResetSegment), i32]),
        "cb_dilate_tiles": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32]),
        "cb_conv_tiled_pool_supported": (i32, [i32, i32, i32]),
        "cb_conv_update_tiled_pool": (i32, [vp, i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32,
                                            i32, i32, i32, i32, i32,
                                            vp, i64, i64, i32, i32, i32, vp, i64, i64, i32, i32, vp, vp, vp, f32, i32]),
        "cb_resize_ws_bytes": (sz, [i32] * 5),
        "cb_resize_bicubic_u8_init": (i32, [vp, vp, i32, i32, i32, i32, i32]),
        "cb_resize_bicubic_u8": (i32, [vp, vp, i64, i64, i64, vp, i64, i64, i64, vp, i32, i32, i32, i32, i32]),
        "cb_resize_bilinear_u8": (i32, [vp, vp, i64, i64, i64, i32, i32, vp, i64, i64, i64, i32, i32, i32,
                                        f32, f32, f32, f32]),
        "cb_map_to_bits": (i32, [vp, vp, vp, i32, i32, i32]),
        "cb_change_detect_sparse": (i32, [vp, i32, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32,
                                          vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, i32, i32]),
        "cb_compact_small_max_words": (i32, []),
        "cb_change_detect_sparse_compact": (i32, [vp, i32, vp, i64, i64, i64, i64, vp, i64, i64, i64, i64, i32,
                                                  vp, vp, vp, vp, vp, i32, i32, i32, i32, f32, i32, i32,
                                                  vp, vp, vp, vp, i32, i32, i32]),
        "cb_pool_compact": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32]),
        "cb_pack_weights": (i32, [vp, i32, i32, vp, vp, i32, i32, i32, i32]),
        "cb_conv_ws_bytes": (sz, []),
        "cb_conv_update": (i32, [vp, i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32,
                                 i32, i32, i32, i32, i32, vp, sz]),
        "cb_conv_update_masked": (i32, [vp, i32, i32, vp, vp, i32, vp, vp, vp, vp, vp, i32, i32, i32, i32,
                                        i32, i32, i32, i32, i32, vp, sz, vp, i32, vp, vp]),
        "cb_maxpool2x2": (i32, [vp, i32, vp, i64, i64, i64, i64, vp, vp, vp, vp, i64, i64, i64,
                                i64, i32, i32, i32, i32, i32, i32]),
        "cb_maxpool2x2_detect": (i32, [vp, i32, vp, i64, i64, i32, vp, vp, vp, vp, i64, i64, i32,
                                       i32, i32, i32, i32, i32, i32, vp, i64, i64, i32, i32, vp, vp,
                                       vp, f32, i32]),
        "cb_gen_xmatrix": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, i32, i32, i32]),
        "cb_matrix_mult": (i32, [vp, i32, vp, vp, vp, vp, i32, i32, i32]),
        "cb_update_output": (i32, [vp, i32, vp, vp, vp, i32, i32, i32, i32]),
        "cb_fg_update": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, f32]),
        "cb_fg_detect": (i32, [vp, vp, i64, i64, i64, i64, vp, i64, i64, i32, vp, vp, vp, vp, i32, i32, i32,
                               i32, f32]),
        "cb_conv_accumulate": (i32, [vp, i32, i32, vp, vp, i32, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                     i32, i32, i32, vp, sz]),
    }
    # the *_streams variants: the plain call's arguments + one row of per-stream counts and its accumulator
    for name in ("cb_dilate_compact", "cb_dilate_compact_tiles", "cb_dilate_tiles", "cb_change_detect_sparse_compact",
                 "cb_conv_update_masked"):
        sig[name + "_streams"] = (i32, sig[name][1] + [vp, vp])
    sig["cb_tail_update_streams"] = (i32, sig["cb_tail_update"][1] + [i32, i32, vp, vp, vp, vp])
    sig["cb_stream_bucket"] = (i32, [vp, vp, vp, i32, i32, vp, vp])
    # the *_thr variants: the newest variant's arguments + the per-stream thresholds (one table per layer)
    for name in ("cb_change_detect_streams", "cb_change_detect_u8_streams", "cb_change_detect_sparse",
                 "cb_change_detect_sparse_compact_streams", "cb_maxpool2x2_detect", "cb_conv_update_tiled_pool",
                 "cb_tail_update_streams"):
        tables = 2 if name == "cb_tail_update_streams" else 1
        sig[name.replace("_streams", "") + "_thr"] = (i32, sig[name][1] + [vp] * tables)
    # the *_zone variants: the *_thr arguments + the watched-pixel zone bitmap
    for name in ("cb_change_detect_thr", "cb_change_detect_u8_thr"):
        sig[name.replace("_thr", "_zone")] = (i32, sig[name][1] + [vp])
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


C = _load()


class CBinferError(RuntimeError):
    pass


def check(status):
    if status != 0:
        raise CBinferError("libcbinfer_sm100: %s (status %d)" % (C.cb_last_error().decode(), status))


def dtype_code(t):
    try:
        return _DTYPES[t.dtype if isinstance(t, torch.Tensor) else t]
    except KeyError:
        raise TypeError("cbinfer_b200 supports float32, float16 and bfloat16 tensors, got %s" % (t,))


def require_cuda(*tensors):
    """The product path is CUDA-only (north star: no CPU fallback)."""
    for t in tensors:
        if not t.is_cuda:
            raise CBinferError("cbinfer_b200 has no CPU path: tensor on %s" % (t.device,))


def stream_ptr(device=None):
    return torch.cuda.current_stream(device).cuda_stream


def channel_pitch(dtype, C_):
    return C.cb_channel_pitch(dtype_code(dtype), C_)
