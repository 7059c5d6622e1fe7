"""ctypes binding of libgnc.so (include/gnc.h).  No fallback: if the CUDA library is
missing or fails, this raises - the product path never computes on the CPU."""
from __future__ import annotations

import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint8, c_uint16, c_uint64,
                    c_void_p)

# GNC_LIB: kernel-development hook (scripts/chain_ab.py loads alternative builds of the same library side by side)
_LIB_PATH = os.environ.get("GNC_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libgnc.so")

GNC_OK, GNC_EINVAL, GNC_ECUDA, GNC_EWORKSPACE, GNC_JPEG_UNSUPPORTED = 0, 1, 2, 3, 4


class GncSeg(Structure):
    """struct gnc_seg (include/gnc.h)."""
    _fields_ = [("base", c_void_p), ("idx", c_void_p), ("ld", c_int64), ("width", c_int32), ("_pad", c_int32)]


class GncTcEpilogue(Structure):
    """struct gnc_tc_epilogue (include/gnc.h)."""
    _fields_ = [("bias", c_void_p),
                ("addend", c_void_p), ("ld_addend", c_int64),
                ("gather0", c_void_p), ("gather0_idx", c_void_p), ("ld_gather0", c_int64),
                ("gather1", c_void_p), ("gather1_idx", c_void_p), ("ld_gather1", c_int64),
                ("relu", c_int32), ("_pad0", c_int32),
                ("gamma", c_void_p), ("beta", c_void_p), ("eps", c_float), ("_pad1", c_int32),
                ("residual", c_void_p), ("ld_residual", c_int64),
                ("dot_w", c_void_p), ("dot_b", c_void_p),
                ("mask", c_void_p), ("ld_mask", c_int64),
                ("residual_idx", c_void_p),
                ("ln_z", c_void_p), ("ld_ln_z", c_int64), ("ln_mean", c_void_p), ("ln_rstd", c_void_p)]


class GncTcChain(Structure):
    """struct gnc_tc_chain (include/gnc.h)."""
    _fields_ = [("nlayers", c_int32), ("_pad0", c_int32),
                ("W", c_void_p * 3), ("ldw", c_int64 * 3), ("bias", c_void_p * 3),
                ("gather0", c_void_p), ("gather0_idx", c_void_p), ("ld_gather0", c_int64),
                ("gather1", c_void_p), ("gather1_idx", c_void_p), ("ld_gather1", c_int64),
                ("gamma", c_void_p), ("beta", c_void_p), ("eps", c_float), ("_pad1", c_int32),
                ("residual", c_void_p), ("residual_idx", c_void_p), ("ld_residual", c_int64),
                ("dot_w", c_void_p), ("dot_b", c_void_p),
                ("gather2", c_void_p), ("gather2_idx", c_void_p), ("ld_gather2", c_int64), ("pre_bias", c_void_p),
                ("operand2", c_void_p), ("ld_operand2", c_int64), ("W_operand2", c_void_p), ("ldw_operand2", c_int64),
                ("narrow_W", c_void_p), ("ld_narrow_W", c_int64), ("narrow_b", c_void_p), ("narrow_k", c_int32), ("_pad2", c_int32),
                ("stash_a1", c_void_p), ("stash_a2", c_void_p), ("stash_z", c_void_p), ("ld_stash", c_int64),
                ("stash_mean", c_void_p), ("stash_rstd", c_void_p),
                ("agg_rowptr", c_void_p), ("agg_eid", c_void_p),
                ("edge_slots", c_int32), ("paired_operand", c_int32)]


class GncBwdReduceItem(Structure):
    """struct gnc_bwd_reduce_item (include/gnc.h)."""
    _fields_ = [("work", c_void_p), ("dW", c_void_p), ("db", c_void_p), ("lddw", c_int64), ("parts", c_int32),
                ("accumulate", c_int32)]


class GncJpegHuff(Structure):
    """struct gnc_jpeg_huff (include/gnc.h)."""
    _fields_ = [("look", c_uint16 * 512), ("maxcode", c_int32 * 18), ("valoff", c_int32 * 17), ("vals", c_uint8 * 256)]


class GncJpegImage(Structure):
    """struct gnc_jpeg_image (include/gnc.h)."""
    _fields_ = [("width", c_int32), ("height", c_int32), ("ncomp", c_int32),
                ("hsamp", c_int32 * 3), ("vsamp", c_int32 * 3), ("qtab", c_int32 * 3), ("dc_tab", c_int32 * 3),
                ("ac_tab", c_int32 * 3),
                ("restart_interval", c_int32), ("mcu_x", c_int32), ("mcu_y", c_int32), ("_pad", c_int32),
                ("scan_offset", c_int64), ("scan_bytes", c_int64), ("n_blocks", c_int64), ("plane_bytes", c_int64),
                ("block_offset", c_int64), ("coef_offset", c_int64), ("plane_offset", c_int64), ("pixel_offset", c_int64),
                ("quant", (c_uint16 * 64) * 4), ("huff", GncJpegHuff * 8)]


class GncJpegScan(Structure):
    """struct gnc_jpeg_scan (include/gnc.h)."""
    _fields_ = [("image", c_int32), ("ncomp", c_int32), ("comp", c_int32 * 3), ("dc_tab", c_int32 * 3), ("ac_tab", c_int32),
                ("Ss", c_int32), ("Se", c_int32), ("Ah", c_int32), ("Al", c_int32), ("restart_interval", c_int32),
                ("offset", c_int64), ("bytes", c_int64)]


class GncJpegChain(Structure):
    """struct gnc_jpeg_chain (include/gnc.h)."""
    _fields_ = [("first_scan", c_int32), ("n_scans", c_int32), ("bytes", c_int64)]


GNC_JPEG_MAX_SCANS, GNC_JPEG_MAX_TABLES = 64, 32

GNC_UNSUPPORTED = GNC_JPEG_UNSUPPORTED
GNC_PNG_MAX_RAW_BYTES = 2 << 20


class GncPngImage(Structure):
    """struct gnc_png_image (include/gnc.h)."""
    _fields_ = [("width", c_int32), ("height", c_int32), ("color_type", c_int32), ("bit_depth", c_int32),
                ("row_bytes", c_int32), ("bpp", c_int32), ("window", c_int32), ("_pad", c_int32),
                ("stream_offset", c_int64), ("stream_bytes", c_int64), ("raw_offset", c_int64), ("raw_bytes", c_int64),
                ("pixel_offset", c_int64), ("palette", (c_uint8 * 3) * 256)]


class GncResizeImage(Structure):
    """struct gnc_resize_image (include/gnc.h)."""
    _fields_ = [("src", c_void_p), ("pitch", c_int64), ("tmp_row", c_int64), ("tab_x", c_int64), ("tab_y", c_int64),
                ("height", c_int32), ("width", c_int32), ("ksize_x", c_int32), ("ksize_y", c_int32)]


class GncError(RuntimeError):
    pass


_P = c_void_p
# name -> (restype, argtypes); mirrors include/gnc.h one to one (tests/test_abi.py checks it)
SIGNATURES = {
    "gnc_version": (c_int, []),
    "gnc_last_error": (c_char_p, []),
    "gnc_launch_count": (c_uint64, []),
    "gnc_reset_launch_count": (None, []),
    "gnc_grid_num_edges": (c_int64, [c_int, c_int, c_int]),
    "gnc_build_pixel_graph_u8": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gnc_build_patch_graph_u8": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gnc_superpixel_workspace": (c_int64, [c_int, c_int]),
    "gnc_build_superpixel_graph": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int64,
                                           _P, _P, _P, _P, _P, _P, _P, _P]),
    "gnc_slic_num_centers": (c_int, [c_int, c_int, c_int]),
    "gnc_slic_workspace_bytes": (c_int64, [c_int, c_int, c_int, c_int]),
    "gnc_slic_labels_u8": (c_int, [_P, c_int, c_int, c_int, c_int, c_float, c_int, _P, _P, _P]),
    "gnc_resize_bicubic_ksize": (c_int, [c_int, c_int]),
    "gnc_resize_bicubic_coeffs": (c_int, [c_int, c_int, _P, _P]),
    "gnc_resize_bicubic_u8": (c_int, [_P, c_int64, c_int, c_int, c_int64, c_int64, c_int, c_int, _P, _P, c_int, _P, _P, c_int,
                                      _P, _P, _P]),
    "gnc_resize_bicubic_ragged_u8": (c_int, [_P, c_int64, c_int, c_int, c_int64, c_int, _P, _P, _P, _P]),
    "gnc_csr_workspace": (c_int64, [c_int64]),
    "gnc_csr_build": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P]),
    "gnc_agg_csr_sum_f32": (c_int, [_P, _P, _P, c_int64, c_int64, c_int, _P, c_int64, c_int, _P]),
    "gnc_agg_csr_sum_pair_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int, c_int64, _P]),
    "gnc_gather_rows_f32": (c_int, [_P, c_int64, _P, c_int64, c_int, _P, c_int64, c_int, _P]),
    "gnc_gather_add_rows_f32": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int, _P, c_int, c_int64,
                                        c_int, _P, c_int64, _P]),
    "gnc_grid_edge_class": (c_int, [c_int, c_int, c_int, c_int, _P, _P]),
    "gnc_grid_pair_slots": (c_int, [c_int, c_int, c_int, _P, _P, _P, _P]),
    "gnc_edge_geometry_f32": (c_int, [_P, c_int, _P, _P, c_int64, _P, _P]),
    "gnc_linear_fwd_f32": (c_int, [POINTER(GncSeg), c_int, c_int64, _P, c_int64, _P, c_int, c_int, _P, c_int64, _P]),
    "gnc_linear_fwd_splitk_workspace": (c_int64, [c_int64, c_int, c_int64]),
    "gnc_linear_fwd_splitk_f32": (c_int, [POINTER(GncSeg), c_int, c_int64, _P, c_int64, _P, c_int, c_int, _P, c_int64,
                                          _P, c_int64, _P]),
    "gnc_linear_narrowk_fwd_f32": (c_int, [_P, c_int64, c_int64, c_int, _P, c_int64, _P, c_int, c_int, _P, c_int64, _P]),
    "gnc_linear_narrowk_wgrad_workspace": (c_int64, [c_int64, c_int, c_int]),
    "gnc_linear_narrowk_wgrad_f32": (c_int, [_P, c_int64, _P, c_int64, _P, c_int64, c_int64, c_int, c_int, _P, c_int64,
                                             _P, c_int, _P, c_int64, _P]),
    "gnc_linear_dgrad_f32": (c_int, [_P, c_int64, c_int64, c_int, _P, c_int64, c_int, _P, c_int64, c_int, _P]),
    "gnc_linear_wgrad_workspace": (c_int64, [c_int64, c_int, c_int]),
    "gnc_linear_wgrad_f32": (c_int, [_P, c_int64, c_int64, c_int, POINTER(GncSeg), c_int, _P, c_int64, c_int,
                                     _P, c_int64, _P]),
    "gnc_colsum_workspace": (c_int64, [c_int64, c_int]),
    "gnc_relu_bwd_colsum_f32": (c_int, [_P, c_int64, _P, c_int64, c_int64, c_int, _P, c_int64, _P, c_int,
                                        _P, c_int64, _P]),
    "gnc_layernorm_fwd_f32": (c_int, [_P, c_int64, c_int64, c_int, _P, _P, c_float, _P, c_int64, _P, c_int64,
                                      _P, _P, _P]),
    "gnc_layernorm_bwd_workspace": (c_int64, [c_int64, c_int]),
    "gnc_layernorm_bwd_f32": (c_int, [_P, c_int64, _P, c_int64, _P, _P, _P, c_int64, c_int, _P, c_int64,
                                      _P, _P, c_int, _P, c_int64, _P]),
    "gnc_tc_linear_f32": (c_int, [_P, c_int64, c_int64, c_int, _P, c_int64, c_int, c_int, POINTER(GncTcEpilogue),
                                  _P, c_int64, _P]),
    "gnc_tc_linear_multi_f32": (c_int, [_P, c_int64, c_int64, c_int, POINTER(c_void_p), POINTER(c_int64), POINTER(c_void_p),
                                        c_int64, _P]),
    "gnc_tc_mlp_chain_f32": (c_int, [_P, c_int64, c_int64, POINTER(GncTcChain), _P, c_int64, _P]),
    "gnc_tc_multi_chain_f32": (c_int, [_P, c_int64, c_int64, c_int, POINTER(c_void_p), POINTER(c_int64), POINTER(c_void_p),
                                       POINTER(c_void_p), c_int64, _P]),
    "gnc_debug_chain_trace": (c_int, [_P, c_int]),
    "gnc_debug_slic_run_length": (c_int, [c_int]),
    "gnc_tc_wgrad_workspace": (c_int64, [c_int64]),
    "gnc_tc_wgrad_f32": (c_int, [_P, c_int64, _P, c_int64, c_int64, c_int, c_int, _P, c_int64, c_int, _P, _P, c_int64,
                                 _P]),
    "gnc_dot_tail_fwd_f32": (c_int, [_P, c_int64, c_int64, c_int, _P, _P, _P, _P]),
    "gnc_dot_tail_bwd_workspace": (c_int64, [c_int64, c_int]),
    "gnc_dot_tail_bwd_f32": (c_int, [_P, c_int64, c_int64, c_int, _P, _P, c_int, _P, c_int64, _P, _P, c_int, _P, c_int64, _P]),
    "gnc_slic_connectivity_workspace": (c_int64, [c_int, c_int, c_int]),
    "gnc_slic_enforce_connectivity": (c_int, [_P, c_int, c_int, c_int, c_int, _P, _P, _P, c_int64, _P]),
    "gnc_segment_readout_f32": (c_int, [_P, _P, c_int, c_int, _P, _P]),
    "gnc_segment_readout_bwd_f32": (c_int, [_P, _P, c_int, c_int, _P, _P]),
    "gnc_cross_entropy_f32": (c_int, [_P, c_int64, _P, c_int, c_int, c_float, _P, _P, _P, c_int64, _P, _P]),
    "gnc_adam_step_f32": (c_int, [_P, _P, _P, _P, c_int64, c_double, c_double, c_double, c_double, c_int64, c_float, _P]),
    "gnc_zero_f32": (c_int, [_P, c_int64, _P]),
    "gnc_tc_bwd_layer_workspace": (c_int64, []),
    "gnc_tc_bwd_layer_f32": (c_int, [_P, c_int64, _P, c_int64, c_int64, _P, c_int64, c_int, _P, c_int64, _P, c_int64,
                                     _P, c_int64, _P, c_int, _P, c_int64, _P]),
    "gnc_debug_slic_connect_streaming": (c_int, [c_int]),
    "gnc_superpixel_batch_offsets": (c_int, [_P, _P, c_int, c_int, c_int64, _P, _P, _P]),
    "gnc_superpixel_batch_compact": (c_int, [_P, _P, _P, c_int, c_int, c_int64, _P, _P, _P, _P, _P, c_int64, _P]),
    "gnc_superpixel_batch_padded": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int64, _P, _P,
                                            _P, _P, _P, _P, _P]),
    "gnc_jpeg_parse": (c_int, [_P, c_int64, POINTER(GncJpegImage)]),
    "gnc_jpeg_pack": (c_int, [_P, _P, c_int, c_int, _P, c_int64, _P, _P, _P]),
    "gnc_jpeg_scratch_bytes": (c_int64, [c_int64, c_int]),
    "gnc_jpeg_decode_rgb_u8": (c_int, [_P, _P, c_int, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "gnc_debug_jpeg_sequential": (c_int, [c_int]),
    "gnc_jpeg_pack_progressive": (c_int, [_P, _P, c_int, c_int, _P, c_int64, _P, _P, _P, c_int64, _P, c_int64, _P, c_int64,
                                          _P]),
    "gnc_jpeg_decode_progressive_rgb_u8": (c_int, [_P, _P, c_int, _P, _P, c_int, _P, c_int64, c_int64, _P, _P, _P, _P]),
    "gnc_debug_jpeg_chains_per_warp": (c_int, [c_int]),
    "gnc_png_pack": (c_int, [_P, _P, c_int, c_int, _P, c_int64, _P, _P, _P]),
    "gnc_png_decode_rgb_u8": (c_int, [_P, _P, c_int, _P, _P, _P, _P]),
    "gnc_tc_bwd_layer_parts": (c_int32, [c_int64]),
    "gnc_tc_bwd_reduce_batch_f32": (c_int, [POINTER(GncBwdReduceItem), c_int32, _P]),
}

_lib = None


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Loads libgnc.so; raises GncError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise GncError(
            f"{_LIB_PATH} not found: build it with `python -m graphnet_classifier_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU fallback for this path.")
    lib = ctypes.CDLL(_LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != GNC_OK:
        msg = load().gnc_last_error()
        raise GncError(f"libgnc {what} failed (code {rc}): {msg.decode() if msg else ''}")


def launch_count() -> int:
    return int(load().gnc_launch_count())


def reset_launch_count() -> None:
    load().gnc_reset_launch_count()
