"""ctypes binding of libeod_memory.so (the C ABI declared in include/eod_memory.h).

There is NO CPU fallback: if the shared library is missing this module raises at import of the first
symbol, and every wrapper raises EodError on a non-zero return code.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_void_p

from .build import SO_PATH

EOD_OK = 0
ORDER_ZX, ORDER_XZ = 0, 1
LAYOUT_CHW, LAYOUT_HWC, LAYOUT_HWC_BF16, LAYOUT_HWC_F16, LAYOUT_CHW_BF16, LAYOUT_CHW_F16 = 0, 1, 2, 3, 4, 5
FUSE_SUM, FUSE_MEM_ONLY, FUSE_IMAGE_ONLY = 0, 1, 2
WRITE_AUTO, WRITE_LDG, WRITE_TMA, WRITE_TMA_DRY, WRITE_DET = 0, 1, 2, 3, 4

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/eod_memory.h one to one
_P = c_void_p
SIGNATURES = {
    "eod_version": [],
    "eod_last_error": [],
    "eod_backproject_quantize": [_P, _P, _P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_int,
                                 c_int, c_int, c_float, _P, _P, _P, _P, _P, _P],
    "eod_backproject_quantize_u16": [_P, c_double, _P, _P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_int,
                                     c_int, c_int, c_float, _P, _P, _P, _P, _P, _P],
    "eod_backproject_count": [_P, c_int, c_double, _P, _P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_int, c_int, c_int,
                              _P, _P, _P, _P],
    "eod_quantize_world": [_P, c_int64, c_float, c_float, c_float, c_int, c_int, c_int, _P, _P],
    "eod_sample_mask": [_P, c_int, c_int, c_int, _P, _P, _P],
    "eod_frame_count": [_P, _P, _P, c_int, c_int, c_int64, _P, _P, _P, _P, c_int, _P],
    "eod_expand_counts": [_P, _P, c_int, c_int, c_int64, _P, _P],
    "eod_write_mean": [_P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int64, _P, c_int, _P, _P, _P],
    "eod_write_mean_det_workspace_bytes": [c_int, c_int, c_int, c_int64, c_int],
    "eod_write_mean_det_status_offset": [c_int, c_int64],
    "eod_write_mean_det": [_P, _P, _P, _P, c_int, c_int, c_int, c_int64, _P, _P, c_int64, _P],
    "eod_write_mean_det_layout": [_P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int64, _P, _P, c_int64, _P],
    "eod_finalize_counts": [_P, c_int, c_int, c_int64, _P, _P, _P, _P, _P, c_int, _P],
    "eod_box_to_image_features": [_P, _P, c_int, c_int, c_int, _P, _P, _P],
    "eod_masks_observed": [_P, _P, c_int, c_int, c_int, _P, _P],
    "eod_write_objects": [_P, _P, _P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int, _P, _P],
    "eod_paste_masks": [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_float, _P, _P, _P],
    "eod_write_objects_pasted": [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P, _P, _P, c_int, c_int, c_int64, c_int, _P, _P],
    "eod_write_objects_det": [_P, _P, _P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int64, _P, _P, c_int64, _P],
    "eod_write_objects_pasted_det": [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P, _P, _P, c_int, c_int, c_int64, _P, _P, c_int64, _P],
    "eod_flush_slots": [_P, _P, _P, _P, c_int, c_int, c_int64, c_int, _P, _P, _P],
    "eod_bilinear_lattice": [_P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "eod_write_max": [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int64, _P, _P, _P, _P, _P, _P],
    "eod_max_winner_list": [_P, c_int, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P],
    "eod_heightmax_contest_depth": [_P, c_int, c_double, _P, _P, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_float, c_int, c_int,
                                    c_int, c_float, c_int, _P, _P, _P, c_int64, _P, _P, _P],
    "eod_heightmax_contest_planes": [_P, _P, _P, c_int, c_int, c_int, c_int, c_int64, _P, _P, _P, c_int64, _P, _P, _P],
    "eod_heightmax_update": [_P, c_int, c_int, c_int, c_int, c_int, c_int64, _P, c_int64, _P, _P, _P, _P, _P, _P, _P, c_int64, _P, _P],
    "eod_heightmax_reset": [_P, c_int, c_int64, c_int, _P, _P, _P, _P],
    "eod_linear_rows": [_P, c_int64, c_int64, _P, _P, c_int64, c_int64, _P, c_float, c_int, _P, c_int, c_int, _P, c_int64, _P, _P],
    "eod_read_pool": [_P, c_int, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int64, _P, _P, _P, _P],
    "eod_normalize_memory": [_P, _P, c_int64, c_int, _P, c_int, _P],
    "eod_read_roi": [c_int, _P, _P, _P, _P, c_int, c_int, _P, _P, c_int, c_int, c_int, c_int, c_float, c_int, _P, _P, _P, _P],
    "eod_semmap_update": [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int64, _P, _P, _P],
    "eod_semmap_decode": [_P, _P, c_int, c_int64, c_float, _P, _P, _P],
    "eod_reset_touched": [_P, _P, _P, c_int64, c_int, _P],
    "eod_reset_episodes": [_P, _P, _P, _P, c_int, c_int64, c_int, _P],
    "eod_refresh_norm16": [_P, _P, _P, _P, c_int, c_int64, c_int, _P],
    "eod_check_indices": [_P, c_int, c_int64, c_int64, _P, _P, _P],
    "eod_remap_indices": [_P, c_int, c_int64, _P, c_int, c_int64, c_int, c_int64, _P, _P, _P],
    "eod_project_split_weights": [_P, c_int, c_int, _P, _P],
    "eod_project_fuse_levels": [c_int, _P, _P, _P, _P, _P, _P, c_float, c_int, c_int, c_int, c_int, c_int, _P],
    "eod_project_fuse": [_P, _P, _P, _P, c_float, c_int, c_int, c_int, c_int, c_int, _P, _P],
    "eod_fuse": [_P, _P, c_float, c_int, c_int64, _P, _P],
}
_RESTYPES = {"eod_last_error": c_char_p, "eod_write_mean_det_workspace_bytes": c_int64, "eod_write_mean_det_status_offset": c_int64}


class EodError(RuntimeError):
    pass


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise EodError(f"{SO_PATH} is missing: build it with `python -m __graft_entry__` or "
                           f"`python embodied-object-detection_b200/build.py` (there is no CPU fallback)")
        handle = ctypes.CDLL(SO_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(handle, name)          # AttributeError here == header/library mismatch
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, c_int)
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != EOD_OK:
        msg = lib().eod_last_error()
        raise EodError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")
