"""Torch-tensor front end of the C ABI: validates shapes/dtypes/devices, passes raw device pointers and the
current CUDA stream to libeod_memory.so.  torch is used for device memory and streams only; every op
here runs a hand-written kernel (no torch compute, no CPU fallback: CPU tensors raise).
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import (FUSE_IMAGE_ONLY, FUSE_MEM_ONLY, FUSE_SUM, LAYOUT_CHW, LAYOUT_CHW_BF16, LAYOUT_CHW_F16, LAYOUT_HWC, LAYOUT_HWC_BF16, LAYOUT_HWC_F16,
                   ORDER_XZ, ORDER_ZX, WRITE_AUTO, WRITE_DET, WRITE_LDG, WRITE_TMA, EodError, check)

# feature dtype of each layout of the mean write (every layout not listed takes fp32)
LAYOUT_DTYPE = {LAYOUT_HWC_BF16: torch.bfloat16, LAYOUT_HWC_F16: torch.float16, LAYOUT_CHW_BF16: torch.bfloat16, LAYOUT_CHW_F16: torch.float16}
# the layout that takes features of a given dtype in the same memory order as an fp32 layout
_LAYOUT_16 = {(LAYOUT_CHW, torch.bfloat16): LAYOUT_CHW_BF16, (LAYOUT_CHW, torch.float16): LAYOUT_CHW_F16,
              (LAYOUT_HWC, torch.bfloat16): LAYOUT_HWC_BF16, (LAYOUT_HWC, torch.float16): LAYOUT_HWC_F16}


def layout_for_dtype(layout: int, dtype: torch.dtype) -> int:
    """The 16-bit variant of an fp32 layout for bf16 / fp16 features; ``layout`` itself for any other dtype."""
    return _LAYOUT_16.get((int(layout), dtype), int(layout))

# kernels launched through this module since import (bench.py reports it as gpu_launches)
launch_count = 0

_LAUNCHES = {"eod_backproject_quantize": 1, "eod_backproject_quantize_u16": 1, "eod_backproject_count": 1, "eod_quantize_world": 1, "eod_sample_mask": 1, "eod_frame_count": 1, "eod_expand_counts": 1, "eod_write_mean": 1, "eod_write_mean_det": 9,
             "eod_write_mean_det_layout": 9,
             "eod_finalize_counts": 1, "eod_box_to_image_features": 1, "eod_masks_observed": 1, "eod_paste_masks": 1, "eod_write_objects_pasted": 1, "eod_bilinear_lattice": 1, "eod_write_objects": 1, "eod_write_objects_det": 9, "eod_write_objects_pasted_det": 9, "eod_flush_slots": 2, "eod_write_max": 2, "eod_read_pool": 2,
             "eod_fuse": 1, "eod_project_split_weights": 1, "eod_project_fuse": 1, "eod_project_fuse_levels": 1, "eod_normalize_memory": 1, "eod_reset_touched": 1, "eod_semmap_update": 1, "eod_semmap_decode": 2,
             "eod_reset_episodes": 1, "eod_refresh_norm16": 1, "eod_check_indices": 1, "eod_remap_indices": 1, "eod_max_winner_list": 1, "eod_linear_rows": 1, "eod_read_roi": 1,
             "eod_heightmax_contest_depth": 1, "eod_heightmax_contest_planes": 1, "eod_heightmax_update": 1, "eod_heightmax_reset": 1}


def _call(name: str, *args) -> None:
    global launch_count
    check(getattr(_lib.lib(), name)(*args), name)
    launch_count += _LAUNCHES[name]


def _dev(t: torch.Tensor, dtype: torch.dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise EodError(f"{name}: tensor is on {t.device}; the spatial memory runs on CUDA only (no CPU fallback)")
    if t.device.index != torch.cuda.current_device():
        raise EodError(f"{name}: tensor is on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()} "
                       f"(kernels launch on the current device: wrap the call in torch.cuda.device(...))")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(ref: Optional[torch.Tensor] = None) -> int:
    """The current stream of the device the operands live on.  The library launches on the CUDA context's current device, so
    a tensor on another device than torch's current one is an error (wrap the call in ``torch.cuda.device(t.device)``)."""
    if ref is not None and ref.device.index is not None and ref.device.index != torch.cuda.current_device():
        raise EodError(f"operands live on {ref.device} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                       f"wrap the call in torch.cuda.device({str(ref.device)!r})")
    return torch.cuda.current_stream().cuda_stream


def backproject_quantize(depth: torch.Tensor, pose: torch.Tensor, shifts: torch.Tensor, intr: Sequence[float], cell: float,
                         map_w: int, map_h: int, order: int = ORDER_ZX, z_clip: float = 0.5, *, want_idx: bool = True,
                         want_q2: bool = False, want_outlier: bool = False, want_height: bool = False,
                         want_world: bool = False, out: Optional[dict] = None, depth_div: float = 1000.0) -> dict:
    """depth (E,H,W) f32 metres - or uint16 sensor units, divided by ``depth_div`` in the kernel as robot_demo.py:515-517 does on
    the host - pose (E,12) f32, shifts (E,6) f32 -> dict(idx, q2, outlier, height, world)."""
    raw = depth.dtype == torch.uint16
    _dev(depth, torch.uint16 if raw else torch.float32, "depth"), _dev(pose, torch.float32, "pose"), _dev(shifts, torch.float32, "shifts")
    E, H, W = depth.shape
    if pose.shape != (E, 12) or shifts.shape != (E, 6):
        raise ValueError("pose must be (E,12) and shifts (E,6)")
    out = {} if out is None else out
    dev = depth.device

    def buf(key, want, shape, dtype):
        if not want:
            return None
        if key not in out:
            out[key] = torch.empty(shape, dtype=dtype, device=dev)
        return _dev(out[key], dtype, key)

    idx = buf("idx", want_idx, (E, H, W), torch.int32)
    q2 = buf("q2", want_q2, (E, H, W, 2), torch.int32)
    outlier = buf("outlier", want_outlier, (E, H, W), torch.uint8)
    height = buf("height", want_height, (E, H, W), torch.float32)
    world = buf("world", want_world, (E, H, W, 3), torch.float32)
    fx, fy, cx, cy = (float(v) for v in intr)
    tail = (pose.data_ptr(), shifts.data_ptr(), E, H, W, fx, fy, cx, cy, float(cell), int(map_w), int(map_h), int(order), float(z_clip),
            _ptr(idx), _ptr(q2), _ptr(outlier), _ptr(height), _ptr(world), _stream())
    if raw:
        _call("eod_backproject_quantize_u16", depth.data_ptr(), float(depth_div), *tail)
    else:
        _call("eod_backproject_quantize", depth.data_ptr(), *tail)
    return out


def backproject_count_supported(H: int, W: int) -> bool:
    return W % 4 == 0 and (H * W) % 128 == 0


def backproject_count(depth: torch.Tensor, pose: torch.Tensor, shifts: torch.Tensor, intr: Sequence[float], cell: float, map_w: int, map_h: int,
                      idx: torch.Tensor, frame_cnt: torch.Tensor, active: Optional[torch.Tensor] = None, order: int = ORDER_ZX,
                      depth_div: float = 1000.0) -> None:
    """Back-projection to cell ids (idx (E,H,W) i32) AND the frame's per-cell pixel counts (frame_cnt (E,cells) i32, accumulated) in one
    launch - eod_backproject_quantize + eod_frame_count(samp=None) of a dense frame-step.  depth f32 or uint16 (/ depth_div)."""
    raw = depth.dtype == torch.uint16
    _dev(depth, torch.uint16 if raw else torch.float32, "depth"), _dev(pose, torch.float32, "pose"), _dev(shifts, torch.float32, "shifts")
    _dev(idx, torch.int32, "idx"), _dev(frame_cnt, torch.int32, "frame_cnt")
    E, H, W = depth.shape
    if pose.shape != (E, 12) or shifts.shape != (E, 6) or tuple(idx.shape) != (E, H, W) or tuple(frame_cnt.shape) != (E, map_w * map_h):
        raise ValueError("backproject_count: pose (E,12), shifts (E,6), idx (E,H,W), frame_cnt (E, map_w*map_h)")
    if active is not None:
        _dev(active, torch.int32, "active")
    fx, fy, cx, cy = (float(v) for v in intr)
    _call("eod_backproject_count", depth.data_ptr(), int(raw), float(depth_div), pose.data_ptr(), shifts.data_ptr(), E, H, W, fx, fy, cx, cy,
          float(cell), int(map_w), int(map_h), int(order), _ptr(active), idx.data_ptr(), frame_cnt.data_ptr(), _stream())


def quantize_world(world: torch.Tensor, map_world_shift: Sequence[float], cell: float, map_w: int, map_h: int,
                   order: int = ORDER_ZX) -> torch.Tensor:
    """world (..., 3) f32 (sensor_data 'projection_indices') -> (..., 1) int32 proj_indices (build_memory_data.py:135-144)."""
    _dev(world, torch.float32, "world")
    if world.shape[-1] != 3:
        raise ValueError("world must be (..., 3)")
    out = torch.empty(world.shape[:-1] + (1,), dtype=torch.int32, device=world.device)
    _call("eod_quantize_world", world.data_ptr(), world.numel() // 3, float(map_world_shift[0]), float(map_world_shift[2]), float(cell),
          int(map_w), int(map_h), int(order), out.data_ptr(), _stream())
    return out


def sample_mask(observed: torch.Tensor, stride: int, samp: Optional[torch.Tensor] = None,
                n_sampled: Optional[torch.Tensor] = None) -> torch.Tensor:
    """observed (E,HW) u8 -> samp (E,HW) u8: every stride-th observed pixel in raster order."""
    _dev(observed, torch.uint8, "observed")
    E, HW = observed.shape
    samp = torch.empty_like(observed) if samp is None else _dev(samp, torch.uint8, "samp")
    _call("eod_sample_mask", observed.data_ptr(), E, HW, int(stride), samp.data_ptr(), _ptr(n_sampled), _stream())
    return samp


def frame_count(idx: torch.Tensor, samp: Optional[torch.Tensor], frame_cnt: torch.Tensor,
                active: Optional[torch.Tensor] = None, slots: Optional["ObjectSlots"] = None) -> None:
    """idx (E,HW) i32, samp (E,HW) u8 | None, frame_cnt (E,cells) i32 scratch (zero on entry);
    active (E) i32 | None: episodes with active <= 0 are skipped (no kept detection -> no write, no visibility);
    slots: when given, every cell that receives samples claims a compact slot (object-regime write)."""
    _dev(idx, torch.int32, "idx"), _dev(frame_cnt, torch.int32, "frame_cnt")
    E, HW = idx.shape[0], idx[0].numel()
    if samp is not None:
        _dev(samp, torch.uint8, "samp")
    if active is not None:
        _dev(active, torch.int32, "active")
    sl = (None, None, None, 0) if slots is None else (slots.slot_of_cell.data_ptr(), slots.slot_cell.data_ptr(), slots.n_slots.data_ptr(), slots.S)
    _call("eod_frame_count", idx.data_ptr(), _ptr(samp), _ptr(active), E, HW, frame_cnt.shape[1], frame_cnt.data_ptr(), *sl, _stream())


class ObjectSlots:
    """Per-frame workspace of the fused object write: a compact slot per touched cell and one zeroed fp32 row per slot
    (all of it is back to zero after flush_slots).  S = ceil(HW / sample_stride) slots always suffice."""

    def __init__(self, n_episodes: int, n_cells: int, channels: int, n_slots_max: int, device: torch.device):
        self.E, self.n_cells, self.C, self.S = n_episodes, n_cells, channels, int(n_slots_max)
        self.slot_of_cell = torch.zeros((n_episodes, n_cells), dtype=torch.int32, device=device)
        self.slot_cell = torch.zeros((n_episodes, self.S), dtype=torch.int32, device=device)
        self.n_slots = torch.zeros((n_episodes,), dtype=torch.int32, device=device)
        self.scratch = torch.zeros((n_episodes, self.S, channels), dtype=torch.float32, device=device)


def expand_counts(idx: torch.Tensor, frame_cnt: torch.Tensor, pix_inv_n: torch.Tensor) -> torch.Tensor:
    """pix_inv_n (E,HW) f32 := 1 / frame_cnt[idx] (after frame_count); feeds write_mean."""
    _dev(idx, torch.int32, "idx"), _dev(frame_cnt, torch.int32, "frame_cnt"), _dev(pix_inv_n, torch.float32, "pix_inv_n")
    E, HW = idx.shape[0], idx[0].numel()
    if pix_inv_n.numel() < E * HW:
        raise ValueError("pix_inv_n must hold E*HW floats")
    _call("eod_expand_counts", idx.data_ptr(), frame_cnt.data_ptr(), E, HW, frame_cnt[0].numel(), pix_inv_n.data_ptr(), _stream())
    return pix_inv_n


def write_mean(feat: torch.Tensor, idx: torch.Tensor, samp: Optional[torch.Tensor], frame_cnt: torch.Tensor,
               sums: torch.Tensor, layout: int = LAYOUT_CHW, variant: int = WRITE_AUTO,
               pix_inv_n: Optional[torch.Tensor] = None, active: Optional[torch.Tensor] = None) -> None:
    """feat (E,C,HW) [CHW] or (E,HW,C) [HWC] f32, (E,HW,C) bf16 / fp16 [LAYOUT_HWC_BF16 / _F16] or (E,C,HW) bf16 / fp16
    [LAYOUT_CHW_BF16 / _F16: widened exactly, fp32 arithmetic; HW % 8 == 0, no pix_inv_n]; sums (E,cells,C) f32 accumulated in
    place.  pix_inv_n: output of expand_counts for this frame (fp32 CHW only).
    active (E) i32 | None: slots with active <= 0 are skipped (give frame_count the same mask)."""
    feat_dtype = LAYOUT_DTYPE.get(int(layout), torch.float32)
    _dev(feat, feat_dtype, "feat"), _dev(idx, torch.int32, "idx"), _dev(sums, torch.float32, "sums")
    _dev(frame_cnt, torch.int32, "frame_cnt")
    E, n_cells, C = sums.shape
    HW = idx[0].numel()
    if feat.numel() != E * C * HW:
        raise ValueError(f"feat has {feat.numel()} elements, expected E*C*HW = {E * C * HW}")
    if samp is not None:
        _dev(samp, torch.uint8, "samp")
    if pix_inv_n is not None:
        _dev(pix_inv_n, torch.float32, "pix_inv_n")
        if pix_inv_n.numel() < E * HW:
            raise ValueError("pix_inv_n must hold E*HW floats")
    if active is not None:
        _dev(active, torch.int32, "active")
        if active.numel() != E:
            raise ValueError("active must hold one int32 per episode")
    _call("eod_write_mean", feat.data_ptr(), int(layout), idx.data_ptr(), _ptr(samp), frame_cnt.data_ptr(), E, C, HW,
          n_cells, sums.data_ptr(), int(variant), _ptr(pix_inv_n), _ptr(active), _stream())


def semmap_update(frame_cnt: torch.Tensor, counts: torch.Tensor, sums: torch.Tensor, zs_weight: torch.Tensor, n_cls: int,
                  intensity: torch.Tensor, cls: torch.Tensor) -> None:
    """Refresh intensity / class of the cells visible in the current frame (call between the write and finalize_counts).
    zs_weight (C, K>=n_cls) f32 as the reference holds it; intensity (E,cells) f32, cls (E,cells) i32."""
    _dev(frame_cnt, torch.int32, "frame_cnt"), _dev(counts, torch.float32, "counts"), _dev(sums, torch.float32, "sums")
    _dev(zs_weight, torch.float32, "zs_weight"), _dev(intensity, torch.float32, "intensity"), _dev(cls, torch.int32, "cls")
    E, n_cells, C = sums.shape
    if zs_weight.shape[0] != C or zs_weight.shape[1] < n_cls:
        raise ValueError("zs_weight must be (C, K) with K >= n_cls")
    _call("eod_semmap_update", frame_cnt.data_ptr(), counts.data_ptr(), sums.data_ptr(), zs_weight.data_ptr(), zs_weight.shape[1],
          int(n_cls), E, C, n_cells, intensity.data_ptr(), cls.data_ptr(), _stream())


def semmap_decode(intensity: torch.Tensor, cls: torch.Tensor, thresh: float, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(E,cells) int32 explicit map: class id, or -1 where the min-max normalised intensity is below thresh."""
    _dev(intensity, torch.float32, "intensity"), _dev(cls, torch.int32, "cls")
    E, n_cells = intensity.shape
    out = torch.empty((E, n_cells), dtype=torch.int32, device=intensity.device) if out is None else _dev(out, torch.int32, "semmap")
    ws = torch.empty((E, 2), dtype=torch.float32, device=intensity.device)
    _call("eod_semmap_decode", intensity.data_ptr(), cls.data_ptr(), E, n_cells, float(thresh), ws.data_ptr(), out.data_ptr(), _stream())
    return out


def reset_touched(counts: torch.Tensor, sums: torch.Tensor, norm16: Optional[torch.Tensor] = None) -> None:
    """memory_reset for library-maintained state: clears the rows of every cell with a non-zero count."""
    _dev(counts, torch.float32, "counts"), _dev(sums, torch.float32, "sums")
    if norm16 is not None:
        _dev(norm16, torch.float16, "norm16")
    C = sums.shape[-1]
    _call("eod_reset_touched", counts.data_ptr(), sums.data_ptr(), _ptr(norm16), counts.numel(), C, _stream())


def reset_episodes(counts: torch.Tensor, sums: torch.Tensor, norm16: Optional[torch.Tensor], mask: torch.Tensor) -> None:
    """Per-slot memory_reset: clears the touched rows of the episodes with mask[e] != 0.  counts (E,cells), sums (E,cells,C)."""
    _dev(counts, torch.float32, "counts"), _dev(sums, torch.float32, "sums"), _dev(mask, torch.int32, "mask")
    if norm16 is not None:
        _dev(norm16, torch.float16, "norm16")
    E, n_cells, C = sums.shape
    if mask.numel() != E:
        raise ValueError("mask must hold one int32 per episode")
    _call("eod_reset_episodes", counts.data_ptr(), sums.data_ptr(), _ptr(norm16), mask.data_ptr(), E, n_cells, C, _stream())


def refresh_norm16(counts: torch.Tensor, sums: torch.Tensor, norm16: torch.Tensor, mask: Optional[torch.Tensor] = None) -> None:
    """norm16[e] := half(sums / counts where counts > 1) for every touched cell of the episodes with mask[e] != 0 (None = all):
    the read table of TEST_TYPE longterm, refreshed at the first frame of a sequence (custom_rcnn.py:482-486)."""
    _dev(counts, torch.float32, "counts"), _dev(sums, torch.float32, "sums"), _dev(norm16, torch.float16, "norm16")
    E, n_cells, C = sums.shape
    if mask is not None:
        _dev(mask, torch.int32, "mask")
        if mask.numel() != E:
            raise ValueError("mask must hold one int32 per episode")
    _call("eod_refresh_norm16", counts.data_ptr(), sums.data_ptr(), norm16.data_ptr(), _ptr(mask), E, n_cells, C, _stream())


def check_indices(idx: torch.Tensor, n_cells: int, want_i32: bool = False) -> Optional[torch.Tensor]:
    """Range check of an externally supplied index plane (int32 / int64, any shape): raises IndexError - like the reference's
    gather does (timm.py:147) - if any id is outside [0, n_cells).  Synchronises (one 4-byte read-back).  want_i32: also return
    the plane as int32 (same shape)."""
    if idx.dtype not in (torch.int32, torch.int64):
        raise TypeError("idx must be int32 or int64")
    _dev(idx, idx.dtype, "idx")
    err = torch.zeros((1,), dtype=torch.int32, device=idx.device)
    out = torch.empty(idx.shape, dtype=torch.int32, device=idx.device) if want_i32 else None
    if idx.numel():
        _call("eod_check_indices", idx.data_ptr(), int(idx.dtype == torch.int64), idx.numel(), int(n_cells), _ptr(out), err.data_ptr(), _stream())
    bad = int(err.item())
    if bad:
        raise IndexError(f"{bad} cell indices are outside [0, {int(n_cells)}): proj_indices do not belong to this map")
    return out


def remap_indices(idx: torch.Tensor, lut: torch.Tensor, n_rows: int, add: int = 1) -> torch.Tensor:
    """explicit_map read mode (loader.py:233-246): int32 plane ``lut[idx] + add`` of the same shape as idx - the rows of the
    (n_rows, C) [zeros; class table] memory.  Raises IndexError, like the reference's numpy / torch gathers, if a cell id is outside
    the map or a class outside the table.  Synchronises (one 4-byte read-back)."""
    for t, name in ((idx, "idx"), (lut, "lut")):
        if t.dtype not in (torch.int32, torch.int64):
            raise TypeError(f"{name} must be int32 or int64")
        _dev(t, t.dtype, name)
    err = torch.zeros((1,), dtype=torch.int32, device=idx.device)
    out = torch.empty(idx.shape, dtype=torch.int32, device=idx.device)
    if idx.numel():
        _call("eod_remap_indices", idx.data_ptr(), int(idx.dtype == torch.int64), idx.numel(), lut.data_ptr(), int(lut.dtype == torch.int64),
              lut.numel(), int(add), int(n_rows), out.data_ptr(), err.data_ptr(), _stream())
    bad = int(err.item())
    if bad:
        raise IndexError(f"{bad} pixels map outside the semantic map / the {int(n_rows)}-row class table")
    return out


class DetWorkspace:
    """Caller-owned workspace of the deterministic writes (write_mean_det, write_objects[_pasted]_det), zero-filled once."""

    def __init__(self, n_episodes: int, channels: int, hw: int, n_cells: int, device: torch.device, runs_per_episode: int = 0):
        lib = _lib.lib()
        self.nbytes = int(lib.eod_write_mean_det_workspace_bytes(n_episodes, channels, hw, n_cells, int(runs_per_episode)))
        if self.nbytes <= 0:
            raise ValueError("bad sizes for the deterministic-write workspace")
        self.buf = torch.zeros((self.nbytes,), dtype=torch.uint8, device=device)
        self._status_off = int(lib.eod_write_mean_det_status_offset(n_episodes, n_cells))

    def overflowed(self) -> bool:
        """True if some run did not fit since the workspace was created (those runs used fp32 reductions)."""
        return bool(self.buf[self._status_off:self._status_off + 4].view(torch.int32).item())


def write_mean_det(feat: torch.Tensor, idx: torch.Tensor, samp: Optional[torch.Tensor], frame_cnt: torch.Tensor,
                   sums: torch.Tensor, ws: DetWorkspace, layout: int = LAYOUT_CHW, active: Optional[torch.Tensor] = None) -> None:
    """Deterministic main pass (HW % 32 == 0): same contract as write_mean, bitwise reproducible.  layout: LAYOUT_CHW (fp32) or
    LAYOUT_HWC / _HWC_BF16 / _HWC_F16 - the same features give the same bits in every layout (16-bit ones widened exactly); the
    16-bit CHW layouts raise EodError.  active (E) i32 | None: slots with active <= 0 are skipped (give frame_count the same mask)."""
    _dev(feat, LAYOUT_DTYPE.get(int(layout), torch.float32), "feat"), _dev(idx, torch.int32, "idx"), _dev(sums, torch.float32, "sums")
    _dev(frame_cnt, torch.int32, "frame_cnt")
    E, n_cells, C = sums.shape
    HW = idx[0].numel()
    if feat.numel() != E * C * HW:
        raise ValueError(f"feat has {feat.numel()} elements, expected E*C*HW = {E * C * HW}")
    if samp is not None:
        _dev(samp, torch.uint8, "samp")
    if active is not None:
        _dev(active, torch.int32, "active")
        if active.numel() != E:
            raise ValueError("active must hold one int32 per episode")
    _call("eod_write_mean_det_layout", feat.data_ptr(), int(layout), idx.data_ptr(), _ptr(samp), frame_cnt.data_ptr(), _ptr(active), E, C, HW,
          n_cells, sums.data_ptr(), ws.buf.data_ptr(), ws.nbytes, _stream())


def finalize_counts(idx: torch.Tensor, frame_cnt: torch.Tensor, counts: torch.Tensor,
                    touched: Optional[torch.Tensor] = None, sums: Optional[torch.Tensor] = None,
                    norm16: Optional[torch.Tensor] = None) -> None:
    """counts += 1 per visible cell, frame_cnt := 0; optionally refresh the normalised fp16 rows (norm16 (E,cells,C))
    of the visible cells from sums."""
    _dev(idx, torch.int32, "idx"), _dev(frame_cnt, torch.int32, "frame_cnt"), _dev(counts, torch.float32, "counts")
    if touched is not None:
        _dev(touched, torch.uint8, "touched")
    C = 0
    if norm16 is not None:
        _dev(norm16, torch.float16, "norm16"), _dev(sums, torch.float32, "sums")
        C = sums.shape[-1]
    E, HW = idx.shape[0], idx[0].numel()
    _call("eod_finalize_counts", idx.data_ptr(), E, HW, counts.shape[1], frame_cnt.data_ptr(), counts.data_ptr(),
          _ptr(touched), _ptr(sums) if norm16 is not None else None, _ptr(norm16), C, _stream())


def box_to_image_features(box_features: torch.Tensor, masks: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """box_features (K,C) f32, masks (K,H,W) bool/u8 -> image_features (1,C,H,W) f32, observed (H,W) bool."""
    _dev(box_features, torch.float32, "box_features")
    if masks.dtype == torch.bool:
        masks = masks.view(torch.uint8)
    _dev(masks, torch.uint8, "masks")
    K, C = box_features.shape
    H, W = masks.shape[1:]
    img = torch.empty((1, C, H, W), dtype=torch.float32, device=masks.device)
    obs = torch.empty((H, W), dtype=torch.uint8, device=masks.device)
    _call("eod_box_to_image_features", box_features.data_ptr(), masks.data_ptr(), K, C, H * W, img.data_ptr(),
          obs.data_ptr(), _stream())
    return img, obs.view(torch.bool)


def _masks_u8(masks: torch.Tensor) -> torch.Tensor:
    if masks.dtype == torch.bool:
        masks = masks.view(torch.uint8)
    return _dev(masks, torch.uint8, "masks")


def masks_observed(masks: torch.Tensor, n_obj: Optional[torch.Tensor] = None, observed: Optional[torch.Tensor] = None) -> torch.Tensor:
    """masks (E,Kmax,H,W) bool/u8, n_obj (E) i32 | None -> observed (E,H*W) u8 (1 where any object covers the pixel)."""
    masks = _masks_u8(masks)
    E, Kmax, H, W = masks.shape
    if n_obj is not None:
        _dev(n_obj, torch.int32, "n_obj")
    observed = torch.empty((E, H * W), dtype=torch.uint8, device=masks.device) if observed is None else _dev(observed, torch.uint8, "observed")
    _call("eod_masks_observed", masks.data_ptr(), _ptr(n_obj), E, Kmax, H * W, observed.data_ptr(), _stream())
    return observed


def write_objects(box_features: torch.Tensor, masks: torch.Tensor, n_obj: Optional[torch.Tensor], idx: torch.Tensor,
                  samp: torch.Tensor, slots: ObjectSlots) -> None:
    """Fused A6+A7 (first half): box_features (E,Kmax,C) f32, masks (E,Kmax,H,W), idx (E,H,W) i32, samp (E,HW) u8;
    the per-pixel object means of the sampled pixels are reduced into slots.scratch."""
    masks = _masks_u8(masks)
    _dev(box_features, torch.float32, "box_features"), _dev(idx, torch.int32, "idx"), _dev(samp, torch.uint8, "samp")
    E, Kmax, H, W = masks.shape
    if box_features.shape != (E, Kmax, slots.C) or slots.E != E:
        raise ValueError("box_features must be (E,Kmax,C) matching masks (E,Kmax,H,W) and the slot workspace")
    if n_obj is not None:
        _dev(n_obj, torch.int32, "n_obj")
    _call("eod_write_objects", box_features.data_ptr(), masks.data_ptr(), _ptr(n_obj), Kmax, idx.data_ptr(), samp.data_ptr(),
          slots.slot_of_cell.data_ptr(), E, slots.C, H * W, slots.n_cells, slots.S, slots.scratch.data_ptr(), _stream())


def _paste_args(mask_probs: torch.Tensor, boxes: torch.Tensor, n_obj: Optional[torch.Tensor]):
    _dev(mask_probs, torch.float32, "mask_probs"), _dev(boxes, torch.float32, "boxes")
    if mask_probs.dim() != 4 or mask_probs.shape[-1] != mask_probs.shape[-2]:
        raise ValueError("mask_probs must be (E,Kmax,S,S): only square mask predictions are supported")
    E, Kmax, S, _ = mask_probs.shape
    if boxes.shape != (E, Kmax, 4):
        raise ValueError("boxes must be (E,Kmax,4) XYXY matching mask_probs (E,Kmax,S,S)")
    if n_obj is not None:
        _dev(n_obj, torch.int32, "n_obj")
    return E, Kmax, S


def paste_masks(mask_probs: torch.Tensor, boxes: torch.Tensor, image_shape: Tuple[int, int], threshold: float = 0.5,
                n_obj: Optional[torch.Tensor] = None, want_masks: bool = True, want_observed: bool = False,
                observed_out: Optional[torch.Tensor] = None):
    """paste_masks_in_image (detectron2 mask_ops.py, custom_rcnn.py:880) for E episodes: mask_probs (E,Kmax,S,S) f32,
    boxes (E,Kmax,4) f32 -> masks (E,Kmax,H,W) bool and / or observed (E,H*W) u8 (OR over the episode's objects)."""
    E, Kmax, S = _paste_args(mask_probs, boxes, n_obj)
    H, W = int(image_shape[0]), int(image_shape[1])
    dev = mask_probs.device
    masks = torch.empty((E, Kmax, H, W), dtype=torch.uint8, device=dev) if want_masks else None
    observed = None
    if want_observed:
        observed = torch.empty((E, H * W), dtype=torch.uint8, device=dev) if observed_out is None else _dev(observed_out, torch.uint8, "observed_out")
        if observed.numel() != E * H * W:
            raise ValueError("observed_out must hold E*H*W bytes")
    if Kmax == 0:
        return (masks.view(torch.bool) if want_masks else None), (observed.zero_() if want_observed else None)
    _call("eod_paste_masks", mask_probs.data_ptr(), boxes.data_ptr(), _ptr(n_obj), E, Kmax, S, H, W, float(threshold),
          _ptr(masks), _ptr(observed), _stream())
    return (masks.view(torch.bool) if want_masks else None), observed


def write_objects_pasted(box_features: torch.Tensor, mask_probs: torch.Tensor, boxes: torch.Tensor, n_obj: Optional[torch.Tensor],
                         idx: torch.Tensor, samp: torch.Tensor, slots: ObjectSlots, threshold: float = 0.5) -> None:
    """write_objects with the pasted-mask test evaluated on the fly: mask_probs (E,Kmax,S,S), boxes (E,Kmax,4), idx (E,H,W)."""
    E, Kmax, S = _paste_args(mask_probs, boxes, n_obj)
    _dev(box_features, torch.float32, "box_features"), _dev(idx, torch.int32, "idx"), _dev(samp, torch.uint8, "samp")
    if idx.dim() != 3:
        raise ValueError("idx must be (E,H,W)")
    _, H, W = idx.shape
    if box_features.shape != (E, Kmax, slots.C) or slots.E != E:
        raise ValueError("box_features must be (E,Kmax,C) matching mask_probs and the slot workspace")
    _call("eod_write_objects_pasted", box_features.data_ptr(), mask_probs.data_ptr(), boxes.data_ptr(), _ptr(n_obj), Kmax, S, H, W,
          float(threshold), idx.data_ptr(), samp.data_ptr(), slots.slot_of_cell.data_ptr(), E, slots.C, slots.n_cells, slots.S,
          slots.scratch.data_ptr(), _stream())


def write_objects_det(box_features: torch.Tensor, masks: torch.Tensor, n_obj: Optional[torch.Tensor], idx: torch.Tensor,
                      samp: torch.Tensor, frame_cnt: torch.Tensor, sums: torch.Tensor, ws: DetWorkspace) -> None:
    """Deterministic object write (HW % 32 == 0): sums[cell] += the cell's mean of the sampled pixels' object means, bit for bit
    what write_mean_det(LAYOUT_CHW) adds for the box_to_image_features image, without building it.  frame_cnt from
    frame_count(idx, samp, frame_cnt, n_obj) (no slots); ws is the DetWorkspace of write_mean_det, sized the same way."""
    masks = _masks_u8(masks)
    _dev(box_features, torch.float32, "box_features"), _dev(idx, torch.int32, "idx"), _dev(samp, torch.uint8, "samp")
    _dev(frame_cnt, torch.int32, "frame_cnt"), _dev(sums, torch.float32, "sums")
    E, Kmax, H, W = masks.shape
    _, n_cells, C = sums.shape
    if box_features.shape != (E, Kmax, C) or sums.shape[0] != E:
        raise ValueError("box_features must be (E,Kmax,C) matching masks (E,Kmax,H,W) and sums (E,cells,C)")
    if n_obj is not None:
        _dev(n_obj, torch.int32, "n_obj")
    _call("eod_write_objects_det", box_features.data_ptr(), masks.data_ptr(), _ptr(n_obj), Kmax, idx.data_ptr(), samp.data_ptr(),
          frame_cnt.data_ptr(), E, C, H * W, n_cells, sums.data_ptr(), ws.buf.data_ptr(), ws.nbytes, _stream())


def write_objects_pasted_det(box_features: torch.Tensor, mask_probs: torch.Tensor, boxes: torch.Tensor, n_obj: Optional[torch.Tensor],
                             idx: torch.Tensor, samp: torch.Tensor, frame_cnt: torch.Tensor, sums: torch.Tensor, ws: DetWorkspace,
                             threshold: float = 0.5) -> None:
    """write_objects_det with the pasted-mask test evaluated on the fly: mask_probs (E,Kmax,S,S), boxes (E,Kmax,4), idx (E,H,W)."""
    E, Kmax, S = _paste_args(mask_probs, boxes, n_obj)
    _dev(box_features, torch.float32, "box_features"), _dev(idx, torch.int32, "idx"), _dev(samp, torch.uint8, "samp")
    _dev(frame_cnt, torch.int32, "frame_cnt"), _dev(sums, torch.float32, "sums")
    if idx.dim() != 3:
        raise ValueError("idx must be (E,H,W)")
    _, H, W = idx.shape
    _, n_cells, C = sums.shape
    if box_features.shape != (E, Kmax, C) or sums.shape[0] != E:
        raise ValueError("box_features must be (E,Kmax,C) matching mask_probs and sums (E,cells,C)")
    _call("eod_write_objects_pasted_det", box_features.data_ptr(), mask_probs.data_ptr(), boxes.data_ptr(), _ptr(n_obj), Kmax, S, H, W,
          float(threshold), idx.data_ptr(), samp.data_ptr(), frame_cnt.data_ptr(), E, C, n_cells, sums.data_ptr(), ws.buf.data_ptr(), ws.nbytes,
          _stream())


def flush_slots(frame_cnt: torch.Tensor, slots: ObjectSlots, sums: torch.Tensor) -> None:
    """sums[cell] += scratch[slot] / n_cell for every claimed slot; the workspace returns to zero."""
    _dev(frame_cnt, torch.int32, "frame_cnt"), _dev(sums, torch.float32, "sums")
    E, n_cells, C = sums.shape
    if (E, n_cells, C) != (slots.E, slots.n_cells, slots.C):
        raise ValueError("sums does not match the slot workspace")
    _call("eod_flush_slots", frame_cnt.data_ptr(), slots.slot_of_cell.data_ptr(), slots.slot_cell.data_ptr(), slots.n_slots.data_ptr(),
          E, C, n_cells, slots.S, slots.scratch.data_ptr(), sums.data_ptr(), _stream())


def bilinear_lattice(src: torch.Tensor, out_hw: Tuple[int, int], step: int) -> torch.Tensor:
    """F.interpolate(src, out_hw, mode='bilinear', align_corners=True)[:, :, ::step, ::step] for src (E,C,h,w) f32."""
    _dev(src, torch.float32, "src")
    E, C, h, w = src.shape
    H, W = int(out_hw[0]), int(out_hw[1])
    out = torch.empty((E, C, -(-H // step), -(-W // step)), dtype=torch.float32, device=src.device)
    _call("eod_bilinear_lattice", src.data_ptr(), E, C, h, w, H, W, int(step), out.data_ptr(), _stream())
    return out


def write_max(height: torch.Tensor, idx: torch.Tensor, outlier: Optional[torch.Tensor], feat: Optional[torch.Tensor],
              height_map: torch.Tensor, key64: torch.Tensor, arg_pix: torch.Tensor, observed: Optional[torch.Tensor],
              state: Optional[torch.Tensor], layout: int = LAYOUT_HWC, pix_stride: int = 1) -> None:
    """height/idx/outlier (E,H,W); feat (E,H,W,C) [HWC] or (E,C,H,W) [CHW]; height_map (E,cells) f32;
    key64 (E,cells) i64 scratch; arg_pix (E,cells) i32; observed (E,cells) u8; state (E,cells,C) f32."""
    _dev(height, torch.float32, "height"), _dev(idx, torch.int32, "idx"), _dev(height_map, torch.float32, "height_map")
    _dev(key64, torch.int64, "key64"), _dev(arg_pix, torch.int32, "arg_pix")
    E, H, W = height.shape
    C = 0
    if feat is not None:
        _dev(feat, torch.float32, "feat"), _dev(state, torch.float32, "state")
        C = state.shape[2]
    if outlier is not None:
        if outlier.dtype == torch.bool:
            outlier = outlier.view(torch.uint8)
        _dev(outlier, torch.uint8, "outlier")
    if observed is not None:
        _dev(observed, torch.uint8, "observed")
    _call("eod_write_max", height.data_ptr(), idx.data_ptr(), _ptr(outlier), _ptr(feat), int(layout), E, C, H, W,
          int(pix_stride), height_map.shape[1], height_map.data_ptr(), key64.data_ptr(), arg_pix.data_ptr(),
          _ptr(observed), _ptr(state), _stream())


def write_max_linear(height: torch.Tensor, idx: torch.Tensor, outlier: Optional[torch.Tensor], feat: torch.Tensor, height_map: torch.Tensor,
                     key64: torch.Tensor, arg_pix: torch.Tensor, observed: Optional[torch.Tensor], state: torch.Tensor, weight: torch.Tensor,
                     bias: Optional[torch.Tensor], layout: int = LAYOUT_HWC, pix_stride: int = 1) -> torch.Tensor:
    """SMNet 'replace' update with the linear layer (model.py of the 3.10 bytecode, src lines 104-128): the height-max contest of
    write_max, then ``state[raised cells] = linlayer(feature[winner pixels])`` as ONE tensor-core row GEMM over the winners only
    (eod_max_winner_list + eod_linear_rows).  feat (E,H,W,C_in) [HWC] or (E,C_in,H,W) [CHW]; weight (C_mem,C_in), bias (C_mem,);
    state (E,cells,C_mem).  Returns the device-side winner count (1,) i32."""
    _dev(feat, torch.float32, "feat"), _dev(state, torch.float32, "state"), _dev(weight, torch.float32, "weight")
    E, H, W = height.shape
    c_in = weight.shape[1]
    if tuple(feat.shape) != ((E, H, W, c_in) if layout == LAYOUT_HWC else (E, c_in, H, W)):
        raise ValueError("write_max_linear: feat does not match (E,H,W,C_in) / (E,C_in,H,W)")
    if state.shape[2] != weight.shape[0]:
        raise ValueError("write_max_linear: state channels must equal weight.shape[0]")
    write_max(height, idx, outlier, None, height_map, key64, arg_pix, observed, None, layout, pix_stride)
    lattice = -(-H // pix_stride) * -(-W // pix_stride)
    src, dst, count = max_winner_list(arg_pix, H, W, c_in, layout, capacity=min(arg_pix.numel(), E * lattice))
    linear_rows(feat, weight, bias, 1.0, out=state.view(-1, state.shape[2]), a_off=src, a_k_stride=1 if layout == LAYOUT_HWC else H * W,
                m_count=count, n_rows=src.numel(), y_dst=dst)
    return count


def linear_rows(a: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor] = None, scale: float = 1.0, *,
                out: Optional[torch.Tensor] = None, a_off: Optional[torch.Tensor] = None, a_k_stride: int = 1, m_count: Optional[torch.Tensor] = None,
                n_rows: Optional[int] = None, y_dst: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Y = scale * (A @ weight^T + bias) in fp32 accuracy on the tensor cores (eod_linear_rows, 3xTF32).
    a: (M,K) f32, ANY strides (a transposed view costs nothing) - or, with ``a_off`` (M_max,) int64 element offsets, the flat f32
    buffer the rows are gathered from (element l of row i at a_off[i] + l * a_k_stride; K = weight.shape[1]; ``m_count`` (1,) i32 on
    the device bounds the rows, ``n_rows`` = M_max).  weight: (N,K) f32, any strides; bias (N,) f32.  out: (rows,N') f32 with unit
    column stride, written at row i or y_dst[i] (int64); default a fresh (M,N)."""
    _devs = [a, weight] + [t for t in (bias, out, a_off, m_count, y_dst) if t is not None]
    for t in _devs:
        if not t.is_cuda or t.device != a.device:
            raise EodError("linear_rows: all tensors must live on one CUDA device (no CPU fallback)")
    if a.dtype != torch.float32 or weight.dtype != torch.float32 or weight.dim() != 2:
        raise TypeError("linear_rows: a and weight must be float32, weight (N,K)")
    N, K = weight.shape
    if a_off is None:
        if a.dim() != 2 or a.shape[1] != K:
            raise ValueError("linear_rows: a must be (M,K)")
        M, a_rs, a_ks = a.shape[0], a.stride(0), a.stride(1)
    else:
        if a_off.dtype != torch.int64 or not a_off.is_contiguous():
            raise TypeError("linear_rows: a_off must be contiguous int64")
        M, a_rs, a_ks = int(a_off.numel() if n_rows is None else n_rows), 0, int(a_k_stride)
    if bias is not None:
        _dev(bias, torch.float32, "bias")
    if out is None:
        if y_dst is not None:
            raise ValueError("linear_rows: scattered rows need an explicit out")
        out = torch.empty((M, N), dtype=torch.float32, device=a.device)
    if out.dtype != torch.float32 or out.dim() != 2 or out.stride(1) != 1 or out.shape[1] < N:
        raise ValueError("linear_rows: out must be (rows, >= N) float32 with unit column stride")
    if m_count is not None:
        _dev(m_count, torch.int32, "m_count")
    if y_dst is not None and (y_dst.dtype != torch.int64 or not y_dst.is_contiguous()):
        raise TypeError("linear_rows: y_dst must be contiguous int64")
    if a.device.index != torch.cuda.current_device():
        raise EodError("linear_rows: tensors are not on the current CUDA device")
    _call("eod_linear_rows", a.data_ptr(), int(a_rs), int(a_ks), _ptr(a_off), weight.data_ptr(), int(weight.stride(0)), int(weight.stride(1)),
          _ptr(bias), float(scale), int(M), _ptr(m_count), int(N), int(K), out.data_ptr(), int(out.stride(0)), _ptr(y_dst), _stream())
    return out


def max_winner_list(arg_pix: torch.Tensor, H: int, W: int, C: int, layout: int = LAYOUT_HWC, capacity: Optional[int] = None):
    """arg_pix (E,cells) i32 of write_max -> (src_off (cap,) i64, dst_row (cap,) i64, count (1,) i32) for linear_rows (the 'replace'
    update: state[dst_row] = linlayer(feat[src_off ...])).  capacity defaults to the number of pixels, the most winners a frame can have."""
    _dev(arg_pix, torch.int32, "arg_pix")
    E, n_cells = arg_pix.shape
    cap = int(min(E * n_cells, E * H * W) if capacity is None else capacity)
    src = torch.empty((cap,), dtype=torch.int64, device=arg_pix.device)
    dst = torch.empty((cap,), dtype=torch.int64, device=arg_pix.device)
    count = torch.empty((1,), dtype=torch.int32, device=arg_pix.device)
    _call("eod_max_winner_list", arg_pix.data_ptr(), E, n_cells, int(H), int(W), int(C), int(layout), src.data_ptr(), dst.data_ptr(),
          count.data_ptr(), cap, _stream())
    return src, dst, count


class HeightMaxScratch:
    """Per-frame scratch of the lock-step height-max write (eod_heightmax_*), all-zero between frames (the update leaves it so):
    key64 (E,cells) i64 packed keys, cell_list (E,list_cap) i32 the cells a frame touched, n_list (E,2) i32, and ``raised`` (1,) i32:
    the number of cells the last update raised (device)."""

    def __init__(self, n_episodes: int, n_cells: int, lattice: int, device: torch.device):
        self.E, self.n_cells, self.list_cap = int(n_episodes), int(n_cells), int(min(n_cells, lattice))
        self.key64 = torch.zeros((self.E, self.n_cells), dtype=torch.int64, device=device)
        self.cell_list = torch.zeros((self.E, self.list_cap), dtype=torch.int32, device=device)
        self.n_list = torch.zeros((self.E, 2), dtype=torch.int32, device=device)
        self.raised = torch.zeros((1,), dtype=torch.int32, device=device)

    def args(self) -> tuple:
        return self.key64.data_ptr(), self.cell_list.data_ptr(), self.list_cap, self.n_list.data_ptr(), self.raised.data_ptr()


def _active(active: Optional[torch.Tensor], E: int) -> Optional[int]:
    if active is None:
        return None
    _dev(active, torch.int32, "active")
    if active.numel() != E:
        raise ValueError("active must hold one int32 per episode")
    return active.data_ptr()


def heightmax_contest_depth(depth: torch.Tensor, pose: torch.Tensor, shifts: torch.Tensor, intr: Sequence[float], cell: float, map_w: int,
                            map_h: int, scratch: HeightMaxScratch, active: Optional[torch.Tensor] = None, pix_stride: int = 1,
                            order: int = ORDER_ZX, z_clip: float = 0.5, depth_div: float = 1000.0) -> None:
    """Height-max contest of one frame with the geometry computed from depth in registers (no idx / outlier / height planes):
    depth (E,H,W) f32 metres or uint16 (/ depth_div), pose (E,12), shifts (E,6); active (E) i32 | None."""
    raw = depth.dtype == torch.uint16
    _dev(depth, torch.uint16 if raw else torch.float32, "depth"), _dev(pose, torch.float32, "pose"), _dev(shifts, torch.float32, "shifts")
    E, H, W = depth.shape
    if pose.shape != (E, 12) or shifts.shape != (E, 6) or scratch.E != E or scratch.n_cells != map_w * map_h:
        raise ValueError("heightmax_contest_depth: pose (E,12), shifts (E,6) and a scratch of E episodes x map_w*map_h cells")
    fx, fy, cx, cy = (float(v) for v in intr)
    _call("eod_heightmax_contest_depth", depth.data_ptr(), int(raw), float(depth_div), pose.data_ptr(), shifts.data_ptr(), E, H, W, fx, fy, cx, cy,
          float(cell), int(map_w), int(map_h), int(order), float(z_clip), int(pix_stride), _active(active, E), *scratch.args(), _stream())


def heightmax_contest_planes(height: torch.Tensor, idx: torch.Tensor, outlier: Optional[torch.Tensor], scratch: HeightMaxScratch,
                             active: Optional[torch.Tensor] = None, pix_stride: int = 1) -> None:
    """Height-max contest of one frame from precomputed planes (create_coco_mp3d.py:157-165): height (E,H,W) f32, idx (E,H,W) i32 cell
    ids in [0, cells), outlier (E,H,W) u8 / bool | None; active (E) i32 | None."""
    _dev(height, torch.float32, "height"), _dev(idx, torch.int32, "idx")
    E, H, W = height.shape
    if tuple(idx.shape) != (E, H, W) or scratch.E != E:
        raise ValueError("heightmax_contest_planes: height and idx (E,H,W) and a scratch of E episodes")
    if outlier is not None:
        if outlier.dtype == torch.bool:
            outlier = outlier.view(torch.uint8)
        _dev(outlier, torch.uint8, "outlier")
        if tuple(outlier.shape) != (E, H, W):
            raise ValueError("heightmax_contest_planes: outlier must be (E,H,W)")
    _call("eod_heightmax_contest_planes", height.data_ptr(), idx.data_ptr(), _ptr(outlier), E, H, W, int(pix_stride), scratch.n_cells,
          _active(active, E), *scratch.args(), _stream())


def _feat_hw(feat: torch.Tensor, layout: int, E: int, C: int, what: str) -> Tuple[int, int]:
    """(H, W) of (E,H,W,C) channels-last or (E,C,H,W) features; EodError if the dtype does not belong to the layout."""
    dtype = LAYOUT_DTYPE.get(int(layout), torch.float32)
    if feat.dtype != dtype:
        raise EodError(f"{what}: layout {int(layout)} takes {dtype} features, got {feat.dtype}")
    _dev(feat, dtype, "feat")
    hwc = int(layout) in (LAYOUT_HWC, LAYOUT_HWC_BF16, LAYOUT_HWC_F16)
    if feat.dim() != 4 or feat.shape[0] != E or feat.shape[3 if hwc else 1] != C:
        raise ValueError(f"{what}: feat must be {'(E,H,W,C)' if hwc else '(E,C,H,W)'} with E={E}, C={C}, got {tuple(feat.shape)}")
    return (feat.shape[1], feat.shape[2]) if hwc else (feat.shape[2], feat.shape[3])


def heightmax_update(feat: torch.Tensor, layout: int, scratch: HeightMaxScratch, height_map: torch.Tensor, observed: torch.Tensor,
                     state: torch.Tensor, linlayer: Optional[Tuple[torch.Tensor, Optional[torch.Tensor]]] = None) -> torch.Tensor:
    """Update of the cells the frame's contest listed: height_map (E,cells) f32 and observed (E,cells) u8 of the raised cells, and
    state (E,cells,C_mem) f32 rows := the winners' feature rows (copy) or ``linlayer(feature rows)`` with linlayer = (weight (C_mem,C)
    f32, bias (C_mem,) | None) on the tensor cores (eod_linear_rows; fp32 features only).  feat (E,C,H,W) [CHW layouts] or (E,H,W,C)
    [HWC layouts] in the layout's dtype.  Returns the device count of raised cells (scratch.raised, valid until the next contest)."""
    _dev(height_map, torch.float32, "height_map"), _dev(observed, torch.uint8, "observed"), _dev(state, torch.float32, "state")
    E, n_cells = height_map.shape
    if (E, n_cells) != (scratch.E, scratch.n_cells) or tuple(observed.shape) != (E, n_cells) or state.dim() != 3 or state.shape[:2] != (E, n_cells):
        raise ValueError("heightmax_update: height_map / observed (E,cells), state (E,cells,C) matching the scratch")
    if linlayer is None:
        C = state.shape[2]
        H, W = _feat_hw(feat, layout, E, C, "heightmax_update")
        _call("eod_heightmax_update", feat.data_ptr(), int(layout), E, C, H, W, n_cells, scratch.cell_list.data_ptr(), scratch.list_cap,
              scratch.n_list.data_ptr(), scratch.key64.data_ptr(), height_map.data_ptr(), observed.data_ptr(), state.data_ptr(), None, None, 0,
              scratch.raised.data_ptr(), _stream())
        return scratch.raised
    weight, bias = linlayer
    if int(layout) not in (LAYOUT_CHW, LAYOUT_HWC):
        raise EodError("heightmax_update: the linlayer update takes fp32 features (LAYOUT_CHW / LAYOUT_HWC)")
    c_in = weight.shape[1]
    H, W = _feat_hw(feat, layout, E, c_in, "heightmax_update")
    if state.shape[2] != weight.shape[0]:
        raise ValueError("heightmax_update: state channels must equal weight.shape[0]")
    cap = E * scratch.list_cap
    if getattr(scratch, "_winners", None) is None or scratch._winners[0].numel() != cap:
        scratch._winners = (torch.empty((cap,), dtype=torch.int64, device=feat.device), torch.empty((cap,), dtype=torch.int64, device=feat.device))
    src, dst = scratch._winners
    _call("eod_heightmax_update", None, int(layout), E, c_in, H, W, n_cells, scratch.cell_list.data_ptr(), scratch.list_cap,
          scratch.n_list.data_ptr(), scratch.key64.data_ptr(), height_map.data_ptr(), observed.data_ptr(), None, src.data_ptr(), dst.data_ptr(),
          cap, scratch.raised.data_ptr(), _stream())
    linear_rows(feat, weight, bias, 1.0, out=state.view(-1, state.shape[2]), a_off=src, a_k_stride=1 if int(layout) == LAYOUT_HWC else H * W,
                m_count=scratch.raised, n_rows=cap, y_dst=dst)
    return scratch.raised


def heightmax_reset(height_map: torch.Tensor, observed: torch.Tensor, state: torch.Tensor, mask: torch.Tensor) -> None:
    """Per-slot reset of the height-max state: the episodes with mask[e] != 0 get height_map = 0, observed = 0 and zero state rows."""
    _dev(height_map, torch.float32, "height_map"), _dev(observed, torch.uint8, "observed"), _dev(state, torch.float32, "state")
    _dev(mask, torch.int32, "mask")
    E, n_cells, C = state.shape
    if mask.numel() != E or tuple(height_map.shape) != (E, n_cells) or tuple(observed.shape) != (E, n_cells):
        raise ValueError("heightmax_reset: mask (E), height_map / observed (E,cells), state (E,cells,C)")
    _call("eod_heightmax_reset", mask.data_ptr(), E, n_cells, C, height_map.data_ptr(), observed.data_ptr(), state.data_ptr(), _stream())


def read_pool(table: torch.Tensor, counts: Optional[torch.Tensor], idx: torch.Tensor, out: Optional[Sequence[torch.Tensor]] = None):
    """table (E,cells,C) f32 sums (+ counts (E,cells) f32) or f16 normalised table; idx (E,H,W) i32/i64.
    Returns [L0, L1, L2] as logical (E,C,h,w) f16 tensors in channels_last memory format."""
    if table.dtype not in (torch.float32, torch.float16):
        raise TypeError("table must be float32 (sums) or float16 (normalised memory)")
    _dev(table, table.dtype, "table")
    if idx.dtype not in (torch.int32, torch.int64):
        raise TypeError("idx must be int32 or int64")
    _dev(idx, idx.dtype, "idx")
    E, n_cells, C = table.shape
    _, H, W = idx.shape
    if counts is not None:
        _dev(counts, torch.float32, "counts")
    if out is None:
        out = [torch.empty((E, H >> s, W >> s, C), dtype=torch.float16, device=table.device) for s in (3, 4, 5)]
    for o in out:
        _dev(o, torch.float16, "level")
    _call("eod_read_pool", table.data_ptr(), int(table.dtype == torch.float16), _ptr(counts), idx.data_ptr(),
          int(idx.dtype == torch.int64), E, C, H, W, n_cells, out[0].data_ptr(), out[1].data_ptr(), out[2].data_ptr(),
          _stream())
    return [o.permute(0, 3, 1, 2) for o in out]


def read_roi(levels: Sequence[torch.Tensor], boxes: torch.Tensor, batch_idx: Optional[torch.Tensor] = None, pooled: int = 7,
             strides: Sequence[int] = (8, 16, 32), sampling_ratio: int = 0, min_level: int = 3, canonical_size: float = 224.0,
             canonical_level: int = 4, want_levels: bool = False, want_valid: bool = False):
    """Per-ROI map features: ROIAlign (aligned, detectron2 ROIAlignV2) of the pooled memory levels over the proposals' boxes with
    the FPN level assignment (detic_roi_heads.py:331-334 applied to the memory levels; see eod_read_roi).
    levels: what read_pool returns - logical (E,C,h,w) fp16 tensors in channels-last memory; boxes (R,4) f32 XYXY image pixels;
    batch_idx (R) i32.  Returns logical (R,C,pooled,pooled) f32 in channels-last memory [, assigned level (R) i32] [, valid (R,pooled,
    pooled) f32: the share of each bin's sample points that lie on the level = ROIAlign of a constant-1 plane].
    Level -1 means the box pools nothing (zero features, valid 0): detectron2 assigns it no level (its size is NaN: inverted in
    exactly one axis, or a NaN coordinate), or its batch_idx lies outside [0, E)."""
    import ctypes
    n = len(levels)
    if not (1 <= n <= 4) or len(strides) != n:
        raise ValueError("read_roi: 1..4 levels with one stride each")
    _dev(boxes, torch.float32, "boxes")
    if boxes.dim() != 2 or boxes.shape[1] != 4:
        raise ValueError("boxes must be (R,4) XYXY")
    R = boxes.shape[0]
    C = levels[0].shape[1]
    dims = [_level_dims(lv, C) for lv in levels]
    E = dims[0][0]
    if any(d[0] != E for d in dims):
        raise ValueError("all levels must share the episode dimension")
    if batch_idx is not None:
        _dev(batch_idx, torch.int32, "batch_idx")
        if batch_idx.numel() != R:
            raise ValueError("batch_idx must hold one int32 per box")
    elif E != 1:
        raise ValueError("batch_idx is required when the levels hold more than one episode")
    out = torch.empty((R, pooled, pooled, C), dtype=torch.float32, device=boxes.device)
    lvl = torch.empty((R,), dtype=torch.int32, device=boxes.device) if want_levels else None
    valid = torch.empty((R, pooled, pooled), dtype=torch.float32, device=boxes.device) if want_valid else None
    if R:
        _call("eod_read_roi", n, (ctypes.c_void_p * n)(*[lv.data_ptr() for lv in levels]), (ctypes.c_int * n)(*[d[1] for d in dims]),
              (ctypes.c_int * n)(*[d[2] for d in dims]), (ctypes.c_float * n)(*[1.0 / float(s) for s in strides]), E, C, boxes.data_ptr(),
              _ptr(batch_idx), R, int(pooled), int(sampling_ratio), int(min_level), float(canonical_size), int(canonical_level),
              out.data_ptr(), _ptr(lvl), _ptr(valid), _stream())
    out = out.permute(0, 3, 1, 2)
    ret = (out,) + ((lvl,) if want_levels else ()) + ((valid,) if want_valid else ())
    return ret if len(ret) > 1 else out


def fuse(res: Optional[torch.Tensor], mem: Optional[torch.Tensor], weight: float, mode: int,
         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    ref = res if res is not None else mem
    if res is not None:
        _dev(res, torch.float32, "res")
    if mem is not None:
        _dev(mem, torch.float32, "mem")
    out = torch.empty_like(ref) if out is None else _dev(out, torch.float32, "out")
    _call("eod_fuse", _ptr(res), _ptr(mem), float(weight), int(mode), ref.numel(), out.data_ptr(), _stream())
    return out


def normalize_memory(sums: torch.Tensor, counts: torch.Tensor, half: bool = False) -> torch.Tensor:
    """create_implicit_memory as a table: sums (..., cells, C) f32, counts (..., cells) f32 -> same shape, f32|f16."""
    _dev(sums, torch.float32, "sums"), _dev(counts, torch.float32, "counts")
    C = sums.shape[-1]
    out = torch.empty(sums.shape, dtype=torch.float16 if half else torch.float32, device=sums.device)
    _call("eod_normalize_memory", sums.data_ptr(), counts.data_ptr(), sums.numel() // C, C, out.data_ptr(), int(half), _stream())
    return out


def project_split_weights(weight: torch.Tensor) -> torch.Tensor:
    """weight (N,K) or (N,K,1,1) f32 -> (2N,K) f16 hi/lo split consumed by project_fuse (N % 128 == 0, K % 64 == 0)."""
    _dev(weight, torch.float32, "weight")
    N = weight.shape[0]
    K = weight.numel() // N
    out = torch.empty((2 * N, K), dtype=torch.float16, device=weight.device)
    _call("eod_project_split_weights", weight.data_ptr(), N, K, out.data_ptr(), _stream())
    return out


def project_fuse(level: torch.Tensor, w_split: torch.Tensor, bias: Optional[torch.Tensor], res: Optional[torch.Tensor],
                 weight: float, mode: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """level: logical (E,K,h,w) f16 in channels-last memory (what read_pool returns) or (E,h,w,K) contiguous;
    w_split (2N,K) f16; bias (N) f32 | None; res (E,N,h,w) f32 NCHW | None (mem_only) -> out (E,N,h,w) f32 NCHW."""
    if level.dim() != 4 or level.dtype != torch.float16 or not level.is_cuda:
        raise TypeError("level must be a 4-d CUDA float16 tensor")
    K = w_split.shape[1]
    if level.shape[1] == K and level.permute(0, 2, 3, 1).is_contiguous():
        E, _, h, w = level.shape
    elif level.shape[3] == K and level.is_contiguous():
        E, h, w, _ = level.shape
    else:
        raise ValueError("level must be channels-last (E,h,w,K) memory with K matching w_split")
    _dev(w_split, torch.float16, "w_split")
    N = w_split.shape[0] // 2
    if bias is not None:
        _dev(bias, torch.float32, "bias")
        if bias.numel() != N:
            raise ValueError("bias must have N elements")
    if mode not in (FUSE_SUM, FUSE_MEM_ONLY):
        raise ValueError("project_fuse: mode must be FUSE_SUM or FUSE_MEM_ONLY")
    if res is not None:
        _dev(res, torch.float32, "res")
        if tuple(res.shape) != (E, N, h, w):
            raise ValueError(f"res must be (E,N,h,w) = {(E, N, h, w)}")
    out = torch.empty((E, N, h, w), dtype=torch.float32, device=level.device) if out is None else _dev(out, torch.float32, "out")
    _call("eod_project_fuse", level.data_ptr(), w_split.data_ptr(), _ptr(bias), _ptr(res), float(weight), int(mode), E, h * w, K, N,
          out.data_ptr(), _stream())
    return out


def _level_dims(level: torch.Tensor, K: int):
    if level.dim() != 4 or level.dtype != torch.float16 or not level.is_cuda:
        raise TypeError("level must be a 4-d CUDA float16 tensor")
    if level.shape[1] == K and level.permute(0, 2, 3, 1).is_contiguous():
        E, _, h, w = level.shape
    elif level.shape[3] == K and level.is_contiguous():
        E, h, w, _ = level.shape
    else:
        raise ValueError("level must be channels-last (E,h,w,K) memory with K matching w_split")
    return E, h, w


def project_fuse_levels(levels: Sequence[torch.Tensor], w_splits: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]],
                        results: Optional[Sequence[torch.Tensor]], weight: float, mode: int,
                        outs: Optional[Sequence[torch.Tensor]] = None, variant: int = 0):
    """project_fuse for up to three pyramid levels in one launch (persistent tcgen05 kernel).  Same per-level contract as
    project_fuse; all levels share E, K and N."""
    import ctypes
    n = len(levels)
    if not (1 <= n <= 3) or len(w_splits) != n or len(biases) != n or (results is not None and len(results) != n):
        raise ValueError("project_fuse_levels: 1..3 levels with matching w_splits / biases / results")
    if mode not in (FUSE_SUM, FUSE_MEM_ONLY):
        raise ValueError("project_fuse_levels: mode must be FUSE_SUM or FUSE_MEM_ONLY")
    if mode == FUSE_SUM and results is None:
        raise EodError("project_fuse_levels: res is required for sum")
    K = w_splits[0].shape[1]
    N = w_splits[0].shape[0] // 2
    dims = [_level_dims(lv, K) for lv in levels]
    E = dims[0][0]
    created = outs is None
    outs = [torch.empty((E, N, h, w), dtype=torch.float32, device=levels[0].device) for _, h, w in dims] if created else list(outs)
    for k in range(n):
        _dev(w_splits[k], torch.float16, "w_split"), _dev(outs[k], torch.float32, "out")
        if dims[k][0] != E or tuple(w_splits[k].shape) != (2 * N, K):
            raise ValueError("all levels must share E, K and N")
        if biases[k] is not None:
            _dev(biases[k], torch.float32, "bias")
        if results is not None:
            _dev(results[k], torch.float32, "res")
            if tuple(results[k].shape) != (E, N, dims[k][1], dims[k][2]):
                raise ValueError("res must be (E,N,h,w) NCHW")
    arr = lambda ptrs: (ctypes.c_void_p * n)(*ptrs)
    hw = (ctypes.c_int * n)(*[h * w for _, h, w in dims])
    _call("eod_project_fuse_levels", n, arr([lv.data_ptr() for lv in levels]), arr([w.data_ptr() for w in w_splits]),
          arr([None if b is None else b.data_ptr() for b in biases]), None if results is None else arr([r.data_ptr() for r in results]),
          arr([o.data_ptr() for o in outs]), hw, float(weight), int(mode), E, K, N, int(variant), _stream())
    return outs
