"""Spatial feature memory: grid state + write/read on the B200 kernels.

Three host-side objects sit above the C ABI:

``EpisodeBatch``
    E independent episodes advanced in lock step (BASELINE config 2 "batched x64"): one launch per stage covers
    all E grids.  This is the throughput path the bench measures:
        project (depth, pose -> cell indices) -> read (pooled fp16 levels) -> write (features -> grid).

``HeightMaxBatch``
    E episodes of the SMNet height-max memory in lock step (BASELINE configs[2]): per frame a contest of the frame's pixels
    for the highest point of every cell and the 'replace' update of the cells it raised.

``SpatialFeatureMemory``
    Single-episode mirror of the memory methods of ``CustomRCNNRecurrent``
    (detic/modeling/meta_arch/custom_rcnn.py:470-477, 681-936, 1019-1042) with the reference's method names,
    argument meaning and state attributes (``implicit_memory``, ``observations``, ``semmap_features``,
    ``observation_count``), so the meta-architecture can delegate to it.

HBM layout per episode: ``sums`` (cells, C) fp32 row = cell ``z*map_w + x``; ``counts`` (cells) fp32;
``frame_cnt`` (cells) int32 scratch, all-zero between frames; ``norm16`` (cells, C) fp16 = the normalised table the
read gathers from, refreshed per frame for the visible cells only.  State never leaves the device.
"""
from __future__ import annotations

import os

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import ops
from ._lib import LAYOUT_CHW, LAYOUT_CHW_BF16, LAYOUT_CHW_F16, LAYOUT_HWC, ORDER_ZX, WRITE_AUTO, WRITE_DET, EodError


def _slot_workspace(slots: Optional[ops.ObjectSlots], E: int, n_cells: int, C: int, HW: int, sample_stride: int,
                    device: torch.device) -> ops.ObjectSlots:
    """``slots`` if it fits a frame of HW pixels sampled every ``sample_stride``-th, else a new workspace of the object write."""
    S = -(-HW // sample_stride)
    if slots is None or slots.S < S or slots.n_cells != n_cells:
        slots = ops.ObjectSlots(E, n_cells, C, S, device)
    return slots


def _write_objects(idx: torch.Tensor, samp: torch.Tensor, frame_cnt: torch.Tensor, slots: Optional[ops.ObjectSlots], sums: torch.Tensor,
                   box_features: torch.Tensor, n_obj: Optional[torch.Tensor], masks: Optional[torch.Tensor] = None,
                   mask_probs: Optional[torch.Tensor] = None, boxes: Optional[torch.Tensor] = None, mask_thresh: float = 0.5,
                   det_ws: Optional[ops.DetWorkspace] = None) -> None:
    """count -> object write -> flush of one frame into ``sums``, with the objects' ``masks``, or with their un-pasted
    ``mask_probs`` and ``boxes`` (pasted inside the write).  frame_cnt stays set for the finalize.
    det_ws: the deterministic write instead (count without the slot table, no flush; ``slots`` is unused)."""
    if det_ws is not None:
        ops.frame_count(idx, samp, frame_cnt, n_obj)
        if masks is not None:
            ops.write_objects_det(box_features, masks, n_obj, idx, samp, frame_cnt, sums, det_ws)
        else:
            ops.write_objects_pasted_det(box_features, mask_probs, boxes, n_obj, idx, samp, frame_cnt, sums, det_ws, mask_thresh)
        return
    ops.frame_count(idx, samp, frame_cnt, n_obj, slots)
    if masks is not None:
        ops.write_objects(box_features, masks, n_obj, idx, samp, slots)
    else:
        ops.write_objects_pasted(box_features, mask_probs, boxes, n_obj, idx, samp, slots, mask_thresh)
    ops.flush_slots(frame_cnt, slots, sums)


class EpisodeBatch:
    """E episodes in lock step.  ``step`` runs the frame on two internal streams so that independent stages overlap:

        geometry stream : project -> count -> expand                    -> read  (needs finalize of frame t-1)
        write stream    :                      write (needs expand)  -> finalize (needs read: it refreshes ``norm16``)

    The read (an L1/L2 gather) runs next to the HBM-bound write instead of in front of it, and with
    ``pipeline=True`` the geometry of frame t+1 runs under the write of frame t (index plane, per-frame counts and
    reciprocal divisors are double buffered).  Results are identical in either mode: the read of frame t always
    sees exactly the state finalised by frame t-1 (custom_rcnn.py:489-515).

    ``pipeline=False`` (default): fully stream-ordered for the caller - on return the caller's stream has been made
    to wait for everything ``step`` enqueued.
    ``pipeline=True``: the caller promises that the geometry inputs of a step - depth / pose / shifts / samp /
    ``proj_indices``, and in ``step_detections`` also the detection tensors and ``n_obj`` - are ready when the step is
    called: they are consumed ahead of the caller's stream (``inputs_ready=False`` drops the promise for one step: the
    geometry then waits for the caller's stream, the write of the previous frame still overlaps).  ``feat`` and every
    mask of ``step`` (``active``, ``reset_mask``, ``refresh_mask``) are ordered on the caller's stream in either mode; a
    step that takes ``active`` does not run ahead of it.  The returned levels are ordered on the caller's stream; grid
    state (``sums``, ``counts``, ``norm16``) must be read after ``join()``.

    In both modes a step's inputs may be overwritten, on the caller's stream, as soon as the NEXT step has returned.

    Lock-step batches of RAGGED episodes (the reference iterates sequences of different lengths one after the other,
    custom_rcnn.py:441-443): ``step(..., active=, reset_mask=, refresh_mask=)`` - slots whose episode has ended are
    skipped by the write (their grid is left alone), a slot that starts a sequence flagged ``memory_reset`` is cleared
    on its own (:470-477), and with ``read_frozen = True`` (TEST_TYPE longterm, :482-486) the fp16 read table is a
    snapshot that only ``refresh_mask`` brings up to date.
    """

    def __init__(self, n_episodes: int, map_w: int, map_h: int, channels: int, height: int = 480, width: int = 640,
                 device: torch.device = torch.device("cuda"), layout: int = LAYOUT_CHW, variant: int = WRITE_AUTO,
                 pipeline: bool = False, fp16_table: bool = True, object_variant: int = WRITE_AUTO):
        if torch.device(device).type != "cuda":
            raise EodError("EpisodeBatch needs a CUDA device (no CPU fallback)")
        if object_variant not in (WRITE_AUTO, WRITE_DET):
            raise ValueError(f"object_variant must be WRITE_AUTO or WRITE_DET, got {object_variant!r}")
        if variant == WRITE_DET and layout in (LAYOUT_CHW_BF16, LAYOUT_CHW_F16):
            raise EodError("variant=WRITE_DET has no deterministic write for 16-bit CHW features (use LAYOUT_HWC_BF16 / _HWC_F16 "
                           "channels-last features, or feed feat.float() with LAYOUT_CHW)")
        self.E, self.map_w, self.map_h, self.C, self.H, self.W = n_episodes, map_w, map_h, channels, height, width
        self.n_cells = map_w * map_h
        self.device, self.layout, self.variant, self.pipeline = torch.device(device), layout, variant, pipeline
        self.object_variant = object_variant
        z = dict(device=self.device)
        self.sums = torch.zeros((self.E, self.n_cells, self.C), dtype=torch.float32, **z)
        self.counts = torch.zeros((self.E, self.n_cells), dtype=torch.float32, **z)
        # always-current normalised fp16 copy of the grid (what create_implicit_memory + .half() would return); only
        # the rows of the cells visible in a frame change, and the write's post-pass refreshes exactly those
        # fp16_table=False drops it (a third of the grid's footprint: 84 instead of 56 resident 1000x1000x512 grids in 180 GB): the read
        # then normalises and rounds the fp32 rows it gathers (same bits, twice the gathered bytes); no longterm snapshot in that mode
        self.norm16 = torch.zeros((self.E, self.n_cells, self.C), dtype=torch.float16, **z) if fp16_table else None
        # per-frame planes, double buffered (frame t uses buffer t & 1)
        self._idx2 = [torch.zeros((self.E, height, width), dtype=torch.int32, **z) for _ in range(2)]
        self._frame_cnt2 = [torch.zeros((self.E, self.n_cells), dtype=torch.int32, **z) for _ in range(2)]
        self._pix_inv_n2: Optional[List[torch.Tensor]] = None      # (E,H,W) f32 reciprocal divisors, created on first use (pixel_divisors mode)
        self.levels = [torch.empty((self.E, height >> s, width >> s, self.C), dtype=torch.float16, **z) for s in (3, 4, 5)]
        self._k = 0
        self._t = 0
        with torch.cuda.device(self.device):
            self._geo = torch.cuda.Stream(priority=0)
            self._wr = torch.cuda.Stream(priority=-1)      # the HBM-bound stage gets the SMs first
        self._pre: Optional[torch.cuda.Stream] = None      # paste / sample stream of the object regime, created on first use
        self._obs2 = self._samp2 = None                    # its per-frame observed / sampled-pixel planes (E, H*W) u8, double buffered
        self._e_fin: Optional[torch.cuda.Event] = None
        self._e_read: Optional[torch.cuda.Event] = None
        self._sync_next = True
        self._slots: Optional[ops.ObjectSlots] = None      # workspace of write_objects, created on first use
        # workspace of the deterministic writes (variant=WRITE_DET and / or object_variant=WRITE_DET: one serves both)
        self._det_ws: Optional[ops.DetWorkspace] = None
        self.det_runs_per_episode = 0                      # 0: HW/4 runs per episode and frame (every object frame with sample_stride >= 4)
        # CHW write: True = the divisors 1/n_cell travel with the tile (expand_counts pre-pass + 4 B per pixel); False = the consumer
        # looks a group's divisor up in frame_cnt itself (one dependent L2 load per group, no pre-pass)
        # (round 2: with the pixels of a tile grouped by cell there are few look-ups, and the pre-pass plus its 158 MB per 64-episode
        # frame-step cost more than they saved: 16.8 k -> 17.6 k frames/s in the bench, same bits)
        self.pixel_divisors = os.environ.get("EOD_PIXEL_DIVISORS", "0") == "1"
        self.fused_count = os.environ.get("EOD_FUSED_COUNT", "1") != "0"      # dense step: eod_backproject_count instead of project + count
        self.read_frozen = False      # True: finalize leaves norm16 alone (longterm snapshot read); refresh_read() updates it
        self.stage_events = None      # dict(stage -> [(start, end) CUDA events]) when profiling is on

    # current frame's planes
    @property
    def idx(self) -> torch.Tensor:
        return self._idx2[self._k]

    @property
    def frame_cnt(self) -> torch.Tensor:
        return self._frame_cnt2[self._k]

    @property
    def pix_inv_n(self) -> torch.Tensor:
        if self._pix_inv_n2 is None:
            self._pix_inv_n2 = [torch.zeros((self.E, self.H, self.W), dtype=torch.float32, device=self.device) for _ in range(2)]
        return self._pix_inv_n2[self._k]

    @property
    def _per_pixel_divisors(self) -> bool:
        """The write takes its divisors from ``pix_inv_n`` (expand_counts pre-pass): only the TMA-staged CHW kernel does."""
        return self.variant != WRITE_DET and self.layout == LAYOUT_CHW and self.pixel_divisors

    def profile(self, on: bool = True) -> None:
        """Record a CUDA-event pair around every stage launch (on the stream it is launched on, no synchronisation added)."""
        self.stage_events = {"project": [], "read": [], "count": [], "expand": [], "write": [], "finalize": []} if on else None

    def _timed(self, stage: str, fn, *args, **kw):
        if self.stage_events is None:
            return fn(*args, **kw)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn(*args, **kw)
        b.record()
        self.stage_events[stage].append((a, b))
        return out

    def stage_ms(self) -> dict:
        """Mean launch duration per stage in ms (call after a synchronize)."""
        return {k: (sum(a.elapsed_time(b) for a, b in v) / len(v) if v else 0.0) for k, v in (self.stage_events or {}).items()}

    def join(self) -> None:
        """Make the caller's current stream wait for everything ``step`` has enqueued on the internal streams."""
        s0 = torch.cuda.current_stream(self.device)
        for ev in (self._e_read, self._e_fin):
            if ev is not None:
                s0.wait_event(ev)

    def reset(self, full: bool = False, mask: Optional[torch.Tensor] = None) -> None:
        """memory_reset (custom_rcnn.py:470-477) for every episode of the batch, or - ``mask`` (E) i32 - for the slots
        with mask[e] != 0 only.  Only rows of cells seen since the last reset can be non-zero, so by default just those
        are cleared (eod_reset_touched / eod_reset_episodes); ``full=True`` rewrites the whole grid (use it if the state
        tensors were modified from outside)."""
        self.join()
        if mask is not None:
            ops.reset_episodes(self.counts, self.sums, self.norm16, mask)
        elif full:
            self.sums.zero_()
            self.counts.zero_()
            if self.norm16 is not None:
                self.norm16.zero_()
            for f in self._frame_cnt2:
                f.zero_()
        else:
            ops.reset_touched(self.counts, self.sums, self.norm16)      # frame_cnt is all-zero between frames already
        self._sync_next = True        # the next step must not run ahead of these fills

    # ---- single stages on the caller's stream (serial use, tests) ------------------------------------------
    def project(self, depth: torch.Tensor, pose: torch.Tensor, shifts: torch.Tensor, intr: Sequence[float], cell: float,
                order: int = ORDER_ZX) -> torch.Tensor:
        """depth (E,H,W) f32, pose (E,12), shifts (E,6) -> self.idx (E,H,W) int32 (A2-A5)."""
        self._timed("project", ops.backproject_quantize, depth, pose, shifts, intr, cell, self.map_w, self.map_h, order,
                    out={"idx": self.idx})
        return self.idx

    def _geometry(self, depth, pose, shifts, intr, cell, order, proj_indices) -> None:
        if proj_indices is None:
            self.project(depth, pose, shifts, intr, cell, order)
        else:
            self._timed("project", self.idx.copy_, proj_indices.reshape(self.E, self.H, self.W))

    def set_indices(self, idx: torch.Tensor, validate: bool = True) -> None:
        """Use precomputed proj_indices (E,H,W) int32 / int64, as the reference does from memory_data/*.h5.  The plane is
        range-checked against this batch's grid (IndexError, one 4-byte read-back); validate=False only for planes that
        eod_backproject_quantize produced for this grid (they are clipped already)."""
        idx = idx.reshape(self.E, self.H, self.W)
        if validate:
            self.idx.copy_(ops.check_indices(idx.contiguous(), self.n_cells, want_i32=True))
        else:
            self.idx.copy_(idx)

    def refresh_read(self, mask: Optional[torch.Tensor] = None) -> None:
        """Bring the fp16 read table up to date with sums / counts for the slots with mask[e] != 0 (None = all): the
        'updated_memory = self.implicit_memory' of custom_rcnn.py:482-486 at the first frame of a sequence."""
        if self.norm16 is None:
            raise EodError("refresh_read: this batch keeps no fp16 read table (fp16_table=False)")
        self.join()
        ops.refresh_norm16(self.counts, self.sums, self.norm16, mask)
        self._sync_next = True

    def read(self) -> List[torch.Tensor]:
        """A10-A12 fused: [L0 (E,C,H/8,W/8), L1, L2] fp16 (channels_last memory)."""
        if self.norm16 is None:
            if self.read_frozen:
                raise EodError("read_frozen (TEST_TYPE longterm) needs the fp16 read table: construct the batch with fp16_table=True")
            return self._timed("read", ops.read_pool, self.sums, self.counts, self.idx, out=self.levels)
        return self._timed("read", ops.read_pool, self.norm16, None, self.idx, out=self.levels)

    def read_roi(self, boxes: torch.Tensor, batch_idx: torch.Tensor, pooled: int = 7) -> torch.Tensor:
        """Per-proposal map features of the CURRENT frame's levels (call after ``step`` / ``read``): boxes (R,4) f32 XYXY in image
        pixels, batch_idx (R) i32 slot of each box -> logical (R,C,pooled,pooled) f32 (see ops.read_roi / eod_read_roi)."""
        return ops.read_roi([l.permute(0, 3, 1, 2) for l in self.levels], boxes, batch_idx, pooled)

    def _count(self, samp: Optional[torch.Tensor], active: Optional[torch.Tensor] = None) -> None:
        self._timed("count", ops.frame_count, self.idx, samp, self.frame_cnt, active)
        if self._per_pixel_divisors:
            self._timed("expand", ops.expand_counts, self.idx, self.frame_cnt, self.pix_inv_n)

    def _det_workspace(self) -> ops.DetWorkspace:
        if self._det_ws is None:
            self._det_ws = ops.DetWorkspace(self.E, self.C, self.H * self.W, self.n_cells, self.device, self.det_runs_per_episode)
        return self._det_ws

    def _object_workspace(self, sample_stride: int) -> dict:
        """The workspace of this frame's object write, as the keywords of _write_objects: the deterministic write's
        (object_variant=WRITE_DET) or the slot table of the reduction-based one."""
        if self.object_variant == WRITE_DET:
            return dict(slots=None, det_ws=self._det_workspace())
        self._slots = _slot_workspace(self._slots, self.E, self.n_cells, self.C, self.H * self.W, sample_stride, self.device)
        return dict(slots=self._slots)

    def _write(self, feat: torch.Tensor, samp: Optional[torch.Tensor], active: Optional[torch.Tensor] = None) -> None:
        if self.variant == WRITE_DET:
            self._timed("write", ops.write_mean_det, feat, self.idx, samp, self.frame_cnt, self.sums, self._det_workspace(), self.layout, active)
            return
        self._timed("write", ops.write_mean, feat, self.idx, samp, self.frame_cnt, self.sums, self.layout, self.variant,
                    self.pix_inv_n if self._per_pixel_divisors else None, active)

    def _finalize(self) -> None:
        # read_frozen (TEST_TYPE longterm): counts only - the fp16 table the read gathers from is a snapshot
        if self.read_frozen or self.norm16 is None:
            self._timed("finalize", ops.finalize_counts, self.idx, self.frame_cnt, self.counts)
        else:
            self._timed("finalize", ops.finalize_counts, self.idx, self.frame_cnt, self.counts, None, self.sums, self.norm16)

    def write(self, feat: torch.Tensor, samp: Optional[torch.Tensor] = None, active: Optional[torch.Tensor] = None) -> None:
        """A7 + A8 for one frame of every episode: feat (E,C,H,W) [CHW] or (E,H,W,C) [HWC] fp32, (E,H,W,C) bf16 / fp16
        [LAYOUT_HWC_BF16 / LAYOUT_HWC_F16] or (E,C,H,W) bf16 / fp16 [LAYOUT_CHW_BF16 / LAYOUT_CHW_F16];
        samp (E,H,W) u8 selects the contributing pixels (None = all); active (E) i32: slots with active <= 0 are skipped."""
        self._count(samp, active)
        self._write(feat, samp, active)
        self._finalize()

    def write_objects(self, box_features: torch.Tensor, masks: torch.Tensor, n_obj: Optional[torch.Tensor] = None,
                      sample_stride: int = 8) -> None:
        """Object-feature regime (the reference's live path, custom_rcnn.py:681-743) for one frame of every episode,
        fused: box_features (E,Kmax,C) f32 (= 50*normalize(feat), :848), masks (E,Kmax,H,W) bool, n_obj (E) i32 kept
        detections per episode (None = Kmax).  Episodes with n_obj == 0 are skipped entirely, counts included (:686).
        With ``object_variant=WRITE_DET`` the write is the deterministic one (bitwise reproducible, see ops.write_objects_det)."""
        ws = self._object_workspace(sample_stride)
        observed = ops.masks_observed(masks, n_obj)
        samp = ops.sample_mask(observed, sample_stride)
        _write_objects(self.idx, samp, self.frame_cnt, ws["slots"], self.sums, box_features, n_obj, masks=masks, det_ws=ws.get("det_ws"))
        self._finalize()

    def write_detections(self, box_features: torch.Tensor, mask_probs: torch.Tensor, boxes: torch.Tensor,
                         n_obj: Optional[torch.Tensor] = None, sample_stride: int = 8, mask_thresh: float = 0.5) -> None:
        """write_objects taking the detector's un-pasted output (custom_rcnn.py:876-880): mask_probs (E,Kmax,S,S) f32 (the
        mask head's 28x28 probabilities), boxes (E,Kmax,4) f32 XYXY.  paste_masks_in_image is folded into the write: the
        (K,480,640) masks are never built - one pass ORs the pasted test into ``observed``, the write re-evaluates it for
        the sampled pixels only."""
        ws = self._object_workspace(sample_stride)
        _, observed = ops.paste_masks(mask_probs, boxes, (self.H, self.W), mask_thresh, n_obj, want_masks=False, want_observed=True)
        samp = ops.sample_mask(observed, sample_stride)
        _write_objects(self.idx, samp, self.frame_cnt, ws["slots"], self.sums, box_features, n_obj,
                       mask_probs=mask_probs, boxes=boxes, mask_thresh=mask_thresh, det_ws=ws.get("det_ws"))
        self._finalize()

    # ---- one frame, overlapped -------------------------------------------------------------------------------
    # The frame protocol that step and step_detections share, one helper per phase; each of the two lays its own stages out on the
    # streams between them.
    def _begin_frame(self, inputs_ready: bool, force_strict: bool) -> Tuple[torch.cuda.Stream, bool, torch.cuda.Event]:
        """Flip the double buffer and mark the caller's stream (``e_in``).  strict: this frame takes its inputs behind ``e_in``
        (not pipelined, first step after a reset / refresh / replay, ``inputs_ready=False`` or ``force_strict``)."""
        s0 = torch.cuda.current_stream(self.device)
        self._k = self._t & 1
        self._t += 1
        strict = (not self.pipeline) or self._sync_next or not inputs_ready or force_strict
        self._sync_next = False
        return s0, strict, s0.record_event()

    def _reset_refresh(self, e_in: torch.cuda.Event, reset_mask: Optional[torch.Tensor],
                       refresh_mask: Optional[torch.Tensor]) -> Optional[torch.cuda.Event]:
        """reset_mask / refresh_mask on the write stream, behind finalize of frame t-1 (same stream) and the caller's masks; the
        returned event orders this frame's read behind them."""
        if reset_mask is None and refresh_mask is None:
            return None
        with torch.cuda.stream(self._wr):
            self._wr.wait_event(e_in)
            if reset_mask is not None:
                ops.reset_episodes(self.counts, self.sums, self.norm16, reset_mask)
            if refresh_mask is not None and self.norm16 is not None:
                ops.refresh_norm16(self.counts, self.sums, self.norm16, refresh_mask)
            return self._wr.record_event()

    def _read_frame(self, strict: bool, e_in: torch.cuda.Event,
                    e_state: Optional[torch.cuda.Event]) -> Tuple[List[torch.Tensor], torch.cuda.Event]:
        """This frame's read on the geometry stream, after the geometry enqueued there: it sees the state finalised by frame t-1
        and this frame's reset / refresh."""
        with torch.cuda.stream(self._geo):
            if not strict:
                self._geo.wait_event(e_in)                 # the caller has consumed the previous frame's levels
            if self._e_fin is not None:
                self._geo.wait_event(self._e_fin)          # norm16 as finalised by frame t-1
            if e_state is not None:
                self._geo.wait_event(e_state)
            levels = self.read()
            return levels, self._geo.record_event()

    def _end_frame(self, s0: torch.cuda.Stream, e_read: torch.cuda.Event, wait_fin: bool,
                   inputs: Sequence[torch.Tensor]) -> torch.cuda.Event:
        """Finalize on the write stream after its stages, then order the levels on the caller's stream and, with ``wait_fin``,
        the whole frame; without it ``inputs`` stay allocated until the write stream is done with them."""
        with torch.cuda.stream(self._wr):
            self._wr.wait_event(e_read)                    # finalize rewrites the norm16 rows the read gathers from
            self._finalize()
            e_fin = self._wr.record_event()
        self._e_read, self._e_fin = e_read, e_fin
        s0.wait_event(e_read)
        if wait_fin:
            s0.wait_event(e_fin)
        else:
            for t in inputs:
                t.record_stream(self._wr)
        return e_fin

    def step(self, depth, pose, shifts, intr, cell, feat, samp=None, order: int = ORDER_ZX, *, active: Optional[torch.Tensor] = None,
             reset_mask: Optional[torch.Tensor] = None, refresh_mask: Optional[torch.Tensor] = None,
             inputs_ready: bool = True, proj_indices: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
        """One frame of the hot path for all E episodes, in the reference's order: the read of frame t sees
        the state written by frame t-1 (custom_rcnn.py:489-515).  See the class docstring for the stream layout and for which
        inputs ``inputs_ready`` covers.
        feat and active / reset_mask / refresh_mask ((E) i32 device tensors, ragged lock-step batches) are ordered on the caller's
        stream: reset_mask clears those slots BEFORE this frame's read (frame['memory_reset'], :470-477), refresh_mask then brings
        their fp16 read table up to date (read_frozen mode, :482-486), active <= 0 slots are neither counted nor written.
        proj_indices (E,H,W) int32: precomputed, range-checked cell indices (memory_data/*.h5) used instead of depth / pose."""
        # active is read by the count on the geometry stream AND by the write: both must see the caller's mask, so a step that
        # takes one runs its geometry behind the caller's stream
        s0, strict, e_in = self._begin_frame(inputs_ready, force_strict=active is not None)
        e_state = self._reset_refresh(e_in, reset_mask, refresh_mask)
        with torch.cuda.stream(self._geo):
            if strict:
                self._geo.wait_event(e_in)                 # inputs (and a preceding reset) are ordered on the caller's stream
            if samp is None and proj_indices is None and self.fused_count and ops.backproject_count_supported(self.H, self.W):
                # dense frame, geometry computed here: the per-cell pixel counts are taken inside the back-projection launch
                self._timed("project", ops.backproject_count, depth, pose, shifts, intr, cell, self.map_w, self.map_h, self.idx, self.frame_cnt,
                            active, order)
                if self._per_pixel_divisors:
                    self._timed("expand", ops.expand_counts, self.idx, self.frame_cnt, self.pix_inv_n)
            else:
                self._geometry(depth, pose, shifts, intr, cell, order, proj_indices)
                self._count(samp, active)
            e_geo = self._geo.record_event()
        levels, e_read = self._read_frame(strict, e_in, e_state)
        with torch.cuda.stream(self._wr):
            self._wr.wait_event(e_in)                      # feat is outside the pipeline promise: always ordered on the caller's stream
            self._wr.wait_event(e_geo)
            self._write(feat, samp, active)
        self._end_frame(s0, e_read, wait_fin=not self.pipeline, inputs=(feat,))
        return levels

    def step_detections(self, depth, pose, shifts, intr, cell, box_features, mask_probs, boxes, n_obj=None, sample_stride: int = 8,
                        mask_thresh: float = 0.5, order: int = ORDER_ZX, *, reset_mask: Optional[torch.Tensor] = None,
                        refresh_mask: Optional[torch.Tensor] = None, proj_indices: Optional[torch.Tensor] = None,
                        inputs_ready: bool = True) -> List[torch.Tensor]:
        """One frame of the reference's LIVE regime for all E episodes (custom_rcnn.py:489-515 with :876-936): read of the
        state left by frame t-1, then the write of this frame's kept detections (un-pasted 28x28 mask probabilities + boxes).
        Three streams, stream-ordered for the caller on entry and exit:

            geometry stream : project ---------------------> read   (needs finalize of frame t-1)
            paste stream    : paste/observed -> sample
            write stream    : (project, sample) count -> write_objects -> flush -> (read) finalize

        The mask pasting and the sampling scan depend on neither the geometry nor the state, and the issue-bound read runs next to
        the latency-bound object write instead of in front of it.  With ``pipeline=True`` the caller's stream is not made to wait for
        this frame's finalize, so project / paste / sample of frame t+1 run under write / flush / finalize of frame t (index plane and
        per-frame counts are double buffered); the state chain read(t) -> finalize(t) -> read(t+1) is what remains serial.  The
        promise of ``pipeline=True`` covers depth / pose / shifts / proj_indices AND box_features / mask_probs / boxes / n_obj
        (``inputs_ready=False`` drops it for one call); reset_mask / refresh_mask are ordered on the caller's stream, as in ``step``.
        A step's inputs may be overwritten once the next step has returned.  Slots whose episode has ended pass n_obj == 0
        (nothing is written, :686).  ``object_variant=WRITE_DET``: the write is the deterministic one (count without slots, no flush)."""
        capturing = torch.cuda.is_current_stream_capturing()
        if self._pre is None:
            with torch.cuda.device(self.device):
                self._pre = torch.cuda.Stream(priority=0)
        ws = self._object_workspace(sample_stride)
        # a side stream joins a capture only by waiting for the capturing stream
        s0, strict, e_in = self._begin_frame(inputs_ready, force_strict=capturing)
        e_state = self._reset_refresh(e_in, reset_mask, refresh_mask)
        with torch.cuda.stream(self._pre):
            if strict:
                self._pre.wait_event(e_in)
            # per-frame planes owned by the batch (double buffered like the index plane): tensors allocated here on the paste stream
            # and consumed on the write stream would make the caching allocator defer their reuse and fall back to cudaMalloc
            if self._obs2 is None:
                self._obs2 = [torch.empty((self.E, self.H * self.W), dtype=torch.uint8, device=self.device) for _ in range(2)]
                self._samp2 = [torch.empty((self.E, self.H * self.W), dtype=torch.uint8, device=self.device) for _ in range(2)]
                self._fin2 = [None, None]
            if self._fin2[self._k] is not None and not capturing:      # a capture cannot wait for an event recorded outside it
                self._pre.wait_event(self._fin2[self._k])      # the write side of frame t-2 has finished with this half
            _, observed = ops.paste_masks(mask_probs, boxes, (self.H, self.W), mask_thresh, n_obj, want_masks=False, want_observed=True,
                                          observed_out=self._obs2[self._k])
            samp = ops.sample_mask(observed, sample_stride, self._samp2[self._k])
            e_samp = self._pre.record_event()
        with torch.cuda.stream(self._geo):
            if strict:
                self._geo.wait_event(e_in)
            self._geometry(depth, pose, shifts, intr, cell, order, proj_indices)
            e_geo = self._geo.record_event()
        levels, e_read = self._read_frame(strict, e_in, e_state)
        with torch.cuda.stream(self._wr):
            if strict:
                self._wr.wait_event(e_in)                  # the detection inputs are inside the pipeline promise
            self._wr.wait_event(e_geo)
            self._wr.wait_event(e_samp)
            _write_objects(self.idx, samp, self.frame_cnt, ws["slots"], self.sums, box_features, n_obj,
                           mask_probs=mask_probs, boxes=boxes, mask_thresh=mask_thresh, det_ws=ws.get("det_ws"))
        # a capture must join every side stream back into the capturing stream
        e_fin = self._end_frame(s0, e_read, wait_fin=not self.pipeline or capturing,
                                inputs=(box_features, mask_probs, boxes) + ((n_obj,) if n_obj is not None else ()))
        self._fin2[self._k] = None if capturing else e_fin      # an event recorded in a capture cannot be waited for outside it
        return levels

    def capture_step_detections(self, depth, pose, shifts, intr, cell, box_features, mask_probs, boxes, n_obj=None, **kw) -> "GraphedDetections":
        """Capture ``step_detections`` for this shape into ONE CUDA graph (the online single-robot loop, robot_demo.py:559-566: a frame
        is ~10 small launches on two streams, so one episode is bound by launch overhead, not by the kernels).  The arguments are
        example inputs of the shapes / dtypes every later frame will have; they are copied into static buffers owned by the returned
        object, whose ``__call__(depth, pose, shifts, box_features, mask_probs, boxes, n_obj)`` copies a frame's inputs in and replays
        the graph.  Results are identical to the eager call (same kernels, same order).  Per-frame keywords (reset_mask, refresh_mask,
        proj_indices) raise ValueError: a graph would apply them at every replay."""
        return GraphedDetections(self, depth, pose, shifts, intr, cell, box_features, mask_probs, boxes, n_obj, kw)


class GraphedDetections:
    """``EpisodeBatch.step_detections`` of one fixed shape as a CUDA graph (see ``capture_step_detections``).  The three pooled
    levels returned by a call live in static buffers: they are valid until the next call."""

    _KEYS = ("depth", "pose", "shifts", "box_features", "mask_probs", "boxes", "n_obj")

    # per-frame inputs that the graph would bake in: the warm-up frame would apply them once and every replay again
    _PER_FRAME = ("reset_mask", "refresh_mask", "proj_indices")

    def __init__(self, batch: "EpisodeBatch", depth, pose, shifts, intr, cell, box_features, mask_probs, boxes, n_obj, kw):
        bad = [k for k in self._PER_FRAME if k in kw]
        if bad:
            raise ValueError(f"capture_step_detections: {', '.join(bad)} cannot be captured (a replay would reuse it every frame); "
                             f"reset / refresh with an eager step or EpisodeBatch.reset / refresh_read between replays")
        self.batch = batch
        given = dict(zip(self._KEYS, (depth, pose, shifts, box_features, mask_probs, boxes, n_obj)))
        self.static = {k: (None if v is None else v.detach().to(batch.device).clone().contiguous()) for k, v in given.items()}
        st = self.static
        args = (st["depth"], st["pose"], st["shifts"], intr, cell, st["box_features"], st["mask_probs"], st["boxes"], st["n_obj"])
        with torch.cuda.device(batch.device):
            batch.join()
            torch.cuda.current_stream().synchronize()
            # everything the step allocates lazily (slot or deterministic-write workspace, the library's per-device state) must exist
            # before the capture; the
            # warm-up frame runs with n_obj = 0, which writes nothing and leaves the grid as it is
            zero_obj = torch.zeros((batch.E,), dtype=torch.int32, device=batch.device)
            batch.step_detections(*args[:8], zero_obj, **kw)
            batch.join()
            torch.cuda.current_stream().synchronize()
            batch._t -= 1                                   # the warm-up frame does not count
            batch._e_fin = batch._e_read = None             # no dependency on work recorded outside the capture
            self.graph = torch.cuda.CUDAGraph()
            side = torch.cuda.Stream()
            with torch.cuda.graph(self.graph, stream=side):
                self.levels = batch.step_detections(*args, **kw)
            batch._t -= 1                                   # capturing enqueues nothing
            batch._e_fin = batch._e_read = None             # replays are ordered by the stream they are launched on
        self._k = batch._k                                  # the double-buffer half the graph was captured on

    def __call__(self, depth, pose, shifts, box_features, mask_probs, boxes, n_obj=None):
        b = self.batch
        for k, v in zip(self._KEYS, (depth, pose, shifts, box_features, mask_probs, boxes, n_obj)):
            dst = self.static[k]
            if dst is None:
                if v is not None:
                    raise ValueError(f"{k}: the graph was captured without this input")
                continue
            if v is None:
                raise ValueError(f"{k}: the graph was captured with this input")
            if v.data_ptr() != dst.data_ptr():
                dst.copy_(v, non_blocking=True)
        b.join()                                            # an eager step before this replay may still be running on the side streams
        b._e_fin = b._e_read = None
        b._k = self._k
        b._t += 1
        self.graph.replay()
        b._sync_next = True                                 # the next eager step must not run ahead of this replay (same planes)
        return self.levels


class HeightMaxBatch:
    """E episodes of the SMNet height-max memory (bytecode-only SMNet.encode, SURVEY 8a row A7') in lock step: BASELINE configs[2].

    Per episode: ``state`` (cells, C_mem) f32, ``height_map`` (cells) f32 = highest inlier height + 1000 seen so far (0 before the
    first), ``observed`` (cells) u8.  A frame is the contest of its [::pix_stride, ::pix_stride] pixels for the highest point of every
    cell - geometry from depth (computed in registers) or from precomputed height / idx / outlier planes - and the update of the cells
    it raised: the winner pixel's feature row is copied into ``state`` ('replace' without a layer), or, with ``linlayer=(weight (C_mem, C)
    f32, bias (C_mem,) | None)``, ``state[cell] = weight @ row + bias`` on the tensor cores (fp32 features only).  Results equal
    ``ops.backproject_quantize`` + ``ops.write_max`` (``write_max_linear``) over the same frames bit for bit.

    ``feat`` is (E,C,H,W) or (E,H,W,C) in the dtype of ``layout`` (LAYOUT_CHW / _HWC fp32, the _BF16 / _F16 variants widened exactly).
    Everything is ordered on the caller's stream, inputs included."""

    def __init__(self, n_episodes: int, map_w: int, map_h: int, channels: int, height: int = 480, width: int = 640,
                 device: torch.device = torch.device("cuda"), layout: int = LAYOUT_CHW, linlayer: Optional[Tuple[torch.Tensor, Optional[torch.Tensor]]] = None,
                 pix_stride: int = 1, order: int = ORDER_ZX, z_clip: float = 0.5, depth_div: float = 1000.0):
        if torch.device(device).type != "cuda":
            raise EodError("HeightMaxBatch needs a CUDA device (no CPU fallback)")
        if linlayer is not None and layout not in (LAYOUT_CHW, LAYOUT_HWC):
            raise EodError("HeightMaxBatch: the linlayer update takes fp32 features (LAYOUT_CHW / LAYOUT_HWC)")
        self.E, self.map_w, self.map_h, self.C, self.H, self.W = n_episodes, map_w, map_h, channels, height, width
        self.n_cells = map_w * map_h
        self.device, self.layout, self.pix_stride, self.order, self.z_clip, self.depth_div = torch.device(device), layout, pix_stride, order, z_clip, depth_div
        self.linlayer = None
        c_mem = channels
        if linlayer is not None:
            weight, bias = linlayer
            if weight.dim() != 2 or weight.shape[1] != channels:
                raise ValueError(f"linlayer weight must be (C_mem, {channels})")
            self.linlayer = (weight.to(self.device, torch.float32).contiguous(),
                             None if bias is None else bias.to(self.device, torch.float32).contiguous())
            c_mem = weight.shape[0]
        z = dict(device=self.device)
        self.state = torch.zeros((self.E, self.n_cells, c_mem), dtype=torch.float32, **z)
        self.height_map = torch.zeros((self.E, self.n_cells), dtype=torch.float32, **z)
        self.observed = torch.zeros((self.E, self.n_cells), dtype=torch.uint8, **z)
        lattice = -(-height // pix_stride) * -(-width // pix_stride)
        self.scratch = ops.HeightMaxScratch(self.E, self.n_cells, lattice, self.device)

    def reset(self, mask: Optional[torch.Tensor] = None) -> None:
        """memory reset of every episode, or - ``mask`` (E) i32 - of the slots with mask[e] != 0 only."""
        if mask is None:
            mask = torch.ones((self.E,), dtype=torch.int32, device=self.device)
        ops.heightmax_reset(self.height_map, self.observed, self.state, mask)

    def step(self, feat: torch.Tensor, *, depth: Optional[torch.Tensor] = None, pose: Optional[torch.Tensor] = None,
             shifts: Optional[torch.Tensor] = None, intr: Optional[Sequence[float]] = None, cell: Optional[float] = None,
             height: Optional[torch.Tensor] = None, idx: Optional[torch.Tensor] = None, outlier: Optional[torch.Tensor] = None,
             active: Optional[torch.Tensor] = None, reset_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One frame of every episode.  Geometry: depth (E,H,W) f32 metres or uint16 (/ depth_div) + pose (E,12) + shifts (E,6) + intr +
        cell, OR precomputed planes height (E,H,W) f32 + idx (E,H,W) i32 cell ids in [0, cells) + outlier (E,H,W) u8 | None.
        active (E) i32: slots with active <= 0 read nothing and keep their state; reset_mask (E) i32: those slots are cleared before
        the frame.  Returns the device count (1,) i32 of cells raised this frame over all episodes (valid until the next step)."""
        geo = depth if depth is not None else height
        if geo is None or tuple(geo.shape) != (self.E, self.H, self.W):
            raise ValueError(f"HeightMaxBatch.step: depth or height of shape {(self.E, self.H, self.W)} is required")
        # features are checked before the contest: a refused update would leave the frame's keys in the scratch
        if ops._feat_hw(feat, self.layout, self.E, self.C, "HeightMaxBatch.step") != (self.H, self.W):
            raise ValueError(f"HeightMaxBatch.step: feat must cover H={self.H}, W={self.W}")
        if self.C % 4 or self.state.shape[2] % 4 or feat.data_ptr() % 16 or self.state.data_ptr() % 16:
            raise EodError("HeightMaxBatch.step: feature and state rows need C % 4 == 0 and 16-byte aligned tensors")
        if reset_mask is not None:
            ops.heightmax_reset(self.height_map, self.observed, self.state, reset_mask)
        if depth is not None:
            if height is not None or idx is not None or outlier is not None:
                raise ValueError("HeightMaxBatch.step: give depth + pose + shifts + intr + cell OR height + idx (+ outlier), not both")
            if pose is None or shifts is None or intr is None or cell is None:
                raise ValueError("HeightMaxBatch.step: depth needs pose, shifts, intr and cell")
            ops.heightmax_contest_depth(depth, pose, shifts, intr, cell, self.map_w, self.map_h, self.scratch, active, self.pix_stride,
                                        self.order, self.z_clip, self.depth_div)
        else:
            if idx is None:
                raise ValueError("HeightMaxBatch.step: height needs idx")
            ops.heightmax_contest_planes(height, idx, outlier, self.scratch, active, self.pix_stride)
        return ops.heightmax_update(feat, self.layout, self.scratch, self.height_map, self.observed, self.state, self.linlayer)


class SpatialFeatureMemory:
    """Reference-facing, one episode in flight (like one ``CustomRCNNRecurrent`` instance).

    semmap_gt_info / replica_map_info: the dicts of SMNet/semmap_GT_info.json / replica_map_info.json used by the map
    size lookup of custom_rcnn.py:704-729; downsample = 10 (:364).
    """

    def __init__(self, mem_feat_dim: int = 512, device: torch.device = torch.device("cuda"), test_type: str = "default",
                 semmap_gt_info: Optional[dict] = None, replica_map_info: Optional[dict] = None, downsample: int = 10,
                 sample_stride: int = 8, height: int = 480, width: int = 640, fused_write: bool = True,
                 zs_weight: Optional[torch.Tensor] = None, obs_score_thresh: float = 0.4, n_semmap_classes: int = 20):
        if torch.device(device).type != "cuda":
            raise EodError("SpatialFeatureMemory needs a CUDA device (no CPU fallback)")
        self.C, self.device, self.test_type = mem_feat_dim, torch.device(device), test_type
        self.fused_write = fused_write      # False: materialise image_features like the reference (box_to_image_features)
        # explicit semantic map (custom_rcnn.py:747-756,938-978): maintained when the CLIP classifier table is given
        self.zs_weight = None if zs_weight is None else zs_weight.to(self.device, torch.float32).contiguous()   # (C, K)
        self.obs_score_thresh, self.n_semmap_classes = obs_score_thresh, n_semmap_classes       # MODEL.MEMORY_OBS_SCORE_THRESH
        self._intensity: Optional[torch.Tensor] = None
        self._cls: Optional[torch.Tensor] = None
        self.semmap_gt_info, self.replica_map_info = semmap_gt_info or {}, replica_map_info or {}
        self.downsample, self.sample_stride, self.H, self.W = downsample, sample_stride, height, width
        self.validate_indices = True                            # range-check externally supplied proj_indices (see _idx32)
        self.implicit_memory: Optional[torch.Tensor] = None     # (cells, C) f32 sums        (custom_rcnn.py:476,759)
        self.observations: Optional[torch.Tensor] = None        # (cells,)  f32 counts      (:477,760)
        self._frame_cnt: Optional[torch.Tensor] = None
        self._touched: Optional[torch.Tensor] = None
        self._slots: Optional[ops.ObjectSlots] = None

    # ---- state ---------------------------------------------------------------------------------------
    def reset(self, n_cells: int) -> None:
        """frame['memory_reset'] (custom_rcnn.py:470-477); the state is created on the device."""
        self.implicit_memory = torch.zeros((n_cells, self.C), dtype=torch.float32, device=self.device)
        self.observations = torch.zeros((n_cells,), dtype=torch.float32, device=self.device)
        self._frame_cnt = torch.zeros((1, n_cells), dtype=torch.int32, device=self.device)
        self._touched = torch.zeros((1, n_cells), dtype=torch.uint8, device=self.device)
        self._intensity = torch.zeros((1, n_cells), dtype=torch.float32, device=self.device)
        self._cls = torch.zeros((1, n_cells), dtype=torch.int32, device=self.device)     # argmax of all-zero logits is class 0

    def map_dims(self, sequence_name: str) -> Tuple[int, int]:
        """(map_w, map_h) as custom_rcnn.py:704-729 resolves them (MP3D table, Replica table, else 200x200)."""
        try:
            map_w, _, map_h = self.semmap_gt_info[sequence_name[0:13]]["dim"]
            return math.ceil(map_w / self.downsample), math.ceil(map_h / self.downsample)
        except KeyError:
            try:
                parts = sequence_name.split("_")
                if len(parts) == 5:
                    env = "_".join((parts[0] + "_" + parts[1] + "_" + parts[2], parts[3]))
                elif len(parts) == 4:
                    env = "_".join((parts[0] + "_" + parts[1], parts[2]))
                else:
                    env = parts[0] + "_" + parts[1]
                map_w, _, map_h = self.replica_map_info[env]["dim"]
                return map_w, map_h
            except Exception:
                return 200, 200

    @property
    def semmap_features(self) -> Optional[torch.Tensor]:
        """(1, C, map_h, map_w) view of the sums (custom_rcnn.py:731-742) when the map dims are known."""
        return None if self.implicit_memory is None or not hasattr(self, "_dims") else \
            self.implicit_memory.reshape(self._dims[1], self._dims[0], self.C).permute(2, 0, 1).unsqueeze(0)

    @property
    def observation_count(self) -> Optional[torch.Tensor]:
        return None if self.observations is None or not hasattr(self, "_dims") else \
            self.observations.reshape(1, self._dims[1], self._dims[0])

    @property
    def semmap(self) -> Optional[torch.Tensor]:
        """(cells,) int32 explicit semantic map as custom_rcnn.py:756 leaves it in ``self.semmap`` (class id, -1 below the
        observation-intensity threshold); None without a classifier table.  Stays on the device."""
        if self.zs_weight is None or self._intensity is None:
            return None
        return ops.semmap_decode(self._intensity, self._cls, self.obs_score_thresh)[0]

    def _finalize(self, idx: torch.Tensor) -> None:
        """End of a write into the live state: the explicit map of the cells the frame saw, then their counts (_frame_cnt back to zero)."""
        if self.zs_weight is not None:
            ops.semmap_update(self._frame_cnt, self.observations.unsqueeze(0), self.implicit_memory.unsqueeze(0), self.zs_weight,
                              self.n_semmap_classes, self._intensity, self._cls)
        ops.finalize_counts(idx, self._frame_cnt, self.observations.unsqueeze(0))

    # ---- read ----------------------------------------------------------------------------------------
    def create_implicit_memory(self, frame: Dict) -> Tuple[torch.Tensor, torch.Tensor]:
        """custom_rcnn.py:762-775,823: (memory / observations where observations > 1, proj_indices)."""
        mem = torch.as_tensor(frame["memory"]).to(self.device, torch.float32).contiguous()
        obs = torch.as_tensor(frame["observations"]).to(self.device, torch.float32).contiguous()
        return ops.normalize_memory(mem, obs), frame["proj_indices"]

    def create_explicit_memory(self, frame: Dict, clip_embeddings: torch.Tensor, semmap: Optional[torch.Tensor] = None
                               ) -> Tuple[torch.Tensor, torch.Tensor, Optional[torch.Tensor]]:
        """MODEL.MEMORY_TYPE 'explicit_map' (SMNet/loader.py:233-246,298; ``create_explicit_memory`` of the older custom_rcnn revision,
        bytecode listing create_explicit_memory_custom_rcnn_py39.txt, src lines 1400-1411): the memory the read gathers from is the class
        table with a zero row in front, ``memory = [0; clip_embeddings]`` (K+1, C), and a pixel's index is the class of the cell it
        falls into, ``proj_indices := (semmap + 1)[proj_indices]`` (-1 'empty' -> row 0).  semmap: (cells,) int class map (-1 = empty);
        default = the live explicit map of this memory (A14, ``self.semmap``).  Returns (memory fp32 (K+1,C), proj_indices int32
        (H,W), ego_observations = observations[proj_indices] or None) - feed the first two to ``read_levels`` / ``MemoryFusion``
        exactly like an implicit memory."""
        table = torch.as_tensor(clip_embeddings).to(self.device, torch.float32)
        memory = torch.cat([torch.zeros((1, table.shape[1]), dtype=torch.float32, device=self.device), table], 0).contiguous()
        sm = self.semmap if semmap is None else torch.as_tensor(semmap).to(self.device)
        if sm is None:
            raise EodError("create_explicit_memory: no semantic map (pass semmap= or construct the memory with zs_weight)")
        if sm.dtype not in (torch.int32, torch.int64):
            sm = sm.to(torch.int64)
        idx = self._index_plane(frame["proj_indices"]).contiguous()
        proj = ops.remap_indices(idx, sm.reshape(-1).contiguous(), memory.shape[0], add=1)
        obs = frame.get("observations")
        ego_obs = None if obs is None else torch.as_tensor(obs).to(self.device).reshape(-1)[idx.long()]
        return memory, proj, ego_obs

    def preprocess_spatial_memory(self, batched_inputs: Sequence[Dict]):
        """custom_rcnn.py:1019-1042: lists of (memory f16, proj_indices int64, observations)."""
        memory, projection, observations = [], [], []
        for x in batched_inputs:
            m = torch.as_tensor(x["memory"]).to(self.device)
            p = self._index_plane(x["proj_indices"])
            o = x.get("observations")
            if o is not None and not torch.is_tensor(o):
                o = torch.as_tensor(o).to(self.device).to(torch.half)
            memory.append(m.to(torch.half))
            projection.append(p.to(torch.long))
            observations.append(o)
        return memory, projection, observations

    def read_levels(self, proj_indices: torch.Tensor, memory: Optional[torch.Tensor] = None,
                    observations: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
        """Fused A10-A12 for this episode: the three pooled fp16 levels (1,C,h,w) from the live state (or from
        an explicit memory table: fp32 sums + observations, or an already normalised fp16 table)."""
        table = self.implicit_memory if memory is None else memory
        counts = self.observations if memory is None else observations
        if table.dtype == torch.float16:
            counts = None
        idx = self._index_plane(proj_indices).unsqueeze(0).contiguous()
        if self.validate_indices:
            ops.check_indices(idx, table.shape[0])
        return ops.read_pool(table.unsqueeze(0).contiguous(), None if counts is None else counts.unsqueeze(0).contiguous(), idx)

    # ---- write ---------------------------------------------------------------------------------------
    def box_to_image_features(self, box_features: torch.Tensor, masks: torch.Tensor):
        """custom_rcnn.py:884-901 (bit-exact)."""
        return ops.box_to_image_features(box_features.to(self.device, torch.float32).contiguous(),
                                         masks.to(self.device).contiguous())

    def _index_plane(self, proj_indices) -> torch.Tensor:
        """An externally supplied plane (h5 / npz proj_indices, (H,W) or (H,W,1)) on the device as int32 / int64 (H,W)."""
        p = torch.as_tensor(proj_indices).to(self.device)
        if p.dim() == 3 and p.shape[-1] == 1:
            p = p.squeeze(2)
        if p.dtype not in (torch.int32, torch.int64):
            p = p.to(torch.int64)
        return p

    def _idx32(self, proj_indices: torch.Tensor, n_cells: Optional[int] = None) -> torch.Tensor:
        """(1, HW) int32 view of an externally supplied plane (see ``_index_plane``).  With n_cells the ids are
        range-checked on the device (IndexError like the reference's gather, one 4-byte read-back); ``validate_indices =
        False`` on the instance skips that for callers whose planes come from eod_backproject_quantize for this very grid."""
        p = self._index_plane(proj_indices)
        if n_cells is not None and self.validate_indices:
            return ops.check_indices(p.contiguous(), n_cells, want_i32=True).reshape(1, -1)
        return p.to(torch.int32).reshape(1, -1).contiguous()

    def _feat_in(self, image_features: torch.Tensor, layout: int, C: int) -> Tuple[torch.Tensor, int]:
        """Image features on the device, contiguous, and the layout the write takes them in: bf16 / fp16 stay 16-bit (half the bytes
        of the write's feature stream, same sums), any other dtype - or a 16-bit image whose rows are not 16-byte aligned
        (H*W % 8 != 0) - is cast to fp32 as before."""
        x = torch.as_tensor(image_features)
        if x.dtype not in (torch.bfloat16, torch.float16) or (x.numel() // C) % 8:
            return x.to(self.device, torch.float32).contiguous(), layout
        return x.to(self.device).contiguous(), ops.layout_for_dtype(layout, x.dtype)

    def _fresh_mean(self, feat: torch.Tensor, idx: torch.Tensor, samp: Optional[torch.Tensor], n_cells: int, C: int,
                    layout: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """Per-cell mean of one frame into a fresh zero table, the live state untouched: (table (cells,C) f32, observed_mem
        (cells,) bool = the cells the frame wrote)."""
        table = torch.zeros((1, n_cells, C), dtype=torch.float32, device=self.device)
        cnt = torch.zeros((1, n_cells), dtype=torch.int32, device=self.device)
        touched = torch.zeros((1, n_cells), dtype=torch.uint8, device=self.device)
        dummy_counts = torch.zeros((1, n_cells), dtype=torch.float32, device=self.device)
        ops.frame_count(idx, samp, cnt)
        ops.write_mean(feat, idx, samp, cnt, table, layout)
        ops.finalize_counts(idx, cnt, dummy_counts, touched)
        return table[0], touched[0].view(torch.bool)

    def project_image_features(self, image_features: torch.Tensor, observed_pixels: torch.Tensor,
                               proj_indices: Sequence[torch.Tensor], memory: Sequence[torch.Tensor]):
        """custom_rcnn.py:903-936: (mean (M,C) f32 in ascending cell order, observed_mem (cells,) bool).  bf16 / fp16 images are
        written as they are (16-bit CHW layout, widened exactly in the kernel: the reference sums ``float()`` of them, :930)."""
        n_cells = memory[0].shape[0]
        C = image_features.shape[1]
        idx = self._idx32(proj_indices[0], n_cells)
        samp = ops.sample_mask(observed_pixels.to(self.device).reshape(1, -1).view(torch.uint8).contiguous(), self.sample_stride)
        feat, layout = self._feat_in(image_features, LAYOUT_CHW, C)
        mean, observed_mem = self._fresh_mean(feat.reshape(1, C, -1), idx, samp, n_cells, C, layout)
        return mean[observed_mem], observed_mem

    def update_implicit_memory(self, inference_results, proj_indices: torch.Tensor, memory: torch.Tensor, frame: Dict,
                               visualise: bool = False) -> None:
        """custom_rcnn.py:681-760.  ``inference_results`` is what ``inference_with_proposals`` returns
        (:882): None (no kept detection -> no write at all, :686) or (boxes, box_features (K,C), masks
        (K,H,W) bool, pred_instances); floating-point masks (K,S,S) are taken as the mask head's probabilities BEFORE
        paste_masks_in_image (:880) and pasted here with ``boxes`` (K,4).  Sums and visibility counts are accumulated in place on the device."""
        if inference_results is None:
            return
        boxes, box_features, masks, _ = inference_results
        if self.implicit_memory is None or self.implicit_memory.shape[0] != memory.shape[0]:
            self.reset(memory.shape[0])
        self._dims = self.map_dims(frame.get("sequence_name", ""))
        if masks.is_floating_point():
            # un-pasted mask-head output (K,S,S) with its boxes: paste_masks_in_image (:880) folded into the write
            if self.fused_write:
                self.write_detections(box_features, masks, boxes, proj_indices)
                return
            masks = self.paste_masks_in_image(masks, boxes, (self.H, self.W))
        if self.fused_write:
            self.write_object_features(box_features, masks, proj_indices)
        else:
            image_features, observed = self.box_to_image_features(box_features, masks)
            self.write_image_features(image_features, observed, proj_indices)

    def paste_masks_in_image(self, masks: torch.Tensor, boxes: torch.Tensor, image_shape: Tuple[int, int],
                             threshold: float = 0.5) -> torch.Tensor:
        """detectron2's paste_masks_in_image as the reference calls it (custom_rcnn.py:880): masks (K,S,S) f32
        probabilities, boxes (K,4) f32 XYXY -> (K,H,W) bool; bit-exact with torch-CPU."""
        if masks.shape[0] == 0:
            return torch.zeros((0,) + tuple(image_shape), dtype=torch.bool, device=self.device)
        m, _ = ops.paste_masks(masks.to(self.device, torch.float32).contiguous().unsqueeze(0),
                               boxes.to(self.device, torch.float32).contiguous().unsqueeze(0), image_shape, threshold)
        return m[0]

    def write_detections(self, box_features: torch.Tensor, mask_probs: torch.Tensor, boxes: torch.Tensor,
                         proj_indices: torch.Tensor, mask_thresh: float = 0.5) -> None:
        """custom_rcnn.py:876-880 + 690-701,738-743 in one go: the kept detections' (K,S,S) mask probabilities and boxes are
        pasted on the fly (no (K,H,W) masks, no (1,C,H,W) image)."""
        idx = self._idx32(proj_indices, self.implicit_memory.shape[0]).view(1, self.H, self.W)
        bf = box_features.to(self.device, torch.float32).contiguous().unsqueeze(0)
        mp = mask_probs.to(self.device, torch.float32).contiguous().unsqueeze(0)
        bx = boxes.to(self.device, torch.float32).contiguous().unsqueeze(0)
        self._slots = _slot_workspace(self._slots, 1, self.implicit_memory.shape[0], self.C, self.H * self.W, self.sample_stride, self.device)
        _, observed = ops.paste_masks(mp, bx, (self.H, self.W), mask_thresh, want_masks=False, want_observed=True)
        samp = ops.sample_mask(observed, self.sample_stride)
        _write_objects(idx, samp, self._frame_cnt, self._slots, self.implicit_memory.unsqueeze(0), bf, None,
                       mask_probs=mp, boxes=bx, mask_thresh=mask_thresh)
        self._finalize(idx)

    def write_object_features(self, box_features: torch.Tensor, masks: torch.Tensor, proj_indices: torch.Tensor) -> None:
        """A6 + A7 + A8 without the (1,C,H,W) image (custom_rcnn.py:690-701,738-743): the per-pixel object mean is
        formed only for the every-``sample_stride``-th observed pixels, on the fly."""
        h, w = masks.shape[-2:]
        idx = self._idx32(proj_indices, self.implicit_memory.shape[0]).view(1, h, w)
        bf = box_features.to(self.device, torch.float32).contiguous().unsqueeze(0)
        m = masks.to(self.device).contiguous().unsqueeze(0)
        self._slots = _slot_workspace(self._slots, 1, self.implicit_memory.shape[0], self.C, h * w, self.sample_stride, self.device)
        observed = ops.masks_observed(m)
        samp = ops.sample_mask(observed, self.sample_stride)
        _write_objects(idx, samp, self._frame_cnt, self._slots, self.implicit_memory.unsqueeze(0), bf, None, masks=m)
        self._finalize(idx)

    def dense_backbone_write(self, p3: torch.Tensor, proj_indices: torch.Tensor, n_cells: int,
                             weight: Optional[torch.Tensor] = None, bias: Optional[torch.Tensor] = None, step: int = 8):
        """Dense backbone-feature write (SURVEY 8a row A7'', bytecode-only older CustomMapFPN.forward): p3 (1,C,h,w) ->
        bilinear (H,W) align_corners=True -> [::step, ::step] -> optional 1x1 projection (map_merge_forward_projection,
        eod_linear_rows) -> per-cell mean with proj_indices[::step, ::step]; returns (memory (cells,C') f32 with the mean in the
        observed cells and zeros elsewhere - the reference REPLACES the memory - and observed_mem (cells,) bool)."""
        idx_full = self._index_plane(proj_indices)
        H, W = idx_full.shape
        f = ops.bilinear_lattice(p3.to(self.device, torch.float32).contiguous(), (H, W), step)
        layout = LAYOUT_CHW
        C = f.shape[1]
        if weight is not None:                             # 1x1 conv == per-sample row GEMM on the tensor cores (fp32 accuracy), output HWC
            w2 = weight.to(self.device, torch.float32).reshape(weight.shape[0], -1)
            b2 = None if bias is None else bias.to(self.device, torch.float32).contiguous()
            f = ops.linear_rows(f[0].reshape(C, -1).t(), w2, b2)          # the CHW lattice is read through a transposed view
            f, C, layout = f.unsqueeze(0), w2.shape[0], LAYOUT_HWC
        else:
            f = f.reshape(1, C, -1).contiguous()
        idx = self._idx32(idx_full[::step, ::step].contiguous(), n_cells)
        return self._fresh_mean(f, idx, None, n_cells, C, layout)

    def write_image_features(self, image_features: torch.Tensor, observed_pixels: Optional[torch.Tensor],
                             proj_indices: torch.Tensor, layout: int = LAYOUT_CHW) -> None:
        """A7 + A8 on the live state: per-cell mean of every ``sample_stride``-th observed pixel, sums +=,
        counts += 1 for all visible cells.  bf16 / fp16 features are written as they are (the 16-bit variant of ``layout``)."""
        idx = self._idx32(proj_indices, self.implicit_memory.shape[0])
        samp = None
        if observed_pixels is not None:
            samp = ops.sample_mask(observed_pixels.to(self.device).reshape(1, -1).view(torch.uint8).contiguous(), self.sample_stride)
        C = self.C
        feat, layout = self._feat_in(image_features, layout, C)
        feat = feat.reshape(1, -1)
        ops.frame_count(idx, samp, self._frame_cnt)
        ops.write_mean(feat, idx, samp, self._frame_cnt, self.implicit_memory.unsqueeze(0), layout)
        self._finalize(idx)
