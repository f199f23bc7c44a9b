"""Episode runner: drives a dataset of (ragged) episodes through an ``EpisodeBatch`` in lock step, the way the
reference's eval loop drives them one after the other (detic/modeling/meta_arch/custom_rcnn.py:441-539).

Reference semantics kept, frame by frame and per episode:
  * order of episodes and ``memory_reset`` flags: SMNet/loader.py:97-117,289-293 (``formats.order_files`` /
    ``formats.memory_reset_flag``);
  * ``memory_reset`` -> zero state BEFORE the frame's read (custom_rcnn.py:470-477);
  * TEST_TYPE default / episodic: the read of every frame sees the latest state; longterm: the read of a whole
    sequence sees the state as it was at the sequence's first frame, after a reset if there was one (:482-491) -
    ``EpisodeBatch.read_frozen`` + a per-slot ``refresh_mask`` at sequence starts;
  * read -> (detector, out of scope) -> write of the same frame (:494-515); a frame without kept detections writes
    nothing (:686);
  * ``save_semmap``: after the write of a sequence's FIRST frame the state is dumped under <out>/memory/<sequence_name>
    with the reference's dataset names (:518-530, ``formats.save_memory``).

What is new is the batching: a STREAM is a maximal chain of consecutive episodes that share one grid (it starts at an
episode whose first frame carries ``memory_reset``: a whole scene for default / longterm, one sequence for episodic).
Streams are independent, so they are dealt round-robin to ranks (no collective, SURVEY 8e) and, inside a rank, to the
R resident grid slots of one ``EpisodeBatch``; a slot that finishes its stream takes the next one from the queue, which
keeps at most R grids resident however many episodes there are (BASELINE configs[4]: 512 episodes of 1000x1000x512
grids in waves of R).  Slots without work are masked out (``active``).

``regime="heightmax"`` runs the same schedule over a ``HeightMaxBatch`` (the SMNet height-max memory, BASELINE configs[2]): no read,
and each episode's map is dumped after its LAST frame (SMNet's encoder hands the finished map to its decoder).

``LockStepSchedule`` is the host-only part (pure Python, tested without a GPU); ``EpisodeRunner`` issues the launches.
"""
from __future__ import annotations

import os
from collections import deque
from dataclasses import dataclass
from typing import Callable, Dict, Iterator, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import formats, ops
from ._lib import LAYOUT_CHW, ORDER_ZX, WRITE_AUTO, WRITE_DET, EodError


def split_streams(reset_first: Sequence[bool]) -> List[List[int]]:
    """Episodes in dataset order -> chains sharing one grid: a new chain starts at every episode whose first frame carries
    memory_reset (SMNet/loader.py:289-293)."""
    streams: List[List[int]] = []
    for i, r in enumerate(reset_first):
        if r or not streams:
            streams.append([])
        streams[-1].append(i)
    return streams


@dataclass
class Step:
    assign: List[Optional[Tuple[int, int]]]        # per slot: (episode index, frame index) or None (idle)
    reset: List[bool]                               # per slot: clear the grid before this frame's read
    seq_start: List[bool]                           # per slot: this is frame 0 of its episode (longterm snapshot, save_semmap)


class LockStepSchedule:
    """Which (episode, frame) every slot processes at every frame-step.  n_frames[i], reset_first[i]: per episode in
    dataset order; rank / world: this rank's share of the streams (stream index % world == rank)."""

    def __init__(self, n_frames: Sequence[int], reset_first: Sequence[bool], n_slots: int, rank: int = 0, world: int = 1):
        if n_slots <= 0 or not (0 <= rank < world):
            raise ValueError("n_slots must be positive and 0 <= rank < world")
        self.n_frames, self.n_slots = [int(n) for n in n_frames], int(n_slots)
        all_streams = split_streams(reset_first)
        self.streams = [s for k, s in enumerate(all_streams) if k % world == rank]
        self.n_streams_total = len(all_streams)

    @property
    def episodes(self) -> List[int]:
        return [e for s in self.streams for e in s]

    @property
    def total_frames(self) -> int:
        return sum(self.n_frames[e] for e in self.episodes)

    def __iter__(self) -> Iterator[Step]:
        queue = deque(self.streams)
        cur: List[Optional[dict]] = [None] * self.n_slots      # dict(eps=[...], k=position in chain, f=frame)
        while True:
            assign: List[Optional[Tuple[int, int]]] = [None] * self.n_slots
            reset = [False] * self.n_slots
            start = [False] * self.n_slots
            for s in range(self.n_slots):
                st = cur[s]
                while True:
                    if st is None:
                        if not queue:
                            break
                        st = dict(eps=queue.popleft(), k=0, f=0, fresh=True)
                    if st["k"] >= len(st["eps"]):
                        st = None
                        continue
                    e = st["eps"][st["k"]]
                    if st["f"] >= self.n_frames[e]:            # episode exhausted (or empty): next one of the chain
                        st["k"] += 1
                        st["f"] = 0
                        continue
                    break
                cur[s] = st
                if st is None:
                    continue
                e = st["eps"][st["k"]]
                assign[s] = (e, st["f"])
                start[s] = st["f"] == 0
                reset[s] = bool(st.pop("fresh", False))          # a slot that takes a new chain always starts from zero
                st["f"] += 1
            if not any(a is not None for a in assign):
                return
            yield Step(assign, reset, start)


class _Staging:
    """Pinned host buffers + device buffers, both double buffered: the pinned copy of step k is not overwritten before its
    asynchronous H2D copy has completed (event), and the device copy of step k is not overwritten while step k's kernels may
    still read it (EpisodeBatch orders everything of step k before whatever the caller enqueues after step k+1)."""

    def __init__(self, device: torch.device):
        self.device = torch.device(device)
        self.pin: Dict[str, List[torch.Tensor]] = {}
        self.dev: Dict[str, List[torch.Tensor]] = {}
        self.done: List[Optional[torch.cuda.Event]] = [None, None]
        self.flip = 0

    def next(self) -> None:
        self.flip ^= 1
        if self.done[self.flip] is not None:
            self.done[self.flip].synchronize()

    def buf(self, key: str, shape, dtype) -> Tuple[torch.Tensor, torch.Tensor]:
        if key not in self.pin or tuple(self.pin[key][0].shape) != tuple(shape):
            self.pin[key] = [torch.zeros(shape, dtype=dtype).pin_memory() for _ in range(2)]
            self.dev[key] = [torch.zeros(shape, dtype=dtype, device=self.device) for _ in range(2)]
        return self.pin[key][self.flip], self.dev[key][self.flip]

    def commit(self) -> None:
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.device))
        self.done[self.flip] = ev


class HostEpisodeProvider:
    """Episodes held on the host as lists of frame dicts - the items of ``formats.EpisodeDataset`` (SMNet/loader.py item
    contract) plus whatever feeds the write.  Per frame: ``sequence_name``, ``memory_reset``, and
        geometry : ``proj_indices`` (H,W[,1]) int32  (memory_data/*.h5)   or   ``depth`` (H,W) f32 + ``pose`` (12,) f32
        write    : ``feat`` (C,H,W) f32 [dense]   or   ``box_features`` (K,C), ``mask_probs`` (K,S,S), ``boxes`` (K,4) [detections]
        height-max planes (create_coco_mp3d.py:157-165), with ``proj_indices``: ``height`` (H,W) f32 and ``outlier`` (H,W) bool / u8
    ``shifts``: per episode (6,) f32 (world_shift_origin xyz, map_world_shift xyz), needed with depth.
    ``feat_dtype``: the dtype ``feat`` is staged in - torch.bfloat16 / torch.float16 feed the 16-bit layouts of ``EpisodeRunner``
    (LAYOUT_CHW_BF16 / _F16 for (C,H,W) frames, LAYOUT_HWC_BF16 / _F16 for (H,W,C) ones) at half the bytes; a frame's ``feat`` may
    be a numpy array or a CPU tensor of any dtype.
    Frames are staged through pinned buffers and copied to the device on the caller's stream."""

    def __init__(self, episodes: Sequence[Sequence[dict]], device: torch.device, shifts: Optional[Sequence[np.ndarray]] = None,
                 k_max: int = 16, feat_dtype: torch.dtype = torch.float32):
        self.episodes, self.device, self.k_max, self.feat_dtype = episodes, torch.device(device), int(k_max), feat_dtype
        self.shifts = None if shifts is None else [np.asarray(s, np.float32) for s in shifts]
        self._st = _Staging(self.device)

    n_episodes = property(lambda self: len(self.episodes))

    def n_frames(self, i: int) -> int:
        return len(self.episodes[i])

    def name(self, i: int) -> str:
        return str(self.episodes[i][0].get("sequence_name", f"episode_{i}")) if len(self.episodes[i]) else f"episode_{i}"

    def reset_flag(self, i: int, f: int) -> bool:
        return bool(self.episodes[i][f].get("memory_reset", False))

    def stage(self, assign: Sequence[Optional[Tuple[int, int]]]) -> dict:
        self._st.next()
        R = len(assign)
        first = next(self.episodes[e][f] for a in assign if a is not None for e, f in [a])
        out: Dict[str, torch.Tensor] = {}
        host: Dict[str, torch.Tensor] = {}

        def put(key, s, value, shape, dtype):
            if key not in host:
                host[key], out[key] = self._st.buf(key, (R,) + tuple(shape), dtype)
            host[key][s] = (value if torch.is_tensor(value) else torch.as_tensor(np.asarray(value))).reshape(shape).to(dtype)

        for s, a in enumerate(assign):
            if a is None:
                continue
            fr = self.episodes[a[0]][a[1]]
            if "proj_indices" in fr:
                pi = np.asarray(fr["proj_indices"])
                pi = pi[..., 0] if pi.ndim == 3 else pi
                put("idx", s, pi, pi.shape, torch.int32)
            else:
                put("depth", s, fr["depth"], np.asarray(fr["depth"]).shape, torch.float32)
                put("pose", s, fr["pose"], (12,), torch.float32)
                put("shifts", s, self.shifts[a[0]], (6,), torch.float32)
            for key, dtype in (("height", torch.float32), ("outlier", torch.uint8)):
                if key in fr:
                    put(key, s, fr[key], np.asarray(fr[key]).shape, dtype)
            if "feat" in fr:
                f = fr["feat"]
                put("feat", s, f, tuple(f.shape) if torch.is_tensor(f) else np.asarray(f).shape, self.feat_dtype)
            elif "box_features" in fr:
                bf, mp, bx = np.asarray(fr["box_features"], np.float32), np.asarray(fr["mask_probs"], np.float32), np.asarray(fr["boxes"], np.float32)
                K = bf.shape[0]
                if K > self.k_max:
                    raise EodError(f"{K} detections in one frame exceed k_max={self.k_max}")
                C = bf.shape[1] if K else int(first["box_features"].shape[1])
                S = mp.shape[-1] if K else int(np.asarray(first["mask_probs"]).shape[-1])
                for key, shape, dtype in (("box_features", (self.k_max, C), torch.float32), ("mask_probs", (self.k_max, S, S), torch.float32),
                                          ("boxes", (self.k_max, 4), torch.float32), ("n_obj", (), torch.int32)):
                    if key not in host:
                        host[key], out[key] = self._st.buf(key, (R,) + shape, dtype)
                host["n_obj"][s] = K
                if K:
                    host["box_features"][s, :K] = torch.from_numpy(bf)
                    host["mask_probs"][s, :K] = torch.from_numpy(mp)
                    host["boxes"][s, :K] = torch.from_numpy(bx)
        if "n_obj" in host:
            for s, a in enumerate(assign):
                if a is None:
                    host["n_obj"][s] = 0
        for key in host:
            out[key].copy_(host[key], non_blocking=True)
        self._st.commit()
        return out


class EpisodeRunner:
    """Lock-step execution of a provider's episodes on one GPU (one rank).

    provider: ``n_episodes``, ``n_frames(i)``, ``name(i)``, ``reset_flag(i, f)``, ``stage(assign) -> dict`` of (R, ...) device
    tensors ordered on the caller's stream: ``idx`` (R,H,W) i32 or ``depth`` (R,H,W) + ``pose`` (R,12) + ``shifts`` (R,6);
    ``feat`` (R,C,H,W) [dense regime] or ``box_features`` (R,K,C) + ``mask_probs`` (R,K,S,S) + ``boxes`` (R,K,4) + ``n_obj`` (R).
    ``trusted_indices = True`` on the provider skips the range check of staged ``idx`` planes.
    ``variant = WRITE_DET``: the dense write is the deterministic one, so a run reproduces bit for bit whatever the slot count and the
    wave a stream lands in (size its workspace with ``batch.det_runs_per_episode``); the detection regime has no deterministic write
    and raises EodError.
    ``regime = "heightmax"``: the slots are a ``HeightMaxBatch`` (``layout`` and ``linlayer`` = (weight, bias) | None as it takes them);
    frames carry ``feat`` and depth + pose or ``proj_indices`` + ``height`` (+ ``outlier``); anything else staged (detections, an index
    plane without heights) raises EodError.  There is no read, so ``on_levels`` is not called; ``save_dir`` receives
    <save_dir>/heightmax/<name> (``formats.save_heightmax``) after each episode's last frame.
    """

    def __init__(self, provider, map_w: int, map_h: int, channels: int, n_slots: int, *, height: int = 480, width: int = 640,
                 device: torch.device = torch.device("cuda"), test_type: str = "default", rank: int = 0, world: int = 1,
                 intr: Optional[Sequence[float]] = None, cell: float = 0.2, order: int = ORDER_ZX, layout: int = LAYOUT_CHW,
                 save_dir: Optional[str] = None, zs_weight: Optional[torch.Tensor] = None, obs_score_thresh: float = 0.4,
                 n_semmap_classes: int = 20, sample_stride: int = 8, mask_thresh: float = 0.5, pipeline: bool = True,
                 variant: int = WRITE_AUTO, regime: str = "mean", linlayer=None):
        from .memory import EpisodeBatch, HeightMaxBatch
        if test_type not in ("default", "episodic", "longterm"):
            raise ValueError(f"unknown TEST_TYPE {test_type!r}")           # detic/config.py:74
        if regime not in ("mean", "heightmax"):
            raise ValueError(f"unknown regime {regime!r} (mean | heightmax)")
        if regime == "heightmax" and variant != WRITE_AUTO:
            raise ValueError("variant selects the mean write; the height-max regime has one update")
        self.regime = regime
        self.provider, self.test_type, self.device = provider, test_type, torch.device(device)
        n = provider.n_episodes
        self.schedule = LockStepSchedule([provider.n_frames(i) for i in range(n)],
                                         [provider.n_frames(i) > 0 and provider.reset_flag(i, 0) for i in range(n)], n_slots, rank, world)
        if regime == "heightmax":
            self.batch = HeightMaxBatch(n_slots, map_w, map_h, channels, height, width, self.device, layout=layout, linlayer=linlayer, order=order)
        else:
            self.batch = EpisodeBatch(n_slots, map_w, map_h, channels, height, width, self.device, layout=layout, variant=variant, pipeline=pipeline)
            self.batch.read_frozen = test_type == "longterm"
        self.intr, self.cell, self.order = intr, float(cell), order
        self.save_dir, self.sample_stride, self.mask_thresh = save_dir, sample_stride, mask_thresh
        self.zs_weight = None if zs_weight is None else zs_weight.to(self.device, torch.float32).contiguous()
        self.obs_score_thresh, self.n_semmap_classes = obs_score_thresh, n_semmap_classes
        self.R = n_slots
        self._masks = _Staging(self.device)
        self.stats = {"frames": 0, "steps": 0, "slot_steps": 0, "resets": 0, "saved": 0}

    # -- explicit semantic map of one slot, for the save (custom_rcnn.py:747-756): full decode of the touched cells -------------
    def _semmap(self, s: int) -> torch.Tensor:
        b = self.batch
        if self.zs_weight is None:
            return torch.full((b.n_cells,), -1, dtype=torch.int32)                               # :474, never decoded
        counts = b.counts[s:s + 1]
        seen = (counts != 0)
        frame_cnt = seen.to(torch.int32)
        intensity = torch.zeros((1, b.n_cells), dtype=torch.float32, device=self.device)
        cls = torch.zeros((1, b.n_cells), dtype=torch.int32, device=self.device)
        # eod_semmap_update expects the counts BEFORE this frame's increment (n = counts + 1)
        ops.semmap_update(frame_cnt, (counts - seen.to(torch.float32)).contiguous(), b.sums[s:s + 1], self.zs_weight, self.n_semmap_classes, intensity, cls)
        return ops.semmap_decode(intensity, cls, self.obs_score_thresh)[0]

    def _save(self, s: int, name: str) -> None:
        self.batch.join()
        path = os.path.join(self.save_dir, "memory", name)
        formats.save_memory(path, self._semmap(s), self.batch.sums[s], self.batch.counts[s])
        self.stats["saved"] += 1

    def _step_heightmax(self, inp: dict, active: torch.Tensor, reset_mask: Optional[torch.Tensor]) -> None:
        other = [k for k in ("box_features", "mask_probs", "boxes", "n_obj") if k in inp]
        if other or "feat" not in inp or ("idx" in inp and "height" not in inp):
            raise EodError(f"height-max runner: a frame needs feat and depth + pose or proj_indices + height (+ outlier); staged: {sorted(inp)}")
        if "idx" in inp:
            geo = dict(height=inp["height"], idx=inp["idx"], outlier=inp.get("outlier"))
        else:
            geo = dict(depth=inp["depth"], pose=inp["pose"], shifts=inp["shifts"], intr=self.intr, cell=self.cell)
        self.batch.step(inp["feat"], active=active, reset_mask=reset_mask, **geo)

    def _save_heightmax(self, s: int, name: str) -> None:
        b = self.batch
        formats.save_heightmax(os.path.join(self.save_dir, "heightmax", name), b.state[s], b.observed[s], b.height_map[s])
        self.stats["saved"] += 1

    def run(self, on_levels: Optional[Callable[[Step, List[torch.Tensor]], None]] = None, max_steps: Optional[int] = None) -> dict:
        """Process this rank's share of the dataset.  on_levels(step, levels): consumer hook, called after every frame-step
        with the three pooled fp16 levels (R,C,h,w) ordered on the caller's stream (idle slots hold stale values).
        With WRITE_DET the stats carry ``det_overflowed``: some run did not fit the workspace (since it was created) and took the
        order-dependent reductions - the result is correct but no longer reproducible."""
        b = self.batch
        self.stats = {k: 0 for k in self.stats}                  # per run() call
        with torch.cuda.device(self.device):
            for k, step in enumerate(self.schedule):
                if max_steps is not None and k >= max_steps:
                    break
                reset = [r or (a is not None and self.provider.reset_flag(a[0], a[1])) for r, a in zip(step.reset, step.assign)]
                refresh = [getattr(b, "read_frozen", False) and (st or r) for st, r in zip(step.seq_start, reset)]
                self._masks.next()
                pin, dev = self._masks.buf("masks", (3, self.R), torch.int32)
                pin.copy_(torch.tensor([[int(a is not None) for a in step.assign], [int(r) for r in reset], [int(r) for r in refresh]], dtype=torch.int32))
                dev.copy_(pin, non_blocking=True)
                self._masks.commit()
                inp = self.provider.stage(step.assign)
                geo = dict(proj_indices=inp["idx"]) if "idx" in inp else dict()
                if "idx" in inp and not getattr(self.provider, "trusted_indices", False):
                    ops.check_indices(inp["idx"], b.n_cells)
                masks = dict(reset_mask=dev[1] if any(reset) else None, refresh_mask=dev[2] if any(refresh) else None)
                depth, pose, shifts = inp.get("depth"), inp.get("pose"), inp.get("shifts")
                if self.regime == "heightmax":
                    self._step_heightmax(inp, dev[0], masks["reset_mask"])
                    levels = None
                elif "feat" in inp:
                    levels = b.step(depth, pose, shifts, self.intr, self.cell, inp["feat"], None, self.order, active=dev[0],
                                    inputs_ready=False, **masks, **geo)
                else:
                    if b.variant == WRITE_DET:
                        raise EodError("EpisodeRunner(variant=WRITE_DET): the object-regime write (detections) is not deterministic")
                    n_obj = torch.where(dev[0] > 0, inp["n_obj"], torch.zeros_like(inp["n_obj"]))
                    levels = b.step_detections(depth, pose, shifts, self.intr, self.cell, inp["box_features"], inp["mask_probs"], inp["boxes"],
                                               n_obj, self.sample_stride, self.mask_thresh, self.order, inputs_ready=False, **masks, **geo)
                self.stats["steps"] += 1
                self.stats["slot_steps"] += self.R
                self.stats["frames"] += sum(a is not None for a in step.assign)
                self.stats["resets"] += sum(reset)
                if self.regime == "heightmax":
                    if self.save_dir:
                        for s, a in enumerate(step.assign):
                            if a is not None and a[1] == self.provider.n_frames(a[0]) - 1:
                                self._save_heightmax(s, self.provider.name(a[0]))
                    continue
                if on_levels is not None:
                    on_levels(step, levels)
                if self.save_dir:
                    for s, (a, st) in enumerate(zip(step.assign, step.seq_start)):
                        if a is not None and st:
                            self._save(s, self.provider.name(a[0]))
            if self.regime == "heightmax":
                return dict(self.stats)
            b.join()
            if b.variant == WRITE_DET:
                self.stats["det_overflowed"] = b._det_ws is not None and b._det_ws.overflowed()
        return dict(self.stats)


class PooledSyntheticProvider:
    """Synthetic dense-regime episodes for workloads too large to hold as depth maps (BASELINE configs[4]: 512 episodes x 100
    frames = 63 GB of fp32 depth): ``pool`` distinct trajectories are ray-cast once on the device (episodes.DeviceEpisodes) and
    episode e replays trajectory e % pool into ITS OWN grid; every episode starts with memory_reset (independent episodes,
    TEST_TYPE episodic).  Features: two resident random (R,C,H,W) slabs used alternately (>> L2), as in bench.py, drawn in fp32 and
    held as ``feat_dtype`` (torch.bfloat16 / torch.float16 feed LAYOUT_CHW_BF16 / _F16).  Input generation only - nothing here is on
    the measured path except one gather of the step's depth / pose rows."""
    trusted_indices = True

    def __init__(self, n_episodes: int, n_frames: int, channels: int, n_slots: int, device, height: int = 480, width: int = 640,
                 map_w: int = 1000, map_h: int = 1000, cell: float = 0.2, pool: int = 64, seed0: int = 1234, lengths=None,
                 feat_dtype: torch.dtype = torch.float32):
        from . import episodes as E_
        from .geometry import transform3d
        self.device = torch.device(device)
        self.n_episodes, self.T, self.pool = int(n_episodes), int(n_frames), int(min(pool, n_episodes))
        self.lengths = None if lengths is None else [int(x) for x in lengths]
        dev_eps = E_.DeviceEpisodes(self.pool, n_frames, self.device, height, width, map_w, map_h, cell, seed0)
        self.depth = torch.empty((self.pool, n_frames, height, width), dtype=torch.float32, device=self.device)
        for t in range(n_frames):
            dev_eps.render(list(range(self.pool)), [t] * self.pool, out=self.depth[:, t])
        T = transform3d(torch.from_numpy(dev_eps.xyzhe.reshape(-1, 5))).reshape(self.pool, n_frames, 4, 4)
        self.T_host = T.numpy()
        self.shift_host = dev_eps.shift
        self.pose = T[:, :, :3, :].reshape(self.pool, n_frames, 12).contiguous().to(self.device)
        self.shifts = torch.from_numpy(np.concatenate([np.zeros_like(dev_eps.shift), dev_eps.shift], 1)).to(self.device)
        gen = torch.Generator(device=self.device).manual_seed(seed0)
        self.feat = [torch.randn((n_slots, channels, height, width), device=self.device, generator=gen).to(feat_dtype) for _ in range(2)]
        self._st = _Staging(self.device)
        self._keep: List[dict] = []
        self._k = 0

    def n_frames(self, i: int) -> int:
        return self.T if self.lengths is None else self.lengths[i]

    def name(self, i: int) -> str:
        return f"synthetic_{i % self.pool}_{i}"

    def reset_flag(self, i: int, f: int) -> bool:
        return f == 0

    def stage(self, assign: Sequence[Optional[Tuple[int, int]]]) -> dict:
        self._st.next()
        R = len(assign)
        pin, dev = self._st.buf("sel", (2, R), torch.int64)
        pin.copy_(torch.tensor([[0 if a is None else a[0] % self.pool for a in assign], [0 if a is None else a[1] for a in assign]], dtype=torch.int64))
        dev.copy_(pin, non_blocking=True)
        self._st.commit()
        out = {"depth": self.depth[dev[0], dev[1]], "pose": self.pose[dev[0], dev[1]], "shifts": self.shifts[dev[0]], "feat": self.feat[self._k & 1]}
        self._k += 1
        self._keep = (self._keep + [out])[-3:]            # gathered rows stay alive until the steps that read them have been ordered
        return out
