"""The layer that schedules the kernels: EpisodeBatch.step / step_detections spread a frame over two or three internal streams,
``pipeline=True`` runs frame t+1's geometry ahead of the caller's stream, capture_step_detections replays a CUDA graph between
eager steps, and the persistent TMA write takes its tiles from the ticket pool or, inside a capture, from a static partition.

Every late-input test delays the caller's stream (``torch.cuda._sleep``) before it produces the inputs there, and asserts that the
stream was still busy when ``step`` returned: the step's work was enqueued before its inputs existed, so an ordering error changes
the result instead of passing unseen.  References: float64 per-cell means (custom_rcnn.py:696-701,917-934) within SUM_TOL of scale,
exact counts / touched sets, and - for the deterministic write variant - a serial twin whose every bit must agree.
Run on the B200 box with `-m gpu`.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
H, W, C, MW, MH, CELL = 96, 128, 128, 60, 45, 0.2
SUM_TOL = 1e-5          # max|a-b| <= SUM_TOL * max|ref|
SLEEP_MS = 50           # how long a late producer keeps the caller's stream busy
KMAX = 6


# --------------------------------------------------------------------------------------------------------
# harness
# --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sleep_cycles(cuda):
    """torch.cuda._sleep cycles that keep a stream busy for about SLEEP_MS on this device (measured: the SM clock is not assumed)."""
    probe = 20_000_000
    torch.cuda._sleep(5 * probe)                              # let the SM clock ramp up first
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    torch.cuda._sleep(probe)
    b.record()
    b.synchronize()
    cycles = int(probe * SLEEP_MS / max(a.elapsed_time(b), 1e-3))
    return min(max(cycles, 2_000_000), 150_000_000)          # bounded: a busy-wait of tens of ms, never a hang


def late(cycles, produce):
    """Delay the caller's current stream, then run ``produce`` on it: what it writes does not exist yet when the next call
    enqueues its work."""
    torch.cuda._sleep(cycles)
    produce()


def assert_busy(what):
    assert not torch.cuda.current_stream().query(), \
        f"{what}: the caller's stream had drained before the step was enqueued - the late producer proves nothing"


def ref_write(sums, counts, feat, idx, samp=None):
    """One frame of the mean write for one episode in float64: sums (cells,C) += per-cell mean of the sampled pixels, counts += 1
    for every cell a pixel falls into (custom_rcnn.py:696-701,917-934).  feat (C,HW) or (C,H,W); returns new arrays and the
    per-cell sample counts."""
    f = np.asarray(feat, np.float64).reshape(sums.shape[1], -1)
    ix = np.asarray(idx).reshape(-1).astype(np.int64)
    sel = np.ones(ix.shape, bool) if samp is None else np.asarray(samp).reshape(-1) != 0
    order = np.argsort(ix[sel], kind="stable")
    cells = ix[sel][order]
    uniq, start, n = np.unique(cells, return_index=True, return_counts=True)
    sums, counts = sums.copy(), counts.copy()
    if uniq.size:
        sums[uniq] += np.add.reduceat(f[:, sel].T[order], start, axis=0) / n[:, None]
    counts[np.unique(ix)] += 1
    n_cell = np.zeros(sums.shape[0], np.int64)
    n_cell[uniq] = n
    return sums, counts, n_cell


def assert_sums(got, ref, what):
    got = got.double().cpu().numpy() if torch.is_tensor(got) else got
    scale = max(float(np.abs(ref).max()), 1e-30)
    err = float(np.abs(got - ref).max())
    assert err <= SUM_TOL * scale, f"{what}: sums off by {err:.3g} (scale {scale:.3g})"


def bits(t):
    t = t.contiguous()
    return t.view({torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype])


def assert_same_bits(a, b, what):
    assert torch.equal(bits(a), bits(b)), f"{what}: {int((bits(a) != bits(b)).sum())} elements differ"


def assert_levels_close(got, ref, what):
    """fp16 levels of two grids that reduced in different orders: at most one ulp, on fewer than 1e-3 of the elements."""
    for k, (x, y) in enumerate(zip(got, ref)):
        d = (bits(x).int() - bits(y).int()).abs()
        assert int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3, f"{what} L{k}: max {int(d.max())} ulp"


def assert_levels_equal_reference(levels, sums, counts, idx, what):
    """The read of a frame against R.read_frame of the state the frame saw (bit-exact: same fp16 table, same pooling)."""
    for e in range(sums.shape[0]):
        ref = R.read_frame(sums[e], counts[e], torch.from_numpy(idx[e]).long())
        for k in range(3):
            assert torch.equal(bits(levels[k][e].cpu()), bits(ref[k][0])), f"{what} slot {e} L{k}"


class Scene:
    pass


@pytest.fixture(scope="module")
def scene(eod, cuda):
    """Three episodes x six frames at 96x128 on a 60x45 grid: device depth / pose / features, oracle cell indices."""
    s = Scene()
    s.E, s.T = 3, 6
    eps = [eod.episodes.make_episode(300 + e, s.T, H, W, MW, MH, CELL) for e in range(s.E)]
    s.intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    s.shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(cuda)
    Tm = [eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps]))) for t in range(s.T)]
    s.depth = [torch.from_numpy(np.stack([ep.depth[t] for ep in eps])).to(cuda) for t in range(s.T)]
    s.pose = [Tm[t][:, :3].reshape(s.E, 12).to(cuda) for t in range(s.T)]
    s.idx = [np.stack([oracle.backproject_quantize(eps[e].depth[t], Tm[t][e].numpy(), s.intr, np.zeros(3, np.float32), eps[e].map_world_shift,
                                                   np.float32(CELL), MW, MH, 0, 0.5, want=("idx",))["idx"] for e in range(s.E)]) for t in range(s.T)]
    s.idx_dev = [torch.from_numpy(i).to(cuda) for i in s.idx]
    g = torch.Generator(device=cuda).manual_seed(5)
    s.feat = [torch.randn((s.E, C, H, W), device=cuda, generator=g) for _ in range(s.T)]
    torch.cuda.synchronize()
    return s


def det_batch(eod, cuda, E, pipeline):
    """Deterministic write variant with room for every run: its bits do not depend on batching or scheduling (DESIGN 3.1b)."""
    b = eod.EpisodeBatch(E, MW, MH, C, H, W, cuda, variant=eod._lib.WRITE_DET, pipeline=pipeline)
    b.det_runs_per_episode = H * W
    return b


def make_dets(eod, rng, n_obj):
    E = len(n_obj)
    bf = np.zeros((E, KMAX, C), np.float32)
    pr = np.zeros((E, KMAX, 28, 28), np.float32)
    bx = np.zeros((E, KMAX, 4), np.float32)
    for e, n in enumerate(n_obj):
        if n:
            f, p, b = eod.episodes.make_mask_head_detections(rng, H, W, C, (int(n), int(n)), 28)
            bf[e, :n], pr[e, :n], bx[e, :n] = f, p, b
    return bf, pr, bx, np.asarray(n_obj, np.int32)


def poison_dets(bf, pr, bx, n_obj):
    """Detection inputs that would write NaN over whole images if a step consumed them."""
    bf.fill_(float("nan"))
    pr.fill_(1.0)
    bx.zero_()
    bx[..., 2] = float(W)
    bx[..., 3] = float(H)
    n_obj.fill_(KMAX)


def i32(v, dev):
    return torch.tensor(v, dtype=torch.int32, device=dev)


def warm(batch, frame):
    """Run one throwaway frame on the batch and clear its grid: the workspaces and streams it creates on first use (and the kernels
    the frame launches) exist before a timed window, so no allocation inside a late-fed step can stall the host until the caller's
    stream has drained."""
    frame(batch)
    batch.reset(full=True)
    torch.cuda.synchronize()


# --------------------------------------------------------------------------------------------------------
# A  step: feat / reset_mask / refresh_mask produced late (memory.py step: the write stream and the state
#    stream wait on the caller's stream before they read them)
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [False, True], ids=["ordered", "pipelined"])
@pytest.mark.parametrize("inputs_ready", [True, False], ids=["ready", "not-ready"])
def test_step_late_feat_and_masks_match_serial_twin_bitwise(eod, cuda, scene, sleep_cycles, pipeline, inputs_ready):
    """feat, reset_mask and refresh_mask are written on the caller's stream after the step was enqueued (TEST_TYPE longterm:
    read_frozen, the fp16 table changes only through refresh_mask).  Against a serial, synchronised twin: sums, counts, norm16
    and levels bitwise equal; sums within SUM_TOL of the float64 reference."""
    s = scene
    a, b = det_batch(eod, cuda, s.E, pipeline), det_batch(eod, cuda, s.E, False)
    a.read_frozen = b.read_frozen = True
    ones = i32([1] * s.E, cuda)
    warm(a, lambda x: x.step(s.depth[0], s.pose[0], s.shifts, s.intr, CELL, s.feat[0], reset_mask=ones, refresh_mask=ones))
    masks = {1: (None, [1, 1, 1]), 2: ([0, 1, 0], [1, 1, 0]), 4: (None, [0, 0, 1]), 5: ([1, 0, 0], None)}    # t -> (reset, refresh)
    feat_buf = torch.empty_like(s.feat[0])
    reset_buf, refresh_buf = torch.empty(s.E, dtype=torch.int32, device=cuda), torch.empty(s.E, dtype=torch.int32, device=cuda)
    ref_s = np.zeros((s.E, MW * MH, C))
    ref_c = np.zeros((s.E, MW * MH))
    for t in range(s.T):
        reset, refresh = masks.get(t, (None, None))
        reset_src = None if reset is None else i32(reset, cuda)
        refresh_src = None if refresh is None else i32(refresh, cuda)
        # the synchronous twin first: it also loads every kernel the frame needs before the timed window
        lb = [l.clone() for l in b.step(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, s.feat[t], reset_mask=reset_src, refresh_mask=refresh_src)]
        feat_buf.fill_(float("nan"))
        reset_buf.fill_(1)                              # read too early, these would reset / refresh every slot
        refresh_buf.fill_(1)
        torch.cuda.synchronize()

        def produce():
            feat_buf.copy_(s.feat[t])
            if reset is not None:
                reset_buf.copy_(reset_src)
            if refresh is not None:
                refresh_buf.copy_(refresh_src)

        late(sleep_cycles, produce)
        la = a.step(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, feat_buf, reset_mask=None if reset is None else reset_buf,
                    refresh_mask=None if refresh is None else refresh_buf, inputs_ready=inputs_ready)
        assert_busy(f"t={t}")
        la = [l.clone() for l in la]
        a.join()
        torch.cuda.synchronize()
        for k in range(3):
            assert_same_bits(la[k], lb[k], f"t={t} level {k}")
        for name in ("sums", "counts", "norm16"):
            assert_same_bits(getattr(a, name), getattr(b, name), f"t={t} {name}")
        for e in range(s.E):
            if reset is not None and reset[e]:
                ref_s[e], ref_c[e] = 0, 0
            ref_s[e], ref_c[e], _ = ref_write(ref_s[e], ref_c[e], s.feat[t][e].cpu().numpy(), s.idx[t][e])
        assert_sums(a.sums, ref_s, f"t={t}")
        assert np.array_equal(a.counts.cpu().numpy(), ref_c), f"t={t}: counts"
    assert not a._det_ws.overflowed()
    assert float(a.norm16.float().abs().max()) > 0 and float(a.counts.max()) >= 2


# --------------------------------------------------------------------------------------------------------
# B  step(pipeline=True, inputs_ready=True) with `active` produced late: the count (geometry stream) and the
#    write (write stream) must see the same mask
# --------------------------------------------------------------------------------------------------------
ACTIVE = [[1, 1, 1], [1, 0, 1], [1, 1, 0], [1, 0, 1], [0, 1, 1], [1, 1, 1]]      # slot 1: 1->0->1->0, slot 2: ->0->1, slot 0: ->0->1


@pytest.mark.parametrize("path", ["backproject_count", "project+frame_count", "proj_indices"])
def test_step_late_active_mask_leaves_idle_slots_bit_identical(eod, cuda, scene, sleep_cycles, path):
    """A slot that is idle in a frame keeps sums, counts and norm16 bit for bit although its feature slab is NaN; the active slots
    follow the float64 reference (counts exact) and every level equals the read of the state the frame saw."""
    s = scene
    a = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda, pipeline=True)
    a.fused_count = path == "backproject_count"
    feat_buf = torch.empty_like(s.feat[0])
    active_buf = i32(ACTIVE[0], cuda)
    ref_s = np.zeros((s.E, MW * MH, C))
    ref_c = np.zeros((s.E, MW * MH))
    for t in range(s.T):
        act = ACTIVE[t]
        act_src = i32(act, cuda)
        torch.cuda.synchronize()
        before = (a.sums.cpu(), a.counts.cpu(), a.norm16.cpu())
        src = s.feat[t].clone()
        for e in range(s.E):
            if not act[e]:
                src[e] = float("nan")                   # an idle slot's slab must not even be read

        def produce():
            feat_buf.copy_(src)
            active_buf.copy_(act_src)

        late(sleep_cycles, produce)
        levels = a.step(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, feat_buf, active=active_buf,
                        proj_indices=s.idx_dev[t] if path == "proj_indices" else None)
        assert_busy(f"t={t}")
        levels = [l.clone() for l in levels]
        a.join()
        torch.cuda.synchronize()
        assert_levels_equal_reference(levels, before[0], before[1], s.idx[t], f"t={t}")
        for e in range(s.E):
            if not act[e]:
                assert torch.equal(bits(a.sums[e].cpu()), bits(before[0][e])), f"t={t}: idle slot {e} sums changed"
                assert torch.equal(a.counts[e].cpu(), before[1][e]), f"t={t}: idle slot {e} counts changed"
                assert torch.equal(bits(a.norm16[e].cpu()), bits(before[2][e])), f"t={t}: idle slot {e} norm16 changed"
                continue
            ref_s[e], ref_c[e], _ = ref_write(ref_s[e], ref_c[e], s.feat[t][e].cpu().numpy(), s.idx[t][e])
            assert_sums(a.sums[e], ref_s[e], f"t={t} slot {e}")
            assert np.array_equal(a.counts[e].cpu().numpy(), ref_c[e]), f"t={t} slot {e}: counts"
    assert float(a.counts.max()) >= 2


# --------------------------------------------------------------------------------------------------------
# C  step_detections(pipeline=True, inputs_ready=False): detection tensors, n_obj and reset_mask produced late
# --------------------------------------------------------------------------------------------------------
def test_step_detections_late_inputs_match_serial_composition(eod, cuda, scene, sleep_cycles):
    """box_features / mask_probs / boxes / n_obj / reset_mask written on the caller's stream after the step was enqueued; a slot
    without detections in one frame.  Against project -> reset -> read -> write_detections on a twin: touched sets and counts
    exact, sums within SUM_TOL, levels within one fp16 ulp."""
    s = scene
    rng = np.random.default_rng(21)
    a = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda, pipeline=True)
    b = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda)
    n_objs = [[6, 3, 2], [6, 0, 3], [2, 6, 0], [4, 3, 6]]
    warm_dets = [torch.from_numpy(x).to(cuda) for x in make_dets(eod, rng, [2, 2, 2])]
    warm(a, lambda x: x.step_detections(s.depth[0], s.pose[0], s.shifts, s.intr, CELL, *warm_dets, reset_mask=i32([1] * s.E, cuda)))
    resets = {2: [1, 0, 0]}
    bufs = (torch.empty((s.E, KMAX, C), device=cuda), torch.empty((s.E, KMAX, 28, 28), device=cuda),
            torch.empty((s.E, KMAX, 4), device=cuda), torch.empty(s.E, dtype=torch.int32, device=cuda))
    reset_buf = torch.empty(s.E, dtype=torch.int32, device=cuda)
    for t, n_obj in enumerate(n_objs):
        dets = [torch.from_numpy(x).to(cuda) for x in make_dets(eod, rng, n_obj)]
        reset = resets.get(t)
        reset_src = None if reset is None else i32(reset, cuda)
        b.project(s.depth[t], s.pose[t], s.shifts, s.intr, CELL)      # the serial twin first (it also loads every kernel of the frame)
        if reset is not None:
            b.reset(mask=reset_src)
        lb = [l.clone() for l in b.read()]
        b.write_detections(*dets)
        poison_dets(*bufs)
        reset_buf.fill_(1)
        torch.cuda.synchronize()

        def produce():
            for dst, src in zip(bufs, dets):
                dst.copy_(src)
            if reset is not None:
                reset_buf.copy_(reset_src)

        late(sleep_cycles, produce)
        la = a.step_detections(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, *bufs, reset_mask=None if reset is None else reset_buf,
                               inputs_ready=False)
        assert_busy(f"t={t}")
        la = [l.clone() for l in la]
        a.join()
        torch.cuda.synchronize()
        assert_levels_close(la, lb, f"t={t}")
        if t == 0:
            for x, y in zip(la, lb):
                assert torch.equal(x, y)                # both tables still empty
        assert torch.equal(a.counts, b.counts), f"t={t}: counts"
        assert torch.equal(a.sums == 0, b.sums == 0), f"t={t}: touched cells"
        assert_sums(a.sums, b.sums.double().cpu().numpy(), f"t={t}")
    assert float(b.counts.max()) >= 2 and float(b.sums.abs().max()) > 0


# --------------------------------------------------------------------------------------------------------
# D  input reuse: a step's inputs may be overwritten once the next step has returned (runner._Staging relies on it)
# --------------------------------------------------------------------------------------------------------
def test_inputs_overwritten_after_the_next_step_change_nothing(eod, cuda, scene):
    """pipeline=True, inputs resident, no host synchronisation: after step t+1 returns, step t's depth / pose / shifts / feat / samp /
    reset_mask (dense) and detection tensors (object regime) are overwritten with NaN or garbage on the caller's stream.  The dense
    batch must equal its serial deterministic twin bit for bit, the object batch its serial twin up to reduction order."""
    s = scene
    nan = float("nan")
    # dense
    a, b = det_batch(eod, cuda, s.E, True), det_batch(eod, cuda, s.E, False)
    g = torch.Generator(device=cuda).manual_seed(8)
    samps = {2: (torch.rand((s.E, H, W), device=cuda, generator=g) < 0.5).to(torch.uint8)}
    resets = {3: [0, 1, 0]}
    torch.cuda.synchronize()
    prev, la = None, []
    for t in range(s.T):
        cur = dict(depth=s.depth[t].clone(), pose=s.pose[t].clone(), shifts=s.shifts.clone(), feat=s.feat[t].clone(),
                   samp=samps[t].clone() if t in samps else None, reset=i32(resets[t], cuda) if t in resets else None)
        levels = a.step(cur["depth"], cur["pose"], cur["shifts"], s.intr, CELL, cur["feat"], cur["samp"], reset_mask=cur["reset"])
        la.append([l.clone() for l in levels])
        if prev is not None:
            for k in ("depth", "pose", "shifts", "feat"):
                prev[k].fill_(nan)
            for k in ("samp", "reset"):
                if prev[k] is not None:
                    prev[k].fill_(1)
        prev = cur
    a.join()
    torch.cuda.synchronize()
    for t in range(s.T):
        lb = b.step(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, s.feat[t], samps.get(t),
                    reset_mask=i32(resets[t], cuda) if t in resets else None)
        for k in range(3):
            assert_same_bits(la[t][k], lb[k], f"dense t={t} level {k}")
    torch.cuda.synchronize()
    for name in ("sums", "counts", "norm16"):
        assert_same_bits(getattr(a, name), getattr(b, name), f"dense {name}")
    # object regime
    rng = np.random.default_rng(4)
    c = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda, pipeline=True)
    d = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda)
    dets = [[torch.from_numpy(x).to(cuda) for x in make_dets(eod, rng, n)] for n in ([6, 2, 4], [3, 6, 0], [5, 1, 6], [2, 4, 3])]
    torch.cuda.synchronize()
    prev, lc = None, []
    for t, det in enumerate(dets):
        cur = [s.depth[t].clone(), s.pose[t].clone()] + [x.clone() for x in det]
        lc.append([l.clone() for l in c.step_detections(cur[0], cur[1], s.shifts, s.intr, CELL, *cur[2:])])
        if prev is not None:
            prev[0].fill_(nan)
            prev[1].fill_(nan)
            poison_dets(*prev[2:])
        prev = cur
    c.join()
    torch.cuda.synchronize()
    for t, det in enumerate(dets):
        assert_levels_close(lc[t], d.step_detections(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, *det), f"objects t={t}")
    torch.cuda.synchronize()
    assert torch.equal(c.counts, d.counts) and torch.equal(c.sums == 0, d.sums == 0)
    assert_sums(c.sums, d.sums.double().cpu().numpy(), "objects")
    assert float(d.sums.abs().max()) > 0


# --------------------------------------------------------------------------------------------------------
# E  graph replays interleaved with pipelined eager steps (GraphedDetections.__call__ -> the next eager step)
# --------------------------------------------------------------------------------------------------------
def test_graph_replays_between_pipelined_eager_steps(eod, cuda, sleep_cycles):
    """A pipeline=True batch alternates replays of its captured step_detections with eager steps; every replay waits behind a late
    producer, so it has not even started when the next eager step is enqueued.  One and two / three eager steps between replays:
    both double-buffer halves meet the graph's.  Frame by frame against an eager pipeline=False twin."""
    E, T = 2, 10
    kinds = "GEGEEGEEEG"
    rng = np.random.default_rng(31)
    eps = [eod.episodes.make_episode(610 + e, T, H, W, MW, MH, CELL) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(cuda)
    depth = [torch.from_numpy(np.stack([ep.depth[t] for ep in eps])).to(cuda) for t in range(T)]
    pose = [eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))[:, :3].reshape(E, 12).to(cuda) for t in range(T)]
    dets = [[torch.from_numpy(x).to(cuda) for x in make_dets(eod, rng, [KMAX - t % 3, 0 if t == 4 else 3])] for t in range(T)]
    a = eod.EpisodeBatch(E, MW, MH, C, H, W, cuda, pipeline=True)
    b = eod.EpisodeBatch(E, MW, MH, C, H, W, cuda)
    graphed = a.capture_step_detections(depth[0], pose[0], shifts, intr, CELL, *dets[0])
    staging = [x.clone() for x in [depth[0], pose[0], shifts] + dets[0]]
    torch.cuda.synchronize()
    la = []
    for t, kind in enumerate(kinds):
        if kind == "G":
            late(sleep_cycles, lambda: [dst.copy_(src) for dst, src in zip(staging, [depth[t], pose[t], shifts] + dets[t])])
            levels = graphed(*staging)
        else:
            levels = a.step_detections(depth[t], pose[t], shifts, intr, CELL, *dets[t])
            if kinds[t - 1] == "G":
                assert_busy(f"t={t}: eager step after a replay")
        la.append([l.clone() for l in levels])
    a.join()
    torch.cuda.synchronize()
    for t in range(T):
        assert_levels_close(la[t], b.step_detections(depth[t], pose[t], shifts, intr, CELL, *dets[t]), f"t={t} ({kinds[t]})")
    torch.cuda.synchronize()
    assert torch.equal(a.counts, b.counts) and torch.equal(a.sums == 0, b.sums == 0)
    assert_sums(a.sums, b.sums.double().cpu().numpy(), "after the last frame")
    assert float(b.counts.max()) >= 2


# --------------------------------------------------------------------------------------------------------
# F  capture refuses per-frame masks and precomputed indices (GraphedDetections.__init__)
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("key", ["reset_mask", "refresh_mask", "proj_indices"])
def test_capture_rejects_per_frame_masks_and_leaves_state_alone(eod, cuda, scene, key):
    """A reset / refresh mask or an index plane would be baked into every replay (and applied by the warm-up frame): the capture
    must raise ValueError before it runs anything, leaving sums / counts / norm16 bit for bit as they were."""
    s = scene
    rng = np.random.default_rng(9)
    a = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda, pipeline=True)
    for t in range(2):
        a.step_detections(s.depth[t], s.pose[t], s.shifts, s.intr, CELL, *[torch.from_numpy(x).to(cuda) for x in make_dets(eod, rng, [4, 3, 5])])
    a.join()
    torch.cuda.synchronize()
    snap = (a.sums.clone(), a.counts.clone(), a.norm16.clone())
    assert float(snap[1].max()) >= 2
    extra = {"reset_mask": i32([1, 1, 1], cuda), "refresh_mask": i32([1, 1, 1], cuda), "proj_indices": s.idx_dev[3]}[key]
    dets = [torch.from_numpy(x).to(cuda) for x in make_dets(eod, rng, [4, 3, 5])]
    with pytest.raises(ValueError):
        a.capture_step_detections(s.depth[2], s.pose[2], s.shifts, s.intr, CELL, *dets, **{key: extra})
    a.join()
    torch.cuda.synchronize()
    assert_same_bits(a.sums, snap[0], "sums")
    assert_same_bits(a.counts, snap[1], "counts")
    assert_same_bits(a.norm16, snap[2], "norm16")


# --------------------------------------------------------------------------------------------------------
# G  every write kernel with `active` (write_mean.cu: LDG / TMA / channels-last skips, frame_count, backproject_count)
# --------------------------------------------------------------------------------------------------------
KERNELS = {"tma": (0, 2), "ldg": (0, 1), "hwc_f32": (1, 0), "hwc_bf16": (2, 0), "hwc_f16": (3, 0)}      # name -> (layout, variant)
GE, GH, GW, GCELLS = 5, 64, 96, 333
ACTIVE_G = [0, 1, 0, 1, 0]                                   # idle slots first, in the middle and last


@pytest.fixture(scope="module")
def geo5(eod, cuda):
    eps = [eod.episodes.make_episode(820 + e, 1, GH, GW, MW, MH, CELL) for e in range(GE)]
    intr = eod.compute_intrinsics(GW, GH, math.radians(67.5))
    shifts = torch.from_numpy(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps])).to(cuda)
    pose = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[0] for ep in eps])))[:, :3].reshape(GE, 12).to(cuda)
    return torch.from_numpy(np.stack([ep.depth[0] for ep in eps])).to(cuda), pose, shifts, intr


@pytest.mark.parametrize("C_", [128, 256, 512])
@pytest.mark.parametrize("kernel", list(KERNELS))
@pytest.mark.parametrize("with_samp", [False, True], ids=["dense", "sampled"])
def test_write_kernels_skip_idle_slots(eod, cuda, geo5, C_, kernel, with_samp):
    """frame_count -> write_mean -> finalize_counts (with the fp16 refresh) under an active mask: idle slots (NaN slabs) keep sums,
    counts, norm16 and touched bit for bit; active slots match the float64 reference, counts and touched sets exact, refreshed
    fp16 rows bit-exact.  backproject_count takes the same mask."""
    ops, layout, variant = eod.ops, *KERNELS[kernel]
    rng = np.random.default_rng(C_ + 7 * layout + variant + 100 * with_samp)
    HW = GH * GW
    act = i32(ACTIVE_G, cuda)
    idle = [e for e in range(GE) if not ACTIVE_G[e]]
    # the fused back-projection count skips idle slots exactly like frame_count
    depth, pose, shifts, intr = geo5
    gidx = torch.empty((GE, GH, GW), dtype=torch.int32, device=cuda)
    gcnt = torch.zeros((GE, MW * MH), dtype=torch.int32, device=cuda)
    ops.backproject_count(depth, pose, shifts, intr, CELL, MW, MH, gidx, gcnt, act)
    ref_cnt = torch.zeros_like(gcnt)
    ops.frame_count(gidx, None, ref_cnt, act)
    assert torch.equal(gcnt, ref_cnt) and not gcnt[idle].any()
    # the write: runs of two to sixteen pixels and isolated pixels, sampled or not
    feat = (rng.standard_normal((GE, C_, HW)) * 3).astype(np.float32)
    if layout in (2, 3):                                      # 16-bit features: the reference sums the exactly widened values
        feat = torch.from_numpy(feat).to(torch.bfloat16 if layout == 2 else torch.float16).float().numpy()
    idx = rng.integers(0, GCELLS, (GE, GH // 2 + 1, GW // 16 + 1)).repeat(2, 1).repeat(16, 2)[:, :GH, :GW].astype(np.int32)
    idx[:, ::5, ::3] = rng.integers(0, GCELLS, idx[:, ::5, ::3].shape)
    samp = (rng.uniform(size=(GE, GH, GW)) < 0.3).astype(np.uint8) if with_samp else None
    sums0 = rng.standard_normal((GE, GCELLS, C_)).astype(np.float32)
    counts0 = rng.integers(0, 4, (GE, GCELLS)).astype(np.float32)
    norm0 = rng.standard_normal((GE, GCELLS, C_)).astype(np.float16)
    f = torch.from_numpy(feat).to(cuda)
    f[idle] = float("nan")
    if layout:
        f = f.transpose(1, 2).contiguous()
        if layout in (2, 3):
            f = f.to(torch.bfloat16 if layout == 2 else torch.float16)
    d_idx, d_samp = torch.from_numpy(idx).to(cuda), None if samp is None else torch.from_numpy(samp).to(cuda)
    d_sums, d_counts, d_norm = (torch.from_numpy(x).to(cuda) for x in (sums0, counts0, norm0))
    d_cnt = torch.zeros((GE, GCELLS), dtype=torch.int32, device=cuda)
    d_touched = torch.zeros((GE, GCELLS), dtype=torch.uint8, device=cuda)
    ops.frame_count(d_idx, d_samp, d_cnt, act)
    ops.write_mean(f, d_idx, d_samp, d_cnt, d_sums, layout, variant, None, act)
    ops.finalize_counts(d_idx, d_cnt, d_counts, d_touched, d_sums, d_norm)
    torch.cuda.synchronize()
    assert not d_cnt.any()                                    # scratch back to zero
    got_s, got_c, got_n, got_t = d_sums.cpu(), d_counts.cpu().numpy(), d_norm.cpu(), d_touched.cpu().numpy()
    for e in range(GE):
        if not ACTIVE_G[e]:
            assert torch.equal(bits(got_s[e]), bits(torch.from_numpy(sums0[e]))), f"idle slot {e}: sums"
            assert np.array_equal(got_c[e], counts0[e]), f"idle slot {e}: counts"
            assert torch.equal(bits(got_n[e]), bits(torch.from_numpy(norm0[e]))), f"idle slot {e}: norm16"
            assert not got_t[e].any(), f"idle slot {e}: touched"
            continue
        rs, rc, n = ref_write(sums0[e].astype(np.float64), counts0[e].astype(np.float64), feat[e], idx[e], None if samp is None else samp[e])
        assert_sums(got_s[e], rs, f"slot {e}")
        assert np.array_equal(got_s[e].numpy()[n == 0], sums0[e][n == 0]), f"slot {e}: cells without samples were written"
        assert np.array_equal(got_c[e], rc), f"slot {e}: counts"
        assert np.array_equal(got_t[e].astype(bool), n > 0), f"slot {e}: touched"
        vis = np.unique(idx[e])
        ref16 = R.create_implicit_memory(got_s[e], torch.from_numpy(got_c[e])).half()
        assert torch.equal(bits(got_n[e][vis]), bits(ref16[vis])), f"slot {e}: refreshed fp16 rows"
        hidden = np.setdiff1d(np.arange(GCELLS), vis)
        assert torch.equal(bits(got_n[e][hidden]), bits(torch.from_numpy(norm0[e][hidden]))), f"slot {e}: hidden fp16 rows"


# --------------------------------------------------------------------------------------------------------
# H  the static tile partition of the TMA write (work == nullptr: every captured launch) against the tickets
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H_,W_,E_", [(32, 40, 1), (32, 41, 1), (32, 41, 3), (480, 640, 2)],
                         ids=["20-groups", "41-tiles", "123-tiles", "480x640x2"])
@pytest.mark.parametrize("with_active", [False, True], ids=["all", "active"])
def test_tma_write_static_partition_in_a_graph(eod, cuda, H_, W_, E_, with_active):
    """frame_count -> write_mean(CHW, TMA) -> finalize_counts captured in a CUDA graph after an eager warm-up, then replayed: a
    captured launch takes the static partition (CTA b: groups b, b+G, ...).  Shapes on the scheduler's edges: an odd tile count
    (group size 1), a last chunk of tickets only partly full, fewer groups than SMs, and 480x640 x 2 (many groups per CTA).  The
    replay and the eager (ticketed) launch both match the float64 reference, counts and touched sets exact; idle slots untouched."""
    ops, lib = eod.ops, eod._lib
    rng = np.random.default_rng(H_ * W_ + E_)
    HW = H_ * W_
    cells = 300 if HW < 5000 else 2000
    act_l = [0 if (with_active and e % 2) else 1 for e in range(E_)]
    act = i32(act_l, cuda) if with_active else None
    feat = rng.standard_normal((E_, C, HW)).astype(np.float32)
    idx = rng.integers(0, cells, (E_, H_ // 2 + 1, W_ // 8 + 1)).repeat(2, 1).repeat(8, 2)[:, :H_, :W_].reshape(E_, HW).astype(np.int32)
    idx[:, ::7] = rng.integers(0, cells, idx[:, ::7].shape)
    sums0 = rng.standard_normal((E_, cells, C)).astype(np.float32)
    counts0 = rng.integers(0, 3, (E_, cells)).astype(np.float32)
    f = torch.from_numpy(feat).to(cuda)
    for e in range(E_):
        if not act_l[e]:
            f[e] = float("nan")
    d_idx = torch.from_numpy(idx).to(cuda)

    def state():
        return (torch.from_numpy(sums0).to(cuda), torch.from_numpy(counts0).to(cuda), torch.zeros((E_, cells), dtype=torch.int32, device=cuda),
                torch.zeros((E_, cells), dtype=torch.uint8, device=cuda))

    def frame(st):
        sums, counts, cnt, touched = st
        ops.frame_count(d_idx, None, cnt, act)
        ops.write_mean(f, d_idx, None, cnt, sums, lib.LAYOUT_CHW, lib.WRITE_TMA, None, act)
        ops.finalize_counts(d_idx, cnt, counts, touched)

    eager = state()
    frame(eager)                                              # ticketed, and the warm-up of the capture
    torch.cuda.synchronize()
    replayed = state()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        frame(replayed)
    torch.cuda.synchronize()
    assert torch.equal(replayed[0].cpu(), torch.from_numpy(sums0))            # capturing ran nothing
    graph.replay()
    torch.cuda.synchronize()
    for name, st in (("eager", eager), ("replay", replayed)):
        assert not st[2].any(), name
        for e in range(E_):
            got_s, got_c, got_t = st[0][e].cpu(), st[1][e].cpu().numpy(), st[3][e].cpu().numpy()
            if not act_l[e]:
                assert torch.equal(bits(got_s), bits(torch.from_numpy(sums0[e]))) and np.array_equal(got_c, counts0[e]) and not got_t.any(), \
                    f"{name}: idle slot {e} changed"
                continue
            rs, rc, n = ref_write(sums0[e].astype(np.float64), counts0[e].astype(np.float64), feat[e], idx[e])
            assert_sums(got_s, rs, f"{name} slot {e}")
            assert np.array_equal(got_c, rc), f"{name} slot {e}: counts"
            assert np.array_equal(got_t.astype(bool), n > 0), f"{name} slot {e}: touched"
    del graph


# --------------------------------------------------------------------------------------------------------
# I  the first ticketed launch of a process inside a capture (launch_tma_kernel: the pool must not be touched there)
# --------------------------------------------------------------------------------------------------------
FIRST_TICKETED_LAUNCH_IN_CAPTURE = r"""
import importlib
import torch
eod = importlib.import_module("embodied-object-detection_b200")
ops, lib = eod.ops, eod._lib
dev = torch.device("cuda:0")
E, C, H, W, cells = 2, 128, 32, 64, 300
g = torch.Generator(device=dev).manual_seed(0)
feat = torch.randn((E, C, H * W), device=dev, generator=g)
idx = torch.randint(0, cells, (E, H // 2, W // 4), device=dev, generator=g, dtype=torch.int32).repeat_interleave(2, 1).repeat_interleave(4, 2)
idx = idx.reshape(E, H * W).contiguous()

def state():
    return torch.zeros((E, cells, C), device=dev), torch.zeros((E, cells), device=dev), torch.zeros((E, cells), dtype=torch.int32, device=dev)

def frame(st, variant):
    sums, counts, cnt = st
    ops.frame_count(idx, None, cnt)
    ops.write_mean(feat, idx, None, cnt, sums, lib.LAYOUT_CHW, variant)
    ops.finalize_counts(idx, cnt, counts)

warm = state()
frame(warm, lib.WRITE_LDG)              # same shape, no ticketed launch: the count / finalize kernels and the library are warm
torch.cuda.synchronize()
captured = state()
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph):
    frame(captured, lib.WRITE_TMA)      # the first launch of the process that would draw a ticket
graph.replay()
eager = state()
frame(eager, lib.WRITE_TMA)
torch.cuda.synchronize()
scale = float(eager[0].abs().max())
for name, st in (("replay", captured), ("ldg", warm)):
    err = float((st[0] - eager[0]).abs().max())
    assert scale > 0 and err <= 1e-6 * scale, (name, err, scale)
    assert torch.equal(st[1], eager[1]) and torch.equal(st[0] == 0, eager[0] == 0), name
print("capture ok")
"""


def test_first_ticketed_launch_of_a_process_inside_a_capture(eod, cuda):
    """In a fresh process whose first TMA write is captured into a graph (eager module loading, so that lazy loading is not a
    confound): the capture and the replay succeed, and the replay equals an eager TMA write and the LDG write of the same frame."""
    env = dict(os.environ, CUDA_MODULE_LOADING="EAGER")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", FIRST_TICKETED_LAUNCH_IN_CAPTURE]
    r = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=240)
    assert r.returncode == 0 and "capture ok" in r.stdout, f"exit {r.returncode}\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"


# --------------------------------------------------------------------------------------------------------
# J  two batches driven from two caller streams (shared ticket pool, tensor-map cache)
# --------------------------------------------------------------------------------------------------------
def test_two_batches_on_two_caller_streams(eod, cuda, scene, sleep_cycles):
    """Two pipelined batches (default TMA write), each driven from its own caller stream with late features, their steps interleaved
    without a host synchronisation.  Each matches its own serial twin (levels within one fp16 ulp) and the float64 reference.
    The features are positive: zero-mean features pool to values near zero, where the last-bit differences of two reduction
    orders span many fp16 ulps."""
    s = scene
    feats = [f.abs() + 0.5 for f in s.feat]
    frames = [list(range(s.T)), list(reversed(range(s.T)))]            # the second batch walks the frames backwards
    batches = [eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda, pipeline=True) for _ in range(2)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    feat_bufs = [[torch.empty_like(feats[0]) for _ in range(2)] for _ in range(2)]      # step t's features live until step t+1 returned
    levels = [[], []]
    torch.cuda.synchronize()
    for t in range(s.T):
        for i in (0, 1):
            f = frames[i][t]
            with torch.cuda.stream(streams[i]):
                buf = feat_bufs[i][t & 1]
                late(sleep_cycles, lambda: buf.copy_(feats[f]))
                lv = batches[i].step(s.depth[f], s.pose[f], s.shifts, s.intr, CELL, buf)
                assert_busy(f"batch {i} t={t}")
                levels[i].append([l.clone() for l in lv])
    for i in (0, 1):
        with torch.cuda.stream(streams[i]):
            batches[i].join()
    torch.cuda.synchronize()
    for i in (0, 1):
        twin = eod.EpisodeBatch(s.E, MW, MH, C, H, W, cuda)
        ref_s = np.zeros((s.E, MW * MH, C))
        ref_c = np.zeros((s.E, MW * MH))
        for t, f in enumerate(frames[i]):
            assert_levels_close(levels[i][t], twin.step(s.depth[f], s.pose[f], s.shifts, s.intr, CELL, feats[f]), f"batch {i} t={t}")
            for e in range(s.E):
                ref_s[e], ref_c[e], _ = ref_write(ref_s[e], ref_c[e], feats[f][e].cpu().numpy(), s.idx[f][e])
        torch.cuda.synchronize()
        assert np.array_equal(batches[i].counts.cpu().numpy(), ref_c), f"batch {i}: counts"
        assert_sums(batches[i].sums, ref_s, f"batch {i}")
