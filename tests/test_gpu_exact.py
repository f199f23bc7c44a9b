"""The accumulating kernels held to the bit on exactly summable inputs (tests/exact_cases.py): the mean write in every variant, the
object write with flush_slots, the frame loop built on them, project_fuse, linear_rows and semmap_update.

On these inputs every partial sum is exact in fp32, so the result does not depend on the reduction order and a correct kernel returns
the float64 result - an fp32 number - bit for bit.  Every assertion here is torch.equal or an equality of raw bits; none uses a
tolerance.  A cell that loses or double-counts one of its 2^18 pixels, a contribution sent to another cell, or a GEMM that drops the
lo term of one K block fails here, where the tolerance tests of test_gpu_parity.py can pass."""
import math

import numpy as np
import pytest
import torch

from oracle import reference_ops as R

import exact_cases as X
from test_gpu_scale import device_sms, semmap_update_sweeps

pytestmark = pytest.mark.gpu


def _t(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t if dtype is None else t.to(dtype)


def _exact32(ref64: np.ndarray) -> torch.Tensor:
    """The fp32 tensor equal to a float64 result that must be an fp32 number."""
    r32 = np.asarray(ref64).astype(np.float32)
    assert np.array_equal(r32.astype(np.float64), ref64), "the reference is not an fp32 number: the case is not exactly summable"
    return torch.from_numpy(r32)


def _same_bits(got: torch.Tensor, ref: torch.Tensor, what) -> None:
    g, r = got.detach().contiguous().cpu(), ref.contiguous().cpu()
    assert g.shape == r.shape and g.dtype == r.dtype, (what, g.shape, r.shape, g.dtype, r.dtype)
    itype = {torch.float32: torch.int32, torch.float16: torch.int16}[g.dtype]
    bad = int((g.view(itype) != r.view(itype)).sum())
    assert bad == 0, (what, f"{bad} elements differ")


def _norm16(sums64: np.ndarray, counts: np.ndarray) -> torch.Tensor:
    """create_implicit_memory(...).half() of an fp32 state (custom_rcnn.py:764-774)."""
    return R.create_implicit_memory(torch.from_numpy(np.asarray(sums64, np.float32)), torch.from_numpy(np.asarray(counts, np.float32))).half()


# ------------------------------------------------------------------------------------------------------------------------------
# mean write: every kernel, with and without samp, active mask, dyadic initial sums, the 2^18-pixel cell
# ------------------------------------------------------------------------------------------------------------------------------
# kind -> (variant, layout, expand): EOD_WRITE_LDG / _TMA on CHW, AUTO on the channels-last layouts, the deterministic write
KINDS = {"ldg": (1, 0, False), "tma": (2, 0, False), "tma+expand": (2, 0, True), "hwc-f32": (0, 1, False), "hwc-bf16": (0, 2, False),
         "hwc-f16": (0, 3, False), "det": (None, 0, False)}
RAGGED_KINDS = {"auto-ldg": (0, 0, False), "hwc-f32": (0, 1, False), "hwc-bf16": (0, 2, False), "hwc-f16": (0, 3, False)}


def _write_case(rng, E, H, W, cells, C, samp_p, big=None, qf=3):
    samp = None
    if samp_p is not None:
        samp = rng.random((E, H, W)) < samp_p
        samp[0, : H // 3] = False                                          # whole tiles without a sample
    max_log2 = 6 if big is None else 12
    idx = np.stack([X.index_plane(rng, H, W, cells, None if samp is None else samp[e], max_log2, big) for e in range(E)])
    feat = X.dyadic(rng, (E, C, H, W), 3, qf)                            # 4 significant bits: exact in bf16 and fp16
    n_max = max(int(X.sample_counts(idx[e], None if samp is None else samp[e], cells).max()) for e in range(E))
    q = qf + int(math.log2(n_max))
    sums0 = X.dyadic(rng, (E, cells, C), 20, q)                          # dyadic initial sums, |x| < 2^(20-q)
    counts0 = rng.integers(0, 4, (E, cells)).astype(np.float32)
    return feat, idx, samp, sums0, counts0, q


def _run_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, active):
    variant, layout, expand = {**KINDS, **RAGGED_KINDS}[kind]
    E, C, H, W = feat.shape
    cells = sums0.shape[1]
    d_idx = _t(idx, cuda)
    d_samp = None if samp is None else _t(samp.astype(np.uint8), cuda)
    d_sums, d_counts = _t(sums0, cuda), _t(counts0, cuda)
    d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    d_touched = torch.zeros((E, cells), dtype=torch.uint8, device=cuda)
    d_norm = torch.zeros((E, cells, C), dtype=torch.float16, device=cuda)
    d_act = None if active is None else _t(active, cuda)
    if layout == 0:
        f_dev = _t(feat, cuda)
    else:
        f_dev = _t(feat.transpose(0, 2, 3, 1), cuda)
        if layout in (2, 3):
            f_dev = f_dev.to(torch.bfloat16 if layout == 2 else torch.float16)
    eod.ops.frame_count(d_idx, d_samp, d_cnt, d_act)
    if variant is None:
        ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda, H * W)
        eod.ops.write_mean_det(f_dev, d_idx, d_samp, d_cnt, d_sums, ws)
    else:
        pix = eod.ops.expand_counts(d_idx, d_cnt, torch.empty((E, H, W), device=cuda)) if expand else None
        eod.ops.write_mean(f_dev, d_idx, d_samp, d_cnt, d_sums, layout, variant, pix, d_act)
    eod.ops.finalize_counts(d_idx, d_cnt, d_counts, d_touched, d_sums, d_norm)
    torch.cuda.synchronize()
    if variant is None:
        assert not ws.overflowed()
    return d_sums, d_counts, d_touched, d_norm, d_cnt


def _check_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, q, active=None):
    E, C = feat.shape[:2]
    cells = sums0.shape[1]
    d_sums, d_counts, d_touched, d_norm, d_cnt = _run_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, active)
    assert int(d_cnt.abs().sum()) == 0, "frame_cnt is not back to zero"
    for e in range(E):
        live = active is None or active[e] > 0
        se = None if samp is None else samp[e]
        ref, bound, n = X.mean_write_f64(sums0[e], feat[e], idx[e], se, cells)
        X.assert_pow2_counts(n)
        X.check_lattice([feat[e], sums0[e], ref], q, bound)
        if not live:
            ref, n = sums0[e].astype(np.float64), np.zeros(cells, np.int64)
        _same_bits(d_sums[e], _exact32(ref), (kind, e, "sums"))
        vis = np.zeros(cells, bool)
        if live:
            vis[np.unique(idx[e])] = True
        counts = counts0[e] + vis
        assert np.array_equal(d_counts[e].cpu().numpy(), counts), (kind, e, "counts")
        assert np.array_equal(d_touched[e].cpu().numpy().astype(bool), n > 0), (kind, e, "touched")
        want16 = torch.where(torch.from_numpy(vis)[:, None], _norm16(ref, counts), torch.zeros((), dtype=torch.float16))
        _same_bits(d_norm[e], want16, (kind, e, "norm16"))
        if samp is not None and live:
            assert (vis & (n == 0)).any()                                    # some cells were visible without a sample (bit 31)


@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("kind", list(KINDS))
def test_mean_write_exact_e3(eod, cuda, kind, C):
    """E=3 at 96x128: dense, sampled (whole tiles without a sample, cells visible without one) with an active mask that idles a slot,
    dyadic initial sums."""
    rng = np.random.default_rng(C + len(kind))
    for samp_p, active in ((None, None), (0.3, np.array([1, 0, 2], np.int32))):
        if KINDS[kind][0] is None:
            active = None                                                    # the deterministic write takes no active mask
        feat, idx, samp, sums0, counts0, q = _write_case(rng, 3, 96, 128, 2700, C, samp_p)
        _check_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, q, active)


@pytest.mark.parametrize("kind", list(RAGGED_KINDS))
def test_mean_write_exact_ragged(eod, cuda, kind):
    """HW % 32 != 0 (30x52): the kernels that take it (AUTO picks the LDG kernel for CHW)."""
    rng = np.random.default_rng(31)
    for C in (128, 256, 512):
        for samp_p, active in ((None, None), (0.5, np.array([2, 0], np.int32))):
            feat, idx, samp, sums0, counts0, q = _write_case(rng, 2, 30, 52, 800, C, samp_p)
            _check_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, q, active)


@pytest.mark.parametrize("kind,C", [(k, 128) for k in KINDS] + [("tma", 256), ("tma", 512)])
def test_mean_write_exact_cell_of_2_18_pixels(eod, cuda, kind, C):
    """480x640 with one cell of 2^18 sampled pixels (a wall filling the frame at close range): one lost or double-counted pixel moves
    its mean by |f| / 2^18."""
    rng = np.random.default_rng(18 + C)
    feat, idx, samp, sums0, counts0, q = _write_case(rng, 1, 480, 640, 4000, C, None, big=1 << 18)
    _check_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, q)
    if kind == "tma":                                                      # the same cell with samples: 2^18 of ~290 k sampled pixels
        samp = (rng.random((1, 480, 640)) < 0.95)
        idx = X.index_plane(rng, 480, 640, 4000, samp[0], 12, 1 << 18)[None]
        _check_write(eod, cuda, kind, feat, idx, samp, sums0, counts0, q)


# ------------------------------------------------------------------------------------------------------------------------------
# object regime: write_objects / write_objects_pasted + flush_slots
# ------------------------------------------------------------------------------------------------------------------------------
def _object_frame(rng, E, H, W, C, cells, n_obj, n_base=6, copies=(1, 2, 4)):
    """Per episode: detections with 1/2/4 overlaps, the idx plane built on the stride-8 sample ranks, garbage beyond n_obj."""
    cases = [X.object_case(rng, H, W, C, n_base, copies=copies) if n_obj[e] else None for e in range(E)]
    Kmax = max([c["masks"].shape[0] for c in cases if c is not None] + [int(max(n_obj)), 1])
    bf = np.full((E, Kmax, C), 1e6, np.float32)
    probs = np.ones((E, Kmax, 28, 28), np.float32)
    boxes = np.tile(np.array([0, 0, W, H], np.float32), (E, Kmax, 1))
    masks = np.ones((E, Kmax, H, W), bool)
    idx = np.empty((E, H, W), np.int32)
    n_obj = np.array(n_obj, np.int32)
    for e in range(E):
        c = cases[e]
        if c is None:
            idx[e] = rng.integers(0, cells, (H, W))
            continue
        k = c["masks"].shape[0]
        n_obj[e] = k
        bf[e, :k], probs[e, :k], boxes[e, :k], masks[e, :k] = c["box_features"], c["probs"], c["boxes"], c["masks"]
        samp = R.sample_mask(torch.from_numpy(c["masks"].any(0)), 8).numpy()
        idx[e] = X.index_plane(rng, H, W, cells, samp, 4)
    return bf, probs, boxes, masks, n_obj, idx


def _object_oracle(sums, counts, bf, masks, idx, n):
    """One frame of the reference chain box_to_image_features -> project_image_features -> accumulate (exact on these inputs)."""
    if not n:
        return sums, counts
    img, obs = R.box_to_image_features(torch.from_numpy(bf[:n]), torch.from_numpy(masks[:n]))
    mean = X.object_mean_f64(bf[:n], masks[:n])
    samp = R.sample_mask(obs, 8).numpy()
    ref, bound, cnt = X.mean_write_f64(sums.numpy(), mean.reshape(-1, *idx.shape), idx, samp, sums.shape[0])
    X.assert_pow2_counts(cnt)
    X.check_lattice([bf[:n], sums.numpy(), ref], 2 + 2 + int(math.log2(max(int(cnt.max()), 1))), bound)
    s, c = R.write_mean_frame(sums, counts, img, obs, torch.from_numpy(idx).long(), stride=8)
    assert np.array_equal(s.numpy().astype(np.float64), ref)
    return s, c


@pytest.mark.parametrize("pasted", [False, True], ids=["masks", "pasted"])
def test_object_write_and_flush_exact_through_ops(eod, cuda, pasted):
    """masks_observed / paste -> sample_mask -> frame_count(slots) -> write_objects[_pasted] -> flush_slots -> finalize_counts:
    ragged n_obj with an empty episode, garbage beyond n_obj, three frames accumulating; then more than 128 objects."""
    rng = np.random.default_rng(40 + pasted)
    H, W, C, mw, mh = 96, 128, 128, 50, 40
    cells = mw * mh
    for E, n_base, copies, frames in ((3, 6, (1, 2, 4), ([1, 0, 1], [1, 1, 0], [0, 1, 1])), (1, 36, (4,), ([1],))):
        slots = eod.ops.ObjectSlots(E, cells, C, -(-H * W // 8), cuda)
        d_sums = torch.zeros((E, cells, C), device=cuda)
        d_counts = torch.zeros((E, cells), device=cuda)
        d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
        sums = [torch.zeros(cells, C) for _ in range(E)]
        counts = [torch.zeros(cells) for _ in range(E)]
        for has in frames:
            bf, probs, boxes, masks, n_obj, idx = _object_frame(rng, E, H, W, C, cells, has, n_base, copies)
            if E == 1:
                assert n_obj[0] > 128
            d_n = _t(n_obj, cuda)
            d_idx = _t(idx, cuda)
            if pasted:
                _, observed = eod.ops.paste_masks(_t(probs, cuda), _t(boxes, cuda), (H, W), 0.5, d_n, want_masks=False, want_observed=True)
            else:
                observed = eod.ops.masks_observed(_t(masks, cuda), d_n)
            samp = eod.ops.sample_mask(observed, 8)
            eod.ops.frame_count(d_idx, samp, d_cnt, d_n, slots)
            if pasted:
                eod.ops.write_objects_pasted(_t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), d_n, d_idx, samp, slots)
            else:
                eod.ops.write_objects(_t(bf, cuda), _t(masks, cuda), d_n, d_idx, samp, slots)
            eod.ops.flush_slots(d_cnt, slots, d_sums)
            eod.ops.finalize_counts(d_idx, d_cnt, d_counts)
            torch.cuda.synchronize()
            assert int(d_cnt.abs().sum()) == 0 and not slots.scratch.any() and not slots.slot_of_cell.any()
            for e in range(E):
                sums[e], counts[e] = _object_oracle(sums[e], counts[e], bf[e], masks[e], idx[e], int(n_obj[e]) if has[e] else 0)
                _same_bits(d_sums[e], sums[e], (E, e, "sums"))
                assert torch.equal(d_counts[e].cpu(), counts[e]), (E, e, "counts")
            slots.n_slots.zero_()


@pytest.mark.parametrize("pasted", [False, True], ids=["write_objects", "write_detections"])
def test_object_write_exact_through_episode_batch(eod, cuda, pasted):
    """EpisodeBatch.write_objects / write_detections: sums, counts and the fp16 table bit for bit, over three frames."""
    rng = np.random.default_rng(50 + pasted)
    E, H, W, C, mw, mh = 3, 96, 128, 256, 50, 40
    cells = mw * mh
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    sums = [torch.zeros(cells, C) for _ in range(E)]
    counts = [torch.zeros(cells) for _ in range(E)]
    for has in ([1, 1, 0], [0, 1, 1], [1, 0, 1]):
        bf, probs, boxes, masks, n_obj, idx = _object_frame(rng, E, H, W, C, cells, has)
        batch.set_indices(_t(idx, cuda))
        if pasted:
            batch.write_detections(_t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(n_obj * np.array(has, np.int32), cuda))
        else:
            batch.write_objects(_t(bf, cuda), _t(masks, cuda), _t(n_obj * np.array(has, np.int32), cuda))
        torch.cuda.synchronize()
        for e in range(E):
            sums[e], counts[e] = _object_oracle(sums[e], counts[e], bf[e], masks[e], idx[e], int(n_obj[e]) if has[e] else 0)
            _same_bits(batch.sums[e], sums[e], (e, "sums"))
            assert torch.equal(batch.counts[e].cpu(), counts[e]), (e, "counts")
            _same_bits(batch.norm16[e], R.create_implicit_memory(sums[e], counts[e]).half(), (e, "norm16"))


# ------------------------------------------------------------------------------------------------------------------------------
# frame loop: step / step_detections with proj_indices against the serial oracle chain write_mean_frame -> read_frame
# ------------------------------------------------------------------------------------------------------------------------------
class _Chain:
    """Serial oracle of one episode: state (sums, counts), the fp16 read table (a snapshot when read_frozen)."""

    def __init__(self, cells, C, frozen):
        self.sums, self.counts, self.frozen = torch.zeros(cells, C), torch.zeros(cells), frozen
        self.table = torch.zeros(cells, C, dtype=torch.float16)

    def reset(self):
        self.sums.zero_(), self.counts.zero_(), self.table.zero_()

    def refresh(self):
        self.table = R.create_implicit_memory(self.sums, self.counts).half()

    def read(self, idx):
        proj = torch.from_numpy(idx).long()
        return R.read_pool(self.table, proj) if self.frozen else R.read_frame(self.sums, self.counts, proj)

    def norm16(self):
        return self.table if self.frozen else R.create_implicit_memory(self.sums, self.counts).half()


def _check_levels(got, ref, what):
    for k in range(3):
        _same_bits(got[k], ref[k][0], what + (k,))


@pytest.mark.parametrize("fp16_table", [True, False], ids=["table", "no-table"])
@pytest.mark.parametrize("variant", ["auto", "det"])
@pytest.mark.parametrize("pipeline", [False, True], ids=["ordered", "pipelined"])
def test_step_frame_loop_exact(eod, cuda, pipeline, variant, fp16_table):
    """Six frames of EpisodeBatch.step(proj_indices=...): samp on some frames, a mid-run reset_mask, refresh_mask (read_frozen with
    the fp16 table in the pipelined mode), active masks (default variant): every frame's three levels, and sums / counts / norm16 at
    the end, equal the serial oracle chain bit for bit."""
    E, H, W, C, mw, mh, T = 3, 96, 128, 128, 60, 45, 6
    cells = mw * mh
    det = variant == "det"
    frozen = fp16_table and pipeline
    rng = np.random.default_rng(60 + 4 * pipeline + 2 * det + fp16_table)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, variant=eod._lib.WRITE_DET if det else eod._lib.WRITE_AUTO, pipeline=pipeline,
                             fp16_table=fp16_table)
    batch.det_runs_per_episode = H * W
    batch.read_frozen = frozen
    chains = [_Chain(cells, C, frozen) for _ in range(E)]
    depth = torch.zeros((E, H, W), device=cuda)
    pose = torch.zeros((E, 12), device=cuda)
    shifts = torch.zeros((E, 6), device=cuda)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    plan = [dict(), dict(samp=0.4), dict(reset=[0, 1, 0], active=[1, 1, 0]), dict(refresh=[1, 0, 1]), dict(samp=0.3, active=[0, 2, 1]),
            dict(reset=[1, 0, 0], refresh=[1, 1, 0])]
    got, want = [], []
    for t in range(T):
        p = plan[t]
        samp = (rng.random((E, H, W)) < p["samp"]) if "samp" in p else None
        idx = np.stack([X.index_plane(rng, H, W, cells, None if samp is None else samp[e], 5) for e in range(E)])
        feat = X.dyadic(rng, (E, C, H, W), 3, 3)
        active = None if det or "active" not in p else np.array(p["active"], np.int32)
        kw = dict(proj_indices=_t(idx, cuda))
        for key in ("reset", "refresh"):
            if key in p:
                kw[key + "_mask"] = _t(np.array(p[key], np.int32), cuda)
        if active is not None:
            kw["active"] = _t(active, cuda)
        levels = batch.step(depth, pose, shifts, intr, 0.2, _t(feat, cuda), None if samp is None else _t(samp.astype(np.uint8), cuda), **kw)
        got.append([l.clone() for l in levels])
        ref_levels = []
        for e, ch in enumerate(chains):
            if p.get("reset", [0] * E)[e]:
                ch.reset()
            if p.get("refresh", [0] * E)[e] and fp16_table:
                ch.refresh()
            ref_levels.append(ch.read(idx[e]))
            if active is None or active[e] > 0:
                se = None if samp is None else samp[e]
                ref, bound, n = X.mean_write_f64(ch.sums.numpy(), feat[e], idx[e], se, cells)
                X.assert_pow2_counts(n)
                X.check_lattice([feat[e], ch.sums.numpy(), ref], 3 + 5, bound)
                ch.sums = _exact32(ref)
                ch.counts[torch.from_numpy(np.unique(idx[e])).long()] += 1
        want.append(ref_levels)
    batch.join()
    torch.cuda.synchronize()
    for t in range(T):
        for e in range(E):
            _check_levels([l[e] for l in got[t]], want[t][e], (t, e))
    for e, ch in enumerate(chains):
        _same_bits(batch.sums[e], ch.sums, (e, "sums"))
        assert torch.equal(batch.counts[e].cpu(), ch.counts), (e, "counts")
        if fp16_table:
            _same_bits(batch.norm16[e], ch.norm16(), (e, "norm16"))
    assert float(batch.counts.max()) >= 3


@pytest.mark.parametrize("fp16_table", [True, False], ids=["table", "no-table"])
@pytest.mark.parametrize("pipeline", [False, True], ids=["ordered", "pipelined"])
def test_step_detections_frame_loop_exact(eod, cuda, pipeline, fp16_table):
    """Five frames of EpisodeBatch.step_detections(proj_indices=...) with ragged n_obj (idle slots pass 0), a reset and a refresh
    (read_frozen with the table in the pipelined mode): levels, sums, counts and norm16 equal the serial oracle chain bit for bit."""
    E, H, W, C, mw, mh = 3, 96, 128, 128, 50, 40
    cells = mw * mh
    frozen = fp16_table and pipeline
    rng = np.random.default_rng(70 + 2 * pipeline + fp16_table)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, pipeline=pipeline, fp16_table=fp16_table)
    batch.read_frozen = frozen
    chains = [_Chain(cells, C, frozen) for _ in range(E)]
    depth = torch.zeros((E, H, W), device=cuda)
    pose = torch.zeros((E, 12), device=cuda)
    shifts = torch.zeros((E, 6), device=cuda)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    plan = [dict(has=[1, 1, 0]), dict(has=[1, 0, 1]), dict(has=[1, 1, 1], reset=[0, 1, 0]), dict(has=[0, 1, 1], refresh=[1, 1, 0]),
            dict(has=[1, 1, 1], refresh=[0, 0, 1])]
    got, want = [], []
    for t, p in enumerate(plan):
        bf, probs, boxes, masks, n_obj, idx = _object_frame(rng, E, H, W, C, cells, p["has"])
        n_obj = n_obj * np.array(p["has"], np.int32)
        kw = dict(proj_indices=_t(idx, cuda))
        for key in ("reset", "refresh"):
            if key in p:
                kw[key + "_mask"] = _t(np.array(p[key], np.int32), cuda)
        args = (_t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(n_obj, cuda))
        levels = batch.step_detections(depth, pose, shifts, intr, 0.2, *args, **kw)
        got.append([l.clone() for l in levels])
        ref_levels = []
        for e, ch in enumerate(chains):
            if p.get("reset", [0] * E)[e]:
                ch.reset()
            if p.get("refresh", [0] * E)[e] and fp16_table:
                ch.refresh()
            ref_levels.append(ch.read(idx[e]))
            ch.sums, ch.counts = _object_oracle(ch.sums, ch.counts, bf[e], masks[e], idx[e], int(n_obj[e]))
        want.append(ref_levels)
    batch.join()
    torch.cuda.synchronize()
    for t in range(len(plan)):
        for e in range(E):
            _check_levels([l[e] for l in got[t]], want[t][e], (t, e))
    for e, ch in enumerate(chains):
        _same_bits(batch.sums[e], ch.sums, (e, "sums"))
        assert torch.equal(batch.counts[e].cpu(), ch.counts), (e, "counts")
        if fp16_table:
            _same_bits(batch.norm16[e], ch.norm16(), (e, "norm16"))
    assert float(batch.counts.max()) >= 2


# ------------------------------------------------------------------------------------------------------------------------------
# projection: project_fuse / project_fuse_levels (tcgen05, fp16 level x hi/lo-split weight) and MemoryFusion
# ------------------------------------------------------------------------------------------------------------------------------
def _proj_ref(x16, Wt, b, res, weight, mode):
    """float64 timm.py:174-184 on (E,h,w,K) levels -> (E,N,h,w), with the lattice check of the split GEMM."""
    E, h, w, K = x16.shape
    x64 = x16.astype(np.float64).reshape(-1, K)
    hi, lo = X.split_weights_f64(Wt)
    assert np.array_equal(hi.astype(np.float64) + lo.astype(np.float64) * 2.0 ** -11, Wt.astype(np.float64))
    mem = x64 @ Wt.astype(np.float64).T + (0 if b is None else b.astype(np.float64))
    mem = mem.reshape(E, h, w, -1).transpose(0, 3, 1, 2) * weight
    ref = mem + res.astype(np.float64) if mode == 0 else mem
    qx = X.lattice_q(x64)
    if lo.any():                                          # the lo accumulator x . W_lo on its own, then x . W_hi + 2^-11 (x . W_lo)
        X.check_lattice([x64 @ lo.astype(np.float64).T], qx + X.lattice_q(lo), float(X.gemm_bound(x64, lo).max()))
    q = max(qx + X.lattice_q(hi), qx + X.lattice_q(lo) + 11 if lo.any() else 0, X.lattice_q(ref), 0 if b is None else X.lattice_q(b))
    bound = weight * (float(X.gemm_bound(x64, Wt).max()) + (0 if b is None else float(np.abs(b).max()))) + \
        (float(np.abs(res).max()) if mode == 0 else 0)
    X.check_lattice([ref], q, bound)
    return _exact32(ref)


@pytest.mark.parametrize("E,h,w,K,N,lo", [(2, 60, 80, 512, 256, False), (3, 15, 20, 512, 256, False), (5, 7, 9, 64, 128, False),
                                          (2, 30, 40, 128, 128, True)])
def test_project_fuse_exact(eod, cuda, E, h, w, K, N, lo):
    """project_fuse and project_fuse_levels variants 1 and 2 (2 needs hw % 4 == 0), SUM / MEM_ONLY, bias on and off: bit for bit.
    ``lo``: weights with a nonzero W_lo, so the lo product and its 2^-11 rescale are exercised exactly."""
    rng = np.random.default_rng(E * 100 + K + lo)
    x16 = X.dyadic(rng, (E, h, w, K), 3, 2, np.float16)
    Wt = X.weights_with_lo(rng, (N, K)) if lo else X.dyadic(rng, (N, K), 3, 4)
    if lo:
        assert (X.split_weights_f64(Wt)[1] != 0).any()
    b = X.dyadic(rng, (N,), 10, 6)
    res = X.dyadic(rng, (E, N, h, w), 12, 6)
    wsplit = eod.ops.project_split_weights(_t(Wt, cuda))
    hi_d, lo_d = X.split_weights_f64(Wt)
    lvl = _t(x16, cuda).permute(0, 3, 1, 2)
    for weight in (5.0, 0.5):
        for mode, bias in ((0, b), (1, b), (0, None), (1, None)):
            ref = _proj_ref(x16, Wt, bias, res, weight, mode)
            bias_d = None if bias is None else _t(bias, cuda)
            res_d = _t(res, cuda) if mode == 0 else None
            _same_bits(eod.ops.project_fuse(lvl, wsplit, bias_d, res_d, weight, mode), ref, (weight, mode, bias is None, "project_fuse"))
            for variant in [1] + ([2] if (h * w) % 4 == 0 else []):
                out = eod.ops.project_fuse_levels([lvl], [wsplit], [bias_d], None if res_d is None else [res_d], weight, mode, variant=variant)[0]
                _same_bits(out, ref, (weight, mode, bias is None, variant))


@pytest.mark.parametrize("variant", [1, 2])
def test_project_fuse_three_levels_many_tiles_exact(eod, cuda, variant):
    """Three levels in one launch at E=24 (many tiles per CTA in the persistent kernel), SUM and MEM_ONLY: every level bit for bit."""
    rng = np.random.default_rng(24 + variant)
    E, K, N = 24, 512, 256
    shapes = [(60, 80), (30, 40), (15, 20)]
    xs = [X.dyadic(rng, (E, h, w, K), 3, 2, np.float16) for h, w in shapes]
    Ws = [X.dyadic(rng, (N, K), 3, 4) for _ in shapes]
    bs = [X.dyadic(rng, (N,), 10, 6) for _ in shapes]
    rs = [X.dyadic(rng, (E, N, h, w), 12, 6) for h, w in shapes]
    lv = [_t(x, cuda) for x in xs]
    ws = [eod.ops.project_split_weights(_t(Wt, cuda)) for Wt in Ws]
    for mode in (0, 1):
        outs = eod.ops.project_fuse_levels(lv, ws, [_t(b, cuda) for b in bs], [_t(r, cuda) for r in rs] if mode == 0 else None, 5.0, mode,
                                           variant=variant)
        for k in range(3):
            _same_bits(outs[k], _proj_ref(xs[k], Ws[k], bs[k], rs[k], 5.0, mode), (mode, k))


def _fusion_case(eod, cuda, rng, C=512, CO=256, H=96, W=128, cells=700):
    fus = eod.MemoryFusion("implicit_memory", "sum", 5, mem_feat_dim=C, ego_feat_dim=CO).to(cuda)
    sd = {}
    for k in range(3):
        sd[f"map_merge_projection{k + 1}.weight"] = torch.from_numpy(X.dyadic(rng, (CO, C, 1, 1), 2, 4))
        sd[f"map_merge_projection{k + 1}.bias"] = torch.from_numpy(X.dyadic(rng, (CO,), 10, 6))
    fus.load_state_dict(sd)
    table = X.dyadic(rng, (cells, C), 3, 2, np.float16)
    idx = rng.integers(0, cells, (H // 8, W // 8)).repeat(8, 0).repeat(8, 1).astype(np.int64)
    idx[::3, ::5] = rng.integers(0, cells, idx[::3, ::5].shape)
    res = [X.dyadic(rng, (1, CO, H >> s, W >> s), 10, 6) for s in (3, 4, 5)]
    levels = R.read_pool(torch.from_numpy(table), torch.from_numpy(idx))
    return fus, sd, table, idx, res, levels


def test_memory_fusion_tensor_core_forward_exact(eod, cuda):
    """MemoryFusion's fused tcgen05 forward (read -> one projection launch for three levels): each fused level bit for bit."""
    rng = np.random.default_rng(81)
    fus, sd, table, idx, res, levels = _fusion_case(eod, cuda, rng)
    with torch.no_grad():
        out = fus([_t(r, cuda) for r in res], [_t(table, cuda)], [_t(idx, cuda)], [None])
    for k in range(3):
        x16 = levels[k].permute(0, 2, 3, 1).contiguous().numpy()
        Wt = sd[f"map_merge_projection{k + 1}.weight"].numpy().reshape(res[k].shape[1], -1)
        _same_bits(out[k], _proj_ref(x16, Wt, sd[f"map_merge_projection{k + 1}.bias"].numpy(), res[k], 5.0, 0), k)


def test_memory_fusion_training_gradients_exact(eod, cuda):
    """The training path (eod_linear_rows forward and backward, incl. the transposed strided views of _LinearFn.backward): outputs and
    the gradients of weight, bias and res equal float64 autograd bit for bit (loss = sum(out * g) with dyadic g)."""
    rng = np.random.default_rng(82)
    fus, sd, table, idx, res, levels = _fusion_case(eod, cuda, rng, C=256, CO=128)
    gs = [X.dyadic(rng, r.shape, 3, 2) for r in res]
    res_g = [_t(r, cuda).requires_grad_(True) for r in res]
    out = fus(res_g, [_t(table, cuda)], [_t(idx, cuda)], [None])
    sum((o * _t(g, cuda)).sum() for o, g in zip(out, gs)).backward()
    for k, conv in enumerate(fus.merge_map_projections):
        w = sd[f"map_merge_projection{k + 1}.weight"].double().requires_grad_(True)
        b = sd[f"map_merge_projection{k + 1}.bias"].double().requires_grad_(True)
        r = torch.from_numpy(res[k]).double().requires_grad_(True)
        x = levels[k].double()
        o = r + 5.0 * torch.nn.functional.conv2d(x, w, b)
        (o * torch.from_numpy(gs[k]).double()).sum().backward()
        x2 = x[0].reshape(x.shape[1], -1).T.numpy()                        # (M, K): the rows of the forward GEMM
        g5 = 5.0 * gs[k][0].reshape(gs[k].shape[1], -1).T                  # (M, N): the gradient of the GEMM output
        assert X.tf32_exact(x2) and X.tf32_exact(g5) and X.tf32_exact(w.detach().numpy())
        X.check_lattice([o.detach().numpy()], X.lattice_q(o.detach().numpy()),
                        5 * (float(X.gemm_bound(x2, w.detach().numpy().reshape(w.shape[0], -1)).max()) + float(b.detach().abs().max()))
                        + float(np.abs(res[k]).max()))
        X.check_lattice([w.grad.numpy()], X.lattice_q(x2) + X.lattice_q(g5), float(X.gemm_bound(g5.T, x2.T).max()))
        X.check_lattice([b.grad.numpy()], X.lattice_q(g5), float(np.abs(g5).sum(0).max()))
        _same_bits(out[k], _exact32(o.detach().numpy()), (k, "out"))
        _same_bits(conv.weight.grad, _exact32(w.grad.numpy()), (k, "grad weight"))
        _same_bits(conv.bias.grad, _exact32(b.grad.numpy()), (k, "grad bias"))
        _same_bits(res_g[k].grad, _exact32(r.grad.numpy()), (k, "grad res"))


# ------------------------------------------------------------------------------------------------------------------------------
# linear_rows (3xTF32 on tcgen05) and the write_max replace path built on it
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,K,N", [(1, 64, 16), (127, 64, 256), (128, 96, 64), (300, 512, 256), (1000, 256, 512), (257, 20, 48)])
def test_linear_rows_exact(eod, cuda, M, K, N):
    """Operands with at most 11 significant bits survive the TF32 split: contiguous, transposed and padded operands, bias and scale,
    gathered rows (a_off) with a device-side count (m_count) scattered to y_dst rows - all bit for bit; other rows untouched."""
    rng = np.random.default_rng(M * 7 + K)
    a = X.dyadic(rng, (M, K), 6, 3)
    w = X.dyadic(rng, (N, K), 6, 6)
    b = X.dyadic(rng, (N,), 10, 9)
    assert X.tf32_exact(a) and X.tf32_exact(w)
    a64, w64, b64 = a.astype(np.float64), w.astype(np.float64), b.astype(np.float64)
    ref = (a64 @ w64.T + b64) * 0.75
    X.check_lattice([ref, a64 @ w64.T], 11, float(X.gemm_bound(a, w).max()) + float(np.abs(b).max()))
    ref32 = _exact32(ref)
    da, dw, db = _t(a, cuda), _t(w, cuda), _t(b, cuda)
    a_t = da.t().contiguous().t()
    w_pad = torch.zeros((N, K + 12), device=cuda)[:, 3:3 + K]
    w_pad.copy_(dw)
    for name, (aa, ww) in {"contiguous": (da, dw), "A transposed view": (a_t, dw), "W padded": (da, w_pad), "both": (a_t, w_pad)}.items():
        _same_bits(eod.ops.linear_rows(aa, ww, db, 0.75), ref32, name)
    _same_bits(eod.ops.linear_rows(da, dw), _exact32(a64 @ w64.T), "no bias")
    perm = torch.from_numpy(rng.permutation(M)).to(cuda)
    n_live = max(1, (2 * M) // 3)
    out = torch.full((M + 5, N), 7.0, device=cuda)
    eod.ops.linear_rows(da, dw, db, 1.0, out=out, a_off=(perm * K).to(torch.int64), m_count=torch.tensor([n_live], dtype=torch.int32, device=cuda),
                        n_rows=M, y_dst=(perm + 5).to(torch.int64))
    live = perm[:n_live].cpu()
    _same_bits(out[(live + 5).to(cuda)], _exact32((a64 @ w64.T + b64)[live.numpy()]), "gathered")
    untouched = torch.ones(M + 5, dtype=torch.bool)
    untouched[live + 5] = False
    assert bool((out.cpu()[untouched] == 7.0).all())


@pytest.mark.parametrize("layout", [0, 1])
def test_write_max_replace_with_linlayer_exact(eod, cuda, layout):
    """SMNet 'replace' with the linear layer: state[raised cells] = F.linear(winner features) bit for bit (float64 reference), other
    rows untouched, over three frames."""
    rng = np.random.default_rng(90 + layout)
    H, W, C_in, C_mem, mw, mh, T, stride = 48, 64, 64, 256, 23, 19, 3, 2
    cells = mw * mh
    lin_w = X.dyadic(rng, (C_mem, C_in), 6, 6)
    lin_b = X.dyadic(rng, (C_mem,), 10, 6)
    state = torch.zeros(cells, C_mem, dtype=torch.float64)
    observed = torch.zeros(cells, dtype=torch.bool)
    hmap = torch.zeros(cells)
    d_state = torch.zeros((1, cells, C_mem), device=cuda)
    d_obs = torch.zeros((1, cells), dtype=torch.uint8, device=cuda)
    d_hmap = torch.zeros((1, cells), device=cuda)
    d_key = torch.zeros((1, cells), dtype=torch.int64, device=cuda)
    d_arg = torch.zeros((1, cells), dtype=torch.int32, device=cuda)
    for t in range(T):
        w2m = np.stack([rng.integers(0, mw, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1), rng.integers(0, mh, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1)], -1)
        inl = rng.uniform(size=(H, W)) < 0.7
        heights = (np.round(rng.uniform(-1.5, 1.0, (H, W)) * 4) / 4).astype(np.float32)
        feat = X.dyadic(rng, (H, W, C_in), 6, 3)
        prev = d_state.clone()
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, torch.from_numpy(feat).double(), torch.from_numpy(w2m),
                                                                torch.from_numpy(inl), torch.from_numpy(heights), mw, stride,
                                                                linlayer=(torch.from_numpy(lin_w).double(), torch.from_numpy(lin_b).double()))
        X.check_lattice([state.numpy()], 9, float(X.gemm_bound(feat.reshape(-1, C_in), lin_w).max()) + float(np.abs(lin_b).max()))
        flat = (w2m[..., 1] * mw + w2m[..., 0]).astype(np.int32)
        f_dev = _t(feat if layout == 1 else feat.transpose(2, 0, 1), cuda)[None].contiguous()
        eod.ops.write_max_linear(_t(heights, cuda)[None], _t(flat, cuda)[None], _t((~inl).view(np.uint8), cuda)[None], f_dev, d_hmap, d_key,
                                 d_arg, d_obs, d_state, _t(lin_w, cuda), _t(lin_b, cuda), layout, stride)
        torch.cuda.synchronize()
        assert np.array_equal((d_arg[0] >= 0).cpu().numpy(), m.numpy())
        _same_bits(d_state[0], _exact32(state.numpy()), t)
        assert torch.equal(d_state[0][~m.to(cuda)], prev[0][~m.to(cuda)])


# ------------------------------------------------------------------------------------------------------------------------------
# semmap_update
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,E,cells", [(128, 2, 900), (512, 2, 900), (128, 3, 250_007)], ids=["128", "512", "128-past-sweep"])
def test_semmap_update_exact(eod, cuda, C, E, cells):
    """intensity = mean |sums| / count (custom_rcnn.py:747-748) bit for bit (C is a power of two); cls = the first argmax of the exact
    float64 dot products with the classifier table (inputs built to have a unique maximum); cells not visible this frame untouched.
    The last case has more rows than one sweep of the kernel's capped grid (606 208 on 148 SMs), with 32-row chunks straddling
    episodes (250 007 % 32 != 0)."""
    if cells > 900:
        assert semmap_update_sweeps(E, cells, device_sms()) > 1 and cells % 32
    rng = np.random.default_rng(C)
    K, n_cls = 21, 20
    zs = X.dyadic(rng, (C, K), 4, 4)
    sums = X.dyadic(rng, (E, cells, C), 8, 3)
    for _ in range(20):                                                    # make the maximum unique in every row
        dots = sums.astype(np.float64) @ zs.astype(np.float64)[:, :n_cls]
        top = np.sort(dots, axis=-1)
        tie = top[..., -1] == top[..., -2]
        if not tie.any():
            break
        sums[tie] = X.dyadic(rng, (int(tie.sum()), C), 8, 3)
    assert not tie.any()
    X.check_lattice([dots], 7, float(np.abs(sums[0]).astype(np.float64).max() * np.abs(zs).sum(0).max() * 2))
    counts = rng.integers(0, 5, (E, cells)).astype(np.float32)
    vis = rng.random((E, cells)) < 0.6
    frame_cnt = np.where(vis, rng.integers(1, 9, (E, cells)), 0).astype(np.int32)
    frame_cnt[0, :5] = np.int32(-2 ** 31)                                  # visible without a sample (bit 31 only)
    vis[0, :5] = True
    inten = torch.full((E, cells), -7.0, device=cuda)
    cls = torch.full((E, cells), -3, dtype=torch.int32, device=cuda)
    eod.ops.semmap_update(_t(frame_cnt, cuda), _t(counts, cuda), _t(sums, cuda), _t(zs, cuda), n_cls, inten, cls)
    torch.cuda.synchronize()
    mean_abs = _exact32(np.abs(sums.astype(np.float64)).sum(-1) / C).numpy()
    n = counts + np.float32(1)
    ref_int = np.where(n > 1, mean_abs / n, mean_abs).astype(np.float32)
    ref_int = np.where(vis, ref_int, np.float32(-7.0))
    ref_cls = np.where(vis, dots.argmax(-1), -3).astype(np.int32)
    _same_bits(inten, torch.from_numpy(ref_int), "intensity")
    assert np.array_equal(cls.cpu().numpy(), ref_cls)
