"""The deterministic object-regime write (write_objects[_pasted]_det, EpisodeBatch(object_variant=WRITE_DET), EpisodeRunner): bit for
bit the dense deterministic write of the box_to_image_features image, against the oracle, reproducible and independent of batching."""
import math
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R

import test_gpu_exact as GX
import test_gpu_runner as TR
from test_gpu_det_layouts import _same_bits, _t

pytestmark = pytest.mark.gpu

CHW = 0
SUM_TOL = 1e-5


def _random_frame(eod, rng, E, H, W, C, cells, has, k_range=(4, 16), block=(4, 8)):
    """Per episode with has[e]: make_mask_head_detections (edge cases in every other one) padded with garbage up to Kmax, a blocky
    index plane with noise; n_obj = 0 where has[e] is 0 (its detections and planes are garbage)."""
    dets = [eod.episodes.make_mask_head_detections(rng, H, W, C, k_range, 28, edge_cases=bool(e % 2)) if has[e] else None for e in range(E)]
    Kmax = max([d[0].shape[0] for d in dets if d is not None] + [1]) + 2
    bf = (rng.standard_normal((E, Kmax, C)) * 1e4).astype(np.float32)
    probs = np.ones((E, Kmax, 28, 28), np.float32)
    boxes = np.tile(np.array([0, 0, W, H], np.float32), (E, Kmax, 1))
    n_obj = np.zeros(E, np.int32)
    for e, d in enumerate(dets):
        if d is not None:
            k = d[0].shape[0]
            bf[e, :k], probs[e, :k], boxes[e, :k], n_obj[e] = d[0], d[1], d[2], k
    by, bx = block
    idx = rng.integers(0, cells, (E, H // by + 1, W // bx + 1)).repeat(by, 1).repeat(bx, 2)[:, :H, :W].astype(np.int32)
    idx[:, ::5, ::7] = rng.integers(0, cells, idx[:, ::5, ::7].shape)
    return bf, probs, boxes, n_obj, idx


def _det_write(eod, cuda, pasted, bf, probs, boxes, masks, n_obj, idx, sums, ws, H, W, stride=8):
    """paste / masks_observed -> sample_mask -> frame_count(n_obj) -> write_objects[_pasted]_det into sums: (samp, frame_cnt)."""
    E, cells = sums.shape[:2]
    d_n = _t(n_obj, cuda)
    if pasted:
        _, observed = eod.ops.paste_masks(probs, boxes, (H, W), 0.5, d_n, want_masks=False, want_observed=True)
    else:
        observed = eod.ops.masks_observed(masks, d_n)
    samp = eod.ops.sample_mask(observed, stride)
    cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    eod.ops.frame_count(idx, samp, cnt, d_n)
    if pasted:
        eod.ops.write_objects_pasted_det(bf, probs, boxes, d_n, idx, samp, cnt, sums, ws)
    else:
        eod.ops.write_objects_det(bf, masks, d_n, idx, samp, cnt, sums, ws)
    return samp, cnt


def _dense_reference(eod, cuda, bf, masks, n_obj, idx, samp, cnt, sums, ws, H, W):
    """Per episode: box_to_image_features of its n_obj objects, then write_mean_det(LAYOUT_CHW) with the same samp, frame_cnt, active."""
    for e in range(sums.shape[0]):
        n = int(n_obj[e])
        if not n:
            continue
        img, _ = eod.ops.box_to_image_features(bf[e, :n].contiguous(), masks[e, :n].contiguous())
        eod.ops.write_mean_det(img, idx[e:e + 1], samp[e:e + 1], cnt[e:e + 1].contiguous(), sums[e:e + 1], ws, layout=CHW,
                               active=_t(n_obj[e:e + 1], cuda))


def _oracle_frame(sums, counts, bf, probs, boxes, masks, n, idx, pasted, H, W, stride=8):
    """custom_rcnn.py:876-936 on the CPU for one episode and frame (masks pasted by the oracle in the pasted case)."""
    if not n:
        return sums, counts
    m = torch.from_numpy(oracle.paste_masks(probs[:n], boxes[:n], H, W, 0.5)) if pasted else torch.from_numpy(masks[:n])
    img, obs = R.box_to_image_features(torch.from_numpy(bf[:n]), m)
    return R.write_mean_frame(sums, counts, img, obs, torch.from_numpy(idx).long(), stride=stride)


def _within(got: torch.Tensor, ref: torch.Tensor, what) -> None:
    err = float((got.cpu() - ref).abs().max())
    assert err <= SUM_TOL * max(float(ref.abs().max()), 1e-30), (what, err)


# ------------------------------------------------------------------------------------------------------------------------------
# 1 + 2. the dense deterministic write's bits, and the oracle
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pasted", [False, True], ids=["masks", "pasted"])
@pytest.mark.parametrize("C", [128, 256, 512])
def test_objects_det_is_the_dense_det_write_of_the_image(eod, cuda, C, pasted):
    """Ragged n_obj with an idle slot and garbage beyond n_obj, three accumulating frames; sums identical bits to the dense deterministic
    write of the box_to_image_features image, within 1e-5 of the oracle, counts exact.  C=128 adds a frame of more than 128 objects."""
    rng = np.random.default_rng(3000 + C + pasted)
    E, H, W, cells = 3, 96, 128, 600
    sums = torch.randn((E, cells, C), device=cuda, generator=torch.Generator(device=cuda).manual_seed(C))
    ref = sums.clone()
    counts = torch.zeros((E, cells), device=cuda)
    o_sums, o_counts = [sums[e].cpu() for e in range(E)], [torch.zeros(cells) for _ in range(E)]
    ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda)
    ws_ref = eod.ops.DetWorkspace(1, C, H * W, cells, cuda)
    frames = [([1, 0, 1], (4, 16)), ([1, 1, 0], (4, 16)), ([0, 1, 1], (4, 16))]
    if C == 128:
        frames.append(([1, 1, 0], (130, 140)))
    for t, (has, k_range) in enumerate(frames):
        bf, probs, boxes, n_obj, idx = _random_frame(eod, rng, E, H, W, C, cells, has, k_range)
        d_bf, d_probs, d_boxes, d_idx = _t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(idx, cuda)
        masks, _ = eod.ops.paste_masks(d_probs, d_boxes, (H, W), 0.5, _t(n_obj, cuda))
        samp, cnt = _det_write(eod, cuda, pasted, d_bf, d_probs, d_boxes, masks, n_obj, d_idx, sums, ws, H, W)
        _dense_reference(eod, cuda, d_bf, masks, n_obj, d_idx, samp, cnt, ref, ws_ref, H, W)
        eod.ops.finalize_counts(d_idx, cnt, counts)
        torch.cuda.synchronize()
        assert not ws.overflowed() and not ws_ref.overflowed()
        _same_bits(sums, ref, (t, "sums vs dense det"))
        for e in range(E):
            o_sums[e], o_counts[e] = _oracle_frame(o_sums[e], o_counts[e], bf[e], probs[e], boxes[e], masks[e].cpu().numpy(), int(n_obj[e]),
                                                   idx[e], pasted, H, W)
            _within(sums[e], o_sums[e], (t, e, "sums vs oracle"))
            assert torch.equal(counts[e].cpu(), o_counts[e]), (t, e, "counts")
    assert float(counts.max()) >= 2


@pytest.mark.parametrize("pasted", [False, True], ids=["masks", "pasted"])
def test_objects_det_exact_against_the_oracle(eod, cuda, pasted):
    """tests/exact_cases.py object frames (every partial sum exact in fp32): bit-exact with the oracle, through the ops, three frames
    with ragged n_obj and an empty slot; then more than 128 objects."""
    rng = np.random.default_rng(60 + pasted)
    H, W, C, mw, mh = 96, 128, 128, 50, 40
    cells = mw * mh
    for E, n_base, copies, frames in ((3, 6, (1, 2, 4), ([1, 0, 1], [1, 1, 0], [0, 1, 1])), (1, 36, (4,), ([1],))):
        ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda)
        d_sums = torch.zeros((E, cells, C), device=cuda)
        d_counts = torch.zeros((E, cells), device=cuda)
        sums = [torch.zeros(cells, C) for _ in range(E)]
        counts = [torch.zeros(cells) for _ in range(E)]
        for has in frames:
            bf, probs, boxes, masks, n_obj, idx = GX._object_frame(rng, E, H, W, C, cells, has, n_base, copies)
            n_eff = np.where(np.array(has) > 0, n_obj, 0).astype(np.int32)
            if E == 1:
                assert n_obj[0] > 128
            d_idx = _t(idx, cuda)
            _, cnt = _det_write(eod, cuda, pasted, _t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(masks, cuda), n_eff, d_idx, d_sums, ws, H, W)
            eod.ops.finalize_counts(d_idx, cnt, d_counts)
            torch.cuda.synchronize()
            assert not ws.overflowed()
            for e in range(E):
                sums[e], counts[e] = GX._object_oracle(sums[e], counts[e], bf[e], masks[e], idx[e], int(n_eff[e]))
                _same_bits(d_sums[e], sums[e], (E, e, "sums"))
                assert torch.equal(d_counts[e].cpu(), counts[e]), (E, e, "counts")


# ------------------------------------------------------------------------------------------------------------------------------
# 3. reproducible, independent of batching; long segments (chunked reduce, bitmap sort)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pasted", [False, True], ids=["masks", "pasted"])
def test_objects_det_reproducible_and_batch_independent(eod, cuda, pasted):
    """480x640, sample_stride 1, E=4: slot 0 is one whole-image object over a single cell (9600 runs: bitmap sort), slot 1 has a cell
    of 400 runs (chunked reduce), slots 2-3 random detections.  Two runs, each slot alone and a permuted slot order: the same bits."""
    rng = np.random.default_rng(77 + pasted)
    E, H, W, C, cells = 4, 480, 640, 128, 3000
    bf, probs, boxes, n_obj, idx = _random_frame(eod, rng, E, H, W, C, cells, [1, 1, 1, 1], (4, 16), block=(8, 16))
    n_obj[0] = 1
    probs[0, 0], boxes[0, 0] = 1.0, (0.0, 0.0, float(W), float(H))            # pastes to the whole image
    idx[0] = 5
    idx[1, :20] = 7                                                          # 400 tiles of one cell: 400 runs
    sums0 = torch.randn((E, cells, C), device=cuda, generator=torch.Generator(device=cuda).manual_seed(9))
    d = dict(bf=_t(bf, cuda), probs=_t(probs, cuda), boxes=_t(boxes, cuda), idx=_t(idx, cuda))
    masks, _ = eod.ops.paste_masks(d["probs"], d["boxes"], (H, W), 0.5, _t(n_obj, cuda))

    def run(order):
        o = torch.as_tensor(order, device=cuda)
        sums = sums0[o].contiguous()
        ws = eod.ops.DetWorkspace(len(order), C, H * W, cells, cuda, H * W)
        _det_write(eod, cuda, pasted, d["bf"][o].contiguous(), d["probs"][o].contiguous(), d["boxes"][o].contiguous(), masks[o].contiguous(),
                   n_obj[np.array(order)], d["idx"][o].contiguous(), sums, ws, H, W, stride=1)
        torch.cuda.synchronize()
        assert not ws.overflowed()
        return sums

    a, b = run([0, 1, 2, 3]), run([0, 1, 2, 3])
    _same_bits(a, b, "two runs")
    for e in range(E):
        _same_bits(run([e])[0], a[e], ("alone", e))
    p = [2, 0, 3, 1]
    perm = run(p)
    for i, e in enumerate(p):
        _same_bits(perm[i], a[e], ("permuted", e))
    # slot 0: every pixel is sampled and holds bf[0, 0], so cell 5 gains exactly that row (float64 reference: an fp32 oracle summing the
    # 307 200 pixels one after the other drifts by ~1e-3 of scale itself); every other cell is untouched
    ref = sums0[0].cpu().double()
    ref[5] += torch.from_numpy(bf[0, 0]).double()
    _within(a[0].double(), ref, "whole-image object")
    keep = torch.arange(cells, device=cuda) != 5
    _same_bits(a[0][keep], sums0[0][keep], "untouched cells")


# ------------------------------------------------------------------------------------------------------------------------------
# 4. overflow: a workspace too small falls back to reductions, still correct
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pasted", [False, True], ids=["masks", "pasted"])
def test_objects_det_overflow_stays_correct(eod, cuda, pasted):
    rng = np.random.default_rng(88 + pasted)
    E, H, W, C, cells = 2, 96, 128, 256, 600
    bf, probs, boxes, n_obj, idx = _random_frame(eod, rng, E, H, W, C, cells, [1, 1], (4, 16))
    d_probs, d_boxes = _t(probs, cuda), _t(boxes, cuda)
    masks, _ = eod.ops.paste_masks(d_probs, d_boxes, (H, W), 0.5, _t(n_obj, cuda))
    sums = torch.zeros((E, cells, C), device=cuda)
    ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda, 16)
    _det_write(eod, cuda, pasted, _t(bf, cuda), d_probs, d_boxes, masks, n_obj, _t(idx, cuda), sums, ws, H, W)
    torch.cuda.synchronize()
    assert ws.overflowed()
    for e in range(E):
        ref, _ = _oracle_frame(torch.zeros(cells, C), torch.zeros(cells), bf[e], probs[e], boxes[e], masks[e].cpu().numpy(), int(n_obj[e]),
                               idx[e], pasted, H, W)
        _within(sums[e], ref, e)


# ------------------------------------------------------------------------------------------------------------------------------
# 5 + 6. EpisodeBatch(object_variant=WRITE_DET): the frame loop and its graph
# ------------------------------------------------------------------------------------------------------------------------------
def _batch(eod, cuda, E, C, H, W, mw, mh, pipeline):
    b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, pipeline=pipeline, object_variant=eod._lib.WRITE_DET)
    return b


@pytest.mark.parametrize("pipeline", [False, True], ids=["ordered", "pipelined"])
def test_episode_batch_objects_det_matches_a_serial_twin(eod, cuda, pipeline):
    """step_detections with reset_mask / refresh_mask, idle slots (n_obj = 0) and late inputs: levels of every frame, sums, counts and
    norm16 bit for bit those of a serial pipeline=False twin; write_detections and write_objects (pasted masks) agree bit for bit."""
    E, C, H, W, mw, mh = 3, 128, 96, 128, 60, 45
    cells = mw * mh
    rng = np.random.default_rng(500 + pipeline)
    a, b = _batch(eod, cuda, E, C, H, W, mw, mh, pipeline), _batch(eod, cuda, E, C, H, W, mw, mh, False)
    a.read_frozen = b.read_frozen = pipeline
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    z = lambda *s: torch.zeros(s, device=cuda)
    plan = [dict(), dict(has=[1, 0, 1]), dict(reset=[0, 1, 0], late=True), dict(refresh=[1, 0, 1]), dict(has=[0, 1, 1], reset=[1, 0, 0], refresh=[1, 1, 0])]
    for t, p in enumerate(plan):
        bf, probs, boxes, n_obj, idx = _random_frame(eod, rng, E, H, W, C, cells, p.get("has", [1, 1, 1]), (2, 8))
        args = (z(E, H, W), z(E, 12), z(E, 6), intr, 0.2, _t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(n_obj, cuda))
        kw = dict(proj_indices=_t(idx, cuda))
        for key in ("reset", "refresh"):
            if key in p:
                kw[key + "_mask"] = _t(np.array(p[key], np.int32), cuda)
        la = [l.clone() for l in a.step_detections(*args, inputs_ready=not p.get("late"), **kw)]
        lb = [l.clone() for l in b.step_detections(*args, **kw)]
        for k in range(3):
            _same_bits(la[k], lb[k], (t, "level", k))
    a.join(), b.join()
    torch.cuda.synchronize()
    assert a._slots is None and not a._det_ws.overflowed()
    _same_bits(a.sums, b.sums, "sums")
    _same_bits(a.counts, b.counts, "counts")
    _same_bits(a.norm16, b.norm16, "norm16")
    assert float(a.counts.max()) >= 3
    # write_detections == write_objects with the pasted masks
    bf, probs, boxes, n_obj, idx = _random_frame(eod, rng, E, H, W, C, cells, [1, 0, 1], (2, 8))
    d_n = _t(n_obj, cuda)
    for x in (a, b):
        x.set_indices(_t(idx, cuda))
    a.write_detections(_t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), d_n)
    masks, _ = eod.ops.paste_masks(_t(probs, cuda), _t(boxes, cuda), (H, W), 0.5, d_n)
    b.write_objects(_t(bf, cuda), masks, d_n)
    torch.cuda.synchronize()
    _same_bits(a.sums, b.sums, "write_detections vs write_objects")
    _same_bits(a.norm16, b.norm16, "norm16 after write_*")


def test_capture_step_detections_objects_det(eod, cuda):
    """A graph of step_detections(object_variant=WRITE_DET): replays equal an eager twin bit for bit, with an eager frame in between."""
    E, C, H, W, mw, mh = 2, 128, 96, 128, 60, 45
    cells = mw * mh
    rng = np.random.default_rng(41)
    a, b = _batch(eod, cuda, E, C, H, W, mw, mh, True), _batch(eod, cuda, E, C, H, W, mw, mh, False)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    ep = eod.episodes.make_episode(7, 4, H, W, mw, mh, 0.2)
    T = eod.transform3d(torch.from_numpy(ep.xyzhe))
    shifts = _t(np.tile(np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]), (E, 1)), cuda)
    Kmax = 8

    def frame(i):
        dets = [eod.episodes.make_mask_head_detections(rng, H, W, C, (2, 6), 28) for _ in range(E)]
        bf, probs, boxes = np.zeros((E, Kmax, C), np.float32), np.zeros((E, Kmax, 28, 28), np.float32), np.zeros((E, Kmax, 4), np.float32)
        n = np.zeros(E, np.int32)
        for e, d in enumerate(dets):
            k = d[0].shape[0]
            bf[e, :k], probs[e, :k], boxes[e, :k], n[e] = d[0], d[1], d[2], k
        depth = _t(np.stack([ep.depth[i % 4]] * E), cuda)
        pose = _t(np.stack([T[i % 4, :3].reshape(12).numpy()] * E), cuda)
        return depth, pose, shifts, _t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(n, cuda)

    f0 = frame(0)
    g = a.capture_step_detections(f0[0], f0[1], f0[2], intr, 0.2, *f0[3:])
    for i in range(4):
        f = frame(i)
        if i == 2:
            la = [l.clone() for l in a.step_detections(f[0], f[1], f[2], intr, 0.2, *f[3:])]
        else:
            la = [l.clone() for l in g(*f)]
        lb = [l.clone() for l in b.step_detections(f[0], f[1], f[2], intr, 0.2, *f[3:])]
        for k in range(3):
            _same_bits(la[k], lb[k], (i, "level", k))
    a.join(), b.join()
    torch.cuda.synchronize()
    _same_bits(a.sums, b.sums, "sums")
    _same_bits(a.counts, b.counts, "counts")
    _same_bits(a.norm16, b.norm16, "norm16")
    assert float(a.counts.max()) >= 2 and not a._det_ws.overflowed()


# ------------------------------------------------------------------------------------------------------------------------------
# 7. EpisodeRunner(variant=WRITE_DET, object_variant=WRITE_DET)
# ------------------------------------------------------------------------------------------------------------------------------
def _run(eod, cuda, episodes, shifts, intr, test_type, n_slots, save_dir):
    provider = eod.HostEpisodeProvider(episodes, cuda, shifts, k_max=8)
    runner = eod.EpisodeRunner(provider, TR.MW, TR.MH, TR.C, n_slots=n_slots, height=TR.H, width=TR.W, device=cuda, test_type=test_type,
                               intr=intr, cell=TR.CELL, variant=eod._lib.WRITE_DET, object_variant=eod._lib.WRITE_DET, save_dir=save_dir)
    got = {}

    def on_levels(step, levels):
        for s, a in enumerate(step.assign):
            if a is not None:
                got[a] = [lv[s].clone() for lv in levels]

    stats = runner.run(on_levels)
    torch.cuda.synchronize()
    assert stats["det_overflowed"] is False
    saved = {}
    for f in os.listdir(os.path.join(save_dir, "memory")):
        _, mem, obs = eod.formats.load_memory(os.path.join(save_dir, "memory", f))
        saved[os.path.splitext(f)[0]] = (mem, obs)
    return got, saved, stats


def _solo(eod, cuda, episodes, shifts, intr, test_type):
    """Every episode replayed one frame at a time through EpisodeBatch(E=1, object_variant=WRITE_DET), in dataset order."""
    batch = eod.EpisodeBatch(1, TR.MW, TR.MH, TR.C, TR.H, TR.W, cuda, variant=eod._lib.WRITE_DET, object_variant=eod._lib.WRITE_DET)
    batch.read_frozen = test_type == "longterm"
    one = torch.ones((1,), dtype=torch.int32, device=cuda)
    levels, saved = {}, {}
    Kmax = 8
    for e, ep in enumerate(episodes):
        for i, fr in enumerate(ep):
            kw = {}
            if fr["memory_reset"] or (e == 0 and i == 0):
                kw["reset_mask"] = one
            if batch.read_frozen and (i == 0 or "reset_mask" in kw):
                kw["refresh_mask"] = one
            K = fr["box_features"].shape[0]
            bf, probs, boxes = np.zeros((1, Kmax, TR.C), np.float32), np.zeros((1, Kmax, 28, 28), np.float32), np.zeros((1, Kmax, 4), np.float32)
            bf[0, :K], probs[0, :K], boxes[0, :K] = fr["box_features"], fr["mask_probs"], fr["boxes"]
            lv = batch.step_detections(_t(fr["depth"], cuda)[None], _t(fr["pose"], cuda)[None], _t(shifts[e], cuda)[None], intr, TR.CELL,
                                       _t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(np.array([K], np.int32), cuda), **kw)
            levels[(e, i)] = [l[0].clone() for l in lv]
            if i == 0:
                batch.join()
                saved[os.path.splitext(fr["sequence_name"])[0]] = (batch.sums[0].cpu().numpy(), batch.counts[0].cpu().numpy())
    batch.join()
    torch.cuda.synchronize()
    assert not batch._det_ws.overflowed()
    return levels, saved


@pytest.mark.parametrize("test_type", ["default", "longterm"])
def test_runner_objects_det_is_reproducible_across_slots_and_waves(eod, cuda, tmp_path, test_type):
    episodes, shifts, intr = TR._dataset(eod, test_type, "detections")
    runs = [_run(eod, cuda, episodes, shifts, intr, test_type, n, str(tmp_path / f"run{k}")) for k, n in enumerate((2, 2, 3))]
    solo_levels, solo_saved = _solo(eod, cuda, episodes, shifts, intr, test_type)
    n_frames = sum(len(ep) for ep in episodes)
    got0, saved0, stats0 = runs[0]
    assert stats0["frames"] == n_frames and len(got0) == n_frames and stats0["steps"] < n_frames
    for got, saved, _ in runs[1:] + [(solo_levels, solo_saved, None)]:
        assert set(got) == set(got0) and set(saved) == set(saved0)
        for key in got0:
            for k in range(3):
                _same_bits(got[key][k], got0[key][k], (key, k))
        for name in saved0:
            assert np.array_equal(saved[name][0].view(np.int32), saved0[name][0].view(np.int32)), name
            assert np.array_equal(saved[name][1], saved0[name][1]), name
    ref_levels, ref_saved = TR._oracle_serial(episodes, test_type, "detections")
    for key, lv in got0.items():
        for k in range(3):
            a, b = lv[k].float().cpu(), ref_levels[key][k][0].float()
            tol = 2e-3 * max(1.0, float(b.abs().max()))
            assert torch.allclose(a, b, rtol=2e-3, atol=tol), (key, k, float((a - b).abs().max()))
    for name, (s_ref, c_ref) in ref_saved.items():
        mem, obs = saved0[os.path.splitext(name)[0]]
        assert np.array_equal(obs, c_ref.numpy()), name
        assert np.abs(mem - s_ref.numpy()).max() <= SUM_TOL * max(float(s_ref.abs().max()), 1e-30), name
