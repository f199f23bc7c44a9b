"""The per-ROI read's CPU oracle (no GPU): oracle.reference_ops.roi_align_f32 restates eod_read_roi's arithmetic in fp32, one rounding
per operation in the kernel's order.  Here it is held bit for bit to torchvision's executed CPU ROIAlign over boxes on and off the
image, and roi_levels - the level ROIPooler pools each box from, -1 for none - to detectron2's assign_boxes_to_levels.
tests/test_gpu_read_roi.py holds the kernel to the same restatement, over the box families defined here."""
import numpy as np
import pytest
import torch

from oracle import reference_ops as R

STRIDES = (8, 16, 32, 64)
H, W = 384, 512                                    # levels 48x64, 24x32, 12x16, 6x8


def level_dims(n_levels, H=H, W=W):
    return [(H // s, W // s) for s in STRIDES[:n_levels]]


def _side_for_level(l, n_bins_side):
    """Length of the other side of a box whose one side is n_bins_side image pixels, so that sqrt(area) = 224 * 2^(l - 1/2): the
    middle of level l's size range (level 0 takes everything below 224, the top level everything above)."""
    return (224.0 * 2.0 ** (l - 0.5)) ** 2 / n_bins_side


def level_edge_sides():
    """Square sides a (image pixels) on detectron2's level knife edges: sqrt(a * a) = 112, 224, 448, 896 and one fp32 ulp on either
    side, and the two neighbouring fp32 sides between which assign_boxes_to_levels really changes level (just below each edge:
    4 + log2(s / 224) rounds up to the integer for s an ulp or two short of it)."""
    sides = []
    for edge in (112.0, 224.0, 448.0, 896.0):
        e = np.float32(edge)
        sides += [np.nextafter(e, np.float32(0)), e, np.nextafter(e, np.float32(np.inf))]
        bits = np.arange(e.view(np.int32) - 64, e.view(np.int32) + 1, dtype=np.int32).view(np.float32)
        z = torch.zeros(len(bits))
        lv = R.assign_boxes_to_levels(torch.stack([z, z, torch.from_numpy(bits), torch.from_numpy(bits)], 1), 2, 6)
        flip = int(np.nonzero(np.diff(lv.numpy()))[0][0])
        sides += [bits[flip], bits[flip + 1]]
    return np.asarray(sides, np.float32)


def roi_box_families(n_levels, P, seed, H=H, W=W):
    """name -> (n,4) f32 XYXY boxes in image pixels for an H x W image with levels at STRIDES[:n_levels]: every family within a few
    image sizes of the frame (a box with an inf corner would take ~2^31 samples per bin, in torchvision and in the kernel alike)."""
    rng = np.random.default_rng(seed)
    dims = level_dims(n_levels, H, W)
    fam = {}
    # proposals clipped to the image, as _create_proposals_from_boxes leaves them
    n = 10
    cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
    s = np.exp(rng.uniform(np.log(8), np.log(2 * max(H, W)), n))
    ar = np.exp(rng.uniform(-1, 1, n))
    b = np.stack([cx - s * np.sqrt(ar) / 2, cy - s / np.sqrt(ar) / 2, cx + s * np.sqrt(ar) / 2, cy + s / np.sqrt(ar) / 2], 1)
    fam["clipped"] = np.stack([b[:, 0].clip(0, W), b[:, 1].clip(0, H), b[:, 2].clip(0, W), b[:, 3].clip(0, H)], 1)
    # partly outside: across each side and each corner, by 10 - 60 % of the box
    out = []
    for dx, dy in ((-1, 0), (1, 0), (0, -1), (0, 1), (-1, -1), (1, -1), (-1, 1), (1, 1)):
        bw, bh = np.exp(rng.uniform(np.log(24), np.log(1.5 * max(H, W)), 2))
        fx, fy = rng.uniform(0.1, 0.6, 2)
        x0 = {-1: -fx * bw, 0: rng.uniform(0, W - bw) if bw < W else -(bw - W) / 2, 1: W - (1 - fx) * bw}[dx]
        y0 = {-1: -fy * bh, 0: rng.uniform(0, H - bh) if bh < H else -(bh - H) / 2, 1: H - (1 - fy) * bh}[dy]
        out.append([x0, y0, x0 + bw, y0 + bh])
    fam["partly_outside"] = np.asarray(out)
    # wholly outside: starting within one level pixel of an edge, on each side for each level (sized to be pooled from that level),
    # and one far away (its samples are all empty)
    out = []
    for l, s in enumerate(STRIDES[:n_levels]):
        a, q = 224.0 * 2.0 ** (l - 0.5), np.exp(rng.uniform(np.log(0.5), np.log(2.0)))
        thick, long_ = a * q, a / q
        gap, y0 = rng.uniform(0, s), rng.uniform(0, H) - long_ / 2
        out += [[W + gap, y0, W + gap + thick, y0 + long_], [-gap - thick, y0, -gap, y0 + long_]]
        x0 = rng.uniform(0, W) - long_ / 2
        out += [[x0, H + gap, x0 + long_, H + gap + thick], [x0, -gap - thick, x0 + long_, -gap]]
    out.append([W + 200, H + 150, W + 300, H + 260])
    fam["outside_near"] = np.asarray(out)
    # sample points exactly on the limits -1 and h / w: one side 2 P level pixels long, so that bins are 2 pixels and the samples sit at
    # rs + 2 ph + iy + 0.5 for sampling_ratio 0 and 2 alike; the first sample row on -1, or the last on h (w)
    out = []
    for l, (s, (h, w)) in enumerate(zip(STRIDES, dims)):
        side, other = 2 * P * s, _side_for_level(l, 2 * P * s)
        ox, oy = (W - other) / 2, (H - other) / 2
        out += [[ox, -s, ox + other, -s + side], [ox, (h - 2 * P + 1) * s, ox + other, (h - 2 * P + 1) * s + side],
                [-s, oy, -s + side, oy + other], [(w - 2 * P + 1) * s, oy, (w - 2 * P + 1) * s + side, oy + other]]
    fam["sample_limits"] = np.asarray(out)
    # zero width / height / both: inside, on the edge, at the level-0 coordinates whose samples land exactly on -1 and h / w, and a
    # zero-width box inverted in height (area -0: level 0)
    h0, w0 = dims[0]
    s0 = STRIDES[0]
    out = [[100, 50, 100, 150], [40, 90, 300, 90], [200, 200, 200, 200], [0, 0, 0, H], [W, 0, W, H], [10, H, 200, H],
           [-s0 / 2, 20, -s0 / 2, 300], [(w0 + 0.5) * s0, 20, (w0 + 0.5) * s0, 300], [30, -s0 / 2, 250, -s0 / 2],
           [30, (h0 + 0.5) * s0, 250, (h0 + 0.5) * s0], [-s0 / 2, -s0 / 2, -s0 / 2, -s0 / 2], [100, 100, 100, 50]]
    fam["zero_size"] = np.asarray(out)
    # inverted in both axes: positive area, so a level; the samples walk backwards from the first corner
    fam["inverted_both"] = np.asarray([[200, 180, 60, 40], [W + 20, H - 10, W - 300, -40], [90, 260, 10, 20], [W, H, 0, 0]])
    # inverted in exactly one axis: negative area, so no level
    fam["inverted_one"] = np.asarray([[10, 10, 5, 40], [300, 20, 60, 200], [40, 300, 200, 100], [-50, 100, -80, 400]])
    nan = np.nan
    fam["nan"] = np.asarray([[nan, 10, 50, 60], [10, nan, 50, 60], [10, 10, nan, 60], [10, 10, 50, nan], [nan, nan, 50, 60],
                             [nan, nan, nan, nan]])
    # level knife edges, at the origin and half off the image
    a = level_edge_sides()
    fam["level_edges"] = np.concatenate([np.stack([0 * a, 0 * a, a, a], 1), np.stack([W - a / 2, H - a / 2, W + a / 2, H + a / 2], 1)])
    return {k: np.asarray(v, np.float32) for k, v in fam.items()}


NO_LEVEL = ("inverted_one", "nan")


def all_boxes(fam):
    names = sorted(fam)
    return np.concatenate([fam[k] for k in names]), np.concatenate([np.full(len(fam[k]), k) for k in names])


def _levels(n_levels, C, seed):
    rng = np.random.default_rng(seed)
    return [(rng.standard_normal((C, h, w)) * rng.choice([1e-2, 1.0, 100.0], (C, 1, 1))).astype(np.float16).astype(np.float32)
            for h, w in level_dims(n_levels)]


def test_box_families_reach_every_branch():
    """The families do what their names say: sample_limits boxes are pooled from the level they were sized for and put a sample
    exactly on -1 and on h / w; no-level families have none and every other box has one."""
    for n_levels in (1, 2, 3, 4):
        for P in (7, 14):
            fam = roi_box_families(n_levels, P, seed=n_levels)
            for k, b in fam.items():
                lv = R.roi_levels(torch.from_numpy(b), n_levels).numpy()
                assert ((lv == -1) if k in NO_LEVEL else (lv >= 0)).all(), (k, lv)
            lv = R.roi_levels(torch.from_numpy(fam["sample_limits"]), n_levels).numpy()
            assert lv.tolist() == [l for l in range(n_levels) for _ in range(4)]
            for (s, (h, w)), b in zip(zip(STRIDES, level_dims(n_levels)), fam["sample_limits"].reshape(-1, 4, 4)):
                first = b[:, :2] / np.float32(s) - np.float32(0.5) + np.float32(0.5)          # the first sample of bin 0 (bins are 2 px)
                last = b[:, 2:] / np.float32(s) - np.float32(0.5) - np.float32(0.5)
                assert first[0, 1] == -1 and last[1, 1] == h and first[2, 0] == -1 and last[3, 0] == w


@pytest.mark.parametrize("P,sr", [(7, 0), (7, 2), (14, 0), (14, 2)])
def test_roi_align_restatement_matches_torchvision_bitwise(P, sr):
    """roi_align_f32 against torchvision.ops.roi_align (executed, CPU, aligned=True) on every box that has a level, at that level: bins
    equal bit for bit, and valid equals ROIAlign of a constant-1 plane within 1e-6.  The boxes reach the empty-sample branch and
    fractional valid shares.  Boxes without a level never reach ROIAlign (ROIPooler skips them; eod_read_roi pools nothing for them);
    torchvision's CPU kernel is not defined for them either (a NaN size becomes INT_MIN samples)."""
    from torchvision.ops import roi_align
    n_levels, C = 4, 16
    levels = _levels(n_levels, C, seed=P + sr)
    boxes, names = all_boxes(roi_box_families(n_levels, P, seed=10 * P + sr))
    lvl = R.roi_levels(torch.from_numpy(boxes), n_levels).numpy()
    got, got_valid, want, want_valid = [], [], [], []
    for b, l in zip(boxes, lvl):
        if l < 0:
            continue
        out, valid = R.roi_align_f32(levels[l], b, 1.0 / STRIDES[l], P, sr)
        got.append(out)
        got_valid.append(valid)
        roi = torch.from_numpy(np.concatenate([[0], b]).astype(np.float32))[None]
        want.append(roi_align(torch.from_numpy(levels[l])[None], roi, (P, P), 1.0 / STRIDES[l], sr, True)[0].numpy())
        want_valid.append(roi_align(torch.ones((1, 1) + levels[l].shape[1:]), roi, (P, P), 1.0 / STRIDES[l], sr, True)[0, 0].numpy())
    got, want, got_valid, want_valid = map(np.stack, (got, want, got_valid, want_valid))
    assert ((got_valid > 0) & (got_valid < 1)).any() and (got_valid == 0).any() and (got_valid == 1).any()
    assert np.abs(got_valid - want_valid).max() <= 1e-6
    diff = got.view(np.uint32) != want.view(np.uint32)
    if diff.any():
        ulps = np.abs(got.view(np.int32).astype(np.int64) - want.view(np.int32).astype(np.int64))[diff]
        if ulps.max() <= 2:
            pytest.skip(f"this torchvision build rounds ROIAlign differently ({int(diff.sum())} values off by <= {int(ulps.max())} ulp, "
                        "e.g. multiply-adds contracted to fma); the restatement follows the uncontracted order of the kernel")
        bad = np.nonzero(diff.reshape(len(got), -1).any(1))[0]
        raise AssertionError(f"restatement != torchvision for {len(bad)} boxes, up to {int(ulps.max())} ulp: {bad[:8].tolist()}")


@pytest.mark.parametrize("n_levels", [1, 2, 3, 4])
def test_no_level_rule_matches_assign_boxes_to_levels(n_levels):
    """roi_levels == assign_boxes_to_levels where that lies in [0, n_levels), -1 elsewhere; -1 exactly for the boxes inverted in one
    axis and the boxes with a NaN coordinate, whose detectron2 level is an out-of-range integer; ROIPooler (roi_read) pools zeros for
    them.  Zero-area boxes, -0 area included, are level 0."""
    boxes, names = all_boxes(roi_box_families(n_levels, 7, seed=3))
    bt = torch.from_numpy(boxes)
    ref = R.assign_boxes_to_levels(bt, 3, 3 + n_levels - 1)
    lv = R.roi_levels(bt, n_levels)
    inside = (ref >= 0) & (ref < n_levels)
    assert torch.equal(lv[inside], ref[inside]) and (lv[~inside] == -1).all()
    no_level = np.isin(names, NO_LEVEL)
    assert np.array_equal(~inside.numpy(), no_level)
    area = (bt[:, 2] - bt[:, 0]) * (bt[:, 3] - bt[:, 1])
    assert (lv[area == 0] == 0).all() and bool((area == 0).any()) and bool(torch.signbit(area[area == 0]).any())
    levels = [torch.from_numpy(x)[None] for x in _levels(n_levels, 4, seed=1)]
    pooled, lvl = R.roi_read(levels, [bt], 7, STRIDES[:n_levels])
    assert torch.equal(lvl, lv)
    assert not pooled[torch.from_numpy(no_level)].any() and pooled[torch.from_numpy(~no_level)].any()
