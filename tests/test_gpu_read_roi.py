"""eod_read_roi (the per-proposal memory read) bit for bit against oracle.reference_ops.roi_align_f32, which
tests/test_read_roi_host.py holds bit for bit to torchvision's executed ROIAlign (run on the B200 box with `-m gpu`).

The boxes are the families of test_read_roi_host: on and across every image border, wholly outside within one level pixel of it,
samples exactly on the -1 and h / w limits, zero-size, inverted, NaN, and on the level knife edges.  Every level is random fp16
data, so each tap of each channel shows in the bits of its bin."""
import gc

import numpy as np
import pytest
import torch

from oracle import reference_ops as R

import test_read_roi_host as HB

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _free_device_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


def _need(nbytes):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes} bytes of free device memory, {free} free")


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _random_levels(rng, E, C, dims):
    """(E,h,w,C) fp16 channels-last levels, channels at three magnitudes."""
    return [(rng.standard_normal((E, h, w, C), dtype=np.float32) * rng.choice([1e-2, 1.0, 100.0], C)).astype(np.float16) for h, w in dims]


def _expected(levels, boxes, bidx, n_levels, P, sr, E, rows=None):
    """What eod_read_roi must return for `rows` (default all): levels[l] (E,h,w,C) fp16 numpy -> bins (n,C,P,P) f32, valid (n,P,P) f32,
    level (n) i32.  A box pools from roi_levels' level of its episode, through the restatement; no level or no episode: nothing."""
    rows = np.arange(len(boxes)) if rows is None else np.asarray(rows)
    C = levels[0].shape[3]
    lvl = R.roi_levels(torch.from_numpy(boxes[rows]), n_levels).numpy().astype(np.int32)
    lvl[(bidx[rows] < 0) | (bidx[rows] >= E)] = -1
    out, valid = np.zeros((len(rows), C, P, P), np.float32), np.zeros((len(rows), P, P), np.float32)
    planes = {}
    for i, (r, l) in enumerate(zip(rows, lvl)):
        if l >= 0:
            key = (l, bidx[r])
            if key not in planes:
                planes[key] = np.ascontiguousarray(levels[l][bidx[r]].transpose(2, 0, 1)).astype(np.float32)
            out[i], valid[i] = R.roi_align_f32(planes[key], boxes[r], 1.0 / HB.STRIDES[l], P, sr)
    return out, valid, lvl


def _assert_bits(got, want, what):
    g, w = np.ascontiguousarray(got).view(np.uint32), np.ascontiguousarray(want).view(np.uint32)
    bad = np.nonzero((g != w).reshape(len(g), -1).any(1))[0]
    assert not len(bad), f"{what}: {len(bad)} of {len(g)} rows differ, first {bad[:8].tolist()}"


def _read(eod, levels_dev, bx, bi, P, sr, n_levels):
    out, lvl, valid = eod.ops.read_roi([l.permute(0, 3, 1, 2) for l in levels_dev], bx, bi, P, HB.STRIDES[:n_levels], sampling_ratio=sr,
                                       want_levels=True, want_valid=True)
    torch.cuda.synchronize()
    return out.cpu().numpy(), lvl.cpu().numpy(), valid.cpu().numpy()


@pytest.mark.parametrize("n_levels", [1, 2, 3, 4])
@pytest.mark.parametrize("sr", [0, 2])
@pytest.mark.parametrize("P", [7, 14])
@pytest.mark.parametrize("C", [128, 256, 512])
def test_read_roi_bitwise_vs_restatement(eod, cuda, C, P, sr, n_levels):
    """Every box family, episodes mixed: bins bit for bit, levels exact with -1 for no level, valid = n_valid / count bit for bit and
    ROIAlign of a ones plane within 1e-6 (not bitwise: w1+w2+w3+w4 rounds).  The case takes the empty-sample branch (fractional
    valid) and has boxes without a level."""
    from torchvision.ops import roi_align
    E = 3
    rng = np.random.default_rng(1000 * C + 100 * P + 10 * sr + n_levels)
    dims = HB.level_dims(n_levels)
    levels = _random_levels(rng, E, C, dims)
    boxes, _ = HB.all_boxes(HB.roi_box_families(n_levels, P, seed=P + n_levels))
    bidx = rng.integers(0, E, len(boxes)).astype(np.int32)
    got, got_lvl, got_valid = _read(eod, [_t(l, cuda) for l in levels], _t(boxes, cuda), _t(bidx, cuda), P, sr, n_levels)
    want, want_valid, want_lvl = _expected(levels, boxes, bidx, n_levels, P, sr, E)
    assert np.array_equal(got_lvl, want_lvl)
    assert (want_lvl == -1).any() and set(range(n_levels)) <= set(want_lvl.tolist())
    _assert_bits(got, want, "bins")
    _assert_bits(got_valid, want_valid, "valid")
    assert ((want_valid > 0) & (want_valid < 1)).any() and (want_valid[want_lvl >= 0] == 0).any()
    for l in range(n_levels):
        sel = np.nonzero(want_lvl == l)[0]
        rois = torch.from_numpy(np.concatenate([np.zeros((len(sel), 1), np.float32), boxes[sel]], 1))
        ones = roi_align(torch.ones((1, 1) + dims[l]), rois, (P, P), 1.0 / HB.STRIDES[l], sr, True)[:, 0].numpy()
        assert np.abs(got_valid[sel] - ones).max() <= 1e-6


def test_read_roi_past_2_31_output_elements(eod, cuda):
    """R = 86 016 ROIs x 49 bins x 512 channels > 2^31 output elements (8.6 GB): the ROIs whose rows straddle and follow element 2^31,
    the last ones and a sample of the first ones, bit for bit (bins, valid, level)."""
    E, C, P, R_, n_levels = 64, 512, 7, 86_016, 3
    assert R_ * P * P * C > 2 ** 31
    dims = HB.level_dims(n_levels)
    _need(R_ * P * P * (C + 1) * 4 + E * sum(h * w for h, w in dims) * C * 2 + R_ * 24 + 2 * 1024 ** 3)
    rng = np.random.default_rng(31)
    levels = _random_levels(rng, E, C, dims)
    fam = HB.roi_box_families(n_levels, P, seed=31)
    pool, _ = HB.all_boxes(fam)
    boxes = pool[np.arange(R_) % len(pool)]
    bidx = (np.arange(R_) * 7 % E).astype(np.int32)
    straddle = 2 ** 31 // (P * P * C)                                   # its row holds element 2^31
    near = np.arange(straddle - 2, straddle + 4)
    boxes[near] = fam["partly_outside"][:len(near)]                   # pooled from a level, with empty samples
    rows = np.unique(np.concatenate([np.arange(8), rng.choice(straddle - 2, 24, replace=False), near, np.arange(R_ - 4, R_)]))
    out, lvl, valid = eod.ops.read_roi([_t(l, cuda).permute(0, 3, 1, 2) for l in levels], _t(boxes, cuda), _t(bidx, cuda), P,
                                       HB.STRIDES[:n_levels], want_levels=True, want_valid=True)
    sel = torch.from_numpy(rows).to(cuda)
    got, got_lvl, got_valid = out[sel].cpu().numpy(), lvl[sel].cpu().numpy(), valid[sel].cpu().numpy()
    del out, lvl, valid
    want, want_valid, want_lvl = _expected(levels, boxes, bidx, n_levels, P, 0, E, rows)
    assert (want_lvl[np.isin(rows, near)] >= 0).all()
    assert np.array_equal(got_lvl, want_lvl)
    _assert_bits(got, want, "bins")
    _assert_bits(got_valid, want_valid, "valid")


def test_read_roi_out_of_range_batch_idx(eod, cuda):
    """batch_idx -1 and E pool nothing (zero bins, valid 0, level -1).  The levels are episodes 1..E of an (E+2)-episode buffer whose
    episodes 0 and E+1 hold a sentinel, so a read through a bad index stays inside the allocation and shows in the result."""
    E, C, P, n_levels = 3, 128, 7, 3
    rng = np.random.default_rng(7)
    dims = HB.level_dims(n_levels)
    bufs = _random_levels(rng, E + 2, C, dims)
    for b in bufs:
        b[0], b[E + 1] = 1000.0, -1000.0
    levels = [b[1:E + 1] for b in bufs]
    fam = HB.roi_box_families(n_levels, P, seed=7)
    boxes = np.concatenate([fam["clipped"], fam["partly_outside"], fam["sample_limits"]])
    bidx = np.resize(np.array([-1, 0, E, 1, 2, -1, E], np.int32), len(boxes))
    dev_bufs = [_t(b, cuda) for b in bufs]
    for sr in (0, 2):
        got, got_lvl, got_valid = _read(eod, [b[1:E + 1] for b in dev_bufs], _t(boxes, cuda), _t(bidx, cuda), P, sr, n_levels)
        want, want_valid, want_lvl = _expected(levels, boxes, bidx, n_levels, P, sr, E)
        bad = (bidx < 0) | (bidx >= E)
        assert (want_lvl[bad] == -1).all() and (want_lvl[~bad] >= 0).all()
        assert np.array_equal(got_lvl, want_lvl)
        _assert_bits(got, want, f"bins, sampling_ratio {sr}")
        _assert_bits(got_valid, want_valid, f"valid, sampling_ratio {sr}")


def _fusion_case(eod, cuda, P, fusion_mode, seed):
    rng = np.random.default_rng(seed)
    C, CO, H, W, cells = 256, 128, 192, 256, 600
    fusion = eod.MemoryFusion("implicit_memory", fusion_mode, 5, mem_feat_dim=C, ego_feat_dim=CO).to(cuda)
    with torch.no_grad():
        for conv in fusion.merge_map_projections:
            conv.bias.uniform_(-2.0, 2.0)                              # a bias that a wrong valid share would visibly misplace
    mem16 = [_t((rng.standard_normal((cells, C)) * 2).astype(np.float16), cuda) for _ in range(2)]
    idx = [_t(rng.integers(0, cells, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1).astype(np.int64), cuda) for _ in range(2)]
    fams = [HB.roi_box_families(3, P, seed=seed + i, H=H, W=W) for i in range(2)]
    boxes = [torch.from_numpy(HB.all_boxes(f)[0]) for f in fams]
    return fusion, mem16, idx, boxes, (H, W, CO)


@pytest.mark.parametrize("P", [7, 14])
@pytest.mark.parametrize("fusion_mode", ["sum", "mem_only"])
def test_memory_fusion_roi_read_off_image_boxes(eod, cuda, fusion_mode, P):
    """MemoryFusion.read_roi(project=True) and fuse_roi over boxes across and outside the image border, against executed ROIAlign
    (R.roi_read) over the fused levels res + w (conv(L) + b), within 1e-4 of scale: the projection bias survives the pooling with each
    bin's share of on-level samples.  Boxes without a level have a memory term of exactly zero."""
    fusion, mem16, idx, boxes, (H, W, CO) = _fusion_case(eod, cuda, P, fusion_mode, seed=40 + P)
    with torch.no_grad():
        levels = fusion.read(mem16, idx, [None, None])
        res = [torch.randn((2, CO, H >> s, W >> s)) for s in (3, 4, 5)]
        memterm = [5.0 * torch.nn.functional.conv2d(l.cpu().float(), c.weight.cpu(), c.bias.cpu()) for l, c in zip(levels, fusion.merge_map_projections)]
        want_mem, lvl = R.roi_read(memterm, boxes, P)
        no_level = lvl == -1
        assert no_level.any() and (lvl >= 0).any()
        proj = fusion.read_roi(mem16, idx, boxes, pooled=P, project=True).cpu()
        assert not proj[no_level].any()
        assert (proj - want_mem).abs().max().item() <= 1e-4 * want_mem.abs().max().item()
        box_features, _ = R.roi_read(res, boxes, P)
        box_features[no_level] = torch.randn_like(box_features[no_level])   # whatever the image-only pooler held there
        got = fusion.fuse_roi(box_features.to(cuda), mem16, idx, boxes).cpu()
    if fusion_mode == "sum":
        want, _ = R.roi_read([r + m for r, m in zip(res, memterm)], boxes, P)
        assert torch.equal(got[no_level], box_features[no_level])
    else:
        want = want_mem
        assert not got[no_level].any()
    ok = ~no_level
    assert (got[ok] - want[ok]).abs().max().item() <= 1e-4 * want.abs().max().item()


def test_episode_batch_read_roi_off_image_boxes(eod, cuda):
    """EpisodeBatch.read_roi after batch.read(): the levels of the current frame pooled over every box family, episodes mixed, bit for
    bit against the restatement."""
    E, C, H, W, mw, mh = 3, 256, 192, 256, 30, 20
    rng = np.random.default_rng(9)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    batch.norm16.copy_(_t((rng.standard_normal((E, mw * mh, C)) * 2).astype(np.float16), cuda))
    batch.set_indices(_t(rng.integers(0, mw * mh, (E, H // 4, W // 4)).repeat(4, 1).repeat(4, 2).astype(np.int64), cuda))
    batch.read()
    boxes, _ = HB.all_boxes(HB.roi_box_families(3, 7, seed=9, H=H, W=W))
    bidx = rng.integers(0, E, len(boxes)).astype(np.int32)
    got = batch.read_roi(_t(boxes, cuda), _t(bidx, cuda))
    torch.cuda.synchronize()
    levels = [l.cpu().numpy() for l in batch.levels]
    want, want_valid, want_lvl = _expected(levels, boxes, bidx, 3, 7, 0, E)
    assert (want_lvl == -1).any() and ((want_valid > 0) & (want_valid < 1)).any()
    _assert_bits(got.cpu().numpy(), want, "bins")
