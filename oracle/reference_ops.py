"""ORACLE (test infrastructure, NOT product code).

Device-neutral torch-CPU restatement of the reference's spatial-feature-memory path.  Every function
cites the reference lines it follows (paths relative to /root/reference/Detic).  The reference hard-codes
``.cuda()`` / ``torch.cuda.FloatTensor`` and imports detectron2, so it cannot be imported as-is; the only
semantic change here is "allocate on the CPU".  Pinning: tests/golden/make_golden.py executes the
reference's *own* source lines (imported projector package; exec of the cited line ranges of
custom_rcnn.py / timm.py with CPU-patched constructors) and the resulting fixtures are compared against
these functions in tests/test_oracle_golden.py.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

# --------------------------------------------------------------------------------------------------
# Geometry (A1-A5)
# --------------------------------------------------------------------------------------------------


def transform3d(xyzhe: torch.Tensor) -> torch.Tensor:
    """(N,5) x,y,z,heading,elevation -> (N,4,4) camera-to-world.  SMNet/projector/core.py:6-34."""
    elev, head = xyzhe[:, 4], xyzhe[:, 3]
    cx, sx = torch.cos(elev), torch.sin(elev)
    cy, sy = torch.cos(head), torch.sin(head)
    T = torch.zeros(xyzhe.shape[0], 4, 4)
    T[:, 0, 0], T[:, 0, 1], T[:, 0, 2], T[:, 0, 3] = cy, sx * sy, cx * sy, xyzhe[:, 0]
    T[:, 1, 1], T[:, 1, 2], T[:, 1, 3] = cx, -sx, xyzhe[:, 1]
    T[:, 2, 0], T[:, 2, 1], T[:, 2, 2], T[:, 2, 3] = -sy, cy * sx, cy * cx, xyzhe[:, 2]
    T[:, 3, 3] = 1
    return T


def intrinsics(width: int, height: int, vfov: float) -> Tuple[float, float, float, float]:
    """fx, fy, cx, cy as the fp32 values the reference holds.  core.py:68-77 (Python-double math, then
    one rounding to fp32 inside torch.Tensor([...]))."""
    hfov = width / height * vfov
    fx = width / (2.0 * math.tan(hfov / 2.0))
    fy = height / (2.0 * math.tan(vfov / 2.0))
    K = torch.Tensor([fx, fy, width / 2.0, height / 2.0])
    return tuple(float(v) for v in K)


def pixel_to_world(depth: torch.Tensor, T: torch.Tensor, vfov: float,
                   world_shift_origin: torch.Tensor) -> torch.Tensor:
    """depth (B,H,W) f32, T (B,4,4) -> world xyz (B,H,W,3).  core.py:80-149,177-225."""
    B, H, W = depth.shape
    fx, fy, cx, cy = (torch.tensor(v, dtype=torch.float32) for v in intrinsics(W, H, vfov))
    u = torch.arange(W).float().view(1, 1, W).expand(B, H, W)
    v = torch.arange(H).float().view(1, H, 1).expand(B, H, W)
    x_scale = (u + 0.5 - cx) / fx            # core.py:107
    y_scale = (v + 0.5 - cy) / fy            # core.py:108
    z = depth / float(1.0)                   # core.py:142
    x = z * x_scale
    y = z * y_scale
    xyz1 = torch.stack((x, y, z, torch.ones_like(z)), dim=3).reshape(B, H * W, 4)   # core.py:148
    world = torch.bmm(T, xyz1.transpose(1, 2)).transpose(1, 2)[:, :, :3]            # core.py:175,214
    world = world - world_shift_origin                                             # core.py:220
    return world.reshape(B, H, W, 3)


def discretize(point_cloud: torch.Tensor, camera_height: torch.Tensor, cell: float, out_w: int, out_h: int,
               z_clip: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """core.py:227-271 -> (pixels_in_map int64 (B,H,W,2) unclipped, mask_outliers bool)."""
    q = (point_cloud[:, :, :, [0, 2]] / cell).round()
    outside = (q[..., 0] >= out_w) + (q[..., 1] >= out_h) + (q[..., 0] < 0) + (q[..., 1] < 0)
    cam_y = camera_height.view(-1, 1, 1).expand(-1, q.shape[1], q.shape[2])
    above = point_cloud[..., 1] > (cam_y + z_clip)
    return q.long(), outside + above


def projector_forward(depth: torch.Tensor, T: torch.Tensor, vfov: float, out_h: int, out_w: int, cell: float,
                      world_shift_origin: torch.Tensor, z_clip: float):
    """projector.py:66-106 with return_heights=True.  depth (B,1,H,W)."""
    d = depth[:, 0]
    no_depth = d == 0
    pc = pixel_to_world(d, T, vfov, world_shift_origin)
    idx2d, outliers = discretize(pc, T[:, 1, 3], cell, out_w, out_h, z_clip)
    return idx2d, no_depth + outliers, pc[..., 1]


def quantize_flat_index(world_xyz: torch.Tensor, map_world_shift: torch.Tensor, cell: float, map_w: int,
                        map_h: int, order: str = "zx") -> torch.Tensor:
    """World xyz (T,H,W,3) f32 -> flat clipped cell index int32 (T,H,W,1).
    SMNet/build_memory_data.py:135-144 (order 'zx': z*map_w+x); robot_demo.py:526-533 (order 'xz':
    x*map_h+z)."""
    p = world_xyz - map_world_shift
    q = (p[:, :, :, [0, 2]] / cell).round().long()
    qx = q[..., 0].clamp(0, map_w - 1)
    qz = q[..., 1].clamp(0, map_h - 1)
    flat = qz * map_w + qx if order == "zx" else qx * map_h + qz
    return flat.to(torch.int32).unsqueeze(-1)


# --------------------------------------------------------------------------------------------------
# Write (A6-A8)
# --------------------------------------------------------------------------------------------------


def paste_masks_in_image(masks: torch.Tensor, boxes: torch.Tensor, image_shape, threshold: float = 0.5, want_values: bool = False,
                         skip_empty: bool = True):
    """detectron2 layers/mask_ops.py paste_masks_in_image + _do_paste_mask as executed on the CPU (call site
    custom_rcnn.py:880): one chunk per mask, skip_empty=True, F.grid_sample(align_corners=False), ``>= threshold``.
    detectron2 is not vendored in /root/reference (README :36-39, git master): this is a restatement of its published
    source; the arithmetic that decides the result (grid construction + grid_sample) is executed by torch itself.
    masks (K,S,S) f32 probabilities, boxes (K,4) f32 XYXY -> (K,H,W) bool.
    skip_empty=False restates the branch _do_paste_mask takes for CUDA tensors (the reference's live path): the whole image
    is sampled instead of the box's integer neighbourhood."""
    img_h, img_w = image_shape
    N = masks.shape[0]
    img_masks = torch.zeros(N, img_h, img_w, dtype=torch.bool)
    values = torch.zeros(N, img_h, img_w) if want_values else None
    for i in range(N):
        m, b = masks[i:i + 1, None], boxes[i:i + 1]
        x0_int, y0_int = torch.clamp(b.min(dim=0).values.floor()[:2] - 1, min=0).to(dtype=torch.int32)
        x1_int = torch.clamp(b[:, 2].max().ceil() + 1, max=img_w).to(dtype=torch.int32)
        y1_int = torch.clamp(b[:, 3].max().ceil() + 1, max=img_h).to(dtype=torch.int32)
        if not skip_empty:
            x0_int, y0_int, x1_int, y1_int = 0, 0, img_w, img_h
        x0, y0, x1, y1 = torch.split(b, 1, dim=1)
        if int(y0_int) >= int(y1_int) or int(x0_int) >= int(x1_int):
            continue        # box entirely outside the image: torch.arange would raise upstream; fast_rcnn_inference clips boxes, so it cannot occur
        img_y = torch.arange(y0_int, y1_int, dtype=torch.float32) + 0.5
        img_x = torch.arange(x0_int, x1_int, dtype=torch.float32) + 0.5
        img_y = (img_y - y0) / (y1 - y0) * 2 - 1
        img_x = (img_x - x0) / (x1 - x0) * 2 - 1
        gx = img_x[:, None, :].expand(1, img_y.size(1), img_x.size(1))
        gy = img_y[:, :, None].expand(1, img_y.size(1), img_x.size(1))
        grid = torch.stack([gx, gy], dim=3)
        if grid.numel() == 0:
            continue
        v = F.grid_sample(m.float(), grid, align_corners=False)[:, 0]
        img_masks[i, int(y0_int):int(y1_int), int(x0_int):int(x1_int)] = (v >= threshold)[0]
        if want_values:
            values[i, int(y0_int):int(y1_int), int(x0_int):int(x1_int)] = v[0]
    return (img_masks, values) if want_values else img_masks


def box_to_image_features(box_features: torch.Tensor, masks: torch.Tensor):
    """custom_rcnn.py:884-901.  box_features (K,C) f32, masks (K,H,W) bool ->
    image_features (1,C,H,W) f32, observed_pixels (H,W) bool."""
    K, C = box_features.shape
    H, W = masks.shape[1:]
    image_features = torch.zeros(1, C, H, W)
    observations = torch.zeros(1, 1, H, W)
    for i in range(K):
        mask = masks[i]
        image_features[:, :, mask] += box_features[i].reshape(1, C, 1)
        observations[:, :, mask] += 1
    observed = (observations > 0)[0, 0]
    image_features[:, :, observed] = image_features[:, :, observed] / observations[:, :, observed]
    return image_features, observed


def project_image_features_dense(image_features, observed_pixels, proj, n_cells: int, stride: int = 8):
    """LITERAL restatement of custom_rcnn.py:903-936 (one-hot bool (P', cells) -> matmul).  Only usable
    when P' * n_cells fits in RAM."""
    C = image_features.shape[1]
    f = image_features[:, :, observed_pixels].squeeze(0).permute(1, 0).reshape(-1, C)
    p = proj[observed_pixels]
    p, f = p[::stride], f[::stride]
    onehot = torch.zeros(p.shape[0], n_cells, dtype=torch.bool)
    onehot[torch.arange(p.shape[0]), p] = True
    onehot = onehot.t()
    observed_mem = torch.any(onehot, dim=1)
    onehot = onehot[observed_mem].to(torch.float32)
    s = torch.matmul(onehot, f.to(torch.float32))
    count = torch.sum(onehot, dim=1).unsqueeze(1)
    return s / count, observed_mem


def project_image_features_sparse(image_features, observed_pixels, proj, n_cells: int, stride: int = 8):
    """Same result set as project_image_features_dense without the one-hot (index_add_); fp32 sums may
    differ from the matmul in summation order only (tolerance 1e-5 of scale)."""
    C = image_features.shape[1]
    f = image_features[:, :, observed_pixels].squeeze(0).permute(1, 0).reshape(-1, C)
    p = proj[observed_pixels]
    p, f = p[::stride].long(), f[::stride].to(torch.float32)
    s = torch.zeros(n_cells, C)
    s.index_add_(0, p, f)
    n = torch.zeros(n_cells)
    n.index_add_(0, p, torch.ones(p.shape[0]))
    observed_mem = n > 0
    return s[observed_mem] / n[observed_mem].unsqueeze(1), observed_mem


def sample_mask(observed_pixels: torch.Tensor, stride: int) -> torch.Tensor:
    """Per-pixel bool: pixel is one of the every-``stride``-th observed pixels in raster order
    (custom_rcnn.py:905-914: boolean-mask compaction is raster order, then ``[::8]``)."""
    flat = observed_pixels.reshape(-1)
    rank = torch.cumsum(flat.to(torch.int64), 0) - 1
    return (flat & (rank % stride == 0)).reshape(observed_pixels.shape)


def accumulate(sums: torch.Tensor, counts: torch.Tensor, mean: torch.Tensor, observed_mem: torch.Tensor,
               proj: torch.Tensor):
    """custom_rcnn.py:696-701,738-743,759-760 on the flat (cells,C)/(cells,) views: sums += scatter(mean);
    counts += 1 for every visible cell (unique(proj))."""
    upd = torch.zeros_like(sums)
    upd[observed_mem] = mean
    vis = torch.zeros_like(counts)
    vis[torch.unique(proj.long())] = 1
    return sums + upd, counts + vis


def write_mean_frame(sums, counts, image_features, observed_pixels, proj, stride: int = 8):
    """One frame of the mean-mode write (A6 output -> A7 -> A8)."""
    mean, observed_mem = project_image_features_sparse(image_features, observed_pixels, proj, sums.shape[0], stride)
    return accumulate(sums, counts, mean, observed_mem, proj)


def dense_backbone_write(p3: torch.Tensor, proj: torch.Tensor, n_cells: int, weight=None, bias=None):
    """A7'' (bytecode-only lineage, SURVEY 8a): p3 (1,C,h,w) -> bilinear (480,640) align_corners ->
    [::8, ::8] -> optional 1x1 conv -> per-cell mean; returns the REPLACED memory (zeros elsewhere)."""
    H, W = proj.shape
    f = F.interpolate(p3, (H, W), mode="bilinear", align_corners=True)[:, :, ::8, ::8]
    if weight is not None:
        f = F.conv2d(f, weight, bias)
    C = f.shape[1]
    f = f[0].reshape(C, -1).t().contiguous()
    p = proj[::8, ::8].reshape(-1).long()
    s = torch.zeros(n_cells, C).index_add_(0, p, f)
    n = torch.zeros(n_cells).index_add_(0, p, torch.ones(p.shape[0]))
    mem = torch.zeros(n_cells, C)
    m = n > 0
    mem[m] = s[m] / n[m].unsqueeze(1)
    return mem, m


def explicit_semmap(sums: torch.Tensor, counts: torch.Tensor, zs_weight: torch.Tensor, thresh: float, n_cls: int = 20):
    """custom_rcnn.py:747-756 + visualise_clip_image_features (:938-978) on the flat views: returns
    (semmap (cells,) int64 with -1 below the threshold, normalised intensity (cells,), logits (cells, n_cls))."""
    inten = sums.abs().mean(dim=1)                                           # :747
    sel = counts > 1
    inten[sel] = inten[sel] / counts[sel]                                    # :748
    inten = (inten - inten.min()) / (inten.max() - inten.min())              # :751
    norm = 50.0 * F.normalize(sums, p=2, dim=1)                              # :949
    scores = torch.mm(norm, zs_weight)[:, :n_cls]                            # :952
    prob = scores.softmax(dim=1)                                             # :955
    _, idx = torch.max(prob, dim=1)                                          # :958
    idx = idx.clone()
    idx[inten < thresh] = -1                                                 # :968 (mask replaces the scores, :964)
    return idx, inten, scores


# --------------------------------------------------------------------------------------------------
# SMNet height-max write (A7', bytecode-only; torch_scatter 1.4.0 scatter_max canonical tie rule)
# --------------------------------------------------------------------------------------------------


def scatter_max_canonical(src: torch.Tensor, index: torch.Tensor, out: torch.Tensor):
    """``out, arg = scatter_max(src, index, dim=0, out=out)`` with the canonical rule of SURVEY 8(c):
    sequential ``if src[i] >= out[idx]: out[idx] = src[i]; arg[idx] = i`` (last/highest index wins ties, an
    equal later value replaces); arg = -1 where not raised.  parity unpinned (torch_scatter absent)."""
    o = out.clone().numpy()
    arg = (-torch.ones(out.shape[0], dtype=torch.int64)).numpy()
    s, ix = src.numpy(), index.numpy()
    # vectorised equivalent of the sequential loop: stable sort by (cell, value, position)
    import numpy as np
    keep = ~np.isnan(s)                      # `NaN >= x` is false: a NaN height never raises a cell and never shadows a finite one
    pos = np.arange(s.shape[0])[keep]
    s, ix = s[keep], ix[keep]
    if s.shape[0]:
        order = np.lexsort((pos, s, ix))
        ixs = ix[order]
        last = np.r_[ixs[1:] != ixs[:-1], True]
        win = order[last]
        cells = ix[win]
        raise_ = s[win] >= o[cells]
        o[cells[raise_]] = s[win][raise_]
        arg[cells[raise_]] = pos[win[raise_]]
    return torch.from_numpy(o), torch.from_numpy(arg)


def smnet_heightmax_frame(state, observed, height_map, feat_hwc, w2m, inliers, heights, map_w: int,
                          downsample: int = 1, linlayer=None):
    """One frame of SMNet.encode (model_test.pyc src lines 62-163, 'replace'-without-linear update):
    returns new (state, observed, height_map, arg, m).  feat_hwc (H,W,C) f32 already interpolated."""
    if downsample > 1:
        w2m, inliers, heights, feat_hwc = (t[::downsample, ::downsample] for t in (w2m, inliers, heights, feat_hwc))
    flat = (map_w * w2m[..., 1].long() + w2m[..., 0].long())[inliers]
    h = heights[inliers] + 1000
    height_map, arg = scatter_max_canonical(h, flat, height_map)
    m = arg >= 0
    observed = observed | m
    state = state.clone()
    if m.any():
        rows = feat_hwc[inliers][arg[m]]
        # model.py (3.10 bytecode, src lines 126-128): mem_update == 'replace' -> state[m] = self.linlayer(tmp_memory)
        state[m] = rows if linlayer is None else F.linear(rows, linlayer[0], linlayer[1])
    return state, observed, height_map, arg, m


# --------------------------------------------------------------------------------------------------
# Read (A10-A13)
# --------------------------------------------------------------------------------------------------


def create_implicit_memory(sums: torch.Tensor, counts: torch.Tensor) -> torch.Tensor:
    """custom_rcnn.py:764-774: sums/count where count > 1, else unchanged."""
    mem = sums.clone()
    sel = counts > 1
    mem[sel] = mem[sel] / counts.unsqueeze(1)[sel]
    return mem


def read_pool(memory16: torch.Tensor, proj: torch.Tensor) -> List[torch.Tensor]:
    """timm.py:147-168 for one image.  memory16 (cells,C) f16, proj (H,W) int64 ->
    [L0 (1,C,H/8,W/8), L1 (1,C,H/16,W/16), L2 (1,C,H/32,W/32)] f16."""
    ego = memory16[proj.long()].permute(2, 0, 1).unsqueeze(0)
    ego = F.avg_pool2d(ego.to(torch.float32), kernel_size=4, stride=4)
    levels = []
    for _ in range(3):
        ego = F.avg_pool2d(ego.to(torch.float32), kernel_size=2, stride=2).to(torch.half)
        levels.append(ego)
    return levels


def project_and_fuse(levels: Sequence[torch.Tensor], results: Sequence[torch.Tensor],
                     weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor], map_feature_weight: float,
                     fusion: str) -> List[torch.Tensor]:
    """timm.py:170-192: mem = conv1x1_l(level.f32) * MAP_FEATURE_WEIGHT ; sum | mem_only | image_only."""
    out = []
    for lvl, res, w, b in zip(levels, results, weights, biases):
        mem = F.conv2d(lvl.to(torch.float32), w, b)
        mem = mem * map_feature_weight
        if fusion == "sum":
            new = mem + res
        elif fusion == "mem_only":
            new = mem
        elif fusion == "image_only":
            new = res
        else:
            raise UnboundLocalError("new_res")       # the reference leaves new_res undefined (timm.py:181-189)
        out.append(new.to(res.dtype))
    return out


def assign_boxes_to_levels(boxes: torch.Tensor, min_level: int = 3, max_level: int = 5, canonical_box_size: int = 224,
                           canonical_level: int = 4) -> torch.Tensor:
    """detectron2 modeling/poolers.py assign_boxes_to_levels (published source restated; detectron2 is not under /root/reference):
    floor(canonical_level + log2(sqrt(area) / canonical_box_size + eps)) clamped to [min_level, max_level], minus min_level."""
    import sys
    box_sizes = torch.sqrt((boxes[:, 2] - boxes[:, 0]) * (boxes[:, 3] - boxes[:, 1]))
    lvl = torch.floor(canonical_level + torch.log2(box_sizes / canonical_box_size + sys.float_info.epsilon))
    lvl = torch.clamp(lvl, min=min_level, max=max_level)
    return lvl.to(torch.int64) - min_level


def roi_levels(boxes: torch.Tensor, n_levels: int) -> torch.Tensor:
    """The level ROIPooler pools each box from: assign_boxes_to_levels with levels 3 .. 3 + n_levels - 1, and -1 where that lies outside
    [0, n_levels).  A box inverted in exactly one axis (negative area) or with a NaN coordinate has a NaN size; torch.clamp keeps the
    NaN and the int64 cast turns it into an out-of-range integer, so ROIPooler's `level_assignments == level` matches no level and the
    box pools zeros.  eod_read_roi reports such a box as level -1."""
    lvl = assign_boxes_to_levels(boxes, 3, 3 + n_levels - 1)
    return torch.where((lvl >= 0) & (lvl < n_levels), lvl, torch.full_like(lvl, -1))


def _f2i(v):
    """C's (int) of an fp32 array as the GPU converts it (cvt.rzi.s32.f32): truncation, saturating, NaN -> 0."""
    import numpy as np
    v = np.asarray(v, np.float32)
    return np.where(np.isnan(v), 0, np.clip(np.trunc(np.nan_to_num(v)), -2.0 ** 31, 2.0 ** 31 - 1)).astype(np.int64)


def roi_align_f32(level, box, scale: float, pooled: int = 7, sampling_ratio: int = 0):
    """ROIAlign (aligned=True, detectron2 ROIAlignV2) of one level over one box, restated in eod_read_roi's arithmetic: level (C,h,w)
    f32 numpy, box 4 XYXY image-pixel coordinates -> (bins (C,pooled,pooled) f32, valid (pooled,pooled) f32 = n_valid / count, the
    share of each bin's sample points that lie on the level, i.e. ROIAlign of a constant-1 plane up to the rounding of w1+w2+w3+w4).
    Every operation is one fp32 rounding, in the order of torchvision's CPU kernel (torchvision/csrc/ops/cpu/roi_align_kernel.cpp):
    sample point, the (-1, h] x (-1, w] test, the clamps, the bilinear weights, val = ((w1 v1 + w2 v2) + w3 v3) + w4 v4, accumulated
    sample by sample (iy outer, ix inner), then / count.  The bins and channels of one box are independent of each other, so the
    arrays run over them while the samples stay sequential: every output element sees exactly the kernel's operation order.
    fp32 -> int casts follow the GPU (NaN -> 0)."""
    import numpy as np
    f = np.float32
    C, h, w = level.shape
    P = f(pooled)
    x1, y1, x2, y2 = (f(v) for v in box)
    sc = f(scale)
    rsw, rsh = f(f(x1 * sc) - f(0.5)), f(f(y1 * sc) - f(0.5))
    rew, reh = f(f(x2 * sc) - f(0.5)), f(f(y2 * sc) - f(0.5))
    roi_w, roi_h = f(rew - rsw), f(reh - rsh)
    bin_h, bin_w = f(roi_h / P), f(roi_w / P)
    gh = sampling_ratio if sampling_ratio > 0 else int(_f2i(np.ceil(f(roi_h / P))))
    gw = sampling_ratio if sampling_ratio > 0 else int(_f2i(np.ceil(f(roi_w / P))))
    count = f(max(gh * gw, 1))
    pb = np.arange(pooled, dtype=f)
    start_y, start_x = (rsh + pb * bin_h).astype(f), (rsw + pb * bin_w).astype(f)           # rs + p * bin, per bin row / column
    acc = np.zeros((C, pooled, pooled), f)
    n_valid = np.zeros((pooled, pooled), np.int64)
    for iy in range(gh):
        yy = (start_y + f(f(f(iy + 0.5) * bin_h) / f(gh))).astype(f)
        for ix in range(gw):
            xx = (start_x + f(f(f(ix + 0.5) * bin_w) / f(gw))).astype(f)
            y, x = np.broadcast_to(yy[:, None], (pooled, pooled)).copy(), np.broadcast_to(xx[None, :], (pooled, pooled)).copy()
            empty = (y < -1.0) | (y > f(h)) | (x < -1.0) | (x > f(w))                       # NaN compares false: not empty
            n_valid += ~empty
            y[y <= 0] = 0
            x[x <= 0] = 0
            y_low, x_low = _f2i(y), _f2i(x)
            top, right = y_low >= h - 1, x_low >= w - 1
            y_low[top], x_low[right] = h - 1, w - 1
            y[top], x[right] = f(h - 1), f(w - 1)
            y_high, x_high = np.where(top, y_low, y_low + 1), np.where(right, x_low, x_low + 1)
            ly, lx = (y - y_low.astype(f)).astype(f), (x - x_low.astype(f)).astype(f)
            hy, hx = (f(1) - ly).astype(f), (f(1) - lx).astype(f)
            w1, w2, w3, w4 = hy * hx, hy * lx, ly * hx, ly * lx
            val = ((w1 * level[:, y_low, x_low] + w2 * level[:, y_low, x_high]) + w3 * level[:, y_high, x_low]) + w4 * level[:, y_high, x_high]
            acc = np.where(empty, acc, acc + val)
    return (acc / count).astype(f), (n_valid.astype(f) / count).astype(f)


def roi_read(levels: Sequence[torch.Tensor], boxes_per_image: Sequence[torch.Tensor], pooled: int = 7, strides=(8, 16, 32)):
    """The box pooling of detic_roi_heads.py:331-334 (detectron2 ROIPooler, ROIAlignV2 = torchvision roi_align(aligned=True),
    sampling_ratio 0) applied to the pooled MEMORY levels: levels[l] (B,C,h,w) -> (sum n_i, C, pooled, pooled) f32, levels (sum n_i;
    -1 for a box ROIPooler pools from no level, see roi_levels).  torchvision's CPU ROIAlign is EXECUTED here; the level assignment is
    the restatement above."""
    from torchvision.ops import roi_align
    boxes = torch.cat(list(boxes_per_image), 0).float()
    bidx = torch.cat([torch.full((b.shape[0], 1), float(i)) for i, b in enumerate(boxes_per_image)], 0)
    rois = torch.cat([bidx, boxes], 1)
    lvl = roi_levels(boxes, len(levels))
    out = torch.zeros(boxes.shape[0], levels[0].shape[1], pooled, pooled)
    for k, (x, s) in enumerate(zip(levels, strides)):
        sel = (lvl == k).nonzero().squeeze(1)
        if sel.numel():
            out[sel] = roi_align(x.float().contiguous(), rois[sel], (pooled, pooled), 1.0 / s, 0, True)
    return out, lvl


def read_frame(sums, counts, proj) -> List[torch.Tensor]:
    """A10 -> A11 -> A12 for one frame."""
    return read_pool(create_implicit_memory(sums, counts).to(torch.half), proj)
