"""Exactly summable inputs for the accumulating kernels (mean write, object write + flush_slots, project_fuse, linear_rows, semmap).

Every value such a case can produce lies on the lattice 2^-q * Z with |x| < 2^(24-q): features are small integers times 2^-k, every
written cell receives a power-of-two number of sampled pixels (so 1/n, x * rcp(n) and x / n are exact), a sampled pixel is covered by
1, 2 or 4 objects, and GEMM operands have at most 11 significant bits.  Then every partial sum is exact in fp32 whatever the reduction
order, the float64 result is an fp32 number, and a correct kernel must return it bit for bit.  ``check_lattice`` asserts the bound
for a given case; tests/test_exact_cases.py checks the promise on the CPU, tests/test_gpu_exact.py holds the kernels to it.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np


def dyadic(rng: np.random.Generator, shape, bits: int, q: int, dtype=np.float32) -> np.ndarray:
    """Integers in [-(2^bits - 1), 2^bits - 1] times 2^-q."""
    m = (1 << bits) - 1
    return (rng.integers(-m, m + 1, shape).astype(np.float64) * 2.0 ** -q).astype(dtype)


def lattice_q(a: np.ndarray, q_max: int = 80) -> int:
    """Smallest q with every element of ``a`` an integer multiple of 2^-q (finite inputs)."""
    a = np.asarray(a, np.float64).reshape(-1)
    a = a[a != 0]
    if a.size == 0:
        return 0
    for q in range(-64, q_max + 1):
        s = np.ldexp(a, q)
        if np.array_equal(s, np.round(s)):
            return q
    raise AssertionError(f"values need more than 2^-{q_max} resolution")


def check_lattice(values: Sequence[np.ndarray], q: int, bound: float) -> None:
    """Assert that every value lies on 2^-q * Z and that ``bound`` (an upper bound of |x| over every partial sum the computation can
    form, in any order) is below 2^(24 - q): then fp32 represents every partial sum exactly."""
    for v in values:
        v = np.asarray(v, np.float64)
        s = np.ldexp(v, q)
        assert np.array_equal(s, np.round(s)), f"a value is off the 2^-{q} lattice (needs 2^-{lattice_q(v)})"
    assert bound < 2.0 ** (24 - q), f"partial sums up to {bound} do not fit 24 bits at 2^-{q}"


def pow2_sizes(rng: np.random.Generator, n: int, max_log2: int, first: Optional[int] = None) -> List[int]:
    """Split n into power-of-two group sizes (random exponents up to max_log2, 1-pixel groups included)."""
    out = [] if first is None else [int(first)]
    left = n - sum(out)
    assert left >= 0
    while left:
        k = int(rng.integers(0, max_log2 + 1))
        s = 1 << k
        while s > left:
            s >>= 1
        out.append(s)
        left -= s
    return out


def index_plane(rng: np.random.Generator, H: int, W: int, cells: int, samp: Optional[np.ndarray] = None, max_log2: int = 5,
                big: Optional[int] = None, n_unsampled_cells: int = 8, mix: float = 0.5) -> np.ndarray:
    """(H,W) int32 cell plane in which every cell holds a power-of-two number of SAMPLED pixels (samp (H,W) bool, None = all).
    Groups are laid out along the sampled pixels in raster order, so they form runs that cross warps, TMA tiles and strips;
    ``mix`` of the 64-pixel windows then permute their labels (same group sizes, non-contiguous groups inside a tile).  Unsampled
    pixels continue the run before them, and some runs of them go to ``n_unsampled_cells`` cells that get no sample at all (visible
    without a sample: frame_cnt bit 31).  ``big``: size of the first group (e.g. 2^18 at 480x640)."""
    HW = H * W
    s = np.ones(HW, bool) if samp is None else np.asarray(samp, bool).reshape(-1)
    pos = np.nonzero(s)[0]
    sizes = pow2_sizes(rng, pos.size, max_log2, big)
    n_unsamp = n_unsampled_cells if samp is not None else 0
    assert len(sizes) + n_unsamp <= cells, f"{len(sizes)} groups + {n_unsamp} unsampled cells > {cells} cells"
    perm = rng.permutation(cells).astype(np.int32)
    lab = np.repeat(perm[: len(sizes)], sizes)
    for w0 in range(0, lab.size, 64):                   # permute labels inside some windows: group sizes are unchanged
        if rng.random() < mix:
            seg = lab[w0:w0 + 64]
            lab[w0:w0 + 64] = seg[rng.permutation(seg.size)]
    idx = np.empty(HW, np.int32)
    if pos.size:
        # each unsampled pixel takes the label of the last sampled pixel before it (the first sampled one before any)
        last = np.maximum.accumulate(np.where(s, np.arange(HW), -1))
        src = np.where(last >= 0, last, pos[0])
        full = np.zeros(HW, np.int32)
        full[pos] = lab
        idx[:] = full[src]
    else:
        idx[:] = perm[0]
    if n_unsamp:
        spare = perm[len(sizes): len(sizes) + n_unsamp]
        un = np.nonzero(~s)[0]
        for c in spare:                                  # a short run of unsampled pixels per spare cell
            if un.size:
                p0 = int(un[rng.integers(0, un.size)])
                run = np.arange(p0, min(p0 + int(rng.integers(1, 40)), HW))
                idx[run[~s[run]]] = c
    return idx.reshape(H, W)


def sample_counts(idx: np.ndarray, samp: Optional[np.ndarray], cells: int) -> np.ndarray:
    i = np.asarray(idx).reshape(-1)
    if samp is not None:
        i = i[np.asarray(samp, bool).reshape(-1)]
    return np.bincount(i, minlength=cells)


def assert_pow2_counts(n: np.ndarray) -> None:
    nz = n[n > 0]
    assert ((nz & (nz - 1)) == 0).all(), "a cell's sample count is not a power of two"


def mean_write_f64(sums0: np.ndarray, feat_chw: np.ndarray, idx: np.ndarray, samp: Optional[np.ndarray], cells: int):
    """float64 sums0 + per-cell mean of the sampled pixels (the mean write of one frame of one episode); also the bound of every
    partial sum (|sums0| + sum |f| / n per cell and channel) and the sample counts."""
    C = feat_chw.shape[0]
    f = np.asarray(feat_chw, np.float64).reshape(C, -1).T
    i = np.asarray(idx).reshape(-1)
    if samp is not None:
        keep = np.asarray(samp, bool).reshape(-1)
        f, i = f[keep], i[keep]
    n = np.bincount(i, minlength=cells)
    s = np.zeros((cells, C))
    a = np.zeros((cells, C))
    if i.size:                                          # float64 sums of lattice values: exact in any order
        order = np.argsort(i, kind="stable")
        fs, cs = f[order], i[order]
        starts = np.r_[0, np.nonzero(cs[1:] != cs[:-1])[0] + 1]
        s[cs[starts]] = np.add.reduceat(fs, starts, axis=0)
        a[cs[starts]] = np.add.reduceat(np.abs(fs), starts, axis=0)
    nn = np.maximum(n, 1)[:, None]
    out = np.asarray(sums0, np.float64) + s / nn
    bound = float((np.abs(np.asarray(sums0, np.float64)) + a / nn).max()) if cells else 0.0
    return out, bound, n


# --------------------------------------------------------------------------------------------------------------------------------
# object regime
# --------------------------------------------------------------------------------------------------------------------------------
def object_boxes(rng: np.random.Generator, H: int, W: int, n_base: int, copies: Sequence[int] = (1, 2, 4), gap: int = 4) -> np.ndarray:
    """(K,4) f32 XYXY boxes: n_base disjoint boxes (cells of a grid, ``gap`` pixels apart so that neither the masks nor their pasted
    neighbourhoods touch), each repeated 1, 2 or 4 times - a covered pixel has 1, 2 or 4 objects."""
    g = int(np.ceil(np.sqrt(n_base)))
    ch, cw = H // g, W // g
    assert ch > 2 * gap + 2 and cw > 2 * gap + 2, "image too small for that many disjoint boxes"
    out = []
    for b in range(n_base):
        r, c = divmod(b, g)
        y0 = r * ch + gap + int(rng.integers(0, 3))
        x0 = c * cw + gap + int(rng.integers(0, 3))
        y1 = (r + 1) * ch - gap - int(rng.integers(0, 3))
        x1 = (c + 1) * cw - gap - int(rng.integers(0, 3))
        box = np.array([x0 + rng.uniform(0, 0.9), y0 + rng.uniform(0, 0.9), x1 - rng.uniform(0, 0.9), y1 - rng.uniform(0, 0.9)], np.float32)
        out += [box] * int(rng.choice(copies))
    return np.stack(out).astype(np.float32)


def object_case(rng: np.random.Generator, H: int, W: int, C: int, n_base: int, bits: int = 4, q: int = 2, probs_size: int = 28,
                copies: Sequence[int] = (1, 2, 4)) -> Dict[str, np.ndarray]:
    """Detections whose pasted masks overlap 1, 2 or 4 times: box_features (K,C) dyadic, mask probabilities (K,S,S) in {0,1} (the
    copies of a box share their probabilities), boxes (K,4), and the masks the oracle pastes from them (K,H,W)."""
    import oracle
    boxes = object_boxes(rng, H, W, n_base, copies)
    K = boxes.shape[0]
    probs = np.empty((K, probs_size, probs_size), np.float32)
    k = 0
    while k < K:
        j = k
        while j < K and np.array_equal(boxes[j], boxes[k]):
            j += 1
        p = (rng.random((probs_size, probs_size)) < 0.75).astype(np.float32)
        p[probs_size // 4: 3 * probs_size // 4, probs_size // 4: 3 * probs_size // 4] = 1.0      # never an empty mask
        probs[k:j] = p
        k = j
    masks = oracle.paste_masks(probs, boxes, H, W, 0.5)
    cover = masks.sum(0)
    assert set(np.unique(cover).tolist()) <= {0, 1, 2, 4}, "pasted masks overlap other than 1, 2 or 4 times"
    return {"box_features": dyadic(rng, (K, C), bits, q), "probs": probs, "boxes": boxes, "masks": masks}


def object_mean_f64(box_features: np.ndarray, masks: np.ndarray) -> np.ndarray:
    """Per-pixel mean of the covering objects' features, float64 (C, H*W) (zero where nothing covers)."""
    K, H, W = masks.shape
    m = masks.reshape(K, -1).astype(np.float64)
    s = np.asarray(box_features, np.float64).T @ m
    cnt = m.sum(0)
    return s / np.maximum(cnt, 1)


# --------------------------------------------------------------------------------------------------------------------------------
# GEMM operands
# --------------------------------------------------------------------------------------------------------------------------------
def gemm_bound(a: np.ndarray, w: np.ndarray) -> np.ndarray:
    """sum_k |a_mk| |w_nk| - bounds every partial sum of a row product, in any order."""
    return np.abs(np.asarray(a, np.float64)) @ np.abs(np.asarray(w, np.float64)).T


def split_weights_f64(w: np.ndarray):
    """The hi / lo terms project_split_weights forms: hi = half(w), lo = half((w - hi) * 2^11)."""
    w = np.asarray(w, np.float32)
    hi = w.astype(np.float16)
    lo = ((w - hi.astype(np.float32)) * np.float32(2048.0)).astype(np.float16)
    return hi, lo


def weights_with_lo(rng: np.random.Generator, shape, hi_bits: int = 3, hi_q: int = 4, lo_q: int = 13) -> np.ndarray:
    """fp32 weights hi + lo with hi = a * 2^-hi_q and a nonzero lo = +-2^-lo_q on about half the entries (below half an fp16 ulp of
    most hi, so the split puts it into W_lo; where hi is small the fp16 hi holds all of it and W_lo is 0)."""
    hi = dyadic(rng, shape, hi_bits, hi_q, np.float64)
    lo = rng.integers(-1, 2, shape) * 2.0 ** -lo_q
    return (hi + lo).astype(np.float32)


def tf32_exact(x: np.ndarray) -> bool:
    """At most 11 significant bits: the 3xTF32 split keeps the value in its big half and the small half is zero."""
    x = np.asarray(x, np.float32).reshape(-1)
    return bool(((x.view(np.uint32) & np.uint32(0x1FFF)) == 0).all())
