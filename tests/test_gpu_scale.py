"""The kernels at the batch sizes the benchmark runs (run on the B200 box with `-m gpu`).

Two kinds of code only run at these sizes:
  * the loop-carried part of every launcher that caps its grid at a multiple of the SM count (the read's prefetch of the next item and
    its (episode, quadrant) carry, the level-2 pool, the reset / refresh / semmap row sweeps, the height-max reset and the passes of the
    height-max update over its cell list, the fusion epilogue, finalize over the cell plane): below the cap every warp gets one item;
  * state rows past element offset 2^31 (byte offset 2^32): BASELINE configs[1] keeps 64 x 250 000 x 256 fp32 sums, configs[2]
    16 x 10^6 x 256.
Every case asserts through the sizing helpers below - one per capped launcher, mirroring its grid formula - that it really takes more
than one trip, so that a changed cap fails here instead of silently no longer reaching the loop.  tests/test_scale_host.py checks the
same shapes against the helpers with 148 SMs on a machine without a GPU.

Results are held to the oracle (oracle.read_pool_f16, reference_ops) bit for bit, to fp64 within the tolerance of
test_linlayer_update_vs_fp64_oracle, or to an independently run path (one episode alone, torch on the device).
"""
import gc
import math
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import path_check
from oracle import reference_ops as R

pytestmark = pytest.mark.gpu

I32_ELEMS = 2 ** 31


# ---- sizing: one helper per capped launcher, the same integer arithmetic as its host code ----------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def device_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def read_ctas_per_sm():
    """EOD_READ_CTAS_PER_SM as read_pool.cu reads it: atoi of the value, 16 when unset or not positive."""
    v = os.environ.get("EOD_READ_CTAS_PER_SM")
    if v is None:
        return 16
    s = v.strip()
    n = len(s) - len(s.lstrip("+-"))
    while n < len(s) and s[n].isdigit():
        n += 1
    try:
        k = int(s[:n])
    except ValueError:
        k = 0
    return k if k > 0 else 16


def read_pool_trips(E, H, W, sms):
    """read_pool_kernel: items (one 16x16 quadrant of one episode) per warp, for the warp that takes the most."""
    n_items = E * (H // 16) * (W // 16)
    blocks = min(_cdiv(n_items, 8), sms * read_ctas_per_sm())
    return _cdiv(n_items, blocks * 8)


def pool_level2_trips(E, H, W, C, sms):
    """pool_level2_kernel: trips of its grid-stride loop over E * (H/32) * (W/32) * C/4 four-channel groups."""
    total = E * (H // 32) * (W // 32) * (C // 4)
    blocks = min(_cdiv(total, 256), sms * 8)
    return _cdiv(total, blocks * 256)


def _row_sweeps(n_rows, sms):
    blocks = min(_cdiv(n_rows, 256), sms * 16)             # 8 warps x 32 rows per block and sweep
    return _cdiv(n_rows, blocks * 256)


def touched_rows_sweeps(E, n_cells, sms):
    """touched_rows_kernel (eod_reset_touched / eod_reset_episodes / eod_refresh_norm16): sweeps over the E * n_cells rows."""
    return _row_sweeps(E * n_cells, sms)


def heightmax_reset_sweeps(E, n_cells, sms):
    """heightmax_reset_kernel: sweeps over the E * n_cells rows."""
    return _row_sweeps(E * n_cells, sms)


def semmap_update_sweeps(E, n_cells, sms):
    """semmap_update_kernel: sweeps over the E * n_cells rows."""
    return _row_sweeps(E * n_cells, sms)


def heightmax_update_pass_cells(E, list_cap, sms):
    """heightmax_update_kernel: listed cells one pass of an episode's blocks covers (8 warps x 32 cells per block)."""
    return min(_cdiv(list_cap, 256), _cdiv(sms * 8, E)) * 256


def fuse_trips(n, sms):
    """fuse_kernel: trips of its grid-stride loop over the n // 4 float4."""
    n4 = n // 4
    blocks = max(1, min(_cdiv(n4, 256), sms * 16))
    return _cdiv(n4, blocks * 256)


def finalize_cells_trips(E, n_cells, HW, sms):
    """finalize_cells_kernel (eod_finalize_counts when the grid is comparable to the image): trips of 2048 cells per block.
    0 when the launcher takes the pixel-driven kernel instead."""
    n_rows = E * n_cells
    if not (n_cells <= 4 * HW and n_rows % 4 == 0):
        return 0
    blocks = min(_cdiv(n_rows, 2048), sms * 16)
    return _cdiv(n_rows // 4, blocks * 512)


# ---- the cases (shapes shared with tests/test_scale_host.py) ------------------------------------------------------------------------
READ_E, READ_H, READ_W, READ_CELLS = 64, 480, 640, 3001
READ_FAR = {"f16": dict(E=18, n_cells=10 ** 6, C=128, e=17), "f32": dict(E=10, n_cells=10 ** 6, C=256, e=9)}
DENSE = dict(E=64, mw=500, mh=500, C=256, H=480, W=640, cell=0.2, frames=3, checked=(0, 34, 63))
DENSE_RESET, DENSE_KEEP = (1, 34, 36, 62, 63), (0, 2, 33, 35, 37, 61)
HMAX = dict(E=16, mw=1000, mh=1000, C=256, H=480, W=640, cell=0.02, frames=3, checked=(0, 9, 15))
HMAX_RESET, HMAX_KEEP = (1, 9, 15), (0, 8, 10, 14)
HLIST = dict(E=64, mw=501, mh=499, C=64, H=480, W=640, cell=0.02, frames=2, lin_c=128)
SWEEP = dict(E=5, n_cells=999 * 1001, C=128)
SWEEP_MASKS = {"one": (0, 1, 0, 0, 0), "alternate": (1, 0, 1, 0, 1), "last": (0, 0, 0, 0, 1)}
FUSE_N = 2_500_003


# ---- helpers ------------------------------------------------------------------------------------------------------------------
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


def _bits(t):
    t = t.contiguous()
    return t.view({torch.float32: torch.int32, torch.float16: torch.int16}.get(t.dtype, t.dtype))


def _mask(E, sel, dev):
    m = torch.zeros((E,), dtype=torch.int32)
    m[list(sel)] = 1
    return m.to(dev)


def _stress_planes(H, W, cells, seed):
    """The id patterns of stress_cases.stress_read at H x W: checkerboard (16 runs per window), 1-px stripes both ways, noise, blocks
    with edges off the 4/8/16 lattice, sparse noise over a coarse tiling."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W]
    return [((yy + xx) % 2) * (cells - 1), xx % cells, yy % cells, rng.integers(0, cells, (H, W)), (yy // 24) * 7 % cells + (xx // 40) % 3,
            np.where(rng.uniform(size=(H, W)) < 0.02, rng.integers(0, cells, (H, W)), (yy // 9 + xx // 13) % cells)]


def _episode_ids(E, H, W, cells, seed=64):
    """(E,H,W) int32: episode e reads pattern e % 6, rolled by (e, 3e) and offset by 131 e - no two episodes read the same."""
    pats = _stress_planes(H, W, cells, seed)
    return np.stack([(np.roll(pats[e % 6], (e, 3 * e), axis=(0, 1)) + 131 * e) % cells for e in range(E)]).astype(np.int32)


def _check_read(got, ref_of, episodes, what):
    lv = [g.contiguous().cpu().numpy().view(np.uint16) for g in got]      # logical (E,C,h,w)
    for e in episodes:
        ref = ref_of(e)
        for k in range(3):
            r = ref[k].view(np.uint16)
            assert np.array_equal(lv[k][e], r), (what, e, k, int((lv[k][e] != r).sum()))


# ---- 1. read past its grid cap ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,table", [(128, "f16"), (256, "f16"), (512, "f16"), (256, "f32")])
def test_read_pool_past_grid_cap_vs_oracle(eod, cuda, C, table):
    """E = 64 at 480x640: every warp walks several quadrants (prefetched ids, stepped (e, qy, qx)) and the level-2 pool loops.  All
    three levels equal oracle.read_pool_f16 bit for bit, int32 and int64 ids; every episode at C = 128, else every 7th and the last."""
    E, H, W, cells = READ_E, READ_H, READ_W, READ_CELLS
    sms = device_sms()
    assert read_pool_trips(E, H, W, sms) > 1 and pool_level2_trips(E, H, W, C, sms) > 1
    _need(E * cells * C * 4 + E * H * W * 12 + E * C * H * W // 16)
    rng = np.random.default_rng(C + (table == "f32"))
    ids = _episode_ids(E, H, W, cells)
    episodes = range(E) if (C, table) == (128, "f16") else sorted(set(range(0, E, 7)) | {E - 1})
    if table == "f16":
        tab = (rng.standard_normal((E, cells, C), dtype=np.float32) * rng.choice([1e-3, 1.0, 300.0], (E, cells, 1))).astype(np.float16)
        tab[:, 0, :8] = [0.0, -0.0, 6e-8, -6e-8, 65504.0, -65504.0, 1.0, -1.0]
        args, ref_table = (_t(tab, cuda), None), lambda e: tab[e]
    else:
        sums = (rng.standard_normal((E, cells, C), dtype=np.float32) * rng.choice([1e-3, 1.0, 300.0], (E, cells, 1))).astype(np.float32)
        sums[:, :5] = -0.0
        sums[:, 5:8] = 7e4                                                             # > fp16 max: rounds to inf like torch
        counts = rng.integers(0, 7, (E, cells)).astype(np.float32)
        args = (_t(sums, cuda), _t(counts, cuda))
        ref_table = lambda e: R.create_implicit_memory(torch.from_numpy(sums[e]), torch.from_numpy(counts[e])).half().numpy()
    refs = {}

    def ref_of(e):
        if e not in refs:
            refs[e] = oracle.read_pool_f16(ref_table(e), ids[e])
        return refs[e]

    for dtype in (np.int32, np.int64):
        got = eod.ops.read_pool(*args, _t(ids.astype(dtype), cuda))
        _check_read(got, ref_of, episodes, (C, table, dtype.__name__))
        del got


# ---- 2. read rows past 2^31 elements ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("table", ["f16", "f32"])
def test_read_pool_rows_past_2_31_elements(eod, cuda, table):
    """The checked episode's first table row lies at element offset >= 2^31; its ids hit the first and the last cell of the grid.
    fp16 table with int32 ids, fp32 sums + counts with int64 ids, against the oracle on that episode."""
    p = READ_FAR[table]
    E, N, C, e = p["E"], p["n_cells"], p["C"], p["e"]
    H, W = READ_H, READ_W
    assert e * N * C >= I32_ELEMS
    elem = 2 if table == "f16" else 4
    _need(E * N * C * elem + E * N * 4 + E * H * W * 8 + E * C * H * W // 16)
    rng = np.random.default_rng(17)
    used = np.unique(np.concatenate([[0, N - 1], rng.integers(0, N, 2000)]))          # sorted: compact id u <-> cell used[u]
    U = len(used)
    compact = _episode_ids(1, H, W, U, seed=5)[0]
    compact[:8, :8] = 0                                                                 # a whole 8x8 block of cell 0
    compact[-1, -16:] = U - 1                                                           # and the last cell, in a mixed window
    vals = rng.standard_normal((U, C), dtype=np.float32) * 3
    dtype = torch.float16 if table == "f16" else torch.float32
    tab = torch.zeros((E, N, C), dtype=dtype, device=cuda)
    rows = _t(used.astype(np.int64), cuda)
    idx = torch.zeros((E, H, W), dtype=torch.int32 if table == "f16" else torch.int64, device=cuda)
    idx[e] = _t(used[compact], cuda).to(idx.dtype)
    if table == "f16":
        tab[e, rows] = _t(vals, cuda).half()
        got = eod.ops.read_pool(tab, None, idx)
        ref16 = vals.astype(np.float16)
    else:
        cnt = rng.integers(0, 7, U).astype(np.float32)
        counts = torch.zeros((E, N), device=cuda)
        tab[e, rows] = _t(vals, cuda)
        counts[e, rows] = _t(cnt, cuda)
        got = eod.ops.read_pool(tab, counts, idx)
        ref16 = R.create_implicit_memory(torch.from_numpy(vals), torch.from_numpy(cnt)).half().numpy()
    _check_read(got, lambda _: oracle.read_pool_f16(ref16, compact), [e], table)


# ---- 3. configs[1] through EpisodeBatch ---------------------------------------------------------------------------------------
def test_configs1_episode_batch_vs_oracle_reset_and_refresh(eod, cuda):
    """E = 64, 500x500, C = 256, 3 frames through EpisodeBatch(pipeline=True) against the oracle frame by frame on episodes 0, 34 (the
    first whose rows start past 2^31 elements) and 63: the TMA write over 64 episodes, finalize over the cell plane past its cap, the
    incremental fp16 table and the read at E = 64.  Then refresh_read(mask) rebuilds the fp16 rows of the selected slots from sums and
    counts, and reset(mask=) clears the selected slots - chunks of 32 rows straddle their boundaries - and nothing else."""
    p = DENSE
    E, mw, mh, C, H, W, cell = p["E"], p["mw"], p["mh"], p["C"], p["H"], p["W"], p["cell"]
    n_cells = mw * mh
    sms = device_sms()
    assert 34 * n_cells * C >= I32_ELEMS > 33 * n_cells * C
    assert finalize_cells_trips(E, n_cells, H * W, sms) > 1 and read_pool_trips(E, H, W, sms) > 1
    assert touched_rows_sweeps(E, n_cells, sms) > 1
    assert all((e * n_cells) % 32 for e in (1, 35, 37, 63))                             # these slots start inside a 32-row chunk
    _need(E * n_cells * C * 6 + E * C * H * W * 4 + 3 * 1024 ** 3)
    eps = {e: eod.episodes.make_episode(1234 + e, p["frames"], H, W, mw, mh, cell) for e in p["checked"]}
    filler = eod.episodes.make_episode(999, p["frames"], H, W, mw, mh, cell)
    all_eps = [eps.get(e, filler) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in all_eps]), cuda)
    Ts = [eod.transform3d(torch.from_numpy(ep.xyzhe)) for ep in all_eps]
    host = {e: dict(depth=eps[e].depth, T=Ts[e].numpy(), shift=eps[e].map_world_shift) for e in p["checked"]}
    slab = torch.empty((E, C, H, W), device=cuda)                  # synced steps: frame t + 1 is generated after frame t's write
    gen = torch.Generator(device=cuda)

    def feat_fn(t):
        def make():
            gen.manual_seed(77 + t)
            return slab.normal_(generator=gen)
        return make

    frames = [dict(depth=_t(np.stack([ep.depth[t] for ep in all_eps]), cuda), pose=torch.stack([T[t, :3].reshape(12) for T in Ts]).to(cuda),
                   feat=feat_fn(t)) for t in range(p["frames"])]
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, pipeline=True)
    res = path_check.check_dense_steps(batch, frames, shifts, intr, cell, host, synced=True)
    assert res["ok"], path_check.summary(res)
    del frames, slab, res
    torch.cuda.empty_cache()

    # refresh_read(mask): the selected checked slots get their fp16 rows back from sums / counts, the unselected one stays as it is
    for e in p["checked"]:
        batch.norm16[e].zero_()
    batch.refresh_read(_mask(E, (34, 63), cuda))
    batch.join()
    torch.cuda.synchronize()
    assert not bool(batch.norm16[0].any())
    for e in (34, 63):
        seen = batch.counts[e] != 0
        assert int(seen.sum()) > 100
        ref = R.create_implicit_memory(batch.sums[e][seen].cpu(), batch.counts[e][seen].cpu()).half()
        assert torch.equal(_bits(batch.norm16[e][seen].cpu()), _bits(ref)), e
        assert not bool(((batch.norm16[e] != 0).any(1) & ~seen).any()), e

    # reset(mask=): selected slots all zero, unselected neighbours bit-identical
    before = {e: (batch.sums[e].clone(), batch.counts[e].clone(), batch.norm16[e].clone()) for e in DENSE_KEEP}
    assert all(bool(batch.counts[e].any()) for e in DENSE_RESET)
    batch.reset(mask=_mask(E, DENSE_RESET, cuda))
    batch.join()
    torch.cuda.synchronize()
    for e in DENSE_RESET:
        assert not bool(batch.sums[e].any()) and not bool(batch.counts[e].any()) and not bool(batch.norm16[e].any()), e
    for e, (s, c, n) in before.items():
        assert torch.equal(_bits(batch.sums[e]), _bits(s)) and torch.equal(batch.counts[e], c) and torch.equal(_bits(batch.norm16[e]), _bits(n)), e


# ---- 4. configs[2] through HeightMaxBatch -------------------------------------------------------------------------------------
def _hmax_episodes(eod, E, T, H, W, mw, mh, cell, seed, room_size=(24.0, 16.0)):
    eps = [eod.episodes.make_episode(seed + e, T, H, W, mw, mh, cell, room_size=room_size) for e in range(E)]
    Ts = [eod.transform3d(torch.from_numpy(ep.xyzhe)) for ep in eps]
    shifts = np.stack([np.concatenate([ep.map_world_shift, np.zeros(3, np.float32)]) for ep in eps])
    return eps, Ts, shifts


def _hmax_oracle(ep, T, feats_hwc, intr, mw, mh, cell, C, linlayer=None, dtype=torch.float32):
    """R.smnet_heightmax_frame over the episode's frames; feats_hwc[t] (H,W,C) CPU."""
    n = mw * mh
    c_mem = C if linlayer is None else linlayer[0].shape[0]
    state, observed, hmap = torch.zeros(n, c_mem, dtype=dtype), torch.zeros(n, dtype=torch.bool), torch.zeros(n)
    for t, f in enumerate(feats_hwc):
        o = oracle.backproject_quantize(ep.depth[t], T[t].numpy(), intr, ep.map_world_shift, np.zeros(3, np.float32), cell, mw, mh, 0, 0.5)
        state, observed, hmap, _, m = R.smnet_heightmax_frame(state, observed, hmap, f.to(dtype), torch.from_numpy(o["q2"]),
                                                              ~torch.from_numpy(o["outlier"].astype(bool)), torch.from_numpy(o["height"]), mw, 1,
                                                              linlayer=linlayer)
    return state, observed, hmap, m


def test_configs2_heightmax_batch_vs_alone_oracle_and_reset(eod, cuda):
    """E = 16, 1000x1000, C = 256, 0.02 m cells, from depth, 3 frames: every episode equals the same episode run alone in one
    HeightMaxBatch(1) bit for bit; episodes 0, 9 (the first past 2^31 elements) and 15 equal R.smnet_heightmax_frame.  Then a masked
    reset over the 16 M rows clears the selected slots and nothing else."""
    p = HMAX
    E, mw, mh, C, H, W, cell, T_ = p["E"], p["mw"], p["mh"], p["C"], p["H"], p["W"], p["cell"], p["frames"]
    n_cells = mw * mh
    sms = device_sms()
    assert 9 * n_cells * C >= I32_ELEMS > 8 * n_cells * C
    assert heightmax_reset_sweeps(E, n_cells, sms) > 1
    _need(E * n_cells * (C * 4 + 13) + (T_ + 1) * E * H * W * C * 4 + n_cells * (C * 4 + 13) + 5 * 1024 ** 3)
    L = eod._lib
    eps, Ts, shifts = _hmax_episodes(eod, E, T_, H, W, mw, mh, cell, seed=4321)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    sh = _t(shifts, cuda)
    depth = [_t(np.stack([ep.depth[t] for ep in eps]), cuda) for t in range(T_)]
    pose = [torch.stack([T[t, :3].reshape(12) for T in Ts]).to(cuda) for t in range(T_)]
    gen = torch.Generator(device=cuda).manual_seed(5)
    feats = [torch.randn((E, H, W, C), device=cuda, generator=gen) for _ in range(T_)]
    batch = eod.HeightMaxBatch(E, mw, mh, C, H, W, cuda, layout=L.LAYOUT_HWC)
    for t in range(T_):
        batch.step(feats[t], depth=depth[t], pose=pose[t], shifts=sh, intr=intr, cell=cell)
    torch.cuda.synchronize()
    assert int(batch.scratch.key64.abs().sum()) == 0 and int(batch.scratch.n_list.abs().sum()) == 0
    assert all(int(batch.observed[e].sum()) > 1000 for e in p["checked"] + HMAX_RESET)   # (two slots of the 16 look out of the map)

    alone = eod.HeightMaxBatch(1, mw, mh, C, H, W, cuda, layout=L.LAYOUT_HWC)
    for e in range(E):
        alone.reset()
        for t in range(T_):
            alone.step(feats[t][e:e + 1], depth=depth[t][e:e + 1], pose=pose[t][e:e + 1], shifts=sh[e:e + 1], intr=intr, cell=cell)
        torch.cuda.synchronize()
        assert torch.equal(_bits(batch.state[e]), _bits(alone.state[0])), e
        assert torch.equal(_bits(batch.height_map[e]), _bits(alone.height_map[0])) and torch.equal(batch.observed[e], alone.observed[0]), e
    del alone
    for e in p["checked"]:
        state, observed, hmap, _ = _hmax_oracle(eps[e], Ts[e], [f[e].cpu() for f in feats], intr, mw, mh, cell, C)
        assert torch.equal(batch.height_map[e].cpu(), hmap) and torch.equal(batch.observed[e].cpu().bool(), observed), e
        assert torch.equal(batch.state[e].cpu(), state), e
        del state
    del feats
    torch.cuda.empty_cache()

    before = {e: (batch.state[e].clone(), batch.height_map[e].clone(), batch.observed[e].clone()) for e in HMAX_KEEP}
    assert all(bool(batch.observed[e].any()) for e in HMAX_RESET)
    batch.reset(_mask(E, HMAX_RESET, cuda))
    torch.cuda.synchronize()
    for e in HMAX_RESET:
        assert not bool(batch.state[e].any()) and not bool(batch.height_map[e].any()) and not bool(batch.observed[e].any()), e
    for e, (s, h, o) in before.items():
        assert torch.equal(_bits(batch.state[e]), _bits(s)) and torch.equal(_bits(batch.height_map[e]), _bits(h)), e
        assert torch.equal(batch.observed[e], o), e


# ---- 5. height-max update past its pass size ----------------------------------------------------------------------------------
def test_heightmax_update_past_its_pass_size(eod, cuda):
    """E = 64 on a 501x499 map (cell count not a multiple of 32), C = 64, 2 frames through ops: some episode lists more cells in a frame
    than one pass of its blocks covers.  Every episode equals its E = 1 run bit for bit and the scratch is clean after every update;
    the linlayer update at this E is within 1e-5 of scale of the fp64 oracle on two episodes."""
    p = HLIST
    E, mw, mh, C, H, W, cell, T_ = p["E"], p["mw"], p["mh"], p["C"], p["H"], p["W"], p["cell"], p["frames"]
    n_cells = mw * mh
    assert n_cells % 32
    sms = device_sms()
    L, ops = eod._lib, eod.ops
    _need(E * n_cells * (p["lin_c"] * 4 + 13) + T_ * E * H * W * C * 4 + E * n_cells * 8 + 2 * 1024 ** 3)
    eps, Ts, shifts = _hmax_episodes(eod, E, T_, H, W, mw, mh, cell, seed=700, room_size=(12.0, 9.0))
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    sh = _t(shifts, cuda)
    depth = [_t(np.stack([ep.depth[t] for ep in eps]), cuda) for t in range(T_)]
    pose = [torch.stack([T[t, :3].reshape(12) for T in Ts]).to(cuda) for t in range(T_)]
    gen = torch.Generator(device=cuda).manual_seed(8)
    feats = [torch.randn((E, H, W, C), device=cuda, generator=gen) for _ in range(T_)]

    def clean(s):
        return int(s.key64.abs().sum()) == 0 and int(s.n_list.abs().sum()) == 0

    scratch = ops.HeightMaxScratch(E, n_cells, H * W, cuda)
    state = torch.zeros((E, n_cells, C), device=cuda)
    hmap = torch.zeros((E, n_cells), device=cuda)
    obs = torch.zeros((E, n_cells), dtype=torch.uint8, device=cuda)
    per_pass = heightmax_update_pass_cells(E, scratch.list_cap, sms)
    listed = []
    for t in range(T_):
        ops.heightmax_contest_depth(depth[t], pose[t], sh, intr, cell, mw, mh, scratch)
        listed.append(scratch.n_list[:, 0].cpu())
        ops.heightmax_update(feats[t], L.LAYOUT_HWC, scratch, hmap, obs, state)
        torch.cuda.synchronize()
        assert clean(scratch), t
    assert int(max(n.max() for n in listed)) > per_pass, per_pass

    s1 = ops.HeightMaxScratch(1, n_cells, H * W, cuda)
    st1, h1, o1 = torch.zeros((1, n_cells, C), device=cuda), torch.zeros((1, n_cells), device=cuda), torch.zeros((1, n_cells), dtype=torch.uint8, device=cuda)
    for e in range(E):
        st1.zero_(), h1.zero_(), o1.zero_()
        for t in range(T_):
            ops.heightmax_contest_depth(depth[t][e:e + 1], pose[t][e:e + 1], sh[e:e + 1], intr, cell, mw, mh, s1)
            ops.heightmax_update(feats[t][e:e + 1], L.LAYOUT_HWC, s1, h1, o1, st1)
        torch.cuda.synchronize()
        assert torch.equal(_bits(state[e]), _bits(st1[0])) and torch.equal(_bits(hmap[e]), _bits(h1[0])) and torch.equal(obs[e], o1[0]), e
    assert clean(s1)
    del state, st1, s1
    torch.cuda.empty_cache()

    # the same frame through the winner list + eod_linear_rows
    rng = np.random.default_rng(33)
    lin_w = (rng.standard_normal((p["lin_c"], C)) / 8).astype(np.float32)
    lin_b = rng.standard_normal(p["lin_c"]).astype(np.float32)
    lin = eod.HeightMaxBatch(E, mw, mh, C, H, W, cuda, layout=L.LAYOUT_HWC, linlayer=(_t(lin_w, cuda), _t(lin_b, cuda)))
    lin.step(feats[0], depth=depth[0], pose=pose[0], shifts=sh, intr=intr, cell=cell)
    torch.cuda.synchronize()
    assert clean(lin.scratch)
    for e in (int(listed[0].argmax()), E - 1):                   # the longest first-frame list, and the last slot
        ref, observed, href, m = _hmax_oracle(eps[e], Ts[e], [feats[0][e].cpu()], intr, mw, mh, cell, C,
                                              linlayer=(torch.from_numpy(lin_w).double(), torch.from_numpy(lin_b).double()), dtype=torch.float64)
        assert int(m.sum()) == int(listed[0][e]), e            # the first frame raises every cell it lists
        assert torch.equal(lin.height_map[e].cpu(), href) and torch.equal(lin.observed[e].cpu().bool(), observed), e
        got = lin.state[e].cpu().double()
        assert float((got[m] - ref[m]).abs().max()) <= 1e-5 * float(ref[m].abs().max()), e
        assert not bool(got[~m].any()), e


# ---- 6. reset, refresh and heightmax-reset sweeps through ops -----------------------------------------------------------------
def _sweep_state(cuda, seed):
    """Synthetic (E, 999*1001, 128) state: non-zero sums / fp16 rows everywhere, counts on ~2 % of the rows and around every episode
    boundary (where the 32-row chunks of a sweep straddle two episodes)."""
    E, N, C = SWEEP["E"], SWEEP["n_cells"], SWEEP["C"]
    gen = torch.Generator(device=cuda).manual_seed(seed)
    sums = torch.randn((E, N, C), device=cuda, generator=gen)
    norm16 = torch.randn((E, N, C), device=cuda, generator=gen).half()
    counts = torch.randint(1, 7, (E, N), device=cuda, generator=gen).float()
    keep = torch.rand((E, N), device=cuda, generator=gen) < 0.02
    keep[:, :40] = keep[:, -40:] = torch.rand((E, 40), device=cuda, generator=gen) < 0.5
    counts *= keep                                                 # count 0 with non-zero sums on the other rows: never touched
    return sums, counts, norm16


@pytest.mark.parametrize("mask", list(SWEEP_MASKS), ids=list(SWEEP_MASKS))
def test_reset_and_refresh_sweeps_vs_torch(eod, cuda, mask):
    """reset_episodes / refresh_norm16 (and reset_touched) over E * n_cells > the rows of one sweep, n_cells % 32 != 0: exactly the rows
    with a non-zero count of the selected slots change - cleared, or norm16 := half(sums / count where count > 1) - bit for bit as
    torch computes it on the device."""
    E, N, C = SWEEP["E"], SWEEP["n_cells"], SWEEP["C"]
    assert touched_rows_sweeps(E, N, device_sms()) > 2 and N % 32
    _need(E * N * C * 12 + E * N * 16)
    sums, counts, norm16 = _sweep_state(cuda, 3)
    m = _mask(E, [e for e, v in enumerate(SWEEP_MASKS[mask]) if v], cuda)
    hit = (counts != 0) & (m[:, None] != 0)
    assert int(hit.sum()) > 0 and int((hit[:, :40]).sum()) > 0

    n = norm16.clone()
    eod.ops.refresh_norm16(counts, sums, n, m)
    c = counts[..., None]
    exp = torch.where(hit[..., None], torch.where(c > 1, sums / c, sums).half(), norm16)
    torch.cuda.synchronize()
    assert torch.equal(_bits(n), _bits(exp))
    del n, exp

    s, cn, n = sums.clone(), counts.clone(), norm16.clone()
    eod.ops.reset_episodes(cn, s, n, m)
    torch.cuda.synchronize()
    assert torch.equal(cn, torch.where(hit, torch.zeros_like(counts), counts))
    assert torch.equal(_bits(s), _bits(torch.where(hit[..., None], torch.zeros_like(sums), sums)))
    assert torch.equal(_bits(n), _bits(torch.where(hit[..., None], torch.zeros_like(norm16), norm16)))
    if mask == "alternate":                                        # and the unmasked reset of the same state
        s.copy_(sums), cn.copy_(counts), n.copy_(norm16)
        eod.ops.reset_touched(cn, s, n)
        torch.cuda.synchronize()
        seen = counts != 0
        assert not bool(cn.any())
        assert torch.equal(_bits(s), _bits(torch.where(seen[..., None], torch.zeros_like(sums), sums)))
        assert torch.equal(_bits(n), _bits(torch.where(seen[..., None], torch.zeros_like(norm16), norm16)))


@pytest.mark.parametrize("mask", list(SWEEP_MASKS), ids=list(SWEEP_MASKS))
def test_heightmax_reset_sweep_vs_torch(eod, cuda, mask):
    """heightmax_reset over E * n_cells > the rows of one sweep: selected slots get height 0 and observed 0 on every row, and zero state
    rows where the cell was observed; state rows of unobserved cells and every row of the other slots are left alone."""
    E, N, C = SWEEP["E"], SWEEP["n_cells"], SWEEP["C"]
    assert heightmax_reset_sweeps(E, N, device_sms()) > 2 and N % 32
    _need(E * N * C * 8 + E * N * 32)
    gen = torch.Generator(device=cuda).manual_seed(4)
    state = torch.randn((E, N, C), device=cuda, generator=gen)
    hmap = torch.rand((E, N), device=cuda, generator=gen) + 999.0
    obs = (torch.rand((E, N), device=cuda, generator=gen) < 0.3).to(torch.uint8)
    obs[:, :40] = (torch.rand((E, 40), device=cuda, generator=gen) < 0.5).to(torch.uint8)
    sel = _mask(E, [e for e, v in enumerate(SWEEP_MASKS[mask]) if v], cuda)[:, None] != 0
    st, h, o = state.clone(), hmap.clone(), obs.clone()
    eod.ops.heightmax_reset(h, o, st, sel[:, 0].int())
    torch.cuda.synchronize()
    assert torch.equal(_bits(h), _bits(torch.where(sel, torch.zeros_like(hmap), hmap)))
    assert torch.equal(o, torch.where(sel, torch.zeros_like(obs), obs))
    assert torch.equal(_bits(st), _bits(torch.where((sel & (obs != 0))[..., None], torch.zeros_like(state), state)))
