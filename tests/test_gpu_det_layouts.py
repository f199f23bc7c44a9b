"""The deterministic write (eod_write_mean_det_layout) on channels-last features and with an active mask, and the runs of EpisodeRunner
it makes reproducible.

Every layout sums a run's sampled pixels in raster order from +0 (16-bit values widened exactly) and the segmented reduce does not look at
the layout, so the same features give the same bits in every layout: det(HWC x) == det(CHW x), det(HWC_BF16 x) == det(CHW x.float()),
on arbitrary inputs - not only on the exactly summable ones of tests/exact_cases.py.  Run on the B200 box with `-m gpu`."""
import math
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R

import exact_cases as X
import test_gpu_runner as TR

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5
CHW, HWC, HWC_BF16, HWC_F16, CHW_BF16, CHW_F16 = 0, 1, 2, 3, 4, 5
CHANNELS_LAST = {HWC: torch.float32, HWC_BF16: torch.bfloat16, HWC_F16: torch.float16}
LAYOUT_IDS = {CHW: "chw", HWC: "hwc", HWC_BF16: "hwc-bf16", HWC_F16: "hwc-f16"}


def _t(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t if dtype is None else t.to(dtype)


def _bits(t: torch.Tensor) -> torch.Tensor:
    t = t.detach().contiguous().cpu()
    return t.view({torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype])


def _same_bits(a: torch.Tensor, b: torch.Tensor, what) -> None:
    assert a.shape == b.shape and a.dtype == b.dtype, (what, a.shape, b.shape, a.dtype, b.dtype)
    bad = int((_bits(a) != _bits(b)).sum())
    assert bad == 0, (what, f"{bad} elements differ")


def _layout_feat(x_chw: torch.Tensor, layout: int) -> torch.Tensor:
    """(E,C,H,W) fp32 device features in ``layout``: channels-last ones permuted and cast to the layout's dtype."""
    if layout == CHW:
        return x_chw.contiguous()
    return x_chw.permute(0, 2, 3, 1).contiguous().to(CHANNELS_LAST[layout])


def _widened(x_chw: torch.Tensor, layout: int) -> torch.Tensor:
    """The fp32 CHW features whose det write must give the bits of ``_layout_feat(x_chw, layout)``."""
    return x_chw.to(CHANNELS_LAST.get(layout, torch.float32)).float().contiguous()


def _det(eod, cuda, feat, layout, idx, samp, sums0, active=None, runs_per_episode=None, ws=None):
    """frame_count -> write_mean_det on a copy of sums0: (sums, workspace)."""
    E, cells, C = sums0.shape
    HW = idx[0].numel()
    d_sums = sums0.clone()
    d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    ws = ws or eod.ops.DetWorkspace(E, C, HW, cells, cuda, HW if runs_per_episode is None else runs_per_episode)
    eod.ops.frame_count(idx, samp, d_cnt, active)
    eod.ops.write_mean_det(feat, idx, samp, d_cnt, d_sums, ws, layout=layout, active=active)
    torch.cuda.synchronize()
    return d_sums, ws


def _oracle_sums(feat_chw: np.ndarray, idx: np.ndarray, samp, sums0: np.ndarray) -> np.ndarray:
    cells = sums0.shape[0]
    s, n = oracle.cell_sums_seq(feat_chw, idx, samp, cells)
    return sums0 + np.where(n[:, None] > 0, s / np.maximum(n, 1)[:, None].astype(np.float32), 0).astype(np.float32)


def _within(got: torch.Tensor, ref: np.ndarray, what) -> None:
    err = float(np.abs(got.cpu().numpy() - ref).max())
    assert err <= SUM_TOL * float(np.abs(ref).max()), (what, err)


# ------------------------------------------------------------------------------------------------------------------------------
# 1. the same bits in every layout, on standard-normal features
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_samp", [False, True], ids=["dense", "sampled"])
@pytest.mark.parametrize("C", [128, 256, 512])
def test_det_layouts_give_the_bits_of_chw(eod, cuda, C, with_samp):
    """Cell 7 of episode 0 has > 256 runs (chunked reduce), cell 9 of episode 1 > 2048 (bitmap sort); the rest is blocky with noise."""
    rng = np.random.default_rng(900 + C + with_samp)
    E, H, W, cells = 2, 64, 128, 300
    idx = rng.integers(10, cells, (E, H // 4 + 1, W // 8 + 1)).repeat(4, 1).repeat(8, 2)[:, :H, :W].astype(np.int32)
    idx[:, ::3, ::5] = rng.integers(10, cells, idx[:, ::3, ::5].shape)
    idx[0, :24, ::4] = 7                                                    # 768 isolated pixels: 768 runs
    idx[1, :56, ::2] = 9                                                    # 3584 runs (fewer than HW in all: the workspace holds them)
    samp = (rng.random((E, H, W)) < 0.8).astype(np.uint8) if with_samp else None
    runs = lambda e, c: int(sum(((idx[e].reshape(-1) == c) & np.r_[True, np.diff(idx[e].reshape(-1)) != 0]
                                 & ((samp[e].reshape(-1) > 0) if with_samp else True))))
    assert runs(0, 7) > 256 and runs(1, 9) > 2048
    x = torch.randn((E, C, H, W), device=cuda, generator=torch.Generator(device=cuda).manual_seed(C))
    sums0 = torch.randn((E, cells, C), device=cuda, generator=torch.Generator(device=cuda).manual_seed(C + 1))
    d_idx, d_samp = _t(idx, cuda), (None if samp is None else _t(samp, cuda))
    ref_chw = {}
    for layout in (HWC, HWC_BF16, HWC_F16):
        xw = _widened(x, layout)
        key = CHANNELS_LAST[layout]
        if key not in ref_chw:
            ref_chw[key], ws = _det(eod, cuda, xw, CHW, d_idx, d_samp, sums0)
            assert not ws.overflowed()
            for e in range(E):
                _within(ref_chw[key][e], _oracle_sums(xw[e].cpu().numpy(), idx[e], None if samp is None else samp[e], sums0[e].cpu().numpy()),
                        (LAYOUT_IDS[layout], e))
        got, ws = _det(eod, cuda, _layout_feat(x, layout), layout, d_idx, d_samp, sums0)
        assert not ws.overflowed()
        _same_bits(got, ref_chw[key], LAYOUT_IDS[layout])


# ------------------------------------------------------------------------------------------------------------------------------
# 2. exactly summable inputs: sums, counts, touched cells and the fp16 table equal the float64 reference bit for bit
# ------------------------------------------------------------------------------------------------------------------------------
def _exact32(ref64: np.ndarray) -> torch.Tensor:
    r32 = np.asarray(ref64).astype(np.float32)
    assert np.array_equal(r32.astype(np.float64), ref64), "the reference is not an fp32 number: the case is not exactly summable"
    return torch.from_numpy(r32)


@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("layout", [HWC, HWC_BF16, HWC_F16, CHW], ids=lambda l: LAYOUT_IDS[l])
def test_det_exact_lattice(eod, cuda, layout, C):
    """E=3 at 96x128 (the case of test_mean_write_exact_e3): dense, then sampled with an active mask that idles a slot."""
    rng = np.random.default_rng(300 + 4 * C + layout)
    E, H, W, cells = 3, 96, 128, 2700
    for samp_p, active in ((None, None), (0.3, np.array([1, 0, 2], np.int32))):
        samp = None
        if samp_p is not None:
            samp = rng.random((E, H, W)) < samp_p
            samp[0, : H // 3] = False
        idx = np.stack([X.index_plane(rng, H, W, cells, None if samp is None else samp[e], 6) for e in range(E)])
        feat = X.dyadic(rng, (E, C, H, W), 3, 3)                            # 4 significant bits: exact in bf16 and fp16
        n_max = max(int(X.sample_counts(idx[e], None if samp is None else samp[e], cells).max()) for e in range(E))
        q = 3 + int(math.log2(n_max))
        sums0 = X.dyadic(rng, (E, cells, C), 20, q)
        counts0 = rng.integers(0, 4, (E, cells)).astype(np.float32)
        d_idx = _t(idx, cuda)
        d_samp = None if samp is None else _t(samp.astype(np.uint8), cuda)
        d_act = None if active is None else _t(active, cuda)
        d_sums, d_counts = _t(sums0, cuda), _t(counts0, cuda)
        d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
        d_touched = torch.zeros((E, cells), dtype=torch.uint8, device=cuda)
        d_norm = torch.zeros((E, cells, C), dtype=torch.float16, device=cuda)
        ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda, H * W)
        eod.ops.frame_count(d_idx, d_samp, d_cnt, d_act)
        eod.ops.write_mean_det(_layout_feat(_t(feat, cuda), layout), d_idx, d_samp, d_cnt, d_sums, ws, layout=layout, active=d_act)
        eod.ops.finalize_counts(d_idx, d_cnt, d_counts, d_touched, d_sums, d_norm)
        torch.cuda.synchronize()
        assert not ws.overflowed() and int(d_cnt.abs().sum()) == 0
        for e in range(E):
            live = active is None or active[e] > 0
            se = None if samp is None else samp[e]
            ref, bound, n = X.mean_write_f64(sums0[e], feat[e], idx[e], se, cells)
            X.assert_pow2_counts(n)
            X.check_lattice([feat[e], sums0[e], ref], q, bound)
            if not live:
                ref, n = sums0[e].astype(np.float64), np.zeros(cells, np.int64)
            _same_bits(d_sums[e], _exact32(ref), (e, "sums"))
            vis = np.zeros(cells, bool)
            if live:
                vis[np.unique(idx[e])] = True
            counts = counts0[e] + vis
            assert np.array_equal(d_counts[e].cpu().numpy(), counts), (e, "counts")
            assert np.array_equal(d_touched[e].cpu().numpy().astype(bool), n > 0), (e, "touched")
            want16 = torch.where(torch.from_numpy(vis)[:, None], R.create_implicit_memory(_exact32(ref), torch.from_numpy(counts)).half(),
                                 torch.zeros((), dtype=torch.float16))
            _same_bits(d_norm[e], want16, (e, "norm16"))


# ------------------------------------------------------------------------------------------------------------------------------
# 3. active mask: idle slots untouched (their NaN slabs unread), the others as in a batch of their own
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", [CHW, HWC, HWC_BF16, HWC_F16], ids=lambda l: LAYOUT_IDS[l])
def test_det_active_mask(eod, cuda, layout):
    rng = np.random.default_rng(40 + layout)
    E, C, H, W, cells = 4, 128, 64, 96, 500
    active = np.array([1, 0, 2, 0], np.int32)
    idx = rng.integers(0, cells, (E, H // 2, W // 4)).repeat(2, 1).repeat(4, 2).astype(np.int32)
    samp = (rng.random((E, H, W)) < 0.6).astype(np.uint8)
    x = torch.randn((E, C, H, W), device=cuda, generator=torch.Generator(device=cuda).manual_seed(layout))
    x[torch.from_numpy(active <= 0).to(cuda)] = float("nan")
    sums0 = torch.randn((E, cells, C), device=cuda)
    counts0 = _t(rng.integers(0, 3, (E, cells)).astype(np.float32), cuda)
    norm0 = R.create_implicit_memory(sums0.cpu().reshape(-1, C), counts0.cpu().reshape(-1)).half().reshape(E, cells, C).to(cuda)

    def frame(sel, act):
        sel = list(sel)
        d_idx, d_samp = _t(idx[sel], cuda), _t(samp[sel], cuda)
        d_sums, d_counts, d_norm = sums0[sel].clone(), counts0[sel].clone(), norm0[sel].clone()
        d_cnt = torch.zeros((len(sel), cells), dtype=torch.int32, device=cuda)
        d_act = None if act is None else _t(act, cuda)
        ws = eod.ops.DetWorkspace(len(sel), C, H * W, cells, cuda, H * W)
        eod.ops.frame_count(d_idx, d_samp, d_cnt, d_act)
        eod.ops.write_mean_det(_layout_feat(x[sel], layout), d_idx, d_samp, d_cnt, d_sums, ws, layout=layout, active=d_act)
        eod.ops.finalize_counts(d_idx, d_cnt, d_counts, None, d_sums, d_norm)
        torch.cuda.synchronize()
        assert not ws.overflowed() and int(d_cnt.abs().sum()) == 0, "frame_cnt is not back to zero"
        return d_sums, d_counts, d_norm

    masked = frame(range(E), active)
    alone = frame([0, 2], None)
    for k, name in enumerate(("sums", "counts", "norm16")):
        ref = (sums0, counts0, norm0)[k]
        for e in (1, 3):
            _same_bits(masked[k][e], ref[e], (e, name, "idle slot changed"))
        for j, e in enumerate((0, 2)):
            _same_bits(masked[k][e], alone[k][j], (e, name))
    assert bool(torch.isfinite(masked[0]).all())


# ------------------------------------------------------------------------------------------------------------------------------
# 4. 480x640 channels-last: run to run, another batching, and an undersized workspace
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", [HWC, HWC_BF16], ids=lambda l: LAYOUT_IDS[l])
def test_det_channels_last_reproducible_full_frame(eod, cuda, layout):
    rng = np.random.default_rng(480 + layout)
    E, C, H, W, cells = 3, 128, 480, 640, 4000
    idx = rng.integers(0, cells, (E, H // 8, W // 16)).repeat(8, 1).repeat(16, 2).astype(np.int32)
    idx[:, ::7, ::3] = rng.integers(0, cells, idx[:, ::7, ::3].shape)      # noisy depth: short runs inside the blocks
    samp = (rng.random((E, H, W)) < 0.5).astype(np.uint8)
    x = torch.randn((E, C, H, W), device=cuda, generator=torch.Generator(device=cuda).manual_seed(7))
    sums0 = torch.randn((E, cells, C), device=cuda)
    d_idx, d_samp = _t(idx, cuda), _t(samp, cuda)
    feat = _layout_feat(x, layout)
    a, ws = _det(eod, cuda, feat, layout, d_idx, d_samp, sums0)
    assert not ws.overflowed()
    b, _ = _det(eod, cuda, feat, layout, d_idx, d_samp, sums0, ws=ws)     # the workspace as the first call left it
    _same_bits(a, b, "run to run")
    order = [2, 0, 1]
    c, _ = _det(eod, cuda, feat[order].contiguous(), layout, d_idx[order].contiguous(), d_samp[order].contiguous(), sums0[order].contiguous())
    _same_bits(a, c[np.argsort(order)], "batch order")
    small, ws = _det(eod, cuda, feat, layout, d_idx, d_samp, sums0, runs_per_episode=64)
    assert ws.overflowed()
    xw = _widened(x, layout).cpu().numpy()
    for e in range(E):
        ref = _oracle_sums(xw[e], idx[e], samp[e], sums0[e].cpu().numpy())
        _within(a[e], ref, (e, "det"))
        _within(small[e], ref, (e, "overflowed"))


# ------------------------------------------------------------------------------------------------------------------------------
# 5. EpisodeBatch(variant=WRITE_DET) on channels-last features, ragged masks, both stream modes
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pipeline", [False, True], ids=["ordered", "pipelined"])
@pytest.mark.parametrize("layout", [HWC, HWC_BF16], ids=lambda l: LAYOUT_IDS[l])
def test_episode_batch_det_channels_last(eod, cuda, layout, pipeline):
    """step(active=, reset_mask=, refresh_mask=) on a channels-last WRITE_DET batch is bit-identical - levels of every frame, sums,
    counts, norm16 - to a serial CHW WRITE_DET twin fed the same (widened) features; idle slots hold NaN features."""
    E, C, H, W, mw, mh = 3, 128, 96, 128, 60, 45
    cells = mw * mh
    rng = np.random.default_rng(70 + 2 * layout + pipeline)
    lib = eod._lib
    a = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, layout=layout, variant=lib.WRITE_DET, pipeline=pipeline)
    b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, layout=CHW, variant=lib.WRITE_DET, pipeline=False)
    for x in (a, b):
        x.det_runs_per_episode = H * W
        x.read_frozen = pipeline                                           # longterm snapshot read in the pipelined case
    depth, pose, shifts = torch.zeros((E, H, W), device=cuda), torch.zeros((E, 12), device=cuda), torch.zeros((E, 6), device=cuda)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    plan = [dict(), dict(samp=0.4, active=[1, 0, 1]), dict(reset=[0, 1, 0], active=[1, 1, 0]), dict(refresh=[1, 0, 1]),
            dict(samp=0.3, active=[0, 2, 1], reset=[1, 0, 0], refresh=[1, 1, 0])]
    gen = torch.Generator(device=cuda).manual_seed(5)
    for t, p in enumerate(plan):
        samp = _t((rng.random((E, H, W)) < p["samp"]).astype(np.uint8), cuda) if "samp" in p else None
        idx = _t(rng.integers(0, cells, (E, H // 2, W // 4)).repeat(2, 1).repeat(4, 2).astype(np.int32), cuda)
        x = torch.randn((E, C, H, W), device=cuda, generator=gen)
        kw = dict(proj_indices=idx)
        for key in ("active", "reset", "refresh"):
            if key in p:
                kw[key if key == "active" else key + "_mask"] = _t(np.array(p[key], np.int32), cuda)
        if "active" in p:
            x[_t(np.array(p["active"]) <= 0, cuda)] = float("nan")
        la = [l.clone() for l in a.step(depth, pose, shifts, intr, 0.2, _layout_feat(x, layout), samp, inputs_ready=False, **kw)]
        lb = [l.clone() for l in b.step(depth, pose, shifts, intr, 0.2, _widened(x, layout), samp, **kw)]
        for k in range(3):
            _same_bits(la[k], lb[k], (t, "level", k))
    a.join(), b.join()
    torch.cuda.synchronize()
    assert not a._det_ws.overflowed() and not b._det_ws.overflowed()
    _same_bits(a.sums, b.sums, "sums")
    _same_bits(a.counts, b.counts, "counts")
    _same_bits(a.norm16, b.norm16, "norm16")
    assert bool(torch.isfinite(a.sums).all()) and float(a.counts.max()) >= 3


def test_episode_batch_det_refuses_16bit_chw_only(eod, cuda):
    lib = eod._lib
    for layout in (CHW_BF16, CHW_F16):
        with pytest.raises(eod.EodError, match="WRITE_DET"):
            eod.EpisodeBatch(2, 10, 5, 128, 8, 64, cuda, layout=layout, variant=lib.WRITE_DET)
    for layout in (CHW, HWC, HWC_BF16, HWC_F16):
        eod.EpisodeBatch(2, 10, 5, 128, 8, 64, cuda, layout=layout, variant=lib.WRITE_DET)


# ------------------------------------------------------------------------------------------------------------------------------
# 6. EpisodeRunner(variant=WRITE_DET): the same bits whatever the slots and waves
# ------------------------------------------------------------------------------------------------------------------------------
def _bf16_exact(episodes):
    """The dataset with every frame's features rounded to bf16 (kept in fp32): the oracle then sees the values the bf16 run writes."""
    return [[dict(fr, feat=torch.from_numpy(fr["feat"]).to(torch.bfloat16).float().numpy()) for fr in ep] for ep in episodes]


def _runner_episodes(episodes, layout):
    """Frames as the runner's provider takes them: (C,H,W) for CHW, (H,W,C) for the channels-last layouts."""
    if layout == CHW:
        return episodes
    return [[dict(fr, feat=np.ascontiguousarray(fr["feat"].transpose(1, 2, 0))) for fr in ep] for ep in episodes]


def _run(eod, cuda, episodes, shifts, intr, test_type, layout, n_slots, save_dir):
    provider = eod.HostEpisodeProvider(_runner_episodes(episodes, layout), cuda, shifts, feat_dtype=CHANNELS_LAST.get(layout, torch.float32))
    runner = eod.EpisodeRunner(provider, TR.MW, TR.MH, TR.C, n_slots=n_slots, height=TR.H, width=TR.W, device=cuda, test_type=test_type,
                               intr=intr, cell=TR.CELL, layout=layout, variant=eod._lib.WRITE_DET, save_dir=save_dir)
    runner.batch.det_runs_per_episode = TR.H * TR.W
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


def _solo(eod, cuda, episodes, shifts, intr, test_type, layout):
    """Every episode replayed one frame at a time through EpisodeBatch(E=1, WRITE_DET), in dataset order."""
    batch = eod.EpisodeBatch(1, TR.MW, TR.MH, TR.C, TR.H, TR.W, cuda, layout=layout, variant=eod._lib.WRITE_DET)
    batch.det_runs_per_episode = TR.H * TR.W
    batch.read_frozen = test_type == "longterm"
    one = torch.ones((1,), dtype=torch.int32, device=cuda)
    levels, saved = {}, {}
    for e, ep in enumerate(_runner_episodes(episodes, layout)):
        for i, fr in enumerate(ep):
            kw = {}
            if fr["memory_reset"] or (e == 0 and i == 0):
                kw["reset_mask"] = one
            if batch.read_frozen and (i == 0 or "reset_mask" in kw):
                kw["refresh_mask"] = one
            if "proj_indices" in fr:
                kw["proj_indices"] = _t(fr["proj_indices"][..., 0], cuda)[None]
                depth = pose = sh = None
            else:
                depth, pose = _t(fr["depth"], cuda)[None], _t(fr["pose"], cuda)[None]
                sh = _t(shifts[e], cuda)[None]
            feat = _t(fr["feat"], cuda, CHANNELS_LAST.get(layout, torch.float32))[None]
            lv = batch.step(depth, pose, sh, intr, TR.CELL, feat, **kw)
            levels[(e, i)] = [l[0].clone() for l in lv]
            if i == 0:
                batch.join()
                saved[os.path.splitext(fr["sequence_name"])[0]] = (batch.sums[0].cpu().numpy(), batch.counts[0].cpu().numpy())
    batch.join()
    torch.cuda.synchronize()
    assert not batch._det_ws.overflowed()
    return levels, saved


@pytest.mark.parametrize("layout", [CHW, HWC_BF16], ids=lambda l: LAYOUT_IDS[l])
@pytest.mark.parametrize("test_type,regime", [("default", "dense-idx"), ("episodic", "dense-depth"), ("longterm", "dense-idx")])
def test_runner_det_is_reproducible_across_slots_and_waves(eod, cuda, tmp_path, test_type, regime, layout):
    episodes, shifts, intr = TR._dataset(eod, test_type, regime)
    if layout == HWC_BF16:
        episodes = _bf16_exact(episodes)
    runs = [_run(eod, cuda, episodes, shifts, intr, test_type, layout, n, str(tmp_path / f"run{k}")) for k, n in enumerate((2, 2, 3))]
    solo_levels, solo_saved = _solo(eod, cuda, episodes, shifts, intr, test_type, layout)
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
    ref_levels, ref_saved = TR._oracle_serial(episodes, test_type, regime)
    for key, lv in got0.items():
        for k in range(3):
            a, b = lv[k].float().cpu(), ref_levels[key][k][0].float()
            tol = 2e-3 * max(1.0, float(b.abs().max()))
            assert torch.allclose(a, b, rtol=2e-3, atol=tol), (key, k, float((a - b).abs().max()))
    for name, (s_ref, c_ref) in ref_saved.items():
        mem, obs = saved0[os.path.splitext(name)[0]]
        assert np.array_equal(obs, c_ref.numpy()), name
        assert np.abs(mem - s_ref.numpy()).max() <= SUM_TOL * max(float(s_ref.abs().max()), 1e-30), name


def test_runner_det_refuses_the_detection_regime(eod, cuda):
    episodes, shifts, intr = TR._dataset(eod, "default", "detections")
    runner = eod.EpisodeRunner(eod.HostEpisodeProvider(episodes, cuda, shifts, k_max=8), TR.MW, TR.MH, TR.C, n_slots=2, height=TR.H,
                               width=TR.W, device=cuda, intr=intr, cell=TR.CELL, variant=eod._lib.WRITE_DET)
    with pytest.raises(eod.EodError, match="not deterministic"):
        runner.run()


# ------------------------------------------------------------------------------------------------------------------------------
# 7. refusals
# ------------------------------------------------------------------------------------------------------------------------------
def test_det_refusals(eod, cuda):
    E, C, H, W, cells = 1, 128, 8, 64, 50
    idx = torch.zeros((E, H, W), dtype=torch.int32, device=cuda)
    sums = torch.zeros((E, cells, C), device=cuda)
    cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda)
    eod.ops.frame_count(idx, None, cnt)
    for layout, dtype in ((CHW_BF16, torch.bfloat16), (CHW_F16, torch.float16)):
        with pytest.raises(eod.EodError, match="16-bit CHW"):
            eod.ops.write_mean_det(torch.zeros((E, C, H, W), dtype=dtype, device=cuda), idx, None, cnt, sums, ws, layout=layout)
    for layout, wrong in ((HWC_BF16, torch.float32), (HWC_F16, torch.bfloat16), (HWC, torch.float16), (CHW, torch.bfloat16)):
        with pytest.raises(TypeError):
            eod.ops.write_mean_det(torch.zeros((E, H, W, C), dtype=wrong, device=cuda), idx, None, cnt, sums, ws, layout=layout)
    H2, W2 = 30, 52                                                         # HW % 32 != 0
    idx2 = torch.zeros((E, H2, W2), dtype=torch.int32, device=cuda)
    ws2 = eod.ops.DetWorkspace(E, C, H2 * W2, cells, cuda)
    for layout in (CHW, HWC, HWC_BF16):
        f = torch.zeros((E, H2, W2, C), dtype=CHANNELS_LAST.get(layout, torch.float32), device=cuda)
        with pytest.raises(eod.EodError, match="HW % 32"):
            eod.ops.write_mean_det(f, idx2, None, cnt, sums, ws2, layout=layout)
    assert not sums.any()
