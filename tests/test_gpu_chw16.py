"""bf16 / fp16 CHW features in the dense mean write (EOD_LAYOUT_CHW_BF16 / _CHW_F16): the 64-pixel TMA ring and the LDG kernel
against the oracle and against the fp32 CHW write on the widened features, idle slots, graph capture (static partition),
EpisodeBatch.step with late features, the reference-facing SpatialFeatureMemory methods, EpisodeRunner over 16-bit providers, and
the refusals.  The 16-bit values are widened exactly, so on exactly summable inputs (tests/exact_cases.py: 4 significant bits,
representable in bf16 and fp16) every result equals the float64 reference - and the fp32 kernel - bit for bit.
Run on the B200 box with `-m gpu`."""
import math

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R

import exact_cases as X

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5          # max|a-b| <= SUM_TOL * max|ref|
LAYOUTS = {"bf16": (4, torch.bfloat16), "f16": (5, torch.float16)}       # EOD_LAYOUT_CHW_BF16, EOD_LAYOUT_CHW_F16
AUTO, LDG, TMA = 0, 1, 2


def _t(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t if dtype is None else t.to(dtype)


def _bits(t):
    t = t.detach().contiguous().cpu()
    return t.view({torch.float32: torch.int32, torch.float16: torch.int16}[t.dtype])


def _same_bits(got, ref, what):
    g, r = _bits(got), _bits(ref)
    assert g.shape == r.shape, (what, g.shape, r.shape)
    bad = int((g != r).sum())
    assert bad == 0, (what, f"{bad} elements differ")


def _exact32(ref64):
    r32 = np.asarray(ref64).astype(np.float32)
    assert np.array_equal(r32.astype(np.float64), ref64), "the reference is not an fp32 number: the case is not exactly summable"
    return torch.from_numpy(r32)


def _write(eod, cuda, f_dev, layout, variant, idx, samp, sums0, counts0, active=None):
    """frame_count -> write_mean -> finalize_counts (with the fp16 table) on fresh copies of the state."""
    E, cells = sums0.shape[:2]
    C = sums0.shape[2]
    d_idx = _t(idx, cuda)
    d_samp = None if samp is None else _t(samp.astype(np.uint8), cuda)
    d_sums, d_counts = _t(sums0, cuda), _t(counts0, cuda)
    d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    d_touched = torch.zeros((E, cells), dtype=torch.uint8, device=cuda)
    d_norm = torch.zeros((E, cells, C), dtype=torch.float16, device=cuda)
    d_act = None if active is None else _t(active, cuda)
    eod.ops.frame_count(d_idx, d_samp, d_cnt, d_act)
    eod.ops.write_mean(f_dev, d_idx, d_samp, d_cnt, d_sums, layout, variant, None, d_act)
    eod.ops.finalize_counts(d_idx, d_cnt, d_counts, d_touched, d_sums, d_norm)
    torch.cuda.synchronize()
    assert int(d_cnt.abs().sum()) == 0, "frame_cnt is not back to zero"
    return d_sums, d_counts, d_touched, d_norm


# ------------------------------------------------------------------------------------------------------------------------------
# 1  oracle parity: both 16-bit layouts, C = 128 / 256 / 512, TMA and LDG explicitly, and a shape only the LDG kernel takes
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_samp", [False, True], ids=["dense", "samp"])
@pytest.mark.parametrize("shape,variant", [((64, 96), LDG), ((64, 96), TMA), ((24, 30), AUTO), ((24, 30), LDG)],
                         ids=["tma-shape-ldg", "tma-shape-tma", "ldg-shape-auto", "ldg-shape-ldg"])
@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("kind", list(LAYOUTS))
def test_chw16_write_vs_oracle(eod, cuda, kind, C, shape, variant, with_samp):
    """Counts, visibility and touched sets exact; refreshed fp16 rows bit-exact; untouched cells unchanged; sums within SUM_TOL of
    scale of the sequential fp32 oracle on the widened features.  24x30 = 720 pixels: HW % 64 != 0, HW % 8 == 0."""
    layout, dtype = LAYOUTS[kind]
    (H, W), E, cells = shape, 3, 200
    rng = np.random.default_rng(C + 7 * variant + H + with_samp)
    f16 = torch.from_numpy(rng.standard_normal((E, C, H * W)).astype(np.float32)).to(dtype)
    feat = f16.float().numpy()                                               # the widened features: what the write must sum
    idx = rng.integers(0, cells, (E, H // 2 + 1, W // 4 + 1)).repeat(2, 1).repeat(4, 2)[:, :H, :W].reshape(E, H * W).astype(np.int32)
    idx[:, ::11] = rng.integers(0, cells, idx[:, ::11].shape)               # isolated pixels: groups that are not runs
    samp = (rng.random((E, H * W)) < 0.4) if with_samp else None
    sums0 = rng.standard_normal((E, cells, C)).astype(np.float32)
    counts0 = rng.integers(0, 3, (E, cells)).astype(np.float32)
    d_sums, d_counts, d_touched, d_norm = _write(eod, cuda, f16.to(cuda), layout, variant, idx, samp, sums0, counts0)
    for e in range(E):
        s, n = oracle.cell_sums_seq(feat[e].reshape(C, H, W), idx[e].reshape(H, W), None if samp is None else samp[e].reshape(H, W), cells)
        ref = sums0[e] + np.where(n[:, None] > 0, s / np.maximum(n, 1)[:, None].astype(np.float32), 0).astype(np.float32)
        got = d_sums[e].cpu().numpy()
        assert np.abs(got - ref).max() <= SUM_TOL * np.abs(ref).max(), (e, np.abs(got - ref).max())
        assert np.array_equal(got[n == 0], sums0[e][n == 0])                # cells without samples are not written at all
        vis = np.zeros(cells, np.float32)
        vis[np.unique(idx[e])] = 1
        assert np.array_equal(d_counts[e].cpu().numpy(), counts0[e] + vis)
        assert np.array_equal(d_touched[e].cpu().numpy().astype(bool), n > 0)
        ref16 = R.create_implicit_memory(d_sums[e].cpu(), d_counts[e].cpu()).half().numpy()
        got16 = d_norm[e].cpu().numpy()
        v = vis.astype(bool)
        assert np.array_equal(got16[v].view(np.uint16), ref16[v].view(np.uint16))
        assert not got16[~v].any()


# ------------------------------------------------------------------------------------------------------------------------------
# 2 + 3  exactly summable inputs: float64 reference and the fp32 kernel on feat.float(), bit for bit; idle slots bit-identical
# ------------------------------------------------------------------------------------------------------------------------------
def _exact_case(rng, E, H, W, cells, C, samp_p, big=None):
    samp = None
    if samp_p is not None:
        samp = rng.random((E, H, W)) < samp_p
        samp[0, : H // 3] = False                                            # whole tiles without a sample
    idx = np.stack([X.index_plane(rng, H, W, cells, None if samp is None else samp[e], 6 if big is None else 12, big) for e in range(E)])
    feat = X.dyadic(rng, (E, C, H, W), 3, 3)                                 # 4 significant bits: exact in bf16 and fp16
    n_max = max(int(X.sample_counts(idx[e], None if samp is None else samp[e], cells).max()) for e in range(E))
    q = 3 + int(math.log2(n_max))
    sums0 = X.dyadic(rng, (E, cells, C), 20, q)
    counts0 = rng.integers(0, 4, (E, cells)).astype(np.float32)
    return feat, idx, samp, sums0, counts0, q


def _check_exact(eod, cuda, kind, variant, feat, idx, samp, sums0, counts0, q, active=None):
    layout, dtype = LAYOUTS[kind]
    E, C, H, W = feat.shape
    cells = sums0.shape[1]
    f16 = _t(feat.reshape(E, C, H * W), cuda, dtype)
    f32 = f16.float()
    assert torch.equal(f32.cpu(), torch.from_numpy(feat.reshape(E, C, H * W)))    # the case is representable in 16 bits
    if active is not None:
        for e in range(E):
            if active[e] <= 0:                                               # an idle slot's features must not even be read
                f16[e] = float("nan")
                f32[e] = float("nan")
    idx2 = idx.reshape(E, H * W)
    samp2 = None if samp is None else samp.reshape(E, H * W)
    got = _write(eod, cuda, f16, layout, variant, idx2, samp2, sums0, counts0, active)
    twin = _write(eod, cuda, f32, 0, variant, idx2, samp2, sums0, counts0, active)            # fp32 CHW kernel, same variant
    for name, a, b in zip(("sums", "counts", "touched", "norm16"), got, twin):
        if a.dtype == torch.uint8:
            assert torch.equal(a, b), (kind, name)
        else:
            _same_bits(a, b.cpu(), (kind, variant, name, "vs fp32 kernel"))
    for e in range(E):
        live = active is None or active[e] > 0
        se = None if samp is None else samp[e]
        ref, bound, n = X.mean_write_f64(sums0[e], feat[e], idx[e], se, cells)
        X.assert_pow2_counts(n)
        X.check_lattice([feat[e], sums0[e], ref], q, bound)
        if not live:
            ref = sums0[e].astype(np.float64)
        _same_bits(got[0][e], _exact32(ref), (kind, variant, e, "sums"))
        vis = np.zeros(cells, np.float32)
        if live:
            vis[np.unique(idx[e])] = 1
        assert np.array_equal(got[1][e].cpu().numpy(), counts0[e] + vis), (kind, e, "counts")
        if not live:
            assert not got[2][e].any() and not got[3][e].any(), (kind, e, "idle slot touched")


@pytest.mark.parametrize("variant", [LDG, TMA], ids=["ldg", "tma"])
@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("kind", list(LAYOUTS))
def test_chw16_write_exact(eod, cuda, kind, C, variant):
    """E=3 at 96x128: dense, and sampled with an active mask that idles a slot (NaN features there); dyadic initial sums."""
    rng = np.random.default_rng(100 + C + variant + len(kind))
    for samp_p, active in ((None, None), (0.3, np.array([1, 0, 2], np.int32))):
        feat, idx, samp, sums0, counts0, q = _exact_case(rng, 3, 96, 128, 2700, C, samp_p)
        _check_exact(eod, cuda, kind, variant, feat, idx, samp, sums0, counts0, q, active)


@pytest.mark.parametrize("kind", list(LAYOUTS))
def test_chw16_write_exact_ragged_and_big_cell(eod, cuda, kind):
    """30x52 (HW % 64 != 0: AUTO takes the LDG kernel) with an idle slot, and 480x640 with one cell of 2^18 pixels on the TMA ring."""
    rng = np.random.default_rng(200 + len(kind))
    feat, idx, samp, sums0, counts0, q = _exact_case(rng, 2, 30, 52, 800, 256, 0.5)
    _check_exact(eod, cuda, kind, AUTO, feat, idx, samp, sums0, counts0, q, np.array([2, 0], np.int32))
    feat, idx, samp, sums0, counts0, q = _exact_case(rng, 1, 480, 640, 4000, 256, None, big=1 << 18)
    _check_exact(eod, cuda, kind, TMA, feat, idx, samp, sums0, counts0, q)


@pytest.mark.parametrize("with_active", [False, True], ids=["all", "active"])
@pytest.mark.parametrize("H_,W_,E_", [(8, 72, 1), (64, 96, 3), (480, 640, 2)])
def test_chw16_tma_write_static_partition_in_a_graph(eod, cuda, H_, W_, E_, with_active):
    """frame_count -> write_mean(CHW bf16, TMA) -> finalize_counts captured in a CUDA graph after an eager (ticketed) launch, then
    replayed (static partition).  8x72: 9 tiles of 64 pixels (odd: pairs of tiles fall back to single tiles).  On exact inputs the
    replay equals the eager launch and the float64 reference bit for bit; idle slots untouched."""
    ops, lib = eod.ops, eod._lib
    C = 256
    rng = np.random.default_rng(H_ * W_ + E_ + with_active)
    cells = max(400, H_ * W_ // 8)                                            # room for every power-of-two group
    act_l = [0 if (with_active and e % 2) else 1 for e in range(E_)]
    act = _t(np.array(act_l, np.int32), cuda) if with_active else None
    feat, idx, _, sums0, counts0, q = _exact_case(rng, E_, H_, W_, cells, C, None)
    f = _t(feat.reshape(E_, C, H_ * W_), cuda, torch.bfloat16)
    for e in range(E_):
        if not act_l[e]:
            f[e] = float("nan")
    d_idx = _t(idx.reshape(E_, -1), cuda)

    def state():
        return (_t(sums0, cuda), _t(counts0, cuda), torch.zeros((E_, cells), dtype=torch.int32, device=cuda),
                torch.zeros((E_, cells), dtype=torch.uint8, device=cuda))

    def frame(st):
        sums, counts, cnt, touched = st
        ops.frame_count(d_idx, None, cnt, act)
        ops.write_mean(f, d_idx, None, cnt, sums, lib.LAYOUT_CHW_BF16, lib.WRITE_TMA, None, act)
        ops.finalize_counts(d_idx, cnt, counts, touched)

    eager = state()
    frame(eager)
    torch.cuda.synchronize()
    replayed = state()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        frame(replayed)
    torch.cuda.synchronize()
    assert torch.equal(replayed[0].cpu(), torch.from_numpy(sums0))            # capturing ran nothing
    graph.replay()
    torch.cuda.synchronize()
    for k in range(4):
        assert torch.equal(_bits(eager[k]) if eager[k].is_floating_point() else eager[k].cpu(),
                           _bits(replayed[k]) if replayed[k].is_floating_point() else replayed[k].cpu()), ("replay vs eager", k)
    for e in range(E_):
        ref, bound, n = X.mean_write_f64(sums0[e], feat[e], idx[e], None, cells)
        X.check_lattice([feat[e], sums0[e], ref], q, bound)
        if not act_l[e]:
            ref = sums0[e].astype(np.float64)
            assert not eager[3][e].any()
        _same_bits(eager[0][e], _exact32(ref), (e, "sums"))


# ------------------------------------------------------------------------------------------------------------------------------
# 4  EpisodeBatch.step with bf16 CHW features: pipelined and stream-ordered, late features, against an fp32 twin
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def sleep_cycles(cuda):
    """torch.cuda._sleep cycles that keep a stream busy for about 50 ms on this device (measured, not assumed)."""
    probe = 20_000_000
    torch.cuda._sleep(5 * probe)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    torch.cuda._sleep(probe)
    b.record()
    b.synchronize()
    return min(max(int(probe * 50 / max(a.elapsed_time(b), 1e-3)), 2_000_000), 150_000_000)


@pytest.mark.parametrize("pipeline", [False, True], ids=["ordered", "pipelined"])
def test_episode_batch_step_bf16_chw_matches_fp32_twin_bitwise(eod, cuda, sleep_cycles, pipeline):
    """Five frames of step(proj_indices=...) with samp on some frames and active masks; the bf16 batch's features are produced on the
    caller's stream after the step was enqueued (the stream is still busy when step returns).  Against a twin fed feat.float() with
    LAYOUT_CHW: every frame's levels, and sums / counts / norm16, bit for bit - and sums equal the float64 reference."""
    E, H, W, C, mw, mh, T = 3, 96, 128, 128, 60, 45, 5
    cells = mw * mh
    rng = np.random.default_rng(70 + pipeline)
    a = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, layout=eod._lib.LAYOUT_CHW_BF16, pipeline=pipeline)
    b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, layout=eod._lib.LAYOUT_CHW, pipeline=pipeline)
    depth, pose, shifts = torch.zeros((E, H, W), device=cuda), torch.zeros((E, 12), device=cuda), torch.zeros((E, 6), device=cuda)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    plan = [dict(), dict(samp=0.4), dict(active=[1, 1, 0]), dict(samp=0.3, active=[0, 2, 1]), dict()]
    feat_buf = torch.empty((E, C, H, W), dtype=torch.bfloat16, device=cuda)
    ref = np.zeros((E, cells, C))
    # warm-up frame (loads every kernel and creates the streams' workspaces), then a clean grid
    for x, f in ((a, feat_buf.zero_()), (b, feat_buf.float())):
        x.step(depth, pose, shifts, intr, 0.2, f, proj_indices=_t(np.zeros((E, H, W), np.int32), cuda))
        x.reset(full=True)
    torch.cuda.synchronize()
    for t in range(T):
        p = plan[t]
        samp = (rng.random((E, H, W)) < p["samp"]) if "samp" in p else None
        idx = np.stack([X.index_plane(rng, H, W, cells, None if samp is None else samp[e], 5) for e in range(E)])
        feat = X.dyadic(rng, (E, C, H, W), 3, 3)
        src = _t(feat, cuda, torch.bfloat16)
        kw = dict(proj_indices=_t(idx, cuda))
        if "active" in p:
            kw["active"] = _t(np.array(p["active"], np.int32), cuda)
        d_samp = None if samp is None else _t(samp.astype(np.uint8), cuda)
        lb = [l.clone() for l in b.step(depth, pose, shifts, intr, 0.2, src.float(), d_samp, **kw)]
        b.join()
        feat_buf.fill_(float("nan"))                                         # read too early, these would poison the grid
        torch.cuda.synchronize()
        torch.cuda._sleep(sleep_cycles)
        feat_buf.copy_(src)
        la = a.step(depth, pose, shifts, intr, 0.2, feat_buf, d_samp, **kw)
        assert not torch.cuda.current_stream().query(), f"t={t}: the caller's stream had drained - the late feature proves nothing"
        la = [l.clone() for l in la]
        a.join()
        torch.cuda.synchronize()
        for k in range(3):
            _same_bits(la[k], lb[k], (t, "level", k))
        for name in ("sums", "counts", "norm16"):
            _same_bits(getattr(a, name), getattr(b, name), (t, name))
        for e in range(E):
            if "active" not in p or p["active"][e] > 0:
                r, bound, n = X.mean_write_f64(ref[e], feat[e], idx[e], None if samp is None else samp[e], cells)
                X.assert_pow2_counts(n)
                X.check_lattice([feat[e], ref[e], r], 3 + 5, bound)
                ref[e] = r
            _same_bits(a.sums[e], _exact32(ref[e]), (t, e, "sums vs float64"))
    assert float(a.counts.max()) >= 3


# ------------------------------------------------------------------------------------------------------------------------------
# 5  reference-facing methods take 16-bit images as they are
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", list(LAYOUTS))
def test_spatial_memory_16bit_images_match_widened_fp32(eod, cuda, kind, monkeypatch):
    """project_image_features and write_image_features with a bf16 / fp16 (1,C,480,640) image equal the same calls on the widened
    fp32 image, bitwise (exact inputs), and the write really takes the 16-bit CHW layout."""
    _, dtype = LAYOUTS[kind]
    H, W, C, cells = 480, 640, 512, 4000
    rng = np.random.default_rng(300 + len(kind))
    observed = rng.random((H, W)) < 0.8
    samp = R.sample_mask(torch.from_numpy(observed), 8).numpy()
    idx = X.index_plane(rng, H, W, cells, samp, 6)
    feat = X.dyadic(rng, (1, C, H, W), 3, 3)
    img16 = _t(feat, cuda, dtype)
    img32 = img16.float()
    layouts = []
    real = eod.ops.write_mean
    monkeypatch.setattr(eod.ops, "write_mean", lambda *a, **k: (layouts.append(a[5] if len(a) > 5 else k.get("layout")), real(*a, **k))[1])
    proj = _t(idx[..., None], cuda)
    outs = {}
    for name, img in (("16", img16), ("32", img32)):
        mem = eod.SpatialFeatureMemory(C, cuda, height=H, width=W)
        mem.reset(cells)
        mean, observed_mem = mem.project_image_features(img, _t(observed, cuda), [proj], [mem.implicit_memory])
        mem.write_image_features(img, _t(observed, cuda), proj)
        torch.cuda.synchronize()
        outs[name] = (mean, observed_mem, mem.implicit_memory.clone(), mem.observations.clone())
    assert layouts == [LAYOUTS[kind][0]] * 2 + [0, 0], layouts
    _same_bits(outs["16"][0], outs["32"][0].cpu(), "mean")
    assert torch.equal(outs["16"][1], outs["32"][1])
    _same_bits(outs["16"][2], outs["32"][2].cpu(), "implicit_memory")
    assert torch.equal(outs["16"][3], outs["32"][3])
    ref, _, n = X.mean_write_f64(np.zeros((cells, C)), feat[0], idx, samp, cells)
    _same_bits(outs["16"][0], _exact32(ref[n > 0]), "mean vs float64")


# ------------------------------------------------------------------------------------------------------------------------------
# 6  EpisodeRunner over 16-bit providers
# ------------------------------------------------------------------------------------------------------------------------------
def _assert_same_state(a, b, what):
    assert torch.equal(a.counts, b.counts), (what, "counts")
    ref = b.sums.double()
    err = float((a.sums.double() - ref).abs().max())
    assert err <= SUM_TOL * max(float(ref.abs().max()), 1e-30), (what, err)
    assert torch.equal((a.sums != 0).any(-1), (b.sums != 0).any(-1)), (what, "touched rows")


def test_runner_pooled_bf16_chw_matches_fp32_run(eod, cuda):
    """PooledSyntheticProvider(feat_dtype=bf16) with LAYOUT_CHW_BF16 lands in the state of the fp32 run on the widened slabs."""
    H, W, C, mw, mh = 96, 128, 256, 60, 45
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    kw = dict(height=H, width=W, map_w=mw, map_h=mh, pool=3, lengths=[3, 2, 4, 1])
    p16 = eod.runner.PooledSyntheticProvider(4, 4, C, 2, cuda, feat_dtype=torch.bfloat16, **kw)
    p32 = eod.runner.PooledSyntheticProvider(4, 4, C, 2, cuda, **kw)
    assert p16.feat[0].dtype == torch.bfloat16 and p32.feat[0].dtype == torch.float32
    assert torch.equal(p16.feat[0].float(), p32.feat[0].to(torch.bfloat16).float())      # same draws, rounded
    p32.feat = [f.float() for f in p16.feat]
    runs = {}
    for name, prov, layout in (("16", p16, eod._lib.LAYOUT_CHW_BF16), ("32", p32, eod._lib.LAYOUT_CHW)):
        r = eod.EpisodeRunner(prov, mw, mh, C, n_slots=2, height=H, width=W, device=cuda, test_type="episodic", intr=intr, cell=0.2,
                              layout=layout)
        stats = r.run()
        torch.cuda.synchronize()
        runs[name] = (r.batch, stats)
    assert runs["16"][1] == runs["32"][1]
    _assert_same_state(runs["16"][0], runs["32"][0], "pooled")
    assert float(runs["16"][0].counts.max()) >= 1


def test_runner_host_f16_matches_fp32_run(eod, cuda):
    """HostEpisodeProvider(feat_dtype=fp16) staging fp32 frames with LAYOUT_CHW_F16 equals the fp32 run on the fp16-rounded frames."""
    H, W, C, mw, mh = 96, 128, 128, 60, 45
    rng = np.random.default_rng(8)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    episodes = []
    for e, n in enumerate((3, 2)):
        frames = []
        for i in range(n):
            idx = rng.integers(0, mw * mh, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1).astype(np.int32)
            frames.append({"sequence_name": f"seq_{e}", "memory_reset": i == 0, "proj_indices": idx[..., None],
                           "feat": rng.standard_normal((C, H, W)).astype(np.float32)})
        episodes.append(frames)
    rounded = [[dict(fr, feat=fr["feat"].astype(np.float16).astype(np.float32)) for fr in ep] for ep in episodes]
    runs = {}
    for name, prov, layout in (("16", eod.HostEpisodeProvider(episodes, cuda, feat_dtype=torch.float16), eod._lib.LAYOUT_CHW_F16),
                               ("32", eod.HostEpisodeProvider(rounded, cuda), eod._lib.LAYOUT_CHW)):
        r = eod.EpisodeRunner(prov, mw, mh, C, n_slots=2, height=H, width=W, device=cuda, test_type="episodic", intr=intr, cell=0.2,
                              layout=layout)
        r.run()
        torch.cuda.synchronize()
        runs[name] = r.batch
    _assert_same_state(runs["16"], runs["32"], "host")


# ------------------------------------------------------------------------------------------------------------------------------
# 7  refusals
# ------------------------------------------------------------------------------------------------------------------------------
def test_chw16_refusals(eod, cuda):
    lib, ops = eod._lib, eod.ops
    E, C, cells = 1, 128, 50
    idx = torch.zeros((E, 64 * 8), dtype=torch.int32, device=cuda)
    cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    sums = torch.zeros((E, cells, C), device=cuda)
    f16 = torch.zeros((E, C, 64 * 8), dtype=torch.bfloat16, device=cuda)
    with pytest.raises(TypeError):
        ops.write_mean(f16, idx, None, cnt, sums, lib.LAYOUT_CHW)             # bf16 features with the fp32 layout
    with pytest.raises(eod.EodError, match="WRITE_DET"):
        eod.EpisodeBatch(E, 10, 5, C, 8, 64, cuda, layout=lib.LAYOUT_CHW_BF16, variant=lib.WRITE_DET)
    with pytest.raises(eod.EodError, match="WRITE_DET"):
        eod.EpisodeBatch(E, 10, 5, C, 8, 64, cuda, layout=lib.LAYOUT_CHW_F16, variant=lib.WRITE_DET)
    odd = torch.zeros((E, 4 * 9), dtype=torch.int32, device=cuda)          # HW = 36: rows of 72 bytes
    with pytest.raises(eod.EodError, match="16-byte aligned"):
        ops.write_mean(torch.zeros((E, C, 36), dtype=torch.float16, device=cuda), odd, None, cnt, sums, lib.LAYOUT_CHW_F16)
    pix = torch.zeros((E, 64 * 8), device=cuda)
    with pytest.raises(eod.EodError, match="pix_inv_n"):
        ops.write_mean(f16, idx, None, cnt, sums, lib.LAYOUT_CHW_BF16, lib.WRITE_AUTO, pix)
    with pytest.raises(eod.EodError, match="HW % 64"):
        ops.write_mean(torch.zeros((E, C, 24 * 30), dtype=torch.bfloat16, device=cuda), torch.zeros((E, 720), dtype=torch.int32, device=cuda),
                       None, cnt, sums, lib.LAYOUT_CHW_BF16, lib.WRITE_TMA)
    torch.cuda.synchronize()
    assert not sums.any()
