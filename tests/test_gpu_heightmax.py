"""Lock-step height-max regime (BASELINE configs[2]: SMNet's top-down height-max projection) on the B200: HeightMaxBatch and the
eod_heightmax_* kernels against the two-pass path (ops.backproject_quantize + ops.write_max / write_max_linear, which stay as they
are) and against the CPU oracle (oracle.reference_ops.smnet_heightmax_frame), plus EpisodeRunner(regime="heightmax").
Run on the B200 box with `-m gpu`."""
import math
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R

pytestmark = pytest.mark.gpu

H, W, MW, MH, CELL = 96, 128, 120, 90, 0.05


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _episodes(eod, E, T, seed=7, mw=MW, mh=MH, cell=CELL, h=H, w=W):
    eps = [eod.episodes.make_episode(seed + e, T, h, w, mw, mh, cell) for e in range(E)]
    Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe for ep in eps]).reshape(-1, 5))).reshape(E, T, 4, 4)
    depth = np.stack([ep.depth for ep in eps], 1)                                    # (T,E,H,W)
    pose = Tm[:, :, :3].reshape(E, T, 12).permute(1, 0, 2).contiguous()              # (T,E,12)
    shifts = np.stack([np.concatenate([ep.map_world_shift, np.zeros(3, np.float32)]) for ep in eps])
    return depth, pose, shifts


class _TwoPass:
    """The existing path per episode: backproject_quantize (idx, outlier, height planes) + write_max into (E,...) state."""

    def __init__(self, E, C, cells, dev, stride=1):
        self.state = torch.zeros((E, cells, C), device=dev)
        self.hmap = torch.zeros((E, cells), device=dev)
        self.obs = torch.zeros((E, cells), dtype=torch.uint8, device=dev)
        self.key = torch.zeros((E, cells), dtype=torch.int64, device=dev)
        self.arg = torch.zeros((E, cells), dtype=torch.int32, device=dev)
        self.stride = stride

    def frame(self, eod, e, depth, pose, shifts, intr, feat, layout, mw=MW, mh=MH, cell=CELL):
        g = eod.ops.backproject_quantize(depth[e:e + 1], pose[e:e + 1], shifts[e:e + 1], intr, cell, mw, mh, want_outlier=True, want_height=True)
        s = slice(e, e + 1)
        eod.ops.write_max(g["height"], g["idx"], g["outlier"], feat[s].contiguous(), self.hmap[s], self.key[s], self.arg[s], self.obs[s],
                          self.state[s], layout, self.stride)
        return int((self.arg[e] >= 0).sum())


def _assert_scratch_clean(batch):
    assert int(batch.scratch.key64.abs().sum()) == 0 and int(batch.scratch.n_list.abs().sum()) == 0


@pytest.mark.parametrize("u16", [False, True], ids=["f32", "u16"])
@pytest.mark.parametrize("stride", [1, 4])
def test_fused_from_depth_equals_two_pass(eod, cuda, u16, stride):
    """From depth: state, height_map and observed bit-identical to backproject_quantize + write_max; the raised count equals the
    cells with arg_pix >= 0; the idle slot is untouched; the key scratch and the lists are zero after every step."""
    E, T, C = 3, 4, 64
    depth, pose, shifts = _episodes(eod, E, T)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    if u16:
        depth = np.minimum(np.round(depth * 1000.0), 65535).astype(np.uint16)
    sh = _t(shifts, cuda)
    batch = eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda, layout=eod._lib.LAYOUT_HWC, pix_stride=stride)
    ref = _TwoPass(E, C, MW * MH, cuda, stride)
    gen = torch.Generator(device=cuda).manual_seed(3)
    idle = 1
    active = torch.tensor([1, 0, 1], dtype=torch.int32, device=cuda)
    total = 0
    for t in range(T):
        d, p = _t(depth[t], cuda), pose[t].to(cuda)
        feat = torch.randn((E, H, W, C), device=cuda, generator=gen)
        feat[idle] = float("nan")                                         # the idle slot's features must not be read
        snap = (batch.state[idle].clone(), batch.height_map[idle].clone(), batch.observed[idle].clone())
        raised = batch.step(feat, depth=d, pose=p, shifts=sh, intr=intr, cell=CELL, active=active)
        n_ref = sum(ref.frame(eod, e, d, p, sh, intr, feat, eod._lib.LAYOUT_HWC) for e in (0, 2))
        torch.cuda.synchronize()
        assert int(raised.item()) == n_ref, t
        total += n_ref
        for e in (0, 2):
            assert torch.equal(batch.height_map[e], ref.hmap[e]), (t, e)
            assert torch.equal(batch.observed[e], ref.obs[e]), (t, e)
            assert torch.equal(batch.state[e], ref.state[e]), (t, e)
        assert torch.equal(batch.state[idle], snap[0]) and torch.equal(batch.height_map[idle], snap[1]) and torch.equal(batch.observed[idle], snap[2])
        _assert_scratch_clean(batch)
    assert total > 100


def _adversarial_frames(rng, T, h, w, mw, mh, C):
    """The scenario of test_write_max_vs_oracle: quantised heights (many exact ties), a frame that raises nothing new, NaN / +-inf."""
    for t in range(T):
        w2m = np.stack([rng.integers(0, mw, (h // 4, w // 4)).repeat(4, 0).repeat(4, 1), rng.integers(0, mh, (h // 4, w // 4)).repeat(4, 0).repeat(4, 1)], -1)
        inl = rng.uniform(size=(h, w)) < 0.7
        heights = (np.round(rng.uniform(-1.5, 1.0, (h, w)) * 4) / 4).astype(np.float32)
        if t == 2:
            heights[:] = heights.min() - 5
        if t == 3:
            heights[rng.uniform(size=(h, w)) < 0.1] = np.nan
            heights[rng.uniform(size=(h, w)) < 0.02] = np.inf
            heights[rng.uniform(size=(h, w)) < 0.02] = -np.inf
        yield w2m, inl, heights, rng.standard_normal((h, w, C)).astype(np.float32)


@pytest.mark.parametrize("layout,stride", [(1, 1), (0, 1), (1, 4)])
def test_planes_adversarial_heights(eod, cuda, layout, stride):
    """From planes: ties, a frame that raises nothing, NaN and +-inf heights - bit-identical to write_max and to the oracle."""
    rng = np.random.default_rng(17 + stride)
    h, w, C, mw, mh, T = 48, 64, 64, 23, 19, 4
    cells = mw * mh
    state, observed, hmap = torch.zeros(cells, C), torch.zeros(cells, dtype=torch.bool), torch.zeros(cells)
    batch = eod.HeightMaxBatch(1, mw, mh, C, h, w, cuda, layout=layout, pix_stride=stride)
    ref = _TwoPass(1, C, cells, cuda, stride)
    for t, (w2m, inl, heights, feat) in enumerate(_adversarial_frames(rng, T, h, w, mw, mh, C)):
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, torch.from_numpy(feat), torch.from_numpy(w2m),
                                                                torch.from_numpy(inl), torch.from_numpy(heights), mw, stride)
        flat = _t((w2m[..., 1] * mw + w2m[..., 0]).astype(np.int32), cuda)[None]
        hd, od = _t(heights, cuda)[None], _t((~inl).view(np.uint8), cuda)[None]
        f_dev = _t(feat if layout == 1 else feat.transpose(2, 0, 1), cuda)[None].contiguous()
        raised = batch.step(f_dev, height=hd, idx=flat, outlier=od)
        eod.ops.write_max(hd, flat, od, f_dev, ref.hmap, ref.key, ref.arg, ref.obs, ref.state, layout, stride)
        torch.cuda.synchronize()
        assert int(raised.item()) == int(m.sum()) == int((ref.arg >= 0).sum()), t
        for got, two_pass, orc in ((batch.height_map[0], ref.hmap[0], hmap), (batch.observed[0], ref.obs[0], observed.to(torch.uint8)),
                                   (batch.state[0], ref.state[0], state)):
            assert torch.equal(got, two_pass) and torch.equal(got.cpu(), orc), t
        _assert_scratch_clean(batch)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16], ids=["bf16", "fp16"])
@pytest.mark.parametrize("hwc", [True, False], ids=["HWC", "CHW"])
def test_16bit_features_equal_fp32_of_widened(eod, cuda, dtype, hwc):
    E, T, C, mw, mh = 2, 3, 64, 300, 240                                    # a 15 m x 12 m map: the whole room
    L = eod._lib
    depth, pose, shifts = _episodes(eod, E, T, seed=21, mw=mw, mh=mh)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    sh = _t(shifts, cuda)
    base = L.LAYOUT_HWC if hwc else L.LAYOUT_CHW
    b16 = eod.HeightMaxBatch(E, mw, mh, C, H, W, cuda, layout=eod.ops.layout_for_dtype(base, dtype))
    b32 = eod.HeightMaxBatch(E, mw, mh, C, H, W, cuda, layout=base)
    gen = torch.Generator(device=cuda).manual_seed(9)
    for t in range(T):
        shape = (E, H, W, C) if hwc else (E, C, H, W)
        f16 = (torch.randn(shape, device=cuda, generator=gen) * 3).to(dtype)
        geo = dict(depth=_t(depth[t], cuda), pose=pose[t].to(cuda), shifts=sh, intr=intr, cell=CELL)
        b16.step(f16, **geo)
        b32.step(f16.float(), **geo)
    torch.cuda.synchronize()
    assert int(b32.observed.sum()) > 100
    assert torch.equal(b16.state, b32.state) and torch.equal(b16.height_map, b32.height_map) and torch.equal(b16.observed, b32.observed)


@pytest.mark.parametrize("layout", [0, 1])
def test_linlayer_update_vs_fp64_oracle(eod, cuda, layout):
    """'replace' update with the linear layer: raised rows within 1e-5 of scale of the fp64 oracle, the other rows untouched bit for
    bit, the raised count and the emitted destination rows equal the oracle's raised set."""
    rng = np.random.default_rng(31 + layout)
    h, w, C_in, C_mem, mw, mh, T, stride = 48, 64, 64, 256, 23, 19, 4, 2
    cells = mw * mh
    lin_w = (rng.standard_normal((C_mem, C_in)) / 8).astype(np.float32)
    lin_b = rng.standard_normal(C_mem).astype(np.float32)
    state, observed, hmap = torch.zeros(cells, C_mem, dtype=torch.float64), torch.zeros(cells, dtype=torch.bool), torch.zeros(cells)
    batch = eod.HeightMaxBatch(1, mw, mh, C_in, h, w, cuda, layout=layout, linlayer=(_t(lin_w, cuda), _t(lin_b, cuda)), pix_stride=stride)
    for t, (w2m, inl, heights, feat) in enumerate(_adversarial_frames(rng, T, h, w, mw, mh, C_in)):
        prev = batch.state.clone()
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, torch.from_numpy(feat).double(), torch.from_numpy(w2m),
                                                                torch.from_numpy(inl), torch.from_numpy(heights), mw, stride,
                                                                linlayer=(torch.from_numpy(lin_w).double(), torch.from_numpy(lin_b).double()))
        flat = _t((w2m[..., 1] * mw + w2m[..., 0]).astype(np.int32), cuda)[None]
        f_dev = _t(feat if layout == 1 else feat.transpose(2, 0, 1), cuda)[None].contiguous()
        count = batch.step(f_dev, height=_t(heights, cuda)[None], idx=flat, outlier=_t((~inl).view(np.uint8), cuda)[None])
        torch.cuda.synchronize()
        n = int(count.item())
        assert n == int(m.sum()), t
        assert set(batch.scratch._winners[1][:n].tolist()) == set(np.nonzero(m.numpy())[0].tolist())
        assert torch.equal(batch.height_map[0].cpu(), hmap) and torch.equal(batch.observed[0].cpu().bool(), observed)
        got = batch.state[0].cpu().double()
        if n:
            assert float((got[m] - state[m]).abs().max()) <= 1e-5 * float(state[m].abs().max())
        assert torch.equal(batch.state[0][~m.to(cuda)], prev[0][~m.to(cuda)])
        state = got.clone()
        _assert_scratch_clean(batch)


def test_batch_equals_single_episodes_and_reset_mask(eod, cuda):
    """E episodes in one batch give the bits of each episode run alone; reset_mask clears exactly its slots before the frame."""
    E, T, C = 3, 4, 32
    depth, pose, shifts = _episodes(eod, E, T, seed=51)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    sh = _t(shifts, cuda)
    batch = eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda)
    alone = [eod.HeightMaxBatch(1, MW, MH, C, H, W, cuda) for _ in range(E)]
    gen = torch.Generator(device=cuda).manual_seed(4)
    reset = torch.tensor([0, 1, 0], dtype=torch.int32, device=cuda)
    for t in range(T):
        feat = torch.randn((E, C, H, W), device=cuda, generator=gen)
        d, p = _t(depth[t], cuda), pose[t].to(cuda)
        rm = reset if t == 2 else None
        batch.step(feat, depth=d, pose=p, shifts=sh, intr=intr, cell=CELL, reset_mask=rm)
        for e in range(E):
            if t == 2 and e == 1:
                alone[e].reset()
            alone[e].step(feat[e:e + 1].contiguous(), depth=d[e:e + 1].contiguous(), pose=p[e:e + 1].contiguous(), shifts=sh[e:e + 1].contiguous(),
                          intr=intr, cell=CELL)
        if t == 2:                                                            # slot 1 now holds exactly this frame
            fresh = eod.HeightMaxBatch(1, MW, MH, C, H, W, cuda)
            fresh.step(feat[1:2].contiguous(), depth=d[1:2].contiguous(), pose=p[1:2].contiguous(), shifts=sh[1:2].contiguous(), intr=intr, cell=CELL)
            assert torch.equal(batch.state[1], fresh.state[0]) and torch.equal(batch.height_map[1], fresh.height_map[0])
    torch.cuda.synchronize()
    for e in range(E):
        assert torch.equal(batch.state[e], alone[e].state[0]) and torch.equal(batch.height_map[e], alone[e].height_map[0])
        assert torch.equal(batch.observed[e], alone[e].observed[0])
    full = eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda)
    full.state.copy_(batch.state), full.height_map.copy_(batch.height_map), full.observed.copy_(batch.observed)
    full.reset(torch.tensor([1, 0, 0], dtype=torch.int32, device=cuda))
    torch.cuda.synchronize()
    assert not bool(full.state[0].any()) and not bool(full.height_map[0].any()) and not bool(full.observed[0].any())
    assert torch.equal(full.state[1:], batch.state[1:]) and torch.equal(full.height_map[1:], batch.height_map[1:])


# ---- runner ---------------------------------------------------------------------------------------------------------------------
RC, RMW, RMH, RCELL = 256, 250, 200, 0.02           # configs[2]-shaped: 256-d features, 0.02 m cells (a small map)
SCENES = {"aaaaaaaaaaa_0": [3, 2, 4], "bbbbbbbbbbb_1": [2, 1], "ccccccccccc_0": [1, 3]}


def _runner_dataset(eod, source):
    rng = np.random.default_rng(5)
    files = [f"{scene}_{k}.h5" for scene, lens in SCENES.items() for k in range(len(lens))]
    rng.shuffle(files)
    ordered = eod.formats.order_files(files, "default")
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    episodes, shifts = [], []
    for f in ordered:
        scene, k = f[:13], int(f.split("_")[-1].split(".")[0])
        n = SCENES[scene][k]
        ep = eod.episodes.make_episode(100 + 7 * len(episodes), n, H, W, RMW, RMH, RCELL)
        Tm = eod.transform3d(torch.from_numpy(ep.xyzhe))
        frames = []
        for i in range(n):
            o = oracle.backproject_quantize(ep.depth[i], Tm[i].numpy(), intr, np.zeros(3, np.float32), ep.map_world_shift, np.float32(RCELL),
                                            RMW, RMH, 0, 0.5, want=("idx", "q2", "outlier", "height"))
            fr = {"sequence_name": f, "memory_reset": eod.formats.memory_reset_flag("default", f, i), "_geo": o,
                  "feat": np.random.default_rng(1000 + 31 * len(episodes) + i).standard_normal((RC, H, W)).astype(np.float32)}
            if source == "planes":
                fr["proj_indices"], fr["height"], fr["outlier"] = o["idx"][..., None], o["height"], o["outlier"].astype(bool)
            else:
                fr["depth"], fr["pose"] = ep.depth[i], Tm[i, :3].reshape(12).numpy()
            frames.append(fr)
        episodes.append(frames)
        shifts.append(np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]))
    return episodes, shifts, intr


def _serial_oracle(episodes):
    """One SMNet encoder, one episode after the other; the map is taken after each episode's last frame."""
    cells = RMW * RMH
    saved = {}
    state = observed = hmap = None
    for ep in episodes:
        for i, fr in enumerate(ep):
            if fr["memory_reset"]:
                state, observed, hmap = torch.zeros(cells, RC), torch.zeros(cells, dtype=torch.bool), torch.zeros(cells)
            o = fr["_geo"]
            state, observed, hmap, _, _ = R.smnet_heightmax_frame(state, observed, hmap, torch.from_numpy(fr["feat"]).permute(1, 2, 0).contiguous(),
                                                                  torch.from_numpy(o["q2"]), ~torch.from_numpy(o["outlier"].astype(bool)),
                                                                  torch.from_numpy(o["height"]), RMW)
        saved[ep[0]["sequence_name"]] = (state.clone(), observed.clone(), hmap.clone())
    return saved


@pytest.mark.parametrize("source", ["depth", "planes"])
def test_runner_heightmax_matches_serial_oracle(eod, cuda, tmp_path, source):
    episodes, shifts, intr = _runner_dataset(eod, source)
    ref = _serial_oracle(episodes)
    dumps = {}
    for slots in (2, 3):
        out = tmp_path / f"r{slots}"
        runner = eod.EpisodeRunner(eod.HostEpisodeProvider(episodes, cuda, shifts), RMW, RMH, RC, n_slots=slots, height=H, width=W, device=cuda,
                                   intr=intr, cell=RCELL, save_dir=str(out), regime="heightmax")
        stats = runner.run(on_levels=lambda *a: pytest.fail("the height-max regime has no read"))
        assert stats["frames"] == sum(len(ep) for ep in episodes) and stats["steps"] < stats["frames"]
        names = sorted(os.listdir(out / "heightmax"))
        assert len(names) == len(ref)
        dumps[slots] = {os.path.splitext(n)[0]: eod.formats.load_heightmax(str(out / "heightmax" / n)) for n in names}
    for n in dumps[2]:
        assert all(np.array_equal(a, b) for a, b in zip(dumps[2][n], dumps[3][n])), n
    for name, (s_ref, o_ref, h_ref) in ref.items():
        got = dumps[2][os.path.splitext(name)[0]]
        assert np.array_equal(got[0], s_ref.numpy()) and np.array_equal(got[1].astype(bool), o_ref.numpy()), name
        assert np.array_equal(got[2], h_ref.numpy()), name
    assert any(o.any() for _, o, _ in ref.values())


def test_runner_heightmax_refuses_other_regime_inputs(eod, cuda):
    episodes, shifts, intr = _runner_dataset(eod, "planes")
    bad = [[{k: v for k, v in fr.items() if k != "height"} for fr in ep] for ep in episodes]        # an index plane without heights
    runner = eod.EpisodeRunner(eod.HostEpisodeProvider(bad, cuda, shifts), RMW, RMH, RC, n_slots=2, height=H, width=W, device=cuda,
                               intr=intr, cell=RCELL, regime="heightmax")
    with pytest.raises(eod.EodError):
        runner.run()
    det = [[dict(sequence_name=fr["sequence_name"], memory_reset=fr["memory_reset"], proj_indices=fr["proj_indices"],
                 box_features=np.zeros((0, RC), np.float32), mask_probs=np.zeros((0, 28, 28), np.float32), boxes=np.zeros((0, 4), np.float32))
            for fr in ep] for ep in episodes]
    runner = eod.EpisodeRunner(eod.HostEpisodeProvider(det, cuda, shifts), RMW, RMH, RC, n_slots=2, height=H, width=W, device=cuda,
                               intr=intr, cell=RCELL, regime="heightmax")
    with pytest.raises(eod.EodError):
        runner.run()


def test_heightmax_config3_full_size(eod, cuda):
    """configs[2] at full size (480x640, C=256, 0.02 m cells, 1000x1000 map) through HeightMaxBatch from depth: equal to the oracle
    bit for bit (state, observed set, height map)."""
    h, w, C, mw, mh, T_ = 480, 640, 256, 1000, 1000, 3
    cells = mw * mh
    ep = eod.episodes.make_episode(4321, T_, h, w, mw, mh, 0.02, room_size=(24.0, 16.0))
    intr = eod.compute_intrinsics(w, h, math.radians(67.5))
    Tm = eod.transform3d(torch.from_numpy(ep.xyzhe))
    sh = _t(np.concatenate([ep.map_world_shift, np.zeros(3, np.float32)])[None], cuda)
    state, observed, hmap = torch.zeros(cells, C), torch.zeros(cells, dtype=torch.bool), torch.zeros(cells)
    batch = eod.HeightMaxBatch(1, mw, mh, C, h, w, cuda, layout=eod._lib.LAYOUT_HWC)
    gen = torch.Generator(device=cuda).manual_seed(5)
    n_raised = 0
    for t in range(T_):
        feat = torch.randn((1, h, w, C), device=cuda, generator=gen)
        raised = batch.step(feat, depth=_t(ep.depth[t:t + 1], cuda), pose=Tm[t:t + 1, :3].reshape(1, 12).to(cuda), shifts=sh, intr=intr, cell=0.02)
        o = oracle.backproject_quantize(ep.depth[t], Tm[t].numpy(), intr, ep.map_world_shift, np.zeros(3, np.float32), 0.02, mw, mh, 0, 0.5)
        inl = ~torch.from_numpy(o["outlier"].astype(bool))
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, feat[0].cpu(), torch.from_numpy(o["q2"]), inl,
                                                                torch.from_numpy(o["height"]), mw, 1)
        torch.cuda.synchronize()
        assert int(raised.item()) == int(m.sum()), t
        assert torch.equal(batch.height_map[0].cpu(), hmap) and torch.equal(batch.observed[0].cpu().bool(), observed)
        assert torch.equal(batch.state[0].cpu(), state), t
        _assert_scratch_clean(batch)
        n_raised += int(m.sum())
    assert n_raised > 1000 and 0 < float(inl.float().mean()) < 1


def test_heightmax_refusals(eod, cuda):
    L = eod._lib
    E, C = 1, 32
    depth, pose, shifts = _episodes(eod, E, 1)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    geo = dict(depth=_t(depth[0], cuda), pose=pose[0].to(cuda), shifts=_t(shifts, cuda), intr=intr, cell=CELL)
    b = eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda)
    with pytest.raises(eod.EodError):                                                     # CPU features
        b.step(torch.zeros((E, C, H, W)), **geo)
    with pytest.raises(eod.EodError):                                                     # CPU geometry
        b.step(torch.zeros((E, C, H, W), device=cuda), **dict(geo, depth=torch.from_numpy(depth[0])))
    with pytest.raises(eod.EodError):                                                     # bf16 features for an fp32 layout
        b.step(torch.zeros((E, C, H, W), dtype=torch.bfloat16, device=cuda), **geo)
    with pytest.raises(eod.EodError):                                                     # fp32 features for a bf16 layout
        eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda, layout=L.LAYOUT_CHW_BF16).step(torch.zeros((E, C, H, W), device=cuda), **geo)
    with pytest.raises(eod.EodError):                                                     # C % 4 != 0
        eod.HeightMaxBatch(E, MW, MH, 30, H, W, cuda, layout=L.LAYOUT_HWC).step(torch.zeros((E, H, W, 30), device=cuda), **geo)
    b2 = eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda, layout=L.LAYOUT_HWC)
    b2.state = torch.zeros(E * MW * MH * C + 1, device=cuda)[1:].view(E, MW * MH, C)     # rows not 16-byte aligned
    with pytest.raises(eod.EodError):
        b2.step(torch.zeros((E, H, W, C), device=cuda), **geo)
    torch.cuda.synchronize()
    assert int(b2.scratch.key64.abs().sum()) == 0                                         # refused before the contest
    with pytest.raises(eod.EodError):
        eod.HeightMaxBatch(E, MW, MH, C, H, W, torch.device("cpu"))
    with pytest.raises(eod.EodError):                                                     # linlayer reads fp32 features only
        eod.HeightMaxBatch(E, MW, MH, C, H, W, cuda, layout=L.LAYOUT_HWC_BF16, linlayer=(torch.zeros(16, C), None))
