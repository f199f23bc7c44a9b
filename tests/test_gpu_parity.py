"""GPU parity tests (run on the B200 box with `-m gpu`).  Every CUDA result goes through the C ABI
(embodied-object-detection_b200.ops -> libeod_memory.so) and is compared with
  * the committed golden fixtures (outputs of the reference's own source, tests/golden/make_golden.py), and
  * the CPU oracle (oracle/) on seeded inputs,
bit-exact for indices / masks / counts / argmax / fp16 read outputs, and within 1e-5 of the feature scale for
accumulated fp32 sums (tolerance stated by BASELINE.json north_star).
"""
import math

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R
from test_gpu_scale import FUSE_N, device_sms, fuse_trips

pytestmark = pytest.mark.gpu

SUM_TOL = 1e-5          # max|a-b| <= SUM_TOL * max|ref|   (SURVEY 8c)


def _unpack(bits, shape):
    return np.unpackbits(bits)[: int(np.prod(shape))].reshape(shape).astype(bool)


def _t(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t if dtype is None else t.to(dtype)


# --------------------------------------------------------------------------------------------------------
# geometry (A1-A5)
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["geometry_small", "geometry_full", "geometry_fine"])
def test_backproject_matches_reference_golden(eod, cuda, golden, name):
    g = golden(name)
    T, H, W = g["depth"].shape
    intr = eod.compute_intrinsics(W, H, float(g["vfov"]))
    depth = _t(g["depth"], cuda)
    pose = _t(g["T"][:, :3, :].reshape(T, 12), cuda)
    zero = np.zeros(3, np.float32)
    cell, mw, mh = float(g["cell"]), int(g["map_w"]), int(g["map_h"])
    # Projector flow (create_coco_mp3d.py): one shift
    sh = _t(np.tile(np.concatenate([g["map_world_shift"], zero]), (T, 1)), cuda)
    r = eod.ops.backproject_quantize(depth, pose, sh, intr, cell, mw, mh, want_q2=True, want_outlier=True, want_height=True)
    assert np.array_equal(r["q2"].cpu().numpy(), g["q2"])
    assert np.array_equal(r["outlier"].cpu().numpy().astype(bool), g["outlier"])
    assert np.array_equal(r["height"].cpu().numpy(), g["height"])
    # PointCloud + build_memory_data flow: shift applied second, clip to the border
    sh = _t(np.tile(np.concatenate([zero, g["map_world_shift"]]), (T, 1)), cuda)
    r = eod.ops.backproject_quantize(depth, pose, sh, intr, cell, mw, mh, want_world=True)
    assert np.array_equal(r["world"].cpu().numpy(), g["world"])
    assert np.array_equal(r["idx"].cpu().numpy(), g["flat"])


@pytest.mark.parametrize("name", ["geometry_small", "geometry_full", "geometry_fine"])
def test_quantize_world_matches_reference_golden(eod, cuda, golden, name):
    """Stored world coordinates -> proj_indices: SMNet/build_memory_data.py:135-143 executed from the reference source."""
    g = golden(name)
    got = eod.ops.quantize_world(_t(g["world"], cuda), g["map_world_shift"], float(g["cell"]), int(g["map_w"]), int(g["map_h"]))
    assert got.shape == g["flat"].shape + (1,) and got.dtype == torch.int32
    assert np.array_equal(got[..., 0].cpu().numpy(), g["flat"])


def test_robot_demo_geometry_matches_reference_golden(eod, cuda, golden):
    """The online robot path (robot_demo.py:514-534 executed from source): millimetre depth, axis-swapped pose, calibrated K,
    flat = q_x * map_h + q_z - through the Projector mirror with explicit intrinsics."""
    g = golden("robot")
    n, H, W = g["depth_mm"].shape
    proj = eod.Projector(math.radians(58), 1, H, W, int(g["map_h"]), int(g["map_w"]), float(g["res"]), np.zeros(3, np.float32), 3,
                         device=cuda, intrinsics=g["K"])
    for t in range(n):
        pv = g["pose_val"][t]
        T = eod.transform3d(torch.FloatTensor(np.array([[pv[0], 0.65, pv[1], -1 * pv[2], np.pi + 0.06]])), axis_swap=True)
        depth = torch.FloatTensor(g["depth_mm"][t] / 1000)[None, None]
        flat = proj.flat_indices(depth, T, g["map_world_shift"], order="xz")
        assert flat.shape == (1, H, W, 1) and flat.dtype == torch.int32
        assert np.array_equal(flat[0, ..., 0].cpu().numpy(), g["flat"][t])
        # raw sensor words straight to the device: the kernel does robot_demo.py:515's fp64 division and fp32 rounding itself
        raw = torch.from_numpy(g["depth_mm"][t].astype(np.uint16))[None, None]
        flat_raw = proj.flat_indices(raw, T, g["map_world_shift"], order="xz")
        assert np.array_equal(flat_raw[0, ..., 0].cpu().numpy(), g["flat"][t])


def test_backproject_u16_depth_every_sensor_word(eod, cuda):
    """All 65 536 uint16 depth words, several divisors, scalar and 4-px kernels: the in-kernel conversion must equal
    torch.FloatTensor(depth_u16 / div) (numpy fp64 true division, then fp32 rounding) bit for bit - checked on the heights / world
    coordinates, which expose the converted depth."""
    words = np.arange(65536, dtype=np.uint16)
    T = eod.transform3d(torch.from_numpy(np.array([[0.3, 0.65, -0.2, 0.4, math.pi + 0.06]], np.float32)), axis_swap=True)
    sh = _t(np.zeros((1, 6), np.float32), cuda)
    pose = T[:, :3].reshape(1, 12).to(cuda)
    for (H, W), div in (((128, 512), 1000.0), ((128, 512), 255.0), ((256, 256), 6553.5), ((65536 // 127 + 1, 127), 1000.0)):
        d = np.resize(words, (H, W))
        intr = eod.compute_intrinsics(W, H, math.radians(58))
        a = eod.ops.backproject_quantize(_t(d[None], cuda), pose, sh, intr, 0.05, 200, 200, 1, want_world=True, want_height=True, depth_div=div)
        ref_depth = torch.FloatTensor(d / div)[None].to(cuda)
        b = eod.ops.backproject_quantize(ref_depth, pose, sh, intr, 0.05, 200, 200, 1, want_world=True, want_height=True)
        for k in ("idx", "world", "height"):
            assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), (H, W, div, k)


def test_backproject_non_finite_depths_follow_torch(eod, cuda):
    """Depth values a sensor should never emit (inf, NaN, 3e38, 1e6): the clipped flat index and the outlier mask must still be what
    the reference's torch-CPU ops return - `.round().long()` of a non-finite / out-of-range float is INT64_MIN on x86, which the
    clip of build_memory_data.py:141-142 turns into cell 0; the outlier test of core.py:253-256 compares the rounded floats."""
    rng = np.random.default_rng(2)
    H, W, mw, mh, cell = 32, 64, 120, 90, 0.1
    depth = rng.uniform(0.3, 9.0, (H, W)).astype(np.float32)
    depth[0, :8] = [np.inf, np.nan, 3e38, 1e6, -np.inf, 0.0, 1e-30, 65504.0]
    xyzhe = np.array([[1.0, 1.25, -2.0, 0.9, math.pi + 0.1]], np.float32)
    T = eod.transform3d(torch.from_numpy(xyzhe))
    vf = math.radians(67.5)
    intr = eod.compute_intrinsics(W, H, vf)
    shift = np.array([-6.0, 0.0, -4.5], np.float32)
    world = R.pixel_to_world(torch.from_numpy(depth[None]), T, vf, torch.zeros(3))
    ref_idx = R.quantize_flat_index(world, torch.from_numpy(shift), cell, mw, mh).numpy().reshape(H, W)
    _, ref_out, _ = R.projector_forward(torch.from_numpy(depth[None, None]), T, vf, mh, mw, cell, torch.from_numpy(shift), 0.5)
    sh = _t(np.concatenate([np.zeros(3, np.float32), shift])[None], cuda)
    got = eod.ops.backproject_quantize(_t(depth[None], cuda), T[:, :3].reshape(1, 12).to(cuda), sh, intr, cell, mw, mh)
    assert np.array_equal(got["idx"][0].cpu().numpy(), ref_idx)
    sh2 = _t(np.concatenate([shift, np.zeros(3, np.float32)])[None], cuda)
    got2 = eod.ops.backproject_quantize(_t(depth[None], cuda), T[:, :3].reshape(1, 12).to(cuda), sh2, intr, cell, mw, mh, want_idx=False, want_outlier=True)
    assert np.array_equal(got2["outlier"][0].cpu().numpy().astype(bool), ref_out[0].numpy())
    for name, d_np in (("oracle", None),):
        o = oracle.backproject_quantize(depth, T[0].numpy(), intr, np.zeros(3, np.float32), shift, np.float32(cell), mw, mh, 0, 0.5, want=("idx",))
        assert np.array_equal(o["idx"], ref_idx)


def test_backproject_randomised_vs_oracle(eod, cuda):
    rng = np.random.default_rng(42)
    H, W, E = 60, 100, 5                                           # ragged: not multiples of the block size
    vfov = math.radians(67.5)
    intr = eod.compute_intrinsics(W, H, vfov)
    depth = rng.uniform(0.0, 10.0, (E, H, W)).astype(np.float32)
    depth[rng.uniform(size=depth.shape) < 0.05] = 0.0
    xyzhe = np.stack([rng.uniform(-5, 5, E), np.full(E, 1.25), rng.uniform(-5, 5, E), rng.uniform(0, 2 * np.pi, E),
                      np.pi + rng.uniform(-0.2, 0.2, E)], 1).astype(np.float32)
    T = eod.transform3d(torch.from_numpy(xyzhe))
    assert torch.equal(T, R.transform3d(torch.from_numpy(xyzhe)))
    shifts = np.concatenate([rng.uniform(-1, 1, (E, 3)), rng.uniform(-8, -2, (E, 3))], 1).astype(np.float32)
    for order in (0, 1):
        for cell, mw, mh in ((0.2, 37, 53), (0.02, 300, 200)):          # small maps: many out-of-map pixels on all sides
            r = eod.ops.backproject_quantize(_t(depth, cuda), T[:, :3].reshape(E, 12).to(cuda), _t(shifts, cuda), intr, cell, mw, mh,
                                             order, 0.5, want_q2=True, want_outlier=True, want_height=True, want_world=True)
            for e in range(E):
                o = oracle.backproject_quantize(depth[e], T[e].numpy(), intr, shifts[e, :3], shifts[e, 3:], cell, mw, mh, order, 0.5)
                for k in ("idx", "q2", "outlier", "height", "world"):
                    assert np.array_equal(r[k][e].cpu().numpy(), o[k]), (k, order, cell, e)
            assert r["outlier"].float().mean().item() > 0.1 and (r["q2"] < 0).any().item()


def test_projector_class_mirrors_reference_api(eod, cuda, golden):
    g = golden("geometry_small")
    T, H, W = g["depth"].shape
    pr = eod.Projector(float(g["vfov"]), 1, H, W, int(g["map_h"]), int(g["map_w"]), float(g["cell"]), g["map_world_shift"], 0.5, device=cuda)
    idx2d, outl, hts = pr.forward(torch.from_numpy(g["depth"][:, None]), torch.from_numpy(g["T"]), return_heights=True)
    assert idx2d.dtype == torch.int64 and outl.dtype == torch.bool
    assert np.array_equal(idx2d.cpu().numpy(), g["q2"]) and np.array_equal(outl.cpu().numpy(), g["outlier"])
    assert np.array_equal(hts.cpu().numpy(), g["height"])
    pc = eod.Projector(float(g["vfov"]), 1, H, W, int(g["map_h"]), int(g["map_w"]), float(g["cell"]), np.zeros(3), 0.5, device=cuda)
    world, nodepth = pc.point_cloud(torch.from_numpy(g["depth"][:, None]), torch.from_numpy(g["T"]))
    assert np.array_equal(world.cpu().numpy(), g["world"]) and np.array_equal(nodepth.cpu().numpy(), g["depth"] == 0)
    flat = pc.flat_indices(torch.from_numpy(g["depth"][:, None]), torch.from_numpy(g["T"]), g["map_world_shift"])
    assert flat.shape == (T, H, W, 1) and np.array_equal(flat[..., 0].cpu().numpy(), g["flat"])


# --------------------------------------------------------------------------------------------------------
# read (A10-A12) and fusion (A13)
# --------------------------------------------------------------------------------------------------------
def test_read_pool_matches_reference_golden(eod, cuda, golden):
    g = golden("read_fuse")
    sums, counts = _t(g["sums"], cuda), _t(g["counts"], cuda)
    mem16 = R.create_implicit_memory(torch.from_numpy(g["sums"]), torch.from_numpy(g["counts"])).to(torch.half)
    for t in range(2):
        idx = _t(g[f"idx{t}"], cuda)
        variants = {
            "fused f32+counts, i32": eod.ops.read_pool(sums[None], counts[None], idx[None]),
            "f16 table, i64": eod.ops.read_pool(mem16.to(cuda)[None].contiguous(), None, idx.long()[None].contiguous()),
            "f16 table, i32": eod.ops.read_pool(mem16.to(cuda)[None].contiguous(), None, idx[None]),
        }
        for name, levels in variants.items():
            for k in range(3):
                got = levels[k].contiguous().cpu().numpy().view(np.uint16)           # logical (1,C,h,w)
                assert got.shape == g[f"level{t}_{k}"].shape
                assert np.array_equal(got, g[f"level{t}_{k}"].view(np.uint16)), (name, t, k)
    norm = eod.ops.normalize_memory(sums, counts)
    assert np.array_equal(norm.cpu().numpy(), R.create_implicit_memory(torch.from_numpy(g["sums"]), torch.from_numpy(g["counts"])).numpy())
    assert np.array_equal(eod.ops.normalize_memory(sums, counts, half=True).cpu().numpy().view(np.uint16), mem16.numpy().view(np.uint16))


@pytest.mark.parametrize("C,E,H,W", [(128, 3, 64, 96), (256, 2, 96, 64), (512, 2, 32, 64)])
def test_read_pool_randomised_vs_oracle(eod, cuda, C, E, H, W):
    rng = np.random.default_rng(C)
    cells = 150
    sums = (rng.standard_normal((E, cells, C)) * rng.choice([1e-3, 1.0, 300.0], (E, cells, 1))).astype(np.float32)
    sums[:, :5] = -0.0                                                         # signed zeros survive the chain
    sums[:, 5:8] = 7e4                                                         # > fp16 max: rounds to inf like torch
    counts = rng.integers(0, 7, (E, cells)).astype(np.float32)
    # piecewise-constant index plane with ragged patches, like a real projection
    idx = (rng.integers(0, cells, (E, H // 4 + 1, W // 8 + 1)).repeat(4, 1).repeat(8, 2)[:, :H, :W]).astype(np.int32)
    idx[:, ::7, ::5] = rng.integers(0, cells, idx[:, ::7, ::5].shape)
    levels = eod.ops.read_pool(_t(sums, cuda), _t(counts, cuda), _t(idx, cuda))
    for e in range(E):
        ref = R.read_frame(torch.from_numpy(sums[e]), torch.from_numpy(counts[e]), torch.from_numpy(idx[e]))
        for k in range(3):
            a = levels[k][e].contiguous().cpu().numpy().view(np.uint16)
            b = ref[k][0].numpy().view(np.uint16)
            assert np.array_equal(a, b), (e, k, np.mean(a != b))


def test_read_pool_signed_zeros_and_adversarial_patterns(eod, cuda):
    """Patterns the randomised test does not reach (from profiles/stress_read.py): a table holding -0.0 (what a tiny negative
    feature becomes in fp16), subnormals and +-65504 in cells that fill whole 8x8 blocks - the reference's window sums start
    from +0, so a gathered -0.0 must come out as +0.0 -, checkerboards (16 runs per window) and 1-pixel stripes."""
    rng = np.random.default_rng(9)
    for C in (128, 256, 512):
        H, W, cells, E = 96, 128, 37, 2
        yy, xx = np.mgrid[0:H, 0:W]
        pats = [(yy // 24) * 7 % cells + (xx // 40) % 3, ((yy + xx) % 2) * (cells - 1), xx % cells, yy % cells]
        table = rng.standard_normal((E, cells, C)).astype(np.float16)
        table[:, :, :8] = np.array([0.0, -0.0, 6e-8, -6e-8, 65504.0, -65504.0, 1.0, -1.0], np.float16)
        table[:, :, 8:16] = np.float16(-1e-9)                               # underflows to -0.0
        for pat in pats:
            idx = np.stack([np.roll(pat, 5 * e, axis=1) for e in range(E)]).astype(np.int32) % cells
            got = eod.ops.read_pool(_t(table, cuda), None, _t(idx, cuda))
            for e in range(E):
                ref = oracle.read_pool_f16(table[e], idx[e])
                for k in range(3):
                    assert np.array_equal(got[k][e].contiguous().cpu().numpy().view(np.uint16), ref[k].view(np.uint16)), (C, e, k)


def test_explicit_map_read_mode(eod, cuda, golden):
    """MODEL.MEMORY_TYPE 'explicit_map' (SMNet/loader.py:233-246,298): memory = [zero row; (20,512) class table], proj_indices =
    (semmap + 1)[proj_indices].  The composed index plane must equal numpy's, and the read of the 21-row table (both as an fp16
    table and as fp32 without counts, through SpatialFeatureMemory.read_levels and MemoryFusion.read) must be bit-identical to
    timm.py:147-168 executed by torch-CPU on the same table (oracle R.read_pool); bad ids raise like the reference's gathers."""
    rng = np.random.default_rng(21)
    H, W, mw, mh, C, K = 96, 128, 70, 50, 512, 20
    clip = rng.standard_normal((K, C)).astype(np.float32)
    clip /= np.linalg.norm(clip, axis=1, keepdims=True)
    semmap = rng.integers(-1, K, (mw * mh,)).astype(np.int64)
    semmap[rng.random(mw * mh) < 0.5] = -1                                            # half the map is unobserved
    yy, xx = np.mgrid[0:H, 0:W]
    proj = ((yy // 5) * mw // 3 + xx // 3) % (mw * mh)
    proj[::9, ::7] = rng.integers(0, mw * mh, proj[::9, ::7].shape)
    obs = rng.integers(0, 5, (mw * mh,)).astype(np.float32)
    mem = eod.SpatialFeatureMemory(C, cuda)
    for idx_dtype, sm_dtype in ((np.int32, np.int64), (np.int64, np.int32), (np.int64, np.int64), (np.int32, np.int32)):
        frame = {"proj_indices": proj.astype(idx_dtype)[..., None], "observations": obs}
        memory, pidx, ego_obs = mem.create_explicit_memory(frame, torch.from_numpy(clip), torch.from_numpy(semmap.astype(sm_dtype)))
        ref_mem = np.insert(clip, 0, np.zeros((1, C)), axis=0).astype(np.float32)      # loader.py:233-235
        ref_idx = (semmap + 1)[proj]                                                  # loader.py:222,242
        assert memory.shape == (K + 1, C) and np.array_equal(memory.cpu().numpy(), ref_mem)
        assert pidx.dtype == torch.int32 and np.array_equal(pidx.cpu().numpy(), ref_idx)
        assert np.array_equal(ego_obs.cpu().numpy(), obs[proj])
    ref = R.read_pool(torch.from_numpy(ref_mem).half(), torch.from_numpy(ref_idx))
    fus = eod.MemoryFusion("implicit_memory", "sum", 5, mem_feat_dim=C, ego_feat_dim=256).to(cuda)
    for name, levels in (("read_levels f16", mem.read_levels(pidx, memory.half())),
                         ("read_levels f32 no counts", mem.read_levels(pidx, memory)),
                         ("MemoryFusion.read", fus.read([memory.half()], [pidx]))):
        for k in range(3):
            assert np.array_equal(levels[k][0].contiguous().cpu().numpy().view(np.uint16), ref[k][0].numpy().view(np.uint16)), (name, k)
    # the same inputs went through the reference's own source (tests/golden/make_golden.py --only-explicit-map): identical outputs
    g = golden("explicit_map")
    assert np.array_equal(g["semmap"], semmap) and np.array_equal(g["proj"], proj) and np.array_equal(g["clip"], clip)
    assert np.array_equal(memory.cpu().numpy(), g["memory"]) and np.array_equal(pidx.cpu().numpy(), g["idx"])
    got = mem.read_levels(pidx, memory.half())
    for k in range(3):
        assert np.array_equal(got[k].contiguous().cpu().numpy().view(np.uint16), g[f"level{k}"].view(np.uint16)), k
    bad = semmap.copy()
    bad[proj[3, 3]] = K + 5                                                           # class outside the table
    with pytest.raises(IndexError):
        mem.create_explicit_memory({"proj_indices": proj}, torch.from_numpy(clip), torch.from_numpy(bad))
    badp = proj.copy()
    badp[0, 0] = mw * mh                                                              # cell outside the map
    with pytest.raises(IndexError):
        mem.create_explicit_memory({"proj_indices": badp}, torch.from_numpy(clip), torch.from_numpy(semmap))


def test_fuse_bit_exact(eod, cuda):
    rng = np.random.default_rng(1)
    assert fuse_trips(FUSE_N, device_sms()) > 1
    for n in (1, 3, 4, 1000, 256 * 60 * 80 + 3, FUSE_N):              # FUSE_N: past the grid cap, so the grid-stride loop turns
        res = rng.standard_normal(n).astype(np.float32)
        mem = (rng.standard_normal(n) * 10).astype(np.float32)
        for w in (5.0, 500.0, 0.3):
            exp = {0: torch.from_numpy(mem) * w + torch.from_numpy(res), 1: torch.from_numpy(mem) * w, 2: torch.from_numpy(res)}
            for mode in (0, 1, 2):
                out = eod.ops.fuse(_t(res, cuda), _t(mem, cuda), w, mode)
                assert np.array_equal(out.cpu().numpy(), exp[mode].numpy()), (n, w, mode)


def test_memory_fusion_module_matches_reference_golden(eod, cuda, golden):
    g = golden("read_fuse")
    C, CO = g["sums"].shape[1], g["w0"].shape[0]
    mem16 = R.create_implicit_memory(torch.from_numpy(g["sums"]), torch.from_numpy(g["counts"])).to(torch.half)
    for fusion in ("sum", "mem_only", "image_only"):
        mod = eod.MemoryFusion("implicit_memory", fusion, 5, mem_feat_dim=C, ego_feat_dim=CO).to(cuda)
        sd = {f"map_merge_projection{k + 1}.{p}": torch.from_numpy(g[f"{q}{k}"]) for k in range(3) for p, q in (("weight", "w"), ("bias", "b"))}
        mod.load_state_dict(sd)
        res = [_t(g[f"res0_{k}"], cuda, torch.float32) for k in range(3)]
        idx = _t(g["idx0"], cuda).long()
        with torch.no_grad():
            out_ref_api = mod(res, [mem16.to(cuda)], [idx], [None])                          # reference call surface
            out_fused = mod(res, [_t(g["sums"], cuda)], [idx], [_t(g["counts"], cuda)])      # fp32 sums + counts
        for out in (out_ref_api, out_fused):
            for k in range(3):
                ref = g[f"fused_{fusion}_0_{k}"]
                assert out[k].shape == ref.shape
                assert np.abs(out[k].cpu().numpy() - ref).max() <= SUM_TOL * np.abs(ref).max(), (fusion, k)
    bad = eod.MemoryFusion("implicit_memory", "ave", 5, mem_feat_dim=C, ego_feat_dim=CO).to(cuda)
    with pytest.raises(UnboundLocalError):
        bad([_t(g[f"res0_{k}"], cuda, torch.float32) for k in range(3)], [mem16.to(cuda)], [_t(g["idx0"], cuda).long()], [None])


@pytest.mark.parametrize("E,h,w,K,N", [(2, 60, 80, 512, 256), (3, 15, 20, 512, 256), (1, 30, 40, 256, 128), (5, 7, 9, 64, 128)])
def test_project_fuse_tensor_core_vs_fp64(eod, cuda, E, h, w, K, N):
    """eod_project_fuse (tcgen05, fp16 level x hi/lo-split fp32 weight) against the fp64 evaluation of timm.py:174-184.
    Tolerance: 1e-5 of the output scale (north star, fp32 accumulations); it must also be as accurate as the fp32 library
    path (torch-CPU matmul of the same operands) up to a small factor - i.e. the split loses nothing that fp32 keeps.
    Tiles with a ragged tail (M % 128 != 0), rows that straddle episodes, bias on/off, sum / mem_only."""
    rng = np.random.default_rng(E * 100 + K)
    x16 = (rng.standard_normal((E, h, w, K)) * 3).astype(np.float16)
    W = (rng.uniform(-1, 1, (N, K)) / math.sqrt(K)).astype(np.float32)
    W[0, :8] = [1e-6, -3e-7, 0.0, 6e-5, 123.456, -1e-3, 2 ** -14, 65504.0]      # sub-fp16-normal, large, exact powers
    b = rng.standard_normal(N).astype(np.float32)
    res = (rng.standard_normal((E, N, h, w)) * 2).astype(np.float32)
    wsplit = eod.ops.project_split_weights(_t(W, cuda))
    lvl = _t(x16, cuda).permute(0, 3, 1, 2)                                      # logical NCHW, channels-last memory
    x64 = torch.from_numpy(x16.astype(np.float64)).reshape(-1, K)
    for weight in (5.0, 500.0):
        for mode, bias in ((0, b), (1, b), (0, None)):
            got = eod.ops.project_fuse(lvl, wsplit, None if bias is None else _t(bias, cuda), _t(res, cuda) if mode == 0 else None, weight, mode)
            variants = [1] + ([2] if (h * w) % 4 == 0 else [])          # tile-per-CTA kernel; persistent kernel (TMA on res: hw % 4 == 0)
            for variant in variants:
                alt = eod.ops.project_fuse_levels([lvl], [wsplit], [None if bias is None else _t(bias, cuda)], [_t(res, cuda)] if mode == 0 else None,
                                                  weight, mode, variant=variant)[0]
                assert (alt.cpu().double() - got.cpu().double()).abs().max().item() <= 2e-6 * got.abs().max().item(), (variant, weight, mode)
            mem64 = x64 @ torch.from_numpy(W.astype(np.float64)).t() + (0 if bias is None else torch.from_numpy(bias.astype(np.float64)))
            mem64 = mem64.reshape(E, h, w, N).permute(0, 3, 1, 2) * weight
            ref64 = (mem64 + torch.from_numpy(res.astype(np.float64))) if mode == 0 else mem64
            mem32 = torch.from_numpy(x16.astype(np.float32)).reshape(-1, K) @ torch.from_numpy(W).t()
            if bias is not None:
                mem32 = mem32 + torch.from_numpy(bias)
            mem32 = mem32.reshape(E, h, w, N).permute(0, 3, 1, 2) * weight
            ref32 = (mem32 + torch.from_numpy(res)) if mode == 0 else mem32
            scale = ref64.abs().max().item()
            err = (got.cpu().double() - ref64).abs().max().item()
            err32 = (ref32.double() - ref64).abs().max().item()
            assert err <= SUM_TOL * scale, (weight, mode, err / scale)
            assert err <= 4 * err32 + 1e-7 * scale, (weight, mode, err, err32)
    with pytest.raises(eod.EodError):
        eod.ops.project_fuse(lvl, wsplit, None, None, 5.0, 0)                    # sum needs res


def test_project_fuse_all_levels_one_launch(eod, cuda):
    """The persistent kernel over the three pyramid levels of E episodes (tiles never straddle episodes; the last tile of an
    episode is ragged: 4800 = 18.75 x 256, 1200, 300) against fp64, and the multi-level launch against per-level launches."""
    rng = np.random.default_rng(99)
    E, K, N = 5, 512, 256
    shapes = [(60, 80), (30, 40), (15, 20)]
    lv = [_t((rng.standard_normal((E, h, w, K)) * 2).astype(np.float16), cuda) for h, w in shapes]
    Ws = [(rng.uniform(-1, 1, (N, K)) / math.sqrt(K)).astype(np.float32) for _ in shapes]
    bs = [rng.standard_normal(N).astype(np.float32) for _ in shapes]
    rs = [rng.standard_normal((E, N, h, w)).astype(np.float32) for h, w in shapes]
    ws = [eod.ops.project_split_weights(_t(W, cuda)) for W in Ws]
    for mode in (0, 1):
        res_d = [_t(r, cuda) for r in rs] if mode == 0 else None
        outs = eod.ops.project_fuse_levels(lv, ws, [_t(b, cuda) for b in bs], res_d, 5.0, mode, variant=2)
        for k, (h, w) in enumerate(shapes):
            x64 = lv[k].cpu().double().reshape(-1, K)
            ref = (x64 @ torch.from_numpy(Ws[k].astype(np.float64)).t() + torch.from_numpy(bs[k].astype(np.float64))).reshape(E, h, w, N).permute(0, 3, 1, 2) * 5.0
            if mode == 0:
                ref = ref + torch.from_numpy(rs[k].astype(np.float64))
            err = (outs[k].cpu().double() - ref).abs().max().item()
            assert err <= SUM_TOL * ref.abs().max().item(), (mode, k, err)
            single = eod.ops.project_fuse_levels([lv[k]], [ws[k]], [_t(bs[k], cuda)], None if mode else [res_d[k]], 5.0, mode, variant=2)[0]
            assert torch.equal(single, outs[k]), (mode, k)          # same tile arithmetic whether launched alone or together


def test_project_fuse_persistent_many_tiles_per_cta_equals_tile_kernel(eod, cuda):
    """Regression for a ring-release race: with several tiles per CTA the persistent kernel must reproduce the
    tile-per-CTA kernel BIT FOR BIT (same UMMA sequence per tile, same epilogue arithmetic), for sum and mem_only, repeatedly."""
    rng = np.random.default_rng(7)
    E, K, N = 24, 512, 256
    shapes = [(60, 80), (30, 40), (15, 20)]
    lv = [_t((rng.standard_normal((E, h, w, K)) * 2).astype(np.float16), cuda) for h, w in shapes]
    ws = [eod.ops.project_split_weights(_t((rng.uniform(-1, 1, (N, K)) / math.sqrt(K)).astype(np.float32), cuda)) for _ in shapes]
    bs = [_t(rng.standard_normal(N).astype(np.float32), cuda) for _ in shapes]
    rs = [_t(rng.standard_normal((E, N, h, w)).astype(np.float32), cuda) for h, w in shapes]
    for mode in (0, 1):
        ref = eod.ops.project_fuse_levels(lv, ws, bs, rs if mode == 0 else None, 5.0, mode, variant=1)
        for rep in range(4):
            got = eod.ops.project_fuse_levels(lv, ws, bs, rs if mode == 0 else None, 5.0, mode, variant=2)
            for k in range(3):
                assert torch.equal(got[k], ref[k]), (mode, rep, k, int((got[k] != ref[k]).sum()))


def test_memory_fusion_tensor_core_and_library_paths_agree(eod, cuda):
    """MemoryFusion forward: the tcgen05 path (inference) and the library-GEMM + eod_fuse path (tensor_core=False) agree
    to the fp32 tolerance on all three levels; with gradients enabled the module takes the autograd path and the
    gradients of the map_merge parameters match a plain-torch restatement (custom_rcnn.py:609-613 trains them)."""
    rng = np.random.default_rng(12)
    C, CO, H, W, cells = 512, 256, 96, 128, 900
    mem16 = _t((rng.standard_normal((cells, C)) * 4).astype(np.float16), cuda)
    idx = _t(rng.integers(0, cells, (H, W)).astype(np.int64), cuda)
    res = [_t(rng.standard_normal((1, CO, H >> s, W >> s)).astype(np.float32), cuda) for s in (3, 4, 5)]
    tc = eod.MemoryFusion("implicit_memory", "sum", 5, mem_feat_dim=C, ego_feat_dim=CO).to(cuda)
    lib = eod.MemoryFusion("implicit_memory", "sum", 5, mem_feat_dim=C, ego_feat_dim=CO, tensor_core=False).to(cuda)
    lib.load_state_dict(tc.state_dict())
    before = eod.ops.launch_count
    with torch.no_grad():
        a = tc(res, [mem16], [idx], [None])
        assert eod.ops.launch_count - before == 1 + 2 + 3 + 1    # index range check + read (L0/L1 + L2 pooling) + 3 weight splits + ONE fused projection launch
        a2 = tc(res, [mem16], [idx], [None])                     # weights unchanged: split cached
        assert eod.ops.launch_count - before == 1 + 2 + 3 + 1 + 1 + 2 + 1
        tc.validate_indices = False                              # planes that eod_backproject_quantize produced for this grid need no check
        tc(res, [mem16], [idx], [None])
        assert eod.ops.launch_count - before == 1 + 2 + 3 + 1 + 1 + 2 + 1 + 2 + 1
        tc.validate_indices = True
        b = lib(res, [mem16], [idx], [None])
    for k in range(3):
        assert torch.equal(a[k], a2[k])
        assert (a[k] - b[k]).abs().max().item() <= SUM_TOL * b[k].abs().max().item(), k
    # training path: gradients flow to the projection parameters and to res
    res_g = [r.clone().requires_grad_(True) for r in res]
    out = tc(res_g, [mem16], [idx], [None])
    loss = sum((o * o).sum() for o in out)
    loss.backward()
    levels = tc.read([mem16], [idx], [None])
    for k, conv in enumerate(tc.merge_map_projections):                       # plain-torch restatement on the CPU in fp64
        w = conv.weight.detach().cpu().double().requires_grad_(True)
        bb = conv.bias.detach().cpu().double().requires_grad_(True)
        r = res[k].cpu().double().requires_grad_(True)
        o = r + 5.0 * torch.nn.functional.conv2d(levels[k].cpu().double(), w, bb)
        (o * o).sum().backward()
        for got, ref in ((conv.weight.grad, w.grad), (conv.bias.grad, bb.grad), (res_g[k].grad, r.grad)):
            assert (got.cpu().double() - ref).abs().max().item() <= 1e-5 * ref.abs().max().item(), k


# --------------------------------------------------------------------------------------------------------
# write, mean mode (A6-A8)
# --------------------------------------------------------------------------------------------------------
def test_sample_mask_and_box_features_bit_exact(eod, cuda):
    rng = np.random.default_rng(3)
    H, W, C = 48, 80, 64
    # plane sizes: 16-pixel vectorised scan (one and several 16 KB steps, ragged last step) and the scalar kernel (HW % 16 != 0)
    for hw in (H * W, 480 * 640, 16 * 1025, 47 * 81):
        for stride in (1, 3, 8):
            obs = rng.uniform(size=(3, hw)) < rng.uniform(0.0, 0.9)
            obs[2] = False                                                 # empty: nothing observed
            obs_u8 = obs.view(np.uint8) * rng.integers(1, 256, obs.shape).astype(np.uint8)      # any non-zero byte counts as observed
            n = torch.zeros(3, dtype=torch.int32, device=cuda)
            samp = eod.ops.sample_mask(_t(obs_u8, cuda), stride, n_sampled=n)
            for e in range(3):
                ref = R.sample_mask(torch.from_numpy(obs[e]), stride).numpy()
                assert np.array_equal(samp[e].cpu().numpy(), ref.astype(np.uint8)), (hw, stride, e)
                assert int(n[e]) == int(ref.sum())
    bf, masks = eod.episodes.make_detections(rng, H, W, C, (7, 9))
    img, observed = eod.ops.box_to_image_features(_t(bf, cuda), _t(masks, cuda))
    ref_img, ref_obs = R.box_to_image_features(torch.from_numpy(bf), torch.from_numpy(masks))
    assert np.array_equal(observed.cpu().numpy(), ref_obs.numpy())
    assert np.array_equal(img.cpu().numpy(), ref_img.numpy())              # same fp32 add order -> bit-exact


def _write_case(eod, cuda, C, E, H, W, cells, layout, variant, with_samp, seed, expand=False):
    rng = np.random.default_rng(seed)
    HW = H * W
    feat = rng.standard_normal((E, C, H, W)).astype(np.float32) * 3
    if layout in (2, 3):        # 16-bit channels-last features: the oracle sums the exactly widened values
        feat = torch.from_numpy(feat).to(torch.bfloat16 if layout == 2 else torch.float16).float().numpy()
    idx = (rng.integers(0, cells, (E, H // 2 + 1, W // 16 + 1)).repeat(2, 1).repeat(16, 2)[:, :H, :W]).astype(np.int32)
    idx[:, ::5, ::3] = rng.integers(0, cells, idx[:, ::5, ::3].shape)
    samp = (rng.uniform(size=(E, H, W)) < 0.3).astype(np.uint8) if with_samp else None
    if with_samp:
        samp[0, : H // 2] = 0                                              # whole tiles without a sampled pixel
    sums0 = rng.standard_normal((E, cells, C)).astype(np.float32)
    counts0 = rng.integers(0, 4, (E, cells)).astype(np.float32)
    d_sums, d_counts = _t(sums0, cuda), _t(counts0, cuda)
    d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    d_touched = torch.zeros((E, cells), dtype=torch.uint8, device=cuda)
    d_idx = _t(idx, cuda)
    d_samp = None if samp is None else _t(samp, cuda)
    f_dev = _t(feat if layout == 0 else feat.transpose(0, 2, 3, 1), cuda)
    if layout in (2, 3):
        f_dev = f_dev.to(torch.bfloat16 if layout == 2 else torch.float16)
    eod.ops.frame_count(d_idx, d_samp, d_cnt)
    pix = eod.ops.expand_counts(d_idx, d_cnt, torch.empty((E, H, W), device=cuda)) if expand else None
    eod.ops.write_mean(f_dev, d_idx, d_samp, d_cnt, d_sums, layout, variant, pix)
    d_norm = torch.zeros((E, cells, C), dtype=torch.float16, device=cuda)
    eod.ops.finalize_counts(d_idx, d_cnt, d_counts, d_touched, d_sums, d_norm)
    torch.cuda.synchronize()
    assert int(d_cnt.abs().sum()) == 0                                     # scratch returned to zero
    for e in range(E):                                                     # refreshed fp16 rows: exactly the visible cells
        vis = np.unique(idx[e])
        ref16 = R.create_implicit_memory(d_sums[e].cpu(), d_counts[e].cpu()).half().numpy()
        got16 = d_norm[e].cpu().numpy()
        assert np.array_equal(got16[vis].view(np.uint16), ref16[vis].view(np.uint16))
        hidden = np.setdiff1d(np.arange(cells), vis)
        assert not got16[hidden].any()
    for e in range(E):
        s, n = oracle.cell_sums_seq(feat[e], idx[e], None if samp is None else samp[e], cells)
        mean = np.where(n[:, None] > 0, s / np.maximum(n, 1)[:, None].astype(np.float32), 0).astype(np.float32)
        ref = sums0[e] + mean
        got = d_sums[e].cpu().numpy()
        assert np.abs(got - ref).max() <= SUM_TOL * np.abs(ref).max(), (e, np.abs(got - ref).max())
        untouched = n == 0
        assert np.array_equal(got[untouched], sums0[e][untouched])         # cells without samples are not written at all
        vis = np.zeros(cells, np.float32)
        vis[np.unique(idx[e])] = 1
        assert np.array_equal(d_counts[e].cpu().numpy(), counts0[e] + vis)
        assert np.array_equal(d_touched[e].cpu().numpy().astype(bool), n > 0)


@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("variant,expand", [(1, False), (2, False), (2, True)], ids=["ldg", "tma", "tma+expand"])   # EOD_WRITE_LDG, EOD_WRITE_TMA
@pytest.mark.parametrize("with_samp", [False, True])
def test_write_mean_chw_vs_oracle(eod, cuda, C, variant, expand, with_samp):
    _write_case(eod, cuda, C, 3, 64, 96, 200, 0, variant, with_samp, seed=C + variant, expand=expand)


@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("with_samp", [False, True])
def test_write_mean_det_reproducible_and_correct(eod, cuda, C, with_samp):
    """EOD_WRITE_DET: bitwise reproducible run to run and under a different batching of the same episodes; within the
    fp32 tolerance of the oracle; cells without samples untouched; an undersized workspace degrades to the atomic path
    (flagged) without losing correctness."""
    rng = np.random.default_rng(40 + C)
    E, H, W, cells = 3, 64, 96, 211
    feat = rng.standard_normal((E, C, H, W)).astype(np.float32) * 3
    idx = (rng.integers(0, cells, (E, H // 2 + 1, W // 16 + 1)).repeat(2, 1).repeat(16, 2)[:, :H, :W]).astype(np.int32)
    idx[:, ::5, ::3] = rng.integers(0, cells, idx[:, ::5, ::3].shape)
    idx[0, :8] = 7                                                         # one long segment: > 32 runs in a cell
    samp = (rng.uniform(size=(E, H, W)) < 0.3).astype(np.uint8) if with_samp else None
    sums0 = rng.standard_normal((E, cells, C)).astype(np.float32)

    def run(order, runs_per_episode=0):
        order = list(order)
        d_idx = _t(idx[order], cuda)
        d_samp = None if samp is None else _t(samp[order], cuda)
        d_sums = _t(sums0[order], cuda)
        d_cnt = torch.zeros((len(order), cells), dtype=torch.int32, device=cuda)
        ws = eod.ops.DetWorkspace(len(order), C, H * W, cells, cuda, runs_per_episode)
        eod.ops.frame_count(d_idx, d_samp, d_cnt)
        eod.ops.write_mean_det(_t(feat[order], cuda), d_idx, d_samp, d_cnt, d_sums, ws)
        out1 = d_sums.clone()                                              # second call: the workspace is reusable as left behind
        d_sums.copy_(_t(sums0[order], cuda))
        eod.ops.write_mean_det(_t(feat[order], cuda), d_idx, d_samp, d_cnt, d_sums, ws)
        torch.cuda.synchronize()
        if not runs_per_episode:
            assert torch.equal(out1, d_sums)                               # run to run: bitwise (unless runs overflowed to atomics)
        inv = np.argsort(order)
        return d_sums.cpu().numpy()[inv], ws.overflowed()

    a, ovf = run(range(E))
    assert not ovf
    b, _ = run([2, 0, 1])
    assert np.array_equal(a, b)                                            # batching order: bitwise
    c, _ = run([1])
    assert np.array_equal(a[1:2], c)                                       # an episode alone: bitwise
    small, ovf = run(range(E), runs_per_episode=5)
    assert ovf
    for e in range(E):
        s_, n = oracle.cell_sums_seq(feat[e], idx[e], None if samp is None else samp[e], cells)
        mean = np.where(n[:, None] > 0, s_ / np.maximum(n, 1)[:, None].astype(np.float32), 0).astype(np.float32)
        ref = sums0[e] + mean
        for got in (a[e], small[e]):
            assert np.abs(got - ref).max() <= SUM_TOL * np.abs(ref).max()
            assert np.array_equal(got[n == 0], sums0[e][n == 0])


def test_write_mean_det_very_long_segment(eod, cuda):
    """A cell with more runs than a warp sorts in shared memory at once (2048) takes the bitmap-sort path of det_reduce and the
    chunked summation (det_chunk / det_final)."""
    rng = np.random.default_rng(77)
    E, C, H, W, cells = 1, 128, 64, 96, 50
    feat = rng.standard_normal((E, C, H, W)).astype(np.float32)
    idx = rng.integers(8, cells, (E, H, W)).astype(np.int32)
    idx[0, :50, ::2] = 7                                                    # 50 rows x 48 isolated pixels = 2400 runs of cell 7
    d_idx, d_feat = _t(idx, cuda), _t(feat, cuda)
    d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
    eod.ops.frame_count(d_idx, None, d_cnt)
    ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda, H * W)
    outs = []
    for _ in range(2):
        d_sums = torch.zeros((E, cells, C), device=cuda)
        eod.ops.write_mean_det(d_feat, d_idx, None, d_cnt, d_sums, ws)
        outs.append(d_sums)
    torch.cuda.synchronize()
    assert not ws.overflowed() and torch.equal(outs[0], outs[1])
    s_, n = oracle.cell_sums_seq(feat[0], idx[0], None, cells)
    ref = np.where(n[:, None] > 0, s_ / np.maximum(n, 1)[:, None].astype(np.float32), 0).astype(np.float32)
    assert n[7] == 2400
    assert np.abs(outs[0][0].cpu().numpy() - ref).max() <= SUM_TOL * np.abs(ref).max()


def test_write_mean_det_bitmap_sort_many_passes_and_batch_independence(eod, cuda):
    """More than 65 536 runs in one episode (the bitmap sort of a long segment needs several passes), two cells with ~77 k runs
    each and a third long one; the result must be bitwise identical run to run AND when the episode sits at another place of
    a larger batch (fixed per-cell summation tree: sorted runs -> chunks of 128 -> chunk sums in order)."""
    rng = np.random.default_rng(5)
    C, H, W, cells = 128, 480, 640, 40
    feat = rng.standard_normal((1, C, H, W)).astype(np.float32)
    idx = np.empty((1, H, W), np.int32)
    idx[0] = 3 + ((np.arange(W) // 2) % 2)[None, :]                          # runs of 2 px alternating cells 3 / 4: 153 600 runs
    idx[0, 100:140, ::4] = 9                                                  # + 6 400 isolated pixels of cell 9
    ref_s, n = oracle.cell_sums_seq(feat[0], idx[0], None, cells)
    ref = np.where(n[:, None] > 0, ref_s / np.maximum(n, 1)[:, None].astype(np.float32), 0).astype(np.float32)
    outs = []
    for E, slot in ((1, 0), (1, 0), (3, 2)):
        f = rng.standard_normal((E, C, H, W)).astype(np.float32)
        ix = rng.integers(10, cells, (E, H, W)).astype(np.int32)
        f[slot], ix[slot] = feat[0], idx[0]
        d_idx, d_feat = _t(ix, cuda), _t(f, cuda)
        d_cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
        eod.ops.frame_count(d_idx, None, d_cnt)
        ws = eod.ops.DetWorkspace(E, C, H * W, cells, cuda, H * W)            # one run per pixel fits
        d_sums = torch.zeros((E, cells, C), device=cuda)
        eod.ops.write_mean_det(d_feat, d_idx, None, d_cnt, d_sums, ws)
        torch.cuda.synchronize()
        assert not ws.overflowed()
        outs.append(d_sums[slot].clone())
        del ws, d_feat
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    assert np.abs(outs[0].cpu().numpy() - ref).max() <= SUM_TOL * np.abs(ref).max()


def test_episode_batch_deterministic_variant(eod, cuda):
    """EpisodeBatch(variant=WRITE_DET) end to end: two identical runs give identical bits (sums, norm16, levels)."""
    E, C, H, W, mw, mh, T_ = 2, 128, 96, 128, 60, 45, 4
    eps = [eod.episodes.make_episode(700 + e, T_, H, W, mw, mh, 0.2) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    gen = torch.Generator(device=cuda).manual_seed(11)
    feat = [torch.randn((E, C, H, W), device=cuda, generator=gen) for _ in range(T_)]
    outs = []
    for rep in range(2):
        batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, variant=4, pipeline=bool(rep))
        batch.det_runs_per_episode = H * W                 # low resolution: a run is ~3 pixels, more than the default HW/4 runs
        lv = []
        for t in range(T_):
            depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
            pose = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))[:, :3].reshape(E, 12).to(cuda)
            torch.cuda.synchronize()
            lv.append([l.clone() for l in batch.step(depth, pose, shifts, intr, 0.2, feat[t])])
        batch.join()
        torch.cuda.synchronize()
        assert not batch._det_ws.overflowed()
        outs.append((batch.sums.clone(), batch.counts.clone(), batch.norm16.clone(), lv))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]) and torch.equal(outs[0][2], outs[1][2])
    for t in range(T_):
        for a, b in zip(outs[0][3][t], outs[1][3][t]):
            assert torch.equal(a, b)
    assert outs[0][0].abs().sum().item() > 0


def test_write_mean_large_grid_pixel_driven_finalize(eod, cuda):
    """cells > 4*HW: eod_finalize_counts walks the pixel plane (atomicExch dedupe) instead of the cell plane;
    E*tiles odd -> the TMA kernel falls back to ungrouped tiles."""
    _write_case(eod, cuda, 128, 3, 32, 96, 13000, 0, 2, True, seed=5, expand=True)
    _write_case(eod, cuda, 256, 1, 32, 32, 5000, 0, 2, False, seed=6, expand=True)


def test_write_mean_chw_ragged_tail_ldg(eod, cuda):
    _write_case(eod, cuda, 256, 2, 30, 52, 90, 0, 0, True, seed=9)        # HW % 32 != 0 -> AUTO picks the LDG kernel


@pytest.mark.parametrize("C", [128, 256, 512])
@pytest.mark.parametrize("layout", [1, 2, 3], ids=["f32", "bf16", "f16"])      # EOD_LAYOUT_HWC, _HWC_BF16, _HWC_F16
def test_write_mean_hwc_vs_oracle(eod, cuda, C, layout):
    _write_case(eod, cuda, C, 2, 30, 52, 90, layout, 0, True, seed=C)
    _write_case(eod, cuda, C, 2, 64, 96, 200, layout, 0, False, seed=C + 1)


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "image-buffer"])
def test_write_path_matches_reference_golden(eod, cuda, golden, fused):
    """Reference call surface (box_to_image_features / project_image_features / update_implicit_memory) against the
    outputs of the reference's own source over a 3-frame sequence."""
    g = golden("write_mean")
    n_cells = int(g["map_w"]) * int(g["map_h"])
    mem = eod.SpatialFeatureMemory(512, cuda, fused_write=fused)
    mem.reset(n_cells)
    for t in range(3):
        K = int(g[f"K{t}"])
        masks = _t(_unpack(g[f"masks{t}"], (K, 480, 640)), cuda)
        bf = _t(g[f"box_features{t}"], cuda)
        proj = _t(g[f"idx{t}"], cuda).long()
        img, observed = mem.box_to_image_features(bf, masks)
        assert np.array_equal(observed.cpu().numpy(), _unpack(g[f"observed{t}"], (480, 640)))
        assert np.array_equal(img[0, :, ::16, ::16].cpu().numpy(), g[f"img_sample{t}"])
        assert np.allclose(img.double().sum(dim=(0, 2, 3)).cpu().numpy(), g[f"img_checksum{t}"], rtol=1e-9)
        mean, observed_mem = mem.project_image_features(img, observed, [proj], [mem.implicit_memory])
        assert np.array_equal(observed_mem.cpu().numpy(), g[f"observed_mem{t}"])              # touched-cell set: exact
        assert np.abs(mean.cpu().numpy() - g[f"mean{t}"]).max() <= SUM_TOL * np.abs(g[f"mean{t}"]).max()
        mem.update_implicit_memory((None, bf, masks, None), proj, mem.implicit_memory, {"sequence_name": "synthetic"})
        assert np.abs(mem.implicit_memory.cpu().numpy() - g[f"sums{t}"]).max() <= SUM_TOL * np.abs(g[f"sums{t}"]).max()
        assert np.array_equal(mem.observations.cpu().numpy(), g[f"counts{t}"])                # visibility counts: exact
        norm, _ = mem.create_implicit_memory({"memory": torch.from_numpy(g[f"sums{t}"]), "observations": torch.from_numpy(g[f"counts{t}"]), "proj_indices": proj})
        assert np.array_equal(norm.cpu().numpy(), g[f"norm{t}"])
    before = mem.implicit_memory.clone()
    mem.update_implicit_memory(None, proj, mem.implicit_memory, {})                           # no detection -> no write (:686)
    assert torch.equal(before, mem.implicit_memory)


def test_explicit_semmap_matches_reference_golden(eod, cuda, golden):
    """semmap kernels on the reference-generated fixture (custom_rcnn.py:747-756,938-978 executed from source): labels
    equal except on rounding edges of the intensity threshold / the top-2 logits."""
    g = golden("semmap")
    sums, counts, zs = (torch.from_numpy(g[k]) for k in ("sums", "counts", "zs_weight"))
    cells = sums.shape[0]
    inten = torch.zeros((1, cells), device=cuda)
    cls = torch.zeros((1, cells), dtype=torch.int32, device=cuda)
    vis = torch.ones((1, cells), dtype=torch.int32, device=cuda)            # every cell "visible": full refresh
    eod.ops.semmap_update(vis, (counts - 1).to(cuda)[None].contiguous(), sums.to(cuda)[None].contiguous(), zs.to(cuda), 20, inten, cls)
    for th in (0.4, 0.1):
        got = eod.ops.semmap_decode(inten, cls, th)[0].cpu().numpy()
        _, ref_inten, scores = R.explicit_semmap(sums, counts, zs, th)
        top2 = scores.topk(2, dim=1).values
        edge = ((ref_inten - th).abs() < 1e-5) | ((top2[:, 0] - top2[:, 1]).abs() < 1e-4)
        ok = (got == g[f"semmap_{th}"]) | edge.numpy()
        assert ok.all(), int((~ok).sum())
        assert int((edge & (counts > 0)).sum()) < 0.01 * cells              # all-zero rows tie on every logit by construction


def test_explicit_semmap_incremental_vs_oracle(eod, cuda):
    """A14: the incrementally maintained explicit map equals the reference's full-grid recomputation
    (custom_rcnn.py:747-756,938-978) after every frame, except where a decision sits on a rounding edge
    (normalised intensity within 1e-5 of the threshold, or top-2 logits closer than 1e-4)."""
    H, W, C, mw, mh, K = 96, 128, 512, 40, 30, 21
    cells = mw * mh
    rng = np.random.default_rng(33)
    zs = torch.from_numpy(rng.standard_normal((C, K)).astype(np.float32))
    zs = zs / zs.norm(dim=0, keepdim=True)
    mem = eod.SpatialFeatureMemory(C, cuda, zs_weight=zs, obs_score_thresh=0.4)
    mem.reset(cells)
    assert (mem.semmap.cpu().numpy() == 0).all()                             # constant intensity: 0/0 -> NaN < thresh is False (reference too)
    sums, counts = torch.zeros(cells, C), torch.zeros(cells)
    for t in range(4):
        idx = (rng.integers(0, cells // 2, (H // 4 + 1, W // 8 + 1)).repeat(4, 0).repeat(8, 1)[:H, :W]).astype(np.int32)
        bf, masks = eod.episodes.make_detections(rng, H, W, C, (5, 9))
        proj = torch.from_numpy(idx).long()
        mem.update_implicit_memory((None, _t(bf, cuda), _t(masks, cuda), None), proj.to(cuda), mem.implicit_memory, {})
        img, obs = R.box_to_image_features(torch.from_numpy(bf), torch.from_numpy(masks))
        sums, counts = R.write_mean_frame(sums, counts, img, obs, proj, stride=8)
        # oracle on the GPU state (the sums agree to 1e-5; the decode is what is under test here)
        ref, inten, scores = R.explicit_semmap(mem.implicit_memory.cpu(), mem.observations.cpu(), zs, 0.4)
        got = mem.semmap.cpu().numpy()
        top2 = scores.topk(2, dim=1).values
        edge = ((inten - 0.4).abs() < 1e-5) | ((top2[:, 0] - top2[:, 1]).abs() < 1e-4)
        ok = (got == ref.numpy()) | edge.numpy()
        assert ok.all(), (t, int((~ok).sum()))
        assert (got >= 0).sum() > 0 and (got == -1).sum() > 0                # both outcomes occur
        assert (mem.implicit_memory.cpu() - sums).abs().max().item() <= SUM_TOL * sums.abs().max().item()


def test_batched_fused_object_write_vs_oracle(eod, cuda):
    """EpisodeBatch.write_objects (masks -> observed -> every 8th -> per-cell mean, no image buffer) against the
    restated reference chain box_to_image_features -> project_image_features -> accumulate, per episode; an episode
    without detections must not change at all (custom_rcnn.py:686)."""
    E, C, H, W, mw, mh, Kmax = 4, 128, 96, 128, 40, 30, 11
    cells = mw * mh
    rng = np.random.default_rng(21)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    sums = [torch.zeros(cells, C) for _ in range(E)]
    counts = [torch.zeros(cells) for _ in range(E)]
    for t in range(3):
        idx = (rng.integers(0, cells, (E, H // 4 + 1, W // 8 + 1)).repeat(4, 1).repeat(8, 2)[:, :H, :W]).astype(np.int32)
        n_obj = np.array([Kmax, 3, 0, 7], np.int32) if t != 1 else np.array([1, 0, 5, Kmax], np.int32)
        bf = np.zeros((E, Kmax, C), np.float32)
        masks = np.zeros((E, Kmax, H, W), bool)
        for e in range(E):
            if n_obj[e]:
                f, m = eod.episodes.make_detections(rng, H, W, C, (int(n_obj[e]), int(n_obj[e])))
                bf[e, : n_obj[e]], masks[e, : n_obj[e]] = f, m
            # garbage beyond n_obj must be ignored
            bf[e, n_obj[e]:] = 1e6
            masks[e, n_obj[e]:] = True
        batch.set_indices(_t(idx, cuda))
        batch.write_objects(_t(bf, cuda), _t(masks, cuda), _t(n_obj, cuda))
        torch.cuda.synchronize()
        for e in range(E):
            if n_obj[e]:
                img, obs = R.box_to_image_features(torch.from_numpy(bf[e, : n_obj[e]]), torch.from_numpy(masks[e, : n_obj[e]]))
                sums[e], counts[e] = R.write_mean_frame(sums[e], counts[e], img, obs, torch.from_numpy(idx[e]).long(), stride=8)
            got = batch.sums[e].cpu().numpy()
            ref = sums[e].numpy()
            assert np.abs(got - ref).max() <= SUM_TOL * max(np.abs(ref).max(), 1e-30), (t, e)
            assert np.array_equal(got == 0, ref == 0)                                     # touched-cell set: exact
            assert np.array_equal(batch.counts[e].cpu().numpy(), counts[e].numpy()), (t, e)
        assert sum(int(f.abs().sum()) for f in batch._frame_cnt2) == 0


# --------------------------------------------------------------------------------------------------------
# mask pasting (custom_rcnn.py:880, detectron2 paste_masks_in_image) and the write fused with it
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["plain", "edge"])
def test_paste_masks_matches_torch_golden(eod, cuda, golden, name):
    """eod_paste_masks against the fixture torch-CPU produced at 480x640 (10 objects; 'edge': sub-pixel box, saturated mask
    whose box-edge value is exactly the threshold, box larger than the image): every pasted bool identical."""
    g = golden("paste")
    H, W = int(g["H"]), int(g["W"])
    probs, boxes = g[name + "_probs"], g[name + "_boxes"]
    K = probs.shape[0]
    ref = _unpack(g[name + "_masks_bits"], (K, H, W))
    masks, observed = eod.ops.paste_masks(_t(probs[None], cuda), _t(boxes[None], cuda), (H, W), float(g["thr"]), want_observed=True)
    assert np.array_equal(masks[0].cpu().numpy(), ref)
    assert np.array_equal(observed[0].cpu().numpy().astype(bool), ref.any(0).reshape(-1))
    mem = eod.SpatialFeatureMemory(128, cuda)
    assert np.array_equal(mem.paste_masks_in_image(torch.from_numpy(probs), torch.from_numpy(boxes), (H, W)).cpu().numpy(), ref)


@pytest.mark.parametrize("H,W,S", [(96, 128, 28), (77, 125, 28), (64, 64, 14), (50, 70, 7)])
def test_paste_masks_randomised_vs_oracle(eod, cuda, H, W, S):
    """Ragged object counts per episode, image sizes that are not multiples of 4, odd mask sizes, thresholds other than 0.5,
    degenerate (zero-extent) boxes: bit-exact against oracle/paste.c; planes beyond n_obj are all False."""
    rng = np.random.default_rng(H * 1000 + W)
    E, Kmax = 3, 9
    n_obj = np.array([Kmax, 4, 0], np.int32)
    probs = rng.uniform(0, 1, (E, Kmax, S, S)).astype(np.float32)
    boxes = np.zeros((E, Kmax, 4), np.float32)
    for e in range(E):
        _, p, b = eod.episodes.make_mask_head_detections(rng, H, W, 8, (Kmax, Kmax), S, edge_cases=(e == 0))
        probs[e], boxes[e] = p, b
    boxes[1, 1] = (10.5, 20.0, 10.5, 40.0)                 # x1 == x0: division by zero -> nothing pasted
    boxes[1, 2] = (30.0, 12.0, 20.0, 5.0)                  # inverted box
    for thr in (0.5, 0.3, 0.0):
        masks, observed = eod.ops.paste_masks(_t(probs, cuda), _t(boxes, cuda), (H, W), thr, _t(n_obj, cuda), want_observed=True)
        masks = masks.cpu().numpy()
        for e in range(E):
            # thr >= 0.5: detectron2's CPU path (integer box neighbourhood) == its CUDA path; below 0.5 the library follows the
            # CUDA path the reference takes (whole image sampled, skip_empty=False)
            ref = oracle.paste_masks(probs[e, : n_obj[e]], boxes[e, : n_obj[e]], H, W, thr, skip_empty=thr >= 0.5)
            assert np.array_equal(masks[e, : n_obj[e]], ref), (thr, e, int((masks[e, : n_obj[e]] != ref).sum()))
            assert not masks[e, n_obj[e]:].any()
            assert np.array_equal(observed[e].cpu().numpy().astype(bool), ref.any(0).reshape(-1) if n_obj[e] else np.zeros(H * W, bool))
    with pytest.raises(eod.EodError):
        eod.ops.paste_masks(_t(probs, cuda), _t(boxes, cuda), (H, W), -1.0)


def test_fused_detection_write_vs_oracle(eod, cuda):
    """EpisodeBatch.write_detections / SpatialFeatureMemory.update_implicit_memory fed with the UN-pasted mask-head output
    (28x28 probabilities + boxes): against oracle paste -> box_to_image_features -> project_image_features -> accumulate.
    Touched-cell sets and visibility counts exact, sums within the fp32 tolerance; identical sets to the two-step path
    (eod_paste_masks -> eod_write_objects)."""
    E, C, H, W, mw, mh, Kmax = 3, 128, 96, 128, 40, 30, 8
    cells = mw * mh
    rng = np.random.default_rng(33)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    twostep = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    single = eod.SpatialFeatureMemory(C, cuda, height=H, width=W)
    single.reset(cells)
    sums = [torch.zeros(cells, C) for _ in range(E)]
    counts = [torch.zeros(cells) for _ in range(E)]
    for t in range(3):
        idx = (rng.integers(0, cells, (E, H // 4 + 1, W // 8 + 1)).repeat(4, 1).repeat(8, 2)[:, :H, :W]).astype(np.int32)
        n_obj = np.array([Kmax, 0, 5], np.int32) if t != 1 else np.array([2, Kmax, 0], np.int32)
        bf = np.full((E, Kmax, C), 1e6, np.float32)
        probs = np.ones((E, Kmax, 28, 28), np.float32)                  # garbage beyond n_obj must be ignored
        boxes = np.tile(np.array([0, 0, W, H], np.float32), (E, Kmax, 1))
        for e in range(E):
            if n_obj[e]:
                f, p, b = eod.episodes.make_mask_head_detections(rng, H, W, C, (int(n_obj[e]), int(n_obj[e])), 28, edge_cases=(e == 2))
                bf[e, : n_obj[e]], probs[e, : n_obj[e]], boxes[e, : n_obj[e]] = f, p, b
        for b_ in (batch, twostep):
            b_.set_indices(_t(idx, cuda))
        batch.write_detections(_t(bf, cuda), _t(probs, cuda), _t(boxes, cuda), _t(n_obj, cuda))
        pasted, _ = eod.ops.paste_masks(_t(probs, cuda), _t(boxes, cuda), (H, W), 0.5, _t(n_obj, cuda))
        twostep.write_objects(_t(bf, cuda), pasted, _t(n_obj, cuda))
        if n_obj[0]:
            single.update_implicit_memory((_t(boxes[0, : n_obj[0]], cuda), _t(bf[0, : n_obj[0]], cuda), _t(probs[0, : n_obj[0]], cuda), None),
                                          _t(idx[0], cuda).long(), single.implicit_memory, {})
        torch.cuda.synchronize()
        for e in range(E):
            if n_obj[e]:
                masks = torch.from_numpy(oracle.paste_masks(probs[e, : n_obj[e]], boxes[e, : n_obj[e]], H, W, 0.5))
                img, obs = R.box_to_image_features(torch.from_numpy(bf[e, : n_obj[e]]), masks)
                sums[e], counts[e] = R.write_mean_frame(sums[e], counts[e], img, obs, torch.from_numpy(idx[e]).long(), stride=8)
            ref = sums[e].numpy()
            for got in (batch.sums[e].cpu().numpy(), twostep.sums[e].cpu().numpy()) + ((single.implicit_memory.cpu().numpy(),) if e == 0 else ()):
                assert np.abs(got - ref).max() <= SUM_TOL * max(np.abs(ref).max(), 1e-30), (t, e)
                assert np.array_equal(got == 0, ref == 0)                                 # touched-cell set: exact
            assert np.array_equal(batch.counts[e].cpu().numpy(), counts[e].numpy()), (t, e)
        assert np.array_equal(single.observations.cpu().numpy(), counts[0].numpy())
    assert sums[0].abs().max() > 0 and sums[1].abs().max() > 0


def test_step_detections_two_streams_matches_serial(eod, cuda):
    """EpisodeBatch.step_detections (geometry/read and paste/write on two streams) against the serial composition
    project -> read -> write_detections, frame by frame: identical indices and fp16 levels (the read sees the state of
    frame t-1), identical touched sets and counts, sums within the reduction-order tolerance."""
    E, C, H, W, mw, mh, Kmax, T = 3, 128, 96, 128, 60, 45, 6, 4
    cell = 0.2
    rng = np.random.default_rng(77)
    eps = [eod.episodes.make_episode(500 + e, T, H, W, mw, mh, cell) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    a = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    c = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, pipeline=True)      # frame t+1's project / paste / sample under frame t's write side
    lc_all, keep = [], []
    for t in range(T):
        Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))
        pose = Tm[:, :3].reshape(E, 12).to(cuda)
        depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
        n_obj = np.array([Kmax, 0 if t == 1 else 3, 2], np.int32)
        bf = np.zeros((E, Kmax, C), np.float32); pr = np.zeros((E, Kmax, 28, 28), np.float32); bx = np.zeros((E, Kmax, 4), np.float32)
        for e in range(E):
            if n_obj[e]:
                f, p, bb = eod.episodes.make_mask_head_detections(rng, H, W, C, (int(n_obj[e]), int(n_obj[e])), 28)
                bf[e, : n_obj[e]], pr[e, : n_obj[e]], bx[e, : n_obj[e]] = f, p, bb
        args = (_t(bf, cuda), _t(pr, cuda), _t(bx, cuda), _t(n_obj, cuda))
        la = [l.clone() for l in a.step_detections(depth, pose, shifts, intr, cell, *args)]
        b.project(depth, pose, shifts, intr, cell)
        lb = [l.clone() for l in b.read()]
        b.write_detections(*args)
        torch.cuda.synchronize()
        keep.append((depth, pose) + args)                                   # the pipelined batch is fed after the loop, back to back
        assert torch.equal(a.idx, b.idx)
        for x, y in zip(la, lb):
            # the two batches reduce in scheduling order: a few fp16 rows of their read tables may differ in the last bit
            d = (x.contiguous().view(torch.int16).int() - y.contiguous().view(torch.int16).int()).abs()
            assert int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3, t
            if t == 0:
                assert torch.equal(x, y)                                       # both tables still empty
        assert torch.equal(a.counts, b.counts) and torch.equal(a.sums == 0, b.sums == 0)
        assert (a.sums - b.sums).abs().max().item() <= SUM_TOL * max(b.sums.abs().max().item(), 1e-30)
        lc_all.append(lb)
    assert b.counts.max().item() >= 2 and b.sums.abs().max().item() > 0
    # pipelined: all frames enqueued without a host synchronisation in between (inputs resident, as the mode requires)
    got = []
    for t, (depth, pose, *args) in enumerate(keep):
        got.append([l.clone() for l in c.step_detections(depth, pose, shifts, intr, cell, *args, inputs_ready=(t != 2))])
    c.join()
    torch.cuda.synchronize()
    assert torch.equal(c.counts, b.counts) and torch.equal(c.sums == 0, b.sums == 0)
    assert (c.sums - b.sums).abs().max().item() <= SUM_TOL * max(b.sums.abs().max().item(), 1e-30)
    for t in range(T):
        for x, y in zip(got[t], lc_all[t]):
            d = (x.contiguous().view(torch.int16).int() - y.contiguous().view(torch.int16).int()).abs()
            assert int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3, t      # tables may differ in the last bit (reduction order)


def test_batch_without_fp16_table_reads_the_same_bits(eod, cuda):
    """EpisodeBatch(fp16_table=False) keeps only sums / counts (a third less memory per grid) and lets the read normalise + round the
    fp32 rows it gathers: levels, counts and sums must equal the default batch bit for bit (same kernels feed both, one stream each,
    deterministic write variant so that the two batches' sums agree exactly), incl. a per-slot reset in the middle."""
    E, C, H, W, mw, mh, T = 2, 128, 96, 128, 60, 45, 4
    cell = 0.2
    eps = [eod.episodes.make_episode(700 + e, T, H, W, mw, mh, cell) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    a = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, variant=eod._lib.WRITE_DET)
    b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, variant=eod._lib.WRITE_DET, fp16_table=False)
    assert b.norm16 is None
    a.det_runs_per_episode = b.det_runs_per_episode = H * W      # room for every run: no fallback to order-dependent reductions
    g = torch.Generator(device=cuda).manual_seed(3)
    for t in range(T):
        Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))
        pose = Tm[:, :3].reshape(E, 12).to(cuda)
        depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
        feat = torch.randn((E, C, H, W), device=cuda, generator=g)
        mask = torch.tensor([0, 1 if t == 2 else 0], dtype=torch.int32, device=cuda) if t == 2 else None
        la = [l.clone() for l in a.step(depth, pose, shifts, intr, cell, feat, reset_mask=mask)]
        lb = [l.clone() for l in b.step(depth, pose, shifts, intr, cell, feat, reset_mask=mask)]
        torch.cuda.synchronize()
        for x, y in zip(la, lb):
            assert torch.equal(x, y), t
        assert torch.equal(a.counts, b.counts), t
        assert torch.equal(a.sums, b.sums), (t, float((a.sums - b.sums).abs().max()), int((a.sums != b.sums).sum()))
    assert float(a.counts.max()) >= 2
    b.read_frozen = True
    with pytest.raises(eod.EodError):
        b.read()


def test_backproject_count_equals_project_then_count(eod, cuda):
    """eod_backproject_count (cell ids + per-cell pixel counts in one launch, one atomic per run over 128 consecutive pixels) against the
    two separate launches: identical idx and frame_cnt - on ray-cast depth, on noise (every pixel its own run), on a constant plane
    (one run per warp), with uint16 depth and with an active mask; sizes it cannot take are refused."""
    rng = np.random.default_rng(12)
    H, W, mw, mh, cell, E = 96, 128, 60, 45, 0.2, 3
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    eps = [eod.episodes.make_episode(900 + e, 1, H, W, mw, mh, cell) for e in range(E)]
    Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[0] for ep in eps])))
    pose = Tm[:, :3].reshape(E, 12).to(cuda)
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    depths = {"raycast": np.stack([ep.depth[0] for ep in eps]),
              "noise": rng.uniform(0.3, 9.0, (E, H, W)).astype(np.float32),
              "plane": np.full((E, H, W), 2.5, np.float32),
              "no depth": np.zeros((E, H, W), np.float32)}
    for name, d in depths.items():
        for raw in (False, True):
            dd = _t((d * 1000).round().clip(0, 65535).astype(np.uint16), cuda) if raw else _t(d, cuda)
            for active in (None, _t(np.array([1, 0, 2], np.int32), cuda)):
                ref_idx = eod.ops.backproject_quantize(dd, pose, shifts, intr, cell, mw, mh)["idx"]
                ref_cnt = torch.zeros((E, mw * mh), dtype=torch.int32, device=cuda)
                eod.ops.frame_count(ref_idx, None, ref_cnt, active)
                idx = torch.empty((E, H, W), dtype=torch.int32, device=cuda)
                cnt = torch.zeros((E, mw * mh), dtype=torch.int32, device=cuda)
                eod.ops.backproject_count(dd, pose, shifts, intr, cell, mw, mh, idx, cnt, active)
                assert torch.equal(idx, ref_idx), (name, raw)
                assert torch.equal(cnt, ref_cnt), (name, raw, active is not None)
                assert int(cnt.sum()) == (H * W * (E if active is None else 2))
    assert not eod.ops.backproject_count_supported(30, 100)
    with pytest.raises(eod.EodError):
        eod.ops.backproject_count(_t(np.ones((1, 30, 100), np.float32), cuda), pose[:1], shifts[:1], intr, cell, mw, mh,
                                  torch.empty((1, 30, 100), dtype=torch.int32, device=cuda), torch.zeros((1, mw * mh), dtype=torch.int32, device=cuda))


def test_divisor_lookup_and_divisor_plane_agree(eod, cuda):
    """The CHW write takes a group's divisor 1/n_cell either from frame_cnt (default since round 2) or from the per-pixel plane that
    eod_expand_counts prepares (``pixel_divisors = True``): same counts, same touched set, sums equal up to reduction order."""
    E, C, H, W, mw, mh, T = 2, 256, 96, 128, 60, 45, 3
    cell = 0.2
    eps = [eod.episodes.make_episode(800 + e, T, H, W, mw, mh, cell) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    a = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    assert a.pixel_divisors is False and a._pix_inv_n2 is None
    b.pixel_divisors = True
    g = torch.Generator(device=cuda).manual_seed(4)
    for t in range(T):
        Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))
        pose = Tm[:, :3].reshape(E, 12).to(cuda)
        depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
        feat = torch.randn((E, C, H, W), device=cuda, generator=g)
        samp = (torch.rand((E, H, W), device=cuda, generator=g) < 0.6).to(torch.uint8) if t == 1 else None
        a.step(depth, pose, shifts, intr, cell, feat, samp)
        b.step(depth, pose, shifts, intr, cell, feat, samp)
    torch.cuda.synchronize()
    assert b._pix_inv_n2 is not None and a._pix_inv_n2 is None
    assert torch.equal(a.counts, b.counts) and torch.equal(a.sums == 0, b.sums == 0)
    assert (a.sums - b.sums).abs().max().item() <= 1e-6 * b.sums.abs().max().item()


def test_graphed_step_detections_matches_eager(eod, cuda):
    """capture_step_detections (one CUDA graph per frame: the online single-robot loop) against the eager step_detections on a twin
    batch, frame by frame, with an eager frame interleaved: identical indices, fp16 levels, counts and touched sets, sums within the
    reduction-order tolerance; a frame without detections (n_obj = 0) writes nothing in either."""
    C, H, W, mw, mh, Kmax, T = 128, 96, 128, 60, 45, 6, 6
    cell = 0.2
    for E in (1, 2):
        rng = np.random.default_rng(78 + E)
        eps = [eod.episodes.make_episode(600 + e, T, H, W, mw, mh, cell) for e in range(E)]
        intr = eod.compute_intrinsics(W, H, math.radians(67.5))
        shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
        a = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
        b = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
        graphed = None
        for t in range(T):
            Tm = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))
            pose = Tm[:, :3].reshape(E, 12).to(cuda)
            depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
            n_obj = np.array([0 if t == 2 else Kmax - (t % 3)] + [3] * (E - 1), np.int32)
            bf = np.zeros((E, Kmax, C), np.float32); pr = np.zeros((E, Kmax, 28, 28), np.float32); bx = np.zeros((E, Kmax, 4), np.float32)
            for e in range(E):
                if n_obj[e]:
                    f, p, bb = eod.episodes.make_mask_head_detections(rng, H, W, C, (int(n_obj[e]), int(n_obj[e])), 28)
                    bf[e, : n_obj[e]], pr[e, : n_obj[e]], bx[e, : n_obj[e]] = f, p, bb
            args = (_t(bf, cuda), _t(pr, cuda), _t(bx, cuda), _t(n_obj, cuda))
            if graphed is None:
                graphed = a.capture_step_detections(depth, pose, shifts, intr, cell, *args)
                assert float(a.sums.abs().max()) == 0.0 and float(a.counts.max()) == 0.0     # capturing wrote nothing
            if t == 3:
                la = [l.clone() for l in a.step_detections(depth, pose, shifts, intr, cell, *args)]      # eager frame in between
            else:
                la = [l.clone() for l in graphed(depth, pose, shifts, *args)]
            lb = [l.clone() for l in b.step_detections(depth, pose, shifts, intr, cell, *args)]
            torch.cuda.synchronize()
            assert torch.equal(a.idx, b.idx), (E, t)
            # the two batches accumulate with fp32 reductions in scheduling order, so their sums - and with them a few fp16 rows of
            # the read table - may differ in the last bit: levels equal up to one fp16 ulp, and exactly wherever the tables agree
            same_table = torch.equal(a.norm16, b.norm16) if t == 0 else None
            for x, y in zip(la, lb):
                d = (x.contiguous().view(torch.int16).int() - y.contiguous().view(torch.int16).int()).abs()
                assert int(d.max()) <= 1 and float((d != 0).float().mean()) < 1e-3, (E, t)
                if same_table:
                    assert torch.equal(x, y), (E, t)
            assert torch.equal(a.counts, b.counts) and torch.equal(a.sums == 0, b.sums == 0), (E, t)
            assert (a.sums - b.sums).abs().max().item() <= SUM_TOL * max(b.sums.abs().max().item(), 1e-30)
        assert b.counts.max().item() >= 2 and b.sums.abs().max().item() > 0


def test_object_write_more_than_128_objects(eod, cuda):
    """Above 128 kept objects per frame the write takes its one-pixel-at-a-time path (the bitmask phase holds 128):
    both the byte-mask and the pasted variant against the oracle chain."""
    E, C, H, W, mw, mh, Kmax = 1, 128, 64, 96, 20, 15, 140
    cells = mw * mh
    rng = np.random.default_rng(140)
    idx = (rng.integers(0, cells, (E, H // 4, W // 8)).repeat(4, 1).repeat(8, 2)).astype(np.int32)
    f, probs, boxes = eod.episodes.make_mask_head_detections(rng, H, W, C, (Kmax, Kmax), 28)
    masks = oracle.paste_masks(probs, boxes, H, W, 0.5)
    img, obs = R.box_to_image_features(torch.from_numpy(f), torch.from_numpy(masks))
    ref, counts = R.write_mean_frame(torch.zeros(cells, C), torch.zeros(cells), img, obs, torch.from_numpy(idx[0]).long(), stride=8)
    for pasted in (False, True):
        batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
        batch.set_indices(_t(idx, cuda))
        if pasted:
            batch.write_detections(_t(f[None], cuda), _t(probs[None], cuda), _t(boxes[None], cuda))
        else:
            batch.write_objects(_t(f[None], cuda), _t(masks[None], cuda))
        got = batch.sums[0].cpu().numpy()
        assert np.abs(got - ref.numpy()).max() <= SUM_TOL * np.abs(ref.numpy()).max(), pasted
        assert np.array_equal(got == 0, ref.numpy() == 0)
        assert np.array_equal(batch.counts[0].cpu().numpy(), counts.numpy())


def test_dense_backbone_write_vs_oracle(eod, cuda):
    """A7'' (bytecode-only lineage): bilinear lattice samples bit-exact vs torch-CPU F.interpolate, per-cell means of the
    projected samples within the fp32 tolerance, observed set exact, memory REPLACED (zeros elsewhere)."""
    rng = np.random.default_rng(8)
    C, h, w, H, W, mw, mh = 256, 60, 80, 480, 640, 120, 90
    cells = mw * mh
    p3 = torch.from_numpy(rng.standard_normal((1, C, h, w)).astype(np.float32))
    proj = torch.from_numpy((rng.integers(0, cells, (H // 16 + 1, W // 16 + 1)).repeat(16, 0).repeat(16, 1)[:H, :W]).astype(np.int64))
    lat = eod.ops.bilinear_lattice(p3.to(cuda), (H, W), 8)
    ref_lat = torch.nn.functional.interpolate(p3, (H, W), mode="bilinear", align_corners=True)[:, :, ::8, ::8]
    assert torch.equal(lat.cpu(), ref_lat)                                  # bit-exact lattice samples
    odd = eod.ops.bilinear_lattice(p3[:, :8, :37, :53].contiguous().to(cuda), (101, 203), 3)
    assert torch.equal(odd.cpu(), torch.nn.functional.interpolate(p3[:, :8, :37, :53], (101, 203), mode="bilinear", align_corners=True)[:, :, ::3, ::3])
    weight = torch.from_numpy(rng.standard_normal((C, C, 1, 1)).astype(np.float32) / 16)
    bias = torch.from_numpy(rng.standard_normal(C).astype(np.float32))
    mem = eod.SpatialFeatureMemory(C, cuda)
    for wgt, b in ((None, None), (weight, bias)):
        got, obs = mem.dense_backbone_write(p3, proj, cells, wgt, b)
        ref, ref_obs = R.dense_backbone_write(p3, proj, cells, wgt, b)
        assert np.array_equal(obs.cpu().numpy(), ref_obs.numpy())
        tol = SUM_TOL if wgt is None else 1e-4                              # library GEMM (TF32-free fp32) vs MKL: summation order
        assert (got.cpu() - ref).abs().max().item() <= tol * ref.abs().max().item()
        assert not got.cpu()[~ref_obs].any()


# --------------------------------------------------------------------------------------------------------
# write, height-max mode (A7')
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout,stride", [(1, 1), (0, 1), (1, 4)])
def test_write_max_vs_oracle(eod, cuda, layout, stride):
    rng = np.random.default_rng(17 + stride)
    H, W, C, mw, mh, T = 48, 64, 64, 23, 19, 4
    cells = mw * mh
    state = torch.zeros(cells, C)
    observed = torch.zeros(cells, dtype=torch.bool)
    hmap = torch.zeros(cells)
    d_state = torch.zeros((1, cells, C), device=cuda)
    d_obs = torch.zeros((1, cells), dtype=torch.uint8, device=cuda)
    d_hmap = torch.zeros((1, cells), device=cuda)
    d_key = torch.zeros((1, cells), dtype=torch.int64, device=cuda)
    d_arg = torch.zeros((1, cells), dtype=torch.int32, device=cuda)
    for t in range(T):
        w2m = np.stack([rng.integers(0, mw, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1), rng.integers(0, mh, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1)], -1)
        inl = rng.uniform(size=(H, W)) < 0.7
        heights = (np.round(rng.uniform(-1.5, 1.0, (H, W)) * 4) / 4).astype(np.float32)        # quantised -> many exact ties
        if t == 2:
            heights[:] = heights.min() - 5                                                       # nothing raised except new cells
        if t == 3:                                                                               # non-finite heights (ADVICE r1): a NaN pixel
            heights[rng.uniform(size=(H, W)) < 0.1] = np.nan                                     # neither raises a cell nor shadows finite ones;
            heights[rng.uniform(size=(H, W)) < 0.02] = np.inf                                    # +inf wins like any maximum, -inf never does
            heights[rng.uniform(size=(H, W)) < 0.02] = -np.inf
        feat = rng.standard_normal((H, W, C)).astype(np.float32)
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, torch.from_numpy(feat), torch.from_numpy(w2m),
                                                                torch.from_numpy(inl), torch.from_numpy(heights), mw, stride)
        flat = (w2m[..., 1] * mw + w2m[..., 0]).astype(np.int32)
        f_dev = _t(feat if layout == 1 else feat.transpose(2, 0, 1), cuda)[None].contiguous()
        eod.ops.write_max(_t(heights, cuda)[None], _t(flat, cuda)[None], _t((~inl).view(np.uint8), cuda)[None], f_dev, d_hmap, d_key, d_arg,
                          d_obs, d_state, layout, stride)
        torch.cuda.synchronize()
        # oracle arg indexes the compacted inlier lattice; convert to raster pixel indices of the full frame
        lat = np.zeros((H, W), bool)
        lat[::stride, ::stride] = True
        pix_of_rank = np.nonzero((inl & lat).reshape(-1))[0]
        arg_pix = np.where(arg.numpy() >= 0, pix_of_rank[np.maximum(arg.numpy(), 0)], -1)
        assert np.array_equal(d_arg[0].cpu().numpy(), arg_pix), t                              # argmax: exact
        assert np.array_equal(d_hmap[0].cpu().numpy(), hmap.numpy())
        assert np.array_equal(d_obs[0].cpu().numpy().astype(bool), observed.numpy())
        assert np.array_equal(d_state[0].cpu().numpy(), state.numpy())                         # winners' features: exact copies
        assert int(d_key.abs().sum()) == 0


@pytest.mark.parametrize("M,K,N", [(1, 64, 16), (127, 64, 256), (128, 96, 64), (300, 512, 256), (1000, 256, 512), (257, 20, 48)])
def test_linear_rows_fp32_accuracy_on_tensor_cores(eod, cuda, M, K, N):
    """eod_linear_rows (3xTF32 on tcgen05, fp32 accumulators in TMEM) against fp64: |error| <= 1e-5 of scale - and not worse than a few
    times the error of the fp32 library GEMM it replaces - for contiguous, transposed (row stride 1) and padded operands, with and
    without bias / scale, K not a multiple of the 32-wide chunk, N over one and two TMEM column blocks."""
    g = torch.Generator(device=cuda).manual_seed(M * 7 + K)
    a = torch.randn((M, K), device=cuda, generator=g) * torch.rand((M, 1), device=cuda, generator=g).mul(6).sub(3).exp()    # rows of very different scale
    w = torch.randn((N, K), device=cuda, generator=g) / K ** 0.5
    b = torch.randn((N,), device=cuda, generator=g)
    ref = (a.double() @ w.double().t() + b.double()) * 0.75
    scale = float(ref.abs().max())
    lib_err = float(((a @ w.t() + b) * 0.75 - ref).abs().max()) / scale
    a_t = a.t().contiguous().t()                                     # same values, row stride 1 / element stride M
    w_pad = torch.zeros((N, K + 12), device=cuda)[:, 3:3 + K]        # unaligned rows, row stride K + 12
    w_pad.copy_(w)
    for name, (aa, ww) in {"contiguous": (a, w), "A transposed view": (a_t, w), "W padded / unaligned": (a, w_pad), "both": (a_t, w_pad)}.items():
        got = eod.ops.linear_rows(aa, ww, b, 0.75)
        err = float((got.double() - ref).abs().max()) / scale
        assert err <= 1e-5 and err <= max(4 * lib_err, 2e-6), (name, err, lib_err)
    if M > 2:                                    # a non-finite input poisons ITS row (inf or NaN: the split turns inf * 0-remainder into NaN), no other
        a_inf = a.clone()
        a_inf[1, 0], a_inf[2, K - 1] = float("inf"), float("nan")
        got = eod.ops.linear_rows(a_inf, w, b, 0.75)
        assert not bool(torch.isfinite(got[1:3]).any())
        keep = torch.ones(M, dtype=torch.bool, device=cuda)
        keep[1:3] = False
        assert float((got[keep].double() - ref[keep]).abs().max()) <= 1e-5 * scale
    nob = eod.ops.linear_rows(a, w)
    assert float((nob.double() - a.double() @ w.double().t()).abs().max()) <= 1e-5 * float((a.double() @ w.double().t()).abs().max())
    # gathered rows + scattered output + device-side row count (the 'replace' update's shape)
    perm = torch.randperm(M, device=cuda, generator=g)
    n_live = max(1, (2 * M) // 3)
    out = torch.full((M + 5, N), 7.0, device=cuda)
    eod.ops.linear_rows(a, w, b, 1.0, out=out, a_off=(perm * K).to(torch.int64), m_count=torch.tensor([n_live], dtype=torch.int32, device=cuda),
                        n_rows=M, y_dst=(perm + 5).to(torch.int64))
    ref2 = a.double() @ w.double().t() + b.double()
    live = perm[:n_live]
    assert float((out[live + 5].double() - ref2[live]).abs().max()) <= 1e-5 * float(ref2.abs().max())
    untouched = torch.ones(M + 5, dtype=torch.bool, device=cuda)
    untouched[live + 5] = False
    assert bool((out[untouched] == 7.0).all())                       # rows beyond the count and unlisted rows are not written


@pytest.mark.parametrize("layout", [0, 1])
def test_write_max_replace_with_linlayer(eod, cuda, layout):
    """SMNet 'replace' update with the linear layer (model.cpython-310.pyc src lines 104-128): state[raised cells] = linlayer(feature[
    winner pixels]).  Contest results (argmax, height map, observed) exact vs the canonical-rule oracle; the raised cells' rows equal
    F.linear of the winners' features (fp64 reference, 1e-5 of scale), every other row is left untouched bit for bit."""
    rng = np.random.default_rng(31 + layout)
    H, W, C_in, C_mem, mw, mh, T, stride = 48, 64, 64, 256, 23, 19, 3, 2
    cells = mw * mh
    lin_w = (rng.standard_normal((C_mem, C_in)) / 8).astype(np.float32)
    lin_b = rng.standard_normal(C_mem).astype(np.float32)
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
        if t == 2:
            heights[:] = heights.min() - 5
        feat = rng.standard_normal((H, W, C_in)).astype(np.float32)
        prev = d_state.clone()
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, torch.from_numpy(feat).double(), torch.from_numpy(w2m),
                                                                torch.from_numpy(inl), torch.from_numpy(heights), mw, stride,
                                                                linlayer=(torch.from_numpy(lin_w).double(), torch.from_numpy(lin_b).double()))
        flat = (w2m[..., 1] * mw + w2m[..., 0]).astype(np.int32)
        f_dev = _t(feat if layout == 1 else feat.transpose(2, 0, 1), cuda)[None].contiguous()
        count = eod.ops.write_max_linear(_t(heights, cuda)[None], _t(flat, cuda)[None], _t((~inl).view(np.uint8), cuda)[None], f_dev, d_hmap, d_key,
                                         d_arg, d_obs, d_state, _t(lin_w, cuda), _t(lin_b, cuda), layout, stride)
        torch.cuda.synchronize()
        assert int(count.item()) == int(m.sum())
        assert np.array_equal(d_hmap[0].cpu().numpy(), hmap.numpy())
        assert np.array_equal(d_obs[0].cpu().numpy().astype(bool), observed.numpy())
        assert np.array_equal((d_arg[0] >= 0).cpu().numpy(), m.numpy())
        got = d_state[0].cpu().double()
        assert float((got - state).abs().max()) <= 1e-5 * float(state.abs().max())
        assert torch.equal(d_state[0][~m.to(cuda)], prev[0][~m.to(cuda)])                       # cells that were not raised keep their rows
        state = got.clone()                                                                     # carry the device rows (no drift between frames)
        assert int(d_key.abs().sum()) == 0


def test_write_max_config3_full_size(eod, cuda):
    """BASELINE configs[2]: SMNet-style height-max projection, 480x640, C=256, 0.02 m cells, 1000x1000 map.  Geometry
    (unclipped cell coordinates, outlier mask, heights) comes from the back-projection kernel exactly as
    create_coco_mp3d.py:157-165 obtains it from Projector.forward(..., return_heights=True); argmax, height map,
    observed set and the winners' feature rows must equal the oracle bit for bit."""
    H, W, C, mw, mh, T_ = 480, 640, 256, 1000, 1000, 3
    cells = mw * mh
    ep = eod.episodes.make_episode(4321, T_, H, W, mw, mh, 0.02, room_size=(24.0, 16.0))     # room larger than the 20 m map: out-of-map pixels
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    Tm = eod.transform3d(torch.from_numpy(ep.xyzhe))
    sh = _t(np.concatenate([ep.map_world_shift, np.zeros(3, np.float32)])[None], cuda)      # Projector subtracts map_world_shift as world_shift_origin
    state = torch.zeros(cells, C)
    observed = torch.zeros(cells, dtype=torch.bool)
    hmap = torch.zeros(cells)
    d_state = torch.zeros((1, cells, C), device=cuda)
    d_obs = torch.zeros((1, cells), dtype=torch.uint8, device=cuda)
    d_hmap = torch.zeros((1, cells), device=cuda)
    d_key = torch.zeros((1, cells), dtype=torch.int64, device=cuda)
    d_arg = torch.zeros((1, cells), dtype=torch.int32, device=cuda)
    gen = torch.Generator(device=cuda).manual_seed(5)
    n_raised = 0
    for t in range(T_):
        r = eod.ops.backproject_quantize(_t(ep.depth[t:t + 1], cuda), Tm[t:t + 1, :3].reshape(1, 12).to(cuda), sh, intr, 0.02, mw, mh,
                                         want_q2=True, want_outlier=True, want_height=True)
        o = oracle.backproject_quantize(ep.depth[t], Tm[t].numpy(), intr, ep.map_world_shift, np.zeros(3, np.float32), 0.02, mw, mh, 0, 0.5)
        assert np.array_equal(r["q2"][0].cpu().numpy(), o["q2"]) and np.array_equal(r["outlier"][0].cpu().numpy(), o["outlier"])
        assert np.array_equal(r["height"][0].cpu().numpy(), o["height"])
        q2 = r["q2"][0]
        flat = (q2[..., 1] * mw + q2[..., 0]).clamp(0, cells - 1).to(torch.int32)             # only inliers are used; they are in range
        feat = torch.randn((1, H, W, C), device=cuda, generator=gen)
        eod.ops.write_max(r["height"], flat[None].contiguous(), r["outlier"], feat, d_hmap, d_key, d_arg, d_obs, d_state, 1, 1)
        torch.cuda.synchronize()
        inl = ~torch.from_numpy(o["outlier"].astype(bool))
        state, observed, hmap, arg, m = R.smnet_heightmax_frame(state, observed, hmap, feat[0].cpu(), torch.from_numpy(o["q2"]), inl,
                                                                torch.from_numpy(o["height"]), mw, 1)
        pix_of_rank = np.nonzero(inl.numpy().reshape(-1))[0]
        arg_pix = np.where(arg.numpy() >= 0, pix_of_rank[np.maximum(arg.numpy(), 0)], -1)
        assert np.array_equal(d_arg[0].cpu().numpy(), arg_pix), t
        assert np.array_equal(d_hmap[0].cpu().numpy(), hmap.numpy())
        assert np.array_equal(d_obs[0].cpu().numpy().astype(bool), observed.numpy())
        assert torch.equal(d_state[0].cpu(), state)
        assert int(d_key.abs().sum()) == 0
        n_raised += int(m.sum())
    assert n_raised > 1000 and 0 < float(inl.float().mean()) < 1                              # the case exercises inliers AND outliers


# --------------------------------------------------------------------------------------------------------
# full-size, size-independent properties (BASELINE sizes: 480x640, C=256, 500x500 grid)
# --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,mw,mh,cell", [(256, 500, 500, 0.2), (512, 1000, 1000, 0.02)], ids=["configs1-2", "configs5"])
def test_full_size_properties(eod, cuda, C, mw, mh, cell):
    E, H, W = 2, 480, 640
    eps = [eod.episodes.make_episode(1234 + e, 3, H, W, mw, mh, cell) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    gen = torch.Generator(device=cuda).manual_seed(0)
    total_vis = torch.zeros(E, device=cuda)
    for t in range(3):
        depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
        T = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))
        pose = T[:, :3].reshape(E, 12).to(cuda)
        feat = torch.randn((E, C, H, W), device=cuda, generator=gen)
        before = batch.sums.clone()
        levels = batch.step(depth, pose, shifts, intr, cell, feat)
        torch.cuda.synchronize()
        for e in range(E):                                              # indices: bit-exact vs the oracle at full size
            o = oracle.backproject_quantize(eps[e].depth[t], T[e].numpy(), intr, np.zeros(3, np.float32), eps[e].map_world_shift, cell, mw, mh, 0, 0.5, want=("idx",))
            assert np.array_equal(batch.idx[e].cpu().numpy(), o["idx"])
        # conservation: sum_c n_c * (delta sums)_c == sum over pixels of the features (per channel)
        delta = batch.sums - before
        for e in range(E):
            cells, n = torch.unique(batch.idx[e].long(), return_counts=True)
            lhs = (delta[e][cells].double() * n[:, None].double()).sum(0)
            rhs = feat[e].double().sum(dim=(1, 2))
            assert (lhs - rhs).abs().max().item() <= 1e-5 * feat[e].abs().sum(dim=(1, 2)).max().item()
            total_vis[e] += cells.numel()
            assert int(batch.counts[e].sum().item()) == int(total_vis[e].item())          # counts: +1 per visible cell per frame
            touched = torch.zeros(mw * mh, dtype=torch.bool, device=cuda)
            touched[cells] = True
            assert (delta[e][~touched] == 0).all().item()
        assert sum(int(f.abs().sum()) for f in batch._frame_cnt2) == 0
    # read after 3 frames vs the C oracle on the downloaded state (bit-exact fp16)
    idx_np = batch.idx.cpu().numpy()
    levels = batch.read()
    torch.cuda.synchronize()
    for e in range(E):
        table16 = R.create_implicit_memory(batch.sums[e].cpu(), batch.counts[e].cpu()).half().numpy()
        L = oracle.read_pool_f16(table16, idx_np[e])
        for k in range(3):
            assert np.array_equal(levels[k][e].contiguous().cpu().numpy().view(np.uint16), L[k].view(np.uint16)), (e, k)
        # the incrementally maintained fp16 table equals a full re-normalisation of the grid
        assert np.array_equal(batch.norm16[e].cpu().numpy().view(np.uint16), table16.view(np.uint16))
    # idempotence: a constant table reads back as that constant at every level
    const = torch.randn(C, device=cuda).half()
    batch.norm16[:] = const
    levels = batch.read()
    for lv in levels:
        assert (lv == const.view(1, C, 1, 1)).all().item()


def test_pipelined_step_matches_stream_ordered_step(eod, cuda):
    """pipeline=True (geometry of frame t+1 under the write of frame t, read next to the write) must give the
    results of the stream-ordered mode: indices and counts bit-exact, sums to atomics-order noise, levels to fp16
    rounding of that noise."""
    E, C, H, W, mw, mh, T_ = 3, 128, 96, 128, 60, 45, 6
    eps = [eod.episodes.make_episode(500 + e, T_, H, W, mw, mh, 0.2) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    depth = [_t(np.stack([ep.depth[t] for ep in eps]), cuda) for t in range(T_)]
    pose = [eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))[:, :3].reshape(E, 12).to(cuda) for t in range(T_)]
    gen = torch.Generator(device=cuda).manual_seed(3)
    feat = [torch.randn((E, C, H, W), device=cuda, generator=gen) for _ in range(T_)]
    torch.cuda.synchronize()
    out = {}
    for mode in (False, True):
        batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda, pipeline=mode)
        lv, ix = [], []
        for rep in range(2):                                   # second pass after a reset: reset must not race the pipeline
            batch.reset()
            lv, ix = [], []
            for t in range(T_):
                levels = batch.step(depth[t], pose[t], shifts, intr, 0.2, feat[t])
                lv.append([l.clone() for l in levels])         # ordered on the caller's stream in both modes
                ix.append(batch.idx.clone() if not mode else None)
        batch.join()
        torch.cuda.synchronize()
        out[mode] = (batch.sums.clone(), batch.counts.clone(), lv, batch.idx.clone(), batch.norm16.clone())
    (s0, c0, l0, i0, n0), (s1, c1, l1, i1, n1) = out[False], out[True]
    assert torch.equal(c0, c1) and torch.equal(i0, i1)
    assert (s0 - s1).abs().max().item() <= 1e-6 * s0.abs().max().item()
    for t in range(T_):
        for a, b in zip(l0[t], l1[t]):
            assert torch.allclose(a.float(), b.float(), rtol=2e-3, atol=2e-3), t
    assert torch.allclose(n0.float(), n1.float(), rtol=2e-3, atol=2e-3)


def test_sparse_reset_clears_everything(eod, cuda):
    """EpisodeBatch.reset() clears only the rows of cells seen since the last reset; the result must be the
    all-zero state of custom_rcnn.py:470-477."""
    E, C, H, W, mw, mh = 2, 128, 96, 128, 60, 45
    eps = [eod.episodes.make_episode(900 + e, 3, H, W, mw, mh, 0.2) for e in range(E)]
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    shifts = _t(np.stack([np.concatenate([np.zeros(3, np.float32), ep.map_world_shift]) for ep in eps]), cuda)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    for t in range(3):
        depth = _t(np.stack([ep.depth[t] for ep in eps]), cuda)
        pose = eod.transform3d(torch.from_numpy(np.stack([ep.xyzhe[t] for ep in eps])))[:, :3].reshape(E, 12).to(cuda)
        batch.step(depth, pose, shifts, intr, 0.2, torch.randn((E, C, H, W), device=cuda))
    assert batch.counts.sum().item() > 0 and batch.sums.abs().sum().item() > 0 and batch.norm16.float().abs().sum().item() > 0
    batch.reset()
    torch.cuda.synchronize()
    assert batch.counts.abs().sum().item() == 0
    assert batch.sums.abs().sum().item() == 0
    assert batch.norm16.float().abs().sum().item() == 0
    assert sum(int(f.abs().sum()) for f in batch._frame_cnt2) == 0


def test_tma_and_ldg_variants_agree_full_size(eod, cuda):
    E, C, H, W, cells = 1, 256, 480, 640, 250000
    ep = eod.episodes.make_episode(77, n_frames=1)
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    T = eod.transform3d(torch.from_numpy(ep.xyzhe[:1]))
    sh = _t(np.concatenate([np.zeros(3, np.float32), ep.map_world_shift])[None], cuda)
    idx = eod.ops.backproject_quantize(_t(ep.depth[:1], cuda), T[:, :3].reshape(1, 12).to(cuda), sh, intr, 0.2, 500, 500)["idx"]
    feat = torch.randn((E, C, H, W), device=cuda)
    outs = []
    for variant in (1, 2):
        sums = torch.zeros((E, cells, C), device=cuda)
        cnt = torch.zeros((E, cells), dtype=torch.int32, device=cuda)
        eod.ops.frame_count(idx, None, cnt)
        eod.ops.write_mean(feat, idx, None, cnt, sums, 0, variant)
        outs.append(sums)
    scale = outs[0].abs().max().item()
    assert (outs[0] - outs[1]).abs().max().item() <= 1e-6 * scale
    s, n = oracle.cell_sums_seq(feat[0].cpu().numpy(), idx[0].cpu().numpy(), None, cells)
    ref = np.where(n[:, None] > 0, s / np.maximum(n, 1)[:, None].astype(np.float32), 0)
    assert np.abs(outs[1][0].cpu().numpy() - ref).max() <= SUM_TOL * np.abs(ref).max()


def test_new_kernels_stay_inside_their_output_buffers(eod, cuda):
    """compute-sanitizer is not available on the pool, so the kernels written this round get a canary check: every output
    tensor is a window of a larger buffer filled with a sentinel, and the bytes on both sides must survive the launch
    (ragged sizes on purpose: partial tiles, partial vectors, last-episode tails)."""
    rng = np.random.default_rng(123)

    def window(shape, dtype, pad=4096):
        n = int(np.prod(shape))
        item = torch.empty((), dtype=dtype).element_size()
        padn = pad // item
        buf = torch.empty(n + 2 * padn, dtype=dtype, device=cuda)
        buf.view(torch.uint8).fill_(0xA5)
        return buf, buf[padn:padn + n].view(shape), padn

    def intact(buf, padn):
        b = buf.view(torch.uint8)
        item = buf.element_size()
        return bool((b[: padn * item] == 0xA5).all()) and bool((b[-padn * item:] == 0xA5).all())

    # read: E=3, 96x160, C=256 / 512 (lanes own 8 / 16 channels)
    for C in (128, 256, 512):
        E, H, W, cells = 3, 96, 160, 700
        table = _t((rng.standard_normal((E, cells, C))).astype(np.float16), cuda)
        idx = _t(rng.integers(0, cells, (E, H, W)).astype(np.int32), cuda)
        bufs = [window((E, H >> s, W >> s, C), torch.float16) for s in (3, 4, 5)]
        eod.ops.read_pool(table, None, idx, out=[b[1] for b in bufs])
        torch.cuda.synchronize()
        assert all(intact(b[0], b[2]) for b in bufs), C
    # paste: odd image size, masks + observed
    E, K, H, W = 2, 5, 77, 125
    probs = _t(rng.uniform(0, 1, (E, K, 28, 28)).astype(np.float32), cuda)
    boxes = _t(np.tile(np.array([-5.0, -3.0, W + 4.0, H + 2.0], np.float32), (E, K, 1)), cuda)
    mb, mv, mp = window((E, K, H * W), torch.uint8)
    ob, ov, op_ = window((E, H * W), torch.uint8)
    eod._lib.check(eod._lib.lib().eod_paste_masks(probs.data_ptr(), boxes.data_ptr(), None, E, K, 28, H, W, 0.5, mv.data_ptr(), ov.data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream), "eod_paste_masks")
    torch.cuda.synchronize()
    assert intact(mb, mp) and intact(ob, op_) and bool(mv.any())
    # projection + fusion: ragged tiles in both kernels
    for variant, (h, w) in ((1, (7, 9)), (2, (15, 20)), (2, (30, 40))):
        E, Kc, N = 3, 128, 128
        lvl = _t(rng.standard_normal((E, h, w, Kc)).astype(np.float16), cuda)
        ws = eod.ops.project_split_weights(_t(rng.standard_normal((N, Kc)).astype(np.float32), cuda))
        res = _t(rng.standard_normal((E, N, h, w)).astype(np.float32), cuda)
        ob, ov, op_ = window((E, N, h, w), torch.float32)
        eod.ops.project_fuse_levels([lvl], [ws], [None], [res], 5.0, 0, outs=[ov], variant=variant)
        torch.cuda.synchronize()
        assert intact(ob, op_), (variant, h, w)
    # row GEMM: ragged last tile, strided output rows (guard bytes between rows too), scattered rows, K tail
    for M, K, N in ((130, 40, 48), (5, 512, 256), (257, 64, 272)):
        a = _t(rng.standard_normal((M, K)).astype(np.float32), cuda)
        w = _t(rng.standard_normal((N, K)).astype(np.float32), cuda)
        ob, ov, op_ = window((M + 3, N + 8), torch.float32)
        dst = torch.randperm(M + 3, device=cuda)[:M].to(torch.int64).contiguous()
        eod.ops.linear_rows(a, w, None, 1.0, out=ov, y_dst=dst, a_off=(torch.arange(M, device=cuda) * K).to(torch.int64), n_rows=M)
        torch.cuda.synchronize()
        assert intact(ob, op_), (M, K, N)
        pad_cols = ov[:, N:].contiguous().view(torch.uint8)
        assert bool((pad_cols == 0xA5).all()), (M, K, N)                                       # the 8 floats behind every output row
        free = torch.ones(M + 3, dtype=torch.bool, device=cuda)
        free[dst] = False
        assert bool((ov[free].contiguous().view(torch.uint8) == 0xA5).all())
        assert float((ov[dst][:, :N].double() - a.double() @ w.double().t()).abs().max()) <= 1e-5 * float((a.double() @ w.double().t()).abs().max())
    # explicit-map index composition
    lut = _t(rng.integers(-1, 20, (999,)).astype(np.int32), cuda)
    src = _t(rng.integers(0, 999, (3, 41, 53)).astype(np.int64), cuda)
    rb, rv, rp = window((3, 41, 53), torch.int32)
    err = torch.zeros(1, dtype=torch.int32, device=cuda)
    eod._lib.check(eod._lib.lib().eod_remap_indices(src.data_ptr(), 1, src.numel(), lut.data_ptr(), 0, lut.numel(), 1, 21, rv.data_ptr(), err.data_ptr(),
                                                    torch.cuda.current_stream().cuda_stream), "eod_remap_indices")
    torch.cuda.synchronize()
    assert intact(rb, rp) and int(err.item()) == 0 and torch.equal(rv.long(), lut.long()[src] + 1)
    # sampling scan: vectorised (HW % 16 == 0) and scalar planes
    for hw in (16 * 1025, 47 * 81):
        obs = _t((rng.uniform(size=(2, hw)) < 0.3).astype(np.uint8), cuda)
        sb, sv, sp = window((2, hw), torch.uint8)
        eod.ops.sample_mask(obs, 8, samp=sv)
        torch.cuda.synchronize()
        assert intact(sb, sp), hw


def test_edge_frames_through_step(eod, cuda):
    """Degenerate frames through the public step APIs against the oracle: the smallest image the read accepts (32x32, one L2
    pixel), a single episode, a frame without depth (every pixel is clipped onto one border cell: a single 1024-pixel run), a
    frame in which no episode has a detection (nothing may change), and a reset in the middle."""
    H = W = 32
    C, mw, mh, cell, E = 128, 9, 7, 0.5, 1
    cells = mw * mh
    intr = eod.compute_intrinsics(W, H, math.radians(67.5))
    rng = np.random.default_rng(3)
    batch = eod.EpisodeBatch(E, mw, mh, C, H, W, cuda)
    shifts = _t(np.array([[0, 0, 0, -2.0, 0, -1.5]], np.float32), cuda)
    sums, counts = torch.zeros(cells, C), torch.zeros(cells)
    xyzhe = np.array([[0.3, 1.25, 0.2, 0.7, math.pi]], np.float32)
    Tm = eod.transform3d(torch.from_numpy(xyzhe))
    pose = Tm[:, :3].reshape(1, 12).to(cuda)
    for t, depth in enumerate((rng.uniform(0.3, 3.0, (1, H, W)).astype(np.float32), np.zeros((1, H, W), np.float32),
                               rng.uniform(0.3, 3.0, (1, H, W)).astype(np.float32))):
        feat = rng.standard_normal((1, C, H, W)).astype(np.float32)
        before = (batch.sums[0].cpu(), batch.counts[0].cpu())
        levels = [l.clone() for l in batch.step(_t(depth, cuda), pose, shifts, intr, cell, _t(feat, cuda))]
        torch.cuda.synchronize()
        idx = oracle.backproject_quantize(depth[0], Tm[0].numpy(), intr, np.zeros(3, np.float32), np.array([-2.0, 0, -1.5], np.float32),
                                          np.float32(cell), mw, mh, 0, 0.5, want=("idx",))["idx"]
        assert np.array_equal(batch.idx[0].cpu().numpy(), idx)
        if t == 1:
            assert len(np.unique(idx)) == 1                                  # no depth: one cell for the whole frame
        ref_levels = R.read_frame(before[0], before[1], torch.from_numpy(idx).long())
        for k in range(3):
            assert np.array_equal(levels[k][0].contiguous().cpu().numpy().view(np.uint16), ref_levels[k][0].numpy().view(np.uint16)), (t, k)
        sums, counts = R.write_mean_frame(sums, counts, torch.from_numpy(feat), torch.ones(H, W, dtype=torch.bool), torch.from_numpy(idx).long(), stride=1)
        assert (batch.sums[0].cpu() - sums).abs().max().item() <= SUM_TOL * sums.abs().max().item(), t
        assert torch.equal(batch.counts[0].cpu(), counts)
    # a frame without any detection: the object write must leave sums, counts and the fp16 table alone
    snap = (batch.sums.clone(), batch.counts.clone(), batch.norm16.clone())
    n_obj = _t(np.zeros(1, np.int32), cuda)
    batch.step_detections(_t(rng.uniform(0.3, 3.0, (1, H, W)).astype(np.float32), cuda), pose, shifts, intr, cell,
                          torch.zeros((1, 4, C), device=cuda), torch.ones((1, 4, 28, 28), device=cuda),
                          _t(np.tile(np.array([0, 0, W, H], np.float32), (1, 4, 1)), cuda), n_obj)
    torch.cuda.synchronize()
    assert torch.equal(batch.sums, snap[0]) and torch.equal(batch.counts, snap[1]) and torch.equal(batch.norm16, snap[2])
    batch.reset()
    torch.cuda.synchronize()
    assert not batch.sums.any() and not batch.counts.any() and not batch.norm16.any()


# --------------------------------------------------------------------------------------------------------
# per-ROI read (north star subsystem 3; detic_roi_heads.py:331-334 applied to the memory levels)
# --------------------------------------------------------------------------------------------------------
def _roi_boxes(rng, n, H, W):
    """Proposal-like boxes: all three FPN levels, fractional corners, boxes on the image border, a degenerate and a full-image one,
    and sizes on the level-assignment knife edges (sqrt(area) = 112, 224, 448 up to an ulp)."""
    cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
    s = np.exp(rng.uniform(np.log(8), np.log(min(H, W)), n))
    ar = np.exp(rng.uniform(-1, 1, n))
    bw, bh = s * np.sqrt(ar), s / np.sqrt(ar)
    b = np.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1)
    b[:, [0, 2]] = np.clip(b[:, [0, 2]], 0, W)
    b[:, [1, 3]] = np.clip(b[:, [1, 3]], 0, H)                         # _create_proposals_from_boxes clips to the image (:314)
    b = b.astype(np.float32)
    extra = [[0, 0, W, H], [10, 10, 10, 40], [3.25, 7.5, 3.25 + 224, 7.5 + 224], [0, 0, 112, 112], [1, 1, 1 + 448, 1 + 448 * 0.999999],
             [5, 5, 5 + np.nextafter(np.float32(224), np.float32(0)), 5 + 224], [W - 9.5, H - 7.25, W, H], [0, 0, 0.5, 0.5]]
    return np.concatenate([b, np.asarray(extra, np.float32)], 0)


@pytest.mark.parametrize("C,E", [(128, 1), (256, 3), (512, 2)])
def test_read_roi_matches_executed_roi_align(eod, cuda, C, E):
    """eod_read_roi against torchvision's CPU ROIAlign (executed) over the oracle's pooled levels, with detectron2's level
    assignment: levels assigned exactly, pooled features within 1e-5 of scale."""
    rng = np.random.default_rng(C + E)
    H, W, cells = 480, 640, 3000
    table = _t((rng.standard_normal((E, cells, C)) * 3).astype(np.float16), cuda)
    idx = _t((rng.integers(0, cells, (E, H // 8, W // 8)).repeat(8, 1).repeat(8, 2)).astype(np.int32), cuda)
    levels = eod.ops.read_pool(table, None, idx)
    boxes = [_roi_boxes(rng, 40, H, W) for _ in range(E)]
    bx = _t(np.concatenate(boxes), cuda)
    bi = _t(np.concatenate([np.full(len(b), e, np.int32) for e, b in enumerate(boxes)]), cuda)
    got, lvl = eod.ops.read_roi(levels, bx, bi, 7, want_levels=True)
    torch.cuda.synchronize()
    assert got.shape == (bx.shape[0], C, 7, 7)
    ref, ref_lvl = R.roi_read([l.cpu() for l in levels], [torch.from_numpy(b) for b in boxes])
    assert np.array_equal(lvl.cpu().numpy(), ref_lvl.numpy())                     # ROI -> level assignment: exact
    assert len(set(ref_lvl.tolist())) == 3                                         # the case exercises all three levels
    err = (got.cpu() - ref).abs().max().item()
    assert err <= SUM_TOL * ref.abs().max().item(), err
    # linearity, i.e. why this IS the reference's per-ROI memory term: pooling the fused level == pooled res + w * conv(pooled memory)
    from torchvision.ops import roi_align
    k = 1
    sel = (ref_lvl == k).nonzero().squeeze(1)
    conv = torch.nn.Conv2d(C, 32, 1).double()
    res = torch.randn(E, 32, H // 16, W // 16, dtype=torch.float64)
    fused = res + 5.0 * conv(levels[k].cpu().double())
    rois = torch.cat([bi.cpu().double()[:, None], bx.cpu().double()], 1)[sel]
    lhs = roi_align(fused, rois, (7, 7), 1 / 16, 0, True)
    pooled_mem = got.cpu().double()[sel]
    rhs = roi_align(res, rois, (7, 7), 1 / 16, 0, True) + 5.0 * conv(pooled_mem)
    inside = (rois[:, 3] - rois[:, 1] > 0) & (rois[:, 4] - rois[:, 2] > 0)        # an empty box pools nothing: the bias has no weight there
    assert (lhs - rhs)[inside].abs().max().item() <= 1e-4 * lhs.abs().max().item()


def test_memory_fusion_read_roi_and_episode_batch_read_roi(eod, cuda):
    """The module-level entry points: MemoryFusion.read_roi (reference-facing, lists per image; project=True returns the memory
    term of box_pooler(fused levels)) and EpisodeBatch.read_roi (levels of the current frame)."""
    rng = np.random.default_rng(5)
    C, CO, H, W, cells = 256, 128, 96, 128, 500
    fusion = eod.MemoryFusion("implicit_memory", "sum", 5, mem_feat_dim=C, ego_feat_dim=CO).to(cuda)
    mem16 = [_t((rng.standard_normal((cells, C)) * 2).astype(np.float16), cuda) for _ in range(2)]
    idx = [_t(rng.integers(0, cells, (H // 4, W // 4)).repeat(4, 0).repeat(4, 1).astype(np.int64), cuda) for _ in range(2)]
    boxes = [torch.from_numpy(_roi_boxes(rng, 12, H, W)[:14]).clamp(0, W) for _ in range(2)]
    for b in boxes:
        b[:, [1, 3]] = b[:, [1, 3]].clamp(0, H)
    roi = fusion.read_roi(mem16, idx, boxes)
    levels = fusion.read(mem16, idx, [None, None])
    ref, ref_lvl = R.roi_read([l.cpu() for l in levels], boxes)
    assert (roi.cpu() - ref).abs().max().item() <= SUM_TOL * ref.abs().max().item()
    with torch.no_grad():
        proj = fusion.read_roi(mem16, idx, boxes, project=True).cpu()
        want = torch.zeros_like(proj)
        # the bias is added per level pixel before the pooling (timm.py:174), so it survives with ROIAlign(constant 1): executed here
        ones, _ = R.roi_read([torch.ones((2, 1) + tuple(l.shape[2:])) for l in levels], boxes)
        for k, conv in enumerate(fusion.merge_map_projections):
            sel = (ref_lvl == k).nonzero().squeeze(1)
            if sel.numel():
                want[sel] = 5.0 * (torch.nn.functional.conv2d(ref[sel], conv.weight.cpu()) + conv.bias.cpu().view(1, -1, 1, 1) * ones[sel])
    assert (proj - want).abs().max().item() <= 1e-4 * want.abs().max().item()
    # fusion at the ROI level (north star (4)): box_pooler(fused levels) == fuse_roi(box_pooler(image-only levels)) by linearity of ROIAlign
    with torch.no_grad():
        res = [torch.randn((2, CO, H >> s_, W >> s_), device=cuda) for s_ in (3, 4, 5)]
        fused = fusion(res, mem16, idx, [None, None])
        pooled_res, _ = R.roi_read([r.cpu() for r in res], boxes)
        pooled_fused, _ = R.roi_read([f.cpu() for f in fused], boxes)
        got_roi = fusion.fuse_roi(pooled_res.to(cuda), mem16, idx, boxes).cpu()
    err_roi = (got_roi - pooled_fused).abs().max().item() / pooled_fused.abs().max().item()
    assert err_roi <= 1e-4, err_roi
    batch = eod.EpisodeBatch(2, 25, 20, C, H, W, cuda)
    batch.norm16.copy_(torch.stack(mem16))
    batch.set_indices(torch.stack(idx))
    batch.read()
    bx = torch.cat(boxes).to(cuda)
    bi = torch.cat([torch.full((len(b),), i, dtype=torch.int32) for i, b in enumerate(boxes)]).to(cuda)
    got = batch.read_roi(bx, bi)
    assert (got.cpu() - ref).abs().max().item() <= SUM_TOL * ref.abs().max().item()
