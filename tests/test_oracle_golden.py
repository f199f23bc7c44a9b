"""The oracle (oracle/geometry.c + oracle/reference_ops.py) against fixtures produced by running the reference's own
source (tests/golden/make_golden.py).  CPU only."""
import os

import numpy as np
import pytest
import torch

import oracle
from oracle import reference_ops as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INTR_480 = (320.0, 359.1853942871094, 320.0, 240.0)


@pytest.mark.parametrize("name", ["geometry_small", "geometry_full", "geometry_fine"])
def test_geometry_c_oracle_matches_reference(golden, name):
    g = golden(name)
    T, H, W = g["depth"].shape
    intr = R.intrinsics(W, H, float(g["vfov"]))
    if (H, W) == (480, 640):
        assert intr == INTR_480
    zero = np.zeros(3, np.float32)
    for t in range(T):
        # Projector flow: single shift = map_world_shift
        o = oracle.backproject_quantize(g["depth"][t], g["T"][t], intr, g["map_world_shift"], zero, float(g["cell"]),
                                        int(g["map_w"]), int(g["map_h"]), 0, 0.5)
        assert np.array_equal(o["q2"], g["q2"][t])
        assert np.array_equal(o["outlier"].astype(bool), g["outlier"][t])
        assert np.array_equal(o["height"], g["height"][t])
        # PointCloud + build_memory_data flow: shift0 = 0, shift1 = map_world_shift, clip
        o = oracle.backproject_quantize(g["depth"][t], g["T"][t], intr, zero, g["map_world_shift"], float(g["cell"]),
                                        int(g["map_w"]), int(g["map_h"]), 0, 0.5)
        assert np.array_equal(o["world"], g["world"][t])
        assert np.array_equal(o["idx"], g["flat"][t])


def test_geometry_torch_restatement_matches_reference(golden):
    g = golden("geometry_fine")
    depth, T = torch.from_numpy(g["depth"]), torch.from_numpy(g["T"])
    shift = torch.from_numpy(g["map_world_shift"])
    assert torch.equal(R.transform3d(torch.from_numpy(g["xyzhe"])), T)
    q2, outl, hts = R.projector_forward(depth[:, None], T, float(g["vfov"]), int(g["map_h"]), int(g["map_w"]),
                                        float(g["cell"]), shift, 0.5)
    assert np.array_equal(q2.numpy().astype(np.int32), g["q2"])
    assert np.array_equal(outl.numpy(), g["outlier"])
    assert np.array_equal(hts.numpy(), g["height"])
    flat = R.quantize_flat_index(torch.from_numpy(g["world"]), shift, float(g["cell"]), int(g["map_w"]), int(g["map_h"]))
    assert np.array_equal(flat[..., 0].numpy(), g["flat"])
    # some pixels must exercise the clip and the outlier mask
    assert g["outlier"].mean() > 0.05 and ((g["q2"] < 0) | (g["q2"] >= int(g["map_w"]))).any()


def _unpack(bits, shape):
    return np.unpackbits(bits)[: int(np.prod(shape))].reshape(shape).astype(bool)


def test_write_restatement_matches_reference(golden):
    g = golden("write_mean")
    n_cells = int(g["map_w"]) * int(g["map_h"])
    sums, counts = torch.zeros(n_cells, 512), torch.zeros(n_cells)
    for t in range(3):
        K = int(g[f"K{t}"])
        masks = torch.from_numpy(_unpack(g[f"masks{t}"], (K, 480, 640)))
        bf = torch.from_numpy(g[f"box_features{t}"])
        proj = torch.from_numpy(g[f"idx{t}"]).long()
        img, observed = R.box_to_image_features(bf, masks)
        assert np.array_equal(observed.numpy(), _unpack(g[f"observed{t}"], (480, 640)))
        assert np.array_equal(img[0, :, ::16, ::16].numpy(), g[f"img_sample{t}"])          # bit-exact (same add order)
        mean_d, om_d = R.project_image_features_dense(img, observed, proj, n_cells)
        mean_s, om_s = R.project_image_features_sparse(img, observed, proj, n_cells)
        assert np.array_equal(om_d.numpy(), g[f"observed_mem{t}"]) and np.array_equal(om_s.numpy(), g[f"observed_mem{t}"])
        scale = np.abs(g[f"mean{t}"]).max()
        assert np.abs(mean_d.numpy() - g[f"mean{t}"]).max() <= 1e-6 * scale
        assert np.abs(mean_s.numpy() - g[f"mean{t}"]).max() <= 1e-5 * scale
        sums, counts = R.accumulate(sums, counts, mean_d, om_d, proj)
        assert np.abs(sums.numpy() - g[f"sums{t}"]).max() <= 1e-5 * np.abs(g[f"sums{t}"]).max()
        assert np.array_equal(counts.numpy(), g[f"counts{t}"])
        norm = R.create_implicit_memory(torch.from_numpy(g[f"sums{t}"]), torch.from_numpy(g[f"counts{t}"]))
        assert np.array_equal(norm.numpy(), g[f"norm{t}"])
        # the sampling mask helper selects exactly the pixels the reference's [::8] keeps
        samp = R.sample_mask(observed, 8)
        assert int(samp.sum()) == (int(observed.sum()) + 7) // 8
        assert np.array_equal(np.unique(proj[samp].numpy()), np.nonzero(g[f"observed_mem{t}"])[0])


def test_read_restatement_matches_reference(golden):
    g = golden("read_fuse")
    sums, counts = torch.from_numpy(g["sums"]), torch.from_numpy(g["counts"])
    mem16 = R.create_implicit_memory(sums, counts).to(torch.half)
    ws = [torch.from_numpy(g[f"w{k}"]) for k in range(3)]
    bs = [torch.from_numpy(g[f"b{k}"]) for k in range(3)]
    for t in range(2):
        proj = torch.from_numpy(g[f"idx{t}"]).long()
        levels = R.read_pool(mem16, proj)
        for k in range(3):
            assert np.array_equal(levels[k].numpy().view(np.uint16), g[f"level{t}_{k}"].view(np.uint16))
        res = [torch.from_numpy(g[f"res{t}_{k}"]).float() for k in range(3)]
        for fusion in (("sum", "mem_only", "image_only") if t == 0 else ("sum",)):
            fused = R.project_and_fuse(levels, res, ws, bs, 5, fusion)
            for k in range(3):
                ref = g[f"fused_{fusion}_{t}_{k}"]
                if fusion == "image_only":
                    assert np.array_equal(fused[k].numpy(), ref)
                else:
                    # the 1x1 conv's fp32 sums round with the CPU's conv kernel (its blocking follows the instruction set and the
                    # thread count), so hosts differ in the last bits (up to ~3e-7 of scale seen): agreement within 1e-6 of scale
                    assert np.abs(fused[k].numpy() - ref).max() <= 1e-6 * np.abs(ref).max(), (fusion, t, k)
        # plain-C pooling chain == torch chain, bit for bit
        L = oracle.read_pool_f16(mem16.numpy(), g[f"idx{t}"])
        for k in range(3):
            assert np.array_equal(L[k].view(np.uint16), levels[k][0].numpy().view(np.uint16))


def test_sequential_cell_sums_c_vs_numpy():
    rng = np.random.default_rng(0)
    C, H, W, cells = 8, 16, 32, 40
    feat = rng.standard_normal((C, H, W)).astype(np.float32)
    idx = rng.integers(0, cells, (H, W)).astype(np.int32)
    samp = (rng.uniform(size=(H, W)) < 0.5).astype(np.uint8)
    s, n = oracle.cell_sums_seq(feat, idx, samp, cells)
    ref = np.zeros((cells, C), np.float32)
    sel = samp.reshape(-1).astype(bool)
    np.add.at(ref, idx.reshape(-1)[sel], feat.reshape(C, -1).T[sel])       # unbuffered, raster order
    assert np.array_equal(s, ref)
    assert np.array_equal(n, np.bincount(idx.reshape(-1)[sel], minlength=cells))


def test_scatter_max_canonical_rule():
    src = torch.tensor([1.0, 5.0, 5.0, 2.0, 7.0, 3.0])
    index = torch.tensor([0, 0, 0, 1, 2, 2])
    out = torch.tensor([0.0, 2.0, 9.0, 4.0])
    o, arg = R.scatter_max_canonical(src, index, out)
    assert o.tolist() == [5.0, 2.0, 9.0, 4.0]
    assert arg.tolist() == [2, 3, -1, -1]         # tie -> highest index; equal to old -> replaced; lower -> -1


def test_explicit_semmap_restatement_matches_reference(golden):
    """custom_rcnn.py:747-751 + visualise_clip_image_features executed from the reference source (semmap.npz) vs the
    oracle restatement: intensity plane and labels bit-exact."""
    g = golden("semmap")
    for th in (0.4, 0.1):
        sem, inten, _ = R.explicit_semmap(torch.from_numpy(g["sums"]), torch.from_numpy(g["counts"]), torch.from_numpy(g["zs_weight"]), th)
        assert np.array_equal(inten.numpy(), g["intensity"])
        assert np.array_equal(sem.numpy(), g[f"semmap_{th}"])


@pytest.mark.parametrize("name", ["plain", "edge"])
def test_paste_masks_c_oracle_matches_torch_golden(golden, name):
    """oracle/paste.c against the fixture produced by torch-CPU (restated paste_masks_in_image, executed F.grid_sample):
    pasted bools identical, sampled values identical bit for bit (pins the fma order of the sampler)."""
    g = golden("paste")
    H, W = int(g["H"]), int(g["W"])
    probs, boxes = g[name + "_probs"], g[name + "_boxes"]
    ref = _unpack(g[name + "_masks_bits"], (probs.shape[0], H, W))
    masks, values = oracle.paste_masks(probs, boxes, H, W, float(g["thr"]), want_values=True)
    assert np.array_equal(masks, ref)
    for k in range(2):
        y0, y1, x0, x1 = g[f"{name}_val{k}_yx"]
        assert np.array_equal(values[k, y0:y1, x0:x1].view(np.uint32), g[f"{name}_val{k}"].view(np.uint32))


def test_paste_masks_torch_restatement_matches_c_oracle_randomised():
    """The torch restatement (executes ATen's grid_sample on this host) and the C restatement agree on seeded detections,
    including boxes that leave the image; skipped on hosts whose ATen build takes the non-vectorised sampler."""
    if torch.backends.cpu.get_cpu_capability() == "DEFAULT":
        pytest.skip("scalar ATen grid_sample rounds differently (no fma); canonical is the AVX2 / AVX-512 build")
    import importlib
    episodes = importlib.import_module("embodied-object-detection_b200.episodes")
    rng = np.random.default_rng(5)
    H, W = 120, 160
    for edge in (False, True):
        _, probs, boxes = episodes.make_mask_head_detections(rng, H, W, 8, (6, 9), 28, edge_cases=edge)
        ref = R.paste_masks_in_image(torch.from_numpy(probs), torch.from_numpy(boxes), (H, W), 0.5).numpy()
        assert np.array_equal(oracle.paste_masks(probs, boxes, H, W, 0.5), ref)
        assert ref.any()


def test_robot_demo_geometry_oracle_and_host_pose_match_reference(eod, golden):
    """Online robot variant (robot_demo.py:40-90,92-225,514-534 executed from source -> robot.npz): the host pose with the axis
    swap is bit-identical to the reference's matmul(T, R), and the C oracle reproduces the column-major flat indices."""
    g = golden("robot")
    H, W = g["depth_mm"].shape[1:]
    K = tuple(float(np.float32(v)) for v in g["K"])
    for t in range(g["depth_mm"].shape[0]):
        pv = g["pose_val"][t]
        xyzhe = torch.FloatTensor(np.array([[pv[0], 0.65, pv[1], -1 * pv[2], np.pi + 0.06]]))       # robot_demo.py:518-519
        T = eod.transform3d(xyzhe, axis_swap=True)
        assert np.array_equal(T.numpy().view(np.uint32), g["T"][t:t + 1].view(np.uint32))
        depth = torch.FloatTensor(g["depth_mm"][t] / 1000).numpy()                                   # :514-516
        out = oracle.backproject_quantize(depth, g["T"][t], K, np.zeros(3, np.float32), g["map_world_shift"], np.float32(g["res"]),
                                          int(g["map_w"]), int(g["map_h"]), 1, 3.0, want=("idx",))
        assert np.array_equal(out["idx"], g["flat"][t])


def test_paste_masks_c_oracle_vs_torch_on_threshold_knife_edges():
    """Masks that sit exactly on the threshold (constant 0.5, {0, 0.5, 1} lattices, +-1e-5 around 0.5), NaN / Inf probabilities,
    integer / half-integer / sub-pixel / oversized boxes: the C restatement and torch-CPU's grid_sample must agree on every pasted
    bool - this is where a different fma order would show."""
    if torch.backends.cpu.get_cpu_capability() == "DEFAULT":
        pytest.skip("scalar ATen grid_sample rounds differently (no fma); canonical is the AVX2 / AVX-512 build")
    rng = np.random.default_rng(1)
    H, W, K = 60, 80, 5
    for case in range(18):
        S = int(rng.choice([28, 14, 7]))
        kind = case % 6
        if kind == 0:   probs = np.full((K, S, S), 0.5, np.float32)
        elif kind == 1: probs = rng.choice([0.0, 0.5, 1.0], (K, S, S)).astype(np.float32)
        elif kind == 2: probs = (rng.integers(0, 3, (K, S, S)) * 0.25 + 0.25).astype(np.float32)
        elif kind == 3: probs = rng.uniform(0.49999, 0.50001, (K, S, S)).astype(np.float32)
        elif kind == 4: probs = rng.uniform(0, 1, (K, S, S)).astype(np.float32)
        else:
            probs = rng.uniform(0, 1, (K, S, S)).astype(np.float32)
            probs[0, 3, 3] = np.nan; probs[1, 2, 2] = np.inf; probs[2, 1, 1] = -np.inf
        boxes = np.zeros((K, 4), np.float32)
        for k in range(K):
            t = k % 5
            if t == 0:   x0, y0 = rng.integers(0, W - 30), rng.integers(0, H - 30); boxes[k] = (x0, y0, x0 + rng.integers(1, 30), y0 + rng.integers(1, 30))
            elif t == 1: x0, y0 = rng.integers(0, W - 30) + 0.5, rng.integers(0, H - 30) + 0.5; boxes[k] = (x0, y0, x0 + 28, y0 + 28)
            elif t == 2: x0, y0 = rng.uniform(-5, W - 4), rng.uniform(-5, H - 4); boxes[k] = (x0, y0, x0 + rng.uniform(0.01, 3), y0 + rng.uniform(0.01, 3))
            elif t == 3: boxes[k] = (rng.uniform(-50, 0), rng.uniform(-50, 0), W + rng.uniform(0, 50), H + rng.uniform(0, 50))
            else:        x0, y0 = rng.uniform(0, W - 40), rng.uniform(0, H - 40); boxes[k] = (x0, y0, x0 + rng.uniform(5, 40), y0 + rng.uniform(5, 40))
        for thr in (0.5, 0.25):
            ref = R.paste_masks_in_image(torch.from_numpy(probs), torch.from_numpy(boxes), (H, W), thr).numpy()
            assert np.array_equal(oracle.paste_masks(probs, boxes, H, W, thr), ref), (case, thr)


def test_bytecode_listings_pin_the_unsourced_write_variants(tmp_path):
    """SURVEY 8a rows A7' / A7'' / A14 exist only as bytecode.  oracle/pyc_disasm.py (own marshal reader: the 3.12 interpreter cannot
    load 3.9 / 3.10 code objects) produced the listings under oracle/disasm/ that the restatements cite; this test pins the
    facts the canonical rules rest on, and - where EOD_REFERENCE_ROOT names a checkout of the original project - that the committed
    listings regenerate from its .pyc files."""
    import re
    from oracle import pyc_disasm
    d = os.path.join(ROOT, "oracle", "disasm")
    enc = open(os.path.join(d, "smnet_encode_model_test_py39.txt")).read()
    # height_map, idx = scatter_max(height + 1000, flat[inliers], dim=0, out=height_map); m = idx >= 0; observed += m
    assert re.search(r"LOAD_GLOBAL\s+\d+\s+\(scatter_max\)", enc) and "('dim', 'out')" in enc
    assert re.search(r"LOAD_CONST\s+\d+\s+\(1000\)\n\s+\d+ INPLACE_ADD", enc)
    i = enc.index("(scatter_max)")
    tail = enc[i:i + 1500]
    assert re.search(r"STORE_FAST\s+\d+\s+\(height_map\)\n\s+\d+ STORE_FAST\s+\d+\s+\(highest_height_indices\)", tail)
    assert re.search(r"\(highest_height_indices\)\n\s+\d+ LOAD_CONST\s+\d+\s+\(0\)\n\s+\d+ COMPARE_OP\s+\d+\s+\(>=\)", tail)
    assert "('size', 'mode', 'align_corners')" in enc and "((480, 640))" in enc and "('bilinear')" in enc
    assert "(rnn)" in enc and "(linlayer)" not in enc                      # model_test: GRU / LSTM update only
    enc310 = open(os.path.join(d, "smnet_encode_model_py310.txt")).read()
    assert "('replace')" in enc310 and "(linlayer)" in enc310              # model.py (3.10): state[m] = linlayer(winners)
    fpn = open(os.path.join(d, "custommapfpn_forward_timm_py39.txt")).read()
    assert "(interpolate)" in fpn and "(map_merge_forward_projection)" in fpn or "(map_merge_memory_projection)" in fpn
    exp = open(os.path.join(d, "create_explicit_memory_custom_rcnn_py39.txt")).read()
    assert "(zs_weight)" in exp or "(semmap)" in exp
    ref_root = os.environ.get("EOD_REFERENCE_ROOT")
    if ref_root:
        made = pyc_disasm.emit(ref_root, str(tmp_path))
        assert len(made) == 4
        for f in made:
            assert open(os.path.join(tmp_path, f)).read() == open(os.path.join(d, f)).read(), f


def test_pyc_disasm_reads_a_minimal_py39_pyc(tmp_path):
    """oracle/pyc_disasm.py on a hand-built CPython 3.9 .pyc (module whose only constant is `def f(): return None`, line 3): the
    single-file mode names the file as given, --emit names it relative to the reference root."""
    import struct
    from oracle import pyc_disasm

    def i32(v):
        return struct.pack("<i", v)

    def tup(*items):
        return b")" + bytes([len(items)]) + b"".join(items)

    def code(name, consts, line):
        ops = b"\x64\x00\x53\x00"                                                      # LOAD_CONST 0, RETURN_VALUE
        return (b"c" + i32(0) * 4 + i32(1) + i32(64) + b"s" + i32(len(ops)) + ops + consts + tup() * 4
                + b"z\x04m.py" + b"z" + bytes([len(name)]) + name.encode() + i32(line) + b"s" + i32(2) + b"\x00\x01")

    pyc = tmp_path / "m.cpython-39.pyc"
    pyc.write_bytes(struct.pack("<H", 3425) + b"\r\n" + bytes(12) + code("<module>", tup(code("f", tup(b"N"), 3)), 1))
    text = pyc_disasm.listing(str(pyc), "f")
    assert text.startswith(f"# {pyc}  ::  f   (CPython 3.9 bytecode, first line 3)\n")
    assert text.splitlines()[-2:] == ["    4      0 LOAD_CONST                   0  (None)", "           2 RETURN_VALUE                  "]
    assert pyc_disasm.listing(str(pyc), "f", str(tmp_path)).startswith("# m.cpython-39.pyc  ::  f   ")


def test_explicit_map_composition_and_read_match_reference(golden):
    """MODEL.MEMORY_TYPE explicit_map: SMNet/loader.py:222,232-246 and timm.py:142-192 executed from source -> explicit_map.npz.  The
    restated composition ((semmap + 1)[proj], zero row in front of the class table) and the oracle's read of the 21-row table must
    equal the reference's outputs bit for bit."""
    g = golden("explicit_map")
    assert np.array_equal(np.insert(g["clip"], 0, np.zeros((1, g["clip"].shape[1])), axis=0).astype(np.float32), g["memory"])
    assert np.array_equal((g["semmap"] + 1)[g["proj"]], g["idx"])
    levels = R.read_pool(torch.from_numpy(g["memory"]).half(), torch.from_numpy(g["idx"]))
    for k in range(3):
        assert np.array_equal(levels[k].numpy().view(np.uint16), g[f"level{k}"].view(np.uint16)), k
