"""CPU checks of what tests/exact_cases.py promises: on its inputs every partial sum is exact in fp32, so the float64 result is an fp32
number whatever the summation order, and the torch-CPU oracle (reference_ops) returns exactly those bits.  tests/test_gpu_exact.py
relies on this to compare the accumulating kernels with torch.equal."""
import numpy as np
import pytest
import torch

from oracle import reference_ops as R

import exact_cases as X


def _orders(rng, v):
    """float32 sums of the rows of v (n, C) in forward, reversed, random, pairwise and 32-chunked order."""
    v = np.asarray(v, np.float32)
    out = {}
    for name, p in (("forward", np.arange(len(v))), ("reversed", np.arange(len(v))[::-1]), ("random", rng.permutation(len(v)))):
        acc = np.zeros(v.shape[1], np.float32)
        for x in v[p]:
            acc = acc + x
        out[name] = acc
    w = v.copy()
    while len(w) > 1:                                    # pairwise tree (odd tail carried up)
        h = len(w) // 2
        nxt = w[:h] + w[h:2 * h]
        w = np.concatenate([nxt, w[2 * h:]]) if len(w) % 2 else nxt
    out["pairwise"] = w[0] if len(w) else np.zeros(v.shape[1], np.float32)
    chunks = [np.sum(v[i:i + 32], axis=0, dtype=np.float32) for i in range(0, len(v), 32)]
    acc = np.zeros(v.shape[1], np.float32)
    for c in chunks:
        acc = acc + c
    out["chunked32"] = acc
    return out


def _cell_sums_any_order(rng, feat_chw, idx, samp, sums0, max_cells=64):
    """Per cell: sums0 + sum(f)/n and sums0 + sum(f/n), each in five orders, against the float64 result."""
    cells = sums0.shape[0]
    ref, bound, n = X.mean_write_f64(sums0, feat_chw, idx, samp, cells)
    C = feat_chw.shape[0]
    f = feat_chw.reshape(C, -1).T
    i = idx.reshape(-1)
    if samp is not None:
        f, i = f[samp.reshape(-1).astype(bool)], i[samp.reshape(-1).astype(bool)]
    written = np.nonzero(n)[0]
    big = written[np.argsort(-n[written])][:4]                           # the largest cells, then a random selection
    pick = np.unique(np.concatenate([big, rng.choice(written, min(max_cells, written.size), replace=False)]))
    for c in pick:
        v = f[i == c]
        inv = np.float32(1.0) / np.float32(n[c])
        for name, s in _orders(rng, v).items():
            assert np.array_equal(sums0[c] + s / np.float32(n[c]), ref[c]), (c, name)
        for name, s in _orders(rng, np.concatenate([sums0[c][None], v * inv])).items():
            assert np.array_equal(s, ref[c]), (c, name, "scaled")
    assert np.array_equal(ref.astype(np.float32).astype(np.float64), ref)
    return ref, bound, n


@pytest.mark.parametrize("H,W,samp_p,big", [(96, 128, None, None), (96, 128, 0.3, None), (30, 52, 0.5, None), (480, 640, None, 1 << 18)],
                         ids=["dense", "sampled", "ragged", "2^18-cell"])
def test_index_plane_counts_are_powers_of_two_and_sums_exact_in_any_order(H, W, samp_p, big):
    rng = np.random.default_rng(H + W)
    C, cells, qf = 8, 3000, 3
    samp = None
    if samp_p is not None:
        samp = rng.random((H, W)) < samp_p
        samp[: H // 3] = False                                            # whole tiles without a sample
    idx = X.index_plane(rng, H, W, cells, samp, max_log2=6, big=big)
    n = X.sample_counts(idx, samp, cells)
    X.assert_pow2_counts(n)
    assert (n == 1).sum() > 0
    if big:
        assert n.max() == big
    vis = np.zeros(cells, bool)
    vis[np.unique(idx)] = True
    if samp is not None:
        assert (vis & (n == 0)).sum() > 0                                  # visible without a sample
    feat = X.dyadic(rng, (C, H, W), 3, qf)
    q = qf + int(np.log2(n.max()))
    sums0 = X.dyadic(rng, (cells, C), 20, q)                              # |sums0| < 2^(20-q): room left for the means
    ref, bound, _ = _cell_sums_any_order(rng, feat, idx, samp, sums0)
    X.check_lattice([feat, sums0], q, bound)


def test_lattice_check_rejects_off_lattice_and_oversized_values():
    X.check_lattice([np.array([0.25, -3.5])], 2, 100.0)
    with pytest.raises(AssertionError):
        X.check_lattice([np.array([0.125])], 2, 1.0)
    with pytest.raises(AssertionError):
        X.check_lattice([np.array([1.0])], 2, 2.0 ** 22)
    assert X.lattice_q(np.array([0.75, 3.0])) == 2 and X.lattice_q(np.array([4.0, 0.0])) == -2


def test_oracle_write_and_read_equal_float64_evaluation():
    """R.write_mean_frame (torch index_add_ in fp32) gives the float64 bits on these inputs over several frames, and R.read_frame
    equals a float64 evaluation of the same read."""
    rng = np.random.default_rng(5)
    H, W, C, cells, T = 96, 128, 16, 2000, 4
    sums = torch.zeros(cells, C)
    counts = torch.zeros(cells)
    s64 = np.zeros((cells, C))
    c64 = np.zeros(cells)
    for t in range(T):
        samp = (rng.random((H, W)) < 0.4) if t % 2 else None
        idx = X.index_plane(rng, H, W, cells, samp, max_log2=5)
        feat = X.dyadic(rng, (1, C, H, W), 3, 2)
        obs = torch.ones(H, W, dtype=torch.bool)
        levels = R.read_frame(sums, counts, torch.from_numpy(idx).long())
        mem = np.where((c64 > 1)[:, None], s64 / np.maximum(c64, 1)[:, None], s64)
        t16 = mem.astype(np.float32).astype(np.float16).astype(np.float64)
        ego = t16[idx.reshape(-1)].reshape(H, W, C)
        l4 = ego.reshape(H // 4, 4, W // 4, 4, C).mean((1, 3))
        for k in range(3):
            l4 = l4.reshape(l4.shape[0] // 2, 2, l4.shape[1] // 2, 2, C).mean((1, 3)).astype(np.float16).astype(np.float64)
            assert np.array_equal(levels[k][0].numpy(), l4.transpose(2, 0, 1)), (t, k)
        if samp is None:
            sums, counts = R.write_mean_frame(sums, counts, torch.from_numpy(feat), obs, torch.from_numpy(idx).long(), stride=1)
        else:
            # the oracle samples every stride-th observed pixel: stride 1 over the observed set = samp
            sums, counts = R.write_mean_frame(sums, counts, torch.from_numpy(feat), torch.from_numpy(samp), torch.from_numpy(idx).long(), stride=1)
        s64, bound, n = X.mean_write_f64(s64, feat[0], idx, samp, cells)
        c64[np.unique(idx)] += 1
        assert np.array_equal(sums.numpy(), s64.astype(np.float32)) and np.array_equal(s64.astype(np.float32).astype(np.float64), s64), t
        assert np.array_equal(counts.numpy(), c64)


def test_object_case_overlaps_and_oracle_chain_exact():
    """Pasted masks overlap 1, 2 or 4 times; idx planes built on the stride-8 sample ranks give power-of-two cells; the oracle chain
    box_to_image_features -> write_mean_frame equals the float64 evaluation; the >128-object case too."""
    rng = np.random.default_rng(8)
    H, W, C, cells = 96, 128, 16, 1500
    for n_base in (6, 40):
        case = X.object_case(rng, H, W, C, n_base)
        masks = case["masks"]
        if n_base == 40:
            assert masks.shape[0] > 40
        obs = masks.any(0)
        samp = R.sample_mask(torch.from_numpy(obs), 8).numpy()
        idx = X.index_plane(rng, H, W, cells, samp, max_log2=4)
        X.assert_pow2_counts(X.sample_counts(idx, samp, cells))
        img, o = R.box_to_image_features(torch.from_numpy(case["box_features"]), torch.from_numpy(masks))
        mean64 = X.object_mean_f64(case["box_features"], masks)
        assert np.array_equal(img[0].reshape(C, -1).numpy(), mean64)
        sums, counts = R.write_mean_frame(torch.zeros(cells, C), torch.zeros(cells), img, o, torch.from_numpy(idx).long(), stride=8)
        ref, bound, n = X.mean_write_f64(np.zeros((cells, C)), mean64.reshape(C, H, W), idx, samp, cells)
        X.check_lattice([case["box_features"]], 2 + 2 + int(np.log2(n.max())), bound)
        assert np.array_equal(sums.numpy().astype(np.float64), ref)


def test_gemm_operands_exact_in_float32():
    """project_fuse operands (fp16 levels x exact-fp16 weights, and a weight with a nonzero W_lo) and linear_rows operands (11
    significant bits): the fp32 GEMM in any order equals the float64 one; the hi / lo split reassembles the weight exactly."""
    rng = np.random.default_rng(9)
    x = X.dyadic(rng, (300, 512), 3, 2, np.float16)
    for w in (X.dyadic(rng, (128, 512), 3, 4), X.weights_with_lo(rng, (128, 512))):
        hi, lo = X.split_weights_f64(w)
        assert np.array_equal(hi.astype(np.float64) + lo.astype(np.float64) * 2.0 ** -11, w.astype(np.float64))
        x64 = x.astype(np.float64)
        ref = x64 @ w.astype(np.float64).T
        q = max(X.lattice_q(x64) + X.lattice_q(hi), X.lattice_q(x64) + X.lattice_q(lo) + 11)
        X.check_lattice([ref], q, float(X.gemm_bound(x64, w).max()))
        assert np.array_equal((x.astype(np.float32) @ w.T).astype(np.float64), ref)
        assert np.array_equal((x.astype(np.float32)[:, ::-1] @ w[:, ::-1].T).astype(np.float64), ref)
    assert (X.split_weights_f64(X.weights_with_lo(rng, (128, 512)))[1] != 0).mean() > 0.2
    a = X.dyadic(rng, (257, 96), 6, 3)
    w = X.dyadic(rng, (48, 96), 6, 6)
    assert X.tf32_exact(a) and X.tf32_exact(w)
    ref = a.astype(np.float64) @ w.astype(np.float64).T
    X.check_lattice([ref], 9, float(X.gemm_bound(a, w).max()))
    assert np.array_equal((a @ w.T).astype(np.float64), ref)
