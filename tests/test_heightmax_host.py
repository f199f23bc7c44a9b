"""Host side of the height-max regime (no GPU needed): the saved-map format and the refusals that happen before any launch."""
import numpy as np
import pytest
import torch


def test_save_load_heightmax_roundtrip(eod, tmp_path):
    rng = np.random.default_rng(0)
    state = rng.standard_normal((12, 8)).astype(np.float32)
    observed = (rng.uniform(size=12) < 0.5).astype(np.uint8)
    hmap = rng.uniform(999, 1001, 12).astype(np.float32)
    path = eod.formats.save_heightmax(str(tmp_path / "heightmax" / "scene_0.npz"), torch.from_numpy(state), torch.from_numpy(observed), hmap)
    s, o, h = eod.formats.load_heightmax(path)
    assert s.dtype == np.float32 and o.dtype == np.uint8 and h.dtype == np.float32
    assert np.array_equal(s, state) and np.array_equal(o, observed) and np.array_equal(h, hmap)
    eod.formats.write_store(str(tmp_path / "partial.npz"), {"state": state})
    with pytest.raises(eod.formats.StoreError):
        eod.formats.load_heightmax(str(tmp_path / "partial.npz"))


def test_heightmax_refuses_cpu(eod):
    with pytest.raises(eod.EodError):
        eod.HeightMaxBatch(1, 10, 10, 8, 16, 16, torch.device("cpu"))
    scratch = type("S", (), {"E": 1, "n_cells": 100})()
    with pytest.raises(eod.EodError):
        eod.ops.heightmax_contest_planes(torch.zeros((1, 16, 16)), torch.zeros((1, 16, 16), dtype=torch.int32), None, scratch)


def test_runner_rejects_unknown_regime(eod):
    provider = eod.HostEpisodeProvider([], torch.device("cpu"))
    with pytest.raises(ValueError):
        eod.EpisodeRunner(provider, 10, 10, 8, n_slots=1, regime="scatter")
    with pytest.raises(ValueError):
        eod.EpisodeRunner(provider, 10, 10, 8, n_slots=1, regime="heightmax", variant=eod._lib.WRITE_DET)
