"""The shapes of tests/test_gpu_scale.py (and of the past-cap cases it shares with test_gpu_parity.py / test_gpu_exact.py) against the
sizing helpers with the B200's 148 SMs: every case must take more than one trip of the loop it is there for.  Runs without a GPU."""
import pytest

import test_gpu_scale as S

SMS = 148


@pytest.fixture(autouse=True)
def _default_read_cap(monkeypatch):
    monkeypatch.delenv("EOD_READ_CTAS_PER_SM", raising=False)


def test_helpers_reproduce_the_launchers_caps():
    # one trip exactly at each cap, two just past it
    assert S.read_pool_trips(1, 16 * 8, 16 * 148 * 16, SMS) == 1 and S.read_pool_trips(1, 16 * 8, 16 * (148 * 16 + 1), SMS) == 2
    assert S.pool_level2_trips(1, 32, 32 * 148 * 8 * 256 // 32, 128, SMS) == 1
    assert S.pool_level2_trips(2, 32, 32 * 148 * 8 * 256 // 32, 128, SMS) == 2
    for f in (S.touched_rows_sweeps, S.heightmax_reset_sweeps, S.semmap_update_sweeps):
        assert f(1, 606_208, SMS) == 1 and f(1, 606_209, SMS) == 2
    assert S.heightmax_update_pass_cells(16, 10 ** 6, SMS) == 18_944 and S.heightmax_update_pass_cells(64, 10 ** 6, SMS) == 4_864
    assert S.heightmax_update_pass_cells(64, 1000, SMS) == 1024                   # small list: the list caps the grid, not the SMs
    assert S.fuse_trips(2_424_832, SMS) == 1 and S.fuse_trips(2_424_836, SMS) == 2
    assert S.finalize_cells_trips(1, 4_849_664, 2 * 10 ** 6, SMS) == 1 and S.finalize_cells_trips(1, 4_849_668, 2 * 10 ** 6, SMS) == 2
    assert S.finalize_cells_trips(2, 2 * 10 ** 6, 480 * 640, SMS) == 0               # grid much larger than the image: pixel-driven kernel


def test_read_cap_follows_the_environment_knob(monkeypatch):
    E, H, W = 16, 480, 640                                                        # 19 200 quadrants
    assert S.read_pool_trips(E, H, W, SMS) == 2
    monkeypatch.setenv("EOD_READ_CTAS_PER_SM", "64")
    assert S.read_ctas_per_sm() == 64 and S.read_pool_trips(E, H, W, SMS) == 1
    for bad in ("0", "-3", "x", ""):
        monkeypatch.setenv("EOD_READ_CTAS_PER_SM", bad)
        assert S.read_ctas_per_sm() == 16
    monkeypatch.setenv("EOD_READ_CTAS_PER_SM", "2abc")                            # atoi reads the leading digits
    assert S.read_ctas_per_sm() == 2


def test_read_cases_loop():
    for C in (128, 256, 512):
        assert S.read_pool_trips(S.READ_E, S.READ_H, S.READ_W, SMS) > 1
        assert S.pool_level2_trips(S.READ_E, S.READ_H, S.READ_W, C, SMS) > 1
    for p in S.READ_FAR.values():
        assert p["e"] < p["E"] and p["e"] * p["n_cells"] * p["C"] >= 2 ** 31


def test_configs1_case_loops_and_lies_past_2_31():
    p = S.DENSE
    n = p["mw"] * p["mh"]
    assert S.finalize_cells_trips(p["E"], n, p["H"] * p["W"], SMS) > 1
    assert S.read_pool_trips(p["E"], p["H"], p["W"], SMS) > 1 and S.touched_rows_sweeps(p["E"], n, SMS) > 1
    first_far = min(e for e in range(p["E"]) if e * n * p["C"] >= 2 ** 31)
    assert first_far == 34 and set(p["checked"]) == {0, first_far, p["E"] - 1}
    assert p["E"] - 1 in S.DENSE_RESET and not set(S.DENSE_RESET) & set(S.DENSE_KEEP)
    straddle = [e for e in S.DENSE_RESET if (e * n) % 32]                        # slots that start inside a 32-row chunk
    assert straddle and any(e - 1 in S.DENSE_RESET for e in straddle) and any(e - 1 in S.DENSE_KEEP for e in straddle)


def test_configs2_case_loops_and_lies_past_2_31():
    p = S.HMAX
    n = p["mw"] * p["mh"]
    assert S.heightmax_reset_sweeps(p["E"], n, SMS) > 1
    assert min(e for e in range(p["E"]) if e * n * p["C"] >= 2 ** 31) == 9 and set(p["checked"]) == {0, 9, p["E"] - 1}
    assert not set(S.HMAX_RESET) & set(S.HMAX_KEEP)


def test_heightmax_list_case_is_ragged():
    p = S.HLIST
    n = p["mw"] * p["mh"]
    assert n % 32 and S.heightmax_update_pass_cells(p["E"], min(n, p["H"] * p["W"]), SMS) == 19 * 256


def test_sweep_cases_loop_and_straddle():
    p = S.SWEEP
    assert p["n_cells"] % 32
    for f in (S.touched_rows_sweeps, S.heightmax_reset_sweeps):
        assert f(p["E"], p["n_cells"], SMS) > 2                                   # later sweeps straddle episodes too
    assert all(len(m) == p["E"] and any(m) for m in S.SWEEP_MASKS.values()) and S.SWEEP_MASKS["last"] == (0,) * (p["E"] - 1) + (1,)
    assert S.semmap_update_sweeps(3, 250_007, SMS) > 1 and 250_007 % 32          # test_gpu_exact.py::test_semmap_update_exact[128-past-sweep]
    assert S.fuse_trips(S.FUSE_N, SMS) > 1 and S.FUSE_N % 4                      # test_gpu_parity.py::test_fuse_bit_exact
