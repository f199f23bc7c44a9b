"""Host-side checks of the deterministic object write (no GPU): argument refusals before any device call and the runner's
object_variant validation."""
import pytest

EOD_ERR_BADARG = -1


def test_objects_det_entry_points_refuse_null_arguments(eod):
    eod.build.build()
    lib = eod._lib.lib()
    P = 0x1000                                    # never dereferenced: the argument checks come first
    E, K, C, HW, cells, ws = 2, 4, 128, 96 * 128, 300, 1 << 20
    full = dict(bf=P, masks=P, n_obj=P, idx=P, samp=P, cnt=P, sums=P, ws=P)
    for missing in ("bf", "masks", "idx", "samp", "cnt", "sums", "ws"):
        a = dict(full, **{missing: None})
        rc = lib.eod_write_objects_det(a["bf"], a["masks"], a["n_obj"], K, a["idx"], a["samp"], a["cnt"], E, C, HW, cells, a["sums"],
                                       a["ws"], ws, None)
        assert rc == EOD_ERR_BADARG, missing
    for bad in (dict(E=0), dict(K=0), dict(HW=0), dict(cells=0), dict(ws=0)):
        s = dict(dict(E=E, K=K, HW=HW, cells=cells, ws=ws), **bad)
        rc = lib.eod_write_objects_det(P, P, P, s["K"], P, P, P, s["E"], C, s["HW"], s["cells"], P, P, s["ws"], None)
        assert rc == EOD_ERR_BADARG, bad
    full = dict(bf=P, probs=P, boxes=P, idx=P, samp=P, cnt=P, sums=P, ws=P)
    for missing in full:
        a = dict(full, **{missing: None})
        rc = lib.eod_write_objects_pasted_det(a["bf"], a["probs"], a["boxes"], P, K, 28, 96, 128, 0.5, a["idx"], a["samp"], a["cnt"], E, C,
                                              cells, a["sums"], a["ws"], ws, None)
        assert rc == EOD_ERR_BADARG, missing
    rc = lib.eod_write_objects_pasted_det(P, P, P, P, K, 0, 96, 128, 0.5, P, P, P, E, C, cells, P, P, ws, None)
    assert rc == EOD_ERR_BADARG
    assert "null pointer" in lib.eod_last_error().decode() or "bad sizes" in lib.eod_last_error().decode()


def test_runner_heightmax_refuses_object_variant(eod):
    with pytest.raises(ValueError, match="object_variant"):
        eod.EpisodeRunner(None, 10, 10, 128, 1, regime="heightmax", object_variant=eod._lib.WRITE_DET)


def test_episode_batch_object_variant_is_checked_before_allocation(eod):
    with pytest.raises(ValueError, match="object_variant"):
        eod.EpisodeBatch(1, 10, 10, 128, 8, 64, "cuda", object_variant=eod._lib.WRITE_TMA)
