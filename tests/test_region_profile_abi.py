"""ml_steric_local_region_profile / ml_region_profile_workspace_bytes without a device: every argument error is
reported before any launch (the pointers below are never dereferenced)."""

import pytest

from momlevel_b200 import _lib

NT, NZ, NCOL, NREG = 2, 3, 300, 4


def _ws_bytes(nv=3, nreg=NREG, nt=1, nz=NZ, ncol=NCOL):
    return _lib.lib().ml_region_profile_workspace_bytes(nv, nreg, nt, nz, ncol)


def _call(region=16, nregions=NREG, outs=(16, 16, 16), ws=256, ws_bytes=None, nt=NT, T=16):
    L = _lib.lib()
    before = L.ml_launch_count()
    if ws_bytes is None:
        ws_bytes = _ws_bytes(sum(o is not None for o in outs) or 1, max(1, min(nregions, 15)))
    rc = L.ml_steric_local_region_profile(0, _lib.F32, T, 16, 16, 16, 16, 16, _lib.F32, 16, 16, 16, region, nregions,
                                          16, -1.0 / 1035.0, nt, NZ, NCOL, *outs, ws, ws_bytes, None)
    assert L.ml_launch_count() == before, "an argument error must return before any launch"
    return rc, L.ml_last_error().decode()


def test_workspace_bytes():
    # one fp64 per-warp partial per (variant, region, step, level, 2048-column segment, warp of 8), plus slack
    for nv, nreg, nt, nz, ncol in ((1, 11, 12, 75, 1440 * 1080), (3, 15, 1, 75, 1440 * 1080), (2, 1, 1, 1, 1),
                                   (3, 7, 13, 7, 4099)):
        assert _ws_bytes(nv, nreg, nt, nz, ncol) == nv * nreg * nt * nz * (-(-ncol // 2048)) * 8 * 8 + 256
    # linear in the regions and in the steps
    one = _ws_bytes(2, 1, 1, 5, 4099) - 256
    for nreg in (1, 2, 7, 15):
        for nt in (1, 3, 12):
            assert _ws_bytes(2, nreg, nt, 5, 4099) - 256 == nreg * nt * one
    # one region is the workspace of ml_steric_local_profile
    assert _ws_bytes(3, 1, 5, 7, 300) == _lib.lib().ml_profile_workspace_bytes(3, 5, 7, 300)


@pytest.mark.parametrize("nregions", [0, -1, 16, 127])
def test_region_count_out_of_range(nregions):
    rc, msg = _call(nregions=nregions)
    assert rc == -2 and "nregions" in msg, msg


def test_null_region():
    rc, msg = _call(region=None)
    assert rc == -1 and "region" in msg, msg


def test_no_output_is_an_error():
    rc, msg = _call(outs=(None, None, None))
    assert rc == -1 and "NULL" in msg


def test_workspace_below_one_step():
    need = _ws_bytes(3)
    rc, msg = _call(ws_bytes=need - 8)
    assert rc == -6 and str(need) in msg, msg
    assert _call(ws=None, ws_bytes=need)[0] == -6
    # the size follows the number of profiles and of regions asked for
    assert _call(outs=(None, 16, None), ws_bytes=_ws_bytes(1) - 8)[0] == -6
    assert _call(nregions=15, ws_bytes=_ws_bytes(3, 15) - 8)[0] == -6


def test_bad_extents_and_alignment():
    assert _call(nt=-1)[0] == -2
    assert _call(T=18)[0] == -7  # an fp32 field that is not 4-byte aligned
    assert _call(ws=260)[0] == -7


def test_column_pressure_of_another_grid():
    L = _lib.lib()
    assert L.ml_set_column_pressure(16, NCOL + 1) == 0
    try:
        rc, msg = _call()
        assert rc == -2 and "column pressure" in msg
    finally:
        L.ml_set_column_pressure(None, 0)
