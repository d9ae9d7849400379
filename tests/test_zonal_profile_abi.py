"""ml_steric_local_zonal_profile / ml_zonal_profile_workspace_bytes without a device: every argument error is
reported before any launch (the pointers below are never dereferenced)."""

import pytest

from momlevel_b200 import _lib

NT, NZ, NY, NX = 2, 3, 5, 300


def _ws_bytes(nv=3, nt=1, nz=NZ, ny=NY, nx=NX):
    return _lib.lib().ml_zonal_profile_workspace_bytes(nv, nt, nz, ny, nx)


def _call(outs=(16, 16, 16), ws=256, ws_bytes=None, nt=NT, nz=NZ, ny=NY, nx=NX, T=16, ptrs=None):
    L = _lib.lib()
    before = L.ml_launch_count()
    if ws_bytes is None:
        ws_bytes = _ws_bytes(sum(o is not None for o in outs) or 1)
    p = dict(T=T, S=16, T_ref=16, S_ref=16, rho_ref=16, v_ref=16, z_i=16, deptho=16, weights=16, p_level=16)
    p.update(ptrs or {})
    rc = L.ml_steric_local_zonal_profile(0, _lib.F32, p["T"], p["S"], p["T_ref"], p["S_ref"], p["rho_ref"], p["v_ref"],
                                         _lib.F32, p["z_i"], p["deptho"], p["weights"], p["p_level"], -1.0 / 1035.0,
                                         nt, nz, ny, nx, *outs, ws, ws_bytes, None)
    assert L.ml_launch_count() == before, "an argument error must return before any launch"
    return rc, L.ml_last_error().decode()


def test_workspace_bytes():
    # one fp64 per-warp partial per (variant, step, level, grid row, 2048-column sub-tile, warp of 8), plus slack
    for nv, nt, nz, ny, nx in ((1, 12, 75, 1080, 1440), (3, 1, 75, 1080, 1440), (2, 1, 1, 1, 1), (3, 13, 7, 9, 4100),
                               (3, 8, 75, 2240, 2880)):
        assert _ws_bytes(nv, nt, nz, ny, nx) == nv * nt * nz * ny * (-(-nx // 2048)) * 8 * 8 + 256
    # linear in the steps and the rows; a grid row is a one-row call of ml_steric_local_profile
    one = _ws_bytes(2, 1, 5, 1, 4099) - 256
    for ny in (1, 2, 7, 300):
        for nt in (1, 3, 12):
            assert _ws_bytes(2, nt, 5, ny, 4099) - 256 == ny * nt * one
    assert _ws_bytes(3, 5, 7, 1, 300) == _lib.lib().ml_profile_workspace_bytes(3, 5, 7, 300)


@pytest.mark.parametrize("name", ["T", "S", "T_ref", "S_ref", "rho_ref", "v_ref", "z_i", "deptho", "weights",
                                  "p_level"])
def test_null_operand(name):
    rc, msg = _call(ptrs={name: None})
    assert rc == -1, msg


def test_no_output_is_an_error():
    rc, msg = _call(outs=(None, None, None))
    assert rc == -1 and "NULL" in msg


@pytest.mark.parametrize("ext", [dict(nt=-1), dict(nz=0), dict(ny=0), dict(ny=-3), dict(nx=0), dict(nx=-1),
                                 dict(ny=1 << 31), dict(nz=1 << 16, ny=1 << 16), dict(nt=1 << 12, nz=1 << 10, ny=1 << 10)],
                         ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()))
def test_bad_extents(ext):
    rc, msg = _call(ws_bytes=1 << 62, **ext)
    assert rc == -2 and "extents" in msg, msg


def test_workspace_below_one_step():
    need = _ws_bytes(3)
    rc, msg = _call(ws_bytes=need - 8)
    assert rc == -6 and str(need) in msg, msg
    assert _call(ws=None, ws_bytes=need)[0] == -6
    # the size follows the number of profiles asked for, and one step is enough
    assert _call(outs=(None, 16, None), ws_bytes=_ws_bytes(1) - 8)[0] == -6
    assert _call(outs=(None, 16, None), ws_bytes=_ws_bytes(1), nt=0)[0] == 0
    assert _call(ws_bytes=need, nt=0)[0] == 0


def test_misaligned_operands_and_workspace():
    assert _call(T=18)[0] == -7  # an fp32 field that is not 4-byte aligned
    assert _call(ptrs={"S_ref": 17})[0] == -7
    assert _call(ws=260)[0] == -7


def test_column_pressure_of_another_grid():
    L = _lib.lib()
    # the column pressure has one value per (y, x) column of the whole plane, not per row
    for n in (NX, NY * NX + 1):
        assert L.ml_set_column_pressure(16, n) == 0
        try:
            rc, msg = _call()
            assert rc == -2 and "column pressure" in msg
        finally:
            L.ml_set_column_pressure(None, 0)
