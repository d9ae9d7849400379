"""ml_steric_local_profile / ml_profile_workspace_bytes without a device: every argument error is reported before
any launch (the pointers below are never dereferenced)."""

import pytest

from momlevel_b200 import _lib

NT, NZ, NCOL = 2, 3, 300


def _ws_bytes(nv=3, nt=NT, nz=NZ, ncol=NCOL):
    return _lib.lib().ml_profile_workspace_bytes(nv, nt, nz, ncol)


def _call(eos=0, dtype=_lib.F32, T=16, T_ref=16, S_ref=16, rho_ref=16, weights=16, vref_dtype=_lib.F32,
          outs=(16, 16, 16), ws=256, ws_bytes=None, nt=NT, nz=NZ, ncol=NCOL):
    L = _lib.lib()
    before = L.ml_launch_count()
    if ws_bytes is None:
        ws_bytes = _ws_bytes(sum(o is not None for o in outs) or 1, nt, nz, ncol)
    rc = L.ml_steric_local_profile(eos, dtype, T, 16, T_ref, S_ref, rho_ref, 16, vref_dtype, 16, 16, weights, 16,
                                   -1.0 / 1035.0, nt, nz, ncol, *outs, ws, ws_bytes, None)
    assert L.ml_launch_count() == before, "an argument error must return before any launch"
    return rc, L.ml_last_error().decode()


def test_workspace_bytes():
    # one fp64 per-warp partial per (variant, step, level, 2048-column segment, warp of 8), plus alignment slack
    for nv, nt, nz, ncol in ((1, 12, 75, 1440 * 1080), (3, 12, 75, 1440 * 1080), (2, 1, 1, 1), (3, 13, 7, 4099)):
        assert _ws_bytes(nv, nt, nz, ncol) == nv * nt * nz * (-(-ncol // 2048)) * 8 * 8 + 256
    assert _ws_bytes(1, 5, 5, 300) < _ws_bytes(2, 5, 5, 300) < _ws_bytes(3, 5, 5, 300)


def test_no_output_is_an_error():
    rc, msg = _call(outs=(None, None, None))
    assert rc == -1 and "NULL" in msg


@pytest.mark.parametrize("arg", ["T", "T_ref", "S_ref", "rho_ref", "weights"])
def test_null_inputs(arg):
    assert _call(**{arg: None})[0] == -1


@pytest.mark.parametrize("kw, code", [
    (dict(eos=9), -4),
    (dict(dtype=5), -3),
    (dict(vref_dtype=7), -3),
    (dict(nz=0), -2),
    (dict(ncol=0), -2),
    (dict(nt=-1), -2),
    (dict(nt=1 << 31), -2),
    (dict(T=18), -7),  # an fp32 field that is not 4-byte aligned
    (dict(ws=260), -7),
])
def test_bad_arguments(kw, code):
    rc, msg = _call(**kw)
    assert rc == code, msg


def test_workspace_too_small_or_missing():
    need = _ws_bytes(3)
    rc, msg = _call(ws_bytes=need - 8)
    assert rc == -6 and str(need) in msg
    assert _call(ws=None, ws_bytes=need)[0] == -6
    # the size follows the number of profiles asked for
    assert _call(outs=(None, 16, None), ws_bytes=_ws_bytes(1) - 8)[0] == -6


def test_column_pressure_of_another_grid():
    L = _lib.lib()
    assert L.ml_set_column_pressure(16, NCOL + 1) == 0
    try:
        rc, msg = _call()
        assert rc == -2 and "column pressure" in msg
    finally:
        L.ml_set_column_pressure(None, 0)
