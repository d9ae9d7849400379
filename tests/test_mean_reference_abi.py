"""ml_mean_state_accumulate / ml_mean_state_bytes without a device: every argument error is reported before any
launch (the pointers below are never dereferenced)."""

import pytest

from momlevel_b200 import _lib

NT, NZ, NCOL = 3, 4, 300


def _bytes(nz=NZ, ncol=NCOL):
    return _lib.lib().ml_mean_state_bytes(nz, ncol)


def _call(dtype=_lib.F32, vdtype=_lib.F32, flags=3, nt=NT, nz=NZ, ncol=NCOL, acc=None, acc_bytes=0, w=None,
          ptrs=None):
    L = _lib.lib()
    before = L.ml_launch_count()
    p = dict(T=16, S=16, V=16, T_mean=16, S_mean=16, V_mean=16)
    p.update(ptrs or {})
    rc = L.ml_mean_state_accumulate(dtype, p["T"], p["S"], p["V"], vdtype, w, nt, nz, ncol, acc, acc_bytes, flags,
                                    p["T_mean"], p["S_mean"], p["V_mean"], None)
    assert L.ml_launch_count() == before, "an argument error must return before any launch"
    return rc, L.ml_last_error().decode()


def test_state_bytes():
    # six fp64 running sums per cell: a weighted sum and a weight sum of T, S and volcello
    for nz, ncol in ((75, 1080 * 1440), (1, 1), (7, 4099), (75, 2240 * 2880)):
        assert _bytes(nz, ncol) == 6 * 8 * nz * ncol
    for nz, ncol in ((0, 5), (5, 0), (-1, 5), (5, -3), (1 << 40, 1 << 30)):
        assert _bytes(nz, ncol) == 0


@pytest.mark.parametrize("name", ["T", "S", "V"])
def test_null_field(name):
    rc, msg = _call(ptrs={name: None})
    assert rc == -1 and name in msg, msg


@pytest.mark.parametrize("name", ["T_mean", "S_mean", "V_mean"])
def test_null_output_with_last(name):
    rc, msg = _call(ptrs={name: None})
    assert rc == -1 and name in msg, msg
    # the outputs are not needed without `last`: the missing accumulator is what is reported then
    assert _call(flags=1, ptrs={name: None})[0] == -6


@pytest.mark.parametrize("dt", [dict(dtype=2), dict(dtype=-1), dict(vdtype=2), dict(vdtype=-1)],
                         ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()))
def test_bad_dtype(dt):
    rc, msg = _call(**dt)
    assert rc == -3, msg


@pytest.mark.parametrize("flags", [4, 8, -1, 7])
def test_bad_flags(flags):
    rc, msg = _call(flags=flags, acc=256, acc_bytes=1 << 40)
    assert rc == -5 and "flags" in msg, msg


@pytest.mark.parametrize("ext", [dict(nt=0), dict(nt=-1), dict(nz=0), dict(nz=-2), dict(ncol=0), dict(ncol=-1),
                                 dict(nz=1 << 40, ncol=1 << 30), dict(nt=1 << 40, nz=1 << 20, ncol=1 << 10)],
                         ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()))
def test_bad_extents(ext):
    rc, msg = _call(acc=256, acc_bytes=1 << 62, **ext)
    assert rc == -2 and "extents" in msg, msg


@pytest.mark.parametrize("flags", [0, 1, 2])
def test_accumulator_needed_unless_first_and_last(flags):
    need = _bytes()
    rc, msg = _call(flags=flags, acc=None, acc_bytes=need)
    assert rc == -6 and str(need) in msg, msg
    rc, msg = _call(flags=flags, acc=256, acc_bytes=need - 8)
    assert rc == -6 and str(need) in msg, msg
    assert _call(flags=flags, acc=260, acc_bytes=need)[0] == -7  # not 8-byte aligned


def test_long_first_and_last_call_needs_the_accumulator():
    # more steps than one launch takes (1024): the launches carry the sums through the accumulator
    assert _call(nt=1025)[0] == -6
    assert _call(nt=1025, acc=256, acc_bytes=_bytes() - 1)[0] == -6


def test_misaligned_operands():
    assert _call(ptrs={"T": 18})[0] == -7  # an fp32 field that is not 4-byte aligned
    assert _call(dtype=_lib.F64, ptrs={"S": 20})[0] == -7  # an fp64 field that is not 8-byte aligned
    assert _call(vdtype=_lib.F64, ptrs={"V": 20})[0] == -7
    assert _call(ptrs={"V_mean": 17})[0] == -7
    assert _call(w=12)[0] == -7
