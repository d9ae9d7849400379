"""CPU tests of the storage dtype that a supplied reference gives the steric entry points (no kernels involved).

An fp64 reference slab handed to fp32 fields must not be rounded to fp32: the device entry points store all four
operands in fp64, and ``core.HostStream`` runs in fp64 unless every value of the slabs is an fp32 value.  The
library is replaced by a recorder, so what is checked is what would cross the C ABI.
"""

import numpy as np
import pytest
import torch

from momlevel_b200 import _lib, core

NZ, NY, NX = 3, 4, 5


class Recorder:
    """Stands in for the CDLL: every entry point records its arguments and returns ML_OK (0)."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append((name, args))
            return 0

        return call

    def args(self, name):
        found = [a for n, a in self.calls if n == name]
        assert len(found) == 1, (name, [n for n, _ in self.calls])
        return found[0]


@pytest.fixture
def rec(monkeypatch):
    r = Recorder()
    monkeypatch.setattr(_lib, "lib", lambda: r)
    monkeypatch.setattr(core, "_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(core, "_stream", lambda: 0)
    return r


def _slabs(seed, dtype, exact=False):
    g = np.random.default_rng(seed)
    T = 2.0 + 25.0 * g.random((NZ, NY, NX))
    S = 33.0 + 3.0 * g.random((NZ, NY, NX))
    T[0, 0, 0] = S[0, 0, 0] = np.nan  # land: NaN must not count as a value that fp32 rounds
    if exact:
        T, S = T.astype(np.float32), S.astype(np.float32)
    return T.astype(dtype), S.astype(dtype)


def _stream(T_ref, S_ref, field_dtype, domain="global", variants=("thermosteric",)):
    V = np.full((NZ, NY, NX), 1.0e9, dtype=np.float32)
    rho = np.full((NZ, NY, NX), 1030.0)
    p = np.arange(NZ, dtype=np.float64) * 1.0e5
    zi = np.arange(NZ + 1, dtype=np.float64) * 10.0
    depth = np.full((NY, NX), 1000.0)
    return core.HostStream(domain, V, p, z_i=zi, deptho=depth, variants=variants,
                           reference={"thetao": T_ref, "so": S_ref, "rho": rho}, dtype=field_dtype)


@pytest.mark.parametrize("domain", ["local", "global"])
@pytest.mark.parametrize("ref_dtype,exact,field_dtype,want", [
    (np.float64, False, torch.float32, _lib.F64),  # a climatology in fp64: the stream runs in fp64
    (np.float32, False, torch.float32, _lib.F32),
    (np.float64, True, torch.float32, _lib.F32),   # an upcast copy of fp32 data: nothing to round, fp32 transfer
    (np.float32, False, torch.float64, _lib.F64),
    (np.float64, False, torch.float64, _lib.F64),
])
def test_host_stream_takes_the_reference_dtype(rec, domain, ref_dtype, exact, field_dtype, want):
    T_ref, S_ref = _slabs(1, ref_dtype, exact)
    hs = _stream(T_ref, S_ref, field_dtype, domain)
    try:
        a = rec.args("ml_host_stream_begin")
        assert a[2] == want
        assert hs.dtype == (torch.float32 if want == _lib.F32 else torch.float64)
        tref, sref = hs._ref["thetao"], hs._ref["so"]
        assert (a[6], a[7]) == (tref.data_ptr(), sref.data_ptr())  # T_ref, S_ref in their own places
        assert tref.dtype == sref.dtype == hs.dtype
        # the slabs that cross are the supplied values, not a rounding of them
        assert np.array_equal(tref.numpy().astype(np.float64), T_ref.astype(np.float64), equal_nan=True)
        assert np.array_equal(sref.numpy().astype(np.float64), S_ref.astype(np.float64), equal_nan=True)
        # blocks follow the stream's dtype
        blk = np.zeros((2, NZ, NY, NX), dtype=np.float32)
        hs.push(blk, blk)
        assert hs._blocks[-1][0].dtype == hs.dtype
    finally:
        hs.abort()


def test_host_stream_one_inexact_slab_is_enough(rec):
    T_ref, _ = _slabs(2, np.float64)
    _, S_ref = _slabs(2, np.float64, exact=True)
    hs = _stream(T_ref, S_ref, torch.float32)
    try:
        assert rec.args("ml_host_stream_begin")[2] == _lib.F64
    finally:
        hs.abort()


def test_host_stream_values_beyond_fp32_range_are_not_exact(rec):
    T_ref, S_ref = _slabs(3, np.float64, exact=True)
    T_ref[1, 1, 1] = 1.0e300  # becomes inf in fp32
    hs = _stream(T_ref, S_ref, torch.float32)
    try:
        assert rec.args("ml_host_stream_begin")[2] == _lib.F64
    finally:
        hs.abort()


def _fields(dtype, nt=2):
    g = np.random.default_rng(7)
    T = torch.from_numpy(2.0 + 25.0 * g.random((nt, NZ, NY, NX))).to(dtype)
    S = torch.from_numpy(33.0 + 3.0 * g.random((nt, NZ, NY, NX))).to(dtype)
    return T, S


@pytest.mark.parametrize("field_dtype,ref_dtype,want", [
    (torch.float32, np.float64, _lib.F64),
    (torch.float64, np.float32, _lib.F64),
    (torch.float32, np.float32, _lib.F32),
])
def test_local_variants_promote_to_the_reference_dtype(rec, field_dtype, ref_dtype, want):
    T, S = _fields(field_dtype)
    T_ref, S_ref = _slabs(4, ref_dtype)
    V = np.full((NZ, NY, NX), 1.0e9)
    p = np.arange(NZ, dtype=np.float64) * 1.0e5
    zi = np.arange(NZ + 1, dtype=np.float64) * 10.0
    core.steric_local_variants(T, S, V, zi, np.full((NY, NX), 1000.0), p, T_ref=T_ref, S_ref=S_ref,
                               rho_ref=np.full((NZ, NY, NX), 1030.0))
    assert rec.args("ml_steric_local_variants")[1] == want


@pytest.mark.parametrize("field_dtype,ref_dtype,want", [
    (torch.float32, np.float64, _lib.F64),
    (torch.float64, np.float32, _lib.F64),
    (torch.float32, np.float32, _lib.F32),
])
def test_global_variants_promote_to_the_reference_dtype(rec, field_dtype, ref_dtype, want):
    T, S = _fields(field_dtype)
    T_ref, S_ref = _slabs(5, ref_dtype)
    V = np.full((NZ, NY, NX), 1.0e9)
    p = np.arange(NZ, dtype=np.float64) * 1.0e5
    _, sums = core.steric_global_variants(T, S, V, p, T_ref=T_ref, S_ref=S_ref)
    a = rec.args("ml_steric_global_variants")
    assert a[1] == want
    assert sums is None and a[15] is None  # a supplied reference: no reference scalars are asked for


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_global_variants_still_detect_a_self_reference(rec, dtype):
    T, S = _fields(dtype, nt=1)
    V = np.full((NZ, NY, NX), 1.0e9)
    p = np.arange(NZ, dtype=np.float64) * 1.0e5
    _, sums = core.steric_global_variants(T, S, V, p)
    a = rec.args("ml_steric_global_variants")
    assert a[1] == (_lib.F32 if dtype == torch.float32 else _lib.F64)
    assert a[4] == a[2] and a[5] == a[3]  # T_ref, S_ref are the fields themselves
    assert sums is not None and a[15] == sums.data_ptr()
