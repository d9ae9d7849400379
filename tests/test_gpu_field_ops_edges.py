"""Spiciness, dz, the reference state, ``delta_rho``, its annual means and the sums of ``calc_masso`` point by point
against the fp64 oracle, on every kernel each entry point can reach.

Each entry of ``csrc/ml_api.cu`` picks its kernel from the storage type, the alignment of its operands, ``ncol % 4``,
``force_direct`` and whether a per-column pressure (a 2-D ``patm``, :class:`core.Pressure`) is set:

* ``flament_spice``: ``k_stream_map<0, 0>`` (fp32, T and S on 16 bytes, ``out`` on 32, ``n % 4 == 0``);
  ``k_spice_vec`` for any other aligned call and under ``force_direct(1)``, followed by ``k_spice`` for the
  ``n % 4`` tail; ``k_spice`` alone when an operand is off 16 bytes.
* ``calc_dz``: ``k_calc_dz``, levels on grid.y and looped past 65535.
* ``reference_state``: ``k_stream_refstate`` (fp32, aligned, ``ncol % 4 == 0``); ``k_reference_state_vec`` (fp64, or
  ``force_direct(1)``, at most 65535 levels); ``k_reference_state`` otherwise; each followed by ``k_reduce_rows``.
* ``delta_rho``: ``k_stream_delta_rho<E, TV>`` (fp32, aligned); ``k_delta_rho<T, E, 4, false>`` (fp64, ``force_direct``,
  or a ``v_ref`` that alone is off 16 bytes); ``k_delta_rho<T, E, 1, false>`` (``ncol % 4 != 0``, an operand off 16
  bytes, a 2-D ``patm``).  ``delta_rho_annual`` takes ``k_delta_rho<T, E, 4 or 1, true>`` by the same rule.
* ``weighted_nansum`` (``derived.calc_masso`` / ``calc_volo``): ``k_weighted_nansum``, rows on grid.y in chunks of
  65535, then ``k_reduce_rows``.

``test_kernel_routes`` checks with the profiler which kernel each geometry reaches, template arguments included; the
parity tests run every case on each geometry.  Tolerances are the suite's: spiciness 1e-12 absolute; dz bit for bit
(the kernel and the oracle do the same subtractions, clamps and one IEEE division); density 1e-10 relative; the
volume and mass sums 1e-13 relative of ``math.fsum`` over the finite terms (positive sums, condition number 1);
``delta_rho`` and its annual means 1e-9 absolute.  NaN patterns must match exactly everywhere.
"""

import math
import re

import numpy as np
import pytest
import torch

from oracle import eos as oeos
from oracle import spice as ospice
from oracle import steric as osteric

pytestmark = pytest.mark.gpu

RHO_RTOL = 1e-10
SUM_RTOL = 1e-13


@pytest.fixture(scope="module")
def core():
    from momlevel_b200 import core

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return core


# ----------------------------------------------------------------------------------------------------- helpers


def _np_dtype(dtype):
    return np.float32 if dtype == torch.float32 else np.float64


def _stored(a, dtype):
    """The fp64 upcast of what the device holds for ``a`` stored as ``dtype``."""
    return np.asarray(a).astype(_np_dtype(dtype)).astype(np.float64)


def _device(a, dtype, offset=False):
    """``a`` on the device as ``dtype``; with ``offset`` a view one element into its buffer, so aligned to its element
    but not to 16 bytes."""
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dtype)
    if not offset:
        return t.cuda()
    base = torch.empty(t.numel() + 1, dtype=dtype, device="cuda")
    view = base[1:].view(t.shape)
    view.copy_(t.cuda())
    assert view.data_ptr() % 16 != 0
    return view


def _kernels(fn):
    """Names of the library's kernels ``fn`` launches, in launch order, with their template arguments (spaces
    dropped): ``"k_delta_rho<float,0,4,false>"``."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = []
    for e in prof.events():
        m = re.search(r"\b(k_\w+)(<[^()]*>)?\(", e.name)
        if m:
            out.append(m.group(1) + (m.group(2) or "").replace(" ", ""))
    return out


class _Forced:
    """``force_direct(1)`` for the calls inside."""

    def __init__(self, core, on=True):
        self.core, self.on = core, on

    def __enter__(self):
        self.prev = self.core.force_direct(1 if self.on else 0)

    def __exit__(self, *exc):
        self.core.force_direct(self.prev)
        return False


def _nan_close(got, want, atol, what):
    assert got.shape == want.shape, what
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN pattern differs"
    m = ~np.isnan(want)
    assert np.isfinite(want[m]).all() and np.isfinite(got[m]).all(), f"{what}: infinite values"
    if m.any():
        err = np.max(np.abs(got[m] - want[m]))
        assert err <= atol, f"{what}: absolute error {err:.3e}"


def _rel_close(got, want, rtol, what):
    assert got.shape == want.shape, what
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN pattern differs"
    m = ~np.isnan(want)
    if m.any():
        err = np.max(np.abs(got[m] - want[m]) / np.abs(want[m]))
        assert err <= rtol, f"{what}: relative error {err:.3e}"


def _same_bits(a, b, what):
    """Equal NaN patterns, and equal bits everywhere else."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    assert a.shape == b.shape, what
    na, nb = np.isnan(a), np.isnan(b)
    assert np.array_equal(na, nb), f"{what}: NaN pattern differs"
    diff = a[~na].view(np.int64) != b[~nb].view(np.int64)
    assert not diff.any(), f"{what}: {int(diff.sum())} values differ, e.g. {a[~na][diff][:3]} vs {b[~nb][diff][:3]}"


def _fsum_close(got, terms, what):
    """``got`` against ``math.fsum`` of the finite ``terms``."""
    want = math.fsum(terms[np.isfinite(terms)].tolist())
    if want == 0.0:
        assert got == 0.0, what
    else:
        assert abs(got - want) <= SUM_RTOL * abs(want), f"{what}: relative error {abs(got - want) / abs(want):.3e}"


# ------------------------------------------------------------------------------------------------- spiciness

SPICE_N = 5 * 2048 + 12  # n % 4 == 0: five whole stream tiles and a short sixth one

# geometry -> (storage, extra points past SPICE_N, T/S off 16 bytes, `out` 16 bytes into its buffer, force_direct)
SPICE_GEOMS = {
    "stream": (torch.float32, 0, False, False, False),
    "forced": (torch.float32, 0, False, False, True),
    "f64": (torch.float64, 0, False, False, False),
    "ragged": (torch.float32, 3, False, False, False),
    "offset": (torch.float32, 0, True, False, False),
    "offset_f64": (torch.float64, 0, True, False, False),
    "out16": (torch.float32, 0, False, True, False),
}


def _spice_fields(n, seed=3):
    rng = np.random.default_rng(seed)
    T = rng.uniform(-2.0, 32.0, n)
    S = rng.uniform(30.0, 40.0, n)
    T[7::97] = np.nan
    S[11::89] = np.nan
    T[3::101] = np.inf
    T[5::103] = -np.inf
    S[13::107] = np.inf
    S[17::109] = -np.inf
    T[19::113] = S[19::113] = np.inf
    T[23::127] = 1.0e70  # T**5 overflows (inf in fp32 storage)
    return T, S


def _spice(core, geom, seed=3):
    dtype, extra, offset, out16, forced = SPICE_GEOMS[geom]
    n = SPICE_N + extra
    T, S = _spice_fields(n, seed)
    Td, Sd = _device(T, dtype, offset), _device(S, dtype, offset)
    out = None
    if out16:
        out = torch.empty(n + 2, dtype=torch.float64, device="cuda")[2:]
        assert out.data_ptr() % 32 == 16
    with _Forced(core, forced):
        got = core.flament_spice(Td, Sd, out=out)
    return got, T, S, dtype


@pytest.mark.parametrize("geom", list(SPICE_GEOMS))
def test_spice_against_oracle(core, geom):
    """flament.py:43-95 with NaN and +-inf in T and S, and a T whose fifth power overflows; those points are NaN, as in
    the reference's power-table sum (an infinite power meets coefficients of both signs)."""
    got, T, S, dtype = _spice(core, geom)
    T64, S64 = _stored(T, dtype), _stored(S, dtype)
    with np.errstate(invalid="ignore", over="ignore"):
        want = ospice.flament_spice(T64, S64)
    assert np.isnan(want[~(np.isfinite(T64) & np.isfinite(S64)) | (np.abs(T64) > 1e60)]).all()
    _nan_close(got.cpu().numpy(), want, 1e-12, f"spice {geom}")


def test_spice_kernels_agree_bitwise(core):
    """k_stream_map, k_spice_vec and k_spice evaluate the same inlined flament_spice on the same values."""
    a = _spice(core, "stream")[0].cpu().numpy()
    b = _spice(core, "forced")[0].cpu().numpy()
    c = _spice(core, "offset")[0].cpu().numpy()
    d = _spice(core, "out16")[0].cpu().numpy()
    _same_bits(a, b, "stream vs vec")
    _same_bits(a, c, "stream vs scalar")
    _same_bits(a, d, "stream vs vec (out on 16 bytes)")
    _same_bits(_spice(core, "f64")[0].cpu().numpy(), _spice(core, "offset_f64")[0].cpu().numpy(), "fp64 vec vs scalar")


# ------------------------------------------------------------------------------------------------------- dz

# interfaces with zero-thickness levels (10-10, 60-60-60), which fraction=True turns into NaN
DZ_ZI = np.array([0.0, 2.5, 10.0, 10.0, 25.0, 60.0, 60.0, 60.0, 100.0, 200.0])
DZ_TOPS = [0.0, 5.0, 25.0, 300.0]               # surface, inside a level, on an interface, below every floor
DZ_BOTTOMS = [None, 3.0, 42.0, 60.0, 1.0e6]     # to the floor, above top 5, inside a level, on an interface, deep


def _dz_depths(z_i):
    """NaN (land), 0, every interface, every level's middle, below the last interface, +inf."""
    mid = 0.5 * (z_i[:-1] + z_i[1:])
    return np.concatenate([[np.nan, 0.0], z_i, mid, [z_i[-1] + 50.0, 1.0e4, np.inf]])


def _dz_case(core, z_i, depth, top, bottom, fraction):
    z_l = 0.5 * (z_i[:-1] + z_i[1:])
    got = core.calc_dz(torch.from_numpy(z_i).cuda(), torch.from_numpy(depth).cuda(), top=top, bottom=bottom,
                       fraction=fraction).cpu().numpy()
    with np.errstate(invalid="ignore"):
        want = osteric.calc_dz(z_l, z_i, depth.reshape(1, -1), top=top, bottom=bottom, fraction=fraction)
    _same_bits(got, want.reshape(got.shape), f"calc_dz top={top} bottom={bottom} fraction={fraction}")
    return got


@pytest.mark.parametrize("fraction", [False, True])
def test_calc_dz_edges(core, fraction):
    """derived.py:295-323 bit for bit: every top x bottom, depths on and between interfaces, NaN, 0 and +inf."""
    depth = _dz_depths(DZ_ZI)
    for top in DZ_TOPS:
        for bottom in DZ_BOTTOMS:
            got = _dz_case(core, DZ_ZI, depth, top, bottom, fraction)
            if fraction:
                assert np.isnan(got[2]).all() and np.isnan(got[5:7]).all()  # the zero-thickness levels


def _dz_grid(nz, seed):
    rng = np.random.default_rng(seed)
    steps = rng.uniform(0.5, 40.0, nz)
    steps[1::7] = 0.0  # repeated interfaces
    return np.concatenate([[0.0], np.cumsum(steps)])


@pytest.mark.parametrize("nz,ncol", [(1, 1), (1, 255), (1, 256), (1, 257), (1, 70000), (75, 1), (75, 255),
                                     (75, 256), (75, 257), (75, 70000), (65536, 257)])
def test_calc_dz_shapes(core, nz, ncol):
    """One column to 70000 columns, one level to 65536 (grid.y holds 65535 levels; the kernel loops past them)."""
    z_i = _dz_grid(nz, nz + ncol)
    rng = np.random.default_rng(ncol)
    pool = _dz_depths(z_i)
    depth = np.where(rng.random(ncol) < 0.5, rng.choice(pool, ncol), rng.uniform(0.0, 1.1 * z_i[-1], ncol))
    cases = [(0.0, None, False), (0.3 * z_i[-1], 0.7 * z_i[-1], True)]
    if nz > 1:
        cases.append((float(z_i[1]), float(z_i[nz // 2]), False))
    if nz > 1000:
        cases = cases[1:2]  # 134 MB of output per call: one call
    for top, bottom, fraction in cases:
        _dz_case(core, z_i, depth, top, bottom, fraction)


def test_calc_dz_derived_level_last(core):
    """derived.calc_dz returns dims (y, x, z); the values are the oracle's, bit for bit."""
    from momlevel_b200 import derived
    from momlevel_b200.labeled import DataArray

    depth = np.resize(_dz_depths(DZ_ZI), 3 * 19).reshape(3, 19)
    z_l = 0.5 * (DZ_ZI[:-1] + DZ_ZI[1:])
    for top, bottom, fraction in ((0.0, None, False), (5.0, 60.0, True), (25.0, 42.0, False)):
        got = derived.calc_dz(DataArray(z_l, ("z_l",)), DataArray(DZ_ZI, ("z_i",)), DataArray(depth, ("yh", "xh")),
                              top=top, bottom=bottom, fraction=fraction)
        assert got.dims == ("yh", "xh", "z_l")
        with np.errstate(invalid="ignore"):
            want = osteric.calc_dz(z_l, DZ_ZI, depth, top=top, bottom=bottom, fraction=fraction)
        _same_bits(np.asarray(got.values), want.transpose(1, 2, 0), f"derived top={top} bottom={bottom}")


# ------------------------------------------------------------------------------------------- reference state

# geometry -> (storage, nx (ny = 3), operands off 16 bytes, 2-D patm, force_direct)
REF_GEOMS = {
    "stream": (torch.float32, 516, False, False, False),
    "forced": (torch.float32, 516, False, False, True),
    "f64": (torch.float64, 516, False, False, False),
    "ragged": (torch.float32, 515, False, False, False),
    "offset": (torch.float32, 516, True, False, False),
    "patm2d": (torch.float32, 516, False, True, False),
}


def _ref_fields(nz, ny, nx, seed):
    rng = np.random.default_rng(seed)
    shape = (nz, ny, nx)
    T = rng.uniform(-2.0, 30.0, shape)
    S = rng.uniform(30.0, 38.0, shape)
    V = rng.uniform(1.0e6, 1.0e9, shape)
    Tf, Sf, Vf = (x.reshape(nz, -1) for x in (T, S, V))  # [level][column] views
    if nz > 2:
        Vf[nz // 2] = np.nan            # a whole dry level
    Tf[0, 1] = np.nan                   # a hole where the volume is present: volo keeps it, masso skips it
    Sf[-1, 2] = np.nan
    Vf[0, 5] = np.nan                   # no volume where T and S are present
    Vf[0, 6:9] = 0.0                    # zero volumes
    Vf[-1, 3] = 0.0
    return T, S, V


def _ref_call(core, geom, eos, nz, seed=5):
    dtype, nx, offset, patm2d, forced = REF_GEOMS[geom]
    ny = 3
    T, S, V = _ref_fields(nz, ny, nx, seed)
    p_level = np.linspace(0.0, 6.0e7, nz) + 101325.0
    patm = np.random.default_rng(seed + 1).uniform(9.0e4, 1.1e5, (ny, nx)) if patm2d else None
    args = [_device(x, dtype, offset) for x in (T, S, V)]
    p = core.Pressure(p_level, patm) if patm2d else p_level
    with _Forced(core, forced):
        rho, sums = core.reference_state(*args, p, eos=eos)
    T64, S64, V64 = (_stored(x, dtype) for x in (T, S, V))
    pres = p_level[:, None, None] + (patm[None] if patm2d else 0.0)
    with np.errstate(invalid="ignore"):
        want = oeos.density(eos, T64, S64, pres)
    return rho.cpu().numpy(), sums.cpu().numpy(), want, V64


@pytest.mark.parametrize("nz", [1, 75])
@pytest.mark.parametrize("eos", ["Wright", "linear"])
@pytest.mark.parametrize("geom", list(REF_GEOMS))
def test_reference_state_against_oracle(core, geom, eos, nz):
    """reference.py:71-80: rho_ref to 1e-10 relative; volo = nansum(V0), masso = nansum(rho_ref * V0) to 1e-13 of
    math.fsum over the finite terms."""
    rho, sums, want, V64 = _ref_call(core, geom, eos, nz)
    _rel_close(rho, want, RHO_RTOL, f"rho_ref {geom} {eos}")
    _fsum_close(float(sums[0]), V64, f"volo {geom}")
    with np.errstate(invalid="ignore"):
        _fsum_close(float(sums[1]), rho * V64, f"masso {geom}")


@pytest.mark.parametrize("eos", ["Wright", "linear"])
def test_reference_state_kernels_agree(core, eos):
    """rho_ref bit for bit on k_stream_refstate, k_reference_state_vec and k_reference_state; the sums (other
    summation orders) to 1e-13."""
    base_rho, base_sums, _, _ = _ref_call(core, "stream", eos, 75)
    for geom in ("forced", "offset"):
        rho, sums, _, _ = _ref_call(core, geom, eos, 75)
        _same_bits(rho, base_rho, f"rho_ref stream vs {geom}")
        assert np.allclose(sums, base_sums, rtol=SUM_RTOL, atol=0), (geom, sums, base_sums)


def test_reference_state_65536_levels(core):
    """More levels than the vectorised kernel takes (grid.y): under force_direct the call falls to k_reference_state,
    whose threads walk all 65536 levels of their column.  One call: the workspace is 2 * nz * 512 doubles."""
    nz, ny, nx = 65536, 3, 4
    T, S, V = _ref_fields(nz, ny, nx, 9)
    p_level = np.linspace(0.0, 6.0e7, nz) + 101325.0
    Td, Sd, Vd = (_device(x, torch.float32) for x in (T, S, V))
    res = {}

    def run():
        with _Forced(core):
            res["out"] = core.reference_state(Td, Sd, Vd, p_level)

    assert _kernels(run) == ["k_reference_state<float,0>", "k_reduce_rows"]
    rho, sums = (x.cpu().numpy() for x in res["out"])
    T64, S64, V64 = (_stored(x, torch.float32) for x in (T, S, V))
    with np.errstate(invalid="ignore"):
        want = oeos.density("Wright", T64, S64, p_level[:, None, None])
        _rel_close(rho, want, RHO_RTOL, "rho_ref nz=65536")
        _fsum_close(float(sums[0]), V64, "volo nz=65536")
        _fsum_close(float(sums[1]), rho * V64, "masso nz=65536")


# ------------------------------------------------------------------------------------------------- delta_rho

# geometry -> (nx (ny = 3: ncol 1548 or 1545), T/S/rho_ref off 16 bytes, v_ref alone off 16 bytes, 2-D patm,
# force_direct)
DR_GEOMS = {
    "aligned": (516, False, False, False, False),   # stream for fp32, k_delta_rho VEC 4 for fp64
    "forced": (516, False, False, False, True),
    "ragged": (515, False, False, False, False),
    "offset": (516, True, False, False, False),
    "patm2d": (516, False, False, True, False),
    "vref_off": (516, False, True, False, False),
}


def _dr_fields(shape, seed):
    nt, nz, ny, nx = shape
    rng = np.random.default_rng(seed)
    T = rng.uniform(-2.0, 30.0, shape)
    S = rng.uniform(30.0, 38.0, shape)
    V = rng.uniform(1.0e6, 1.0e9, shape[1:])
    V[:, 0, :2] = np.nan
    V[nz // 2, 1] = np.nan
    T[nt - 1, 0, 0, 3] = np.nan
    S[0, nz - 1, ny - 1, 4] = np.nan
    # rho_ref: a reference density the oracle and the kernel share (here near step 0), NaN at one point under a
    # present volume
    with np.errstate(invalid="ignore"):
        rho_ref = oeos.wright_density(T[0], S[0], (np.arange(nz) * 80.0e4 + 101325.0)[:, None, None])
    rho_ref = np.where(np.isnan(rho_ref), 1027.0, rho_ref) + rng.normal(0.0, 0.05, rho_ref.shape)
    rho_ref[1 % nz, 2, 7] = np.nan
    return T, S, V, rho_ref


def _dr_inputs(core, geom, dtype, vdtype, shape, bcast, seed):
    nx, offset, vref_off, patm2d, forced = DR_GEOMS[geom]
    nt, nz, ny, _ = shape
    shape = (nt, nz, ny, nx)
    T, S, V, rho_ref = _dr_fields(shape, seed)
    if bcast == "t_bcast":
        T = T[0]
    elif bcast == "s_bcast":
        S = S[0]
    p_level = np.arange(nz) * 80.0e4 + 101325.0
    patm = np.random.default_rng(seed + 1).uniform(-2.0e4, 2.0e4, (ny, nx)) if patm2d else None
    dev = dict(
        T=_device(T, dtype, offset), S=_device(S, dtype, offset), rho_ref=_device(rho_ref, torch.float64, offset),
        v_ref=_device(V, vdtype, offset or vref_off),
        p=core.Pressure(p_level, patm) if patm2d else p_level,
        kw=dict(t_bcast=bcast == "t_bcast", s_bcast=bcast == "s_bcast"), forced=forced)
    T64, S64 = _stored(T, dtype), _stored(S, dtype)
    if bcast == "t_bcast":
        T64 = T64[None]
    elif bcast == "s_bcast":
        S64 = S64[None]
    pres = p_level[:, None, None] + (patm[None] if patm2d else 0.0)
    with np.errstate(invalid="ignore"):
        rho = np.broadcast_to(oeos.wright_density(T64, S64, pres[None]), shape)
    V64 = _stored(V, vdtype)
    want = np.where(~np.isnan(V64)[None], rho - rho_ref[None], np.nan)
    return dev, want, V64, rho, rho_ref


def _dr_run(core, dev, weights=None):
    with _Forced(core, dev["forced"]):
        if weights is None:
            return core.delta_rho(dev["T"], dev["S"], dev["rho_ref"], dev["v_ref"], dev["p"], **dev["kw"])
        return core.delta_rho_annual(dev["T"], dev["S"], dev["rho_ref"], dev["v_ref"], dev["p"], weights, **dev["kw"])


DTYPES = [torch.float32, torch.float64]


@pytest.mark.parametrize("vdtype", DTYPES, ids=["v32", "v64"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("geom", list(DR_GEOMS))
def test_delta_rho_against_oracle(core, geom, dtype, vdtype):
    """steric.py:151-153 with the rho_ref the oracle uses: NaN under a missing volume, under a NaN rho_ref and at NaN
    T or S; no broadcast, t_bcast and s_bcast; fields and v_ref of either storage."""
    for i, bcast in enumerate(("none", "t_bcast", "s_bcast")):
        dev, want, _, _, _ = _dr_inputs(core, geom, dtype, vdtype, (3, 5, 3, 0), bcast, seed=20 + i)
        got = _dr_run(core, dev).cpu().numpy()
        _nan_close(got, want, 1e-9, f"delta_rho {geom} {bcast}")


@pytest.mark.parametrize("vdtype", DTYPES, ids=["v32", "v64"])
def test_delta_rho_stream_more_pairs_than_ctas(core, vdtype):
    """k_stream_delta_rho with 75 levels of 8340 columns: five tiles a level, the last one 148 columns short of whole,
    375 (level, segment) pairs for at most 2 CTAs per SM, so CTAs own several pairs."""
    nt, nz, ny, nx = 2, 75, 4, 2085
    T, S, V, rho_ref = _dr_fields((nt, nz, ny, nx), 31)
    p_level = np.arange(nz) * 80.0e4 + 101325.0
    args = (_device(T, torch.float32), _device(S, torch.float32), _device(rho_ref, torch.float64),
            _device(V, vdtype), torch.from_numpy(p_level).cuda())
    res = {}
    ks = _kernels(lambda: res.update(out=core.delta_rho(*args)))
    assert ks == [f"k_stream_delta_rho<0,{'float' if vdtype == torch.float32 else 'double'}>"], ks
    T64, S64 = _stored(T, torch.float32), _stored(S, torch.float32)
    with np.errstate(invalid="ignore"):
        rho = oeos.wright_density(T64, S64, p_level[None, :, None, None])
    want = np.where(~np.isnan(_stored(V, vdtype))[None], rho - rho_ref[None], np.nan)
    _nan_close(res["out"].cpu().numpy(), want, 1e-9, "stream delta_rho, pairs > CTAs")


# ---------------------------------------------------------------------------------------- delta_rho_annual

DAYS_NOLEAP = np.array([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], np.float64)


def _days_in_month(calendar, nt):
    years = nt // 12
    if calendar == "360_day":
        w = np.full(nt, 30.0)
    else:
        w = np.tile(DAYS_NOLEAP, years)
        if calendar == "julian":
            w[1::12][np.arange(years) % 4 == 0] = 29.0  # the first year of the series is a leap year
    w[5] = 0.0  # a month of weight 0, next to the missing months of one cell (below)
    return w


def _annual_oracle(want_monthly, w):
    """Per cell and year, sum(w * d) / sum(w) over the months whose anomaly is present; 0 / 0 = NaN where none is."""
    nt = want_monthly.shape[0]
    d = want_monthly.reshape((nt // 12, 12) + want_monthly.shape[1:])
    ww = w.reshape((nt // 12, 12) + (1,) * (want_monthly.ndim - 1))
    present = ~np.isnan(d)
    num = np.where(present, ww * np.where(present, d, 0.0), 0.0).sum(axis=1)
    den = np.where(present, ww, 0.0).sum(axis=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        return num / den


ANNUAL_GEOMS = ["aligned", "forced", "ragged", "offset", "patm2d"]


@pytest.mark.parametrize("nt", [12, 24, 120])
@pytest.mark.parametrize("calendar", ["noleap", "julian", "360_day"])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_delta_rho_annual_against_oracle(core, nt, calendar, dtype):
    """util.py:84-87 applied to steric.py:151-158, with a numpy oracle built from oracle.eos densities: a missing
    month in one cell, a whole missing year in another (NaN), a month of weight 0 among missing months (0 / 0 = NaN
    in a third cell, a normal mean in a fourth); VEC 4 and VEC 1."""
    w = _days_in_month(calendar, nt)
    for geom in ANNUAL_GEOMS:
        nx = DR_GEOMS[geom][0]
        T, S, V, rho_ref = _dr_fields((nt, 3, 3, nx), 40 + nt)
        # cell (z=2, y=1, x=9): one missing month; x=10: the whole last year; x=11: months 4 and 6 missing around
        # the weight-0 month 5, the rest of year 0 missing too (only month 5 is present: 0 / 0); x=12: months 4, 6
        # missing, the others present
        T[3, 2, 1, 9] = np.nan
        S[nt - 12:, 2, 1, 10] = np.nan
        T[[m for m in range(12) if m != 5], 2, 1, 11] = np.nan
        S[[4, 6], 2, 1, 12] = np.nan
        dev, want, _, _, _ = _dr_arrays(core, geom, dtype, T, S, V, rho_ref, seed=nt)
        got = _dr_run(core, dev, torch.from_numpy(w).cuda()).cpu().numpy()
        oracle = _annual_oracle(want, w)
        assert np.isnan(oracle[-1, 2, 1, 10]) and np.isnan(oracle[0, 2, 1, 11]) and np.isfinite(oracle[0, 2, 1, 12])
        assert np.isfinite(oracle[0, 2, 1, 9])
        _nan_close(got, oracle, 1e-9, f"annual {geom} nt={nt} {calendar}")


def _dr_arrays(core, geom, dtype, T, S, V, rho_ref, seed):
    """As _dr_inputs, for fields built by the caller (no broadcast, v_ref stored as the fields)."""
    nx, offset, vref_off, patm2d, forced = DR_GEOMS[geom]
    nt, nz, ny, _ = T.shape
    p_level = np.arange(nz) * 80.0e4 + 101325.0
    patm = np.random.default_rng(seed + 1).uniform(-2.0e4, 2.0e4, (ny, nx)) if patm2d else None
    dev = dict(T=_device(T, dtype, offset), S=_device(S, dtype, offset), rho_ref=_device(rho_ref, torch.float64, offset),
               v_ref=_device(V, dtype, offset or vref_off), p=core.Pressure(p_level, patm) if patm2d else p_level,
               kw={}, forced=forced)
    T64, S64, V64 = (_stored(x, dtype) for x in (T, S, V))
    pres = p_level[:, None, None] + (patm[None] if patm2d else 0.0)
    with np.errstate(invalid="ignore"):
        rho = oeos.wright_density(T64, S64, pres[None])
    want = np.where(~np.isnan(V64)[None], rho - rho_ref[None], np.nan)
    return dev, want, V64, rho, rho_ref


def test_delta_rho_annual_rejects_partial_years(core):
    """nt % 12 != 0: ML_ERR_SHAPE from the library before any launch (core asserts the same before calling it)."""
    from momlevel_b200 import _lib

    L = _lib.lib()
    nt, nz, ncol = 13, 2, 8
    T = torch.zeros((nt, nz, ncol), dtype=torch.float32, device="cuda")
    V = torch.ones((nz, ncol), dtype=torch.float32, device="cuda")
    rho = torch.zeros((nz, ncol), dtype=torch.float64, device="cuda")
    p = torch.zeros(nz, dtype=torch.float64, device="cuda")
    w = torch.ones(nt, dtype=torch.float64, device="cuda")
    out = torch.empty((2, nz, ncol), dtype=torch.float64, device="cuda")
    before = L.ml_launch_count()
    for n in (13, 11, 1):
        rc = L.ml_delta_rho_annual(0, _lib.F32, T.data_ptr(), T.data_ptr(), 0, 0, rho.data_ptr(), V.data_ptr(), _lib.F32,
                                   p.data_ptr(), w.data_ptr(), n, nz, ncol, out.data_ptr(), None)
        assert rc == -2 and b"whole years" in L.ml_last_error(), rc
    assert L.ml_launch_count() == before
    with pytest.raises(AssertionError):
        core.delta_rho_annual(T, T, rho, V, p.cpu().numpy(), w)


# -------------------------------------------------------------------------------- weighted sums (calc_masso)


def _wns_fields(nrows, n, seed, a_dtype=np.float64):
    rng = np.random.default_rng(seed)
    a = rng.uniform(990.0, 1060.0, (nrows, n)).astype(a_dtype)
    a[::7, 1] = np.nan
    a[nrows // 2] = np.nan  # a row with nothing to sum: 0
    w = rng.uniform(1.0e6, 1.0e9, n).astype(np.float32)
    w[n - 1] = np.nan
    return a, w


def _wns_check(got, a, w):
    terms = a.astype(np.float64) * w.astype(np.float64)[None]
    for r in range(terms.shape[0]):
        _fsum_close(float(got[r]), terms[r], f"row {r}")


@pytest.mark.parametrize("a_dtype", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("nrows", [65535, 65536, 70001])
def test_weighted_nansum_rows_past_one_grid(core, nrows, a_dtype):
    """Each row against math.fsum (1e-13), and each row's bits equal the same row summed in a call with fewer rows:
    the rows are launched in chunks of 65535 and a row's partials do not depend on its chunk."""
    n = 5
    a, w = _wns_fields(nrows, n, nrows, a_dtype)
    ad, wd = torch.from_numpy(a).cuda(), torch.from_numpy(w).cuda()
    got = core.weighted_nansum(ad, wd, nrows=nrows).cpu().numpy()
    _wns_check(got, a, w)
    for lo, hi in ((0, 65535), (65530, min(nrows, 65540)), (nrows - 1, nrows), (nrows // 2, nrows // 2 + 1)):
        part = core.weighted_nansum(ad[lo:hi], wd, nrows=hi - lo).cpu().numpy()
        _same_bits(part, got[lo:hi], f"rows [{lo}, {hi}) of {nrows}")


def test_calc_masso_derived_long_series(core):
    """derived.calc_masso(rho, volcello) on a 70001-step density (3-hourly output over 24 years)."""
    from momlevel_b200 import derived
    from momlevel_b200.labeled import DataArray

    nt, ny, nx = 70001, 2, 3
    a, w = _wns_fields(nt, ny * nx, 17)
    masso = derived.calc_masso(DataArray(a.reshape(nt, ny, nx), ("time", "yh", "xh")),
                               DataArray(w.reshape(ny, nx), ("yh", "xh")))
    assert masso.dims == ("time",)
    _wns_check(np.asarray(masso.values), a, w)


# ------------------------------------------------------------------------------------------------- route map


def test_kernel_routes(core):
    """Which kernel each geometry of the parity tests reaches, template arguments included."""
    def spice(geom):
        return _kernels(lambda: _spice(core, geom))

    assert spice("stream") == ["k_stream_map<0,0>"]
    assert spice("forced") == ["k_spice_vec<float>"]
    assert spice("f64") == ["k_spice_vec<double>"]
    assert spice("ragged") == ["k_spice_vec<float>", "k_spice<float>"]
    assert spice("offset") == ["k_spice<float>"]
    assert spice("offset_f64") == ["k_spice<double>"]
    assert spice("out16") == ["k_spice_vec<float>"]

    z_i = _dz_grid(75, 1)
    depth = torch.from_numpy(np.linspace(0.0, z_i[-1], 257)).cuda()
    zi = torch.from_numpy(z_i).cuda()
    assert _kernels(lambda: core.calc_dz(zi, depth, top=3.0, bottom=500.0, fraction=True)) == ["k_calc_dz"]

    def ref(geom, eos="Wright"):
        return _kernels(lambda: _ref_call(core, geom, eos, 7))

    assert ref("stream") == ["k_stream_refstate<0>", "k_reduce_rows"]
    assert ref("stream", "linear") == ["k_stream_refstate<1>", "k_reduce_rows"]
    assert ref("forced") == ["k_reference_state_vec<float,0>", "k_reduce_rows"]
    assert ref("f64") == ["k_reference_state_vec<double,0>", "k_reduce_rows"]
    assert ref("ragged") == ["k_reference_state<float,0>", "k_reduce_rows"]
    assert ref("offset") == ["k_reference_state<float,0>", "k_reduce_rows"]
    assert ref("patm2d") == ["k_reference_state<float,0>", "k_reduce_rows"]

    def dr(geom, dtype=torch.float32, vdtype=torch.float32, bcast="none", annual=False):
        dev = _dr_inputs(core, geom, dtype, vdtype, (12, 3, 3, 0), bcast, seed=1)[0]
        w = torch.ones(12, dtype=torch.float64, device="cuda") if annual else None
        return _kernels(lambda: _dr_run(core, dev, w))

    assert dr("aligned") == ["k_stream_delta_rho<0,float>"]
    assert dr("aligned", vdtype=torch.float64, bcast="t_bcast") == ["k_stream_delta_rho<0,double>"]
    assert dr("forced") == ["k_delta_rho<float,0,4,false>"]
    assert dr("aligned", torch.float64) == ["k_delta_rho<double,0,4,false>"]
    assert dr("aligned", torch.float64, torch.float32, "s_bcast") == ["k_delta_rho<double,0,4,false>"]
    assert dr("vref_off") == ["k_delta_rho<float,0,4,false>"]
    assert dr("vref_off", vdtype=torch.float64) == ["k_delta_rho<float,0,4,false>"]
    assert dr("ragged") == ["k_delta_rho<float,0,1,false>"]
    assert dr("offset", torch.float64) == ["k_delta_rho<double,0,1,false>"]
    assert dr("patm2d") == ["k_delta_rho<float,0,1,false>"]
    assert dr("aligned", annual=True) == ["k_delta_rho<float,0,4,true>"]
    assert dr("aligned", torch.float64, annual=True) == ["k_delta_rho<double,0,4,true>"]
    assert dr("ragged", annual=True) == ["k_delta_rho<float,0,1,true>"]
    assert dr("offset", annual=True) == ["k_delta_rho<float,0,1,true>"]
    assert dr("patm2d", annual=True) == ["k_delta_rho<float,0,1,true>"]

    a = torch.rand((65535, 5), dtype=torch.float64, device="cuda")
    w = torch.rand(5, dtype=torch.float32, device="cuda")
    assert _kernels(lambda: core.weighted_nansum(a, w, nrows=65535)) == ["k_weighted_nansum<double,float>",
                                                                          "k_reduce_rows"]
    b = torch.rand((3 * 65535 + 1, 5), dtype=torch.float32, device="cuda")
    assert _kernels(lambda: core.weighted_nansum(b, None, nrows=b.shape[0])) == \
        ["k_weighted_nansum<float,float>"] * 4 + ["k_reduce_rows"]
