"""The stratification kernels (``csrc/ml_strat.cu``) against ``oracle.stratification`` at their edges.

``test_gpu_strat.py`` checks the reference's known answers and two layouts.  This file covers what
that leaves open: every level-axis position, the extents around the 16-level ``cp.async`` ring and
the 512-level limit, more than 65535 outer slabs, NaN holes at the one-sided stencil ends, a
stretched grid, non-default constants, and the cells ``adjust_negative_n2`` fills with 1e-8.

``adjusted[0] = adjusted[0].fillna(1e-8)`` (derived.py:63) indexes the array's FIRST axis: the
surface level of ``(z, y, x)``, the first time step of ``(time, z, y, x)``, every time step of
member 0 of ``(member, time, z, y, x)`` and the row y = 0 of ``(y, x, z)``.  Each field below has
columns that are unstable at the top in slabs inside and outside that index, so the oracle's answer
depends on where the fill goes; every test asserts that it does before it compares.

Tolerance: 1e-10 of the largest |oracle| in the same (outer, level) row, so a deep level is held
to its own magnitude and not to the surface's.  NaN patterns match exactly, and so do the cells
set to 1e-8.  ``adjust_negative_n2`` on an existing field only copies values, so it matches
bit for bit.
"""

import numpy as np
import pytest
import torch

from oracle import eos as oeos
from oracle import steric as osteric
from oracle import stratification as ostrat

pytestmark = pytest.mark.gpu

FILL = 1.0e-8  # derived.py:63


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


# ----------------------------------------------------------------------------- fields


def _grid(nz, depth=6500.0):
    """OM4-like stretched levels (about 2 m thick at the surface, 250 m at depth for nz = 75)."""
    k = np.arange(nz, dtype=np.float64)
    dz = 2.0 + 248.0 * (k / max(nz - 1, 1)) ** 2.2
    z_i = np.concatenate([[0.0], np.cumsum(dz)])
    z_i *= depth / z_i[-1]
    return z_i, 0.5 * (z_i[1:] + z_i[:-1])


def _column_view(a, z_axis):
    nouter = int(np.prod(a.shape[:z_axis], dtype=np.int64))
    return a.reshape(nouter, a.shape[z_axis], -1)


def _fill_slabs(shape, z_axis):
    """Outer slabs of ``adjusted[0]`` for ``z_axis >= 1`` (the level axis leading fills the surface instead)."""
    return int(np.prod(shape[1:z_axis], dtype=np.int64))


def _make(shape, z_axis, z_l, seed=0):
    """fp64 T, S with noise at every level (so no row of gradients cancels to nothing) and planted columns.

    Returns ``(T, S, tops)``: ``tops`` maps "inside" / "outside" to the (slab, column) cells whose top
    three levels are statically unstable, in slabs inside and outside ``adjusted[0]``.
    """
    rng = np.random.default_rng(seed)
    zs = [1] * len(shape)
    zs[z_axis] = -1
    z = z_l.reshape(zs)
    T = 2.0 + 18.0 * np.exp(-z / 700.0) + rng.normal(0.0, 0.05, shape)
    S = 35.2 - 0.9 * np.exp(-z / 300.0) + rng.normal(0.0, 0.01, shape)
    Tv, Sv = _column_view(T, z_axis), _column_view(S, z_axis)
    nouter, nz, ncol = Tv.shape
    k = _fill_slabs(shape, z_axis) if z_axis > 0 else 0
    if k > 0:
        inside = sorted({0, k // 2, k - 1, min(1, k - 1)})
        outside = sorted({s for s in (k, k + 1, (k + nouter) // 2, nouter - 2, nouter - 1) if k <= s < nouter})
    else:  # the surface level of every slab is filled
        inside, outside = sorted({0, nouter // 2, nouter - 1}), []
    tops = {"inside": [(s, 0) for s in inside], "outside": [(s, 0) for s in outside]}
    m = min(3, nz - 1)
    for s, c in tops["inside"] + tops["outside"]:
        Tv[s, :m, c] = Tv[s, m, c] - 0.5 * np.arange(m, 0, -1)  # warmer with depth: N2 < 0 at the top
        Sv[s, :m + 1, c] = Sv[s, m, c]
    used = set(tops["inside"] + tops["outside"])
    spread = sorted({int(s) for s in np.linspace(0, nouter - 1, 24)} | set(outside))
    cols = sorted({int(c) for c in np.linspace(0, ncol - 1, 16)})
    free = [(s, c) for s in spread for c in cols if (s, c) not in used]
    assert len(free) >= 11, "field too small for the planted columns"

    # a column unstable from top to bottom outside the fill: the forward fill has nothing to carry
    neg = next(((s, c) for s, c in free if s in outside), free[0])
    free.remove(neg)
    Tv[neg[0], :, neg[1]] = 2.0 + 15.0 * z_l / z_l[-1]
    Sv[neg[0], :, neg[1]] = 35.0
    holes = [(v, lev) for v in (Tv, Sv) for lev in (0, 1, nz - 2, nz - 1)]
    for (arr, lev), (s, c) in zip(holes, free):
        arr[s, lev, c] = np.nan
    rest = free[len(holes):]
    if len(rest) >= 2:
        s, c = rest[0]
        Tv[s, :, c] = np.nan  # land
        Sv[s, :, c] = np.nan
        s, c = rest[1]
        Tv[s, 2:, c] = np.nan  # wet in the top two levels only
        Sv[s, 2:, c] = np.nan
    return T, S, tops


def _stored(T, S, dtype):
    """The tensors handed to the kernels and the fp64 upcast of exactly those values for the oracle."""
    if dtype == torch.float32:
        T, S = T.astype(np.float32), S.astype(np.float32)
    return (torch.from_numpy(T).cuda(), torch.from_numpy(S).cuda(), T.astype(np.float64), S.astype(np.float64))


# ----------------------------------------------------------------------------- comparisons


def _rows(a, z_axis):
    """One row per (outer, level) pair.  A level-last field has one cell per such pair, so its rows
    are gathered along the axes between the first and the level axis: every x of one (y, level)."""
    if z_axis == a.ndim - 1 and a.ndim > 1:
        a = np.moveaxis(a, -1, 1)
        return a.reshape(a.shape[0] * a.shape[1], -1)
    return a.reshape(int(np.prod(a.shape[:z_axis + 1], dtype=np.int64)), -1)


def _check(got, want, z_axis, rtol=1e-10, where=None, what="", floor=0.0):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, what
    gn, wn = np.isnan(got), np.isnan(want)
    assert np.array_equal(gn, wn), f"{what}: NaN pattern differs at {np.argwhere(gn != wn)[:5].tolist()}"
    gi, wi = np.isinf(got), np.isinf(want)
    assert np.array_equal(gi, wi) and np.array_equal(got[gi], want[wi]), f"{what}: infinities differ"
    fin = np.isfinite(want) if where is None else (np.isfinite(want) & where)
    g, w, f = _rows(got, z_axis), _rows(want, z_axis), _rows(fin, z_axis)
    scale = np.maximum(np.where(f, np.abs(w), 0.0).max(axis=1, keepdims=True), floor)
    err = np.where(f, np.abs(g - w), 0.0)
    bad = err > rtol * scale
    if bad.any():
        r, c = np.argwhere(bad)[0]
        raise AssertionError(f"{what}: {int(bad.sum())} cells off, first row {r} col {c}: got {g[r, c]!r} want {w[r, c]!r} "
                             f"(row scale {scale[r, 0]:.3e})")


def _check_adjusted(got, want, z_axis, what="adjusted N2"):
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(got == FILL, want == FILL), \
        f"{what}: filled cells differ at {np.argwhere((got == FILL) != (want == FILL))[:5].tolist()}"
    _check(got, want, z_axis, what=what)


def _adjust_without_fill(n2, z_axis):
    """The oracle's adjustment with ``adjusted[0]`` moved onto a dummy leading slab (z_axis >= 1)."""
    pad = np.concatenate([np.full_like(n2[:1], np.nan), n2], axis=0)
    return ostrat.adjust_negative_n2(pad, z_axis=z_axis)[1:]


def _assert_fill_matters(want_adj, n2, z_axis, tops):
    """The planted unstable tops take 1e-8 inside ``adjusted[0]`` and stay NaN outside it."""
    wv = _column_view(want_adj, z_axis)
    for s, c in tops["inside"]:
        assert wv[s, 0, c] == FILL, ("planted top not filled by the oracle", s, c)
    for s, c in tops["outside"]:
        assert np.isnan(wv[s, 0, c]), ("planted top outside the fill is not NaN", s, c)
    if z_axis > 0:
        nv = _column_view(_adjust_without_fill(n2, z_axis), z_axis)
        for s, c in tops["inside"]:
            assert np.isnan(nv[s, 0, c])  # without the fill the oracle would say NaN there


def _ratio(T, S, p_level, z_l, eos, z_axis):
    """The oracle's density ratio R = beta dS/dz / (alpha dT/dz), to leave out where R is close to one."""
    shape = [1] * T.ndim
    shape[z_axis] = -1
    p = np.asarray(p_level, np.float64).reshape(shape)
    if eos == "Wright":
        alpha, beta = oeos.wright_alpha(T, S, p), oeos.wright_beta(T, S, p)
    else:
        alpha, beta = oeos.linear_alpha(T, S, p), oeos.linear_beta(T, S, p)
    with np.errstate(divide="ignore", invalid="ignore"):
        return (beta * np.gradient(S, z_l, axis=z_axis, edge_order=2)) / (
            alpha * np.gradient(T, z_l, axis=z_axis, edge_order=2))


def _check_angle(got, T, S, p_level, z_l, eos, z_axis):
    """The angle's error is that of R times d(angle)/dR = (180 / pi) / (1 + R^2), so it is absolute: a small
    angle near R = -1 (where 1 + R cancels) carries the error of any other.  Its scale is therefore at least
    90 degrees, the range of the angle, and not the magnitude of a row that may hold a single cell."""
    want = ostrat.calc_stability_angle(T, S, p_level, z_l, eos=eos, z_axis=z_axis)
    with np.errstate(invalid="ignore"):
        ok = np.abs(1.0 - _ratio(T, S, p_level, z_l, eos, z_axis)) > 1e-6
    assert np.array_equal(np.isnan(got), np.isnan(want)), "Turner angle: NaN pattern differs"
    _check(np.where(ok, got, np.nan), np.where(ok, want, np.nan), z_axis, what="Turner angle", floor=90.0)
    assert ok[np.isfinite(want)].mean() > 0.99  # the comparison is not vacuous


def _oracle_wave_speed(n2, dz, z_axis):
    """``sum_z sqrt(adjusted N2) dz / pi`` (derived.py:821) from the oracle's adjustment, for any leading axes."""
    if n2.ndim == 4 and z_axis == 1:
        return ostrat.calc_wave_speed(n2, dz)[0]
    adj = ostrat.adjust_negative_n2(n2, z_axis=z_axis)
    with np.errstate(invalid="ignore"):
        return np.nansum(np.sqrt(adj) * dz, axis=z_axis) / np.pi


def _dz(z_i, z_l, hshape, seed):
    """Partial bottom cells: a sea floor between interfaces, some land."""
    rng = np.random.default_rng(seed)
    depth = rng.uniform(5.0, z_i[-1], hshape)
    depth.flat[3::7] = np.nan
    return osteric.calc_dz(z_l, z_i, depth)


# ----------------------------------------------------------------------------- one full check


def _run_all(ml, shape, z_axis, dtype, eos, seed=0, gravity=-9.8, patm=101325.0, wave=True, labeled_dims=None):
    from momlevel_b200 import core

    nz = shape[z_axis]
    z_i, z_l = _grid(nz)
    T, S, tops = _make(shape, z_axis, z_l, seed)
    Tg, Sg, T64, S64 = _stored(T, S, dtype)
    n2_want = ostrat.calc_n2(T64, S64, z_l, eos=eos, gravity=gravity, patm=patm, z_axis=z_axis)
    adj_want = ostrat.calc_n2(T64, S64, z_l, eos=eos, gravity=gravity, patm=patm, z_axis=z_axis, adjust_negative=True)
    _assert_fill_matters(adj_want, n2_want, z_axis, tops)

    n2 = core.calc_n2(Tg, Sg, z_l, eos=eos, gravity=gravity, patm=patm, z_axis=z_axis)
    _check(n2.cpu().numpy(), n2_want, z_axis, what="N2")
    adj = core.calc_n2(Tg, Sg, z_l, eos=eos, gravity=gravity, patm=patm, z_axis=z_axis, adjust_negative=True)
    _check_adjusted(adj.cpu().numpy(), adj_want, z_axis)
    # on an existing field the adjustment only moves values: bit for bit
    moved = core.adjust_negative_n2(torch.from_numpy(n2_want).cuda(), z_axis=z_axis).cpu().numpy()
    assert np.array_equal(moved, ostrat.adjust_negative_n2(n2_want, z_axis=z_axis), equal_nan=True)

    p_level = z_l * 1.02e4 + 3.0e4  # not the z_l * 1e4 of the reference's own test
    tu = core.stability_angle(Tg, Sg, p_level, z_l, eos=eos, z_axis=z_axis).cpu().numpy()
    _check_angle(tu, T64, S64, p_level, z_l, eos, z_axis)

    if wave and 0 < z_axis < len(shape) - 1:
        dz = _dz(z_i, z_l, shape[z_axis + 1:], seed + 1)
        c1 = core.wave_speed(torch.from_numpy(n2_want).cuda(), torch.from_numpy(dz).cuda(), z_axis=z_axis).cpu().numpy()
        want = _oracle_wave_speed(n2_want, dz, z_axis)
        assert c1.shape == want.shape
        assert np.array_equal(c1 == 0.0, want == 0.0)
        assert np.all(np.abs(c1 - want) <= 1e-12 * np.abs(want)), np.abs(c1 - want).max()
        assert (want > 0).any()

    if labeled_dims is not None:
        zc = labeled_dims[z_axis]
        ta = ml.DataArray(Tg, labeled_dims, coords={zc: z_l})
        sa = ml.DataArray(Sg, labeled_dims, coords={zc: z_l})
        lab = ml.derived.calc_n2(ta, sa, eos=eos, gravity=gravity, patm=patm, zcoord=zc, adjust_negative=True)
        assert lab.dims == labeled_dims
        assert np.array_equal(lab.values, adj.cpu().numpy(), equal_nan=True)
        lab2 = ml.derived.adjust_negative_n2(ml.DataArray(torch.from_numpy(n2_want).cuda(), labeled_dims), zcoord=zc)
        assert np.array_equal(lab2.values, moved, equal_nan=True)
    return adj


# ----------------------------------------------------------------------------- tests


LAYOUTS = {
    "z0_3d": ((20, 6, 43), 0, ("z_l", "yh", "xh")),
    "z1_4d": ((3, 20, 5, 43), 1, ("time", "z_l", "yh", "xh")),
    "z2_5d_ensemble": ((2, 3, 20, 4, 33), 2, ("member", "time", "z_l", "yh", "xh")),
    "level_last": ((5, 7, 20), 2, ("yh", "xh", "z_l")),
}


@pytest.mark.parametrize("eos", ["Wright", "linear"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_layouts(ml, layout, dtype, eos):
    """Every output at every level-axis position, through ``core`` and through ``derived`` (labeled)."""
    shape, z_axis, dims = LAYOUTS[layout]
    _run_all(ml, shape, z_axis, dtype, eos, seed=3, labeled_dims=dims)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("nz", [3, 4, 14, 15, 16, 17, 18, 31, 33, 75, 512])
def test_level_extents(ml, nz, dtype):
    """Around the ring: it prefetches 15 levels and reuses slots from level 16 on.  nz = 512 with fp64
    storage takes exactly 48 KB of dynamic shared memory (4 nz 8 B of coefficients and pressure, 2 rings of
    16 x 128 x 8 B)."""
    _run_all(ml, (2, nz, 3, 43), 1, dtype, "Wright", seed=nz)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("ncol", [1, 127, 128, 129, 4099])
def test_column_counts(ml, ncol, dtype):
    """A partial last block of 128 columns, exactly one block, one column."""
    _run_all(ml, (24, 18, 1, ncol), 1, dtype, "linear" if ncol % 2 else "Wright", seed=ncol)


def test_level_limits(ml):
    from momlevel_b200 import core

    for nz in (2, 513):
        T = torch.full((2, nz, 8), 10.0, device="cuda")
        z_l = np.arange(nz, dtype=np.float64) + 1.0
        with pytest.raises(ml._lib.MLError):
            core.calc_n2(T, T, z_l)
        with pytest.raises(ml._lib.MLError):
            core.calc_n2(T, T, z_l, adjust_negative=True)
        with pytest.raises(ml._lib.MLError):
            core.stability_angle(T, T, z_l * 1e4, z_l)


@pytest.mark.parametrize("gravity,patm", [(-9.80665, 0.0), (-9.81, 2.5e5)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_gravity_and_patm(ml, dtype, gravity, patm):
    _run_all(ml, (2, 75, 4, 37), 1, dtype, "Wright", seed=11, gravity=gravity, patm=patm, wave=False)
    _run_all(ml, (2, 2, 16, 3, 19), 2, dtype, "linear", seed=12, gravity=gravity, patm=patm, wave=False)


SLABS = {
    "65535_slabs": ((65535, 3, 1, 8), 1),
    "65536_slabs": ((65536, 3, 1, 8), 1),  # the last slab is alone in its launch and holds no fill
    "ensemble_65536_slabs": ((2, 32768, 3, 1, 8), 2),
    "ensemble_fill_across_65535": ((1, 70000, 3, 1, 4), 2),
    "level_last_300x250": ((300, 250, 20), 2),
}


@pytest.mark.parametrize("case", list(SLABS))
def test_many_slabs(ml, case):
    """Above 65535 outer slabs (the grid.y limit of one launch) and fills that span a launch boundary."""
    shape, z_axis = SLABS[case]
    _run_all(ml, shape, z_axis, torch.float32, "Wright", seed=5)


def test_repeatable(ml):
    """A second call gives the same bits, for a field in one launch and for one in two."""
    from momlevel_b200 import core

    for shape, z_axis in (((3, 33, 5, 43), 1), ((65536, 3, 1, 8), 1), ((40, 30, 17), 2)):
        nz = shape[z_axis]
        z_i, z_l = _grid(nz)
        T, S, _ = _make(shape, z_axis, z_l, 9)
        Tg, Sg, _, _ = _stored(T, S, torch.float32)
        for call in (lambda: core.calc_n2(Tg, Sg, z_l, z_axis=z_axis),
                     lambda: core.calc_n2(Tg, Sg, z_l, z_axis=z_axis, adjust_negative=True),
                     lambda: core.stability_angle(Tg, Sg, z_l * 1e4, z_l, z_axis=z_axis)):
            a, b = call().cpu().numpy(), call().cpu().numpy()
            assert np.array_equal(a.view(np.int64), b.view(np.int64))
        n2 = core.calc_n2(Tg, Sg, z_l, z_axis=z_axis)
        if z_axis < len(shape) - 1:
            dz = torch.from_numpy(_dz(z_i, z_l, shape[z_axis + 1:], 1)).cuda()
            a, b = (core.wave_speed(n2, dz, z_axis=z_axis).cpu().numpy() for _ in range(2))
            assert np.array_equal(a.view(np.int64), b.view(np.int64))
        a, b = (core.adjust_negative_n2(n2, z_axis=z_axis).cpu().numpy() for _ in range(2))
        assert np.array_equal(a.view(np.int64), b.view(np.int64))
