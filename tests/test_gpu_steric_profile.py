"""steric_profile() and ml_steric_local_profile: the area-weighted steric, thermosteric and halosteric height change
by model level against the numpy reference (tests/profile_oracle.py), its sum over the levels against the weighted
mean of steric()'s local height, and the bit-identities the kernels promise (one pass against one launch per
variant, ring against plain loads, run against run).

Tolerance: the GPU evaluates the density with a lean reciprocal and FMA contraction, numpy with IEEE division, so
rho and rho_ref each differ by a few ulp of ~1030 kg m-3 (~1e-12 kg m-3).  Against a density change of ~0.03 kg m-3
that is ~1e-11 of a term, more than 1e-12, so a (step, level) value may differ by 1e-12 of the sum of its terms'
magnitudes plus that density floor times the sum of its weights m * w * dz."""

import importlib.util
import pathlib
import sys

import numpy as np
import pytest
import torch

from momlevel_b200 import synth
import profile_oracle  # tests/profile_oracle.py
from oracle import steric as osteric

pytestmark = pytest.mark.gpu

VARIANTS = ("steric", "thermosteric", "halosteric")
RHO_FLOOR = 2e-15 * 1100.0  # kg m-3: a few ulp of the density, the difference of two fp64 evaluations of it
NZ = 10


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


def _case(nt, ny, nx, dtype=torch.float32, seed=7, hole=False, vmask=False, weights="area"):
    """Fields, grid and column weights; ``hole``: NaN T and S at wet cells; ``vmask``: a reference volume that
    disagrees with the bathymetry; ``weights``: "area", "nan_zero" (NaN and 0 weights) or "basin"."""
    grid = synth.make_grid(NZ, ny, nx, seed=seed, device="cpu")
    T, S, V = synth.make_fields(grid, nt, seed=seed, dtype=dtype)  # V: the cell volume [nz, ny, nx]
    wet = torch.nonzero(~torch.isnan(V))
    if hole:
        for k, i in enumerate((len(wet) // 2, len(wet) // 5, len(wet) // 9)):
            z, y, x = (int(j) for j in wet[i])
            (T if k % 2 == 0 else S)[(k * 3) % nt, z, y, x] = float("nan")
    if vmask:
        for i in (len(wet) // 3, len(wet) // 7, 0):  # no reference volume at wet cells, the surface one included
            z, y, x = (int(j) for j in wet[i])
            V[z, y, x] = float("nan")
        dry = torch.nonzero(torch.isnan(V[0]))
        if len(dry):  # a volume under a column the bathymetry calls land
            y, x = (int(j) for j in dry[len(dry) // 2])
            V[0, y, x] = 1.0e9
            T[:, 0, y, x], S[:, 0, y, x] = 12.0, 35.0
    area = grid["areacello"].clone().to(torch.float64)
    if weights == "nan_zero":
        area.view(-1)[::7] = float("nan")
        area.view(-1)[3::11] = 0.0
    elif weights == "basin":
        area = area * (torch.arange(nx)[None, :] < nx // 2)
    return grid, T, S, V, area


def _np(x):
    return x.detach().cpu().numpy().astype(np.float64) if isinstance(x, torch.Tensor) else np.asarray(x, np.float64)


def _oracle_ref(grid, T, S, V, t0=0, patm=101325.0, eos="Wright"):
    V4 = np.broadcast_to(_np(V), tuple(T.shape))  # the volume of every step
    return osteric.reference_state(_np(T), _np(S), V4, _np(grid["areacello"]), _np(grid["z_l"]), patm=patm, eos=eos,
                                   time_index=t0)


def _gpu(ml, grid, T, S, V, w, t0=0, eos="Wright", patm=None, variants=VARIANTS):
    """core.steric_local_profile on device tensors, the reference state being step ``t0`` (core.reference_state)."""
    dev = torch.device("cuda")
    T, S, V = T.to(dev), S.to(dev), V.to(dev)
    p = grid["z_l"].to(dev, torch.float64) * 1.0e4
    if patm is None:
        p = p + 101325.0
    else:
        p = ml.core.Pressure(p, torch.as_tensor(patm, dtype=torch.float64, device=dev))
    rho, _ = ml.core.reference_state(T[t0], S[t0], V, p, eos=eos)
    return ml.core.steric_local_profile(T, S, T[t0], S[t0], rho, V, grid["z_i"].to(dev), grid["deptho"].to(dev), p,
                                        w.to(dev), eos=eos, variants=variants)


def _check(got, grid, T, S, V, w, ref, variant, eos="Wright", patm=101325.0):
    want, scale = profile_oracle.steric_profile(_np(T), _np(S), _np(grid["z_l"]), _np(grid["z_i"]), _np(grid["deptho"]),
                                                ref, weights=_np(w), eos=eos, variant=variant, patm=patm)
    m = ~np.isnan(ref["volcello"][0])
    dz = osteric.calc_dz(_np(grid["z_l"]), _np(grid["z_i"]), _np(grid["deptho"]))
    wsum = np.nansum(np.abs(m * np.nan_to_num(_np(w), nan=0.0))[None] * dz, axis=(1, 2)) / np.nansum(_np(w))
    tol = 1e-12 * scale + RHO_FLOOR / 1035.0 * wsum[None]
    g = got.cpu().numpy()
    assert g.shape == want.shape and np.isfinite(g).all()
    err = np.abs(g - want)
    assert (err <= tol).all(), (variant, float(err.max()), float((err / np.maximum(tol, 1e-300)).max()))


# ------------------------------------------------------------------------------------------ shapes and options


SHAPES = [  # (nt, ny, nx): columns aligned and two whole tiles, ragged, less than a tile, aligned past a tile
    (1, 32, 128),
    (5, 13, 37),
    (12, 12, 20),
    (13, 20, 132),
]


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_oracle_parity(ml, shape, dtype, eos):
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    got = _gpu(ml, grid, T, S, V, w, eos=eos)
    ref = _oracle_ref(grid, T, S, V, eos=eos)
    for v in VARIANTS:
        _check(got[v], grid, T, S, V, w, ref, v, eos=eos)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("opts", [
    dict(hole=True),
    dict(vmask=True),
    dict(weights="nan_zero"),
    dict(weights="basin"),
    dict(hole=True, vmask=True, weights="nan_zero", t0=3),
], ids=["holes", "vmask", "nan_zero_weights", "basin", "all_ref3"])
def test_oracle_parity_edges(ml, opts, dtype):
    t0 = opts.pop("t0", 0)
    grid, T, S, V, w = _case(7, 20, 132, dtype=dtype, **opts)
    got = _gpu(ml, grid, T, S, V, w, t0=t0)
    ref = _oracle_ref(grid, T, S, V, t0=t0)
    for v in VARIANTS:
        _check(got[v], grid, T, S, V, w, ref, v)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_supplied_reference_that_is_not_step_0(ml, dtype):
    grid, T, S, V, w = _case(6, 16, 64, dtype=dtype)
    got = _gpu(ml, grid, T, S, V, w, t0=4)
    ref = _oracle_ref(grid, T, S, V, t0=4)
    for v in VARIANTS:
        _check(got[v], grid, T, S, V, w, ref, v)
        assert (got[v][4] == 0).all()  # the step that is the reference state


def test_2d_patm(ml):
    grid, T, S, V, w = _case(5, 16, 64, hole=True)
    patm = 101325.0 + 50.0 * np.sin(np.arange(16 * 64).reshape(16, 64))
    got = _gpu(ml, grid, T, S, V, w, patm=patm)
    assert ml.core.last_path() == 1  # the column pressure takes the plain-load kernel
    ref = _oracle_ref(grid, T, S, V, patm=patm)
    for v in VARIANTS:
        _check(got[v], grid, T, S, V, w, ref, v, patm=patm)


# -------------------------------------------------------------------------------------------- identities


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_levels_sum_to_the_weighted_mean_of_steric_height(ml, dtype):
    ds = synth.make_dataset(5, NZ, 20, 132, seed=11, device="cuda", dtype=dtype)
    prof, _ = ml.steric_profile(ds, variant=list(VARIANTS))
    area = ds["areacello"].data.to(torch.float64)
    for v in VARIANTS:
        eta = ml.steric(ds, variant=v)[0][v].data
        terms = area[None] * eta
        want = torch.nansum(terms, dim=(1, 2)) / torch.nansum(area)
        got = prof[v].data.sum(dim=1)
        scale = torch.nansum(terms.abs(), dim=(1, 2)) / torch.nansum(area)
        # eta comes from another kernel: its densities may round differently, as against the oracle
        dz = ml.core.calc_dz(ds["z_i"].data, ds["deptho"].data)
        wsum = float(torch.nansum(area[None] * dz) / torch.nansum(area))
        tol = 1e-12 * scale + RHO_FLOOR / 1035.0 * wsum
        assert ((got - want).abs() <= tol).all(), (v, float((got - want).abs().max()))


def test_self_reference_step_0_is_exactly_zero(ml):
    for dtype, shape in ((torch.float32, (4, NZ, 20, 132)), (torch.float64, (4, NZ, 13, 37))):
        ds = synth.make_dataset(*shape, seed=3, device="cuda", dtype=dtype)
        for eos in ("Wright", "Linear"):
            prof, _ = ml.steric_profile(ds, variant=list(VARIANTS), equation_of_state=eos)
            for v in VARIANTS:
                assert (prof[v].data[0] == 0).all(), (dtype, eos, v)
                assert (prof[v].data[1:] != 0).any()


def _pairs():
    return [("steric", "thermosteric"), ("steric", "halosteric"), ("thermosteric", "halosteric"), VARIANTS]


@pytest.mark.parametrize("dtype, shape", [(torch.float32, (12, 32, 128)), (torch.float32, (5, 13, 37)),
                                          (torch.float64, (5, 20, 132))], ids=["ring", "ragged", "f64"])
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_one_pass_equals_one_launch_per_variant(ml, dtype, shape, eos):
    grid, T, S, V, w = _case(*shape, dtype=dtype, hole=True, vmask=True)
    single = {v: _gpu(ml, grid, T, S, V, w, t0=2, eos=eos, variants=v)[v] for v in VARIANTS}
    for names in _pairs():
        got = _gpu(ml, grid, T, S, V, w, t0=2, eos=eos, variants=names)
        for v in names:
            assert torch.equal(got[v], single[v]), (names, v)
    prev = ml.core.force_direct(2)  # one launch per variant inside the library
    try:
        split = _gpu(ml, grid, T, S, V, w, t0=2, eos=eos)
    finally:
        ml.core.force_direct(prev)
    for v in VARIANTS:
        assert torch.equal(split[v], single[v])


@pytest.mark.parametrize("shape", [(12, 32, 128), (7, 12, 20), (3, 20, 132)])
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_ring_and_plain_loads_agree_bit_for_bit(ml, shape, eos):
    grid, T, S, V, w = _case(*shape, hole=True, vmask=True, weights="nan_zero")
    ring = _gpu(ml, grid, T, S, V, w, t0=1, eos=eos)
    assert ml.core.last_path() == 2
    prev = ml.core.force_direct(1)
    try:
        plain = _gpu(ml, grid, T, S, V, w, t0=1, eos=eos)
        assert ml.core.last_path() == 1
    finally:
        ml.core.force_direct(prev)
    for v in VARIANTS:
        assert torch.equal(ring[v], plain[v]), v


def test_reproducible(ml):
    grid, T, S, V, w = _case(13, 32, 128, hole=True)
    a = _gpu(ml, grid, T, S, V, w)
    b = _gpu(ml, grid, T, S, V, w)
    for v in VARIANTS:
        assert torch.equal(a[v], b[v])


def test_launches_its_own_kernels(ml):
    grid, T, S, V, w = _case(3, 16, 64)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _gpu(ml, grid, T, S, V, w)
        torch.cuda.synchronize()
    names = {e.name for e in prof.events()}
    assert any("k_stream_profile" in n for n in names), sorted(names)
    assert any("k_reduce_rows" in n for n in names)


# ------------------------------------------------------------------------------------------------- public call


def test_public_call_on_the_reference_test_data(ml):
    ds = ml.test_data.generate_test_data()
    f = lambda k: np.asarray(ds[k].values, dtype=np.float64)  # noqa: E731
    ref = osteric.reference_state(f("thetao"), f("so"), f("volcello"), f("areacello"), f("z_l"))
    grid = {k: torch.from_numpy(f(k)) for k in ("z_l", "z_i", "deptho", "areacello")}
    res, reference = ml.steric_profile(ds, variant=list(VARIANTS))
    for v in VARIANTS:
        assert res[v].dims == ("time", "z_l") and res[v].encoding["dtype"] == "float32"
        single, _ = ml.steric_profile(ds, variant=v)
        assert np.array_equal(np.asarray(single[v].values), np.asarray(res[v].values))
        _check(torch.as_tensor(np.asarray(res[v].values)), grid, f("thetao"), f("so"), f("volcello"),
               grid["areacello"], ref, v)


def test_public_call_basin_weights_and_supplied_reference(ml):
    ds = synth.make_dataset(6, NZ, 20, 132, seed=9, device="cuda", dtype=torch.float32)
    _, reference = ml.steric(ds)
    basin = ds["areacello"].data * (torch.arange(132, device="cuda")[None, :] < 60)
    res, ref2 = ml.steric_profile(ds, variant=("halosteric", "steric"), weights=basin, reference=reference)
    assert ref2 is reference
    f = lambda k: ds[k].data  # noqa: E731
    want = ml.core.steric_local_profile(f("thetao"), f("so"), reference["thetao"].data, reference["so"].data,
                                        reference["rho"].data, reference["volcello"].data, f("z_i"), f("deptho"),
                                        f("z_l").to(torch.float64) * 1.0e4 + 101325.0, basin,
                                        variants=("halosteric", "steric"))
    for v in ("halosteric", "steric"):
        assert torch.equal(res[v].data, want[v])


@pytest.fixture()
def xr(monkeypatch):
    if importlib.util.find_spec("xarray") is None:
        monkeypatch.syspath_prepend(str(pathlib.Path(__file__).resolve().parent / "_stubs"))
        monkeypatch.delitem(sys.modules, "xarray", raising=False)
    import xarray

    yield xarray
    if getattr(xarray, "__version__", "").endswith("stub"):
        sys.modules.pop("xarray", None)


def test_xarray_round_trip(ml, xr):
    lab = ml.test_data.generate_test_data()
    ds = xr.Dataset(attrs={"title": "config 1"})
    for name, var in lab.variables.items():
        ds[name] = xr.DataArray(np.asarray(var.values), dims=var.dims, attrs=dict(var.attrs))
    result, reference = ml.steric_profile(ds, variant=list(VARIANTS))
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    want, _ = ml.steric_profile(lab, variant=list(VARIANTS))
    for v in VARIANTS:
        assert result[v].dims == ("time", "z_l")
        assert np.array_equal(np.asarray(result[v].values), np.asarray(want[v].values))
