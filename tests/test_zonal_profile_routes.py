"""steric_profile(zonal=True) without a device: the checks before any work, what reaches
core.steric_local_zonal_profile, and the result's dims, y coordinate, row weights, attrs, encoding and annual means.
The device call is replaced by a recorder; the numbers are checked on the GPU in tests/test_gpu_zonal_profile.py."""

import importlib
import pathlib
import sys

import numpy as np
import pytest
import torch

import momlevel_b200 as ml
from momlevel_b200 import core, synth
from momlevel_b200.labeled import ChunkedArray, DataArray, Dataset

steric_mod = importlib.import_module("momlevel_b200.steric")
VARIANTS = ("steric", "thermosteric", "halosteric")
NY, NX = 20, 32


def _small(nt=3, nz=12):
    return synth.make_dataset(nt, nz, NY, NX, seed=5, device="cpu", dtype=torch.float32)


def _reference(ds):
    """A reference state with the variables and ranks steric_profile checks (its values are never computed with)."""
    ref = Dataset()
    for k in ("thetao", "so", "volcello"):
        ref[k] = DataArray(np.asarray(ds[k].values)[0].copy(), ds[k].dims[1:])
    ref["rho"] = DataArray(np.full(ds["thetao"].shape[1:], 1030.0), ds["thetao"].dims[1:])
    ref["areacello"] = DataArray(np.asarray(ds["areacello"].values), ds["areacello"].dims)
    for k, v in (("volo", 2.0), ("masso", 2060.0), ("rhoga", 1030.0)):
        ref[k] = DataArray(np.float64(v), ())
    return ref


class _Recorder:
    """Stands in for core.steric_local_zonal_profile: records what is asked, returns 10 * row + variant index."""

    def __init__(self):
        self.calls = []

    def profile(self, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, rhozero=1035.0,
                eos="Wright", variants=VARIANTS):
        self.calls.append({"variants": tuple(variants), "weights": np.asarray(weights, dtype=np.float64).copy(),
                           "shape": tuple(T.shape), "eos": eos, "rhozero": rhozero, "p": p_level})
        nt, nz, ny = T.shape[0], T.shape[1], T.shape[2]
        j = torch.arange(ny, dtype=torch.float64)
        profs = {v: (10 * j + VARIANTS.index(v)).expand(nt, nz, ny).clone() for v in variants}
        return profs, 100.0 + j


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(core, "steric_local_zonal_profile", r.profile)
    monkeypatch.setattr(steric_mod, "setup_reference_state", lambda dset, **kw: _reference(dset))
    return r


def _no_work(monkeypatch):
    def no_work(*a, **k):
        raise AssertionError("work started before the arguments were checked")

    monkeypatch.setattr(core, "steric_local_profile", no_work)
    monkeypatch.setattr(core, "steric_local_region_profile", no_work)
    monkeypatch.setattr(core, "steric_local_zonal_profile", no_work)
    monkeypatch.setattr(steric_mod, "setup_reference_state", no_work)


# ------------------------------------------------------------------------------------------------------ validation


def test_zonal_with_regions_raises_before_any_work(monkeypatch):
    _no_work(monkeypatch)
    monkeypatch.setattr(steric_mod, "validate_dataset", lambda *a, **k: (_ for _ in ()).throw(AssertionError()))
    monkeypatch.setattr(steric_mod, "_pressure", lambda *a, **k: (_ for _ in ()).throw(AssertionError()))
    with pytest.raises(ValueError, match="regions"):
        ml.steric_profile(_small(), zonal=True, regions=np.ones((NY, NX)))
    with pytest.raises(ValueError, match="regions"):
        ml.steric_profile(_small(), zonal=True, regions=np.ones((NY, NX)), region_codes=[1])


@pytest.mark.parametrize("shape", [(NY, NX - 1), (NX, NY), (NY * NX,), (1, NX), (NY,)],
                         ids=["short_x", "transposed", "flat", "one_row", "one_column"])
def test_weights_of_the_wrong_shape(monkeypatch, shape):
    _no_work(monkeypatch)
    with pytest.raises(ValueError, match="weights"):
        ml.steric_profile(_small(), zonal=True, weights=np.ones(shape))


def test_fields_not_laid_out_time_z_y_x(monkeypatch):
    _no_work(monkeypatch)
    ds = _small()
    swapped = Dataset()
    for name, var in ds.variables.items():
        if name in ("thetao", "so", "volcello"):
            swapped[name] = DataArray(np.ascontiguousarray(np.swapaxes(np.asarray(var.values), 0, 1)),
                                      ("z_l", "time", "yh", "xh"))
        else:
            swapped[name] = var
    with pytest.raises(ValueError, match="laid out"):
        ml.steric_profile(swapped, zonal=True)
    flat = Dataset()  # (time, z, column): no grid rows
    for name, var in ds.variables.items():
        v = np.asarray(var.values)
        if name in ("thetao", "so", "volcello"):
            flat[name] = DataArray(v.reshape(v.shape[0], v.shape[1], -1).copy(), ("time", "z_l", "col"))
        else:
            flat[name] = var
    with pytest.raises(ValueError):
        ml.steric_profile(flat, zonal=True)


def test_chunked_fields_are_not_supported_yet(rec):
    ds = _small()
    for name in ("thetao", "so", "volcello"):
        full = ds[name].values

        def blocks(full=full):
            yield np.array(full[:2])
            yield np.array(full[2:])

        ds[name] = DataArray(ChunkedArray(full.shape, full.dtype, (2, full.shape[0] - 2), blocks), ds[name].dims,
                             attrs=ds[name].attrs)
    with pytest.raises(NotImplementedError):
        ml.steric_profile(ds, zonal=True)
    assert rec.calls == []


# ------------------------------------------------------------------------------------------ what reaches the core


@pytest.mark.parametrize("variant", ["halosteric", VARIANTS, ("thermosteric", "steric")])
def test_one_core_call_and_the_result(rec, variant):
    ds = _small()
    ds["yh"].attrs = {"long_name": "h point nominal latitude", "units": "degrees_north"}
    res, _ = ml.steric_profile(ds, variant=variant, zonal=True, equation_of_state="Linear", rhozero=1025.0,
                               dtype="float64")
    names = (variant,) if isinstance(variant, str) else tuple(variant)
    nt, nz = ds["thetao"].shape[:2]
    assert len(rec.calls) == 1
    call = rec.calls[0]
    assert call["variants"] == names and call["eos"] == "Linear" and call["rhozero"] == 1025.0
    assert call["shape"] == (nt, nz, NY, NX)
    np.testing.assert_array_equal(call["weights"], np.asarray(ds["areacello"].values, dtype=np.float64))
    for v in names:
        r = res[v]
        assert r.dims == ("time", "z_l", "yh") and r.shape == (nt, nz, NY)
        assert r.attrs == {"long_name": f"{v.capitalize()} height adjustment by level and grid row, area-weighted mean",
                           "units": "m"}
        assert r.encoding["dtype"] == "float64"
        got = np.asarray(r.values)
        for j in range(NY):
            assert (got[:, :, j] == 10 * j + VARIANTS.index(v)).all()
    assert res["zonal_weight"].dims == ("yh",)
    np.testing.assert_array_equal(np.asarray(res["zonal_weight"].values), 100.0 + np.arange(NY))
    assert res["zonal_weight"].attrs == {"long_name": "Sum of the column weights of the grid row (nansum(w))"}
    # the y coordinate of the dataset, with its attrs, and the level coordinate
    np.testing.assert_array_equal(np.asarray(res["yh"].values), np.asarray(ds["yh"].values))
    assert res["yh"].attrs == {"long_name": "h point nominal latitude", "units": "degrees_north"}
    np.testing.assert_array_equal(np.asarray(res["z_l"].values), np.asarray(ds["z_l"].values))
    assert "xh" not in res.variables and "region" not in res.variables


def test_without_a_y_coordinate_none_is_attached(rec):
    ds = _small()
    bare = Dataset()
    for name, var in ds.variables.items():
        if name != "yh":
            bare[name] = var
    res, _ = ml.steric_profile(bare, zonal=True)
    assert res["steric"].dims == ("time", "z_l", "yh") and "yh" not in res.variables


def test_basin_weights_reach_the_core(rec):
    ds = _small()
    basin = np.asarray(ds["areacello"].values, dtype=np.float64) * (np.arange(NX)[None, :] < 12)
    basin[3, 5] = np.nan
    ref = _reference(ds)
    res, ref2 = ml.steric_profile(ds, zonal=True, weights=basin, reference=ref)
    assert ref2 is ref
    np.testing.assert_array_equal(rec.calls[0]["weights"], basin)
    ml.steric_profile(ds, zonal=True, weights=DataArray(basin, ds["areacello"].dims), reference=ref)
    np.testing.assert_array_equal(rec.calls[1]["weights"], basin)


def test_a_2d_patm_reaches_the_core_as_a_column_pressure(rec):
    ds = _small()
    patm = np.full(ds["areacello"].shape, 101325.0) + np.arange(NX)[None, :]
    ml.steric_profile(ds, patm=patm, reference=_reference(ds), zonal=True)
    assert isinstance(rec.calls[0]["p"], core.Pressure)


def test_annual_means(rec):
    ds = _small(nt=24)
    days = np.tile([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], 2).astype(np.float64)
    res, _ = ml.steric_profile(ds, variant=["steric", "halosteric"], annual=True, days_in_month=days, zonal=True)
    assert [c["variants"] for c in rec.calls] == [("steric", "halosteric")]
    assert res["halosteric"].shape == (2, 12, NY) and res["halosteric"].dims == ("time", "z_l", "yh")
    got = np.asarray(res["halosteric"].values)
    assert (got[:, :, 3] == 32.0).all()
    assert res["zonal_weight"].dims == ("yh",)


def test_zonal_false_makes_the_calls_of_before(monkeypatch):
    calls = []

    def profile(T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, rhozero=1035.0, eos="Wright",
                variants=VARIANTS):
        calls.append((tuple(variants), tuple(T.shape), eos, rhozero))
        return {v: torch.zeros((T.shape[0], T.shape[1]), dtype=torch.float64) for v in variants}

    def not_zonal(*a, **k):
        raise AssertionError("zonal=False must not take the zonal route")

    monkeypatch.setattr(core, "steric_local_profile", profile)
    monkeypatch.setattr(core, "steric_local_zonal_profile", not_zonal)
    monkeypatch.setattr(steric_mod, "setup_reference_state", lambda dset, **kw: _reference(dset))
    res, _ = ml.steric_profile(_small(), variant=list(VARIANTS))
    res2, _ = ml.steric_profile(_small(), variant=list(VARIANTS), zonal=False)
    assert calls == [(VARIANTS, (3, 12, NY, NX), "Wright", 1035.0)] * 2
    for r in (res, res2):
        assert r["steric"].dims == ("time", "z_l") and "zonal_weight" not in r.variables


# ---------------------------------------------------------------------------------------------- xarray round trip


@pytest.fixture()
def xr(monkeypatch):
    if importlib.util.find_spec("xarray") is None:
        monkeypatch.syspath_prepend(str(pathlib.Path(__file__).resolve().parent / "_stubs"))
        monkeypatch.delitem(sys.modules, "xarray", raising=False)
    import xarray

    yield xarray
    if getattr(xarray, "__version__", "").endswith("stub"):
        sys.modules.pop("xarray", None)


def test_xarray_round_trip(rec, xr):
    lab = _small()
    ds = xr.Dataset(attrs={"title": "section"})
    for name, var in lab.variables.items():
        ds[name] = xr.DataArray(np.asarray(var.values), dims=var.dims, attrs=dict(var.attrs))
    basin = xr.DataArray(np.asarray(lab["areacello"].values) * 2.0, dims=lab["areacello"].dims)
    result, reference = ml.steric_profile(ds, variant=["thermosteric"], zonal=True, weights=basin)
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    assert result["thermosteric"].dims == ("time", "z_l", "yh")
    assert result["zonal_weight"].dims == ("yh",)
    np.testing.assert_array_equal(np.asarray(result["yh"].values), np.asarray(lab["yh"].values))
    np.testing.assert_array_equal(rec.calls[0]["weights"], np.asarray(lab["areacello"].values) * 2.0)
