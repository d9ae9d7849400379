"""steric_profile() without a device: validation, what reaches core.steric_local_profile, and the result's dims,
attrs, encoding and annual means.  The device call is replaced by a recorder; the numbers are checked on the GPU in
tests/test_gpu_steric_profile.py."""

import importlib
import pathlib
import sys

import numpy as np
import pytest
import torch

import momlevel_b200 as ml
from momlevel_b200 import core, synth
from momlevel_b200.labeled import ChunkedArray, DataArray, Dataset
import profile_oracle  # tests/profile_oracle.py
from oracle import steric as osteric

steric_mod = importlib.import_module("momlevel_b200.steric")
VARIANTS = ("steric", "thermosteric", "halosteric")


def _small(nt=3, nz=12, ny=20, nx=32):
    return synth.make_dataset(nt, nz, ny, nx, seed=5, device="cpu", dtype=torch.float32)


def _np(ds, k):
    return np.asarray(ds[k].values, dtype=np.float64)


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
    """Stands in for core.steric_local_profile: records what is asked, returns variant index + call number."""

    def __init__(self):
        self.calls = []

    def profile(self, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, rhozero=1035.0, eos="Wright",
                variants=VARIANTS):
        self.calls.append({"variants": tuple(variants), "T_ref": tuple(np.shape(T_ref)), "S_ref": tuple(np.shape(S_ref)),
                           "weights": np.asarray(weights, dtype=np.float64).copy(), "eos": eos, "rhozero": rhozero,
                           "p": p_level})
        shape = (T.shape[0], T.shape[1])
        return {v: torch.full(shape, float(VARIANTS.index(v)), dtype=torch.float64) for v in variants}


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(core, "steric_local_profile", r.profile)
    monkeypatch.setattr(steric_mod, "setup_reference_state", lambda dset, **kw: _reference(dset))
    return r


# ------------------------------------------------------------------------------------------------------ validation


@pytest.mark.parametrize("bad", ["barotropic", "Steric", [], (), ("steric", "steric"), ["steric", "x"], [None]])
def test_unknown_or_repeated_variants_raise_before_any_work(monkeypatch, bad):
    def no_work(*a, **k):
        raise AssertionError("work started before the variant was checked")

    monkeypatch.setattr(steric_mod, "validate_dataset", no_work)
    monkeypatch.setattr(steric_mod, "setup_reference_state", no_work)
    monkeypatch.setattr(core, "steric_local_profile", no_work)
    with pytest.raises(ValueError):
        ml.steric_profile(_small(), variant=bad)


@pytest.mark.parametrize("shape", [(20, 31), (32, 20), (640,), (1, 20, 32)])
def test_weights_that_do_not_match_the_grid_raise(rec, shape):
    with pytest.raises(ValueError, match="horizontal grid"):
        ml.steric_profile(_small(), weights=np.ones(shape))
    assert rec.calls == []


def test_wrong_layout_raises(rec):
    ds = _small()
    for k in ("thetao", "so"):
        ds[k] = DataArray(np.ascontiguousarray(np.swapaxes(ds[k].values, 0, 1)), ("z_l", "time") + ds[k].dims[2:],
                          attrs=ds[k].attrs)
    with pytest.raises(ValueError, match="laid out"):
        ml.steric_profile(ds)
    assert rec.calls == []


def test_missing_interfaces_raise(rec):
    ds = _small()
    ds = ds.drop_vars(["z_i"])
    with pytest.raises(ValueError):
        ml.steric_profile(ds)
    assert rec.calls == []


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
        ml.steric_profile(ds, variant=list(VARIANTS))
    assert rec.calls == []


# ------------------------------------------------------------------------------------------ what reaches the core


@pytest.mark.parametrize("variant", ["thermosteric", VARIANTS, ("halosteric", "steric")])
def test_one_core_call_and_the_result(rec, variant):
    ds = _small()
    res, ref = ml.steric_profile(ds, variant=variant, equation_of_state="Linear", rhozero=1025.0)
    names = (variant,) if isinstance(variant, str) else tuple(variant)
    nt, nz, ny, nx = ds["thetao"].shape
    assert len(rec.calls) == 1
    call = rec.calls[0]
    assert call["variants"] == names and call["eos"] == "Linear" and call["rhozero"] == 1025.0
    assert call["T_ref"] == (nz, ny, nx) and call["S_ref"] == (nz, ny, nx)
    np.testing.assert_array_equal(call["weights"], _np(ds, "areacello"))  # areacello by default
    assert [v for v in VARIANTS if v in res.variables] == [v for v in VARIANTS if v in names]
    for v in names:
        r = res[v]
        assert r.dims == ("time", "z_l") and r.shape == (nt, nz)
        assert r.attrs == {"long_name": f"{v.capitalize()} height adjustment by level, area-weighted mean", "units": "m"}
        assert r.encoding["dtype"] == "float32"
        assert (np.asarray(r.values) == VARIANTS.index(v)).all()
    np.testing.assert_array_equal(np.asarray(res["z_l"].values), _np(ds, "z_l"))
    assert res["z_l"].attrs == ds["z_l"].attrs
    assert np.asarray(res["time"].values).shape == (nt,)


def test_basin_weights_and_a_supplied_reference(rec):
    ds = _small()
    basin = _np(ds, "areacello") * (np.arange(32)[None, :] < 16)
    ref = _reference(ds)
    res, ref2 = ml.steric_profile(ds, weights=basin, reference=ref, dtype="float64")
    assert ref2 is ref
    np.testing.assert_array_equal(rec.calls[0]["weights"], basin)
    assert res["steric"].encoding["dtype"] == "float64"
    # a labelled DataArray and a torch tensor are taken as they are
    ml.steric_profile(ds, weights=DataArray(basin, ds["areacello"].dims), reference=ref)
    ml.steric_profile(ds, weights=torch.from_numpy(basin), reference=ref)
    for c in rec.calls[1:]:
        np.testing.assert_array_equal(c["weights"], basin)


def test_a_2d_patm_reaches_the_core_as_a_column_pressure(rec):
    ds = _small()
    patm = np.full(ds["areacello"].shape, 101325.0) + np.arange(32)[None, :]
    ml.steric_profile(ds, patm=patm, reference=_reference(ds))
    assert isinstance(rec.calls[0]["p"], core.Pressure)


def test_annual_means(rec):
    ds = _small(nt=24)
    days = np.tile([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], 2).astype(np.float64)
    res, _ = ml.steric_profile(ds, variant=["steric", "halosteric"], annual=True, days_in_month=days)
    assert [c["variants"] for c in rec.calls] == [("steric", "halosteric")]
    assert res["halosteric"].shape == (2, 12) and res["halosteric"].dims == ("time", "z_l")
    assert (np.asarray(res["halosteric"].values) == 2.0).all()
    assert res["steric"].attrs["units"] == "m"


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
    ds = xr.Dataset(attrs={"title": "profile"})
    for name, var in lab.variables.items():
        ds[name] = xr.DataArray(np.asarray(var.values), dims=var.dims, attrs=dict(var.attrs))
    w = xr.DataArray(np.asarray(lab["areacello"].values) * 0.5, dims=lab["areacello"].dims)
    result, reference = ml.steric_profile(ds, variant=["thermosteric"], weights=w)
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    assert result["thermosteric"].dims == ("time", "z_l")
    assert result["thermosteric"].attrs["long_name"] == "Thermosteric height adjustment by level, area-weighted mean"
    np.testing.assert_array_equal(rec.calls[0]["weights"], np.asarray(lab["areacello"].values) * 0.5)


# ------------------------------------------------------------------------------------------------------- the oracle


@pytest.mark.parametrize("variant", VARIANTS)
def test_oracle_sums_over_levels_to_the_weighted_mean_height(variant):
    ds = _small()
    T, S, V = _np(ds, "thetao"), _np(ds, "so"), _np(ds, "volcello")
    area = _np(ds, "areacello")
    ref = osteric.reference_state(T, S, V, area, _np(ds, "z_l"))
    eta, _ = osteric.steric_local(T, S, _np(ds, "z_l"), _np(ds, "z_i"), _np(ds, "deptho"), ref, variant=variant)
    prof, scale = profile_oracle.steric_profile(T, S, _np(ds, "z_l"), _np(ds, "z_i"), _np(ds, "deptho"), ref,
                                                variant=variant)
    want = np.nansum(area[None] * eta, axis=(1, 2)) / np.nansum(area)
    np.testing.assert_allclose(prof.sum(axis=1), want, rtol=0, atol=1e-12 * scale.sum(axis=1).max())
    np.testing.assert_array_equal(prof[0], 0.0)  # the reference state is step 0
