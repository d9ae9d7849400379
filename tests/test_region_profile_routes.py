"""steric_profile(regions=...) without a device: the checks on the region map and its codes, what reaches
core.steric_local_region_profile, and the result's dims, region coordinate, weights, attrs, encoding and annual
means.  The device call is replaced by a recorder; the numbers are checked on the GPU in
tests/test_gpu_region_profile.py."""

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


def _basins():
    """CMIP-like codes: 0 (land) in the first columns, then 1, 2, 3 and 5 in blocks, NaN and -1 in a few columns."""
    r = np.zeros((NY, NX))
    r[:, 4:12] = 1
    r[:, 12:20] = 2
    r[:10, 20:] = 3
    r[10:, 20:] = 5
    r[0, 0] = np.nan
    r[1, 1] = -1
    return r


class _Recorder:
    """Stands in for core.steric_local_region_profile: records what is asked, returns 10 * region + variant index."""

    def __init__(self):
        self.calls = []

    def profile(self, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, region_index, nregions,
                rhozero=1035.0, eos="Wright", variants=VARIANTS):
        self.calls.append({"variants": tuple(variants), "weights": np.asarray(weights, dtype=np.float64).copy(),
                           "index": np.asarray(region_index).copy(), "nregions": nregions, "eos": eos,
                           "rhozero": rhozero, "p": p_level})
        nt, nz = T.shape[0], T.shape[1]
        r = torch.arange(nregions, dtype=torch.float64)[:, None, None]
        profs = {v: (10 * r + VARIANTS.index(v)).expand(nregions, nt, nz).clone() for v in variants}
        return profs, 100.0 + torch.arange(nregions, dtype=torch.float64)


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(core, "steric_local_region_profile", r.profile)
    monkeypatch.setattr(steric_mod, "setup_reference_state", lambda dset, **kw: _reference(dset))
    return r


# ------------------------------------------------------------------------------------------------------ validation


def _bad_cases():
    r = _basins()
    frac = r.copy()
    frac[3, 7] = 1.5
    inf = r.copy()
    inf[2, 2] = np.inf
    many = np.arange(NY * NX, dtype=np.float64).reshape(NY, NX) % 16  # 16 codes present
    return [
        dict(regions=frac),                                    # a finite non-integral code
        dict(regions=inf),
        dict(regions=np.ones((NY, NX - 1))),                   # not the horizontal grid
        dict(regions=np.ones((NX, NY))),
        dict(regions=np.ones((NY * NX,))),
        dict(regions=many),                                    # more than 15 codes present
        dict(regions=r, region_codes=list(range(16))),         # more than 15 codes selected
        dict(regions=r, region_codes=[1, 2, 1]),               # a duplicate
        dict(regions=r, region_codes=[1, -2]),                 # a negative code
        dict(regions=r, region_codes=[1, 2.5]),
        dict(regions=r, region_codes=[]),
        dict(region_codes=[1, 2]),                             # codes without a map
        dict(regions=np.full((NY, NX), np.nan)),               # no code at all
    ]


@pytest.mark.parametrize("kw", _bad_cases(), ids=[
    "fraction", "inf", "short_x", "transposed", "flat", "16_present", "16_selected", "duplicate", "negative",
    "fraction_code", "no_codes", "codes_without_map", "all_nan"])
def test_bad_maps_and_codes_raise_before_any_work(monkeypatch, kw):
    def no_work(*a, **k):
        raise AssertionError("work started before the region map was checked")

    monkeypatch.setattr(steric_mod, "validate_dataset", no_work)
    monkeypatch.setattr(steric_mod, "setup_reference_state", no_work)
    monkeypatch.setattr(steric_mod, "_pressure", no_work)
    monkeypatch.setattr(core, "steric_local_profile", no_work)
    monkeypatch.setattr(core, "steric_local_region_profile", no_work)
    with pytest.raises(ValueError) as err:
        ml.steric_profile(_small(), **kw)
    if "region_codes" in kw:
        assert "region_codes" in str(err.value)


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
        ml.steric_profile(ds, regions=_basins())
    assert rec.calls == []


# ------------------------------------------------------------------------------------------ what reaches the core


def test_default_codes_are_the_sorted_non_negative_codes_present(rec):
    ds = _small()
    res, _ = ml.steric_profile(ds, regions=_basins()[:, ::-1].copy())
    assert np.asarray(res["region"].values).tolist() == [0, 1, 2, 3, 5]
    assert rec.calls[0]["nregions"] == 5


def test_index_of_each_column(rec):
    ds = _small()
    r = _basins()
    ml.steric_profile(ds, regions=r, region_codes=[5, 1, 2, 3])
    idx = rec.calls[0]["index"]
    assert idx.shape == (NY, NX) and idx.dtype == np.int8
    want = np.full((NY, NX), -1)
    for i, c in enumerate([5, 1, 2, 3]):
        want[r == c] = i
    np.testing.assert_array_equal(idx, want)
    # NaN, negative and unselected (0) codes are in no region
    assert idx[0, 0] == -1 and idx[1, 1] == -1 and (idx[:, 2:4] == -1).all()
    assert rec.calls[0]["nregions"] == 4


@pytest.mark.parametrize("kind", ["numpy_int", "numpy_float", "torch", "labelled"])
def test_map_types(rec, kind):
    ds = _small()
    r = np.nan_to_num(_basins(), nan=-1.0)
    arg = {"numpy_int": r.astype(np.int16), "numpy_float": r, "torch": torch.from_numpy(r).to(torch.int32),
           "labelled": DataArray(r, ds["areacello"].dims)}[kind]
    res, _ = ml.steric_profile(ds, regions=arg)
    assert np.asarray(res["region"].values).tolist() == [0, 1, 2, 3, 5]
    want = np.full((NY, NX), -1)
    for i, c in enumerate([0, 1, 2, 3, 5]):
        want[r == c] = i
    np.testing.assert_array_equal(rec.calls[0]["index"], want)


@pytest.mark.parametrize("variant", ["halosteric", VARIANTS, ("thermosteric", "steric")])
def test_one_core_call_and_the_result(rec, variant):
    ds = _small()
    codes = [1, 2, 3, 5, 7]  # 7 has no columns: the core gives its NaN, the result keeps its place
    res, _ = ml.steric_profile(ds, variant=variant, regions=_basins(), region_codes=codes,
                               equation_of_state="Linear", rhozero=1025.0, dtype="float64")
    names = (variant,) if isinstance(variant, str) else tuple(variant)
    nt, nz = ds["thetao"].shape[:2]
    assert len(rec.calls) == 1
    call = rec.calls[0]
    assert call["variants"] == names and call["eos"] == "Linear" and call["rhozero"] == 1025.0
    np.testing.assert_array_equal(call["weights"], np.asarray(ds["areacello"].values, dtype=np.float64))
    for v in names:
        r = res[v]
        assert r.dims == ("time", "region", "z_l") and r.shape == (nt, len(codes), nz)
        assert r.attrs == {"long_name": f"{v.capitalize()} height adjustment by level and region, area-weighted mean",
                           "units": "m"}
        assert r.encoding["dtype"] == "float64"
        got = np.asarray(r.values)
        for i in range(len(codes)):
            assert (got[:, i] == 10 * i + VARIANTS.index(v)).all()
    assert res["region"].dims == ("region",) and np.asarray(res["region"].values).tolist() == codes
    assert res["region_weight"].dims == ("region",)
    np.testing.assert_array_equal(np.asarray(res["region_weight"].values), 100.0 + np.arange(len(codes)))
    np.testing.assert_array_equal(np.asarray(res["z_l"].values), np.asarray(ds["z_l"].values))


def test_weights_reach_the_core(rec):
    ds = _small()
    basin = np.asarray(ds["areacello"].values, dtype=np.float64) * 0.5
    ref = _reference(ds)
    res, ref2 = ml.steric_profile(ds, regions=_basins(), weights=basin, reference=ref)
    assert ref2 is ref
    np.testing.assert_array_equal(rec.calls[0]["weights"], basin)


def test_a_2d_patm_reaches_the_core_as_a_column_pressure(rec):
    ds = _small()
    patm = np.full(ds["areacello"].shape, 101325.0) + np.arange(NX)[None, :]
    ml.steric_profile(ds, patm=patm, reference=_reference(ds), regions=_basins())
    assert isinstance(rec.calls[0]["p"], core.Pressure)


def test_annual_means(rec):
    ds = _small(nt=24)
    days = np.tile([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], 2).astype(np.float64)
    res, _ = ml.steric_profile(ds, variant=["steric", "halosteric"], annual=True, days_in_month=days,
                               regions=_basins(), region_codes=[2, 3])
    assert [c["variants"] for c in rec.calls] == [("steric", "halosteric")]
    assert res["halosteric"].shape == (2, 2, 12) and res["halosteric"].dims == ("time", "region", "z_l")
    got = np.asarray(res["halosteric"].values)
    assert (got[:, 0] == 2.0).all() and (got[:, 1] == 12.0).all()
    assert res["region_weight"].dims == ("region",) and np.asarray(res["region"].values).tolist() == [2, 3]


def test_without_regions_the_call_is_unchanged(monkeypatch):
    calls = []

    def profile(T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, rhozero=1035.0, eos="Wright",
                variants=VARIANTS):
        calls.append(tuple(variants))
        return {v: torch.zeros((T.shape[0], T.shape[1]), dtype=torch.float64) for v in variants}

    def no_regions(*a, **k):
        raise AssertionError("no region map was given")

    monkeypatch.setattr(core, "steric_local_profile", profile)
    monkeypatch.setattr(core, "steric_local_region_profile", no_regions)
    monkeypatch.setattr(steric_mod, "setup_reference_state", lambda dset, **kw: _reference(dset))
    res, _ = ml.steric_profile(_small(), variant=list(VARIANTS))
    assert calls == [VARIANTS]
    assert res["steric"].dims == ("time", "z_l") and "region" not in res.variables


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
    basins = xr.DataArray(_basins(), dims=lab["areacello"].dims)
    result, reference = ml.steric_profile(ds, variant=["thermosteric"], regions=basins, region_codes=[1, 2])
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    assert result["thermosteric"].dims == ("time", "region", "z_l")
    assert np.asarray(result["region"].values).tolist() == [1, 2]
    assert result["region_weight"].dims == ("region",)
    np.testing.assert_array_equal(rec.calls[0]["index"][:, 4:12], 0)
