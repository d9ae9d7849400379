"""steric_layers(variant=[...]) / ml_steric_local_layers_variants without a device: the validation of the variant
list, the argument errors the library reports before any launch, and which core entry point each kind of call
reaches.  The device calls are replaced (no GPU here); the numbers are checked on the GPU in
tests/test_gpu_layers_variants.py."""

import ctypes
import importlib

import numpy as np
import pytest
import torch

import momlevel_b200 as ml
from momlevel_b200 import _lib, core, synth
from momlevel_b200.labeled import DataArray, Dataset

steric_mod = importlib.import_module("momlevel_b200.steric")
VARIANTS = ("steric", "thermosteric", "halosteric")


def _small(nt=3, nz=12, ny=20, nx=32):
    return synth.make_dataset(nt, nz, ny, nx, seed=5, device="cpu", dtype=torch.float32)


def _reference(ds):
    """A reference state with the variables and ranks steric_layers checks (its values are never computed with)."""
    ref = Dataset()
    for k in ("thetao", "so", "volcello"):
        ref[k] = DataArray(np.asarray(ds[k].values)[0].copy(), ds[k].dims[1:])
    ref["rho"] = DataArray(np.full(ds["thetao"].shape[1:], 1030.0), ds["thetao"].dims[1:])
    ref["areacello"] = DataArray(np.asarray(ds["areacello"].values), ds["areacello"].dims)
    for k, v in (("volo", 2.0), ("masso", 2060.0), ("rhoga", 1030.0)):
        ref[k] = DataArray(np.float64(v), ())
    return ref


class _Recorder:
    """Stands in for core.steric_local_layers and core.steric_local_layers_variants: records what is asked."""

    def __init__(self):
        self.calls = []

    def layers(self, T, S, rho_ref, v_ref, z_i, deptho, p_level, edges, rhozero=1035.0, eos="Wright", t_bcast=False,
               s_bcast=False):
        full = S if t_bcast else T
        self.calls.append(("layers", t_bcast, s_bcast, eos))
        return torch.full((full.shape[0], len(edges) - 1) + tuple(full.shape[2:]), float(len(self.calls)),
                          dtype=torch.float64)

    def layers_variants(self, T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, edges, rhozero=1035.0,
                        eos="Wright", variants=VARIANTS):
        self.calls.append(("layers_variants", tuple(variants), tuple(np.shape(T_ref)), tuple(np.shape(S_ref)), eos))
        shape = (T.shape[0], len(edges) - 1) + tuple(T.shape[2:])
        return {v: torch.full(shape, float(VARIANTS.index(v)), dtype=torch.float64) for v in variants}


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(core, "steric_local_layers", r.layers)
    monkeypatch.setattr(core, "steric_local_layers_variants", r.layers_variants)
    monkeypatch.setattr(steric_mod, "setup_reference_state", lambda dset, **kw: _reference(dset))
    return r


# ---------------------------------------------------------------------------------------------- the variant list


@pytest.mark.parametrize("bad", [[], (), ("steric", "steric"), ["steric", "barotropic"], ("Steric",), [None]])
def test_bad_variant_lists_raise_value_error_before_any_work(monkeypatch, bad):
    def no_work(*a, **k):
        raise AssertionError("work started before the variant list was checked")

    monkeypatch.setattr(steric_mod, "validate_dataset", no_work)
    monkeypatch.setattr(steric_mod, "setup_reference_state", no_work)
    monkeypatch.setattr(core, "steric_local_layers_variants", no_work)
    with pytest.raises(ValueError):
        ml.steric_layers(_small(), variant=bad)


def test_variant_names():
    assert core.variant_names(["halosteric", "steric"]) == ("halosteric", "steric")
    assert core.variant_names("thermosteric") == ("thermosteric",)
    assert core.variant_names(VARIANTS) == VARIANTS
    for bad in ([], ["steric", "steric"], ["x"]):
        with pytest.raises(ValueError):
            core.variant_names(bad)


# ------------------------------------------------------------------------------------------ which call is made


def test_a_string_takes_one_layered_call(rec):
    res, _ = ml.steric_layers(_small(), variant="thermosteric")
    assert rec.calls == [("layers", False, True, "Wright")]
    assert set(res.variables) >= {"thermosteric", "layer_top", "layer_bottom"}


@pytest.mark.parametrize("names", [VARIANTS, ("halosteric", "steric"), ["thermosteric"]])
def test_a_list_takes_one_multi_variant_call(rec, names):
    ds = _small()
    res, ref = ml.steric_layers(ds, variant=names, depth_edges=(0, 100, None), equation_of_state="Linear")
    nz, ny, nx = ds["thetao"].shape[1:]
    assert rec.calls == [("layers_variants", tuple(names), (nz, ny, nx), (nz, ny, nx), "Linear")]
    assert [v for v in VARIANTS if v in res.variables] == [v for v in VARIANTS if v in names]
    for v in names:
        r = res[v]
        assert r.dims == ("time", "depth_layer", "yh", "xh") and r.shape == (3, 2, ny, nx)
        assert r.attrs == {"long_name": f"{v.capitalize()} height adjustment", "units": "m",
                           "depth_edges": [0.0, 100.0, float("inf")]}
        assert r.encoding["dtype"] == "float32"
        assert (np.asarray(r.values) == VARIANTS.index(v)).all()
    assert list(res["layer_top"].values) == [0.0, 100.0] and list(res["layer_bottom"].values) == [100.0, np.inf]


def test_a_supplied_reference_and_annual_means(rec):
    ds = _small(nt=24)
    days = np.tile([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], 2).astype(np.float64)
    ref = _reference(ds)
    res, ref2 = ml.steric_layers(ds, variant=["steric", "halosteric"], reference=ref, annual=True, days_in_month=days)
    assert ref2 is ref
    assert [c[0] for c in rec.calls] == ["layers_variants"]
    assert res["halosteric"].shape[0] == 2 and res["halosteric"].dims[:2] == ("time", "depth_layer")


def test_chunked_fields_still_raise(rec):
    from momlevel_b200.labeled import ChunkedArray

    ds = _small()
    for name in ("thetao", "so", "volcello"):
        full = ds[name].values

        def blocks(full=full):
            yield np.array(full[:2])
            yield np.array(full[2:])

        ds[name] = DataArray(ChunkedArray(full.shape, full.dtype, (2, full.shape[0] - 2), blocks), ds[name].dims,
                             attrs=ds[name].attrs)
    with pytest.raises(NotImplementedError):
        ml.steric_layers(ds, variant=list(VARIANTS))
    assert rec.calls == []


# --------------------------------------------------------------------------------------- ABI errors before a launch


def _call(edges, nlayers, T=16, rho_ref=16, outs=(16, 16, 16), eos=0):
    L = _lib.lib()
    e = None if edges is None else np.ascontiguousarray(edges, dtype=np.float64)
    ptr = None if e is None else e.ctypes.data_as(ctypes.c_void_p)
    rc = L.ml_steric_local_layers_variants(eos, _lib.F32, T, 16, 16, 16, rho_ref, 16, _lib.F32, 16, 16, 16, -1.0 / 1035.0,
                                           ptr, nlayers, 2, 3, 300, *outs, None)
    return rc, L.ml_last_error().decode()


@pytest.mark.parametrize("edges, nlayers", [
    ([0.0, 700.0], 0),
    ([float(i) for i in range(10)], 9),
    ([0.0, 700.0, 700.0], 2),
    ([0.0, 2000.0, 700.0], 2),
    ([-5.0, 700.0], 1),
    ([0.0, float("nan")], 1),
    ([0.0, float("inf"), 2000.0], 2),
    ([float("-inf"), 0.0], 1),
])
def test_abi_rejects_bad_layers_with_a_shape_error(edges, nlayers):
    rc, msg = _call(edges, nlayers)
    assert rc == -2, msg  # ML_ERR_SHAPE
    assert "layer" in msg


def test_abi_rejects_null_pointers_and_no_output():
    assert _call(None, 1)[0] == -1
    assert _call([0.0, float("inf")], 1, T=None)[0] == -1
    assert _call([0.0, float("inf")], 1, rho_ref=None)[0] == -1
    rc, msg = _call([0.0, float("inf")], 1, outs=(None, None, None))
    assert rc == -1 and "NULL" in msg
    assert _call([0.0, float("inf")], 1, eos=9)[0] == -4  # unknown equation of state
