"""setup_reference_state(period=...) without a device: the checks before any work, what reaches each route of
core (device-resident, host-resident, chunked), which blocks of a chunked field are read, and the reference Dataset's
variables, dims, dtypes and attrs.  The device calls are replaced by a recorder; the numbers are checked on the GPU
in tests/test_gpu_mean_reference.py."""

import importlib
import pathlib
import sys

import numpy as np
import pytest
import torch

import momlevel_b200 as ml
from momlevel_b200 import core, util
from momlevel_b200.labeled import ChunkedArray, DataArray, Dataset

reference_mod = importlib.import_module("momlevel_b200.reference")
NT, NZ, NY, NX = 10, 3, 4, 5


def _fields():
    """T[t] = t + cell / 1000, S[t] = 35 + t, V[t] = 1 + t: the steps a route sees are readable from T[:, 0, 0, 0]."""
    cell = np.arange(NZ * NY * NX, dtype=np.float64).reshape(NZ, NY, NX) / 1000.0
    t = np.arange(NT, dtype=np.float64).reshape(NT, 1, 1, 1)
    T = (t + cell).astype(np.float32)
    S = (35.0 + t + 0 * cell).astype(np.float32)
    V = (1.0 + t + 0 * cell).astype(np.float32)
    return T, S, V


def _chunked(a, chunks):
    def blocks():
        t = 0
        for n in chunks:
            yield a[t: t + n]
            t += n

    return ChunkedArray(a.shape, a.dtype, chunks, blocks)


def _dataset(T=None, S=None, V=None):
    T0, S0, V0 = _fields()
    dims = ("time", "z_l", "yh", "xh")
    ds = Dataset()
    ds["time"] = DataArray(np.arange(NT, dtype=np.float64), ("time",))
    ds["z_l"] = DataArray(np.linspace(5.0, 500.0, NZ), ("z_l",))
    ds["thetao"] = DataArray(T0 if T is None else T, dims, attrs={"units": "degC"})
    ds["so"] = DataArray(S0 if S is None else S, dims, attrs={"units": "psu"})
    ds["volcello"] = DataArray(V0 if V is None else V, dims, attrs={"units": "m3"})
    ds["areacello"] = DataArray(np.full((NY, NX), 3.6111092e14 / (NY * NX)), ("yh", "xh"))
    return ds


def _loop_mean(T, S, V, w):
    out = []
    for x in (T, S, V):
        x = np.asarray(x, dtype=np.float64)
        s = np.zeros(x.shape[1:])
        ws = np.zeros(x.shape[1:])
        for t in range(x.shape[0]):
            ok = ~np.isnan(x[t])
            s[ok] = s[ok] + w[t] * x[t][ok]
            ws[ok] = ws[ok] + w[t]
        out.append(torch.from_numpy(s / ws))
    return tuple(out)


class _Recorder:
    """Stands in for the device calls of core: records the steps, weights and dtypes each route hands over."""

    def __init__(self):
        self.calls = []

    def mean_state(self, T, S, V, weights=None):
        w = np.ones(T.shape[0]) if weights is None else weights.cpu().numpy()
        self.calls.append({"route": "device", "steps": np.asarray(T[:, 0, 0, 0], dtype=np.float64).round().astype(int),
                           "weights": None if weights is None else w.copy(), "dtypes": (T.dtype, S.dtype, V.dtype)})
        return _loop_mean(T.numpy(), S.numpy(), V.numpy(), w)

    def mean_state_blocks(self, pieces, shape, dtype, v_dtype, weights=None, max_steps=1):
        blocks = []
        for p in pieces:
            assert all(int(b.shape[0]) == int(p[0].shape[0]) for b in p) and 0 < int(p[0].shape[0]) <= max_steps
            assert all(tuple(b.shape[1:]) == tuple(shape) for b in p)
            blocks.append(tuple(np.array(b.numpy() if isinstance(b, torch.Tensor) else b, dtype=np.float64) for b in p))
        T, S, V = (np.concatenate([b[j] for b in blocks]) for j in range(3))
        w = np.ones(T.shape[0]) if weights is None else np.asarray(weights)
        self.calls.append({"route": "host", "steps": T[:, 0, 0, 0].round().astype(int), "lens": [len(b[0]) for b in blocks],
                           "weights": None if weights is None else w.copy(), "dtypes": (dtype, v_dtype)})
        return _loop_mean(T, S, V, w)

    def reference_state(self, T0, S0, V0, p_level, eos="Wright", out=None):
        self.calls.append({"route": "reference_state", "T0": np.asarray(T0.numpy() if isinstance(T0, torch.Tensor) else T0, dtype=np.float64), "eos": eos,
                           "dtype": getattr(T0, "dtype", None), "p": p_level})
        return torch.full(tuple(T0.shape), 1030.0, dtype=torch.float64), torch.tensor([2.0, 2060.0], dtype=torch.float64)


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(core, "mean_state", r.mean_state)
    monkeypatch.setattr(core, "mean_state_blocks", r.mean_state_blocks)
    monkeypatch.setattr(core, "reference_state", r.reference_state)
    monkeypatch.setattr(core, "to_device", lambda x, dtype=None: torch.as_tensor(np.asarray(x)))
    return r


def _no_work(monkeypatch):
    def no_work(*a, **k):
        raise AssertionError("work started before the arguments were checked")

    for name in ("mean_state", "mean_state_blocks", "reference_state", "to_device"):
        monkeypatch.setattr(core, name, no_work)
    monkeypatch.setattr(reference_mod, "_pressure", no_work)


# ------------------------------------------------------------------------------------------------------ validation


@pytest.mark.parametrize("kw", [
    dict(period=3), dict(period=[0, 3]), dict(period=(0, 3)), dict(period=slice(0, 6, 2)), dict(period=slice(6, 0, -1)),
    dict(period=slice(5, 5)), dict(period=slice(7, 2)), dict(period=slice(20, 30)), dict(period=slice(-3, -5)),
    dict(period=slice(0, 4), time_index=2), dict(period=slice(0, 4), time_index=-1),
    dict(period_weights=np.ones(NT)),
    dict(period=slice(0, 4), period_weights=np.ones(3)), dict(period=slice(0, 4), period_weights=np.ones(5)),
    dict(period=slice(0, 4), period_weights=np.ones((4, 1))), dict(period=slice(0, 4), period_weights=2.0),
    dict(period=slice(0, 4), period_weights=[1.0, np.nan, 1.0, 1.0]),
    dict(period=slice(0, 4), period_weights=[1.0, np.inf, 1.0, 1.0]),
    dict(period=slice(0, 4), period_weights=[1.0, -0.5, 1.0, 1.0]),
    dict(period=slice(0, 4), period_weights=[0.0, 0.0, 0.0, 0.0]),
    dict(period=slice(0, 4), period_weights=["a", "b", "c", "d"]),
], ids=lambda kw: ",".join(f"{k}={v!r}" for k, v in kw.items())[:60])
def test_bad_period_or_weights_raise_before_any_work(monkeypatch, kw):
    _no_work(monkeypatch)
    with pytest.raises(ValueError):
        reference_mod.setup_reference_state(_dataset(), **kw)


def test_period_steps_normalises_with_slice_indices():
    assert reference_mod.period_steps(slice(None), NT)[:2] == (0, NT)
    assert reference_mod.period_steps(slice(-4, None), NT)[:2] == (NT - 4, NT)
    assert reference_mod.period_steps(slice(2, 100), NT)[:2] == (2, NT)
    assert reference_mod.period_steps(slice(3, 4, 1), NT)[:2] == (3, 4)
    w = reference_mod.period_steps(slice(0, 3), NT, torch.tensor([31, 28, 31]))[2]
    assert w.dtype == np.float64 and w.tolist() == [31.0, 28.0, 31.0]


# ------------------------------------------------------------------------------------------------ period=None


def test_period_none_runs_the_one_step_code(rec):
    ref = reference_mod.setup_reference_state(_dataset(), time_index=4)
    assert [c["route"] for c in rec.calls] == ["reference_state"]
    T, _, _ = _fields()
    np.testing.assert_array_equal(rec.calls[0]["T0"], T[4].astype(np.float64))
    assert rec.calls[0]["dtype"] == np.float32  # the slab as stored, not averaged and not promoted
    assert np.asarray(ref["thetao"].values).dtype == np.float32 and "reference_period" not in ref.attrs


# ---------------------------------------------------------------------------------------------------- routes


def _check_reference(ref, start, stop, weights):
    T, S, V = _fields()
    w = np.ones(stop - start) if weights is None else np.asarray(weights, dtype=np.float64)
    want = _loop_mean(T[start:stop], S[start:stop], V[start:stop], w)
    assert set(ref.variables) >= {"thetao", "so", "volcello", "rho", "volo", "masso", "rhoga", "areacello"}
    for name, m in zip(("thetao", "so", "volcello"), want):
        assert ref[name].dims == ("z_l", "yh", "xh")
        assert np.asarray(ref[name].values).dtype == np.float64  # never rounded to the fields' fp32
        np.testing.assert_array_equal(np.asarray(ref[name].values), m.numpy())
        assert ref[name].attrs["cell_methods"] == "time: mean"
    assert ref["thetao"].attrs["units"] == "degC"
    assert ref["rho"].dims == ("z_l", "yh", "xh") and ref["rho"].attrs["units"] == "kg m-3"
    assert float(ref["volo"].values) == 2.0 and float(ref["masso"].values) == 2060.0
    assert float(ref["rhoga"].values) == 1030.0
    assert ref.attrs["reference_period"] == f"{start}:{stop}"
    assert ref.attrs["reference_period_weights"] == ("equal" if weights is None else "supplied")
    util.validate_dataset(ref, reference=True, strict=False)


@pytest.mark.parametrize("weights", [None, [31.0, 28.0, 0.0, 30.0, 31.0]])
def test_host_numpy_route(rec, weights):
    ref = reference_mod.setup_reference_state(_dataset(), period=slice(2, 7), period_weights=weights)
    host = [c for c in rec.calls if c["route"] == "host"]
    assert len(host) == 1 and [c["route"] for c in rec.calls].count("device") == 0
    assert host[0]["steps"].tolist() == [2, 3, 4, 5, 6]
    assert host[0]["dtypes"] == (torch.float32, torch.float32)
    if weights is None:
        assert host[0]["weights"] is None
    else:
        np.testing.assert_array_equal(host[0]["weights"], weights)
    # the reference state is evaluated on the fp64 means
    rs = [c for c in rec.calls if c["route"] == "reference_state"]
    assert len(rs) == 1 and rs[0]["dtype"] == torch.float64
    _check_reference(ref, 2, 7, weights)


def test_host_cpu_tensor_route_and_mixed_dtypes(rec):
    T, S, V = _fields()
    ds = _dataset(torch.from_numpy(T), torch.from_numpy(S.astype(np.float64)), torch.from_numpy(V.astype(np.float64)))
    ref = reference_mod.setup_reference_state(ds, period=slice(-3, None))
    host = [c for c in rec.calls if c["route"] == "host"]
    assert host[0]["steps"].tolist() == [7, 8, 9]
    assert host[0]["dtypes"] == (torch.float64, torch.float64)  # T and S share a dtype; V keeps its own
    _check_reference(ref, 7, 10, None)


def test_host_blocks_are_capped(rec, monkeypatch):
    step = NZ * NY * NX * 4
    monkeypatch.setattr(reference_mod, "PERIOD_BLOCK_BYTES", 2 * step)
    reference_mod.setup_reference_state(_dataset(), period=slice(1, 8))
    host = [c for c in rec.calls if c["route"] == "host"][0]
    assert host["lens"] == [2, 2, 2, 1] and host["steps"].tolist() == list(range(1, 8))


@pytest.mark.parametrize("period, read", [(slice(1, 6), (3, 2, 4)), (slice(0, 1), (1, 1, 1)), (slice(8, 10), (4, 4, 5)),
                                          (slice(5, 7), (3, 3, 5))])
def test_chunked_route_reads_no_block_past_the_period(rec, period, read):
    T, S, V = _fields()
    cT, cS, cV = _chunked(T, (1, 4, 2, 3)), _chunked(S, (3, 3, 3, 1)), _chunked(V, (2, 1, 1, 2, 4))
    ref = reference_mod.setup_reference_state(_dataset(cT, cS, cV), period=period, period_weights=np.arange(1.0, 1.0 + period.stop - period.start))
    host = [c for c in rec.calls if c["route"] == "host"]
    assert len(host) == 1
    assert host[0]["steps"].tolist() == list(range(period.start, period.stop))
    np.testing.assert_array_equal(host[0]["weights"], np.arange(1.0, 1.0 + period.stop - period.start))
    # the blocks up to the one holding the period's last step are produced, none after it
    assert (cT.blocks_read, cS.blocks_read, cV.blocks_read) == read
    _check_reference(ref, period.start, period.stop, np.arange(1.0, 1.0 + period.stop - period.start))


def test_chunked_pieces_follow_every_boundary(rec):
    T, S, V = _fields()
    ds = _dataset(_chunked(T, (1, 4, 2, 3)), _chunked(S, (3, 3, 3, 1)), V)
    reference_mod.setup_reference_state(ds, period=slice(0, NT))
    host = [c for c in rec.calls if c["route"] == "host"][0]
    # boundaries of T at 1, 5, 7 and of S at 3, 6, 9: pieces are cut at their union
    assert host["lens"] == [1, 2, 2, 1, 1, 2, 1]


@pytest.mark.parametrize("weights", [None, [1.0, 2.0, 3.0]])
def test_device_route(rec, monkeypatch, weights):
    monkeypatch.setattr(reference_mod, "_device_resident", lambda data: True)
    ref = reference_mod.setup_reference_state(_dataset(), period=slice(4, 7), period_weights=weights)
    dev = [c for c in rec.calls if c["route"] == "device"]
    assert len(dev) == 1 and not [c for c in rec.calls if c["route"] == "host"]
    assert dev[0]["steps"].tolist() == [4, 5, 6]
    assert (dev[0]["weights"] is None) == (weights is None)
    if weights is not None:
        np.testing.assert_array_equal(dev[0]["weights"], weights)
    _check_reference(ref, 4, 7, weights)


def test_device_route_is_chosen_only_without_chunked_fields():
    T, S, V = _fields()
    assert not reference_mod._device_resident([T, S, V])
    assert not reference_mod._device_resident([torch.from_numpy(T), S, V])


def test_fields_must_lead_with_time(rec):
    ds = _dataset()
    ds["volcello"] = DataArray(_fields()[2][0], ("z_l", "yh", "xh"))
    with pytest.raises(ValueError, match="volcello"):
        reference_mod.setup_reference_state(ds, period=slice(0, 3))


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


def test_xarray_in_xarray_out(rec, xr):
    lab = _dataset()
    ds = xr.Dataset(attrs={"title": "control"})
    for name, var in lab.variables.items():
        ds[name] = xr.DataArray(np.asarray(var.values), dims=var.dims, attrs=dict(var.attrs))
    ref = reference_mod.setup_reference_state(ds, period=slice(0, 5), period_weights=[1.0, 2.0, 3.0, 4.0, 5.0])
    assert type(ref).__module__.startswith("xarray")
    assert ref.attrs["reference_period"] == "0:5" and ref.attrs["reference_period_weights"] == "supplied"
    assert ref["thetao"].dims == ("z_l", "yh", "xh") and np.asarray(ref["thetao"].values).dtype == np.float64
    want = _loop_mean(*(f[0:5] for f in _fields()), np.arange(1.0, 6.0))
    np.testing.assert_array_equal(np.asarray(ref["so"].values), want[1].numpy())
    assert [c["route"] for c in rec.calls] == ["host", "reference_state"]
