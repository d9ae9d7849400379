"""steric_variants(domain="global") and ml_steric_global_variants: the global steric, thermosteric and halosteric
series from one pass over T and S, against the oracle, against three single-height calls (bit for bit), and across
the routes (device-resident, host-resident, chunked)."""

import importlib
import importlib.util
import pathlib
import sys

import numpy as np
import pytest
import torch

from oracle import steric as osteric
from oracle import testdata

pytestmark = pytest.mark.gpu

VARIANTS = ("steric", "thermosteric", "halosteric")
ETA_ATOL = 1e-9  # m
REFERENCE_RESULTS = {  # tests/test_steric.py:32-41
    "reference_thetao": 1921.05772939,
    "reference_so": 4388.81731882,
    "reference_vol": 125921.15458782,
    "reference_rho": 128781.63975736,
    "global_reference_vol": 125921.15458782,
    "global_reference_rho": 1030.2309221,
}


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


def _check_reference(reference):
    rs = reference.sum()
    assert float(rs["thetao"]) == pytest.approx(REFERENCE_RESULTS["reference_thetao"], abs=5e-9)
    assert float(rs["so"]) == pytest.approx(REFERENCE_RESULTS["reference_so"], abs=5e-9)
    assert float(rs["volcello"]) == pytest.approx(REFERENCE_RESULTS["reference_vol"], abs=5e-9)
    assert float(rs["rho"]) == pytest.approx(REFERENCE_RESULTS["reference_rho"], abs=5e-9)
    assert float(rs["volo"]) == pytest.approx(REFERENCE_RESULTS["global_reference_vol"], abs=5e-9)
    assert float(rs["rhoga"]) == pytest.approx(REFERENCE_RESULTS["global_reference_rho"], abs=5e-8)


def _series(res):
    return {v: np.asarray(res[v].values) for v in VARIANTS}


# ------------------------------------------------------------------------------------ config 1 against the oracle


def test_config1_against_the_oracle(ml):
    ds = ml.test_data.generate_test_data()
    res, ref = ml.steric_variants(ds, domain="global")
    _check_reference(ref)
    assert set(ref.variables) >= {"thetao", "so", "volcello", "rho", "volo", "masso", "rhoga", "areacello"}
    o = testdata.generate_test_data()
    oref = osteric.reference_state(o["thetao"], o["so"], o["volcello"], o["areacello"], o["z_l"])
    href = float(res["reference_height"])
    assert res["reference_height"].attrs == {"long_name": "Reference column height", "units": "m"}
    stale = {"steric": 6.29048941e-14, "thermosteric": -1.38053154e-13, "halosteric": 1.98293992e-13}
    for v in VARIANTS:
        eta, o_href, _ = osteric.steric_global(o["thetao"], o["so"], o["z_l"], oref, variant=v)
        assert href == pytest.approx(o_href, rel=1e-13)
        assert res[v].dims == ("time",)
        assert res[v].attrs == {"long_name": f"{v.capitalize()} height adjustment", "units": "m"}
        assert res[v].encoding["dtype"] == "float32"
        assert np.allclose(np.exp(res[v].values / href), np.exp(eta / o_href), rtol=1e-13, atol=0)  # the log argument
        assert np.allclose(res[v].values, eta, rtol=0, atol=ETA_ATOL)
        assert np.allclose(float(res.sum()[v]), stale[v])  # the reference's vacuous checks (tests/test_steric.py:80-125)
    assert np.allclose(href, 3.4726688e-10)


# ------------------------------------------------------------------ masses: bit-identical to three single launches


def _fields(nt, nz, ny, nx, dtype=torch.float32, seed=11, holes=True):
    from momlevel_b200 import synth

    grid = synth.make_grid(nz, ny, nx, seed=seed, device="cpu")
    T, S, V = synth.make_fields(grid, nt, seed=seed, dtype=dtype)
    T, S, V = T.cuda().contiguous(), S.cuda().contiguous(), V.cuda().contiguous()
    if holes:
        wet = torch.nonzero(~torch.isnan(V))
        z, y, x = (int(i) for i in wet[len(wet) // 2])
        T[nt // 2, z, y, x] = float("nan")  # a hole at a wet cell of one step: the repair pass
        land = torch.nonzero(torch.isnan(T[0]))
        if len(land):
            z, y, x = (int(i) for i in land[len(land) // 3])
            V[z, y, x] = 1.0e9  # a volume where the fields are missing
        z, y, x = (int(i) for i in wet[len(wet) // 4])
        V[z, y, x] = float("nan")  # and none where they are present
    pres = (grid["z_l"] * 1.0e4 + 101325.0).numpy()
    return T, S, V, pres


def _three_launches(core, T, S, V, pres, Tr, Sr, eos="Wright"):
    return {"steric": core.steric_global(T, S, V, pres, eos=eos),
            "thermosteric": core.steric_global(T, Sr, V, pres, eos=eos, s_bcast=True),
            "halosteric": core.steric_global(Tr, S, V, pres, eos=eos, t_bcast=True)}


@pytest.mark.parametrize("nt", [1, 4, 5, 12, 13, 25])
@pytest.mark.parametrize("hw", [(16, 64), (12, 100)])
def test_one_pass_masses_are_bit_identical_to_three_launches(ml, nt, hw):
    from momlevel_b200 import core

    T, S, V, pres = _fields(nt, 10, *hw)
    for selfref in (True, False):
        Tr, Sr = (T[0], S[0]) if selfref else (T[-1].clone(), S[-1].clone())
        before = core.launch_count()
        got, sums = core.steric_global_variants(T, S, V, pres, T_ref=None if selfref else Tr, S_ref=None if selfref else Sr)
        launches = core.launch_count() - before
        assert core.last_path() == 2  # ML_PATH_TMA: the one-pass kernel
        want = _three_launches(core, T, S, V, pres, Tr, Sr)
        for v in VARIANTS:
            assert torch.equal(got[v], want[v]), v
            assert torch.isfinite(got[v]).all()
        if selfref:
            rho_w, sums_w = core.reference_state(T[0], S[0], V, pres)
            assert torch.allclose(sums, sums_w, rtol=1e-13, atol=0)
        else:
            assert sums is None
        # the one-pass kernel is what ran: with it turned off the same call takes more launches, same bits
        prev = core.force_direct(2)
        try:
            before = core.launch_count()
            again, sums2 = core.steric_global_variants(T, S, V, pres, T_ref=None if selfref else Tr, S_ref=None if selfref else Sr)
            assert core.launch_count() - before > launches
        finally:
            core.force_direct(prev)
        for v in VARIANTS:
            assert torch.equal(again[v], want[v])
    # a subset of the variants
    got, _ = core.steric_global_variants(T, S, V, pres, variants=("steric", "halosteric"))
    want = _three_launches(core, T, S, V, pres, T[0], S[0])
    assert set(got) == {"steric", "halosteric"}
    assert torch.equal(got["steric"], want["steric"]) and torch.equal(got["halosteric"], want["halosteric"])


@pytest.mark.parametrize("case", ["fp64", "ncol_not_multiple_of_4", "ncol_below_256"])
def test_fallback_shapes_match_three_launches(ml, case):
    from momlevel_b200 import core

    shape = {"fp64": (7, 6, 16, 32), "ncol_not_multiple_of_4": (7, 6, 17, 31), "ncol_below_256": (7, 6, 8, 16)}[case]
    T, S, V, pres = _fields(*shape, dtype=torch.float64 if case == "fp64" else torch.float32)
    before = core.launch_count()
    got, sums = core.steric_global_variants(T, S, V, pres)
    launches = core.launch_count() - before
    path = core.last_path()
    assert path == (1 if case == "ncol_below_256" else 2)  # what the last single-height launch took
    prev = core.force_direct(2)
    try:
        before = core.launch_count()
        core.steric_global_variants(T, S, V, pres)
        assert core.launch_count() - before == launches  # the one-pass kernel did not take these shapes
    finally:
        core.force_direct(prev)
    want = _three_launches(core, T, S, V, pres, T[0], S[0])
    for v in VARIANTS:
        assert torch.equal(got[v], want[v]), v
    _, sums_w = core.reference_state(T[0], S[0], V, pres)
    assert torch.allclose(sums, sums_w, rtol=1e-13, atol=0)


# ---------------------------------------------------------------- equation of state, supplied reference, 2-D patm


def _close_series(a, b, href):
    for v in VARIANTS:
        assert np.allclose(np.exp(a[v] / href), np.exp(b[v] / href), rtol=1e-13, atol=0), v


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_equations_of_state_match_steric(ml, eos):
    from momlevel_b200 import synth

    ds = synth.make_dataset(6, 8, 16, 64, seed=4, device="cuda", dtype=torch.float32)
    res, ref = ml.steric_variants(ds, domain="global", equation_of_state=eos)
    href = float(res["reference_height"])
    want = {}
    for v in VARIANTS:
        r, wref = ml.steric(ds, domain="global", variant=v, equation_of_state=eos)
        want[v] = np.asarray(r[v].values)
        assert float(r["reference_height"]) == pytest.approx(href, rel=1e-13)
    assert float(ref["volo"]) == pytest.approx(float(wref["volo"]), rel=1e-13)
    _close_series(_series(res), want, href)


def test_supplied_reference(ml):
    # tests/test_steric.py:128-137: the reference state of another dataset (seed 999)
    dset = ml.test_data.generate_test_data()
    _, reference = ml.steric(ml.test_data.generate_test_data(seed=999))
    res, ref = ml.steric_variants(dset, domain="global", reference=reference)
    assert ref is reference
    for v in VARIANTS:
        want, _ = ml.steric(dset, domain="global", variant=v, reference=reference)
        assert np.array_equal(res[v].values, want[v].values)
    assert float(res["reference_height"]) == float(want["reference_height"])


def test_two_dimensional_patm_matches_steric(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(5, 8, 16, 64, seed=6, device="cuda", dtype=torch.float32)
    patm = 101325.0 + 500.0 * torch.rand((16, 64), generator=torch.Generator().manual_seed(2), dtype=torch.float64).numpy()
    res, _ = ml.steric_variants(ds, domain="global", patm=patm)
    href = float(res["reference_height"])
    want = {v: np.asarray(ml.steric(ds, domain="global", variant=v, patm=patm)[0][v].values) for v in VARIANTS}
    _close_series(_series(res), want, href)
    flat, _ = ml.steric_variants(ds, domain="global")
    assert not np.array_equal(flat["steric"].values, res["steric"].values)


# ------------------------------------------------------------------------------------------- the routes agree


def _chunked_dataset(ds, chunks):
    from momlevel_b200.labeled import ChunkedArray, DataArray

    out = ds.copy()
    made = {}
    for name in ("thetao", "so", "volcello"):
        full = ds[name].values
        cuts = np.cumsum((0,) + tuple(chunks))

        def blocks(full=full, cuts=cuts):
            for a, b in zip(cuts[:-1], cuts[1:]):
                yield np.array(full[a:b])

        made[name] = ChunkedArray(full.shape, full.dtype, chunks, blocks)
        out[name] = DataArray(made[name], ds[name].dims, attrs=ds[name].attrs)
    return out, made


def _moved(ds, fn):
    from momlevel_b200.labeled import DataArray

    out = ds.copy()
    for name in ds.variables:
        d = ds[name].data
        if isinstance(d, torch.Tensor):
            out[name] = DataArray(fn(d), ds[name].dims, attrs=ds[name].attrs)
    return out


def test_routes_agree_bit_for_bit(ml, monkeypatch):
    from momlevel_b200 import synth

    steric_mod = importlib.import_module("momlevel_b200.steric")
    ds = synth.make_dataset(13, 10, 16, 64, seed=9, device="cpu", dtype=torch.float32)
    dev = _moved(ds, lambda t: t.cuda())
    host = _moved(ds, lambda t: t.numpy())
    chunks = (5, 1, 7)
    cds, made = _chunked_dataset(ds, chunks)
    monkeypatch.setattr(steric_mod, "HOST_ROUTE_MIN_BYTES", 0)
    assert steric_mod._variants_route(host, np.zeros(10), "time", "z_l", "z_i", "global") == "host"
    got = {}
    for name, d in (("device", dev), ("host", host), ("chunked", cds)):
        res, ref = ml.steric_variants(d, domain="global")
        got[name] = (_series(res), float(res["reference_height"]), float(ref["volo"]), float(ref["masso"]))
    assert made["thetao"].blocks_read == len(chunks) and made["so"].blocks_read == len(chunks)
    for name in ("host", "chunked"):
        for v in VARIANTS:
            assert np.array_equal(got[name][0][v], got["device"][0][v]), (name, v)
        assert got[name][1:] == got["device"][1:]
    # and against three single-height calls, to rounding of the reference scalars
    for v in VARIANTS:
        want, _ = ml.steric(dev, domain="global", variant=v)
        assert np.allclose(np.exp(got["device"][0][v] / got["device"][1]),
                           np.exp(np.asarray(want[v].values) / float(want["reference_height"])), rtol=1e-13, atol=0)
    # the local domain on chunked fields: one pass over the blocks, the device-resident heights
    cds, made = _chunked_dataset(ds, chunks)
    loc_c, _ = ml.steric_variants(cds)
    loc_d, _ = ml.steric_variants(dev)
    assert made["thetao"].blocks_read == len(chunks)
    for v in VARIANTS:
        assert np.array_equal(np.asarray(loc_c[v].values), np.asarray(loc_d[v].values), equal_nan=True), v


# ------------------------------------------------------------------------------------------ annual, xarray, ABI


@pytest.mark.parametrize("domain", ["local", "global"])
def test_annual_is_the_annual_average_of_the_monthly_series(ml, domain):
    from momlevel_b200.util import annual_average

    d3 = ml.test_data.generate_test_data(start_year=1983, nyears=2, calendar="julian")
    res, _ = ml.steric_variants(d3, domain=domain, annual=True)
    monthly, _ = ml.steric_variants(d3, domain=domain)
    want = annual_average(monthly, tcoord="time")
    assert len(res["time"]) == 2
    for v in VARIANTS:
        assert np.array_equal(np.asarray(res[v].values), np.asarray(want[v].values), equal_nan=True)
        assert res[v].shape[0] == 2
    if domain == "global":
        single, _ = ml.steric(d3, domain="global", annual=True)
        assert np.allclose(res["steric"].values, single["steric"].values, rtol=0, atol=ETA_ATOL)


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
    result, reference = ml.steric_variants(ds, domain="global")
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    want, wref = ml.steric_variants(lab, domain="global")
    for v in VARIANTS:
        assert result[v].dims == ("time",)
        assert np.array_equal(np.asarray(result[v].values), np.asarray(want[v].values))
        assert result[v].attrs == {"long_name": f"{v.capitalize()} height adjustment", "units": "m"}
    assert float(np.asarray(result["reference_height"].values)) == float(want["reference_height"])
    for name in ("thetao", "so", "volcello", "rho", "volo", "masso", "rhoga", "areacello"):
        assert name in reference.variables
    again, _ = ml.steric_variants(ds, domain="global", reference=reference)
    assert np.array_equal(np.asarray(again["steric"].values), np.asarray(want["steric"].values))


def test_abi_errors(ml):
    from momlevel_b200 import _lib

    L = _lib.lib()
    nt, nz, ncol = 3, 4, 256
    T = torch.zeros((nt, nz, ncol), dtype=torch.float32, device="cuda")
    S = torch.zeros_like(T)
    V = torch.ones((nz, ncol), dtype=torch.float32, device="cuda")
    p = torch.zeros(nz, dtype=torch.float64, device="cuda")
    out = torch.empty((3, nt), dtype=torch.float64, device="cuda")
    sums = torch.empty(2, dtype=torch.float64, device="cuda")
    need = L.ml_workspace_bytes(3 * nt, nz, ncol)
    ws = torch.empty(need // 8 + 1, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def call(outs, sums_ptr, nbytes, Tr=T, Sr=S):
        return L.ml_steric_global_variants(0, 0, T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), V.data_ptr(), 0,
                                           p.data_ptr(), nt, nz, ncol, *outs, sums_ptr, ws.data_ptr(), nbytes, stream)

    ptrs = [out[i].data_ptr() for i in range(3)]
    assert call([None, None, None], sums.data_ptr(), need) == -1  # no output
    assert b"output" in L.ml_last_error()
    assert call(ptrs, None, need) == -1  # a self-reference without sums
    assert call(ptrs, sums.data_ptr(), need - 1) == -6  # workspace one byte short
    assert call(ptrs, sums.data_ptr(), need) == 0
    torch.cuda.synchronize()
    assert torch.isfinite(out).all()
