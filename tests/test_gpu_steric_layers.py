"""steric_layers() and ml_steric_local_layers: the local height by depth layer from one pass over T and S, against
the numpy reference (tests/layers_oracle.py), bit for bit against ml_steric_local for the single layer (0, None),
across both kernel families, with holes, a 2-D patm, annual means and the xarray adapter."""

import importlib.util
import pathlib
import sys

import numpy as np
import pytest
import torch

import layers_oracle  # tests/layers_oracle.py
from oracle import steric as osteric
from oracle import testdata

pytestmark = pytest.mark.gpu

VARIANTS = ("steric", "thermosteric", "halosteric")
ETA_ATOL = 1e-9  # m


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


def _edge_sets(z_i):
    """Edge sets on synth.vertical_grid(75): 700 m and 2000 m fall inside levels 36 and 51."""
    assert z_i[36] < 700.0 < z_i[37] and z_i[51] < 2000.0 < z_i[52]
    e_if = float(z_i[20])   # an edge on an interface
    third = (float(z_i[37]) - 700.0) / 3.0
    return [
        (0.0, 700.0, 2000.0, None),
        (0.0, e_if, 700.0, 700.0 + third, 700.0 + 2 * third, 2000.0, None),  # level 36 feeds four layers, two inside it
        (e_if, 2000.0, 6000.0, 6400.0),                          # starts below the surface; the last layers lie below
        (0.0, 700.0, 2000.0, 6000.0, None),                      # most floors: 0.0 there
    ]


def _fields(nt, ny, nx, dtype=torch.float32, seed=7, hole=False):
    from momlevel_b200 import synth

    grid = synth.make_grid(75, ny, nx, seed=seed, device="cpu")
    T, S, V = synth.make_fields(grid, nt, seed=seed, dtype=dtype)
    if hole:  # a missing value at a wet cell of one step: the repair pass
        wet = torch.nonzero(~torch.isnan(V))
        z, y, x = (int(i) for i in wet[len(wet) // 2])
        T[nt // 2, z, y, x] = float("nan")
        z, y, x = (int(i) for i in wet[len(wet) // 5])
        S[nt - 1, z, y, x] = float("nan")
    return grid, T, S, V


def _oracle(grid, T, S, V, edges, variant, eos="Wright", patm=101325.0):
    f = lambda t: t.double().cpu().numpy()  # noqa: E731
    z_l, z_i, depth, area = (f(grid[k]) for k in ("z_l", "z_i", "deptho", "areacello"))
    Tn, Sn = f(T), f(S)
    ref = osteric.reference_state(Tn, Sn, f(V)[None].repeat(Tn.shape[0], 0), area, z_l, patm=patm, eos=eos)
    return layers_oracle.steric_local_layers(Tn, Sn, z_l, z_i, depth, ref, edges, patm=patm, eos=eos, variant=variant)


def _device_call(core, grid, T, S, V, edges, variant, eos="Wright"):
    """reference state from step 0 on the device, then one layered call; returns eta [nt, nl, ny, nx] (numpy)."""
    Td, Sd, Vd = T.cuda(), S.cuda(), V.cuda()
    pres = (grid["z_l"] * 1.0e4 + 101325.0).cuda()
    rho, _ = core.reference_state(Td[0], Sd[0], Vd, pres, eos=eos)
    Tx, Sx, tb, sb = Td, Sd, False, False
    if variant == "thermosteric":
        Sx, sb = Sd[0].clone(), True
    elif variant == "halosteric":
        Tx, tb = Td[0].clone(), True
    args = (Tx, Sx, rho, Vd, grid["z_i"], grid["deptho"], pres)
    return args, dict(eos=eos, t_bcast=tb, s_bcast=sb)


def _close(got, want, atol=ETA_ATOL):
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want))
    m = ~np.isnan(want)
    assert float(np.max(np.abs(got[m] - want[m]), initial=0.0)) <= atol


# --------------------------------------------------------------------------------------------------- oracle parity


@pytest.mark.parametrize("family", ["tma", "direct"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
@pytest.mark.parametrize("variant", VARIANTS)
def test_oracle_parity(ml, family, dtype, eos, variant):
    core = ml.core
    cases = [(13, 12, 100), (5, 13, 101), (25, 16, 64)]  # aligned rows, ragged rows (rank-1 maps), a 12-step chunk + 1
    if dtype == torch.float32:
        cases.append((12, 13, 101))
    for nt, ny, nx in cases:
        grid, T, S, V = _fields(nt, ny, nx, dtype)
        args, kw = _device_call(core, grid, T, S, V, None, variant, eos)
        for edges in _edge_sets(grid["z_i"].numpy()):
            prev = core.force_direct(1 if family == "direct" else 0)
            try:
                got = core.steric_local_layers(*args, edges, **kw)
                path = core.last_path()
            finally:
                core.force_direct(prev)
            assert path == (1 if family == "direct" else 2)
            assert got.shape == (nt, len(edges) - 1, ny, nx)
            _close(got.cpu().numpy(), _oracle(grid, T, S, V, edges, variant, eos))


def test_layers_below_the_floor_are_zero_and_dry_columns_nan(ml):
    core = ml.core
    grid, T, S, V = _fields(5, 12, 100)
    args, kw = _device_call(core, grid, T, S, V, None, "steric")
    got = core.steric_local_layers(*args, (0.0, 700.0, 2000.0, 6000.0, None), **kw).cpu().numpy()
    depth = grid["deptho"].numpy()
    land = np.isnan(depth)
    assert land.any() and np.isnan(got[:, :, land]).all()
    z_i = grid["z_i"].numpy()
    shallow = ~land & (depth <= z_i[51])  # the floor lies above the cell that holds 2000 m (calc_dz: see the quirk)
    assert shallow.any()
    assert (got[:, 2:, shallow] == 0.0).all()  # nansum of zero terms
    assert np.isfinite(got[:, :, ~land]).all()


@pytest.mark.parametrize("nt", [1, 5, 12, 13, 25])
def test_oracle_test_data_config1(ml, nt):
    """The reference's 5x5x5 test dataset (direct family: fewer than 256 columns), steps repeated to nt."""
    o = testdata.generate_test_data()
    reps = -(-nt // o["thetao"].shape[0])
    T = np.concatenate([o["thetao"]] * reps)[:nt]
    S = np.concatenate([o["so"]] * reps)[:nt]
    ref = osteric.reference_state(o["thetao"], o["so"], o["volcello"], o["areacello"], o["z_l"])
    for edges in [(0.0, 15.0, 100.0, None), (0.0, 10.0, 1000.0, 5000.0, None), (0.0, None)]:
        for variant in VARIANTS:
            want = layers_oracle.steric_local_layers(T, S, o["z_l"], o["z_i"], o["deptho"], ref, edges, variant=variant)
            tb, sb = variant == "halosteric", variant == "thermosteric"
            got = ml.core.steric_local_layers(ref["thetao"] if tb else T, ref["so"] if sb else S, ref["rho"],
                                              ref["volcello"], o["z_i"], o["deptho"], o["z_l"] * 1.0e4 + 101325.0,
                                              edges, t_bcast=tb, s_bcast=sb)
            _close(got.cpu().numpy(), want)


# ------------------------------------------------------------------------- (0, None) is ml_steric_local bit for bit


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("family", ["tma", "direct"])
def test_single_layer_is_bit_identical_to_steric_local(ml, family, dtype):
    core = ml.core
    for ny, nx in ((12, 100), (13, 101)):
        grid, T, S, V = _fields(13, ny, nx, dtype, hole=True)
        for variant in VARIANTS:
            args, kw = _device_call(core, grid, T, S, V, None, variant)
            prev = core.force_direct(1 if family == "direct" else 0)
            try:
                got = core.steric_local_layers(*args, (0.0, None), **kw)
                p1 = core.last_path()
                want, _ = core.steric_local(*args, **kw)
                p2 = core.last_path()
            finally:
                core.force_direct(prev)
            assert p1 == p2 == (1 if family == "direct" else 2)
            assert torch.equal(got[:, 0].contiguous().view(torch.int64), want.view(torch.int64)), variant


@pytest.mark.parametrize("variant", VARIANTS)
def test_public_single_layer_equals_steric(ml, variant):
    from momlevel_b200 import synth

    ds = synth.make_dataset(13, 75, 12, 100, seed=3, device="cuda")
    _, ref = ml.steric(ds, variant=variant)
    res, _ = ml.steric(ds, variant=variant, reference=ref)
    lay, ref2 = ml.steric_layers(ds, depth_edges=(0, None), reference=ref, variant=variant)
    assert ref2 is ref
    assert lay[variant].dims == ("time", "depth_layer", "yh", "xh")
    assert torch.equal(lay[variant].data[:, 0].contiguous().view(torch.int64), res[variant].data.contiguous().view(torch.int64))


# -------------------------------------------------------------------------------------------- partition and holes


def test_layers_partition_the_column(ml):
    core = ml.core
    grid, T, S, V = _fields(13, 12, 100)
    z_i = grid["z_i"].numpy()
    args, kw = _device_call(core, grid, T, S, V, None, "steric")
    # no layer starts and ends inside one cell: calc_dz gives such a layer min(bottom - z_i[k], z_i[k+1] - top), not
    # bottom - top (the oracle parity above covers that case)
    edges = (0.0, float(z_i[20]), 700.0, 2000.0, 6000.0, None)
    lay = core.steric_local_layers(*args, edges, **kw).cpu().numpy()
    full, _ = core.steric_local(*args, **kw)
    full = full.cpu().numpy()
    depth = np.nan_to_num(grid["deptho"].numpy(), nan=0.0)
    quirk = np.zeros(depth.shape, dtype=bool)
    for e in edges[1:-1]:
        k = int(np.searchsorted(z_i, e, side="right")) - 1
        if z_i[k] != e:  # an edge inside cell k: a floor inside that cell counts on both sides (calc_dz)
            quirk |= (depth > z_i[k]) & (depth < z_i[k + 1])
    assert quirk.any()
    ok = ~np.isnan(full) & ~quirk[None]
    np.testing.assert_allclose(lay.sum(axis=1)[ok], full[ok], rtol=0, atol=1e-12)
    q = np.broadcast_to(quirk[None, None], lay.shape)
    _close(lay[q].reshape(-1), _oracle(grid, T, S, V, edges, "steric")[q].reshape(-1))


@pytest.mark.parametrize("family", ["tma", "direct"])
def test_holes_at_wet_cells_are_skipped_in_every_layer(ml, family):
    core = ml.core
    for nt, ny, nx in ((13, 12, 100), (5, 13, 101)):
        grid, T, S, V = _fields(nt, ny, nx, hole=True)
        args, kw = _device_call(core, grid, T, S, V, None, "steric")
        for edges in _edge_sets(grid["z_i"].numpy()):
            prev = core.force_direct(1 if family == "direct" else 0)
            try:
                got = core.steric_local_layers(*args, edges, **kw).cpu().numpy()
            finally:
                core.force_direct(prev)
            want = _oracle(grid, T, S, V, edges, "steric")
            _close(got, want)
            # the poisoned columns are finite in every layer: nothing stale or NaN is left from the first sweep
            depth = grid["deptho"].numpy()
            assert np.isfinite(got[:, :, ~np.isnan(depth)]).all()


# ------------------------------------------------------------------------------------------------ the public call


def test_public_call_with_a_2d_patm(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(5, 75, 12, 100, seed=4, device="cuda")
    patm = 101325.0 + 500.0 * torch.rand((12, 100), dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    res, _ = ml.steric_layers(ds, patm=patm.numpy())
    assert ml.core.last_path() == 1  # a column pressure takes the direct family
    grid = {k: ds[k].data.cpu() for k in ("z_l", "z_i", "deptho", "areacello")}
    want = _oracle(grid, ds["thetao"].data, ds["so"].data, ds["volcello"].data[0], (0.0, 700.0, 2000.0, None),
                   "steric", patm=patm.numpy())
    _close(res["steric"].values, want)


def test_public_call_result_and_supplied_reference(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(13, 75, 13, 101, seed=6, device="cuda")
    res, ref = ml.steric_layers(ds, variant="thermosteric", depth_edges=(0, 700, 2000, None))
    assert set(res.variables) >= {"thermosteric", "layer_top", "layer_bottom"} and "delta_rho" not in res.variables
    v = res["thermosteric"]
    assert v.dims == ("time", "depth_layer", "yh", "xh") and v.shape == (13, 3, 13, 101)
    assert v.attrs["long_name"] == "Thermosteric height adjustment" and v.attrs["units"] == "m"
    assert v.attrs["depth_edges"] == [0.0, 700.0, 2000.0, float("inf")]
    assert v.encoding["dtype"] == "float32"
    assert list(res["layer_top"].values) == [0.0, 700.0, 2000.0]
    assert list(res["layer_bottom"].values) == [700.0, 2000.0, np.inf]
    assert np.array_equal(np.asarray(res["time"].values), np.asarray(ds["time"].values))
    again, ref2 = ml.steric_layers(ds, variant="thermosteric", reference=ref)
    assert ref2 is ref
    assert torch.equal(again["thermosteric"].data.view(torch.int64), v.data.view(torch.int64))
    # host-resident (numpy) fields go to the device and give the same heights
    host = ds.copy()
    for k in ("thetao", "so", "volcello", "deptho", "areacello", "z_l", "z_i"):
        host[k] = ml.DataArray(ds[k].data.cpu().numpy(), ds[k].dims, attrs=ds[k].attrs)
    h, _ = ml.steric_layers(host, variant="thermosteric")
    assert np.array_equal(h["thermosteric"].values, v.values, equal_nan=True)


def test_public_call_annual_means(ml):
    from momlevel_b200 import synth
    from momlevel_b200.util import annual_average

    ds = synth.make_dataset(24, 75, 12, 100, seed=8, device="cuda")
    days = np.tile([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], 2).astype(np.float64)
    monthly, _ = ml.steric_layers(ds, variant="halosteric")
    annual, _ = ml.steric_layers(ds, variant="halosteric", annual=True, days_in_month=days)
    want = annual_average(monthly, days_in_month=days)
    assert annual["halosteric"].dims == ("time", "depth_layer", "yh", "xh") and annual["halosteric"].shape[0] == 2
    assert np.array_equal(annual["halosteric"].values, want["halosteric"].values, equal_nan=True)
    assert list(annual["layer_bottom"].values) == [700.0, 2000.0, np.inf]


def test_public_call_errors(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(3, 75, 12, 100, seed=9, device="cuda")
    for bad in ((0.0, 700.0, 700.0), (0.0, float("nan")), (0.0, float("inf"), 9.0), (-1.0, None), (0.0,),
                tuple(float(i) for i in range(10))):
        with pytest.raises(ValueError):
            ml.steric_layers(ds, depth_edges=bad)
    with pytest.raises(ValueError):
        ml.steric_layers(ds, variant="barotropic")


def test_abi_errors_with_device_operands(ml):
    import ctypes

    from momlevel_b200 import _lib

    core, L = ml.core, _lib.lib()
    grid, T, S, V = _fields(2, 12, 100)
    (Td, Sd, rho, Vd, z_i, depth, pres), _ = _device_call(core, grid, T, S, V, None, "steric")
    z_i, depth = z_i.cuda(), depth.cuda()
    eta = torch.empty((2, 8, 1200), dtype=torch.float64, device="cuda")

    def call(edges, nl, v_ref=Vd.data_ptr(), out=eta.data_ptr()):
        e = np.asarray(edges, dtype=np.float64)
        return L.ml_steric_local_layers(0, _lib.F32, Td.data_ptr(), Sd.data_ptr(), 0, 0, rho.data_ptr(), v_ref, _lib.F32,
                                        z_i.data_ptr(), depth.data_ptr(), pres.data_ptr(), -1 / 1035.0,
                                        e.ctypes.data_as(ctypes.c_void_p), nl, 2, 75, 1200, out, None)

    assert call([0.0, 700.0, 500.0], 2) == -2
    assert call([0.0, np.nan], 1) == -2
    assert call([0.0, np.inf, 3000.0], 2) == -2
    assert call([0.0, 1.0], 0) == -2
    assert call(np.arange(10.0), 9) == -2
    assert call([0.0, np.inf], 1, v_ref=None) == -1
    assert call([0.0, np.inf], 1, out=None) == -1
    assert call([0.0, 700.0, np.inf], 2) == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ xarray round trip


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
    edges = (0.0, 15.0, 100.0, None)
    result, reference = ml.steric_layers(ds, depth_edges=edges)
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    want, _ = ml.steric_layers(lab, depth_edges=edges)
    assert result["steric"].dims == ("time", "depth_layer", "yh", "xh")
    assert np.array_equal(np.asarray(result["steric"].values), want["steric"].values, equal_nan=True)
    assert result["steric"].attrs == {"long_name": "Steric height adjustment", "units": "m",
                                      "depth_edges": [0.0, 15.0, 100.0, float("inf")]}
    assert list(np.asarray(result["layer_top"].values)) == [0.0, 15.0, 100.0]
    assert list(np.asarray(result["layer_bottom"].values)) == [15.0, 100.0, np.inf]
    assert result["layer_top"].dims == ("depth_layer",)
    again, _ = ml.steric_layers(ds, depth_edges=edges, reference=reference)
    assert np.array_equal(np.asarray(again["steric"].values), want["steric"].values, equal_nan=True)
