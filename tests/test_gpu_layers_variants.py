"""steric_layers(variant=[...]) and ml_steric_local_layers_variants: the steric, thermosteric and halosteric heights
by depth layer from one pass over T and S, bit for bit against one ml_steric_local_layers launch per height (one-pass
and fallback shapes), against ml_steric_local_variants for the single layer (0, None), against the numpy reference
(tests/layers_oracle.py), and the public call against one steric_layers call per name."""

import ctypes
import importlib.util
import itertools
import pathlib
import sys

import numpy as np
import pytest
import torch

import layers_oracle  # tests/layers_oracle.py
from oracle import steric as osteric

pytestmark = pytest.mark.gpu

VARIANTS = ("steric", "thermosteric", "halosteric")
ETA_ATOL = 1e-9  # m
CHUNKS = (4, 6, 12)  # the instantiated chunk widths of the one-pass layered kernel


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


def _fields(nt, ny, nx, dtype=torch.float32, seed=7, hole=False, vmask=False):
    from momlevel_b200 import synth

    grid = synth.make_grid(75, ny, nx, seed=seed, device="cpu")
    T, S, V = synth.make_fields(grid, nt, seed=seed, dtype=dtype)
    wet = torch.nonzero(~torch.isnan(V))
    if hole:  # a missing value at a wet cell of one step: the repair pass
        z, y, x = (int(i) for i in wet[len(wet) // 2])
        T[nt // 2, z, y, x] = float("nan")
        z, y, x = (int(i) for i in wet[len(wet) // 5])
        S[nt - 1, z, y, x] = float("nan")
    if vmask:  # a reference volume that is missing at cells the bathymetry calls wet
        for i in (len(wet) // 3, len(wet) // 7, 2 * len(wet) // 3):
            z, y, x = (int(j) for j in wet[i])
            V[z, y, x] = float("nan")
    return grid, T, S, V


class _Case:
    """Device operands of one layered call with the reference state taken from step `ref_step` of the fields."""

    def __init__(self, core, grid, T, S, V, eos="Wright", ref_step=0, pres=None):
        self.core, self.eos, self.grid = core, eos, grid
        self.T, self.S, self.V = T.cuda(), S.cuda(), V.cuda()
        self.Tr, self.Sr = self.T[ref_step].clone(), self.S[ref_step].clone()
        self.pres = (grid["z_l"] * 1.0e4 + 101325.0).cuda() if pres is None else pres
        self.rho, _ = core.reference_state(self.Tr, self.Sr, self.V, self.pres, eos=eos)
        self.z_i, self.depth = grid["z_i"].cuda(), grid["deptho"].cuda()

    def one_call(self, edges, variants=VARIANTS):
        return self.core.steric_local_layers_variants(self.T, self.S, self.Tr, self.Sr, self.rho, self.V, self.z_i,
                                                      self.depth, self.pres, edges, eos=self.eos, variants=variants)

    def launches(self, edges, variant):
        """one ml_steric_local_layers launch for one height"""
        T, S, tb, sb = self.T, self.S, False, False
        if variant == "thermosteric":
            S, sb = self.Sr, True
        elif variant == "halosteric":
            T, tb = self.Tr, True
        return self.core.steric_local_layers(T, S, self.rho, self.V, self.z_i, self.depth, self.pres, edges, eos=self.eos,
                                             t_bcast=tb, s_bcast=sb)


def _bits(t):
    return t.contiguous().view(torch.int64)


def _same(got, want, what=""):
    assert got.shape == want.shape, what
    assert torch.equal(_bits(got), _bits(want)), what  # NaNs compare equal only as the same bits


def _counted(core, fn):
    before = core.launch_count()
    out = fn()
    torch.cuda.synchronize()
    return out, core.launch_count() - before


def _close(got, want, atol=ETA_ATOL):
    assert got.shape == want.shape
    assert np.array_equal(np.isnan(got), np.isnan(want))
    m = ~np.isnan(want)
    assert float(np.max(np.abs(got[m] - want[m]), initial=0.0)) <= atol


# ------------------------------------------------------------------------------------- one pass == three launches


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
@pytest.mark.parametrize("chunk", (0,) + CHUNKS)
def test_one_pass_is_bit_identical_to_three_launches(ml, eos, chunk):
    core = ml.core
    prev = core.variants_chunk(chunk)
    try:
        for nt in (1, 5, 12, 13, 25):
            grid, T, S, V = _fields(nt, 12, 100)
            case = _Case(core, grid, T, S, V, eos)
            for edges in _edge_sets(grid["z_i"].numpy()):
                got, n_one = _counted(core, lambda: case.one_call(edges))
                assert core.last_path() == 2
                old = core.force_direct(2)
                try:
                    ab, n_three = _counted(core, lambda: case.one_call(edges))
                finally:
                    core.force_direct(old)
                assert n_one < n_three, (n_one, n_three)  # the one-pass kernel ran, not three launches
                for v in VARIANTS:
                    want = case.launches(edges, v)
                    _same(got[v], want, (nt, edges, v))
                    _same(ab[v], want, (nt, edges, v))
    finally:
        core.variants_chunk(prev)


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_supplied_reference_holes_and_a_volume_mask(ml, eos):
    """A reference that is not step 0, holes at wet cells (the repair pass of every layer of every height) and a
    reference volume that disagrees with the bathymetry."""
    core = ml.core
    for nt, chunk in ((13, 0), (25, 6), (5, 4)):
        grid, T, S, V = _fields(nt, 12, 100, hole=True, vmask=True)
        case = _Case(core, grid, T, S, V, eos, ref_step=min(3, nt - 1))
        prev = core.variants_chunk(chunk)
        try:
            for edges in _edge_sets(grid["z_i"].numpy()):
                got = case.one_call(edges)
                assert core.last_path() == 2
                for v in VARIANTS:
                    _same(got[v], case.launches(edges, v), (nt, edges, v))
                # the repaired columns are finite in every layer where the surface holds water
                wet = ~torch.isnan(case.V[0]).cpu()
                assert torch.isfinite(got["steric"].cpu()[:, :, wet]).all()
        finally:
            core.variants_chunk(prev)


def test_every_pair_of_outputs(ml):
    core = ml.core
    grid, T, S, V = _fields(13, 12, 100, hole=True)
    case = _Case(core, grid, T, S, V)
    edges = _edge_sets(grid["z_i"].numpy())[1]
    want = {v: case.launches(edges, v) for v in VARIANTS}
    _, n_single = _counted(core, lambda: case.launches(edges, "steric"))
    for k in (1, 2, 3):
        for names in itertools.permutations(VARIANTS, k):
            got, n = _counted(core, lambda: case.one_call(edges, names))
            assert set(got) == set(names)
            for v in names:
                _same(got[v], want[v], (names, v))
            if k == 1:
                assert n == n_single  # one height: its own ml_steric_local_layers launch
            else:
                assert n < k * n_single


# ------------------------------------------------------------------------------------------------- fallback shapes


@pytest.mark.parametrize("shape", ["fp64", "ragged", "narrow", "column_pressure"])
def test_fallback_shapes_are_three_launches(ml, shape):
    core = ml.core
    dtype = torch.float64 if shape == "fp64" else torch.float32
    ny, nx = {"ragged": (13, 101), "narrow": (12, 20)}.get(shape, (12, 100))  # 1313 columns; 240 < 256 columns
    grid, T, S, V = _fields(13, ny, nx, dtype, hole=True)
    pres = None
    if shape == "column_pressure":
        patm = 101325.0 + 500.0 * torch.rand((ny, nx), dtype=torch.float64, generator=torch.Generator().manual_seed(1))
        pres = core.Pressure((grid["z_l"] * 1.0e4).cuda(), patm.cuda())
    case = _Case(core, grid, T, S, V, pres=pres)
    for edges in _edge_sets(grid["z_i"].numpy()):
        got, n = _counted(core, lambda: case.one_call(edges))
        want, n3 = {}, 0
        for v in VARIANTS:
            want[v], nv = _counted(core, lambda: case.launches(edges, v))
            n3 += nv
        assert n == n3  # no one-pass kernel: one ml_steric_local_layers per height
        for v in VARIANTS:
            _same(got[v], want[v], (shape, edges, v))
        if shape == "column_pressure":
            assert core.last_path() == 1


# ---------------------------------------------------------------------------------------------------- one layer


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_single_layer_equals_local_variants(ml, eos):
    core = ml.core
    for nt in (5, 13):
        grid, T, S, V = _fields(nt, 12, 100, hole=True)
        case = _Case(core, grid, T, S, V, eos, ref_step=1)
        lay = case.one_call((0.0, None))
        full, _, _ = core.steric_local_variants(case.T, case.S, case.V, case.z_i, case.depth, case.pres, T_ref=case.Tr,
                                                S_ref=case.Sr, rho_ref=case.rho, eos=eos)
        for v in VARIANTS:
            _same(lay[v][:, 0], full[v], v)


# ------------------------------------------------------------------------------------------------------- the oracle


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_oracle_parity(ml, dtype, eos):
    core = ml.core
    for nt, ny, nx in ((13, 12, 100), (5, 13, 101)):
        grid, T, S, V = _fields(nt, ny, nx, dtype)
        case = _Case(core, grid, T, S, V, eos)
        f = lambda t: t.double().cpu().numpy()  # noqa: E731
        z_l, z_i, depth, area = (f(grid[k]) for k in ("z_l", "z_i", "deptho", "areacello"))
        Tn, Sn = f(T), f(S)
        ref = osteric.reference_state(Tn, Sn, f(V)[None].repeat(nt, 0), area, z_l, eos=eos)
        for edges in _edge_sets(grid["z_i"].numpy()):
            got = case.one_call(edges)
            for v in VARIANTS:
                want = layers_oracle.steric_local_layers(Tn, Sn, z_l, z_i, depth, ref, edges, eos=eos, variant=v)
                _close(got[v].cpu().numpy(), want)


# ------------------------------------------------------------------------------------------------ the public call


def _host_copy(ml, ds):
    host = ds.copy()
    for k in ("thetao", "so", "volcello", "deptho", "areacello", "z_l", "z_i"):
        host[k] = ml.DataArray(ds[k].data.cpu().numpy(), ds[k].dims, attrs=ds[k].attrs)
    return host


def _public_same(ml, ds, names=VARIANTS, **kw):
    res, ref = ml.steric_layers(ds, variant=list(names), **kw)
    for v in names:
        one, _ = ml.steric_layers(ds, variant=v, **kw)
        a, b = res[v], one[v]
        assert a.dims == b.dims and a.attrs == b.attrs and a.encoding["dtype"] == b.encoding["dtype"]
        assert np.array_equal(np.asarray(a.values).view(np.int64), np.asarray(b.values).view(np.int64)), v
    assert list(res["layer_top"].values) == list(one["layer_top"].values)
    assert list(res["layer_bottom"].values) == list(one["layer_bottom"].values)
    return res, ref


@pytest.mark.parametrize("where", ["device", "host"])
def test_public_list_equals_one_call_per_name(ml, where):
    from momlevel_b200 import synth

    ds = synth.make_dataset(13, 75, 12, 100, seed=6, device="cuda")
    if where == "host":
        ds = _host_copy(ml, ds)
    before = ml.core.launch_count()
    res, ref = _public_same(ml, ds)
    assert ml.core.launch_count() > before
    assert set(res.variables) >= {*VARIANTS, "layer_top", "layer_bottom"} and "delta_rho" not in res.variables
    assert res["halosteric"].dims == ("time", "depth_layer", "yh", "xh") and res["halosteric"].shape == (13, 3, 12, 100)
    # a supplied reference, a subset and a one-element list
    _public_same(ml, ds, reference=ref)
    _public_same(ml, ds, names=("halosteric", "thermosteric"), reference=ref)
    one, _ = ml.steric_layers(ds, variant=["thermosteric"], reference=ref)
    alone, _ = ml.steric_layers(ds, variant="thermosteric", reference=ref)
    assert set(one.variables) == set(alone.variables)
    assert torch.equal(_bits(torch.as_tensor(np.asarray(one["thermosteric"].values))),
                       _bits(torch.as_tensor(np.asarray(alone["thermosteric"].values))))


def test_public_list_one_pass_on_device_fields(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(13, 75, 12, 100, seed=6, device="cuda")
    _, ref = ml.steric_layers(ds, variant="steric")
    before = ml.core.launch_count()
    ml.steric_layers(ds, variant=list(VARIANTS), reference=ref)
    n_one = ml.core.launch_count() - before
    before = ml.core.launch_count()
    for v in VARIANTS:
        ml.steric_layers(ds, variant=v, reference=ref)
    assert ml.core.launch_count() - before > n_one


def test_public_list_annual_and_2d_patm(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(24, 75, 12, 100, seed=8, device="cuda")
    days = np.tile([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], 2).astype(np.float64)
    res, _ = _public_same(ml, ds, annual=True, days_in_month=days)
    assert res["steric"].shape[0] == 2
    patm = 101325.0 + 500.0 * torch.rand((12, 100), dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    _public_same(ml, ds, patm=patm.numpy())
    assert ml.core.last_path() == 1  # a column pressure takes the direct family


def test_public_list_errors(ml):
    from momlevel_b200 import synth

    ds = synth.make_dataset(3, 75, 12, 100, seed=9, device="cuda")
    for bad in ([], ("steric", "steric"), ["steric", "barotropic"], ("Steric",)):
        with pytest.raises(ValueError):
            ml.steric_layers(ds, variant=bad)


def test_abi_errors_with_device_operands(ml):
    from momlevel_b200 import _lib

    core, L = ml.core, _lib.lib()
    grid, T, S, V = _fields(2, 12, 100)
    c = _Case(core, grid, T, S, V)
    eta = [torch.empty((2, 8, 1200), dtype=torch.float64, device="cuda") for _ in range(3)]

    def call(edges, nl, rho=c.rho.data_ptr(), outs=tuple(e.data_ptr() for e in eta), eos=0):
        e = np.asarray(edges, dtype=np.float64)
        return L.ml_steric_local_layers_variants(eos, _lib.F32, c.T.data_ptr(), c.S.data_ptr(), c.Tr.data_ptr(),
                                                 c.Sr.data_ptr(), rho, c.V.data_ptr(), _lib.F32, c.z_i.data_ptr(),
                                                 c.depth.data_ptr(), c.pres.data_ptr(), -1 / 1035.0,
                                                 e.ctypes.data_as(ctypes.c_void_p), nl, 2, 75, 1200, *outs, None)

    assert call([0.0, 700.0, 500.0], 2) == -2
    assert call([0.0, np.nan], 1) == -2
    assert call([0.0, np.inf, 3000.0], 2) == -2
    assert call([0.0, 1.0], 0) == -2
    assert call(np.arange(10.0), 9) == -2
    assert call([0.0, np.inf], 1, rho=None) == -1
    assert call([0.0, np.inf], 1, outs=(None, None, None)) == -1
    assert call([0.0, np.inf], 1, eos=7) == -4
    assert call([0.0, 700.0, np.inf], 2) == 0
    assert call([0.0, 700.0, np.inf], 2, outs=(None, eta[1].data_ptr(), None)) == 0
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
    result, reference = ml.steric_layers(ds, depth_edges=edges, variant=list(VARIANTS))
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    for v in VARIANTS:
        want, _ = ml.steric_layers(ds, depth_edges=edges, variant=v)
        assert result[v].dims == ("time", "depth_layer", "yh", "xh")
        assert np.array_equal(np.asarray(result[v].values), np.asarray(want[v].values), equal_nan=True)
        assert result[v].attrs == want[v].attrs
    assert list(np.asarray(result["layer_bottom"].values)) == [15.0, 100.0, np.inf]
    again, _ = ml.steric_layers(ds, depth_edges=edges, variant=("thermosteric", "halosteric"), reference=reference)
    assert np.array_equal(np.asarray(again["halosteric"].values), np.asarray(result["halosteric"].values), equal_nan=True)
