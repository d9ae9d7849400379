"""steric_profile(zonal=True) and ml_steric_local_zonal_profile: the height change by level of every grid row (a
latitude-depth section), against a numpy reference of its own (the formula of tests/profile_oracle.py with the nansum
over x only), and the bit-identities the kernels promise: row j equals ml_steric_local_profile on row j sliced out
alone, numerators and quotients, and the bits depend neither on the chunks of the time axis, nor on the kernel
family, nor on one launch per variant, nor on the run.  The oracle tolerance is that of
tests/test_gpu_steric_profile.py, taken per (t, z, j)."""

import importlib.util
import json
import pathlib
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from momlevel_b200 import _lib, synth
from momlevel_b200.labeled import DataArray, Dataset
from oracle import steric as osteric

pytestmark = pytest.mark.gpu

VARIANTS = ("steric", "thermosteric", "halosteric")
RHO_FLOOR = 2e-15 * 1100.0  # kg m-3: a few ulp of the density, the difference of two fp64 evaluations of it
NZ = 6


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


def _land_row(ny):
    return ny - 2 if ny >= 3 else None


def _case(nt, ny, nx, dtype=torch.float32, seed=7):
    """Fields, grid and column weights with every edge at once: holes at wet cells, a reference volume that disagrees
    with the bathymetry, an all-land row (zero weight: a NaN row), a basin mask, NaN and zero weights."""
    grid = synth.make_grid(NZ, ny, nx, seed=seed, device="cpu")
    land = _land_row(ny)
    if land is not None:
        grid["deptho"][land] = float("nan")
        grid["areacello"][land] = 0.0
    T, S, V = synth.make_fields(grid, nt, seed=seed, dtype=dtype)
    wet = torch.nonzero(~torch.isnan(V))
    for k, i in enumerate((len(wet) // 2, len(wet) // 5, len(wet) // 9)):
        z, y, x = (int(j) for j in wet[i])
        (T if k % 2 == 0 else S)[(k * 3) % nt, z, y, x] = float("nan")
    for i in (len(wet) // 3, len(wet) // 7, 0):  # no reference volume at wet cells, the surface one included
        z, y, x = (int(j) for j in wet[i])
        V[z, y, x] = float("nan")
    dry = torch.nonzero(torch.isnan(V[0]))
    dry = dry[dry[:, 0] != (-1 if land is None else land)]
    if len(dry):  # a volume under a column the bathymetry calls land
        y, x = (int(j) for j in dry[len(dry) // 2])
        V[0, y, x] = 1.0e9
        T[:, 0, y, x], S[:, 0, y, x] = 12.0, 35.0
    w = grid["areacello"].clone().to(torch.float64) * (torch.arange(nx)[None, :] < max(1, 3 * nx // 4))  # a basin
    w.view(-1)[::7] = float("nan")
    w.view(-1)[3::11] = 0.0
    return grid, T, S, V, w


def _np(x):
    return x.detach().cpu().numpy().astype(np.float64) if isinstance(x, torch.Tensor) else np.asarray(x, np.float64)


def _patm2d(ny, nx):
    return 101325.0 + 50.0 * np.sin(np.arange(ny * nx, dtype=np.float64).reshape(ny, nx))


def _ops(ml, grid, T, S, V, w, t0=0, eos="Wright", patm=None):
    """Device operands of core.steric_local_zonal_profile, the reference state being step ``t0``."""
    dev = torch.device("cuda")
    T, S, V = T.to(dev), S.to(dev), V.to(dev)
    p = grid["z_l"].to(dev, torch.float64) * 1.0e4
    p = p + 101325.0 if patm is None else ml.core.Pressure(p, torch.as_tensor(patm, dtype=torch.float64, device=dev))
    rho, _ = ml.core.reference_state(T[t0], S[t0], V, p, eos=eos)
    return (T, S, T[t0].contiguous(), S[t0].contiguous(), rho, V, grid["z_i"].to(dev), grid["deptho"].to(dev), p,
            w.to(dev))


def _row(ml, ops, j):
    """The operands of grid row j alone, each in an allocation of its own (a row-sliced dataset)."""
    T, S, Tr, Sr, rho, V, z_i, depth, p, w = ops
    sl = lambda x: x[..., j:j + 1, :].clone(memory_format=torch.contiguous_format)  # noqa: E731
    if isinstance(p, ml.core.Pressure):
        p = ml.core.Pressure(p.level, sl(p.column))
    return (sl(T), sl(S), sl(Tr), sl(Sr), sl(rho), sl(V), z_i, sl(depth), p, sl(w))


def _same(a, b):
    return torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(b, nan=7.0)) and torch.equal(a.isnan(), b.isnan())


def _dt(x):
    return _lib.F32 if x.dtype == torch.float32 else _lib.F64


def _abi(ml, ops, ws_steps=None, poison=False, eos="Wright", zonal=True):
    """Numerators of every variant: ml_steric_local_zonal_profile [nt, nz, ny] with a workspace of ``ws_steps`` steps
    (NaN-filled if ``poison``), or ml_steric_local_profile [nt, nz] (``zonal=False``)."""
    L = _lib.lib()
    T, S, Tr, Sr, rho, V, z_i, depth, p, w = ops
    nt, nz, ny, nx = T.shape
    col = None
    if isinstance(p, ml.core.Pressure):
        p, col = p.level, p.column.to(torch.float64).contiguous()
    if zonal:
        nbytes = L.ml_zonal_profile_workspace_bytes(3, ws_steps or nt, nz, ny, nx)
    else:
        nbytes = L.ml_profile_workspace_bytes(3, nt, nz, ny * nx)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=T.device)
    if poison:
        ws.fill_(float("nan"))
    out = {v: torch.empty((nt, nz, ny) if zonal else (nt, nz), dtype=torch.float64, device=T.device) for v in VARIANTS}
    args = ({"Wright": 0, "Linear": 1}[eos], _dt(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(),
            rho.data_ptr(), V.data_ptr(), _dt(V), z_i.data_ptr(), depth.data_ptr(), w.data_ptr(), p.data_ptr(),
            -1.0 / 1035.0, nt, nz) + ((ny, nx) if zonal else (ny * nx,)) + (
            out["steric"].data_ptr(), out["thermosteric"].data_ptr(), out["halosteric"].data_ptr(), ws.data_ptr(),
            nbytes, None)
    if col is not None:
        _lib.check(L.ml_set_column_pressure(col.data_ptr(), col.numel()))
    try:
        _lib.check((L.ml_steric_local_zonal_profile if zonal else L.ml_steric_local_profile)(*args))
    finally:
        if col is not None:
            L.ml_set_column_pressure(None, 0)
    torch.cuda.synchronize()
    return out


def _oracle(grid, T, S, V, w, t0, eos, variant, patm):
    """``(section[t, z, j], tolerance[t, z, j])``: the profile_oracle formula with the nansum over x only."""
    Tn, Sn = _np(T), _np(S)
    ref = osteric.reference_state(Tn, Sn, np.broadcast_to(_np(V), Tn.shape), _np(grid["areacello"]), _np(grid["z_l"]),
                                  patm=patm, eos=eos, time_index=t0)
    _, drho = osteric.steric_local(Tn, Sn, _np(grid["z_l"]), _np(grid["z_i"]), _np(grid["deptho"]), ref, patm=patm,
                                   eos=eos, variant=variant)
    dz = osteric.calc_dz(_np(grid["z_l"]), _np(grid["z_i"]), _np(grid["deptho"]))
    m = ~np.isnan(ref["volcello"][0])
    wn = _np(w)
    mw = m * np.nan_to_num(wn, nan=0.0)
    terms = mw[None, None] * dz[None] * drho
    coef = -1.0 / 1035.0
    with np.errstate(invalid="ignore", divide="ignore"):
        W = np.nansum(wn, axis=1)
        want = coef * np.nansum(terms, axis=3) / W
        scale = abs(coef) * np.nansum(np.abs(terms), axis=3) / W
        wsum = np.nansum(np.abs(mw)[None] * dz, axis=2) / W
    return want, 1e-12 * scale + RHO_FLOOR / 1035.0 * wsum[None], W


# ---------------------------------------------------------------------------------------------------- oracle

RING = [(1, 300, 4), (5, 40, 36), (12, 16, 360), (13, 6, 1440), (5, 3, 2048), (12, 3, 2052), (1, 5, 2880),
        (5, 2, 4100), (12, 1, 360)]
PLAIN = [(13, 30, 35), (5, 4, 1441)]  # nx % 4 != 0: plain loads


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", RING + PLAIN, ids=lambda s: "x".join(map(str, s)))
def test_oracle_parity_and_the_row_alone(ml, shape, dtype, eos):
    nt, ny, nx = shape
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    t0 = min(2, nt - 1)  # a supplied reference that is not step 0
    for patm in ([None, _patm2d(ny, nx)] if dtype == torch.float32 else [None]):
        ops = _ops(ml, grid, T, S, V, w, t0=t0, eos=eos, patm=patm)
        got, totals = ml.core.steric_local_zonal_profile(*ops, eos=eos)
        ring = dtype == torch.float32 and patm is None and shape in RING
        assert ml.core.last_path() == (2 if ring else 1)
        for v in VARIANTS:
            want, tol, W = _oracle(grid, T, S, V, w, t0, eos, v, 101325.0 if patm is None else patm)
            g = got[v].cpu().numpy()
            assert g.shape == want.shape == (nt, NZ, ny)
            assert np.array_equal(np.isnan(g), np.isnan(want)), v
            ok = ~np.isnan(want)
            err = np.abs(g - want)[ok]
            assert (err <= tol[ok]).all(), (v, float(err.max()))
        np.testing.assert_allclose(totals.cpu().numpy(), W, rtol=1e-13, atol=0)
        land = _land_row(ny)
        if land is not None:
            assert totals[land] == 0 and got["steric"][:, :, land].isnan().all()
        # bit for bit ml_steric_local_profile on the row alone: numerators and the quotients of core
        num = _abi(ml, ops, eos=eos)
        for j in sorted({0, ny // 2, ny - 1} | ({land} if land is not None else set())):
            row = _row(ml, ops, j)
            want_num = _abi(ml, row, eos=eos, zonal=False)
            want_q = ml.core.steric_local_profile(*row, eos=eos)
            for v in VARIANTS:
                assert torch.equal(num[v][:, :, j], want_num[v]), (j, v)
                assert _same(got[v][:, :, j], want_q[v]), (j, v)
            assert totals[j] == torch.nansum(row[-1])


# --------------------------------------------------------------------------------------------- bit identities

GEOMS = [(torch.float32, (12, 16, 360)), (torch.float32, (5, 3, 2052)), (torch.float32, (4, 3, 4100)),
         (torch.float32, (5, 13, 37)), (torch.float64, (5, 20, 132))]
GIDS = ["ring", "ring_2052", "ring_4100", "ragged", "f64"]


@pytest.mark.parametrize("dtype, shape", GEOMS, ids=GIDS)
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_routes_chunks_and_runs_agree(ml, dtype, shape, eos):
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    ops = _ops(ml, grid, T, S, V, w, t0=1, eos=eos)
    whole = _abi(ml, ops, eos=eos)
    ring = ml.core.last_path() == 2
    assert ring == (dtype == torch.float32 and shape[2] % 4 == 0)
    for v in VARIANTS:
        assert torch.isfinite(whole[v]).all()
    # a NaN-filled workspace of one, two and all steps, and a second run
    for steps in (1, 2, shape[0]):
        got = _abi(ml, ops, steps, poison=True, eos=eos)
        for v in VARIANTS:
            assert torch.equal(got[v], whole[v]), (steps, v)
    again = _abi(ml, ops, eos=eos)
    # plain loads, and one launch per variant
    runs = {}
    for mode in (1, 2):
        prev = ml.core.force_direct(mode)
        try:
            runs[mode] = _abi(ml, ops, 1, poison=True, eos=eos)
            assert ml.core.last_path() == (1 if mode == 1 or not ring else 2)
        finally:
            ml.core.force_direct(prev)
    for v in VARIANTS:
        assert torch.equal(again[v], whole[v]) and torch.equal(runs[1][v], whole[v]) and torch.equal(runs[2][v],
                                                                                                     whole[v]), v
    # one variant at a time through core gives the bits of the one pass
    prof, totals = ml.core.steric_local_zonal_profile(*ops, eos=eos)
    for v in VARIANTS:
        assert _same(prof[v], whole[v] / totals)
        assert _same(ml.core.steric_local_zonal_profile(*ops, eos=eos, variants=v)[0][v], prof[v])


@pytest.mark.parametrize("dtype, shape", [(torch.float32, (12, 1, 2052)), (torch.float32, (5, 1, 37)),
                                          (torch.float64, (5, 1, 132))], ids=["ring", "ragged", "f64"])
def test_one_row_grid_is_the_profile(ml, dtype, shape):
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    ops = _ops(ml, grid, T, S, V, w, t0=3)
    num, want_num = _abi(ml, ops), _abi(ml, ops, zonal=False)
    prof, totals = ml.core.steric_local_zonal_profile(*ops)
    want = ml.core.steric_local_profile(*ops)
    for v in VARIANTS:
        assert torch.equal(num[v][:, :, 0], want_num[v])
        assert torch.equal(prof[v][:, :, 0], want[v])
    assert totals[0] == torch.nansum(ops[-1])


@pytest.mark.parametrize("dtype, shape", GEOMS, ids=GIDS)
def test_rows_combine_into_the_profile(ml, dtype, shape):
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    ops = _ops(ml, grid, T, S, V, w, t0=2)
    prof, W = ml.core.steric_local_zonal_profile(*ops)
    whole = ml.core.steric_local_profile(*ops)
    for v in VARIANTS:
        comb = torch.nansum(prof[v] * W, dim=2) / W.sum()
        # the tolerance of the whole-grid profile: rounding of the row sums and of the recombination
        _, tol, Wrow = _oracle(grid, T, S, V, w, 2, "Wright", v, 101325.0)
        bound = np.nansum(tol * Wrow, axis=2) / Wrow.sum() + 1e-15 * np.abs(whole[v].cpu().numpy())
        assert (np.abs(comb.cpu().numpy() - whole[v].cpu().numpy()) <= bound).all(), v


def _kernels(fn):
    """``(kernel, template arguments)`` of every library kernel ``fn`` launches, the arguments in the form
    ``("0", "7", "true", "false")`` whichever form the demangler gave them (``(bool)1``, ``(int)7``)."""
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = set()
    for e in prof.events():
        m = re.search(r"\b(k_\w+)(?:<([^<>]*)>)?\(", e.name)
        if m:
            args = [re.sub(r"^\((?:bool|int|unsigned int)\)", "", a.strip()) for a in (m.group(2) or "").split(",")]
            flags = [{"1": "true", "0": "false"}.get(a, a) for a in args[-2:]]  # ZON, REG
            out.add((m.group(1), tuple(args[:-2] + flags)))
    return out


_ROUTE_PROBE = """
import json, sys
import torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import momlevel_b200 as ml
import test_gpu_zonal_profile as t
dtype = getattr(torch, sys.argv[2])
grid, T, S, V, w = t._case(3, int(sys.argv[3]), int(sys.argv[4]), dtype=dtype)
ops = t._ops(ml, grid, T, S, V, w)
z = t._kernels(lambda: ml.core.steric_local_zonal_profile(*ops))
p = t._kernels(lambda: ml.core.steric_local_profile(*ops))
print(json.dumps({"zonal": sorted(z), "plain": sorted(p)}))
"""


@pytest.mark.parametrize("dtype, shape, kernel, storage", [("float32", (16, 64), "k_stream_profile", None),
                                                           ("float32", (13, 37), "k_profile_direct", "float"),
                                                           ("float64", (16, 64), "k_profile_direct", "double")],
                         ids=["ring", "ragged", "f64"])
def test_kernel_routes(ml, dtype, shape, kernel, storage):
    """The zonal call runs the zonal mode (ZON, REG = true, false) of the route's kernel and k_reduce_rows; the call
    without it runs the mode of before (false, false).  The profiler runs in an interpreter of its own, so what earlier
    tests did to its state in this process does not decide what it records."""
    root = pathlib.Path(__file__).resolve().parent.parent
    res = subprocess.run([sys.executable, "-c", _ROUTE_PROBE, str(root), dtype, *map(str, shape)], capture_output=True,
                         text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])

    def modes(names):
        return {tuple(a[-2:]) for k, a in names if k == kernel and (storage is None or a[0] == storage)}

    assert modes(got["zonal"]) == {("true", "false")}, got["zonal"]
    assert any(k == "k_reduce_rows" for k, _ in got["zonal"]), got["zonal"]
    assert modes(got["plain"]) == {("false", "false")}, got["plain"]


# ------------------------------------------------------------------------------------------------- public call


def _row_dataset(ds, j):
    """``ds`` cut to grid row j: every (y, x) field sliced to [..., j:j+1, :] in an allocation of its own."""
    out = Dataset()
    for name, var in ds.variables.items():
        d = var.data
        if "yh" in var.dims:
            ax = var.dims.index("yh")
            d = d.narrow(ax, j, 1).clone(memory_format=torch.contiguous_format) if isinstance(d, torch.Tensor) else \
                np.ascontiguousarray(np.take(np.asarray(d), [j], axis=ax))
        out[name] = DataArray(d, var.dims, attrs=dict(var.attrs))
    return out


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_public_call(ml, dtype):
    nt, ny, nx = 6, 12, 132
    grid, T, S, V, w = _case(nt, ny, nx, dtype=dtype)
    dev = torch.device("cuda")
    ds = synth.dataset_from_fields({k: v.to(dev) for k, v in grid.items()}, T.to(dev), S.to(dev), V.to(dev))
    other = synth.make_dataset(1, NZ, ny, nx, seed=21, device="cuda", dtype=dtype)
    _, supplied = ml.steric(other)  # a reference that is not a step of ds
    for patm, ref in ((101325.0, None), (101325.0, supplied), (_patm2d(ny, nx), None)):
        res, ref2 = ml.steric_profile(ds, variant=list(VARIANTS), zonal=True, weights=w.numpy(), reference=ref,
                                      patm=patm, strict=False)
        assert ml.core.last_path() == (2 if dtype == torch.float32 and np.ndim(patm) == 0 else 1)
        assert np.asarray(res["yh"].values).tolist() == list(range(ny))
        for v in VARIANTS:
            assert res[v].dims == ("time", "z_l", "yh") and res[v].shape == (nt, NZ, ny)
        if ref is None:  # against the oracle: the reference is step 0
            for v in VARIANTS:
                want, tol, W = _oracle(grid, T, S, V, w, 0, "Wright", v, patm)
                g = np.asarray(res[v].values)
                assert np.array_equal(np.isnan(g), np.isnan(want))
                ok = ~np.isnan(want)
                assert (np.abs(g - want)[ok] <= tol[ok]).all(), v
            np.testing.assert_allclose(np.asarray(res["zonal_weight"].values), W, rtol=1e-13, atol=0)
        # row j is, bit for bit, the public call on the row-sliced dataset with the row-sliced reference
        for j in (0, ny // 2, _land_row(ny), ny - 1):
            rref = _row_dataset(ref2, j)
            rw = np.ascontiguousarray(w.numpy()[j:j + 1])
            rp = patm if np.ndim(patm) == 0 else np.ascontiguousarray(patm[j:j + 1])
            one, _ = ml.steric_profile(_row_dataset(ds, j), variant=list(VARIANTS), weights=rw, reference=rref,
                                       patm=rp, strict=False)
            for v in VARIANTS:
                assert _same(res[v].data[:, :, j], one[v].data), (j, v)


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
    result, reference = ml.steric_profile(ds, variant=list(VARIANTS), zonal=True)
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    want, _ = ml.steric_profile(lab, variant=list(VARIANTS), zonal=True)
    ydim = lab["thetao"].dims[2]
    for v in VARIANTS:
        assert result[v].dims == ("time", lab["thetao"].dims[1], ydim)
        assert np.array_equal(np.asarray(result[v].values), np.asarray(want[v].values), equal_nan=True)
    assert np.array_equal(np.asarray(result["zonal_weight"].values), np.asarray(want["zonal_weight"].values))
