"""steric_profile(regions=...) and ml_steric_local_region_profile: the height change by level of every region of a
region map, against the numpy reference (tests/profile_oracle.py) called with the region's masked weights, and the
bit-identities the kernels promise: region r equals ml_steric_local_profile with weights where(region == r, w, 0),
one region equals the call without regions, and the bits depend neither on the chunks of the time axis, nor on the
kernel family, nor on the run.  The oracle tolerance is that of tests/test_gpu_steric_profile.py."""

import importlib.util
import pathlib
import sys

import numpy as np
import pytest
import torch

from momlevel_b200 import _lib, synth
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


def _case(nt, ny, nx, dtype=torch.float32, seed=7, hole=False):
    grid = synth.make_grid(NZ, ny, nx, seed=seed, device="cpu")
    T, S, V = synth.make_fields(grid, nt, seed=seed, dtype=dtype)
    if hole:
        wet = torch.nonzero(~torch.isnan(V))
        for k, i in enumerate((len(wet) // 2, len(wet) // 5, len(wet) // 9)):
            z, y, x = (int(j) for j in wet[i])
            (T if k % 2 == 0 else S)[(k * 3) % nt, z, y, x] = float("nan")
    area = grid["areacello"].clone().to(torch.float64)
    area.view(-1)[::13] = float("nan")
    return grid, T, S, V, area


def _map(kind, ny, nx, seed=3):
    """A region index [ny, nx] (-1: no region) and its number of regions."""
    g = torch.Generator().manual_seed(seed)
    if kind == "blocks":  # coherent: longitude sectors x two latitude bands, and an excluded strip
        x = torch.arange(nx)[None, :].expand(ny, nx)
        y = torch.arange(ny)[:, None].expand(ny, nx)
        idx = (x * 3 // nx) * 2 + (y * 2 // ny)
        idx = torch.where(x < max(1, nx // 10), -1, idx)
        return idx, 6
    if kind == "random":  # every warp touches many regions
        return torch.randint(-1, 11, (ny, nx), generator=g), 11
    if kind == "fifteen":
        return torch.randint(0, 15, (ny, nx), generator=g), 15
    if kind == "empty":  # regions 1 and 4 have no columns
        idx = torch.randint(0, 3, (ny, nx), generator=g)
        return torch.where(idx == 1, 3, idx), 5
    if kind == "one":
        return torch.zeros((ny, nx), dtype=torch.int64), 1
    raise ValueError(kind)


def _np(x):
    return x.detach().cpu().numpy().astype(np.float64) if isinstance(x, torch.Tensor) else np.asarray(x, np.float64)


def _ops(ml, grid, T, S, V, w, t0=0, eos="Wright"):
    dev = torch.device("cuda")
    T, S, V = T.to(dev), S.to(dev), V.to(dev)
    p = grid["z_l"].to(dev, torch.float64) * 1.0e4 + 101325.0
    rho, _ = ml.core.reference_state(T[t0], S[t0], V, p, eos=eos)
    return (T, S, T[t0], S[t0], rho, V, grid["z_i"].to(dev), grid["deptho"].to(dev), p, w.to(dev))


def _region(ml, ops, idx, nreg, eos="Wright", variants=VARIANTS):
    return ml.core.steric_local_region_profile(*ops, idx, nreg, eos=eos, variants=variants)


def _masked(ml, ops, idx, r, eos="Wright", variants=VARIANTS):
    w = ops[-1]
    mw = torch.where(idx.to(w.device).reshape(w.shape) == r, w, 0.0)
    return ml.core.steric_local_profile(*ops[:-1], mw, eos=eos, variants=variants)


def _same(a, b):
    return torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(b, nan=7.0)) and torch.equal(a.isnan(), b.isnan())


# ---------------------------------------------------------------------------------------------------- oracle


SHAPES = [(1, 32, 128), (5, 13, 37), (12, 12, 20), (13, 20, 132)]


@pytest.mark.parametrize("eos", ["Wright", "Linear"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_oracle_parity(ml, shape, dtype, eos):
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    idx, nreg = _map("blocks", *shape[1:])
    got, totals = _region(ml, _ops(ml, grid, T, S, V, w, eos=eos), idx, nreg, eos=eos)
    V4 = np.broadcast_to(_np(V), tuple(T.shape))
    ref = osteric.reference_state(_np(T), _np(S), V4, _np(grid["areacello"]), _np(grid["z_l"]), eos=eos)
    m = ~np.isnan(ref["volcello"][0])
    dz = osteric.calc_dz(_np(grid["z_l"]), _np(grid["z_i"]), _np(grid["deptho"]))
    for r in range(nreg):
        mw = np.where(_np(idx) == r, _np(w), 0.0)
        assert abs(float(totals[r]) / np.nansum(mw) - 1) < 1e-13
        wsum = np.nansum(np.abs(m * np.nan_to_num(mw, nan=0.0))[None] * dz, axis=(1, 2)) / np.nansum(mw)
        for v in VARIANTS:
            want, scale = profile_oracle.steric_profile(_np(T), _np(S), _np(grid["z_l"]), _np(grid["z_i"]),
                                                        _np(grid["deptho"]), ref, weights=mw, eos=eos, variant=v)
            g = got[v][r].cpu().numpy()
            tol = 1e-12 * scale + RHO_FLOOR / 1035.0 * wsum[None]
            assert g.shape == want.shape and np.isfinite(g).all()
            err = np.abs(g - want)
            assert (err <= tol).all(), (r, v, float(err.max()))


# --------------------------------------------------------------------------------------------- bit identities


GEOMS = [(torch.float32, (12, 32, 128)), (torch.float32, (5, 13, 37)), (torch.float64, (5, 20, 132))]


@pytest.mark.parametrize("kind", ["blocks", "random", "fifteen", "empty"])
@pytest.mark.parametrize("dtype, shape", GEOMS, ids=["ring", "ragged", "f64"])
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_each_region_is_the_masked_weights_call(ml, dtype, shape, kind, eos):
    grid, T, S, V, w = _case(*shape, dtype=dtype, hole=True)
    ops = _ops(ml, grid, T, S, V, w, t0=2, eos=eos)
    idx, nreg = _map(kind, *shape[1:])
    got, totals = _region(ml, ops, idx, nreg, eos=eos)
    assert ml.core.last_path() == (2 if shape == (12, 32, 128) else 1)
    for r in range(nreg):
        want = _masked(ml, ops, idx, r, eos=eos)
        for v in VARIANTS:
            assert _same(got[v][r], want[v]), (kind, r, v)
        if not (idx == r).any():
            assert totals[r] == 0 and got["steric"][r].isnan().all()


@pytest.mark.parametrize("dtype, shape", GEOMS, ids=["ring", "ragged", "f64"])
def test_one_region_is_the_call_without_regions(ml, dtype, shape):
    grid, T, S, V, w = _case(*shape, dtype=dtype, hole=True)
    ops = _ops(ml, grid, T, S, V, w)
    idx, _ = _map("one", *shape[1:])
    got, totals = _region(ml, ops, idx, 1)
    want = ml.core.steric_local_profile(*ops)
    for v in VARIANTS:
        assert torch.equal(got[v][0], want[v]), v
    assert totals[0] == torch.nansum(ops[-1])


def _abi(ml, ops, idx, nreg, ws_steps, poison=False, eos="Wright"):
    """ml_steric_local_region_profile with a workspace of ``ws_steps`` steps (NaN-filled if ``poison``); the
    numerators [nreg, nt, nz] of each variant."""
    L = _lib.lib()
    T, S, Tr, Sr, rho, V, z_i, depth, p, w = ops
    z_i, depth = z_i.to(torch.float64), depth.to(torch.float64)
    nt, nz = T.shape[:2]
    ncol = T[0, 0].numel()
    ri = idx.to(torch.int8).reshape(-1).to(T.device)
    nbytes = L.ml_region_profile_workspace_bytes(3, nreg, ws_steps, nz, ncol)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=T.device)
    if poison:
        ws.fill_(float("nan"))
    out = {v: torch.empty((nreg, nt, nz), dtype=torch.float64, device=T.device) for v in VARIANTS}
    dt = _lib.F32 if T.dtype == torch.float32 else _lib.F64
    vdt = _lib.F32 if V.dtype == torch.float32 else _lib.F64
    _lib.check(L.ml_steric_local_region_profile(
        {"Wright": 0, "Linear": 1}[eos], dt, T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), rho.data_ptr(),
        V.data_ptr(), vdt, z_i.data_ptr(), depth.data_ptr(), w.data_ptr(),
        ri.data_ptr(), nreg, p.data_ptr(), -1.0 / 1035.0, nt, nz, ncol, out["steric"].data_ptr(),
        out["thermosteric"].data_ptr(), out["halosteric"].data_ptr(), ws.data_ptr(), nbytes, None))
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("dtype, shape", GEOMS, ids=["ring", "ragged", "f64"])
@pytest.mark.parametrize("kind", ["blocks", "random"])
def test_chunks_and_a_poisoned_workspace(ml, dtype, shape, kind):
    grid, T, S, V, w = _case(*shape, dtype=dtype, hole=True)
    ops = _ops(ml, grid, T, S, V, w, t0=1)
    idx, nreg = _map(kind, *shape[1:])
    whole = _abi(ml, ops, idx, nreg, shape[0])
    for steps in (1, 2, shape[0]):
        got = _abi(ml, ops, idx, nreg, steps, poison=True)
        for v in VARIANTS:
            assert torch.equal(got[v], whole[v]), (steps, v)
            assert torch.isfinite(got[v]).all()
    # the numerators are those core divides
    prof, totals = _region(ml, ops, idx, nreg)
    for v in VARIANTS:
        assert _same(prof[v], whole[v] / totals[:, None, None])


@pytest.mark.parametrize("shape", [(12, 32, 128), (7, 12, 20)])
@pytest.mark.parametrize("kind", ["blocks", "random"])
@pytest.mark.parametrize("eos", ["Wright", "Linear"])
def test_ring_plain_split_and_repeat_agree(ml, shape, kind, eos):
    grid, T, S, V, w = _case(*shape, hole=True)
    ops = _ops(ml, grid, T, S, V, w, t0=1, eos=eos)
    idx, nreg = _map(kind, *shape[1:])
    ring, _ = _region(ml, ops, idx, nreg, eos=eos)
    assert ml.core.last_path() == 2
    again, _ = _region(ml, ops, idx, nreg, eos=eos)
    runs = {}
    for mode in (1, 2):
        prev = ml.core.force_direct(mode)
        try:
            runs[mode], _ = _region(ml, ops, idx, nreg, eos=eos)
            if mode == 1:
                assert ml.core.last_path() == 1
        finally:
            ml.core.force_direct(prev)
    for v in VARIANTS:
        assert _same(ring[v], again[v]) and _same(ring[v], runs[1][v]) and _same(ring[v], runs[2][v]), v
    # one variant at a time gives the same bits as the one pass
    for v in VARIANTS:
        assert _same(_region(ml, ops, idx, nreg, eos=eos, variants=v)[0][v], ring[v])


def _kernels(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events()}


@pytest.mark.parametrize("dtype, shape, family", [(torch.float32, (3, 16, 64), "k_stream_profile<"),
                                                  (torch.float32, (3, 13, 37), "k_profile_direct<float"),
                                                  (torch.float64, (3, 16, 64), "k_profile_direct<double")],
                         ids=["ring", "ragged", "f64"])
def test_kernel_routes(ml, dtype, shape, family):
    grid, T, S, V, w = _case(*shape, dtype=dtype)
    ops = _ops(ml, grid, T, S, V, w)
    idx, nreg = _map("blocks", *shape[1:])
    names = _kernels(lambda: _region(ml, ops, idx, nreg))
    assert any(family in n and "true>" in n for n in names), sorted(names)
    assert any("k_reduce_rows" in n for n in names)
    plain = _kernels(lambda: ml.core.steric_local_profile(*ops))
    assert any(family in n and "false>" in n for n in plain), sorted(plain)
    assert not any("true>" in n for n in plain if "profile" in n)


# ------------------------------------------------------------------------------------------------- public call


def _public_masked(ml, ds, codes, regions, **kw):
    area = np.asarray(ds["areacello"].values, dtype=np.float64)
    w = kw.pop("weights", area)
    return [ml.steric_profile(ds, weights=np.where(regions == c, w, 0.0), **kw)[0] for c in codes]


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
def test_public_call_equals_the_masked_public_calls(ml, dtype):
    ds = synth.make_dataset(6, NZ, 20, 132, seed=9, device="cuda", dtype=dtype)
    ds["thetao"].data[2, 1, 4, 40] = float("nan")  # a hole at a wet cell
    ds["so"].data[4, 0, 7, 90] = float("nan")
    regions = np.floor(np.arange(132)[None, :] / 30.0) + 0 * np.arange(20)[:, None]
    regions[3, :10] = np.nan
    regions[5, 5:9] = -3
    codes = [4, 1, 0, 2]
    other = synth.make_dataset(1, NZ, 20, 132, seed=21, device="cuda", dtype=dtype)
    _, supplied = ml.steric(other)  # a reference that is not step 0 of ds
    for ref in (None, supplied):
        res, ref2 = ml.steric_profile(ds, variant=list(VARIANTS), regions=regions, region_codes=codes, reference=ref)
        if ref is not None:
            assert ref2 is ref
        want = _public_masked(ml, ds, codes, regions, variant=list(VARIANTS), reference=ref2)
        area = np.asarray(ds["areacello"].values, np.float64)
        for i, c in enumerate(codes):
            for v in VARIANTS:
                assert torch.equal(res[v].data[:, i], want[i][v].data), (i, v)
            w = torch.as_tensor(np.where(regions == c, area, 0.0), device="cuda")
            assert float(res["region_weight"].data[i]) == float(torch.nansum(w))
    # one code everywhere is the call without regions
    one, _ = ml.steric_profile(ds, variant=list(VARIANTS), regions=np.full((20, 132), 3))
    plain, _ = ml.steric_profile(ds, variant=list(VARIANTS))
    for v in VARIANTS:
        assert torch.equal(one[v].data[:, 0], plain[v].data)


def test_public_call_2d_patm(ml):
    ds = synth.make_dataset(6, NZ, 16, 64, seed=4, device="cuda", dtype=torch.float32)
    regions = (np.arange(64)[None, :] // 16 + 0 * np.arange(16)[:, None]).astype(np.int32)
    patm = 101325.0 + 50.0 * np.sin(np.arange(16 * 64).reshape(16, 64))
    _, reference = ml.steric(ds, patm=patm)
    res, _ = ml.steric_profile(ds, regions=regions, patm=patm, reference=reference, variant=list(VARIANTS))
    assert ml.core.last_path() == 1  # the column pressure takes the plain-load kernel
    want = _public_masked(ml, ds, [0, 1, 2, 3], regions, patm=patm, reference=reference, variant=list(VARIANTS))
    for i in range(4):
        for v in VARIANTS:
            assert torch.equal(res[v].data[:, i], want[i][v].data)


def test_public_call_supplied_reference_of_a_later_step(ml):
    grid, T, S, V, w = _case(6, 16, 64)
    ops = _ops(ml, grid, T, S, V, grid["areacello"].to(torch.float64), t0=4)
    idx, nreg = _map("blocks", 16, 64)
    got, _ = _region(ml, ops, idx, nreg)
    for v in VARIANTS:
        assert (got[v][:, 4] == 0).all()  # the step that is the reference state
        assert (got[v][:, :4] != 0).any()


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
    shape = tuple(np.shape(lab["areacello"].values))
    regions = (np.arange(shape[1])[None, :] % 3 + 0 * np.arange(shape[0])[:, None]).astype(np.float64)
    result, reference = ml.steric_profile(ds, variant=list(VARIANTS), regions=xr.DataArray(regions,
                                                                                           dims=lab["areacello"].dims))
    assert type(result).__module__.startswith("xarray") and type(reference).__module__.startswith("xarray")
    want, _ = ml.steric_profile(lab, variant=list(VARIANTS), regions=regions)
    for v in VARIANTS:
        assert result[v].dims == ("time", "region", "z_l")
        assert np.array_equal(np.asarray(result[v].values), np.asarray(want[v].values), equal_nan=True)
    assert np.asarray(result["region"].values).tolist() == [0, 1, 2]
