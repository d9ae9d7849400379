"""GPU parity of setup_reference_state(period=...) against a numpy oracle of its own.

The oracle of the means is a loop over t in fp64 that does what the kernel promises: ``s = s + w * x`` and
``ws = ws + w`` where x is not NaN, each rounded, then ``s / ws``.  So the means must be bit-identical to it on every
route: one launch, plain loads, uneven blocks, T and S chunked at different boundaries, pinned or pageable host memory,
a NaN-poisoned accumulator started with ``first``, launches carried through the accumulator.  ``rho`` is
``oracle.eos`` at the mean state (1e-10 relative), ``volo`` / ``masso`` are ``math.fsum`` over the mean slabs (1e-12
relative), and the heights of every steric entry point with ``reference=`` the period reference are the oracle's with
the mean reference (1e-9 m).

The data has intermittent NaN holes whose patterns differ between T, S and V, land cells that are NaN in every step,
zero weights on some steps and days-in-month weights.
"""

import json
import math
import pathlib
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from momlevel_b200.labeled import ChunkedArray
from oracle import eos as oeos
from oracle import steric as osteric

pytestmark = pytest.mark.gpu

ETA_ATOL = 1e-9  # m
RHO_RTOL = 1e-10
SUM_RTOL = 1e-12
VARIANTS = ("steric", "thermosteric", "halosteric")
DIMS = ("time", "z_l", "yh", "xh")
DAYS = np.array([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], dtype=np.float64)
GRIDS = {"aligned": (6, 8, 16), "ragged": (5, 7, 13), "nz1": (1, 6, 20)}


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


def oracle_means(T, S, V, w=None):
    """The period means: a loop over t in fp64, NaN skipped per field and cell."""
    out = []
    nt = T.shape[0]
    w = np.ones(nt) if w is None else np.asarray(w, dtype=np.float64)
    for x in (T, S, V):
        s = np.zeros(x.shape[1:])
        ws = np.zeros(x.shape[1:])
        for t in range(nt):
            xt = np.asarray(x[t], dtype=np.float64)
            ok = ~np.isnan(xt)
            s[ok] = s[ok] + w[t] * xt[ok]
            ws[ok] = ws[ok] + w[t]
        with np.errstate(invalid="ignore"):
            out.append(s / ws)
    return out


def _case(nt, nz, ny, nx, dtype=np.float32, vdtype=None, seed=0):
    """Fields with intermittent holes (a pattern per field), land columns NaN in every step, and a grid."""
    from momlevel_b200 import synth

    vdtype = dtype if vdtype is None else vdtype
    rng = np.random.default_rng(seed)
    z_i, z_l = synth.vertical_grid(nz)
    land = rng.random((ny, nx)) < 0.2
    land[0, 0] = True
    land[ny // 2, nx // 2] = False
    depth = np.where(land, np.nan, rng.random((ny, nx)) * (z_i[-1] - 10.0) + 10.0)
    dry = np.isnan(depth)[None] | (z_i[:-1, None, None] >= np.nan_to_num(depth)[None])
    area = np.where(land, 0.0, 0.5 + rng.random((ny, nx)))
    area = area / area.sum() * synth.OCEAN_AREA
    T = 2.0 + 18.0 * np.exp(-z_l / 1000.0)[None, :, None, None] + 3.0 * rng.standard_normal((nt, nz, ny, nx))
    S = 35.0 + rng.standard_normal((nt, nz, ny, nx))
    dz = np.minimum(np.clip(np.nan_to_num(depth)[None] - z_i[:-1, None, None], 0.0, None), np.diff(z_i)[:, None, None])
    V = (dz * area)[None] * (1.0 + 0.01 * rng.standard_normal((nt, nz, ny, nx)))
    for x in (T, S, V):
        x[:, dry] = np.nan
        x[rng.random(x.shape) < 0.15] = np.nan  # intermittent holes, independent per field
    T[:, 0, ny // 2, nx // 2] = np.nan  # a wet cell with no temperature in any step
    grid = {"z_i": z_i, "z_l": z_l, "deptho": depth, "areacello": area}
    return grid, T.astype(dtype), S.astype(dtype), V.astype(vdtype)


def _weights(nt, kind):
    if kind is None:
        return None
    w = np.resize(DAYS, nt).copy()
    if kind == "zeros":
        w[1::3] = 0.0
    return w


def _dataset(ml, grid, T, S, V, device="cuda"):
    def put(x):
        t = torch.from_numpy(np.ascontiguousarray(x))
        return t.to(device) if device != "numpy" else np.ascontiguousarray(x)

    nt, nz, ny, nx = T.shape
    ds = ml.Dataset()
    ds["time"] = ml.DataArray(np.arange(nt, dtype=np.float64), ("time",))
    ds["z_l"] = ml.DataArray(put(grid["z_l"]), ("z_l",))
    ds["z_i"] = ml.DataArray(put(grid["z_i"]), ("z_i",))
    ds["yh"] = ml.DataArray(np.arange(ny, dtype=np.float64), ("yh",))
    ds["xh"] = ml.DataArray(np.arange(nx, dtype=np.float64), ("xh",))
    for k, x in (("thetao", T), ("so", S), ("volcello", V)):
        ds[k] = ml.DataArray(put(x), DIMS)
    ds["deptho"] = ml.DataArray(put(grid["deptho"]), ("yh", "xh"))
    ds["areacello"] = ml.DataArray(put(grid["areacello"]), ("yh", "xh"))
    return ds


def _chunked(ml, a, chunks):
    def blocks():
        t = 0
        for n in chunks:
            yield a[t: t + n]
            t += n

    return ChunkedArray(a.shape, a.dtype, chunks, blocks)


def _same_bits(got, want, what=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN pattern differs"
    m = ~np.isnan(want)
    bad = got[m].view(np.int64) != want[m].view(np.int64)
    assert not bad.any(), f"{what}: {int(bad.sum())} cells differ, max {np.abs(got[m] - want[m]).max():.3e}"


def _close_nan(a, b, atol=0.0, rtol=0.0, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: NaN pattern differs"
    m = ~np.isnan(b)
    if m.any():
        err = np.abs(a[m] - b[m])
        assert np.all(err <= atol + rtol * np.abs(b[m])), f"{what}: max err {err.max():.3e}"


def _oracle_reference(grid, means, patm, eos):
    Tm, Sm, Vm = means
    pres = osteric._pres3(grid["z_l"], patm)
    rho = oeos.density(eos, Tm, Sm, pres)
    volo = math.fsum(Vm[~np.isnan(Vm)].tolist())
    mv = rho * Vm
    masso = math.fsum(mv[~np.isnan(mv)].tolist())
    return {"thetao": Tm, "so": Sm, "volcello": Vm, "rho": rho, "volo": volo, "masso": masso, "rhoga": masso / volo,
            "areacello": np.asarray(grid["areacello"])}


def _check_reference(ref, grid, means, patm, eos):
    o = _oracle_reference(grid, means, patm, eos)
    for k in ("thetao", "so", "volcello"):
        _same_bits(ref[k].values, o[k], k)
    _close_nan(ref["rho"].values, np.where(np.isnan(o["rho"]), np.nan, o["rho"]), rtol=RHO_RTOL, what="rho")
    assert abs(float(ref["volo"].values) - o["volo"]) <= SUM_RTOL * abs(o["volo"])
    assert abs(float(ref["masso"].values) - o["masso"]) <= SUM_RTOL * abs(o["masso"])
    return o


# ------------------------------------------------------------------------------------------- oracle parity


CASES = [
    # fields, volcello, eos, patm, grid, weights
    (np.float32, np.float32, "Wright", "scalar", "aligned", "days"),
    (np.float32, np.float32, "Wright", "2d", "ragged", "zeros"),
    (np.float32, np.float32, "linear", "scalar", "nz1", None),
    (np.float64, np.float64, "Wright", "scalar", "ragged", "days"),
    (np.float64, np.float64, "linear", "2d", "aligned", "zeros"),
    (np.float64, np.float32, "Wright", "scalar", "aligned", "zeros"),
    (np.float64, np.float32, "Wright", "2d", "nz1", "days"),
    (np.float32, np.float64, "linear", "scalar", "ragged", None),
]


@pytest.mark.parametrize("fdt, vdt, eos, patm_kind, grid_name, wkind", CASES,
                         ids=[f"{np.dtype(c[0]).name}-v{np.dtype(c[1]).name}-{c[2]}-{c[3]}-{c[4]}-{c[5]}" for c in CASES])
@pytest.mark.parametrize("storage", ["device", "numpy", "chunked"])
def test_period_reference_matches_the_oracle(ml, fdt, vdt, eos, patm_kind, grid_name, wkind, storage):
    nz, ny, nx = GRIDS[grid_name]
    grid, T, S, V = _case(14, nz, ny, nx, fdt, vdt, seed=nz * 100 + nx)
    start, stop = 1, 12
    w = _weights(stop - start, wkind)
    patm = 101325.0 if patm_kind == "scalar" else 101325.0 + 500.0 * np.random.default_rng(1).random((ny, nx))
    ds = _dataset(ml, grid, T, S, V, device="cuda" if storage == "device" else "numpy")
    if storage == "chunked":
        ds["thetao"] = ml.DataArray(_chunked(ml, T, (1, 4, 2, 5, 2)), DIMS)
        ds["so"] = ml.DataArray(_chunked(ml, S, (3, 3, 3, 3, 2)), DIMS)
    ref = ml.reference.setup_reference_state(ds, patm=patm, eos=eos, period=slice(start, stop), period_weights=w)
    means = oracle_means(T[start:stop], S[start:stop], V[start:stop], w)
    _check_reference(ref, grid, means, patm, eos)
    assert ref.attrs["reference_period"] == f"{start}:{stop}"
    if storage == "chunked":
        assert ds["thetao"]._data.blocks_read == 4 and ds["so"]._data.blocks_read == 4  # nothing past step 11


def test_a_cell_with_no_value_is_nan_and_zero_weights_drop_steps(ml):
    grid, T, S, V = _case(6, 4, 8, 16, seed=3)
    T[:, 1, 2, 3] = np.nan
    T[0, 1, 2, 4] = np.nan
    T[1:, 1, 2, 4] = 5.0
    T[:, 1, 2, 5] = np.arange(6, dtype=np.float32)
    w = np.array([1.0, 0.0, 0.0, 2.0, 0.0, 0.0])
    ref = ml.reference.setup_reference_state(_dataset(ml, grid, T, S, V), period=slice(0, 6), period_weights=w)
    got = ref["thetao"].values
    assert np.isnan(got[1, 2, 3])
    assert np.isnan(got[0, 0, 0])  # land
    assert got[1, 2, 4] == 5.0  # only step 3 has weight and a value
    assert got[1, 2, 5] == 2.0  # (0 * 1 + 3 * 2) / 3


# ------------------------------------------------------------------------------------- bits across routes


def _core_means(ml, T, S, V, w=None, **kw):
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    wt = dev(w) if w is not None else None
    return [m.cpu().numpy() for m in ml.core.mean_state(dev(T), dev(S), dev(V), weights=wt, **kw)]


@pytest.mark.parametrize("fdt, vdt", [(np.float32, np.float32), (np.float64, np.float64), (np.float64, np.float32)])
def test_means_are_the_same_bits_on_every_route(ml, fdt, vdt):
    grid, T, S, V = _case(12, 6, 8, 16, fdt, vdt, seed=7)
    w = _weights(12, "zeros")
    want = oracle_means(T, S, V, w)
    one = _core_means(ml, T, S, V, w)
    for a, b, k in zip(one, want, "TSV"):
        _same_bits(a, b, f"one launch {k}")
    prev = ml.core.force_direct(1)
    try:
        plain = _core_means(ml, T, S, V, w)
    finally:
        ml.core.force_direct(prev)
    for a, b, k in zip(plain, want, "TSV"):
        _same_bits(a, b, f"plain loads {k}")
    # bases that are not 16-byte aligned take the plain loads
    dev = []
    for x in (T, S, V):
        flat = torch.empty(x.size + 1, dtype=torch.from_numpy(x).dtype, device="cuda")
        view = flat[1:].view(x.shape)
        view.copy_(torch.from_numpy(x))
        dev.append(view)
    off = ml.core.mean_state(*dev, weights=torch.from_numpy(w).cuda())
    for a, b, k in zip(off, want, "TSV"):
        _same_bits(a.cpu().numpy(), b, f"unaligned {k}")
    # uneven blocks through the accumulator, pinned and pageable host memory
    for lens in ([1, 4, 2, 5], [12], [5, 7]):
        for pinned in (False, True):
            def pieces():
                t = 0
                for n in lens:
                    blk = [torch.from_numpy(np.ascontiguousarray(x[t: t + n])) for x in (T, S, V)]
                    yield [b.pin_memory() for b in blk] if pinned else [b.numpy() for b in blk]
                    t += n

            dt = torch.float32 if fdt == np.float32 else torch.float64
            vt = torch.float32 if vdt == np.float32 else torch.float64
            got = ml.core.mean_state_blocks(pieces(), T.shape[1:], dt, vt, weights=w, max_steps=max(lens))
            for a, b, k in zip(got, want, "TSV"):
                _same_bits(a.cpu().numpy(), b, f"blocks {lens} pinned={pinned} {k}")


def test_poisoned_accumulator_and_long_calls(ml):
    grid, T, S, V = _case(1030, 2, 3, 8, seed=11)
    w = np.resize(DAYS, 1030)
    want = oracle_means(T, S, V, w)
    dev = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()  # noqa: E731
    Td, Sd, Vd, wd = dev(T), dev(S), dev(V), dev(w)
    nbytes = ml.core.mean_state_bytes(2, 24)
    assert nbytes == 6 * 8 * 2 * 24
    acc = torch.full((nbytes // 8,), float("nan"), dtype=torch.float64, device="cuda")
    # `first` does not read the accumulator, whatever it holds
    ml.core.mean_state_accumulate(Td[:3], Sd[:3], Vd[:3], wd[:3], acc, first=True, last=False)
    ml.core.mean_state_accumulate(Td[3:700], Sd[3:700], Vd[3:700], wd[3:700], acc, first=False, last=False)
    got = ml.core.mean_state_accumulate(Td[700:], Sd[700:], Vd[700:], wd[700:], acc, first=False, last=True)
    for a, b, k in zip(got, want, "TSV"):
        _same_bits(a.cpu().numpy(), b, f"three calls {k}")
    # one call longer than a launch takes (1024 steps): launches carry the sums through the accumulator
    for direct in (0, 1):
        prev = ml.core.force_direct(direct)
        try:
            got = ml.core.mean_state(Td, Sd, Vd, weights=wd)
        finally:
            ml.core.force_direct(prev)
        for a, b, k in zip(got, want, "TSV"):
            _same_bits(a.cpu().numpy(), b, f"1030 steps direct={direct} {k}")


def test_one_step_period_is_the_time_index_reference(ml):
    grid, T, S, V = _case(5, 6, 8, 16, seed=5)
    up = _dataset(ml, grid, T.astype(np.float64), S.astype(np.float64), V.astype(np.float64))
    ds = _dataset(ml, grid, T, S, V)
    for i in (0, 3):
        a = ml.reference.setup_reference_state(ds, period=slice(i, i + 1))
        b = ml.reference.setup_reference_state(up, time_index=i)
        for k in ("thetao", "so", "volcello", "rho"):
            _same_bits(a[k].values, b[k].values, f"{k} step {i}")
        for k in ("volo", "masso", "rhoga"):
            assert float(a[k].values) == float(b[k].values), k


# -------------------------------------------------------------------------------------- the kernel per route


_ROUTE_PROBE = """
import json, re, sys
import numpy as np
import torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import momlevel_b200 as ml
import test_gpu_mean_reference as t

def kernels(fn):
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({m.group(1) for e in prof.events() for m in [re.search(r"\\b(k_\\w+)", e.name)] if m})

out = {}
for name, shape in (("aligned", (4, 8, 16)), ("ragged", (4, 7, 13))):
    grid, T, S, V = t._case(6, *shape, seed=2)
    out[name] = kernels(lambda: t._core_means(ml, T, S, V))
    ml.core.force_direct(1)
    out[name + "_direct"] = kernels(lambda: t._core_means(ml, T, S, V))
    ml.core.force_direct(0)
print(json.dumps(out))
"""


def test_kernel_per_route(ml):
    """The vector kernel takes aligned rows; ragged rows and ml_set_force_direct(1) take the plain loads.  The
    profiler runs in an interpreter of its own, so what earlier tests did in this process does not decide it."""
    root = pathlib.Path(__file__).resolve().parent.parent
    res = subprocess.run([sys.executable, "-c", _ROUTE_PROBE, str(root)], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    got = json.loads(res.stdout.strip().splitlines()[-1])
    assert got["aligned"] == ["k_mean_state_vec"], got
    assert got["aligned_direct"] == ["k_mean_state"], got
    assert got["ragged"] == ["k_mean_state"], got
    assert got["ragged_direct"] == ["k_mean_state"], got


# ------------------------------------------------------------------------------------------ end to end


def _heights(ml, ds, ref, chunked):
    out = {}
    for v in VARIANTS:
        for dom in ("local", "global"):
            r, _ = ml.steric(ds, variant=v, domain=dom, reference=ref)
            out[("steric", v, dom)] = np.asarray(r[v].values)
    for dom in ("local", "global"):
        r, _ = ml.steric_variants(ds, reference=ref, domain=dom)
        for v in VARIANTS:
            out[("steric_variants", v, dom)] = np.asarray(r[v].values)
    if not chunked:  # steric_layers and steric_profile take whole arrays only
        r, _ = ml.steric_layers(ds, depth_edges=(0, None), variant=list(VARIANTS), reference=ref)
        for v in VARIANTS:
            out[("steric_layers", v, "local")] = np.asarray(r[v].values)[:, 0]
        r, _ = ml.steric_profile(ds, variant=list(VARIANTS), reference=ref)
        for v in VARIANTS:
            out[("steric_profile", v, "local")] = np.asarray(r[v].values)
    return out


@pytest.mark.parametrize("fdt", [np.float32, np.float64])
@pytest.mark.parametrize("storage", ["device", "chunked"])
def test_steric_with_a_period_reference(ml, fdt, storage):
    from momlevel_b200 import synth

    nt = 12
    ds0 = synth.make_dataset(nt, 8, 10, 16, seed=4, device="cpu", dtype=torch.float32)
    T, S = (np.asarray(ds0[k].values).astype(fdt) for k in ("thetao", "so"))
    V = np.ascontiguousarray(np.asarray(ds0["volcello"].values)).astype(fdt)
    T[3, 2, 4, 5] = np.nan  # an intermittent hole: the mean of that cell skips a step
    grid = {k: np.asarray(ds0[k].values, dtype=np.float64) for k in ("z_i", "z_l", "deptho", "areacello")}
    w = DAYS.copy()
    ds = _dataset(ml, grid, T, S, V, device="cuda" if storage == "device" else "numpy")
    if storage == "chunked":
        ds["thetao"] = ml.DataArray(_chunked(ml, T, (4, 4, 4)), DIMS)
        ds["so"] = ml.DataArray(_chunked(ml, S, (6, 6)), DIMS)
    ref = ml.reference.setup_reference_state(ds, period=slice(0, nt), period_weights=w)
    o = _check_reference(ref, grid, oracle_means(T, S, V, w), 101325.0, "Wright")
    T64, S64 = T.astype(np.float64), S.astype(np.float64)
    want = {}
    for v in VARIANTS:
        want[(v, "local")] = osteric.steric_local(T64, S64, grid["z_l"], grid["z_i"], grid["deptho"], o, variant=v)[0]
        want[(v, "global")] = osteric.steric_global(T64, S64, grid["z_l"], o, variant=v)[0]
    got = _heights(ml, ds, ref, storage == "chunked")
    from profile_oracle import steric_profile as oprofile

    for (func, v, dom), val in got.items():
        if func == "steric_profile":
            want_p, scale = oprofile(T64, S64, grid["z_l"], grid["z_i"], grid["deptho"], o, variant=v)
            assert np.all(np.abs(val - want_p) <= 1e-12 + 1e-10 * scale), (func, v)
            continue
        _close_nan(val, want[(v, dom)], atol=ETA_ATOL, what=f"{func} {v} {dom}")
