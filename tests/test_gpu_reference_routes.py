"""GPU parity of the supplied-reference routes and of the host path against the oracle.

A reference state can come from anywhere -- a climatology, fp64 arithmetic, another run -- so it need not be stored
like the fields.  Every route a call can take (device-resident fields, host-resident fields streamed through device
windows, fields that arrive block by block) must give the oracle's heights and masses for it.  The host path itself
(``ml_steric_local_host``, ``ml_host_stream_*``) is checked over storage, equation of state, ``rhozero``, grid,
packing mode, packing threads, window width and pinned or pageable memory.

Tolerances are the suite's: 1e-9 m on heights, 1e-10 relative on density, 1e-12 relative on volumes and masses.
Two routes that run different kernel families agree within ``1e-11 + 1e-13 * scale``; a packed transfer gives the
bits of a dense one.
"""

import importlib
import itertools

import numpy as np
import pytest
import torch

from oracle import steric as osteric

pytestmark = pytest.mark.gpu

ETA_ATOL = 1e-9  # m
RHO_RTOL = 1e-10
SUM_RTOL = 1e-12
VARIANTS = ("steric", "thermosteric", "halosteric")
DIMS = ("time", "z_l", "yh", "xh")
NP = {"f32": np.float32, "f64": np.float64}
TORCH = {"f32": torch.float32, "f64": torch.float64}


@pytest.fixture(scope="module")
def ml():
    import momlevel_b200

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return momlevel_b200


@pytest.fixture(autouse=True)
def _default_packing(ml):
    yield
    ml.core.host_packing(1)


def _close_nan(a, b, atol=0.0, rtol=0.0, what=""):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: NaN pattern differs"
    m = ~np.isnan(b)
    if m.any():
        err = np.abs(a[m] - b[m])
        assert np.all(err <= atol + rtol * np.abs(b[m])), f"{what}: max err {err.max():.3e}"


def _families_agree(a, b, what=""):
    """Two routes that may run different kernel families: fp64 accuracy, ~1e-12 m where a height is a residue."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)), what
    err = float(np.max(np.abs(np.nan_to_num(a - b)), initial=0.0))
    scale = float(np.max(np.abs(np.nan_to_num(b)), initial=0.0))
    assert err <= 1e-11 + 1e-13 * scale, f"{what}: {err:.3e} at scale {scale:.3e}"


def _bits(a, b, what=""):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    assert a.shape == b.shape and torch.equal(a.view(torch.int64), b.view(torch.int64)), what


def _disagreeing_masks(ds, seed):
    """Host fields whose volcello mask, bathymetry and data holes disagree, with junk T/S under missing volumes."""
    T, S = ds["thetao"].data.clone(), ds["so"].data.clone()
    V = ds["volcello"].data[0].clone()
    depth = ds["deptho"].data.clone()
    shape = tuple(T.shape)
    g = torch.Generator().manual_seed(seed)
    for k in range(40):
        t, z, y, x = (int(torch.randint(0, n, (1,), generator=g)) for n in shape)
        (T if k % 2 else S)[t, z, y, x] = float("nan")
    for _ in range(30):
        z, y, x = (int(torch.randint(0, n, (1,), generator=g)) for n in shape[1:])
        V[z, y, x] = float("nan") if torch.isfinite(V[z, y, x]) else 1.0e9
    for _ in range(12):
        y, x = (int(torch.randint(0, n, (1,), generator=g)) for n in shape[2:])
        depth[y, x] = float("nan") if torch.isfinite(depth[y, x]) else 3000.0
    # data where the reference volume is missing: the reference never reads it, the packed rows never carry it
    junk = torch.isnan(V).unsqueeze(0) & (torch.rand(shape, generator=g) < 0.3)
    T[junk] = 25.0
    S[junk] = 31.0
    return T, S, V, depth


def _off_fp32_grid(x, seed):
    """fp64 values that are not fp32 values (synth draws its fields in fp32): a relative nudge of ~1e-9."""
    g = torch.Generator().manual_seed(seed)
    return x * (1.0 + 1.0e-9 * torch.rand(x.shape, generator=g, dtype=torch.float64))


def _chunked_dataset(ml, ds, chunks):
    """The same Dataset with thetao / so / volcello held as blocks along time (what dask-backed variables are)."""
    from momlevel_b200.labeled import ChunkedArray

    out = ds.copy()
    for name in ("thetao", "so", "volcello"):
        full = np.ascontiguousarray(ds[name].values)
        cuts = np.cumsum((0,) + tuple(chunks))

        def blocks(full=full, cuts=cuts):
            for a, b in zip(cuts[:-1], cuts[1:]):
                yield np.array(full[a:b])

        out[name] = ml.DataArray(ChunkedArray(full.shape, full.dtype, chunks, blocks), ds[name].dims, attrs=ds[name].attrs)
    return out


# ------------------------------------------------------------------------ a. supplied references, every route

ROUTE_GRIDS = {"tma": (5, 30, 12, 100), "ragged": (5, 30, 37, 53)}  # fp32 ncol 1200: TMA family; ncol 1961: ragged
CHUNKS = (1, 3, 1)


def _time_mean_reference(ml, ds, ref_dt):
    """A reference that is not step 0: the fp64 time mean of the fields, stored as ``ref_dt``; the volume is the
    fields' own, ``rho`` is the oracle's.  Returns ``(Dataset, oracle reference dict)``."""
    f64 = lambda k: ds[k].values.astype(np.float64)  # noqa: E731
    T, S = f64("thetao"), f64("so")
    Tm, Sm = T.mean(0).astype(NP[ref_dt]), S.mean(0).astype(NP[ref_dt])
    V0 = np.ascontiguousarray(ds["volcello"].values[0])
    o = osteric.reference_state(Tm[None].astype(np.float64), Sm[None].astype(np.float64), V0[None].astype(np.float64),
                                f64("areacello"), f64("z_l"))
    ref = ml.Dataset()
    for k, v in (("thetao", Tm), ("so", Sm), ("volcello", V0), ("rho", o["rho"])):
        ref[k] = ml.DataArray(v, DIMS[1:])
    for k in ("volo", "masso", "rhoga"):
        ref[k] = ml.DataArray(np.float64(o[k]), ())
    ref["areacello"] = ds["areacello"]
    return ref, o


def _route_datasets(ml, ds):
    dev, host = ds.copy(), ds.copy()
    for k in ("thetao", "so", "volcello"):
        dev[k] = ml.DataArray(ds[k].data.cuda().contiguous(), DIMS)
        host[k] = ml.DataArray(np.ascontiguousarray(ds[k].values), DIMS)
    for k in ("deptho", "areacello", "z_l", "z_i"):
        dev[k] = ml.DataArray(torch.as_tensor(ds[k].values).cuda(), ds[k].dims)
    return {"device": dev, "host": host, "chunked": _chunked_dataset(ml, host, CHUNKS)}


def _every_call(ml, d, ref, route):
    out = {}
    for v in VARIANTS:
        for dom in ("local", "global"):
            r, _ = ml.steric(d, variant=v, domain=dom, reference=ref)
            out[("steric", v, dom)] = r[v].values
    for dom in ("local", "global"):
        r, _ = ml.steric_variants(d, reference=ref, domain=dom)
        for v in VARIANTS:
            out[("steric_variants", v, dom)] = r[v].values
    if route != "chunked":  # steric_layers takes whole arrays only
        r, _ = ml.steric_layers(d, depth_edges=(0, None), variant=list(VARIANTS), reference=ref)
        for v in VARIANTS:
            assert r[v].shape[1] == 1
            out[("steric_layers", v, "local")] = r[v].values[:, 0]
    return out


@pytest.mark.parametrize("grid", sorted(ROUTE_GRIDS))
@pytest.mark.parametrize("fields,refdt", [("f32", "f64"), ("f64", "f32"), ("f32", "f32"), ("f64", "f64")])
def test_supplied_reference_on_every_route(ml, monkeypatch, grid, fields, refdt):
    """A reference stored unlike the fields gives the oracle's heights and masses on every entry point and route:
    an fp64 reference with fp32 fields is used as it is, not rounded to the fields' dtype."""
    from momlevel_b200 import synth

    steric_mod = importlib.import_module("momlevel_b200.steric")
    monkeypatch.setattr(steric_mod, "HOST_ROUTE_MIN_BYTES", 0)
    ds = synth.make_dataset(*ROUTE_GRIDS[grid], seed=3, device="cpu", dtype=TORCH[fields])
    if fields == "f64":
        for i, k in enumerate(("thetao", "so")):
            ds[k] = ml.DataArray(_off_fp32_grid(ds[k].data, i), DIMS)
    ref, o = _time_mean_reference(ml, ds, refdt)
    f64 = lambda k: ds[k].values.astype(np.float64)  # noqa: E731
    T, S, z_l, z_i, depth = f64("thetao"), f64("so"), f64("z_l"), f64("z_i"), f64("deptho")
    want = {}
    for v in VARIANTS:
        want[(v, "local")] = osteric.steric_local(T, S, z_l, z_i, depth, o, variant=v)[0]
        want[(v, "global")] = osteric.steric_global(T, S, z_l, o, variant=v)[0]
    if refdt == "f64":
        # the fixture can tell a used reference from one rounded to fp32
        r32 = dict(o, thetao=o["thetao"].astype(np.float32).astype(np.float64),
                   so=o["so"].astype(np.float32).astype(np.float64))
        rounded = osteric.steric_local(T, S, z_l, z_i, depth, r32, variant="thermosteric")[0]
        assert np.nanmax(np.abs(rounded - want[("thermosteric", "local")])) > 100 * ETA_ATOL
    routes = _route_datasets(ml, ds)
    got = {route: _every_call(ml, d, ref, route) for route, d in routes.items()}
    single = {key[1:]: val for key, val in got["device"].items() if key[0] == "steric"}  # the single-variant device call
    for route, results in got.items():
        for (func, v, dom), val in results.items():
            what = f"{route} {func} {v} {dom}"
            if dom == "local":
                _close_nan(val, want[(v, dom)], atol=ETA_ATOL, what=what)
            else:
                assert val.shape == want[(v, dom)].shape and np.all(np.isfinite(val)), what
                assert np.max(np.abs(val - want[(v, dom)])) < ETA_ATOL, what
            _families_agree(val, single[(v, dom)], what=what)


# -------------------------------------------------------------------------------- b. the host path itself

HOST_GRIDS = {  # (nz, ny, nx); 5 steps each
    "ncol35": (75, 5, 7),         # fewer columns than a tile: the direct family
    "ncol1000": (1, 10, 100),     # aligned rows, a partial last 32-column presence group
    "ncol1961": (12, 37, 53),     # ragged rows: rank-1-map kernels, two unpack blocks per row, a partial group
    "ncol133385": (3, 259, 515),  # ragged, three 64 K-column packing segments, a partial group
}
NT = 5
STORAGES = ("f32/f32", "f64/f64", "f32/f64", "f64/f32")  # fields / reference volume
AXES = {
    "storage": STORAGES,
    "grid": tuple(HOST_GRIDS),
    "eos": ("Wright", "linear"),
    "rhozero": (1035.0, 1025.0),
    "mode": (1, 2, 3, 4),
    "threads": (0, 1, 3),
    "window": (1, 2, NT),
    "src_pinned": (False, True),
    "out_pinned": (False, True),
}


def _pairwise(axes, seed):
    """A seeded greedy covering of every pair of values of two axes: a few dozen cases instead of the product."""
    rng = np.random.default_rng(seed)
    names = list(axes)
    sizes = [len(axes[k]) for k in names]
    pairs = lambda c: {(i, c[i], j, c[j]) for i, j in itertools.combinations(range(len(names)), 2)}  # noqa: E731
    uncovered = set()
    for i, j in itertools.combinations(range(len(names)), 2):
        uncovered |= {(i, a, j, b) for a in range(sizes[i]) for b in range(sizes[j])}
    cases = []
    while uncovered:
        todo = sorted(uncovered)
        best, gain = None, -1
        for _ in range(48):
            c = [int(rng.integers(n)) for n in sizes]
            i, a, j, b = todo[int(rng.integers(len(todo)))]
            c[i], c[j] = a, b
            g = len(pairs(c) & uncovered)
            if g > gain:
                best, gain = c, g
        uncovered -= pairs(best)
        cases.append({k: axes[k][v] for k, v in zip(names, best)})
    return cases


HOST_CASES = _pairwise(AXES, seed=2024)
_HOST_DATA = {}


def _host_data(ml, storage, grid, eos, rhozero):
    """Masked fields of one storage and grid, and the oracle's heights, masses and scalars for them (cached)."""
    from momlevel_b200 import synth

    key = (storage, grid, eos, rhozero)
    if key in _HOST_DATA:
        return _HOST_DATA[key]
    fdt, vdt = storage.split("/")
    ds = synth.make_dataset(NT, *HOST_GRIDS[grid], seed=17, device="cpu", dtype=TORCH[fdt])
    T, S, V, depth = _disagreeing_masks(ds, seed=5)
    if fdt == "f64":
        T, S = _off_fp32_grid(T, 1), _off_fp32_grid(S, 2)
    if vdt != fdt:
        # a volume stored unlike the fields; an fp64 one is not fp32-representable, so indexing it as fp32 shows
        V = V.double() * (1.0 + 2.0**-30) if vdt == "f64" else V.float()
    z_l, z_i = ds["z_l"].values.astype(np.float64), ds["z_i"].values.astype(np.float64)
    T64, S64, V64 = T.double().numpy(), S.double().numpy(), V.double().numpy()
    o = osteric.reference_state(T64, S64, V64[None], ds["areacello"].values, z_l, eos=eos)
    eta = {v: osteric.steric_local(T64, S64, z_l, z_i, depth.numpy(), o, rhozero=rhozero, eos=eos, variant=v)[0]
           for v in VARIANTS}
    masso = osteric.steric_global(T64, S64, z_l, o, eos=eos)[2]
    data = dict(T=T, S=S, V=V, depth=depth.numpy(), z_i=z_i, p=z_l * 1.0e4 + 101325.0, o=o, eta=eta, masso=masso)
    _HOST_DATA.clear()  # one grid at a time is enough: the cases are not ordered by grid
    _HOST_DATA[key] = data
    return data


def _stream_through(hs, T, S, w):
    """Push ``T, S`` in blocks of ``w`` steps; the outputs of every block, complete (after ``finish``)."""
    try:
        blocks = [hs.push(T[t:t + w], S[t:t + w]) for t in range(0, T.shape[0], w)]
        rho, sums = hs.finish()
    finally:
        hs.abort()  # after a failure: this thread may open the next stream
    return {v: torch.cat([b[v] for b in blocks]) for v in hs.variants}, rho, sums


def _run_host(ml, case, d, mode):
    """Heights of the three variants, reference scalars, steric masses and ``host_last_transfer()`` of the local and
    the global call."""
    core = ml.core
    core.host_packing(mode, case["threads"])
    storage, w, eos, rz = case["storage"], case["window"], case["eos"], case["rhozero"]
    T, S, V = d["T"], d["S"], d["V"]
    if case["src_pinned"]:
        T, S, V = T.pin_memory(), S.pin_memory(), V.pin_memory()
    hshape = tuple(T.shape[2:])
    if storage != "f32/f64":
        # whole arrays: ml_steric_local_variants_host (an fp32 volume with fp64 fields is promoted first)
        outs = None
        if case["out_pinned"]:
            outs = {v: torch.empty((NT,) + hshape, dtype=torch.float64).pin_memory() for v in VARIANTS}
        etas, _, sums = core.steric_local_host(T, S, V, d["z_i"], d["depth"], d["p"], rhozero=rz, eos=eos,
                                               steps_per_window=w, variants=True, eta_out=outs)
        if outs is not None:
            assert all(etas[v] is outs[v] for v in VARIANTS)
        local = core.host_last_transfer()
        masso = core.steric_global_host(T, S, V, d["p"], eos=eos, steps_per_window=w)
        return etas, sums, masso, local, core.host_last_transfer(), None
    # fp32 fields with an fp64 volume: only the stream takes a volume stored unlike the fields
    hs = core.HostStream("local", V, d["p"], z_i=d["z_i"], deptho=d["depth"], variants=VARIANTS, rhozero=rz, eos=eos,
                         max_block_steps=w, dtype=torch.float32)
    etas, _, sums = _stream_through(hs, T, S, w)
    path = core.last_path()
    local = core.host_last_transfer()
    hs = core.HostStream("global", V, d["p"], variants=("steric",), eos=eos, max_block_steps=w, dtype=torch.float32)
    masso = _stream_through(hs, T, S, w)[0]["steric"]
    return etas, sums, masso, local, core.host_last_transfer(), path


@pytest.mark.parametrize("case", HOST_CASES, ids=lambda c: "-".join(str(c[k]) for k in AXES))
def test_host_path_matrix(ml, case):
    """Every cell: the oracle's heights, scalars and masses, and the bits of the same call with packing off."""
    d = _host_data(ml, case["storage"], case["grid"], case["eos"], case["rhozero"])
    etas0, sums0, masso0, (bytes0, f0l), (_, f0g), _ = _run_host(ml, case, d, 0)
    etas, sums, masso, (nbytes, fl), (_, fg), path = _run_host(ml, case, d, case["mode"])
    assert f0l == f0g == 0.0
    for v in VARIANTS:
        _close_nan(etas[v].numpy(), d["eta"][v], atol=ETA_ATOL, what=v)
        _bits(etas[v], etas0[v], what=f"{v}: packed against dense")
    assert sums == sums0
    assert sums[0] == pytest.approx(d["o"]["volo"], rel=SUM_RTOL)
    assert sums[1] == pytest.approx(d["o"]["masso"], rel=SUM_RTOL)
    assert np.allclose(masso.numpy(), d["masso"], rtol=SUM_RTOL, atol=0)
    _bits(masso, masso0, what="masses: packed against dense")
    if case["storage"] == "f32/f32" and not case["src_pinned"]:
        # from pageable memory every row crosses packed, as exactly its present cells
        assert fl == 1.0
        assert nbytes == _packed_bytes(bytes0, d["V"], NT)
    if case["storage"] != "f32/f32":
        # fp64 storage or a volume stored unlike the fields: every row crosses as it is
        assert fl == fg == 0.0
    if case["storage"] == "f32/f64":
        assert path == 1, "a volume stored unlike the fields takes the direct family"


def _packed_bytes(dense_bytes, V, nt):
    """Host-to-device bytes of a local fp32 call whose rows all cross packed, from those of the dense call: T and S
    of the cells whose reference volume is present, the level offsets and one flag per row instead of whole rows."""
    nz, ncol = V.shape[0], V[0].numel()
    present = int((~torch.isnan(V)).sum())
    return dense_bytes - 2 * 4 * nt * nz * ncol + 2 * 4 * nt * present + 8 * (nz + 1) + nt * nz


def test_host_packed_fraction(ml):
    """Packing applies to masked fp32 rows only: it is off for fp64 storage, a volume stored unlike the fields and a
    call that wants rho_ref back, and it compresses rows in mode 2 from pinned memory."""
    core = ml.core
    d = _host_data(ml, "f32/f32", "ncol1961", "Wright", 1035.0)
    T, S, V = d["T"].pin_memory(), d["S"].pin_memory(), d["V"].pin_memory()
    args = (d["z_i"], d["depth"], d["p"])
    core.host_packing(0)
    eta0, _, _ = core.steric_local_host(T, S, V, *args)
    core.host_packing(2)
    eta, _, _ = core.steric_local_host(T, S, V, *args)
    assert core.host_last_transfer()[1] > 0.0
    _bits(eta, eta0)
    core.host_packing(0)
    core.steric_local_host(d["T"], d["S"], d["V"], *args)
    dense_bytes = core.host_last_transfer()[0]
    core.host_packing(2)
    eta, _, _ = core.steric_local_host(d["T"], d["S"], d["V"], *args)  # pageable: every row packed
    assert core.host_last_transfer() == (_packed_bytes(dense_bytes, d["V"], NT), 1.0)
    _bits(eta, eta0)
    eta, rho, _ = core.steric_local_host(T, S, V, *args, want_rho_ref=True)
    assert core.host_last_transfer()[1] == 0.0
    _bits(eta, eta0)
    _close_nan(rho.numpy(), d["o"]["rho"], rtol=RHO_RTOL)
    eta, _, _ = core.steric_local_host(T.double(), S.double(), V.double(), *args)
    assert core.host_last_transfer()[1] == 0.0
    _close_nan(eta.numpy(), d["eta"]["steric"], atol=ETA_ATOL)
    hs = core.HostStream("local", V.double().pin_memory(), d["p"], z_i=d["z_i"], deptho=d["depth"], max_block_steps=NT)
    out, _, _ = _stream_through(hs, T, S, NT)
    assert core.host_last_transfer()[1] == 0.0
    _close_nan(out["steric"].numpy(), d["eta"]["steric"], atol=ETA_ATOL)


# ------------------------------------------------------------------------------------- core.HostStream directly

SUBSETS = [s for n in (1, 2, 3) for s in itertools.combinations(VARIANTS, n)]
STREAM_BLOCKS = (1, 3, 2, 1)


@pytest.fixture(scope="module")
def stream_case(ml):
    """fp32 fields on a masked 1000-column grid; a supplied fp64 reference (the time mean, not fp32-representable)."""
    from momlevel_b200 import synth

    ds = synth.make_dataset(sum(STREAM_BLOCKS), 12, 20, 50, seed=23, device="cpu", dtype=torch.float32)
    T, S, V, depth = _disagreeing_masks(ds, seed=9)
    z_l, z_i = ds["z_l"].values.astype(np.float64), ds["z_i"].values.astype(np.float64)
    p = z_l * 1.0e4 + 101325.0
    T64, S64, V64 = T.double().numpy(), S.double().numpy(), V.double().numpy()
    area = ds["areacello"].values
    self_o = osteric.reference_state(T64, S64, V64[None], area, z_l)
    Tm, Sm = T64.mean(0), S64.mean(0)
    sup_o = osteric.reference_state(Tm[None], Sm[None], V64[None], area, z_l)
    want = {}
    for name, o in (("self", self_o), ("supplied", sup_o)):
        for v in VARIANTS:
            want[(name, v, "local")] = osteric.steric_local(T64, S64, z_l, z_i, depth.numpy(), o, variant=v)[0]
            want[(name, v, "global")] = osteric.steric_global(T64, S64, z_l, o, variant=v)[2]
    Td, Sd, Vd = T.cuda(), S.cuda(), V.cuda()
    dev = {}
    etas, _, _ = ml.core.steric_local_variants(Td, Sd, Vd, z_i, depth.numpy(), p)
    m, _ = ml.core.steric_global_variants(Td, Sd, Vd, p)
    for v in VARIANTS:
        dev[("self", v, "local")], dev[("self", v, "global")] = etas[v].cpu().numpy(), m[v].cpu().numpy()
    etas, _, _ = ml.core.steric_local_variants(Td, Sd, Vd, z_i, depth.numpy(), p, T_ref=Tm, S_ref=Sm, rho_ref=sup_o["rho"])
    m, _ = ml.core.steric_global_variants(Td, Sd, Vd, p, T_ref=Tm, S_ref=Sm)
    for v in VARIANTS:
        dev[("supplied", v, "local")], dev[("supplied", v, "global")] = etas[v].cpu().numpy(), m[v].cpu().numpy()
    return dict(T=T, S=S, V=V, depth=depth.numpy(), z_i=z_i, p=p, self_o=self_o, sup_o=sup_o, Tm=Tm, Sm=Sm, want=want,
                dev=dev)


@pytest.mark.parametrize("ref", ["self", "supplied"])
@pytest.mark.parametrize("domain", ["local", "global"])
@pytest.mark.parametrize("subset", SUBSETS, ids="+".join)
def test_host_stream_variant_subsets(ml, stream_case, subset, domain, ref):
    """Any subset of the variants, either domain, step 0 or a supplied fp64 reference, pushed in uneven blocks that
    start with a single step: the oracle's heights or masses and those of the device-resident calls."""
    c = stream_case
    local = domain == "local"
    reference = None
    if ref == "supplied":
        reference = {"thetao": c["Tm"], "so": c["Sm"], "rho": c["sup_o"]["rho"]}
    want_rho = local and ref == "self" and len(subset) % 2 == 1  # rho_ref back from some of the self-reference streams
    hs = ml.core.HostStream(domain, c["V"], c["p"], z_i=c["z_i"] if local else None, deptho=c["depth"] if local else None,
                            variants=subset, reference=reference, max_block_steps=max(STREAM_BLOCKS),
                            want_rho_ref=want_rho, want_sums=ref == "self")
    outs, t = [], 0
    try:
        for n in STREAM_BLOCKS:
            outs.append(hs.push(c["T"][t:t + n].numpy(), c["S"][t:t + n].numpy()))
            t += n
        rho, sums = hs.finish()
    finally:
        hs.abort()  # after a failure: this thread may open the next stream
    # an fp64 reference is not rounded to the fp32 fields: the stream runs in fp64
    assert hs.dtype == (torch.float64 if ref == "supplied" else torch.float32)
    for v in subset:
        got = torch.cat([o[v] for o in outs]).numpy()
        want = c["want"][(ref, v, domain)]
        if local:
            _close_nan(got, want, atol=ETA_ATOL, what=v)
        else:
            assert np.allclose(got, want, rtol=SUM_RTOL, atol=0), v
        _families_agree(got, c["dev"][(ref, v, domain)], what=v)
    assert all(set(o) == set(subset) for o in outs)
    if ref == "self":
        o = c["self_o"]
        assert sums[0] == pytest.approx(o["volo"], rel=SUM_RTOL) and sums[1] == pytest.approx(o["masso"], rel=SUM_RTOL)
    else:
        assert sums is None
    if want_rho:
        _close_nan(rho.numpy(), c["self_o"]["rho"], rtol=RHO_RTOL)
    else:
        assert rho is None
