"""steric.py -- local and global steric sea level (mirrors ``src/momlevel/steric.py:17-196``).

Same signature, same result/reference Datasets, same errors.  The hot loop -- equation of
state, density anomaly, bathymetry-clipped column integral, or the volume-weighted global
sum -- is one fused CUDA kernel per call (``ml_steric_local`` / ``ml_steric_global``); the
4-D ``delta_rho`` field is produced on first access so a call that only needs the height
writes only the 2-D field.
"""

import weakref

import numpy as np
import torch

from . import core
from .labeled import ChunkedArray, DataArray, Dataset
from .reference import _pressure, setup_reference_state
from .util import annual_average, calendar_axis, default_coords, validate_dataset, whole_years_in_order

__all__ = ["halosteric", "steric", "steric_layers", "steric_variants", "thermosteric"]


def steric(
    dset,
    reference=None,
    coord_names=None,
    varname_map=None,
    rhozero=1035.0,
    patm=101325.0,
    equation_of_state="Wright",
    variant="steric",
    domain="local",
    dtype="float32",
    strict=True,
    annual=False,
    verbose=False,
    days_in_month=None,
):
    """Steric, thermosteric or halosteric sea level change relative to a reference state.

    Arguments as ``momlevel.steric`` (steric.py:17-82).  ``days_in_month`` is the one
    addition: the annual-mean weights when ``annual=True`` and the time axis carries no
    calendar.  With a calendar time axis (cftime objects, as MOM6 output decodes to) the years
    and weights are read from it, as the reference does (util.py:79-87).

    Returns ``(result, reference)``.
    """
    xarray_in = type(dset).__module__.startswith("xarray")
    if xarray_in:
        from . import xarray_io

        dset_x = dset
        # only what the path reads is converted; dask-backed fields stay in blocks (labeled.ChunkedArray)
        t_, z_, zb_ = default_coords(coord_names)
        needed = {"thetao", "so", "volcello", "areacello", "deptho", t_, z_, zb_}
        needed |= {k for k, v in (varname_map or {}).items() if v in needed}
        dset = xarray_io.from_xarray(dset, names=sorted(needed))
        if reference is not None:
            assert type(reference).__module__.startswith("xarray"), "`reference` must be an xarray Dataset"
            reference = xarray_io.from_xarray(reference)

    annual_drho = False  # set when delta_rho is produced as annual means by the fused kernel
    # steric.py:84-91
    dset = dset.rename(varname_map)
    tcoord, zcoord, zbounds = default_coords(coord_names)
    additional_vars = None if domain == "global" else [zbounds, "deptho"]
    # The fused default path on device-resident fields reads every value-dependent check back together with
    # volo / masso AFTER the kernel is queued (one synchronisation instead of five in front of the launch);
    # an invalid dataset raises exactly what it raised before, a few milliseconds later.
    deferred = (reference is None and domain == "local" and variant in VARIANTS
                and _on_one_cuda_device(dset, ("thetao", "so", "volcello", "areacello", "deptho", zcoord, zbounds)))
    validate_dataset(dset, strict=strict, additional_vars=additional_vars, area_total=False if deferred else None)

    # steric.py:96
    pres = _pressure(dset, zcoord, patm)

    # steric.py:98-112
    fused_eta = None
    streamed = None    # heights / masses of fields that arrive block by block (dask-backed variables)
    area_total = None  # areacello.sum(), when the fused path has already read it back
    if variant in VARIANTS and _chunked(dset):
        # the fields exist only as blocks along time: streamed through the device as they are produced
        # (core.HostStream), never asked for as whole arrays
        if reference is not None:
            assert isinstance(reference, Dataset), "`reference` must be an xarray Dataset"
        reference, streamed = _streamed(dset, reference, pres, equation_of_state, (variant,), domain, rhozero, tcoord,
                                        zcoord, zbounds, verbose)
        streamed = streamed[variant]
        if domain != "global":
            fused_eta = streamed
    elif reference is not None:
        assert isinstance(reference, Dataset), "`reference` must be an xarray Dataset"
        if verbose:
            print("Using supplied reference state")
    else:
        array_patm = isinstance(pres, core.Pressure)  # a 2-D patm: device kernels only (ml_set_column_pressure)
        if domain != "global" and variant in VARIANTS and not array_patm and _host_resident(dset, tcoord, zcoord, zbounds):
            # fields in host memory (numpy, what xarray hands over): streamed through device windows by the
            # library, level rows packed to their present cells on the way (ml_steric_local_host)
            reference, fused_eta = _selfref_host(dset, pres, equation_of_state, variant, rhozero, tcoord, zcoord,
                                                 zbounds)
        elif domain != "global" and variant in ("steric", "thermosteric", "halosteric"):
            # reference state and column integral in one pass over T, S (ml_steric_local_selfref)
            reference, fused_eta, area_total = _selfref(dset, pres, equation_of_state, variant, rhozero, tcoord, zcoord,
                                                        zbounds, deferred, strict, additional_vars)
        else:
            reference = setup_reference_state(dset, patm=patm, eos=equation_of_state, coord_names=coord_names)
        if verbose:
            print("Generating reference state from first timestep")
    validate_dataset(reference, reference=True, strict=strict, area_total=area_total)

    # steric.py:115-125: which field, if any, is held at its reference value
    if variant == "thermosteric":
        thetao, so, t_bcast, s_bcast = dset["thetao"], reference["so"], False, True
    elif variant == "halosteric":
        thetao, so, t_bcast, s_bcast = reference["thetao"], dset["so"], True, False
    elif variant == "steric":
        thetao, so, t_bcast, s_bcast = dset["thetao"], dset["so"], False, False
    else:
        raise ValueError(f"Unknown variant '{variant}' passed to `steric`")

    full = dset["so"] if t_bcast else dset["thetao"]
    if full.dims[0] != tcoord or full.dims[1] != zcoord:
        raise ValueError(f"expecting fields laid out ({tcoord}, {zcoord}, y, x), got {full.dims}")
    hdims = full.dims[2:]
    result = Dataset()

    if domain == "global":
        # steric.py:134-147
        v_ref = reference["volcello"].data
        if streamed is not None:
            masso = streamed.numpy()
        elif (variant in VARIANTS and not isinstance(pres, core.Pressure)
                and _host_resident(dset, tcoord, zcoord, zbounds, need_depth=False)
                and not (isinstance(v_ref, torch.Tensor) and v_ref.is_cuda)):
            # fields in host memory (a daily series does not fit in HBM): streamed through device windows, level rows
            # packed to the cells of the reference volume on the way; the thermo- / halosteric variants keep their
            # reference slab on the device for the whole series (ml_host_stream_*)
            masso = _global_host(dset, reference, (variant,), pres, equation_of_state)[variant].numpy()
        else:
            masso = core.steric_global(thetao.data, so.data, v_ref, pres, eos=equation_of_state,
                                       t_bcast=t_bcast, s_bcast=s_bcast).cpu().numpy()
        volo, rhoga = float(reference["volo"]), float(reference["rhoga"])
        expansion_coeff = np.log(rhoga / (masso / volo))
        reference_height = volo / float(reference["areacello"].sum())
        sealevel = reference_height * expansion_coeff
        result["reference_height"] = DataArray(np.float64(reference_height), (), attrs={
            "long_name": "Reference column height", "units": "m"})
        result["reference_height"].encoding["dtype"] = dtype
        result[variant] = DataArray(sealevel, (tcoord,))
    else:
        # steric.py:150-166
        if fused_eta is not None:  # the fused pass has checked the depths and integrated already
            eta = fused_eta
        else:
            _check_depths(dset, zcoord, zbounds)
            eta = core.steric_local(thetao.data, so.data, reference["rho"].data, reference["volcello"].data,
                                    dset[zbounds].data, dset["deptho"].data, pres, want_delta_rho=False,
                                    rhozero=rhozero, eos=equation_of_state, t_bcast=t_bcast, s_bcast=s_bcast)[0]

        def _delta_rho():
            return core.delta_rho(thetao.data, so.data, reference["rho"].data, reference["volcello"].data, pres,
                                  eos=equation_of_state, t_bcast=t_bcast, s_bcast=s_bcast)

        if streamed is not None:
            def _delta_rho():  # noqa: F811 -- block by block again; the result is as large as the inputs
                return _delta_rho_streamed(thetao, so, reference, pres, equation_of_state, t_bcast, s_bcast)

        drho_shape = full.shape
        if streamed is not None:
            fused_weights = None  # blocks need not hold whole years: the monthly anomaly is averaged when it is read
        elif annual and days_in_month is None and tcoord in dset.variables:
            # util.py:79-87: year and days-in-month of every step come from the calendar objects of the time axis
            cal = calendar_axis(dset[tcoord].values)
            if cal is not None and whole_years_in_order(cal[0]):
                fused_weights = cal[1]
            else:
                fused_weights = None
        else:
            fused_weights = days_in_month
        if annual and fused_weights is not None:
            # steric.py:181-182 averages every result variable, the 4-D anomaly included: its annual means
            # come out of one fused pass instead of averaging a materialised monthly field
            weights = np.asarray(fused_weights, dtype=np.float64)
            assert weights.size == full.shape[0] and weights.size % 12 == 0, \
                "annual averaging needs whole years of monthly data"

            def _delta_rho():  # noqa: F811
                return core.delta_rho_annual(thetao.data, so.data, reference["rho"].data, reference["volcello"].data,
                                             pres, weights, eos=equation_of_state, t_bcast=t_bcast, s_bcast=s_bcast)

            drho_shape = (full.shape[0] // 12,) + tuple(full.shape[1:])
            annual_drho = True
        result["delta_rho"] = DataArray.lazy(_delta_rho, drho_shape, full.dims, attrs={
            "long_name": "change in in situ density from reference state", "units": "kg m-3"})
        result["delta_rho"].encoding["dtype"] = dtype
        result[variant] = DataArray(eta, (tcoord,) + hdims)

    # steric.py:169-179
    result[variant].attrs = {"long_name": f"{variant.capitalize()} height adjustment", "units": "m"}
    result[variant].encoding["dtype"] = dtype
    for var in set(result.dims):
        if var in dset.variables:
            coord = dset[var].copy(deep=False)
            coord.attrs = dict(dset[var].attrs)
            result[var] = coord

    if annual:
        fused = result["delta_rho"] if annual_drho else None  # already annual, and still lazy
        if fused is not None:
            result = result.drop_vars(["delta_rho"])
        result = annual_average(result, tcoord=tcoord, days_in_month=days_in_month)
        if fused is not None:
            result["delta_rho"] = fused

    if xarray_in:
        return xarray_io.to_xarray(result, like=dset_x), xarray_io.to_xarray(reference, like=dset_x)
    return (result, reference)


def _all_nonnegative(arr):
    """``np.all(nan_to_num(x, nan=0) >= 0)`` without leaving the device a tensor lives on (NaN passes)."""
    data = arr.data
    if isinstance(data, torch.Tensor):
        return not bool((data < 0).any())
    return not bool(np.any(np.asarray(data) < 0))


def _check_depths(dset, zcoord, zbounds):
    """derived.py:284-292: calc_dz's sign checks."""
    arrs = [dset["deptho"].data, dset[zcoord].data, dset[zbounds].data]
    if all(isinstance(a, torch.Tensor) and a.is_cuda for a in arrs):  # one read-back for the three flags
        neg = torch.stack([(a < 0).any() for a in arrs]).cpu()
        assert not bool(neg[0]), "Depth values must all be positive-definite"
        assert not bool(neg[1]), "Vertical coordinate levels must all be positive-definite"
        assert not bool(neg[2]), "Vertical coordinate interfaces must all be positive-definite"
        return
    assert _all_nonnegative(dset["deptho"]), "Depth values must all be positive-definite"
    assert _all_nonnegative(dset[zcoord]), "Vertical coordinate levels must all be positive-definite"
    assert _all_nonnegative(dset[zbounds]), "Vertical coordinate interfaces must all be positive-definite"


def _reference_from_pass(dset, tcoord, eos, rho, sums, pres=None):
    """The reference Dataset of reference.py:57-83 around a rho_ref / {volo, masso} pair a fused pass produced.

    ``rho=None``: the pass did not store the reference density (its volume-weighted sums are all the height
    needs); ``reference["rho"]`` then evaluates it on first access, like ``delta_rho`` in the result.
    """
    reference = Dataset()
    for name in ("thetao", "so", "volcello"):
        reference[name] = dset[name].isel({tcoord: 0}).squeeze().reset_coords(drop=True)
    scalar_attrs = {
        "volo": {"standard_name": "sea_water_volume", "long_name": "Sea Water Volume", "units": "m3"},
        "masso": {"standard_name": "sea_water_mass", "long_name": "Sea Water Mass", "units": "kg"},
        "rhoga": {"long_name": "Global Average Sea Water Density", "units": "kg m-3"}}
    on_device = isinstance(sums, torch.Tensor) and sums.is_cuda
    if on_device:
        # the pass is still running: the scalars are read back (one synchronisation, shared) when first looked at
        memo = {}

        def _host():
            if "v" not in memo:
                memo["v"] = sums.cpu().numpy()
            return memo["v"]

        scalars = {"volo": lambda: np.asarray(np.float64(_host()[0])),
                   "masso": lambda: np.asarray(np.float64(_host()[1])),
                   "rhoga": lambda: np.asarray(np.float64(_host()[1]) / np.float64(_host()[0]))}
    else:
        volo, masso = (float(x) for x in sums)
    rho_attrs = {"standard_name": "sea_water_density", "long_name": "In situ sea water density",
                 "comment": f"calculated with the {eos} equation of state", "units": "kg m-3"}
    if rho is None:
        T0, S0, V0 = (reference[k].data for k in ("thetao", "so", "volcello"))
        reference["rho"] = DataArray.lazy(lambda: core.reference_state(T0, S0, V0, pres, eos=eos)[0],
                                          reference["thetao"].shape, reference["thetao"].dims, attrs=rho_attrs)
    else:
        reference["rho"] = DataArray(rho, reference["thetao"].dims, attrs=rho_attrs)
    if on_device:
        for k in ("volo", "masso", "rhoga"):
            reference[k] = DataArray.lazy(scalars[k], (), (), attrs=scalar_attrs[k])
    else:
        reference["volo"] = DataArray(np.float64(volo), (), attrs=scalar_attrs["volo"])
        reference["masso"] = DataArray(np.float64(masso), (), attrs=scalar_attrs["masso"])
        reference["rhoga"] = DataArray(np.float64(masso) / np.float64(volo), (), attrs=scalar_attrs["rhoga"])
    reference["areacello"] = dset["areacello"]
    return reference


# Value checks of the static grid arrays (areacello.sum() within 2 % of the real ocean, util.py:669-694; depths and
# coordinates positive-definite, derived.py:284-292) that a device-resident Dataset has already passed.  An entry
# stands for the very tensor objects it was made from (weak references) at the version they had (torch bumps
# ``_version`` on every in-place write): a second call on the same grid neither launches the checks nor waits for
# them, so nothing in it synchronises with the device.
_CHECKED_GRIDS = {}


def _checked_before(arrs):
    ent = _CHECKED_GRIDS.get(tuple(id(a) for a in arrs))
    if ent is None:
        return None
    refs, versions, area_total = ent
    for a, r, v in zip(arrs, refs, versions):
        if r() is not a or a._version != v:
            return None
    return area_total


def _remember_checked(arrs, area_total):
    if len(_CHECKED_GRIDS) >= 16:
        _CHECKED_GRIDS.clear()
    _CHECKED_GRIDS[tuple(id(a) for a in arrs)] = (tuple(weakref.ref(a) for a in arrs), tuple(a._version for a in arrs),
                                                   area_total)


HOST_ROUTE_MIN_BYTES = 1 << 26  # fields smaller than this are simply copied to the device


def _host_resident(dset, tcoord, zcoord, zbounds, need_depth=True):
    """Whether ``steric()`` should take the host route: every input lives in host memory (numpy or CPU tensors),
    the fields are laid out ``(time, z, y, x)`` in one piece, and there is enough of them for the streaming to pay."""
    try:
        names = ("thetao", "so", "volcello", zcoord) + (("deptho", zbounds) if need_depth else ())
        arrs = [dset[n].data for n in names]
        if any(isinstance(a, torch.Tensor) and a.is_cuda for a in arrs):
            return False
        T, S, V = (dset[n] for n in ("thetao", "so", "volcello"))
        if not (T.dims == S.dims == V.dims and T.ndim == 4 and T.dims[0] == tcoord and T.dims[1] == zcoord):
            return False
        if not (T.shape == S.shape == V.shape and (not need_depth or dset["deptho"].shape == T.shape[2:])):
            return False
        for a in arrs[:2]:
            if not (a.is_contiguous() if isinstance(a, torch.Tensor) else a.flags["C_CONTIGUOUS"]):
                return False
        nbytes = 2 * int(np.prod(T.shape)) * (4 if str(arrs[0].dtype).endswith("float32") else 8)
        return nbytes >= HOST_ROUTE_MIN_BYTES
    except (KeyError, AttributeError, TypeError):
        return False


def _device_grid_checks(dset, zcoord, zbounds, strict, additional_vars):
    """The value checks of a device-resident Dataset's grid arrays, queued BEHIND the launch they guard: one read-back
    of {areacello total, three sign flags} the first time these tensors are seen, nothing after that
    (``_checked_before``).  Raises what the eager checks raise (util.py:783-792, derived.py:284-292); returns
    ``areacello.sum()``."""
    arrs = (dset["areacello"].data, dset["deptho"].data, dset[zcoord].data, dset[zbounds].data)
    area_total = _checked_before(arrs)
    if area_total is not None:
        validate_dataset(dset, strict=strict, additional_vars=additional_vars, area_total=area_total)
        return area_total
    host = torch.stack([torch.nansum(arrs[0].to(torch.float64))]
                       + [(a < 0).any().to(torch.float64) for a in arrs[1:]]).cpu()  # the one synchronisation
    area_total = float(host[0])
    validate_dataset(dset, strict=strict, additional_vars=additional_vars, area_total=area_total)  # util.py:783-792
    assert not bool(host[1]), "Depth values must all be positive-definite"  # derived.py:284-292
    assert not bool(host[2]), "Vertical coordinate levels must all be positive-definite"
    assert not bool(host[3]), "Vertical coordinate interfaces must all be positive-definite"
    _remember_checked(arrs, area_total)
    return area_total


def _selfref_host(dset, pres, eos, variant, rhozero, tcoord, zcoord, zbounds):
    """``setup_reference_state(dset)`` + the local column integral for fields that live in HOST memory.

    The library streams the time steps through device windows (``ml_steric_local_host`` /
    ``ml_steric_local_variants_host``); the heights come back as host arrays.  Returns ``(reference, eta)``.
    """
    from .util import eos_func_from_str

    eos_func_from_str(eos)
    _check_depths(dset, zcoord, zbounds)
    T, S = dset["thetao"].data, dset["so"].data
    V0 = dset["volcello"].isel({tcoord: 0}).squeeze().data
    step_bytes = 2 * int(np.prod(dset["thetao"].shape[1:])) * 4
    spw = int(min(max(1, -(-(1 << 28) // step_bytes)), dset["thetao"].shape[0]))  # windows of >= 256 MB
    etas, _, (volo, masso) = core.steric_local_host(
        T, S, V0, _host_numpy(dset[zbounds].data), _host_numpy(dset["deptho"].data), _host_numpy(pres),
        rhozero=rhozero, eos=eos, steps_per_window=spw, variants=False if variant == "steric" else (variant,))
    eta = etas if variant == "steric" else etas[variant]
    sums = torch.tensor([volo, masso], dtype=torch.float64)
    return _reference_from_pass(dset, tcoord, eos, None, sums, pres), eta


def _host_numpy(x):
    return x.detach().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _on_one_cuda_device(dset, names):
    try:
        devs = {dset[n].data.device for n in names if isinstance(dset[n].data, torch.Tensor)}
        return len(devs) == 1 and next(iter(devs)).type == "cuda" and all(
            isinstance(dset[n].data, torch.Tensor) for n in names)
    except (KeyError, AttributeError):
        return False


def _selfref(dset, pres, eos, variant, rhozero, tcoord, zcoord, zbounds, deferred=False, strict=True,
             additional_vars=None):
    """``setup_reference_state(dset)`` (reference.py:57-83) with the local column integral fused in.

    Returns ``(reference, eta, area_total)``; ``area_total`` is ``areacello.sum()`` when the value checks were
    deferred (read back with volo / masso after the launch), else ``None``.
    """
    from .util import eos_func_from_str

    eos_func_from_str(eos)
    if not deferred:
        _check_depths(dset, zcoord, zbounds)
    T0 = dset["thetao"].isel({tcoord: 0}).squeeze().data
    S0 = dset["so"].isel({tcoord: 0}).squeeze().data
    V0 = dset["volcello"].isel({tcoord: 0}).squeeze().data
    T = T0 if variant == "halosteric" else dset["thetao"].data
    S = S0 if variant == "thermosteric" else dset["so"].data
    eta, rho, sums = core.steric_local_selfref(
        T, S, V0, dset[zbounds].data, dset["deptho"].data, pres, rhozero=rhozero, eos=eos,
        t_bcast=variant == "halosteric", s_bcast=variant == "thermosteric", want_rho_ref=False)
    area_total = None
    if deferred:  # the value checks ride behind the kernel; volo / masso stay on the device until they are looked at
        area_total = _device_grid_checks(dset, zcoord, zbounds, strict, additional_vars)
    return _reference_from_pass(dset, tcoord, eos, rho, sums, pres), eta, area_total


def _global_host(dset, reference, variants, pres, eos, tcoord="time"):
    """``calc_masso(rho, reference.volcello)`` per step (steric.py:135) for fields in host memory, for each of
    ``variants`` -- two or more of them from one pass over the fields.  ``reference=None``: the reference state is
    step 0 of the fields (its volume taken from ``dset``).  Returns ``{variant: CPU tensor [nt]}``."""
    T, S = dset["thetao"].data, dset["so"].data
    nt = int(T.shape[0])
    step_bytes = 2 * int(np.prod(T.shape[1:])) * (4 if str(T.dtype).endswith("float32") else 8)
    spw = int(min(max(1, -(-(1 << 28) // step_bytes)), nt))  # windows of >= 256 MB
    ref = None
    if reference is not None and any(v != "steric" for v in variants):
        ref = {"thetao": _host_array(reference["thetao"]), "so": _host_array(reference["so"])}
    V = reference["volcello"] if reference is not None else dset["volcello"].isel({tcoord: 0}).squeeze()
    f32 = str(T.dtype).endswith("float32") and str(S.dtype).endswith("float32")
    hs = core.HostStream("global", _host_array(V), _host_numpy(pres), variants=tuple(variants), reference=ref,
                         eos=eos, max_block_steps=spw, dtype=torch.float32 if f32 else torch.float64)
    outs = []
    try:
        for t in range(0, nt, spw):
            outs.append(hs.push(T[t: t + spw], S[t: t + spw]))
        hs.finish()
    except BaseException:
        hs.abort()
        raise
    return {v: torch.cat([o[v] for o in outs]) if len(outs) != 1 else outs[0][v] for v in variants}


def _chunked(dset):
    """Whether thetao or so exists only as blocks along time (a dask-backed variable, ``labeled.ChunkedArray``)."""
    try:
        return any(isinstance(dset[n]._data, ChunkedArray) for n in ("thetao", "so"))
    except (KeyError, AttributeError):
        return False


def _block_iter(arr):
    """``(chunks, iterator of numpy blocks)`` of a field: its own blocks, or the whole host array as one block."""
    if isinstance(arr, ChunkedArray):
        return arr.chunks, arr.blocks()
    a = arr.detach().cpu().numpy() if isinstance(arr, torch.Tensor) else np.asarray(arr)
    return (a.shape[0],), iter([a])


def _aligned_blocks(T, S):
    """Blocks of T and S cut at the union of their block boundaries (views, no copies): ``(max_len, iterator)``."""
    ct, it_t = _block_iter(T)
    cs, it_s = _block_iter(S)
    assert sum(ct) == sum(cs), "thetao and so must have the same number of time steps"
    cuts = sorted(set(np.cumsum(ct).tolist()) | set(np.cumsum(cs).tolist()))
    lens = np.diff([0] + cuts).tolist()

    def gen():
        bt = bs = None
        ot = os_ = 0
        for n in lens:
            if bt is None or ot >= bt.shape[0]:
                bt, ot = next(it_t), 0
            if bs is None or os_ >= bs.shape[0]:
                bs, os_ = next(it_s), 0
            yield bt[ot: ot + n], bs[os_: os_ + n]
            ot += n
            os_ += n

    return (max(lens) if lens else 1), gen()


def _host_array(x):
    x = x.data if isinstance(x, DataArray) else x
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _streamed(dset, reference, pres, eos, variants, domain, rhozero, tcoord, zcoord, zbounds, verbose=False,
              first_step_sums=None):
    """The heights (local) or masses (global) of fields that arrive block by block, and the reference Dataset.

    One pass over the blocks of ``thetao`` / ``so`` through ``core.HostStream`` for all of ``variants``: a block is
    packed, copied and integrated while the next one is being produced, and at most two blocks are alive at a time.
    With ``reference=None`` the reference state is step 0 of the first block (steric.py:105-107); its
    ``{volo, masso}`` come from the stream, or from ``first_step_sums(T0, S0, V0)`` when that is given.
    Returns ``(reference, {variant: CPU tensor})``.
    """
    from .util import eos_func_from_str

    eos_func_from_str(eos)
    if isinstance(pres, core.Pressure):
        raise NotImplementedError("a 2-D `patm` together with chunked (dask-backed) fields")
    local = domain != "global"
    if local:
        _check_depths(dset, zcoord, zbounds)
    T, S = dset["thetao"], dset["so"]
    if not (T.dims == S.dims and T.ndim == 4 and T.dims[0] == tcoord and T.dims[1] == zcoord and T.shape == S.shape):
        raise ValueError(f"expecting fields laid out ({tcoord}, {zcoord}, y, x), got {T.dims} and {S.dims}")
    supplied = reference is not None
    if supplied:
        if verbose:
            print("Using supplied reference state")
        V0 = _host_array(reference["volcello"])
        ref = {"rho": _host_array(reference["rho"])} if local else {}
        if any(v != "steric" for v in variants):
            ref.update(thetao=_host_array(reference["thetao"]), so=_host_array(reference["so"]))
        if not ref:  # the masses of the steric variant need the reference volume only
            ref = None
    else:
        if verbose:
            print("Generating reference state from first timestep")
        V0 = _host_array(dset["volcello"].isel({tcoord: 0}).squeeze())
        ref = None
    max_len, blocks = _aligned_blocks(T._data, S._data)
    dt = torch.float32 if str(T._data.dtype).endswith("float32") and str(S._data.dtype).endswith("float32") else torch.float64
    hs = core.HostStream("local" if local else "global", V0, _host_numpy(pres),
                         z_i=_host_array(dset[zbounds]) if local else None,
                         deptho=_host_array(dset["deptho"]) if local else None, variants=tuple(variants), reference=ref,
                         rhozero=rhozero, eos=eos, max_block_steps=max_len, dtype=dt,
                         want_sums=not supplied and first_step_sums is None)
    outs, first = [], None
    try:
        for Tb, Sb in blocks:
            if first is None and not supplied:  # step 0 becomes the reference Dataset (reference.py:60-68)
                first = (np.array(Tb[0]), np.array(Sb[0]))
            outs.append(hs.push(Tb, Sb))
        _, sums = hs.finish()
    except BaseException:
        hs.abort()
        raise
    out = {v: torch.cat([o[v] for o in outs]) if len(outs) != 1 else outs[0][v] for v in variants}
    if not supplied:
        if first_step_sums is not None:
            sums = first_step_sums(first[0], first[1], V0)
        sub = Dataset()
        hdims = T.dims[1:]
        sub["thetao"] = DataArray(first[0], hdims, attrs=T.attrs)
        sub["so"] = DataArray(first[1], hdims, attrs=S.attrs)
        sub["volcello"] = DataArray(V0, hdims, attrs=dset["volcello"].attrs)
        sub["areacello"] = dset["areacello"]
        for name in hdims:
            if name in dset.variables:
                sub[name] = dset[name]
        sub = _with_time_axis(sub, tcoord)
        sums = sums if isinstance(sums, torch.Tensor) else torch.tensor(sums, dtype=torch.float64)
        reference = _reference_from_pass(sub, tcoord, eos, None, sums, pres)
    return reference, out


def _with_time_axis(sub, tcoord):
    """A one-step Dataset around the reference slabs, so that ``_reference_from_pass`` can take its step 0."""
    out = Dataset()
    for k, v in sub.variables.items():
        if k in ("thetao", "so", "volcello"):
            d = v.data
            out[k] = DataArray(d[None] if not isinstance(d, torch.Tensor) else d.unsqueeze(0), (tcoord,) + v.dims, attrs=v.attrs)
        else:
            out[k] = v
    return out


def _delta_rho_streamed(thetao, so, reference, pres, eos, t_bcast, s_bcast):
    """``delta_rho`` (steric.py:151-158) of chunked fields: one ``ml_delta_rho`` per block, gathered on the host."""
    full = so if t_bcast else thetao
    rho_ref, v_ref = reference["rho"].data, reference["volcello"].data
    parts = []
    if t_bcast or s_bcast:
        fixed = (thetao if t_bcast else so).data
        _, it = _block_iter(full._data)
        for blk in it:
            a = core.delta_rho(fixed if t_bcast else blk, blk if t_bcast else fixed, rho_ref, v_ref, pres, eos=eos,
                               t_bcast=t_bcast, s_bcast=s_bcast)
            parts.append(a.cpu())
    else:
        _, it = _aligned_blocks(thetao._data, so._data)
        for Tb, Sb in it:
            parts.append(core.delta_rho(Tb, Sb, rho_ref, v_ref, pres, eos=eos).cpu())
    return torch.cat(parts)


VARIANTS = ("steric", "thermosteric", "halosteric")


def steric_variants(dset, reference=None, coord_names=None, varname_map=None, rhozero=1035.0, patm=101325.0,
                    equation_of_state="Wright", dtype="float32", strict=True, verbose=False, domain="local", annual=False,
                    days_in_month=None):
    """Steric, thermosteric and halosteric sea level from one call, in either domain.

    Equivalent to ``steric(dset)``, ``thermosteric(dset)`` and ``halosteric(dset)`` (steric.py:115-121 only
    changes which operand of the equation of state is held at its reference value) with the validation, the
    reference state and the result assembly done once, and T and S read once for the three.  Arguments as
    :func:`steric`.  Returns ``(result, reference)``: ``domain="local"`` gives the three height fields,
    ``domain="global"`` the three ``(time,)`` series and ``reference_height``.  There is no ``delta_rho`` (one per
    variant): ask :func:`steric` for the variant whose 4-D anomaly is wanted.
    """
    xarray_in = type(dset).__module__.startswith("xarray")
    if xarray_in:
        from . import xarray_io

        dset_x = dset
        # only what the path reads is converted; dask-backed fields stay in blocks (labeled.ChunkedArray)
        t_, z_, zb_ = default_coords(coord_names)
        needed = {"thetao", "so", "volcello", "areacello", "deptho", t_, z_, zb_}
        needed |= {k for k, v in (varname_map or {}).items() if v in needed}
        dset = xarray_io.from_xarray(dset, names=sorted(needed))
        if reference is not None:
            assert type(reference).__module__.startswith("xarray"), "`reference` must be an xarray Dataset"
            reference = xarray_io.from_xarray(reference)
    dset = dset.rename(varname_map)
    tcoord, zcoord, zbounds = default_coords(coord_names)
    args = (dset, reference, tcoord, zcoord, zbounds, rhozero, patm, equation_of_state, strict, verbose)
    if domain == "global":
        result, reference = _global_variants(*args)
    else:
        result, reference = _local_variants(*args)
    for variant in VARIANTS:
        result[variant].attrs = {"long_name": f"{variant.capitalize()} height adjustment", "units": "m"}  # steric.py:169-172
        result[variant].encoding["dtype"] = dtype
    if "reference_height" in result.variables:
        result["reference_height"].encoding["dtype"] = dtype
    for var in set(result.dims):
        if var in dset.variables:
            coord = dset[var].copy(deep=False)
            coord.attrs = dict(dset[var].attrs)
            result[var] = coord
    if annual:  # steric.py:181-182
        result = annual_average(result, tcoord=tcoord, days_in_month=days_in_month)
    if xarray_in:
        return xarray_io.to_xarray(result, like=dset_x), xarray_io.to_xarray(reference, like=dset_x)
    return (result, reference)


def _variants_route(dset, pres, tcoord, zcoord, zbounds, domain):
    """Where the fields of a three-variant call live, which decides how they are read once for the three:
    ``"chunked"`` (blocks along time: one ``core.HostStream`` pass over the blocks), ``"host"`` (whole arrays in host
    memory, large enough for the streaming to pay: one ``HostStream`` pass / ``ml_steric_local_variants_host``) or
    ``"device"`` (one call of the one-pass entry point on device tensors)."""
    if _chunked(dset):
        return "chunked"
    if not isinstance(pres, core.Pressure) and _host_resident(dset, tcoord, zcoord, zbounds, need_depth=domain != "global"):
        return "host"
    return "device"


def _first_step_sums(eos):
    """``{volo, masso}`` of the reference state that is step 0 of the fields, as the device route evaluates them (the
    self-reference pass of ``ml_steric_global_variants``), for the routes that stream the fields from host memory:
    all three routes then give the same reference scalars, and so the same series, bit for bit."""

    def sums(T0, S0, V0, pres):
        return core.steric_global_variants(np.asarray(T0)[None], np.asarray(S0)[None], V0, pres, eos=eos)[1]

    return sums


def _global_variants(dset, reference, tcoord, zcoord, zbounds, rhozero, patm, eos, strict, verbose):
    """The global branch (steric.py:134-147) for the three variants: masses from one pass, then the ln formula."""
    from .util import eos_func_from_str

    validate_dataset(dset, strict=strict, additional_vars=None)  # steric.py:84-91: no z_i / deptho in this domain
    pres = _pressure(dset, zcoord, patm)
    eos_func_from_str(eos)
    T, S = dset["thetao"], dset["so"]
    if T.dims[0] != tcoord or T.dims[1] != zcoord or S.dims != T.dims:
        raise ValueError(f"expecting fields laid out ({tcoord}, {zcoord}, y, x), got {T.dims}")
    supplied = reference is not None
    if supplied:
        assert isinstance(reference, Dataset), "`reference` must be an xarray Dataset"
        if verbose:
            print("Using supplied reference state")
        validate_dataset(reference, reference=True, strict=strict)
    elif verbose:
        print("Generating reference state from first timestep")
    route = _variants_route(dset, pres, tcoord, zcoord, zbounds, "global")
    sums_of = _first_step_sums(eos)
    if route == "chunked":
        reference, masso = _streamed(dset, reference, pres, eos, VARIANTS, "global", rhozero, tcoord, zcoord, zbounds,
                                     first_step_sums=lambda T0, S0, V0: sums_of(T0, S0, V0, pres))
    elif route == "host":
        masso = _global_host(dset, reference, VARIANTS, pres, eos, tcoord)
        if not supplied:
            T0, S0 = (_host_array(dset[k].isel({tcoord: 0}).squeeze()) for k in ("thetao", "so"))
            V0 = _host_array(dset["volcello"].isel({tcoord: 0}).squeeze())
            reference = _reference_from_pass(dset, tcoord, eos, None, sums_of(T0, S0, V0, pres), pres)
    elif supplied:
        masso, _ = core.steric_global_variants(T.data, S.data, reference["volcello"].data, pres, T_ref=reference["thetao"].data,
                                               S_ref=reference["so"].data, eos=eos)
    else:
        V0 = dset["volcello"].isel({tcoord: 0}).squeeze().data
        masso, sums = core.steric_global_variants(T.data, S.data, V0, pres, eos=eos)
        reference = _reference_from_pass(dset, tcoord, eos, None, sums, pres)
    if not supplied:
        validate_dataset(reference, reference=True, strict=strict)
    # steric.py:136-147
    volo, rhoga = float(reference["volo"]), float(reference["rhoga"])
    reference_height = volo / float(reference["areacello"].sum())
    result = Dataset()
    result["reference_height"] = DataArray(np.float64(reference_height), (), attrs={
        "long_name": "Reference column height", "units": "m"})
    for variant in VARIANTS:
        m = masso[variant]
        m = m.cpu().numpy() if isinstance(m, torch.Tensor) else np.asarray(m)
        result[variant] = DataArray(reference_height * np.log(rhoga / (m / volo)), (tcoord,))
    return result, reference


def _local_variants(dset, reference, tcoord, zcoord, zbounds, rhozero, patm, eos, strict, verbose):
    """The local branch (steric.py:150-166) for the three variants: the heights from one pass over T and S."""
    from .util import eos_func_from_str

    # device-resident fields without a supplied reference: the value checks ride behind the launch, as in steric()
    deferred = reference is None and _on_one_cuda_device(
        dset, ("thetao", "so", "volcello", "areacello", "deptho", zcoord, zbounds))
    validate_dataset(dset, strict=strict, additional_vars=[zbounds, "deptho"], area_total=False if deferred else None)
    pres = _pressure(dset, zcoord, patm)
    eos_func_from_str(eos)
    if not deferred:
        _check_depths(dset, zcoord, zbounds)
    area_total = None
    full = dset["thetao"]
    if full.dims[0] != tcoord or full.dims[1] != zcoord or dset["so"].dims != full.dims:
        raise ValueError(f"expecting fields laid out ({tcoord}, {zcoord}, y, x), got {full.dims}")
    args = (full.data, dset["so"].data)
    tail = (dset[zbounds].data, dset["deptho"].data, pres)
    kw = dict(rhozero=rhozero, eos=eos)
    route = _variants_route(dset, pres, tcoord, zcoord, zbounds, "local")
    if reference is not None:
        assert isinstance(reference, Dataset), "`reference` must be an xarray Dataset"
        if verbose:
            print("Using supplied reference state")
        validate_dataset(reference, reference=True, strict=strict)
        if route == "chunked":
            _, etas = _streamed(dset, reference, pres, eos, VARIANTS, "local", rhozero, tcoord, zcoord, zbounds)
        else:
            etas, _, _ = core.steric_local_variants(*args, reference["volcello"].data, *tail, T_ref=reference["thetao"].data,
                                                    S_ref=reference["so"].data, rho_ref=reference["rho"].data, **kw)
    else:
        if verbose:
            print("Generating reference state from first timestep")
        V0 = dset["volcello"].isel({tcoord: 0}).squeeze().data
        if route == "chunked":
            reference, etas = _streamed(dset, None, pres, eos, VARIANTS, "local", rhozero, tcoord, zcoord, zbounds)
        elif route == "host":
            # fields in host memory: one pass over PCIe feeds the three integrations (ml_steric_local_variants_host)
            step_bytes = 2 * int(np.prod(full.shape[1:])) * 4
            spw = int(min(max(1, -(-(1 << 28) // step_bytes)), full.shape[0]))
            etas, _, (volo, masso) = core.steric_local_host(
                *args, V0, _host_numpy(dset[zbounds].data), _host_numpy(dset["deptho"].data), _host_numpy(pres),
                steps_per_window=spw, variants=True, **kw)
            reference = _reference_from_pass(dset, tcoord, eos, None,
                                             torch.tensor([volo, masso], dtype=torch.float64), pres)
        else:
            etas, rho, sums = core.steric_local_variants(*args, V0, *tail, **kw)
            if deferred:
                area_total = _device_grid_checks(dset, zcoord, zbounds, strict, [zbounds, "deptho"])
            reference = _reference_from_pass(dset, tcoord, eos, rho, sums)
        validate_dataset(reference, reference=True, strict=strict, area_total=area_total)
    result = Dataset()
    for variant in VARIANTS:
        result[variant] = DataArray(etas[variant], (tcoord,) + full.dims[2:])
    return result, reference


def steric_layers(dset, depth_edges=(0.0, 700.0, 2000.0, None), reference=None, coord_names=None, varname_map=None,
                  rhozero=1035.0, patm=101325.0, equation_of_state="Wright", variant="steric", dtype="float32",
                  strict=True, annual=False, days_in_month=None, verbose=False):
    """Local steric, thermosteric or halosteric sea level change split by depth layer (0-700 m, 700-2000 m and
    2000 m to the sea floor by default), from one pass over T and S.

    Layer ``b`` is the local height of :func:`steric` with ``calc_dz(top=depth_edges[b], bottom=depth_edges[b+1])``
    (derived.py:249-325) as the cell thickness; ``None`` as the last edge means "to the sea floor".  A layer wholly
    below a wet column's floor is 0.0; a column whose surface is dry is NaN in every layer.  Like ``calc_dz``, a
    partial bottom cell that straddles an inner edge counts in full towards the layer above the edge, so there the
    layers add up to more than the full-column height.  The remaining arguments are those of :func:`steric` with
    ``domain="local"``; ``reference=None`` builds the reference state from the first step first.

    ``variant`` may also be a list or tuple of distinct names from ``("steric", "thermosteric", "halosteric")``: the
    validation, the reference state and the move of T and S to the device are then done once, and one pass over T
    and S gives every height asked for (a sea-level budget: how much of a layer's change is warming and how much is
    freshening).  Each result variable is the one a call with that name alone returns, bit for bit.

    Returns ``(result, reference)``: ``result[variant]`` has dims ``(time, depth_layer, y, x)``, ``result["layer_top"]``
    and ``result["layer_bottom"]`` are ``(depth_layer,)`` (``inf``: the sea floor).  There is no ``delta_rho``:
    it is the field :func:`steric` returns.
    """
    edges = core.layer_edges(depth_edges)
    names = None if isinstance(variant, str) else core.variant_names(variant)
    xarray_in = type(dset).__module__.startswith("xarray")
    if xarray_in:
        from . import xarray_io

        dset_x = dset
        t_, z_, zb_ = default_coords(coord_names)
        needed = {"thetao", "so", "volcello", "areacello", "deptho", t_, z_, zb_}
        needed |= {k for k, v in (varname_map or {}).items() if v in needed}
        dset = xarray_io.from_xarray(dset, names=sorted(needed))
        if reference is not None:
            assert type(reference).__module__.startswith("xarray"), "`reference` must be an xarray Dataset"
            reference = xarray_io.from_xarray(reference)

    # steric.py:84-91
    dset = dset.rename(varname_map)
    tcoord, zcoord, zbounds = default_coords(coord_names)
    if _chunked(dset):
        raise NotImplementedError("steric_layers takes device-resident or in-memory fields; chunked (dask-backed) "
                                  "fields are not supported yet")
    validate_dataset(dset, strict=strict, additional_vars=[zbounds, "deptho"])
    pres = _pressure(dset, zcoord, patm)  # steric.py:96

    # steric.py:98-112
    if reference is not None:
        assert isinstance(reference, Dataset), "`reference` must be an xarray Dataset"
        if verbose:
            print("Using supplied reference state")
    else:
        reference = setup_reference_state(dset, patm=patm, eos=equation_of_state, coord_names=coord_names)
        if verbose:
            print("Generating reference state from first timestep")
    validate_dataset(reference, reference=True, strict=strict)

    if names is not None:
        # the heights asked for from one call: T_ref, S_ref are the reference slabs (steric.py:115-121)
        full = dset["thetao"]
        if full.dims[0] != tcoord or full.dims[1] != zcoord or dset["so"].dims != full.dims:
            raise ValueError(f"expecting fields laid out ({tcoord}, {zcoord}, y, x), got {full.dims}")
        _check_depths(dset, zcoord, zbounds)
        etas = core.steric_local_layers_variants(full.data, dset["so"].data, reference["thetao"].data,
                                                 reference["so"].data, reference["rho"].data,
                                                 reference["volcello"].data, dset[zbounds].data, dset["deptho"].data,
                                                 pres, edges, rhozero=rhozero, eos=equation_of_state, variants=names)
    else:
        # steric.py:115-125
        if variant == "thermosteric":
            thetao, so, t_bcast, s_bcast = dset["thetao"], reference["so"], False, True
        elif variant == "halosteric":
            thetao, so, t_bcast, s_bcast = reference["thetao"], dset["so"], True, False
        elif variant == "steric":
            thetao, so, t_bcast, s_bcast = dset["thetao"], dset["so"], False, False
        else:
            raise ValueError(f"Unknown variant '{variant}' passed to `steric`")
        full = dset["so"] if t_bcast else dset["thetao"]
        if full.dims[0] != tcoord or full.dims[1] != zcoord:
            raise ValueError(f"expecting fields laid out ({tcoord}, {zcoord}, y, x), got {full.dims}")

        _check_depths(dset, zcoord, zbounds)
        etas = {variant: core.steric_local_layers(thetao.data, so.data, reference["rho"].data,
                                                  reference["volcello"].data, dset[zbounds].data, dset["deptho"].data,
                                                  pres, edges, rhozero=rhozero, eos=equation_of_state, t_bcast=t_bcast,
                                                  s_bcast=s_bcast)}
    result = Dataset()
    # steric.py:169-179, plus the edges
    for name in names or (variant,):
        result[name] = DataArray(etas[name], (tcoord, "depth_layer") + full.dims[2:], attrs={
            "long_name": f"{name.capitalize()} height adjustment", "units": "m",
            "depth_edges": [float(e) for e in edges]})
        result[name].encoding["dtype"] = dtype
    result["layer_top"] = DataArray(edges[:-1].copy(), ("depth_layer",), attrs={
        "long_name": "Top of depth layer", "units": "m"})
    result["layer_bottom"] = DataArray(edges[1:].copy(), ("depth_layer",), attrs={
        "long_name": "Bottom of depth layer (inf: the sea floor)", "units": "m"})
    for var in set(result.dims):
        if var in dset.variables:
            coord = dset[var].copy(deep=False)
            coord.attrs = dict(dset[var].attrs)
            result[var] = coord
    if annual:  # steric.py:181-182
        result = annual_average(result, tcoord=tcoord, days_in_month=days_in_month)
    if xarray_in:
        return xarray_io.to_xarray(result, like=dset_x), xarray_io.to_xarray(reference, like=dset_x)
    return (result, reference)


def halosteric(*args, **kwargs):
    """Wrapper for halosteric calculation (steric.py:187-190)."""
    result, reference = steric(*args, **kwargs, variant="halosteric")
    return (result, reference)


def thermosteric(*args, **kwargs):
    """Wrapper for thermosteric calculation (steric.py:193-196)."""
    result, reference = steric(*args, **kwargs, variant="thermosteric")
    return (result, reference)
