"""reference.py -- sea level reference state (mirrors ``src/momlevel/reference.py:15-85``).

One fused kernel (``ml_reference_state``) evaluates the reference density and both global
sums in a single pass over the ``time_index`` slab.  With ``period=`` the slabs are the time means
of a baseline period (``ml_mean_state_accumulate``, one pass over T, S and volcello) and the same
kernel runs on them.
"""

import numpy as np
import torch

from . import core, util
from .labeled import ChunkedArray, DataArray, Dataset

__all__ = ["setup_reference_state"]


def _pressure(dset, zcoord, patm):
    """steric.py:96 / reference.py:54: 1 m ~ 1 dbar = 1e4 Pa, plus the surface pressure.

    ``patm`` is a scalar (a per-level pressure vector comes back) or a 2-D field over the horizontal dims of the
    dataset -- sea-level pressure from a reanalysis, say -- which the reference broadcasts by dimension name into
    ``pres[z, y, x]``; a :class:`core.Pressure` (per-level part + per-column part) comes back then.
    """
    z = dset[zcoord].data
    on_device = isinstance(z, torch.Tensor) and z.is_cuda
    if not isinstance(patm, (int, float, np.floating, np.integer)):
        nd = getattr(patm, "ndim", np.ndim(patm))
        if nd == 0:
            patm = float(patm)
        elif nd == 2:
            hdims = tuple(d for d in dset["thetao"].dims if d not in (zcoord,))[-2:]
            pdims = getattr(patm, "dims", None)
            if isinstance(patm, (DataArray, torch.Tensor)):
                col = patm.data
            else:  # numpy, or an xarray.DataArray (its .values)
                col = np.asarray(patm.values if hasattr(patm, "values") else patm)
            if pdims is not None and tuple(pdims) != hdims:
                if set(pdims) != set(hdims):
                    raise ValueError(f"`patm` has dims {tuple(pdims)}, expecting the horizontal dims {hdims}")
                col = col.T  # name-based broadcasting: the order of the dims does not matter to the reference
            hshape = tuple(dset["thetao"].shape[-2:])
            if tuple(np.shape(col)) != hshape:
                raise ValueError(f"`patm` has shape {tuple(np.shape(col))}, expecting {hshape}")
            level = (z.to(torch.float64) * 1.0e4) if on_device else np.asarray(dset[zcoord].values, dtype=np.float64) * 1.0e4
            return core.Pressure(level, col)
        else:
            raise NotImplementedError("momlevel_b200 takes `patm` as a scalar or as a 2-D (y, x) field")
    if on_device:  # stays on the device: no read-back in front of the launch
        return (z.to(torch.float64) * 1.0e4) + float(patm)
    return (np.asarray(dset[zcoord].values, dtype=np.float64) * 1.0e4) + float(patm)


def setup_reference_state(dset, patm=101325.0, eos="Wright", coord_names=None, time_index=0, period=None,
                          period_weights=None):
    """Generate the reference dataset (reference.py:15-85).

    Returns a Dataset with ``thetao``, ``so``, ``volcello``, ``rho`` (3-D), ``volo``,
    ``masso``, ``rhoga`` (scalars) and ``areacello``.

    ``period``: a ``slice`` of time positions (step ``None`` or 1) whose time mean is the reference state -- a
    climatology such as 1995-2014, or the first 20 years of a control run -- instead of the one step ``time_index``.
    ``period_weights``: one finite weight >= 0 per step of the period (days in month, say), with a positive sum;
    equal weights by default.  For each cell and each of ``thetao``, ``so`` and ``volcello`` on its own the mean is
    ``sum_t w_t x_t / sum_t w_t`` over the steps where that field is not NaN (xarray's skipna ``weighted(...).mean``);
    a cell with no value in the period is NaN.  ``rho`` is the density of the mean state, ``EOS(mean T, mean S, p)``,
    not the mean density: it is the state the thermosteric and halosteric variants hold fixed.  ``volo``, ``masso``
    and ``rhoga`` are formed from the mean slabs as from one step.

    The means are kept in fp64 whatever the fields' dtype, so ``steric(dset, reference=ref)`` with the thermo- or
    halosteric variant runs on fp64 storage, and a chunked (dask-backed) stream with such a reference runs in fp64
    (the promotion rule of ``core.HostStream``).  The Dataset's ``reference_period`` attribute records the period as
    ``"start:stop"`` and ``reference_period_weights`` whether it was ``"equal"`` or ``"supplied"``.  Fields on the
    device are averaged there in one pass; host-resident and chunked fields are streamed through the device block by
    block, reading no block past the period.  An ``xarray.Dataset`` in gives an ``xarray.Dataset`` out.
    """
    if period is not None or period_weights is not None:
        return _period_reference(dset, patm, eos, coord_names, time_index, period, period_weights)
    tcoord, zcoord, _ = util.default_coords(coord_names)
    util.eos_func_from_str(eos)
    pres = _pressure(dset, zcoord, patm)

    reference = Dataset()
    for name in ("thetao", "so", "volcello"):
        reference[name] = dset[name].isel({tcoord: time_index}).squeeze().reset_coords(drop=True)

    rho, sums = core.reference_state(reference["thetao"].data, reference["so"].data, reference["volcello"].data,
                                     pres, eos=eos)
    volo, masso = (float(x) for x in sums.cpu())
    reference["rho"] = DataArray(rho, reference["thetao"].dims, attrs={
        "standard_name": "sea_water_density",
        "long_name": "In situ sea water density",
        "comment": f"calculated with the {eos} equation of state",
        "units": "kg m-3",
    })
    reference["volo"] = DataArray(np.float64(volo), (), attrs={
        "standard_name": "sea_water_volume", "long_name": "Sea Water Volume", "units": "m3"})
    reference["masso"] = DataArray(np.float64(masso), (), attrs={
        "standard_name": "sea_water_mass", "long_name": "Sea Water Mass", "units": "kg"})
    reference["rhoga"] = DataArray(np.float64(masso) / np.float64(volo), (), attrs={
        "long_name": "Global Average Sea Water Density", "units": "kg m-3"})
    reference["areacello"] = dset["areacello"]
    return reference


def period_steps(period, nt, period_weights=None):
    """``(start, stop, weights)`` of a ``period`` slice over ``nt`` steps, checked; ``weights`` is ``None`` (equal)
    or a float64 array of one weight per step.  Raises ``ValueError`` for a period that is not a forward slice, an
    empty period, or weights that are not finite, >= 0 and of positive sum, one per step."""
    if not isinstance(period, slice):
        raise ValueError(f"`period` must be a slice of time positions, got {type(period).__name__}")
    if period.step not in (None, 1):
        raise ValueError(f"`period` must have a step of None or 1, got {period.step}")
    start, stop, _ = period.indices(int(nt))
    if stop <= start:
        raise ValueError(f"`period` {period} selects no time step of the {nt}")
    if period_weights is None:
        return start, stop, None
    try:
        w = np.asarray(period_weights.detach().cpu() if isinstance(period_weights, torch.Tensor) else period_weights,
                       dtype=np.float64)
    except (TypeError, ValueError) as e:
        raise ValueError(f"`period_weights` must be numbers: {e}") from None
    if w.ndim != 1 or w.shape[0] != stop - start:
        raise ValueError(f"`period_weights` must be 1-D with one weight per step of the period ({stop - start}), "
                         f"got shape {w.shape}")
    if not np.all(np.isfinite(w)) or np.any(w < 0.0) or not w.sum() > 0.0:
        raise ValueError("`period_weights` must be finite and >= 0 with a positive sum")
    return start, stop, np.ascontiguousarray(w)


def _period_reference(dset, patm, eos, coord_names, time_index, period, period_weights):
    """``setup_reference_state(period=...)``: the reference state of the period's time-mean T, S and volcello."""
    if period is None:
        raise ValueError("`period_weights` needs a `period`")
    if time_index != 0:
        raise ValueError("give either `time_index` or `period`, not both")
    xarray_in = type(dset).__module__.startswith("xarray")
    if xarray_in:
        from . import xarray_io

        dset_x = dset
        t_, z_, _ = util.default_coords(coord_names)
        dset = xarray_io.from_xarray(dset, names=["thetao", "so", "volcello", "areacello", t_, z_])
    tcoord, zcoord, _ = util.default_coords(coord_names)
    fields = [dset[name] for name in ("thetao", "so", "volcello")]
    for name, f in zip(("thetao", "so", "volcello"), fields):
        if f.dims[0] != tcoord:
            raise ValueError(f"`period` needs '{name}' laid out ({tcoord}, {zcoord}, ...), got {f.dims}")
    nt = int(fields[0].shape[0])
    if any(int(f.shape[0]) != nt for f in fields) or not fields[0].shape == fields[1].shape == fields[2].shape:
        raise ValueError(f"thetao, so and volcello must have the same shape, got {[tuple(f.shape) for f in fields]}")
    start, stop, weights = period_steps(period, nt, period_weights)
    util.eos_func_from_str(eos)
    pres = _pressure(dset, zcoord, patm)

    data = [f._data for f in fields]
    if _device_resident(data):
        # device-resident fields (those that are not are copied over, the period only): one pass, one launch
        T, S, V = (core.to_device(d[start:stop]) for d in data)
        w = torch.from_numpy(weights).to(T.device) if weights is not None else None
        means = core.mean_state(T, S, V, weights=w)
    else:
        means = _period_mean_host(data, start, stop, weights)

    reference = Dataset(attrs={"reference_period": f"{start}:{stop}",
                               "reference_period_weights": "equal" if weights is None else "supplied"})
    hdims = fields[0].dims[1:]
    for name, f, m in zip(("thetao", "so", "volcello"), fields, means):
        reference[name] = DataArray(m, hdims, attrs={**f.attrs, "cell_methods": f"{tcoord}: mean"})
    rho, sums = core.reference_state(means[0], means[1], means[2], pres, eos=eos)
    volo, masso = (float(x) for x in sums.cpu())
    reference["rho"] = DataArray(rho, hdims, attrs={
        "standard_name": "sea_water_density",
        "long_name": "In situ sea water density",
        "comment": f"calculated with the {eos} equation of state from the time-mean thetao and so of the period",
        "units": "kg m-3",
    })
    reference["volo"] = DataArray(np.float64(volo), (), attrs={
        "standard_name": "sea_water_volume", "long_name": "Sea Water Volume", "units": "m3"})
    reference["masso"] = DataArray(np.float64(masso), (), attrs={
        "standard_name": "sea_water_mass", "long_name": "Sea Water Mass", "units": "kg"})
    reference["rhoga"] = DataArray(np.float64(masso) / np.float64(volo), (), attrs={
        "long_name": "Global Average Sea Water Density", "units": "kg m-3"})
    reference["areacello"] = dset["areacello"]
    if xarray_in:
        return xarray_io.to_xarray(reference, like=dset_x)
    return reference


def _device_resident(data):
    """Whether the period means run on the device-resident route: a field is on the device and none is chunked."""
    return (any(isinstance(d, torch.Tensor) and d.is_cuda for d in data)
            and not any(isinstance(d, ChunkedArray) for d in data))


PERIOD_BLOCK_BYTES = 1 << 29  # host blocks are cut to at most this many bytes of one field (but at least one step)


def _host_blocks(arr, start, stop, cap):
    """``(t0, block)`` for the blocks of a host field that overlap steps ``[start, stop)``, in order.  A chunked field
    yields its own blocks, skipping those before the period without copying them and producing none after the one
    that holds step ``stop - 1``; an in-memory field yields views of ``cap`` steps of the period."""
    if isinstance(arr, ChunkedArray):
        t0 = 0
        it = arr.blocks()
        for n in arr.chunks:
            if t0 >= stop:
                return
            blk = next(it)
            if t0 + n > start:
                yield t0, blk
            t0 += n
        return
    for t0 in range(start, stop, cap):
        yield t0, arr[t0: min(t0 + cap, stop)]


def _period_pieces(data, start, stop, cap):
    """Blocks of T, S and V cut at the union of their boundaries, inside ``[start, stop)`` and at most ``cap`` steps
    long: ``(T, S, V)`` views in step order.  One block per field is held at a time."""
    its = [_host_blocks(d, start, stop, cap) for d in data]
    cur = [(0, None)] * 3
    t = start
    while t < stop:
        for j in range(3):
            t0, blk = cur[j]
            while blk is None or t0 + int(blk.shape[0]) <= t:
                t0, blk = next(its[j])
            cur[j] = (t0, blk)
        hi = min([stop, t + cap] + [t0 + int(blk.shape[0]) for t0, blk in cur])
        yield tuple(blk[t - t0: hi - t0] for t0, blk in cur)
        t = hi


def _period_mean_host(data, start, stop, weights):
    """The period means of fields in host memory (numpy, CPU tensors or chunked): streamed through the device."""
    def dt(d):
        s = str(d.dtype)
        return torch.float32 if s.endswith("float32") else torch.float64

    fdt = torch.float32 if dt(data[0]) == dt(data[1]) == torch.float32 else torch.float64
    shape = tuple(int(s) for s in data[0].shape[1:])
    step_bytes = max(4 if fdt == torch.float32 else 8, 4 if dt(data[2]) == torch.float32 else 8) * int(np.prod(shape))
    cap = max(1, PERIOD_BLOCK_BYTES // step_bytes)
    return core.mean_state_blocks(_period_pieces(data, start, stop, cap), shape, fdt, dt(data[2]), weights=weights,
                                  max_steps=cap)
