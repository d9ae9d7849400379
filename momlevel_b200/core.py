"""Array-level API: torch CUDA tensors (or numpy / DLPack objects) in, fp64 CUDA tensors out.

Thin marshalling over the C ABI (``_lib``): torch is the allocator and the stream owner,
every number is computed by libmomlevel_b200's kernels.  Field layout is MOM6 order
``[t][z][y][x]``; trailing horizontal dims are flattened into ``ncol`` for the library.

Each function names the reference code it stands in for; see include/momlevel_b200.h.
"""

import ctypes

import numpy as np
import torch

from . import _lib

__all__ = [
    "to_device",
    "eos_eval",
    "flament_spice",
    "calc_dz",
    "reference_state",
    "steric_local",
    "steric_local_selfref",
    "steric_local_layers",
    "steric_local_layers_variants",
    "steric_local_profile",
    "steric_local_region_profile",
    "steric_local_zonal_profile",
    "layer_edges",
    "delta_rho",
    "steric_global",
    "steric_global_variants",
    "steric_local_host",
    "host_packing",
    "host_last_transfer",
    "host_pack_simd",
    "host_last_timings",
    "host_last_pack_threads",
    "last_path",
    "launch_count",
    "force_direct",
    "variants_chunk",
    "HostStream",
    "weighted_nansum",
    "Pressure",
    "host_release",
]


def _device():
    if not torch.cuda.is_available():
        raise _lib.MLError(-8, "no CUDA device: momlevel_b200 has no CPU path")
    return torch.device("cuda", torch.cuda.current_device())


def to_device(x, dtype=None):
    """numpy / DLPack / torch -> contiguous CUDA tensor (fp32 and fp64 kept, others -> fp64)."""
    dev = _device()
    if isinstance(x, torch.Tensor):
        t = x
    elif isinstance(x, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(x))
    elif hasattr(x, "__dlpack__"):
        t = torch.from_dlpack(x)
    else:
        t = torch.as_tensor(np.asarray(x, dtype=np.float64))
    if dtype is None:
        dtype = t.dtype if t.dtype in (torch.float32, torch.float64) else torch.float64
    return t.to(device=dev, dtype=dtype, non_blocking=True).contiguous()


def _field_dtype(*ts):
    """Common storage dtype of the 3-D/4-D operands (fp32 only if all are fp32)."""
    return torch.float32 if all(t.dtype == torch.float32 for t in ts) else torch.float64


def _dt_id(t):
    return _lib.F32 if t.dtype == torch.float32 else _lib.F64


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _eos_id(eos):
    # util.py:243-249
    assert isinstance(eos, str), "Expecting string for equation of state"
    key = eos.lower()
    if key not in _lib.EOS_IDS:
        raise ValueError(f"Unknown equation of state: {key}")
    return _lib.EOS_IDS[key]


def _f64(x):
    return to_device(x, torch.float64)


class Pressure:
    """``z_l * 1e4 + patm`` (steric.py:96, reference.py:54) when ``patm`` is a 2-D field: the per-level part
    ``[nz]`` and the per-column part ``[ny, nx]``; the kernels evaluate the EOS at ``level[z] + column[y, x]``.
    Every function of this module that takes ``p_level`` takes one of these instead of a plain vector."""

    def __init__(self, level, column):
        self.level = level
        self.column = column


class _ColumnPressure:
    """Context manager: hand the per-column pressure offset to the library for the calls inside (this thread)."""

    def __init__(self, column):
        self.column = None if column is None else _f64(column).contiguous()

    def __enter__(self):
        if self.column is not None:
            _lib.check(_lib.lib().ml_set_column_pressure(self.column.data_ptr(), self.column.numel()))
        return self

    def __exit__(self, *exc):
        if self.column is not None:
            _lib.lib().ml_set_column_pressure(None, 0)
        return False


def _pressure_parts(p):
    """``(p_level, context manager)`` for a plain per-level vector or a :class:`Pressure`."""
    if isinstance(p, Pressure):
        return p.level, _ColumnPressure(p.column)
    return p, _ColumnPressure(None)


def last_path():
    return _lib.lib().ml_last_path()


def launch_count():
    return int(_lib.lib().ml_launch_count())


def force_direct(on):
    """``True`` / 1: direct kernel family only; 2: TMA family without the one-pass three-height kernel; 0: default."""
    return _lib.lib().ml_set_force_direct(2 if on == 2 else (1 if on else 0))


def variants_chunk(tc=0):
    """Time steps per register chunk of the one-pass three-height kernel (4, 6, 8, 12; 0 = default); returns previous."""
    return _lib.lib().ml_set_variants_chunk(int(tc))


# --------------------------------------------------------------------------- elementwise


def eos_eval(eos, func, T, S, p=None, z_axis=None, t_bcast=False, s_bcast=False):
    """``momlevel.eos.<eos>.<func>(T, S, p)`` elementwise, fp64 out, shape of the full operand.

    ``p`` may be a scalar, an array of the full shape, or -- with ``z_axis`` naming the
    level axis of the fields -- a per-level vector ``[nz]`` (what steric.py:96 builds).
    With ``t_bcast`` / ``s_bcast`` that operand lacks the leading (time) axis of the other
    and is broadcast over it (steric.py:115-121); the level axis is then axis 1.
    """
    L = _lib.lib()
    if func not in _lib.FUNC_IDS:
        raise ValueError(f"Unknown equation of state function: {func}")
    eos_id = _eos_id(eos)
    T, S = to_device(T), to_device(S)
    dt = _field_dtype(T, S)
    T, S = T.to(dt), S.to(dt)
    full = S if t_bcast else T
    if t_bcast or s_bcast:
        small = T if t_bcast else S
        if full.dim() < 2 or tuple(small.shape) != tuple(full.shape[1:]):
            raise ValueError("broadcast operand must match the trailing dims of the other")
        z_axis = 1
    elif T.shape != S.shape:
        raise ValueError("T and S must have the same shape")
    if z_axis is not None:
        z_axis = z_axis % full.dim()
        nouter = int(np.prod(full.shape[:z_axis], dtype=np.int64))
        nz = int(full.shape[z_axis])
        ncol = int(np.prod(full.shape[z_axis + 1:], dtype=np.int64))
    else:
        nouter, nz, ncol = 1, 1, full.numel()
    pt, pmode = None, _lib.P_SCALAR
    if p is not None:
        pt = _f64(p)
        if pt.numel() == 1:
            pmode = _lib.P_SCALAR
        elif z_axis is not None and pt.dim() <= 1 and pt.numel() == nz:
            pmode = _lib.P_PER_LEVEL
        elif pt.numel() == full.numel():
            pmode = _lib.P_FULL
        else:
            raise ValueError("pressure must be a scalar, a per-level vector (with z_axis) or full-shape")
    elif eos_id == 0:
        raise ValueError("the Wright equation of state needs a pressure")
    out = torch.empty(full.shape, dtype=torch.float64, device=full.device)
    _lib.check(
        L.ml_eos_eval(eos_id, _lib.FUNC_IDS[func], _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                      pt.data_ptr() if pt is not None else None, pmode, nouter, nz, ncol, out.data_ptr(), _stream())
    )
    return out


def flament_spice(T, S, out=None):
    """``momlevel.spice.flament.spice`` (flament.py:43-95); ``out`` may hand in the fp64 result tensor."""
    L = _lib.lib()
    T, S = to_device(T), to_device(S)
    assert T.shape == S.shape, "thetao and so must have the same shape"  # flament.py:75
    dt = _field_dtype(T, S)
    T, S = T.to(dt), S.to(dt)
    if out is None:
        out = torch.empty(T.shape, dtype=torch.float64, device=T.device)
    assert out.dtype == torch.float64 and out.is_contiguous() and out.numel() == T.numel() and out.device == T.device
    _lib.check(L.ml_flament_spice(_dt_id(T), T.data_ptr(), S.data_ptr(), T.numel(), out.data_ptr(), _stream()))
    return out


def calc_dz(z_i, deptho, top=0.0, bottom=None, fraction=False):
    """``derived.calc_dz`` (derived.py:295-323) -> ``[nz] + deptho.shape`` fp64."""
    L = _lib.lib()
    z_i, depth = _f64(z_i), _f64(deptho)
    nz = z_i.numel() - 1
    out = torch.empty((nz,) + tuple(depth.shape), dtype=torch.float64, device=depth.device)
    _lib.check(
        L.ml_calc_dz(z_i.data_ptr(), depth.data_ptr(), float(top), float(bottom) if bottom is not None else 0.0,
                     int(bottom is not None), int(bool(fraction)), nz, depth.numel(), out.data_ptr(), _stream())
    )
    return out


# ------------------------------------------------------------------------- stratification


def _column_view(x, z_axis):
    """``(nouter, nz, ncol)`` of a C-contiguous field whose level axis is ``z_axis``."""
    z_axis = z_axis % x.dim()
    return (int(np.prod(x.shape[:z_axis], dtype=np.int64)), int(x.shape[z_axis]),
            int(np.prod(x.shape[z_axis + 1:], dtype=np.int64)))


def _fill_mode(shape, z_axis):
    # adjust_negative_n2's ``adjusted[0]`` is index 0 of the FIRST axis (derived.py:63): the surface level
    # when the level axis leads, otherwise every outer slab whose first index is 0 -- the first time step of
    # (time, z, y, x), every time step of member 0 of (member, time, z, y, x), the row y = 0 of (y, x, z)
    z_axis = z_axis % len(shape)
    if z_axis == 0:
        return 0
    return int(np.prod(shape[1:z_axis], dtype=np.int64))


def calc_n2(T, S, z_l, eos="Wright", gravity=-9.8, patm=101325.0, z_axis=1, adjust_negative=False):
    """``derived.calc_n2`` at cell centres (derived.py:391-411), fp64 out, same shape as ``T``."""
    L = _lib.lib()
    T, S = to_device(T), to_device(S)
    assert T.shape == S.shape, "thetao and so must have the same shape"
    dt = _field_dtype(T, S)
    T, S = T.to(dt), S.to(dt)
    nouter, nz, ncol = _column_view(T, z_axis)
    z = _f64(z_l)
    assert z.numel() == nz, "one level coordinate per level"
    out = torch.empty(T.shape, dtype=torch.float64, device=T.device)
    _lib.check(
        L.ml_calc_n2(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), z.data_ptr(), float(gravity), float(patm),
                     int(bool(adjust_negative)), _fill_mode(T.shape, z_axis), nouter, nz, ncol, out.data_ptr(), _stream())
    )
    return out


def adjust_negative_n2(n2, z_axis=1):
    """``derived.adjust_negative_n2`` (derived.py:30-71) on an existing field."""
    L = _lib.lib()
    n2 = _f64(n2)
    nouter, nz, ncol = _column_view(n2, z_axis)
    out = torch.empty_like(n2)
    _lib.check(L.ml_adjust_negative_n2(n2.data_ptr(), _fill_mode(n2.shape, z_axis), nouter, nz, ncol, out.data_ptr(),
                                       _stream()))
    return out


def stability_angle(T, S, p_level, z_l, eos="Wright", z_axis=1):
    """``derived.calc_stability_angle`` (derived.py:714-766) with a per-level pressure."""
    L = _lib.lib()
    T, S = to_device(T), to_device(S)
    assert T.shape == S.shape, "thetao and so must have the same shape"
    dt = _field_dtype(T, S)
    T, S = T.to(dt), S.to(dt)
    nouter, nz, ncol = _column_view(T, z_axis)
    z, p = _f64(z_l), _f64(p_level)
    assert z.numel() == nz and p.numel() == nz
    out = torch.empty(T.shape, dtype=torch.float64, device=T.device)
    _lib.check(
        L.ml_stability_angle(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), p.data_ptr(), z.data_ptr(), nouter,
                             nz, ncol, out.data_ptr(), _stream())
    )
    return out


def wave_speed(n2, dz, z_axis=1):
    """``(sqrt(adjust_negative_n2(n2)) * dz).sum(z) / pi`` (derived.py:821); ``dz`` is ``[nz][...]``."""
    L = _lib.lib()
    n2, dz = _f64(n2), _f64(dz)
    nouter, nz, ncol = _column_view(n2, z_axis)
    assert dz.numel() == nz * ncol, "dz must be [nz][columns]"
    z_axis = z_axis % n2.dim()
    out = torch.empty(tuple(n2.shape[:z_axis]) + tuple(n2.shape[z_axis + 1:]), dtype=torch.float64, device=n2.device)
    _lib.check(L.ml_wave_speed(n2.data_ptr(), dz.data_ptr(), _fill_mode(n2.shape, z_axis), nouter, nz, ncol,
                               out.data_ptr(), _stream()))
    return out


# ------------------------------------------------------------------------------ reducing


def _workspace(nt, nz, ncol, device):
    n = _lib.lib().ml_workspace_bytes(nt, nz, ncol)
    return torch.empty((n + 7) // 8, dtype=torch.float64, device=device), n


def reference_state(T0, S0, V0, p_level, eos="Wright", out=None):
    """``reference.setup_reference_state`` arithmetic (reference.py:71-80).

    Returns ``(rho_ref [nz,...] fp64, sums fp64[2] = {volo, masso})`` on the device; ``out`` may hand
    in those two tensors when the caller manages streams.
    """
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T0, S0, V0 = to_device(T0), to_device(S0), to_device(V0)
    dt = _field_dtype(T0, S0, V0)
    T0, S0, V0 = T0.to(dt), S0.to(dt), V0.to(dt)
    assert T0.shape == S0.shape == V0.shape
    nz = T0.shape[0]
    ncol = T0.numel() // nz
    p = _f64(p_level)
    if out is not None:
        rho, sums = out
        assert rho.dtype == sums.dtype == torch.float64 and rho.is_contiguous() and rho.numel() == T0.numel()
        assert sums.numel() == 2
    else:
        rho = torch.empty(T0.shape, dtype=torch.float64, device=T0.device)
        sums = torch.empty(2, dtype=torch.float64, device=T0.device)
    ws, nbytes = _workspace(2, nz, ncol, T0.device)
    with _pcol:
        _lib.check(
            L.ml_reference_state(_eos_id(eos), _dt_id(T0), T0.data_ptr(), S0.data_ptr(), V0.data_ptr(), p.data_ptr(), nz,
                                 ncol, rho.data_ptr(), sums.data_ptr(), ws.data_ptr(), nbytes, _stream())
        )
    return rho, sums


def weighted_nansum(a, w=None, nrows=1):
    """``out[r] = nansum(a[r] * w)`` (``w=None``: ``nansum(a[r])``) for ``a`` viewed as ``[nrows, n]`` -- the sums of
    ``derived.calc_masso`` (derived.py:435-438) and ``derived.calc_volo`` (:787-789) on fields that already exist,
    in two fixed-order stages and without the ``rho * volcello`` temporary.  fp64 ``[nrows]`` on the device."""
    L = _lib.lib()
    a = to_device(a)
    n = a.numel() // max(int(nrows), 1)
    wt = None
    if w is not None:
        wt = to_device(w)
        assert wt.numel() == n, "one weight per point of a row"
    out = torch.empty(int(nrows), dtype=torch.float64, device=a.device)
    ws = torch.empty(int(nrows) * 1184, dtype=torch.float64, device=a.device)
    _lib.check(L.ml_calc_masso(_dt_id(a), a.data_ptr(), _dt_id(wt) if wt is not None else 0,
                               wt.data_ptr() if wt is not None else None, int(nrows), n, out.data_ptr(), ws.data_ptr(),
                               ws.numel() * 8, _stream()))
    return out


def _steric_operands(T, S, t_bcast, s_bcast):
    T, S = to_device(T), to_device(S)
    dt = _field_dtype(T, S)
    T, S = T.to(dt), S.to(dt)
    full = S if t_bcast else T
    nt, nz = full.shape[0], full.shape[1]
    hshape = tuple(full.shape[2:])
    ncol = int(np.prod(hshape, dtype=np.int64))
    if t_bcast or s_bcast:
        small = T if t_bcast else S
        if tuple(small.shape) != tuple(full.shape[1:]):
            raise ValueError("broadcast operand must be [nz][...]")
    elif T.shape != S.shape:
        raise ValueError("T and S must have the same shape")
    return T, S, nt, nz, ncol, hshape


def steric_local(T, S, rho_ref, v_ref, z_i, deptho, p_level, rhozero=1035.0, eos="Wright", t_bcast=False,
                 s_bcast=False, want_delta_rho=False, eta_out=None):
    """Local branch of ``steric.steric`` (steric.py:128,150-166).

    Returns ``(eta [nt,...], delta_rho [nt,nz,...] or None)`` fp64 on the device; ``eta_out`` may hand in
    the height tensor when the caller manages streams.
    """
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, t_bcast, s_bcast)
    rho_ref = _f64(rho_ref)
    v_ref = to_device(v_ref)
    z_i, depth, p = _f64(z_i), _f64(deptho), _f64(p_level)
    assert rho_ref.numel() == nz * ncol and v_ref.numel() == nz * ncol and depth.numel() == ncol
    assert z_i.numel() == nz + 1 and p.numel() == nz
    if eta_out is not None:
        eta = eta_out
        assert eta.dtype == torch.float64 and eta.is_contiguous() and eta.numel() == nt * ncol
    else:
        eta = torch.empty((nt,) + hshape, dtype=torch.float64, device=T.device)
    drho = torch.empty((nt, nz) + hshape, dtype=torch.float64, device=T.device) if want_delta_rho else None
    with _pcol:
        _lib.check(
            L.ml_steric_local(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                              rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref), z_i.data_ptr(), depth.data_ptr(),
                              p.data_ptr(), -1.0 / rhozero, nt, nz, ncol, eta.data_ptr(),
                              drho.data_ptr() if drho is not None else None, _stream())
        )
    return eta, drho


def layer_edges(edges):
    """Depth-layer edges as a float64 numpy array: ``None`` as the last edge means "to the sea floor" and becomes
    ``inf`` (``calc_dz(bottom=None)`` is ``calc_dz(bottom=inf)``, derived.py:297-298).  Raises ``ValueError`` unless
    there are 2 to ``MAX_LAYERS + 1`` edges, strictly increasing, >= 0, with only the last one infinite."""
    try:
        vals = list(edges)
    except TypeError:
        raise ValueError(f"depth edges must be a sequence of depths, got {edges!r}") from None
    if not 2 <= len(vals) <= _lib.MAX_LAYERS + 1:
        raise ValueError(f"depth edges must give 1 to {_lib.MAX_LAYERS} layers, got {len(vals)} edges")
    out = []
    for i, v in enumerate(vals):
        if v is None:
            if i != len(vals) - 1:
                raise ValueError("only the last depth edge may be None (to the sea floor)")
            v = np.inf
        try:
            v = float(v)
        except (TypeError, ValueError):
            raise ValueError(f"depth edge {v!r} is not a number") from None
        if np.isnan(v) or v < 0.0 or (np.isinf(v) and i != len(vals) - 1):
            raise ValueError(f"depth edges must be >= 0 and finite except the last, got {v!r}")
        if out and not v > out[-1]:
            raise ValueError(f"depth edges must be strictly increasing, got {vals!r}")
        out.append(v)
    return np.asarray(out, dtype=np.float64)


def steric_local_layers(T, S, rho_ref, v_ref, z_i, deptho, p_level, edges, rhozero=1035.0, eos="Wright", t_bcast=False,
                        s_bcast=False):
    """The local branch (steric.py:150-166) split by depth layer: layer ``b`` integrates with
    ``calc_dz(top=edges[b], bottom=edges[b+1])`` (derived.py:249-325) in place of the full-column thickness.

    ``edges`` as :func:`layer_edges`.  Returns ``eta [nt, nlayers, ...]`` fp64 on the device, from one pass over
    T and S (``ml_steric_local_layers``).
    """
    L = _lib.lib()
    e = layer_edges(edges)
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, t_bcast, s_bcast)
    rho_ref = _f64(rho_ref)
    v_ref = to_device(v_ref)
    z_i, depth, p = _f64(z_i), _f64(deptho), _f64(p_level)
    assert rho_ref.numel() == nz * ncol and v_ref.numel() == nz * ncol and depth.numel() == ncol
    assert z_i.numel() == nz + 1 and p.numel() == nz
    nl = e.size - 1
    eta = torch.empty((nt, nl) + hshape, dtype=torch.float64, device=T.device)
    with _pcol:
        _lib.check(
            L.ml_steric_local_layers(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                                     rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref), z_i.data_ptr(),
                                     depth.data_ptr(), p.data_ptr(), -1.0 / rhozero,
                                     e.ctypes.data_as(ctypes.c_void_p), nl, nt, nz, ncol, eta.data_ptr(), _stream())
        )
    return eta


VARIANTS = ("steric", "thermosteric", "halosteric")


def variant_names(variants):
    """``variants`` as a tuple of distinct names from :data:`VARIANTS`; ``ValueError`` for an empty sequence, a
    duplicate or an unknown name."""
    names = (variants,) if isinstance(variants, str) else tuple(variants)
    unknown = [v for v in names if v not in VARIANTS]
    if unknown:
        raise ValueError(f"Unknown variants {unknown}: expected names from {VARIANTS}")
    if not names:
        raise ValueError("at least one variant is required")
    if len(set(names)) != len(names):
        raise ValueError(f"variants must be distinct, got {list(names)}")
    return names


def steric_local_layers_variants(T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, edges, rhozero=1035.0,
                                 eos="Wright", variants=VARIANTS):
    """:func:`steric_local_layers` for the steric, thermosteric and halosteric heights (steric.py:115-121) in one call.

    ``T_ref, S_ref, rho_ref`` are the reference state (``reference["thetao"]``, ``["so"]``, ``["rho"]``); ``variants``
    may name a subset.  Returns ``{variant: eta [nt, nlayers, ...]}`` fp64 on the device, from one pass over T and S
    when the fields suit it (``ml_steric_local_layers_variants``).
    """
    L = _lib.lib()
    names = variant_names(variants)
    e = layer_edges(edges)
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, False, False)
    Tr, Sr = to_device(T_ref), to_device(S_ref)
    dt = _field_dtype(T, S, Tr, Sr)
    T, S, Tr, Sr = T.to(dt), S.to(dt), Tr.to(dt), Sr.to(dt)
    rho_ref = _f64(rho_ref)
    v_ref = to_device(v_ref)
    z_i, depth, p = _f64(z_i), _f64(deptho), _f64(p_level)
    assert Tr.numel() == nz * ncol and Sr.numel() == nz * ncol and rho_ref.numel() == nz * ncol
    assert v_ref.numel() == nz * ncol and depth.numel() == ncol and z_i.numel() == nz + 1 and p.numel() == nz
    nl = e.size - 1
    eta = {v: torch.empty((nt, nl) + hshape, dtype=torch.float64, device=T.device) for v in names}
    ptr = lambda v: eta[v].data_ptr() if v in eta else None  # noqa: E731
    with _pcol:
        _lib.check(
            L.ml_steric_local_layers_variants(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(),
                                              Sr.data_ptr(), rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref),
                                              z_i.data_ptr(), depth.data_ptr(), p.data_ptr(), -1.0 / rhozero,
                                              e.ctypes.data_as(ctypes.c_void_p), nl, nt, nz, ncol, ptr("steric"),
                                              ptr("thermosteric"), ptr("halosteric"), _stream())
        )
    return eta


def steric_local_profile(T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, rhozero=1035.0,
                         eos="Wright", variants=VARIANTS):
    """The area-weighted height change of each level, ``-1/rhozero * nansum_col(m * w * dz * delta_rho) /
    nansum(w)`` (steric.py:115-121, :151-166, derived.py:295-318), for the variants asked for.

    ``T_ref, S_ref, rho_ref`` are the reference state (``reference["thetao"]``, ``["so"]``, ``["rho"]``); ``weights``
    is one weight per column (``areacello``, or ``areacello`` times a basin mask; NaN counts as 0).  Returns
    ``{variant: [nt, nz]}`` fp64 on the device, from one pass over T and S (``ml_steric_local_profile``).
    """
    L = _lib.lib()
    names = variant_names(variants)
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, _ = _steric_operands(T, S, False, False)
    Tr, Sr = to_device(T_ref), to_device(S_ref)
    dt = _field_dtype(T, S, Tr, Sr)
    T, S, Tr, Sr = T.to(dt), S.to(dt), Tr.to(dt), Sr.to(dt)
    rho_ref = _f64(rho_ref)
    v_ref = to_device(v_ref)
    z_i, depth, p, w = _f64(z_i), _f64(deptho), _f64(p_level), _f64(weights)
    assert Tr.numel() == nz * ncol and Sr.numel() == nz * ncol and rho_ref.numel() == nz * ncol
    assert v_ref.numel() == nz * ncol and depth.numel() == ncol and z_i.numel() == nz + 1 and p.numel() == nz
    if w.numel() != ncol:
        raise ValueError(f"one weight per column: got {w.numel()} weights for {ncol} columns")
    prof = {v: torch.empty((nt, nz), dtype=torch.float64, device=T.device) for v in names}
    nbytes = L.ml_profile_workspace_bytes(len(names), nt, nz, ncol)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=T.device)
    ptr = lambda v: prof[v].data_ptr() if v in prof else None  # noqa: E731
    with _pcol:
        _lib.check(
            L.ml_steric_local_profile(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(),
                                      rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref), z_i.data_ptr(),
                                      depth.data_ptr(), w.data_ptr(), p.data_ptr(), -1.0 / rhozero, nt, nz, ncol,
                                      ptr("steric"), ptr("thermosteric"), ptr("halosteric"), ws.data_ptr(), nbytes,
                                      _stream())
        )
    total = torch.nansum(w)
    return {v: prof[v] / total for v in names}


REGION_WORKSPACE_BYTES = 512 << 20  # the most steric_local_region_profile allocates for partials; the time axis is chunked


def steric_local_region_profile(T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, region_index,
                                nregions, rhozero=1035.0, eos="Wright", variants=VARIANTS):
    """:func:`steric_local_profile` for every region of a region map, from one pass over T and S
    (``ml_steric_local_region_profile``).

    ``region_index`` holds one integer per column: in ``[0, nregions)`` the column's region, any other value (e.g.
    -1) no region; ``1 <= nregions <= 15``.  Region ``r`` is, bit for bit, :func:`steric_local_profile` with
    ``weights=where(region_index == r, weights, 0)``.  Returns ``({variant: [nregions, nt, nz]}, totals[nregions])``
    fp64 on the device: the profiles already divided by ``totals``, each region's ``nansum`` of the weights (0/0,
    NaN, for a region without columns).
    """
    L = _lib.lib()
    names = variant_names(variants)
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, _ = _steric_operands(T, S, False, False)
    Tr, Sr = to_device(T_ref), to_device(S_ref)
    dt = _field_dtype(T, S, Tr, Sr)
    T, S, Tr, Sr = T.to(dt), S.to(dt), Tr.to(dt), Sr.to(dt)
    rho_ref = _f64(rho_ref)
    v_ref = to_device(v_ref)
    z_i, depth, p, w = _f64(z_i), _f64(deptho), _f64(p_level), _f64(weights)
    assert Tr.numel() == nz * ncol and Sr.numel() == nz * ncol and rho_ref.numel() == nz * ncol
    assert v_ref.numel() == nz * ncol and depth.numel() == ncol and z_i.numel() == nz + 1 and p.numel() == nz
    if w.numel() != ncol:
        raise ValueError(f"one weight per column: got {w.numel()} weights for {ncol} columns")
    nregions = int(nregions)
    if not 1 <= nregions <= _lib.MAX_REGIONS:
        raise ValueError(f"nregions={nregions}: between 1 and {_lib.MAX_REGIONS} regions")
    ri = torch.as_tensor(region_index, device=T.device)
    if ri.numel() != ncol:
        raise ValueError(f"one region index per column: got {ri.numel()} for {ncol} columns")
    ri = torch.where((ri >= 0) & (ri < nregions), ri, -1).to(torch.int8).reshape(w.shape).contiguous()
    prof = {v: torch.empty((nregions, nt, nz), dtype=torch.float64, device=T.device) for v in names}
    step = L.ml_region_profile_workspace_bytes(len(names), nregions, 1, nz, ncol) - 256
    steps = max(1, min(nt, (REGION_WORKSPACE_BYTES - 256) // step))
    nbytes = L.ml_region_profile_workspace_bytes(len(names), nregions, steps, nz, ncol)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=T.device)
    ptr = lambda v: prof[v].data_ptr() if v in prof else None  # noqa: E731
    with _pcol:
        _lib.check(
            L.ml_steric_local_region_profile(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(),
                                             Sr.data_ptr(), rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref),
                                             z_i.data_ptr(), depth.data_ptr(), w.data_ptr(), ri.data_ptr(), nregions,
                                             p.data_ptr(), -1.0 / rhozero, nt, nz, ncol, ptr("steric"),
                                             ptr("thermosteric"), ptr("halosteric"), ws.data_ptr(), nbytes, _stream())
        )
    # each total as steric_local_profile forms it from the masked weights, so that the quotients match bit for bit
    totals = torch.stack([torch.nansum(torch.where(ri == r, w, 0.0)) for r in range(nregions)])
    return {v: prof[v] / totals[:, None, None] for v in names}, totals


def steric_local_zonal_profile(T, S, T_ref, S_ref, rho_ref, v_ref, z_i, deptho, p_level, weights, rhozero=1035.0,
                               eos="Wright", variants=VARIANTS):
    """:func:`steric_local_profile` for every grid row at once, from one pass over T and S
    (``ml_steric_local_zonal_profile``).

    ``T, S`` are ``[nt, nz, ny, nx]``, ``weights`` is ``[ny, nx]``.  Row ``j`` is, bit for bit,
    :func:`steric_local_profile` on the operands of row ``j`` alone (sliced to ``[..., j:j+1, :]``).  Returns
    ``({variant: [nt, nz, ny]}, totals[ny])`` fp64 on the device: the sections already divided by ``totals``, each
    row's ``nansum`` of the weights (0/0, NaN, for a row whose weights sum to 0).
    """
    L = _lib.lib()
    names = variant_names(variants)
    p_level, _pcol = _pressure_parts(p_level)
    T, S = to_device(T), to_device(S)
    if T.dim() != 4 or tuple(S.shape) != tuple(T.shape):
        raise ValueError(f"fields laid out (time, z, y, x): got {tuple(T.shape)} and {tuple(S.shape)}")
    T, S, nt, nz, ncol, _ = _steric_operands(T, S, False, False)
    ny, nx = T.shape[2], T.shape[3]
    Tr, Sr = to_device(T_ref), to_device(S_ref)
    dt = _field_dtype(T, S, Tr, Sr)
    T, S, Tr, Sr = T.to(dt), S.to(dt), Tr.to(dt), Sr.to(dt)
    rho_ref = _f64(rho_ref)
    v_ref = to_device(v_ref)
    z_i, depth, p, w = _f64(z_i), _f64(deptho), _f64(p_level), _f64(weights)
    assert Tr.numel() == nz * ncol and Sr.numel() == nz * ncol and rho_ref.numel() == nz * ncol
    assert v_ref.numel() == nz * ncol and depth.numel() == ncol and z_i.numel() == nz + 1 and p.numel() == nz
    if tuple(w.shape) != (ny, nx):
        raise ValueError(f"weights of shape {tuple(w.shape)} do not match the horizontal grid {(ny, nx)}")
    prof = {v: torch.empty((nt, nz, ny), dtype=torch.float64, device=T.device) for v in names}
    step = L.ml_zonal_profile_workspace_bytes(len(names), 1, nz, ny, nx) - 256
    steps = max(1, min(nt, (REGION_WORKSPACE_BYTES - 256) // step))
    nbytes = L.ml_zonal_profile_workspace_bytes(len(names), steps, nz, ny, nx)
    ws = torch.empty((nbytes + 7) // 8, dtype=torch.float64, device=T.device)
    ptr = lambda v: prof[v].data_ptr() if v in prof else None  # noqa: E731
    with _pcol:
        _lib.check(
            L.ml_steric_local_zonal_profile(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(),
                                            Sr.data_ptr(), rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref),
                                            z_i.data_ptr(), depth.data_ptr(), w.data_ptr(), p.data_ptr(),
                                            -1.0 / rhozero, nt, nz, ny, nx, ptr("steric"), ptr("thermosteric"),
                                            ptr("halosteric"), ws.data_ptr(), nbytes, _stream())
        )
    # each total as steric_local_profile forms it, torch.nansum of the row's weights in a buffer of their own, so that
    # the quotients match bit for bit: torch's reduction order follows the alignment of its input, so every row is
    # first given a start aligned as a fresh allocation is (one copy), then summed alone
    pitch = -(-nx // 64) * 64  # 512 bytes
    wp = w.new_zeros((ny, pitch))
    wp[:, :nx] = w
    totals = torch.stack([torch.nansum(wp[j, :nx]) for j in range(ny)])
    return {v: prof[v] / totals for v in names}, totals


def delta_rho(T, S, rho_ref, v_ref, p_level, eos="Wright", t_bcast=False, s_bcast=False):
    """``where(v_ref.notnull(), rho - rho_ref, nan)`` time-first (steric.py:151-158), fp64 on the device."""
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, t_bcast, s_bcast)
    rho_ref, v_ref, p = _f64(rho_ref), to_device(v_ref), _f64(p_level)
    assert rho_ref.numel() == nz * ncol and v_ref.numel() == nz * ncol and p.numel() == nz
    out = torch.empty((nt, nz) + hshape, dtype=torch.float64, device=T.device)
    with _pcol:
        _lib.check(
            L.ml_delta_rho(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                           rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref), p.data_ptr(), nt, nz, ncol,
                           out.data_ptr(), _stream())
        )
    return out


def delta_rho_annual(T, S, rho_ref, v_ref, p_level, days_in_month, eos="Wright", t_bcast=False, s_bcast=False):
    """Annual means of ``delta_rho`` weighted by ``days_in_month`` (util.py:84-87 applied to steric.py:151-158).

    ``[nt/12, nz, ...]`` fp64 on the device; the monthly 4-D anomaly is never materialised.
    """
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, t_bcast, s_bcast)
    rho_ref, v_ref, p, w = _f64(rho_ref), to_device(v_ref), _f64(p_level), _f64(days_in_month)
    assert rho_ref.numel() == nz * ncol and v_ref.numel() == nz * ncol and p.numel() == nz
    assert w.numel() == nt and nt % 12 == 0, "annual averaging needs whole years of monthly data"
    out = torch.empty((nt // 12, nz) + hshape, dtype=torch.float64, device=T.device)
    with _pcol:
        _lib.check(
            L.ml_delta_rho_annual(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                                  rho_ref.data_ptr(), v_ref.data_ptr(), _dt_id(v_ref), p.data_ptr(), w.data_ptr(), nt, nz,
                                  ncol, out.data_ptr(), _stream())
        )
    return out


def selfref_outputs(T, S, t_bcast=False, s_bcast=False):
    """Empty ``(eta, rho_ref, sums)`` for :func:`steric_local_selfref`, allocated on the current stream."""
    full = S if t_bcast else T
    nt, nz, hshape = full.shape[0], full.shape[1], tuple(full.shape[2:])
    dev = full.device
    return (torch.empty((nt,) + hshape, dtype=torch.float64, device=dev),
            torch.empty((nz,) + hshape, dtype=torch.float64, device=dev),
            torch.empty(2, dtype=torch.float64, device=dev))


def steric_local_selfref(T, S, v_ref, z_i, deptho, p_level, rhozero=1035.0, eos="Wright", t_bcast=False, s_bcast=False,
                         out=None, want_rho_ref=True):
    """``setup_reference_state`` + the local branch in one pass; reference = step 0 (steric.py:105-107).

    A broadcast operand is the step-0 slab of that field.  Returns
    ``(eta [nt,...], rho_ref [nz,...], sums fp64[2] = {volo, masso})`` on the device; ``out`` may
    hand in those three tensors (see :func:`selfref_outputs`) when the caller manages streams.
    ``want_rho_ref=False`` asks the library not to store the reference density (7 % of the traffic of a
    12-step call); ``rho_ref`` is then ``None`` unless the layout needs it internally (more than 12 steps, or
    fields the TMA family does not take), in which case it is produced anyway.
    """
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, t_bcast, s_bcast)
    v_ref = to_device(v_ref)
    z_i, depth, p = _f64(z_i), _f64(deptho), _f64(p_level)
    assert v_ref.numel() == nz * ncol and depth.numel() == ncol and z_i.numel() == nz + 1 and p.numel() == nz
    if out is not None:
        eta, rho, sums = out
    else:
        eta = torch.empty((nt,) + hshape, dtype=torch.float64, device=T.device)
        sums = torch.empty(2, dtype=torch.float64, device=T.device)
        rho = torch.empty((nz,) + hshape, dtype=torch.float64, device=T.device) if want_rho_ref else None
    assert eta.dtype == sums.dtype == torch.float64 and eta.is_contiguous()
    assert eta.numel() == nt * ncol and sums.numel() == 2
    assert rho is None or (rho.dtype == torch.float64 and rho.is_contiguous() and rho.numel() == nz * ncol)
    ws, nbytes = _workspace(2, nz, ncol, T.device)

    def call(rho_t):
        return L.ml_steric_local_selfref(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                                         v_ref.data_ptr(), _dt_id(v_ref), z_i.data_ptr(), depth.data_ptr(), p.data_ptr(),
                                         -1.0 / rhozero, nt, nz, ncol, eta.data_ptr(),
                                         rho_t.data_ptr() if rho_t is not None else None, sums.data_ptr(),
                                         ws.data_ptr(), nbytes, _stream())

    with _pcol:
        rc = call(rho)
        if rc == -1 and rho is None:  # ML_ERR_NULL: this layout needs the field itself
            rho = torch.empty((nz,) + hshape, dtype=torch.float64, device=T.device)
            rc = call(rho)
        _lib.check(rc)
    return eta, rho, sums


def steric_local_variants(T, S, v_ref, z_i, deptho, p_level, T_ref=None, S_ref=None, rho_ref=None, rhozero=1035.0,
                          eos="Wright", want_rho_ref=True):
    """Steric, thermosteric and halosteric height in one call (steric.py:115-121, :150-166).

    ``T_ref, S_ref`` default to step 0 of ``T, S`` (what ``steric()`` does without ``reference=``); with
    ``rho_ref=None`` the reference density is evaluated on the way.  The four operands are stored in one dtype:
    fp32 only if all four are fp32, so an fp64 reference slab is never rounded to fp32 fields.  Returns
    ``({"steric": eta, "thermosteric": eta, "halosteric": eta}, rho_ref, sums or None)`` on the device.
    ``want_rho_ref=False`` (self-reference calls only) asks the library not to store the reference density when
    the one-pass kernel does not need the field; ``rho_ref`` is then ``None`` unless the layout needs it.
    """
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, hshape = _steric_operands(T, S, False, False)
    Tr = T[0] if T_ref is None else to_device(T_ref)
    Sr = S[0] if S_ref is None else to_device(S_ref)
    dt = _field_dtype(T, S, Tr, Sr)
    T, S, Tr, Sr = T.to(dt), S.to(dt), Tr.to(dt), Sr.to(dt)
    assert Tr.is_contiguous() and Sr.is_contiguous() and Tr.numel() == nz * ncol and Sr.numel() == nz * ncol
    v_ref = to_device(v_ref)
    z_i, depth, p = _f64(z_i), _f64(deptho), _f64(p_level)
    assert v_ref.numel() == nz * ncol and depth.numel() == ncol and z_i.numel() == nz + 1 and p.numel() == nz
    eta = torch.empty((3, nt) + hshape, dtype=torch.float64, device=T.device)
    sums, ws, nbytes = None, None, 0
    if rho_ref is None:
        store = want_rho_ref or T_ref is not None or S_ref is not None
        rho = torch.empty((nz,) + hshape, dtype=torch.float64, device=T.device) if store else None
        sums = torch.empty(2, dtype=torch.float64, device=T.device)
        ws, nbytes = _workspace(2, nz, ncol, T.device)
        rho_in = None
    else:
        rho = _f64(rho_ref)
        assert rho.numel() == nz * ncol
        rho_in = rho.data_ptr()

    def call(rho_t):
        return L.ml_steric_local_variants(
            _eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), rho_in, v_ref.data_ptr(),
            _dt_id(v_ref), z_i.data_ptr(), depth.data_ptr(), p.data_ptr(), -1.0 / rhozero, nt, nz, ncol,
            eta[0].data_ptr(), eta[1].data_ptr(), eta[2].data_ptr(),
            rho_t.data_ptr() if (rho_ref is None and rho_t is not None) else None,
            sums.data_ptr() if sums is not None else None, ws.data_ptr() if ws is not None else None, nbytes, _stream())

    with _pcol:
        rc = call(rho)
        if rc == -1 and rho is None:  # ML_ERR_NULL: this layout needs the field itself
            rho = torch.empty((nz,) + hshape, dtype=torch.float64, device=T.device)
            rc = call(rho)
        _lib.check(rc)
    return {"steric": eta[0], "thermosteric": eta[1], "halosteric": eta[2]}, rho, sums


def steric_global(T, S, v_ref, p_level, eos="Wright", t_bcast=False, s_bcast=False):
    """``calc_masso(rho, reference.volcello)`` of the global branch (steric.py:135) -> ``masso[nt]``."""
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, _ = _steric_operands(T, S, t_bcast, s_bcast)
    v_ref = to_device(v_ref)
    p = _f64(p_level)
    assert v_ref.numel() == nz * ncol and p.numel() == nz
    masso = torch.empty(nt, dtype=torch.float64, device=T.device)
    ws, nbytes = _workspace(nt, nz, ncol, T.device)
    with _pcol:
        _lib.check(
            L.ml_steric_global(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), int(t_bcast), int(s_bcast),
                               v_ref.data_ptr(), _dt_id(v_ref), p.data_ptr(), nt, nz, ncol, masso.data_ptr(),
                               ws.data_ptr(), nbytes, _stream())
        )
    return masso


GLOBAL_VARIANTS = VARIANTS


def steric_global_variants(T, S, v_ref, p_level, T_ref=None, S_ref=None, eos="Wright", variants=GLOBAL_VARIANTS):
    """The masses of the global steric, thermosteric and halosteric series in one call (steric.py:115-121, :135).

    ``T_ref, S_ref`` default to step 0 of ``T, S`` (what ``steric()`` does without ``reference=``); the sums
    ``{volo, masso}`` of that reference state are then produced on the way.  ``variants`` may name a subset.
    The four operands are stored in one dtype: fp32 only if all four are fp32, so an fp64 reference slab is never
    rounded to fp32 fields.
    Returns ``({variant: masso[nt]}, sums fp64[2] or None)`` on the device (``ml_steric_global_variants``).
    """
    L = _lib.lib()
    p_level, _pcol = _pressure_parts(p_level)
    T, S, nt, nz, ncol, _ = _steric_operands(T, S, False, False)
    if (T_ref is None) != (S_ref is None):
        raise ValueError("T_ref and S_ref are given together or not at all")
    Tr = T if T_ref is None else to_device(T_ref)
    Sr = S if S_ref is None else to_device(S_ref)
    dt = _field_dtype(T, S, Tr, Sr)
    T, S, Tr, Sr = T.to(dt), S.to(dt), Tr.to(dt).contiguous(), Sr.to(dt).contiguous()
    selfref = Tr.data_ptr() == T.data_ptr() and Sr.data_ptr() == S.data_ptr()  # step 0 of the fields themselves
    assert selfref or (Tr.numel() == nz * ncol and Sr.numel() == nz * ncol)
    v_ref = to_device(v_ref)
    p = _f64(p_level)
    assert v_ref.numel() == nz * ncol and p.numel() == nz
    unknown = set(variants) - set(GLOBAL_VARIANTS)
    if unknown or not variants:
        raise ValueError(f"Unknown variants {sorted(unknown)}" if unknown else "at least one variant is required")
    masso = torch.empty((3, nt), dtype=torch.float64, device=T.device)
    sums = torch.empty(2, dtype=torch.float64, device=T.device) if selfref else None
    ws, nbytes = _workspace(3 * nt, nz, ncol, T.device)
    ptr = lambda i: masso[i].data_ptr() if GLOBAL_VARIANTS[i] in variants else None  # noqa: E731
    with _pcol:
        _lib.check(
            L.ml_steric_global_variants(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(),
                                        v_ref.data_ptr(), _dt_id(v_ref), p.data_ptr(), nt, nz, ncol, ptr(0), ptr(1), ptr(2),
                                        sums.data_ptr() if sums is not None else None, ws.data_ptr(), nbytes, _stream())
        )
    return {v: masso[i] for i, v in enumerate(GLOBAL_VARIANTS) if v in variants}, sums


def _host_tensor(x):
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    assert t.device.type == "cpu"
    return t.contiguous()


def steric_local_host(T, S, V0, z_i, deptho, p_level, rhozero=1035.0, eos="Wright", steps_per_window=1,
                      want_rho_ref=False, eta_out=None, variants=False):
    """End-to-end host call: HOST arrays in (numpy or CPU torch, pinned for speed), CPU tensors out.

    ``reference_state`` + ``steric_local`` for variant="steric" with the reference taken
    from time step 0; copies are pipelined against the kernels inside the library.
    Returns ``(eta [nt,...], rho_ref or None, (volo, masso))``.  With ``variants=True`` ``eta`` is a dict
    ``{"steric", "thermosteric", "halosteric"}``: the fields cross PCIe once and every window is
    integrated three times on the device (``ml_steric_local_variants_host``); a tuple of names asks for steric
    plus those.  ``eta_out`` may hand in
    the output tensor (or, with ``variants``, a dict of them) -- pinned memory keeps the read-back asynchronous.
    """
    L = _lib.lib()
    _device()
    T, S, V0 = _host_tensor(T), _host_tensor(S), _host_tensor(V0)
    dt = _field_dtype(T, S, V0)
    T, S, V0 = T.to(dt), S.to(dt), V0.to(dt)
    nt, nz = T.shape[0], T.shape[1]
    hshape = tuple(T.shape[2:])
    ncol = int(np.prod(hshape, dtype=np.int64))
    z_i = _host_tensor(np.asarray(z_i, dtype=np.float64))
    depth = _host_tensor(np.asarray(deptho, dtype=np.float64))
    p = _host_tensor(np.asarray(p_level, dtype=np.float64))
    outs = eta_out if isinstance(eta_out, dict) else {"steric": eta_out}
    eta = outs.get("steric")
    if eta is None:
        eta = torch.empty((nt,) + hshape, dtype=torch.float64)
    rho = torch.empty((nz,) + hshape, dtype=torch.float64) if want_rho_ref else None
    sums = torch.empty(2, dtype=torch.float64)
    head = (_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), V0.data_ptr(), z_i.data_ptr(), depth.data_ptr(),
            p.data_ptr(), -1.0 / rhozero, nt, nz, ncol, int(steps_per_window))
    tail = (rho.data_ptr() if rho is not None else None, sums.data_ptr())
    if not variants:
        _lib.check(L.ml_steric_local_host(*head, eta.data_ptr(), *tail))
        return eta, rho, (float(sums[0]), float(sums[1]))
    wanted = ("thermosteric", "halosteric") if variants is True else tuple(v for v in variants if v != "steric")
    extra = {}
    for name in ("thermosteric", "halosteric"):
        if name in wanted:
            extra[name] = outs.get(name) if outs.get(name) is not None else torch.empty_like(eta)
    ptr = lambda name: extra[name].data_ptr() if name in extra else None  # noqa: E731
    _lib.check(L.ml_steric_local_variants_host(*head, eta.data_ptr(), ptr("thermosteric"), ptr("halosteric"), *tail))
    return {"steric": eta, **extra}, rho, (float(sums[0]), float(sums[1]))


def host_packing(mode=1, threads=0):
    """How the ``*_host`` calls of this thread move level rows: 0 = as they are, 1 = compressed to their
    present cells where the host cores have time for it (default), 2 = every row with absent cells compressed.
    The results do not depend on it (``ml_host_set_packing``)."""
    _lib.check(_lib.lib().ml_host_set_packing(int(mode), int(threads)))


def host_last_transfer():
    """``(host->device bytes, share of level rows that crossed packed)`` of this thread's last ``*_host`` call."""
    L = _lib.lib()
    return int(L.ml_host_last_h2d_bytes()), float(L.ml_host_last_packed_fraction())


def host_last_pack_threads():
    """Packing threads of this thread's last window: with ``host_packing(1, 0)`` the library tunes the number itself."""
    return int(_lib.lib().ml_host_last_pack_threads())


def host_last_timings():
    """Host wall time of this thread's last ``steric_local_host`` call in ms: presence index, windows, drain, whole call."""
    out = (ctypes.c_double * 4)()
    _lib.check(_lib.lib().ml_host_last_timings(ctypes.cast(out, ctypes.c_void_p)))
    return {"presence_index_ms": out[0], "windows_ms": out[1], "drain_ms": out[2], "call_ms": out[3]}


def host_pack_simd():
    """512 when the host-side packing loops run their AVX-512 bodies, 0 for the scalar ones."""
    return int(_lib.lib().ml_pack_simd())


def steric_global_host(T, S, v_ref, p_level, eos="Wright", steps_per_window=1):
    """Per-step masses of the global branch (steric.py:135) for HOST arrays, streamed through device windows.

    Returns ``masso[nt]`` as a CPU tensor; ``distributed.global_sea_level`` applies the ``ln`` formula.
    """
    L = _lib.lib()
    _device()
    host = _host_tensor
    T, S, v_ref = host(T), host(S), host(v_ref)
    dt = _field_dtype(T, S, v_ref)
    T, S, v_ref = T.to(dt), S.to(dt), v_ref.to(dt)
    assert T.shape == S.shape and tuple(v_ref.shape) == tuple(T.shape[1:])
    nt, nz = T.shape[0], T.shape[1]
    ncol = int(np.prod(T.shape[2:], dtype=np.int64))
    p = host(np.asarray(p_level, dtype=np.float64))
    masso = torch.empty(nt, dtype=torch.float64)
    _lib.check(L.ml_steric_global_host(_eos_id(eos), _dt_id(T), T.data_ptr(), S.data_ptr(), v_ref.data_ptr(),
                                       p.data_ptr(), nt, nz, ncol, int(steps_per_window), masso.data_ptr()))
    return masso


VARIANT_BITS = {"steric": 1, "thermosteric": 2, "halosteric": 4}


class HostStream:
    """The host path for fields that arrive block by block (``ml_host_stream_begin / push / finish``).

    What a dask-backed Dataset is to the reference (derived.py:624-630 ``dask="allowed"``; example.ipynb cell 4 opens
    the model output with ``chunks={"time": 1, ...}``): the 4-D fields never exist as one array.  ``push`` takes one
    block of consecutive time steps ``[nt_block, nz, ...]`` of T and S (numpy or CPU tensors; pinned memory keeps
    the copies asynchronous) and returns the block's outputs -- CPU tensors ``[nt_block, ...]`` per variant for
    ``domain="local"``, ``[nt_block]`` masses for ``domain="global"`` -- which are complete once :meth:`finish`
    has returned.  With ``reference=None`` the reference state is step 0 of the first block; otherwise
    ``reference = {"thetao", "so", "rho"}`` (host arrays) is a supplied reference (steric.py:98-103).
    ``dtype`` is how the blocks are stored on their way to the device.  An fp32 stream runs in fp64 when a supplied
    ``thetao`` or ``so`` slab is fp64 and one of its values does not survive a round trip through fp32, so that the
    slab is never rounded; an fp64 slab that is an upcast copy of fp32 data keeps the fp32 transfer.  ``self.dtype``
    is the dtype the stream runs in.  The stream holds at most the current and the previous block alive.
    """

    def __init__(self, domain, v_ref, p_level, z_i=None, deptho=None, variants=("steric",), reference=None,
                 rhozero=1035.0, eos="Wright", max_block_steps=1, dtype=torch.float32, want_rho_ref=False, want_sums=False):
        L = _lib.lib()
        _device()
        self.local = domain == "local"
        if domain not in ("local", "global"):
            raise ValueError(f"Unknown domain '{domain}'")
        self.variants = tuple(variants)
        mask = 0
        for v in self.variants:
            mask |= VARIANT_BITS[v]
        host = _host_tensor
        self._v = host(v_ref)
        if self._v.dtype not in (torch.float32, torch.float64):
            self._v = self._v.to(torch.float64)
        self.nz = int(self._v.shape[0])
        self.hshape = tuple(self._v.shape[1:])
        self.ncol = int(np.prod(self.hshape, dtype=np.int64))
        self._p = host(np.asarray(_host_np(p_level), dtype=np.float64))
        self._zi = host(np.asarray(_host_np(z_i), dtype=np.float64)) if z_i is not None else None
        self._depth = host(np.asarray(_host_np(deptho), dtype=np.float64)) if deptho is not None else None
        if self.local:
            assert self._zi is not None and self._depth is not None, "the local domain needs z_i and deptho"
            assert self._zi.numel() == self.nz + 1 and self._depth.numel() == self.ncol
        assert self._p.numel() == self.nz
        self._ref = None
        tref = sref = rref = None
        if reference is not None:
            self._ref = {k: host(reference[k]) for k in ("thetao", "so", "rho") if reference.get(k) is not None}
            if dtype == torch.float32 and not all(_fp32_exact(self._ref[k]) for k in ("thetao", "so") if k in self._ref):
                dtype = torch.float64
            if "thetao" in self._ref:
                self._ref["thetao"] = self._ref["thetao"].to(dtype)
                self._ref["so"] = self._ref["so"].to(dtype)
                tref, sref = self._ref["thetao"].data_ptr(), self._ref["so"].data_ptr()
            if "rho" in self._ref:
                self._ref["rho"] = self._ref["rho"].to(torch.float64)
                rref = self._ref["rho"].data_ptr()
        self.dtype = dtype
        self.want_rho_ref = bool(want_rho_ref)
        self.max_block_steps = int(max_block_steps)
        handle = ctypes.c_void_p()
        _lib.check(L.ml_host_stream_begin(
            _lib.DOMAIN_LOCAL if self.local else _lib.DOMAIN_GLOBAL, _eos_id(eos), _dt_id(torch.empty(0, dtype=dtype)), mask,
            self._v.data_ptr(), _dt_id(self._v), tref, sref, rref,
            self._zi.data_ptr() if self._zi is not None else None,
            self._depth.data_ptr() if self._depth is not None else None, self._p.data_ptr(), -1.0 / rhozero, self.nz,
            self.ncol, self.max_block_steps, (1 if want_rho_ref else 0) | (2 if want_sums else 0), ctypes.byref(handle)))
        self._h = handle
        self._blocks = []   # (T, S) of the current and the previous block
        self._outs = []     # every output tensor, in push order
        self.steps = 0

    def push(self, T_block, S_block):
        if self._h is None:
            raise RuntimeError("the stream is closed")
        T, S = _host_tensor(T_block).to(self.dtype), _host_tensor(S_block).to(self.dtype)
        assert T.shape == S.shape and tuple(T.shape[1:]) == (self.nz,) + self.hshape, \
            f"block of shape {tuple(T.shape)}, expecting [nt, {self.nz}, {self.hshape}]"
        nt = int(T.shape[0])
        shape = (nt,) + self.hshape if self.local else (nt,)
        out = {v: torch.empty(shape, dtype=torch.float64) for v in self.variants}
        ptr = lambda v: out[v].data_ptr() if v in out else None  # noqa: E731
        rc = _lib.lib().ml_host_stream_push(self._h, T.data_ptr(), S.data_ptr(), nt, ptr("steric"), ptr("thermosteric"),
                                            ptr("halosteric"))
        if rc != 0:
            msg = _lib.lib().ml_last_error().decode("utf-8", "replace")
            self.abort()
            raise _lib.MLError(rc, msg)
        self._blocks = (self._blocks + [(T, S)])[-2:]  # the previous block is released by the NEXT push
        self._outs.append(out)
        self.steps += nt
        return out

    def finish(self):
        """Wait for the tail; returns ``(rho_ref [nz, ...] or None, (volo, masso) or None)``."""
        if self._h is None:
            raise RuntimeError("the stream is closed")
        rho = torch.empty((self.nz,) + self.hshape, dtype=torch.float64) if self.want_rho_ref else None
        sums = torch.zeros(2, dtype=torch.float64)
        h, self._h = self._h, None
        _lib.check(_lib.lib().ml_host_stream_finish(h, rho.data_ptr() if rho is not None else None, sums.data_ptr()))
        self._blocks = []
        return rho, ((float(sums[0]), float(sums[1])) if self._ref is None else None)

    def abort(self):
        if self._h is not None:
            h, self._h = self._h, None
            _lib.lib().ml_host_stream_abort(h)
        self._blocks = []

    def __del__(self):
        try:
            self.abort()
        except Exception:  # noqa: BLE001 -- interpreter shutdown
            pass


def _host_np(x):
    return x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)


def _fp32_exact(t):
    """Whether every value of the host tensor ``t`` survives a round trip through fp32 (NaN stays NaN)."""
    if t.dtype == torch.float32:
        return True
    t = t.to(torch.float64)
    return bool(((t.to(torch.float32).to(torch.float64) == t) | torch.isnan(t)).all())


def host_release():
    """Free the device windows, pinned staging, streams and worker threads that the ``*_host`` calls of THIS thread
    keep between calls (``ml_host_release``).  Registered to run at interpreter exit for the importing thread; a
    program that calls the host path from short-lived worker threads should call it before each of them ends."""
    if _lib._LIB is not None:
        _lib._LIB.ml_host_release()


import atexit  # noqa: E402

atexit.register(host_release)
