"""``core.eos_eval`` point by point against ``oracle.eos``, on each of its three kernels.

``ml_eos_eval`` picks a kernel from the call's shape and alignment (``launch_eos`` in ``csrc/ml_api.cu``):

* the ring-staged stream kernel (``k_stream_map``): density of fp32 fields with a scalar or per-level
  pressure, 16-byte aligned operands, ``ncol % 4 == 0``;
* ``k_eos_eval_vec``, four columns per thread: any other aligned call with ``ncol % 4 == 0``, and every
  such call under ``force_direct(1)``;
* ``k_eos_eval``, one column per thread: ``ncol % 4 != 0`` or an operand that is not 16-byte aligned.

``test_kernel_paths`` checks with the profiler which kernel each geometry below reaches; the parity tests
then cover every function x equation of state x storage x pressure mode x broadcast on each of them.
Tolerances against the fp64 oracle on the upcast inputs: density 1e-10 relative; the derivatives 1e-11 of
the largest |oracle| of their (outer, level) row, because alpha changes sign near the temperature of
maximum density and a relative bound would be meaningless there.
"""

import numpy as np
import pytest
import torch

from oracle import eos as oeos

pytestmark = pytest.mark.gpu

FUNCS = ["density", "drho_dtemp", "drho_dsal", "alpha", "beta"]
NT, NZ, NY = 3, 7, 5


@pytest.fixture(scope="module")
def core():
    from momlevel_b200 import core

    assert torch.cuda.is_available(), "GPU tests need a CUDA device: there is no CPU path"
    return core


def _oracle(eos, func, T, S, p):
    f = getattr(oeos, f"{eos.lower()}_{func}")
    with np.errstate(invalid="ignore", divide="ignore"):
        out = f(T, S, p)
    return np.broadcast_to(np.asarray(out, np.float64), np.broadcast_shapes(T.shape, S.shape))


def _fields(shape, seed):
    """T across the temperature of maximum density (so alpha changes sign), S fresh to salty, a few NaNs."""
    rng = np.random.default_rng(seed)
    T = rng.uniform(-2.0, 30.0, shape)
    S = rng.uniform(0.0, 40.0, shape)
    T.flat[::97] = np.nan
    S.flat[5::89] = np.nan
    return T, S


def _device(a, dtype, offset):
    """``a`` on the device as ``dtype``; with ``offset`` a view that starts one element into its buffer, so
    it is aligned to its element but not to 16 bytes."""
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dtype)
    if not offset:
        return t.cuda()
    base = torch.empty(t.numel() + 1, dtype=dtype, device="cuda")
    view = base[1:].view(t.shape)
    view.copy_(t.cuda())
    assert view.data_ptr() % 16 != 0
    return view


def _rows_close(got, want, func, what):
    assert got.shape == want.shape, what
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what}: NaN pattern differs"
    m = np.isfinite(want)
    assert np.array_equal(m, np.isfinite(got)), what
    if func == "density":
        err = np.abs(got[m] - want[m]) / np.abs(want[m])
        assert err.max() <= 1e-10, f"{what}: relative error {err.max():.3e}"
        return
    g = got.reshape(-1, got.shape[-2] * got.shape[-1])
    w = want.reshape(-1, want.shape[-2] * want.shape[-1])
    f = m.reshape(w.shape)
    scale = np.where(f, np.abs(w), 0.0).max(axis=1, keepdims=True)
    err = np.where(f, np.abs(g - w), 0.0)
    assert np.all(err <= 1e-11 * scale), f"{what}: max error / row scale {(err / np.maximum(scale, 1e-300)).max():.3e}"


# geometry -> (ncol = NY * nx, offset view, force_direct)
GEOMS = {
    "aligned": (16, False, False),   # stream kernel (fp32 density, row pressure) or k_eos_eval_vec
    "forced": (16, False, True),     # k_eos_eval_vec for every call
    "ragged": (13, False, False),    # k_eos_eval: ncol % 4 != 0
    "offset": (16, True, False),     # k_eos_eval: bases off 16-byte alignment
}


def _call(core, eos, func, dtype, geom, pmode, bcast, seed):
    nx, offset, forced = GEOMS[geom]
    shape = (NT, NZ, NY, nx)
    T, S = _fields(shape, seed)
    z_l = np.linspace(2.5, 5500.0, NZ)
    if bcast == "t_bcast":
        T = T[0]
    elif bcast == "s_bcast":
        S = S[0]
    store = np.float32 if dtype == torch.float32 else np.float64
    T64, S64 = T.astype(store).astype(np.float64), S.astype(store).astype(np.float64)
    if pmode == "scalar":
        p, p_or = 2.0e7, 2.0e7
    elif pmode == "level":
        p = z_l * 1.0e4 + 101325.0
        p_or = p.reshape(NZ, 1, 1)
    else:
        p = np.random.default_rng(seed + 1).uniform(0.0, 6.0e7, shape)
        p_or = p
    Tg, Sg = _device(T, dtype, offset), _device(S, dtype, offset)
    pg = torch.from_numpy(p).cuda() if isinstance(p, np.ndarray) else p
    prev = core.force_direct(1 if forced else 0)
    try:
        got = core.eos_eval(eos, func, Tg, Sg, pg, z_axis=1, t_bcast=bcast == "t_bcast", s_bcast=bcast == "s_bcast")
    finally:
        core.force_direct(prev)
    Tb, Sb = np.broadcast_arrays(T64, S64)
    return got.cpu().numpy(), _oracle(eos, func, Tb, Sb, p_or)


@pytest.mark.parametrize("geom", list(GEOMS))
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("func", FUNCS)
@pytest.mark.parametrize("eos", ["Wright", "linear"])
def test_against_oracle(core, eos, func, dtype, geom):
    """Every pressure mode and broadcast of one function, storage and kernel."""
    for i, pmode in enumerate(("scalar", "level", "full")):
        for j, bcast in enumerate(("none", "t_bcast", "s_bcast")):
            got, want = _call(core, eos, func, dtype, geom, pmode, bcast, seed=10 * i + j)
            _rows_close(got, want, func, f"{eos} {func} {geom} p={pmode} {bcast}")


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if "k_eos_eval" in e.name or "k_stream" in e.name]


def test_kernel_paths(core):
    """Which kernel each geometry of the parity tests reaches."""
    def names(func, dtype, geom, pmode="level", bcast="none"):
        ks = _kernels(lambda: _call(core, "Wright", func, dtype, geom, pmode, bcast, seed=1))
        assert len(ks) == 1, ks
        return ks[0]

    assert "k_stream" in names("density", torch.float32, "aligned")
    assert "k_stream" in names("density", torch.float32, "aligned", "scalar", "t_bcast")
    for args in (("density", torch.float32, "forced"), ("density", torch.float64, "aligned"),
                 ("density", torch.float32, "aligned", "full"), ("alpha", torch.float32, "aligned"),
                 ("beta", torch.float64, "aligned", "scalar", "s_bcast")):
        assert "k_eos_eval_vec" in names(*args), args
    for args in (("density", torch.float32, "ragged"), ("density", torch.float32, "offset"),
                 ("drho_dtemp", torch.float64, "offset", "full"), ("alpha", torch.float64, "ragged")):
        n = names(*args)
        assert "k_eos_eval" in n and "k_eos_eval_vec" not in n, (args, n)


@pytest.mark.parametrize("ncol", [3, 4])
@pytest.mark.parametrize("func", ["density", "alpha", "drho_dsal"])
def test_more_rows_than_one_grid(core, func, ncol):
    """nouter * nz = 75000 rows of a few columns: the kernels walk rows beyond gridDim.y (<= 65535)."""
    shape = (300, 250, 1, ncol)
    T, S = _fields(shape, 7)
    z_l = np.linspace(1.0, 6000.0, 250)
    p = z_l * 1.0e4 + 101325.0
    got = core.eos_eval("Wright", func, torch.from_numpy(T).cuda(), torch.from_numpy(S).cuda(),
                        torch.from_numpy(p).cuda(), z_axis=1).cpu().numpy()
    _rows_close(got, _oracle("Wright", func, T, S, p.reshape(1, -1, 1, 1)), func, f"{func} ncol={ncol}")


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("eos", ["Wright", "linear"])
def test_scalar_and_vector_kernels_agree_bitwise(core, eos, dtype):
    """``k_eos_eval`` and ``k_eos_eval_vec`` evaluate the same inlined ``eos_func<EOS, FUNC>`` on the same
    inputs, so an aligned call and the same values in an offset view give the same bits."""
    for func in FUNCS:
        for pmode in ("scalar", "level", "full"):
            a, _ = _call(core, eos, func, dtype, "forced", pmode, "none", seed=3)
            b, _ = _call(core, eos, func, dtype, "offset", pmode, "none", seed=3)
            assert np.array_equal(a.view(np.int64), b.view(np.int64)), (func, pmode)
