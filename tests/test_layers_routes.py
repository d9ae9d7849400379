"""steric_layers() / ml_steric_local_layers without a device: edge validation, the oracle's layered height, the
partial-cell rule of calc_dz at an inner edge, and the argument errors the library reports before any launch."""

import ctypes

import numpy as np
import pytest
import torch

import momlevel_b200 as ml
from momlevel_b200 import _lib, synth
from momlevel_b200.labeled import ChunkedArray, DataArray
import layers_oracle  # tests/layers_oracle.py
from oracle import steric as osteric


def _small(nt=3, nz=12, ny=20, nx=32):
    return synth.make_dataset(nt, nz, ny, nx, seed=5, device="cpu", dtype=torch.float32)


def _np(ds, k):
    return np.asarray(ds[k].values, dtype=np.float64)


# --------------------------------------------------------------------------------------------------- edge validation


@pytest.mark.parametrize("edges", [
    (0.0,),                          # no layer
    (),
    tuple(range(0, 1000, 100)),      # 9 layers, one more than ML_MAX_LAYERS
    (0.0, 700.0, 700.0, None),       # not strictly increasing
    (0.0, 2000.0, 700.0),
    (-1.0, 700.0),                   # negative
    (0.0, float("nan"), 2000.0),     # NaN
    (0.0, float("inf"), 2000.0),     # an infinity that is not last
    (0.0, None, 2000.0),             # None that is not last
    (None, 700.0),
    (0.0, "deep"),
    5.0,                             # not a sequence
])
def test_bad_depth_edges_raise_value_error_before_any_work(edges):
    with pytest.raises(ValueError):
        ml.steric_layers(_small(), depth_edges=edges)


def test_layer_edges_normalise_none_to_inf():
    e = ml.core.layer_edges((0, 700, 2000, None))
    assert e.dtype == np.float64 and list(e) == [0.0, 700.0, 2000.0, np.inf]
    assert list(ml.core.layer_edges([100.0, float("inf")])) == [100.0, np.inf]
    assert ml.core.layer_edges(np.arange(9.0)).size == _lib.MAX_LAYERS + 1


def test_chunked_fields_are_not_supported_yet():
    ds = _small()
    cds = ds.copy()
    for name in ("thetao", "so", "volcello"):
        full = ds[name].values

        def blocks(full=full):
            yield np.array(full[:2])
            yield np.array(full[2:])

        cds[name] = DataArray(ChunkedArray(full.shape, full.dtype, (2, full.shape[0] - 2), blocks), ds[name].dims,
                              attrs=ds[name].attrs)
    with pytest.raises(NotImplementedError):
        ml.steric_layers(cds)


# ------------------------------------------------------------------------------------------------------- the oracle


@pytest.mark.parametrize("variant", ["steric", "thermosteric", "halosteric"])
def test_oracle_single_layer_is_steric_local(variant):
    ds = _small()
    T, S, V = _np(ds, "thetao"), _np(ds, "so"), _np(ds, "volcello")
    ref = osteric.reference_state(T, S, V, _np(ds, "areacello"), _np(ds, "z_l"))
    want, _ = osteric.steric_local(T, S, _np(ds, "z_l"), _np(ds, "z_i"), _np(ds, "deptho"), ref, variant=variant)
    got = layers_oracle.steric_local_layers(T, S, _np(ds, "z_l"), _np(ds, "z_i"), _np(ds, "deptho"), ref, (0.0, None),
                                      variant=variant)
    assert got.shape == (T.shape[0], 1) + T.shape[2:]
    np.testing.assert_array_equal(got[:, 0], want)


def test_oracle_layers_partition_the_column_away_from_straddling_cells():
    ds = _small()
    z_i = _np(ds, "z_i")
    T, S, V = _np(ds, "thetao"), _np(ds, "so"), _np(ds, "volcello")
    ref = osteric.reference_state(T, S, V, _np(ds, "areacello"), _np(ds, "z_l"))
    edges = (0.0, float(z_i[3]), 0.5 * float(z_i[6] + z_i[7]), None)  # one edge on an interface, one inside a cell
    full, _ = osteric.steric_local(T, S, _np(ds, "z_l"), z_i, _np(ds, "deptho"), ref)
    lay = layers_oracle.steric_local_layers(T, S, _np(ds, "z_l"), z_i, _np(ds, "deptho"), ref, edges)
    depth = np.nan_to_num(_np(ds, "deptho"), nan=0.0)
    straddle = (depth > z_i[6]) & (depth < z_i[7])  # the floor lies inside the cell that holds the inner edge
    ok = ~np.isnan(full) & ~straddle[None]
    np.testing.assert_allclose(lay.sum(axis=1)[ok], full[ok], rtol=0, atol=1e-12)


def test_partial_cell_straddling_an_edge_counts_on_both_sides():
    # cell 650-750 m, sea floor at 720 m, edge at 700 m: calc_dz gives 50 m above the edge and 50 m below it,
    # against 70 m for the whole column (derived.py:316-318 assumes the cell reaches its bottom interface)
    z_i = np.array([0.0, 650.0, 750.0])
    z_l = 0.5 * (z_i[1:] + z_i[:-1])
    depth = np.full((1, 1), 720.0)
    above = osteric.calc_dz(z_l, z_i, depth, top=0.0, bottom=700.0)[:, 0, 0]
    below = osteric.calc_dz(z_l, z_i, depth, top=700.0, bottom=None)[:, 0, 0]
    whole = osteric.calc_dz(z_l, z_i, depth)[:, 0, 0]
    assert list(above) == [650.0, 50.0] and list(below) == [0.0, 50.0] and list(whole) == [650.0, 70.0]
    # ... and so the layered heights of a column with a density change in that cell add up to 100/70 of it
    T = np.array([[[[10.0]], [[4.0]]], [[[10.0]], [[5.0]]]])
    S = np.full_like(T, 35.0)
    V = np.ones((2, 2, 1, 1))
    ref = osteric.reference_state(T, S, V, np.ones((1, 1)), z_l)
    full, _ = osteric.steric_local(T, S, z_l, z_i, depth, ref)
    lay = layers_oracle.steric_local_layers(T, S, z_l, z_i, depth, ref, (0.0, 700.0, None))
    assert full[1, 0, 0] != 0.0
    np.testing.assert_allclose(lay[1, :, 0, 0], [full[1, 0, 0] * 50 / 70, full[1, 0, 0] * 50 / 70], rtol=1e-14)


# --------------------------------------------------------------------------------------- ABI errors before a launch


def _call(edges, nlayers, T=16, rho_ref=16, eta=16):
    L = _lib.lib()
    e = None if edges is None else np.ascontiguousarray(edges, dtype=np.float64)
    ptr = None if e is None else e.ctypes.data_as(ctypes.c_void_p)
    rc = L.ml_steric_local_layers(0, _lib.F32, T, 16, 0, 0, rho_ref, 16, _lib.F32, 16, 16, 16, -1.0 / 1035.0, ptr,
                                  nlayers, 2, 3, 300, eta, None)
    return rc, L.ml_last_error().decode()


@pytest.mark.parametrize("edges, nlayers", [
    ([0.0, 700.0], 0),
    ([float(i) for i in range(10)], 9),
    ([0.0, 700.0, 700.0], 2),
    ([0.0, 2000.0, 700.0], 2),
    ([-5.0, 700.0], 1),
    ([0.0, float("nan")], 1),
    ([0.0, float("inf"), 2000.0], 2),
    ([float("-inf"), 0.0], 1),
])
def test_abi_rejects_bad_layers_with_a_shape_error(edges, nlayers):
    rc, msg = _call(edges, nlayers)
    assert rc == -2, msg  # ML_ERR_SHAPE
    assert "layer" in msg


def test_abi_rejects_null_pointers():
    assert _call(None, 1)[0] == -1
    assert _call([0.0, float("inf")], 1, T=None)[0] == -1
    assert _call([0.0, float("inf")], 1, rho_ref=None)[0] == -1
    assert _call([0.0, float("inf")], 1, eta=None)[0] == -1
    L = _lib.lib()
    e = np.array([0.0, np.inf])
    assert L.ml_steric_local_layers(9, 0, 16, 16, 0, 0, 16, 16, 0, 16, 16, 16, -1.0, e.ctypes.data_as(ctypes.c_void_p), 1,
                                    1, 1, 1, 16, None) == -4  # unknown equation of state
