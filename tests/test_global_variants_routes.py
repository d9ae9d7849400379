"""CPU checks of steric_variants(domain="global"): which library calls each kind of input makes, the validation, and
the result Dataset.  The device calls are replaced (no GPU here); the numbers are checked on the GPU in
tests/test_gpu_global_variants.py."""

import importlib

import numpy as np
import pytest
import torch

import momlevel_b200 as ml
from momlevel_b200 import core, synth
from momlevel_b200.labeled import ChunkedArray, DataArray

steric_mod = importlib.import_module("momlevel_b200.steric")
VARIANTS = ("steric", "thermosteric", "halosteric")
VOLO, MASSO = 2.0, 2070.0


class _Recorder:
    """Stands in for core.HostStream (ml_host_stream_*) and core.steric_global_variants: records what is asked."""

    def __init__(self):
        self.calls = []
        rec = self

        class FakeStream:
            def __init__(self, domain, v_ref, p_level, variants=("steric",), reference=None, eos="Wright",
                         max_block_steps=1, dtype=torch.float32, want_sums=False, **kw):
                self.variants = variants
                rec.calls.append(["begin", domain, tuple(np.shape(v_ref)), variants,
                                  None if reference is None else sorted(reference), eos, max_block_steps, want_sums])

            def push(self, T, S):
                rec.calls.append(["push", tuple(T.shape)])
                # M_v(t) = rhoga * volo * exp(-k) with k = 0, 1, 2 per variant: a known series comes out
                return {v: torch.full((T.shape[0],), MASSO * np.exp(-1e-6 * VARIANTS.index(v)), dtype=torch.float64)
                        for v in self.variants}

            def finish(self):
                rec.calls.append(["finish"])
                return None, None

            def abort(self):
                rec.calls.append(["abort"])

        def fake_global_variants(T, S, v_ref, p_level, T_ref=None, S_ref=None, eos="Wright", variants=VARIANTS):
            rec.calls.append(["one_pass", tuple(np.shape(T)), T_ref is None, eos])
            nt = int(np.shape(T)[0])
            masso = {v: torch.full((nt,), MASSO * np.exp(-1e-6 * VARIANTS.index(v)), dtype=torch.float64)
                     for v in variants}
            return masso, (torch.tensor([VOLO, MASSO], dtype=torch.float64) if T_ref is None else None)

        self.stream = FakeStream
        self.one_pass = fake_global_variants


@pytest.fixture
def rec(monkeypatch):
    r = _Recorder()
    monkeypatch.setattr(core, "HostStream", r.stream)
    monkeypatch.setattr(core, "steric_global_variants", r.one_pass)
    return r


def _small():
    return synth.make_dataset(5, 12, 20, 32, seed=5, device="cpu", dtype=torch.float32)


def _check_result(res, ds):
    assert set(res.variables) >= {"reference_height", *VARIANTS}
    assert res["reference_height"].dims == () and res["reference_height"].attrs == {
        "long_name": "Reference column height", "units": "m"}
    assert res["reference_height"].encoding["dtype"] == "float32"
    href = VOLO / float(ds["areacello"].values.sum())
    assert float(res["reference_height"]) == pytest.approx(href, rel=1e-15)
    for k, v in enumerate(VARIANTS):
        assert res[v].dims == ("time",) and res[v].shape == (ds["thetao"].shape[0],)
        assert res[v].attrs == {"long_name": f"{v.capitalize()} height adjustment", "units": "m"}
        assert res[v].encoding["dtype"] == "float32"
        # href * ln(rhoga / (M / volo)) with M = masso * exp(-1e-6 k)
        assert np.allclose(res[v].values, href * 1e-6 * k, rtol=1e-9, atol=1e-18)
    assert "time" in res.variables


def test_host_resident_fields_make_one_stream_for_the_three_masses(rec, monkeypatch):
    ds = _small()
    monkeypatch.setattr(steric_mod, "HOST_ROUTE_MIN_BYTES", 0)
    res, ref = ml.steric_variants(ds, domain="global")
    begins = [c for c in rec.calls if c[0] == "begin"]
    assert begins == [["begin", "global", (12, 20, 32), VARIANTS, None, "Wright", 5, False]]
    assert [c[0] for c in rec.calls if c[0] in ("push", "finish")] == ["push", "finish"]  # one window of 5 steps
    # the reference scalars: the one-pass self-reference of step 0 only (the same sums as the device route)
    assert [c for c in rec.calls if c[0] == "one_pass"] == [["one_pass", (1, 12, 20, 32), True, "Wright"]]
    _check_result(res, ds)
    assert set(ref.variables) >= {"thetao", "so", "volcello", "rho", "volo", "masso", "rhoga", "areacello"}
    assert ref["rho"].is_lazy
    assert float(ref["volo"]) == VOLO and float(ref["rhoga"]) == MASSO / VOLO


def test_host_resident_fields_with_a_supplied_reference(rec, monkeypatch):
    ds = _small()
    monkeypatch.setattr(steric_mod, "HOST_ROUTE_MIN_BYTES", 0)
    ref_in = ml.Dataset()
    for k in ("thetao", "so", "volcello"):
        ref_in[k] = DataArray(ds[k].values[0], ("z_l", "yh", "xh"))
    ref_in["rho"] = DataArray(np.full((12, 20, 32), 1035.0), ("z_l", "yh", "xh"))
    ref_in["volo"] = DataArray(np.float64(VOLO), ())
    ref_in["masso"] = DataArray(np.float64(MASSO), ())
    ref_in["rhoga"] = DataArray(np.float64(MASSO / VOLO), ())
    ref_in["areacello"] = ds["areacello"]
    res, ref = ml.steric_variants(ds, domain="global", reference=ref_in)
    assert rec.calls[0] == ["begin", "global", (12, 20, 32), VARIANTS, ["so", "thetao"], "Wright", 5, False]
    assert not [c for c in rec.calls if c[0] == "one_pass"]
    assert ref is ref_in
    _check_result(res, ds)


def test_chunked_fields_make_one_pass_over_the_blocks(rec):
    ds = _small()
    chunks = (2, 1, 2)
    cds = ds.copy()
    made = {}
    for name in ("thetao", "so", "volcello"):
        full = ds[name].values
        cuts = np.cumsum((0,) + chunks)

        def blocks(full=full, cuts=cuts):
            for a, b in zip(cuts[:-1], cuts[1:]):
                yield np.array(full[a:b])

        made[name] = ChunkedArray(full.shape, full.dtype, chunks, blocks)
        cds[name] = DataArray(made[name], ds[name].dims, attrs=ds[name].attrs)
    res, ref = ml.steric_variants(cds, domain="global")
    assert made["thetao"].blocks_read == len(chunks) and made["so"].blocks_read == len(chunks)
    assert [c for c in rec.calls if c[0] == "begin"] == [["begin", "global", (12, 20, 32), VARIANTS, None, "Wright", 2, False]]
    assert [c[1] for c in rec.calls if c[0] == "push"] == [(2, 12, 20, 32), (1, 12, 20, 32), (2, 12, 20, 32)]
    assert [c for c in rec.calls if c[0] == "one_pass"] == [["one_pass", (1, 12, 20, 32), True, "Wright"]]
    _check_result(res, ds)
    assert float(ref["volo"]) == VOLO


def test_validation_matches_steric_global(rec):
    ds = _small()
    # no z_i / deptho needed in the global domain
    res, _ = ml.steric_variants(ds.drop_vars(["deptho", "z_i"]), domain="global")
    _check_result(res, ds)
    for bad in (ds.drop_vars(["volcello"]), ds.drop_vars(["areacello"])):
        with pytest.raises(ValueError, match="Errors found in dataset.") as want:
            ml.steric(bad, domain="global")
        with pytest.raises(ValueError, match="Errors found in dataset.") as got:
            ml.steric_variants(bad, domain="global")
        assert str(got.value) == str(want.value)
    scaled = ds.copy()
    scaled["areacello"] = ds["areacello"] * 2.0
    with pytest.raises(ValueError, match="Errors found in dataset."):
        ml.steric_variants(scaled, domain="global")


def test_unknown_equation_of_state(rec):
    with pytest.raises(ValueError, match="Unknown equation of state"):
        ml.steric_variants(_small(), domain="global", equation_of_state="teos10")
    assert rec.calls == []
