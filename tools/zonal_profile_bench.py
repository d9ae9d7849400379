"""The height change by level of every grid row (a latitude-depth section) from one pass, against the whole-grid
profile and against the composition a user has without it.

    python tools/zonal_profile_bench.py [--out FILE] [--quick] [--reps N]

fp32, device-resident, three shapes: OM4p25 x 12, an OM4p125-shaped window of 8 daily steps (nx = 2880: two 2048-column
sub-tiles per row) and a 1-degree grid (360 x 320 x 75) x 12.  Alternated in the same run, CUDA events around each
call after warm-up; the entry points are called through the C ABI with their buffers allocated beforehand (the
workspace of the zonal call capped at core.REGION_WORKSPACE_BYTES, as core allocates it):
  1. ml_steric_local_zonal_profile, steric only;
  2. the same, the three variants from one pass;
  3. the same three variants as three single-variant calls;
  4. ml_steric_local_profile, steric only (the whole-grid profile, for scale);
  5. ml_delta_rho + ml_calc_dz + a torch weighted nansum over x per row (what a user composes today; OM4p25 only);
  6. core.steric_local_zonal_profile (with its per-row weight totals) and steric_profile(ds, zonal=True) against
     steric_profile(ds) (OM4p25 only; the public calls build the reference state each time).
The largest difference of 1 against 5 and whether 2 and 3 are bit-identical are recorded.  The card's name, power
limit and SM clocks are read in the same run.  --quick runs small shapes as a rehearsal: its times are not a
measurement.  One JSON document is written to --out (default profiles/r09_zonal_profile.json).
"""

import argparse
import json
import pathlib
import statistics
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

import momlevel_b200 as ml  # noqa: E402
from momlevel_b200 import _lib, core, synth  # noqa: E402

VARIANTS = ("steric", "thermosteric", "halosteric")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fns, reps):
    """Alternate the calls; CUDA events around each.  Returns {name: [ms]}."""
    out = {k: [] for k in fns}
    for f in fns.values():  # warm-up: module load, attributes, allocator
        f()
        f()
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, f in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            out[name].append(e0.elapsed_time(e1))
    return out


def one_shape(shape, reps, whole):
    nt, nz, ny, nx = shape
    L = _lib.lib()
    ds = synth.make_dataset(nt, nz, ny, nx, seed=123, device="cuda", dtype=torch.float32)
    T, S, V = ds["thetao"].data, ds["so"].data, ds["volcello"].data[0]
    z_i, depth = ds["z_i"].data.to(torch.float64), ds["deptho"].data.to(torch.float64)
    area = ds["areacello"].data.to(torch.float64).contiguous()
    pres = (ds["z_l"].data * 1.0e4 + 101325.0).to(torch.float64)
    rho, _ = core.reference_state(T[0], S[0], V, pres)
    Tr, Sr = T[0].contiguous(), S[0].contiguous()
    vdt = _lib.F32 if V.dtype == torch.float32 else _lib.F64
    cap = core.REGION_WORKSPACE_BYTES - 256

    def zbuf(nv):
        steps = max(1, min(nt, cap // (L.ml_zonal_profile_workspace_bytes(nv, 1, nz, ny, nx) - 256)))
        nbytes = L.ml_zonal_profile_workspace_bytes(nv, steps, nz, ny, nx)
        return torch.empty((nbytes + 7) // 8, dtype=torch.float64, device="cuda"), nbytes, steps

    ws_z1, ws_z3 = zbuf(1), zbuf(3)
    pbytes = L.ml_profile_workspace_bytes(1, nt, nz, ny * nx)
    ws_p = torch.empty((pbytes + 7) // 8, dtype=torch.float64, device="cuda")
    one = {v: torch.empty((nt, nz, ny), dtype=torch.float64, device="cuda") for v in VARIANTS}
    three = {v: torch.empty((nt, nz, ny), dtype=torch.float64, device="cuda") for v in VARIANTS}
    prof_out = torch.empty((nt, nz), dtype=torch.float64, device="cuda")

    def zonal(outs, names, ws):
        ptr = lambda v: outs[v].data_ptr() if v in names else None  # noqa: E731
        _lib.check(L.ml_steric_local_zonal_profile(
            0, _lib.F32, T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), rho.data_ptr(), V.data_ptr(), vdt,
            z_i.data_ptr(), depth.data_ptr(), area.data_ptr(), pres.data_ptr(), -1.0 / 1035.0, nt, nz, ny, nx,
            ptr("steric"), ptr("thermosteric"), ptr("halosteric"), ws[0].data_ptr(), ws[1], None))

    def profile():
        _lib.check(L.ml_steric_local_profile(
            0, _lib.F32, T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), rho.data_ptr(), V.data_ptr(), vdt,
            z_i.data_ptr(), depth.data_ptr(), area.data_ptr(), pres.data_ptr(), -1.0 / 1035.0, nt, nz, ny * nx,
            prof_out.data_ptr(), None, None, ws_p.data_ptr(), pbytes, None))

    def split():
        for v in VARIANTS:
            zonal(one, (v,), ws_z1)

    def composed():
        drho = core.delta_rho(T, S, rho, V, pres)
        dz = core.calc_dz(z_i, depth)
        wet = ~torch.isnan(V[0])
        w = torch.where(wet, torch.nan_to_num(area, nan=0.0), torch.zeros_like(area))
        return (-1.0 / 1035.0) * torch.nansum(w * dz[None] * drho, dim=3)  # numerators [nt, nz, ny]

    fns = {"zonal_steric": lambda: zonal(three, ("steric",), ws_z1),
           "zonal_three": lambda: zonal(three, VARIANTS, ws_z3),
           "zonal_three_as_three_calls": split,
           "profile_steric": profile}
    if whole:
        fns["composed"] = composed
        fns["core_zonal_steric"] = lambda: core.steric_local_zonal_profile(T, S, Tr, Sr, rho, V, z_i, depth, pres, area,
                                                                           variants="steric")
        fns["public_zonal"] = lambda: ml.steric_profile(ds, zonal=True)[0]["steric"].data
        fns["public_profile"] = lambda: ml.steric_profile(ds)[0]["steric"].data
    zonal(three, VARIANTS, ws_z3)
    path = core.last_path()
    split()
    torch.cuda.synchronize()
    busy = -(-nx // 4) if nx < 2048 else 256  # threads of a CTA that hold points of a sub-tile (the first one)
    rec = {"shape": list(shape), "path": {1: "plain loads", 2: "ring"}.get(path, path),
           "sub_tiles_per_row": -(-nx // 2048), "threads_with_points_of_256": min(busy, 256),
           "zonal_steps_per_chunk": {"steric": ws_z1[2], "three": ws_z3[2]},
           "reduce_rows_blocks": nt * nz * ny,
           "one_pass_bit_identical_to_three_calls": all(torch.equal(three[v], one[v]) for v in VARIANTS)}
    if whole:
        zonal(three, ("steric",), ws_z1)
        W = torch.stack([torch.nansum(area[j]) for j in range(ny)])  # rows with W = 0 are NaN in both
        rec["max_abs_diff_zonal_vs_composed_m"] = float((three["steric"] / W - composed() / W).abs().nan_to_num().max())
        torch.cuda.empty_cache()
    t = timed(fns, reps)
    for k, v in t.items():
        rec[f"{k}_ms"] = {"best": min(v), "median": statistics.median(v), "all": v}
    med = lambda k: rec[f"{k}_ms"]["median"]  # noqa: E731
    rec["zonal_steric_over_profile_steric_median"] = med("zonal_steric") / med("profile_steric")
    rec["three_calls_over_one_pass_median"] = med("zonal_three_as_three_calls") / med("zonal_three")
    if whole:
        rec["composed_over_zonal_steric_median"] = med("composed") / med("zonal_steric")
        rec["public_zonal_over_public_profile_median"] = med("public_zonal") / med("public_profile")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r09_zonal_profile.json"))
    ap.add_argument("--quick", action="store_true", help="small shapes, a rehearsal rather than a measurement")
    ap.add_argument("--reps", type=int, default=15)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    reps = 3 if args.quick else args.reps
    om4p125 = synth.CONFIGS["om4p125"]
    shapes = {"om4p25x12": (3, 75, 64, 96) if args.quick else synth.CONFIGS["om4p25"],
              "om4p125_window8": (2, 75, 48, 2880) if args.quick else (8,) + om4p125[1:],
              "one_degree_x12": (2, 75, 32, 360) if args.quick else (12, 75, 320, 360)}
    rec = {"gpu (name, power limit, max SM clock, SM clock) before": card(), "quick": bool(args.quick),
           "dtype": "float32", "device_resident": True, "reps": reps,
           "timing": "CUDA events around each call, calls alternated, two warm-up calls each"}
    for name, shape in shapes.items():
        rec[name] = one_shape(shape, reps, whole=name == "om4p25x12")
        torch.cuda.empty_cache()
    rec["gpu (name, power limit, max SM clock, SM clock) after"] = card()
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not (isinstance(vv, dict) and "all" in vv)}
                          if isinstance(v, dict) else v) for k, v in rec.items()}), flush=True)
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
