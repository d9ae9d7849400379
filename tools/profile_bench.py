"""The area-weighted height change by model level from one pass, against the full-column height and against the
composition a user has without it.

    python tools/profile_bench.py [--out FILE] [--quick] [--reps N]

fp32, device-resident, two shapes: OM4p25 x 12 and an OM4p125-shaped window of 8 daily steps (both above L2 size).
Alternated in the same run, CUDA events around each call after warm-up:
  1. ml_steric_local_profile, steric only;
  2. ml_steric_local_profile, the three variants from one pass;
  3. the same three from one launch each (ml_set_force_direct(2));
  4. ml_steric_local (the full-column height, for scale);
  5. ml_delta_rho + ml_calc_dz + a torch weighted nansum over (y, x) (what a user composes today; OM4p25 only);
  6. steric_profile(ds), the public call with reference=None (OM4p25 only).
The largest difference between the outputs of 1 and 5 is recorded, and whether 2 and 3 are bit-identical.  --quick
runs small shapes as a rehearsal: its times are not a measurement.  One JSON document is written to --out (default
profiles/r07_steric_profile.json).
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
from momlevel_b200 import core, synth  # noqa: E402

VARIANTS = ("steric", "thermosteric", "halosteric")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
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
    ds = synth.make_dataset(nt, nz, ny, nx, seed=123, device="cuda", dtype=torch.float32)
    T, S, V = ds["thetao"].data, ds["so"].data, ds["volcello"].data[0]
    z_i, depth, area = ds["z_i"].data, ds["deptho"].data, ds["areacello"].data.to(torch.float64)
    pres = ds["z_l"].data * 1.0e4 + 101325.0
    rho, _ = core.reference_state(T[0], S[0], V, pres)
    Tr, Sr = T[0], S[0]

    def prof1():
        return core.steric_local_profile(T, S, Tr, Sr, rho, V, z_i, depth, pres, area, variants="steric")

    def prof3():
        return core.steric_local_profile(T, S, Tr, Sr, rho, V, z_i, depth, pres, area)

    def prof3_split():
        prev = core.force_direct(2)
        try:
            return core.steric_local_profile(T, S, Tr, Sr, rho, V, z_i, depth, pres, area)
        finally:
            core.force_direct(prev)

    def full():
        return core.steric_local(T, S, rho, V, z_i, depth, pres)[0]

    def composed():
        drho = core.delta_rho(T, S, rho, V, pres)
        dz = core.calc_dz(z_i, depth)
        wet = ~torch.isnan(V[0])
        w = torch.where(wet, torch.nan_to_num(area, nan=0.0), torch.zeros_like(area))
        return (-1.0 / 1035.0) * torch.nansum(w * dz[None] * drho, dim=(2, 3)) / torch.nansum(area)

    fns = {"profile_steric": prof1, "profile_three": prof3, "profile_three_split": prof3_split, "full_column": full}
    if whole:  # the composition's fp64 temporaries of the larger shape would not fit beside its fields
        fns["composed"] = composed
        fns["public"] = lambda: ml.steric_profile(ds)[0]["steric"].data
    p3, p3s = prof3(), prof3_split()
    prof1()
    path = core.last_path()
    t = timed(fns, reps)
    ncol = ny * nx
    pts, lvl = nt * nz * ncol, nz * ncol
    # algorithmic bytes: T and S (fp32) once; per (level, column) rho_ref (fp64) and v_ref (fp32); per column
    # deptho, the weight and the surface mask
    col = ncol * (8 + 8 + 4)
    bytes_prof1 = 2 * pts * 4 + lvl * 12 + col
    bytes_prof3 = bytes_prof1 + lvl * 8  # T_ref and S_ref (fp32)
    # the composition: delta_rho written and read, dz written and read, plus its inputs
    bytes_comp = 2 * pts * 4 + lvl * 12 + 2 * pts * 8 + 2 * lvl * 8 + col
    rec = {"shape": list(shape), "path": {1: "plain loads", 2: "ring"}.get(path, path),
           "one_pass_bit_identical_to_split": all(bool(torch.equal(p3[v], p3s[v])) for v in VARIANTS),
           "algorithmic_bytes": {"profile_steric": bytes_prof1, "profile_three": bytes_prof3, "composed": bytes_comp}}
    if whole:
        a, b = prof1()["steric"], composed()
        rec["max_abs_diff_profile_vs_composed_m"] = float((a - b).abs().max())
        rec["max_abs_profile_m"] = float(b.abs().max())
    for k, v in t.items():
        rec[f"{k}_ms"] = {"best": min(v), "median": statistics.median(v), "all": v}
    med = lambda k: rec[f"{k}_ms"]["median"]  # noqa: E731
    if whole:
        rec["composed_over_profile_steric_median"] = med("composed") / med("profile_steric")
    rec["profile_steric_over_full_column_median"] = med("profile_steric") / med("full_column")
    rec["profile_three_over_split_median"] = med("profile_three") / med("profile_three_split")
    rec["profile_steric_gb_per_s_best"] = bytes_prof1 / rec["profile_steric_ms"]["best"] / 1e6
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r07_steric_profile.json"))
    ap.add_argument("--quick", action="store_true", help="small shapes, a rehearsal rather than a measurement")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    reps = 3 if args.quick else args.reps
    om4p125 = synth.CONFIGS["om4p125"]
    shapes = {"om4p25x12": (3, 75, 64, 96) if args.quick else synth.CONFIGS["om4p25"],
              "om4p125_window8": (2, 75, 48, 80) if args.quick else (8,) + om4p125[1:]}
    rec = {"gpu (name, power limit, max SM clock)": card(), "quick": bool(args.quick), "dtype": "float32",
           "device_resident": True, "reps": reps,
           "timing": "CUDA events around each call, calls alternated, two warm-up calls each"}
    for name, shape in shapes.items():
        rec[name] = one_shape(shape, reps, whole=name == "om4p25x12")
        torch.cuda.empty_cache()
    print(json.dumps({k: ({kk: vv for kk, vv in v.items() if not (isinstance(vv, dict) and "all" in vv)}
                          if isinstance(v, dict) else v) for k, v in rec.items()}), flush=True)
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
