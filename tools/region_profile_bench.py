"""The height change by level of 11 regions from one pass, against one region and against the 11 masked-weight calls
a user makes without it.

    python tools/region_profile_bench.py [--out FILE] [--quick] [--reps N]

fp32, device-resident, two shapes: OM4p25 x 12 and an OM4p125-shaped window of 8 daily steps (both above L2 size).
Alternated in the same run, CUDA events around each call after warm-up, each entry point called through the C ABI
with its buffers allocated beforehand (the workspace of the region calls capped at core.REGION_WORKSPACE_BYTES, as
core allocates it):
  1. ml_steric_local_region_profile, 11 coherent regions (4 longitude sectors x 3 latitude bands, the last two
     merged), steric only;
  2. the same, the three variants from one pass;
  3. ml_steric_local_profile, steric only, one region (for scale);
  4. 11 ml_steric_local_profile calls with weights where(region == r, w, 0) (what a user does without regions);
  5. ml_steric_local_region_profile with a per-column random map of 11 codes, steric only (the worst case: every
     warp touches every region);
  6. steric_profile(ds, regions=...) against 11 steric_profile(ds, weights=...) calls (OM4p25 only; the public
     calls build the reference state each time).
Whether 1 and 4 are bit-identical is recorded.  --quick runs small shapes as a rehearsal: its times are not a
measurement.  One JSON document is written to --out (default profiles/r08_region_profile.json).
"""

import argparse
import json
import pathlib
import statistics
import subprocess
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import momlevel_b200 as ml  # noqa: E402
from momlevel_b200 import _lib, core, synth  # noqa: E402

VARIANTS = ("steric", "thermosteric", "halosteric")
NREG = 11


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


def coherent(ny, nx):
    y = torch.arange(ny)[:, None].expand(ny, nx)
    x = torch.arange(nx)[None, :].expand(ny, nx)
    return torch.clamp((x * 4 // nx) * 3 + y * 3 // ny, max=NREG - 1)


def one_shape(shape, reps, whole):
    nt, nz, ny, nx = shape
    ncol = ny * nx
    L = _lib.lib()
    ds = synth.make_dataset(nt, nz, ny, nx, seed=123, device="cuda", dtype=torch.float32)
    T, S, V = ds["thetao"].data, ds["so"].data, ds["volcello"].data[0]
    z_i, depth = ds["z_i"].data.to(torch.float64), ds["deptho"].data.to(torch.float64)
    area = ds["areacello"].data.to(torch.float64).reshape(-1).contiguous()
    pres = (ds["z_l"].data * 1.0e4 + 101325.0).to(torch.float64)
    rho, _ = core.reference_state(T[0], S[0], V, pres)
    Tr, Sr = T[0].contiguous(), S[0].contiguous()
    maps = {"coherent": coherent(ny, nx), "random": torch.randint(0, NREG, (ny, nx), generator=torch.Generator().manual_seed(5))}
    idx = {k: v.reshape(-1).to(torch.int8).cuda() for k, v in maps.items()}
    masked = [torch.where(idx["coherent"] == r, area, 0.0) for r in range(NREG)]
    vdt = _lib.F32 if V.dtype == torch.float32 else _lib.F64

    def buffers(nv, nreg, steps):
        nbytes = L.ml_region_profile_workspace_bytes(nv, nreg, steps, nz, ncol)
        return torch.empty((nbytes + 7) // 8, dtype=torch.float64, device="cuda"), nbytes

    step3 = L.ml_region_profile_workspace_bytes(3, NREG, 1, nz, ncol) - 256
    step1 = L.ml_region_profile_workspace_bytes(1, NREG, 1, nz, ncol) - 256
    cap = core.REGION_WORKSPACE_BYTES - 256
    ws_r1 = buffers(1, NREG, max(1, min(nt, cap // step1)))
    ws_r3 = buffers(3, NREG, max(1, min(nt, cap // step3)))
    ws_p1 = buffers(1, 1, nt)
    outs = {v: torch.empty((NREG, nt, nz), dtype=torch.float64, device="cuda") for v in VARIANTS}
    masked_out = torch.empty((NREG, nt, nz), dtype=torch.float64, device="cuda")

    def region(names, which, ws):
        ptr = lambda v: outs[v].data_ptr() if v in names else None  # noqa: E731
        _lib.check(L.ml_steric_local_region_profile(
            0, _lib.F32, T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), rho.data_ptr(), V.data_ptr(), vdt,
            z_i.data_ptr(), depth.data_ptr(), area.data_ptr(), idx[which].data_ptr(), NREG, pres.data_ptr(),
            -1.0 / 1035.0, nt, nz, ncol, ptr("steric"), ptr("thermosteric"), ptr("halosteric"), ws[0].data_ptr(), ws[1],
            None))

    def plain(w, out):
        _lib.check(L.ml_steric_local_profile(
            0, _lib.F32, T.data_ptr(), S.data_ptr(), Tr.data_ptr(), Sr.data_ptr(), rho.data_ptr(), V.data_ptr(), vdt,
            z_i.data_ptr(), depth.data_ptr(), w.data_ptr(), pres.data_ptr(), -1.0 / 1035.0, nt, nz, ncol, out.data_ptr(),
            None, None, ws_p1[0].data_ptr(), ws_p1[1], None))

    def masked_calls():
        for r in range(NREG):
            plain(masked[r], masked_out[r])

    fns = {"region_steric": lambda: region(("steric",), "coherent", ws_r1),
           "region_three": lambda: region(VARIANTS, "coherent", ws_r3),
           "one_region_steric": lambda: plain(area, masked_out[0]),
           "masked_11_steric": masked_calls,
           "region_random_steric": lambda: region(("steric",), "random", ws_r1)}
    regions_np = maps["coherent"].numpy()
    area_np = np.asarray(ds["areacello"].values, dtype=np.float64)
    if whole:
        fns["public_regions"] = lambda: ml.steric_profile(ds, regions=regions_np)[0]["steric"].data
        fns["public_11_masked"] = lambda: [ml.steric_profile(ds, weights=np.where(regions_np == r, area_np, 0.0))
                                           for r in range(NREG)]
    region(("steric",), "coherent", ws_r1)
    path = core.last_path()
    masked_calls()
    torch.cuda.synchronize()
    rec = {"shape": list(shape), "regions": NREG, "path": {1: "plain loads", 2: "ring"}.get(path, path),
           "region_steps_per_chunk": {"steric": max(1, min(nt, cap // step1)), "three": max(1, min(nt, cap // step3))},
           "region_numerators_bit_identical_to_masked_calls": bool(torch.equal(outs["steric"], masked_out))}
    t = timed(fns, reps)
    for k, v in t.items():
        rec[f"{k}_ms"] = {"best": min(v), "median": statistics.median(v), "all": v}
    med = lambda k: rec[f"{k}_ms"]["median"]  # noqa: E731
    rec["region_steric_over_one_region_median"] = med("region_steric") / med("one_region_steric")
    rec["masked_11_over_region_steric_median"] = med("masked_11_steric") / med("region_steric")
    rec["region_three_over_region_steric_median"] = med("region_three") / med("region_steric")
    rec["region_random_over_region_steric_median"] = med("region_random_steric") / med("region_steric")
    if whole:
        rec["public_11_over_public_regions_median"] = med("public_11_masked") / med("public_regions")
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r08_region_profile.json"))
    ap.add_argument("--quick", action="store_true", help="small shapes, a rehearsal rather than a measurement")
    ap.add_argument("--reps", type=int, default=15)
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
