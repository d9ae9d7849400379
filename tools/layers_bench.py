"""The local height by depth layer from one pass, against the full-column height and against the composition a
user has without it.

    python tools/layers_bench.py [--out FILE] [--quick] [--reps N]

OM4p25 x 12 (fp32, device-resident, above L2 size), edges (0, 700, 2000, None).  Alternated in the same run, CUDA
events around each call after warm-up:
  1. ml_steric_local (the full column);
  2. ml_steric_local_layers;
  3. ml_delta_rho + ml_calc_dz(top, bottom) per layer + a torch reduction over z (what a user composes today);
  4. steric_layers(ds), the public call with reference=None (reference-state pass included).
The largest difference between the outputs of 2 and 3 is recorded.  --quick runs a small shape as a rehearsal:
its times are not a measurement.  One JSON document is written to --out (default profiles/r04_steric_layers.json).
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

EDGES = (0.0, 700.0, 2000.0, None)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fns, reps):
    """Alternate the calls; CUDA events around each.  Returns {name: [ms]}."""
    out = {k: [] for k in fns}
    for f in fns.values():  # warm-up: module load, tensor maps, attributes, allocator
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r04_steric_layers.json"))
    ap.add_argument("--quick", action="store_true", help="small shape, a rehearsal rather than a measurement")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    nt, nz, ny, nx = (3, 75, 64, 96) if args.quick else synth.CONFIGS["om4p25"]
    reps = 3 if args.quick else args.reps
    gpu = card()
    ds = synth.make_dataset(nt, nz, ny, nx, seed=123, device="cuda", dtype=torch.float32)
    T, S, V = ds["thetao"].data, ds["so"].data, ds["volcello"].data[0]
    z_i, depth = ds["z_i"].data, ds["deptho"].data
    pres = ds["z_l"].data * 1.0e4 + 101325.0
    rho, _ = core.reference_state(T[0], S[0], V, pres)
    edges = core.layer_edges(EDGES)
    ncol = ny * nx

    def full():
        return core.steric_local(T, S, rho, V, z_i, depth, pres)[0]

    def layers():
        return core.steric_local_layers(T, S, rho, V, z_i, depth, pres, EDGES)

    def composed():
        drho = core.delta_rho(T, S, rho, V, pres)
        out = torch.empty((nt, len(edges) - 1, ny, nx), dtype=torch.float64, device="cuda")
        for b in range(len(edges) - 1):
            bottom = None if edges[b + 1] == float("inf") else float(edges[b + 1])
            dz = core.calc_dz(z_i, depth, top=float(edges[b]), bottom=bottom).reshape(nz, ny, nx)
            out[:, b] = (-1.0 / 1035.0) * torch.nansum(dz[None] * drho, dim=1)
        return torch.where(torch.isnan(V[0])[None, None], torch.full_like(out, float("nan")), out)

    def public():
        return ml.steric_layers(ds, depth_edges=EDGES)[0]["steric"].data

    a, b = layers(), composed()
    wet = ~torch.isnan(b)
    same_mask = bool(torch.equal(torch.isnan(a), torch.isnan(b)))
    max_diff = float((a[wet] - b[wet]).abs().max()) if bool(wet.any()) else 0.0
    paths = {}
    full()
    paths["full"] = core.last_path()
    layers()
    paths["layers"] = core.last_path()
    t = timed({"full": full, "layers": layers, "composed": composed, "public": public}, reps)
    pts = nt * nz * ncol
    lvl = nz * ncol
    nl = len(edges) - 1
    # algorithmic bytes: T and S (fp32) once; rho_ref (fp64) and v_ref (fp32) once per call; the heights (fp64)
    bytes_full = 2 * pts * 4 + lvl * 12 + nt * ncol * 8
    bytes_layers = 2 * pts * 4 + lvl * 12 + nl * nt * ncol * 8
    # the composition: delta_rho written and read once per layer, plus the layer's dz field written and read
    bytes_composed = 2 * pts * 4 + lvl * 12 + pts * 8 + nl * (pts * 8 + 2 * lvl * 8) + nl * nt * ncol * 8
    rec = {"gpu": gpu, "quick": bool(args.quick), "shape": [nt, nz, ny, nx], "edges": [float(e) for e in edges],
           "dtype": "float32", "device_resident": True, "reps": reps, "paths": paths,
           "timing": "CUDA events around each call, calls alternated, two warm-up calls each",
           "max_abs_diff_layers_vs_composed_m": max_diff, "nan_masks_equal": same_mask,
           "algorithmic_bytes": {"full": bytes_full, "layers": bytes_layers, "composed": bytes_composed}}
    for k, v in t.items():
        rec[f"{k}_ms"] = {"best": min(v), "median": statistics.median(v), "all": v}
    rec["layers_over_full_median"] = rec["layers_ms"]["median"] / rec["full_ms"]["median"]
    rec["composed_over_layers_median"] = rec["composed_ms"]["median"] / rec["layers_ms"]["median"]
    rec["public_over_layers_median"] = rec["public_ms"]["median"] / rec["layers_ms"]["median"]
    rec["layers_gb_per_s"] = bytes_layers / rec["layers_ms"]["best"] / 1e6
    print(json.dumps({k: v for k, v in rec.items() if not isinstance(v, dict) or "all" not in v}), flush=True)
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
