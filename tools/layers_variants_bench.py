"""The steric, thermosteric and halosteric heights by depth layer from one pass, against one layered launch per height.

    python tools/layers_variants_bench.py [--out FILE] [--quick] [--reps N]

Edges (0, 700, 2000, None), fp32.  Alternated in the same run, CUDA events around each call after warm-up, best and
median:
  OM4p25 x 12, device-resident (above L2 size):
    1. ml_steric_local_layers_variants, the one pass (and each instantiated chunk width of it, the candidates for
       the main width);
    2. three ml_steric_local_layers launches;
    3. ml_steric_local_variants, the full column, for context;
    4. steric_layers(ds, variant=VARIANTS) against three steric_layers(ds, variant=v) calls, on a device-resident
       Dataset and on an in-memory CPU Dataset (the public calls, reference-state pass and host-to-device copies
       included; events around a call that ends in a device synchronise).
  A window of 8 daily OM4p125-shaped steps, device-resident: 1 and 2 again.
The largest difference between the outputs of 1 and 2 is recorded (it must be 0: the one pass is bit-identical).
--quick runs small shapes as a rehearsal: its times are not a measurement.  One JSON document is written to --out
(default profiles/r05_layers_variants.json).
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
VARIANTS = ("steric", "thermosteric", "halosteric")
CHUNKS = (4, 6, 12)  # instantiated chunk widths of the one-pass layered kernel


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fns, reps, warmup=2):
    """Alternate the calls; CUDA events around each, each call ends in a device synchronise.  Returns {name: [ms]}."""
    out = {k: [] for k in fns}
    for f in fns.values():  # warm-up: module load, tensor maps, attributes, allocator
        for _ in range(warmup):
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


def stats(v):
    return {"best": min(v), "median": statistics.median(v), "all": v}


def max_diff(a, b):
    """(largest |a - b| where both are numbers, NaN masks equal, bit-identical)"""
    same_mask = bool(torch.equal(torch.isnan(a), torch.isnan(b)))
    m = ~torch.isnan(a) & ~torch.isnan(b)
    d = float((a[m] - b[m]).abs().max()) if bool(m.any()) else 0.0
    return d, same_mask, bool(torch.equal(a.view(torch.int64), b.view(torch.int64)))


def device_case(name, nt, nz, ny, nx, reps, chunks=False):
    ds = synth.make_dataset(nt, nz, ny, nx, seed=123, device="cuda", dtype=torch.float32)
    T, S, V = ds["thetao"].data, ds["so"].data, ds["volcello"].data[0]
    z_i, depth = ds["z_i"].data, ds["deptho"].data
    pres = ds["z_l"].data * 1.0e4 + 101325.0
    Tr, Sr = T[0].clone(), S[0].clone()
    rho, _ = core.reference_state(Tr, Sr, V, pres)

    def one_pass():
        return core.steric_local_layers_variants(T, S, Tr, Sr, rho, V, z_i, depth, pres, EDGES)

    def three():
        return {"steric": core.steric_local_layers(T, S, rho, V, z_i, depth, pres, EDGES),
                "thermosteric": core.steric_local_layers(T, Sr, rho, V, z_i, depth, pres, EDGES, s_bcast=True),
                "halosteric": core.steric_local_layers(Tr, S, rho, V, z_i, depth, pres, EDGES, t_bcast=True)}

    def full_column():
        return core.steric_local_variants(T, S, V, z_i, depth, pres, T_ref=Tr, S_ref=Sr, rho_ref=rho)[0]

    rec = {"shape": [nt, nz, ny, nx], "dtype": "float32", "device_resident": True, "reps": reps}
    a, b = one_pass(), three()
    rec["paths"] = {}
    n0 = core.launch_count()
    one_pass()
    torch.cuda.synchronize()
    rec["paths"]["one_pass"] = {"family": core.last_path(), "launches": core.launch_count() - n0}
    n0 = core.launch_count()
    three()
    torch.cuda.synchronize()
    rec["paths"]["three"] = {"family": core.last_path(), "launches": core.launch_count() - n0}
    rec["max_abs_diff_one_pass_vs_three_m"] = {}
    for v in VARIANTS:
        d, same_mask, same_bits = max_diff(a[v], b[v])
        rec["max_abs_diff_one_pass_vs_three_m"][v] = {"max_abs_diff": d, "nan_masks_equal": same_mask,
                                                      "bit_identical": same_bits}
    del a, b
    fns = {"one_pass": one_pass, "three_launches": three, "full_column_variants": full_column}
    if chunks:
        for tc in CHUNKS:
            def at(tc=tc):
                prev = core.variants_chunk(tc)
                try:
                    return one_pass()
                finally:
                    core.variants_chunk(prev)
            fns[f"one_pass_tc{tc}"] = at
    t = timed(fns, reps)
    for k, v in t.items():
        rec[f"{k}_ms"] = stats(v)
    rec["three_over_one_pass_median"] = rec["three_launches_ms"]["median"] / rec["one_pass_ms"]["median"]
    rec["one_pass_over_full_column_median"] = rec["one_pass_ms"]["median"] / rec["full_column_variants_ms"]["median"]
    pts, lvl, ncol, nl = nt * nz * ny * nx, nz * ny * nx, ny * nx, len(EDGES) - 1
    # algorithmic bytes: T and S (fp32) once; T_ref, S_ref, v_ref (fp32) and rho_ref (fp64) once; 3 layered heights
    rec["one_pass_bytes"] = 2 * pts * 4 + lvl * (3 * 4 + 8) + 3 * nl * nt * ncol * 8
    rec["one_pass_gb_per_s"] = rec["one_pass_bytes"] / rec["one_pass_ms"]["best"] / 1e6
    print(json.dumps({name: {k: v for k, v in rec.items() if not isinstance(v, dict) or "all" not in v}}), flush=True)
    return rec, ds


def public_case(ds, reps):
    def one_call():
        r = ml.steric_layers(ds, depth_edges=EDGES, variant=list(VARIANTS))[0]
        return [r[v].data for v in VARIANTS]

    def three_calls():
        return [ml.steric_layers(ds, depth_edges=EDGES, variant=v)[0][v].data for v in VARIANTS]

    a, b = one_call(), three_calls()
    bits = all(torch.equal(torch.as_tensor(x).view(torch.int64), torch.as_tensor(y).view(torch.int64))
               for x, y in zip(a, b))
    del a, b
    t = timed({"list": one_call, "three_calls": three_calls}, reps, warmup=1)
    rec = {"bit_identical": bits}
    for k, v in t.items():
        rec[f"{k}_ms"] = stats(v)
    rec["three_over_list_median"] = rec["three_calls_ms"]["median"] / rec["list_ms"]["median"]
    print(json.dumps({k: v for k, v in rec.items() if not isinstance(v, dict) or "all" not in v}), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r05_layers_variants.json"))
    ap.add_argument("--quick", action="store_true", help="small shapes, a rehearsal rather than a measurement")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    reps = 3 if args.quick else args.reps
    res = {"gpu": card(), "quick": bool(args.quick), "edges": [float(e) for e in core.layer_edges(EDGES)],
           "timing": "CUDA events around each call, calls alternated, warm-up calls first; best and median"}
    shape = (3, 75, 64, 96) if args.quick else synth.CONFIGS["om4p25"]
    res["om4p25"], ds = device_case("om4p25", *shape, reps, chunks=True)
    res["om4p25"]["public_device"] = public_case(ds, max(3, reps // 4))
    host = ds.copy()
    for k in ("thetao", "so", "volcello", "deptho", "areacello", "z_l", "z_i"):
        host[k] = ml.DataArray(ds[k].data.cpu().numpy(), ds[k].dims, attrs=ds[k].attrs)
    del ds
    torch.cuda.empty_cache()
    res["om4p25"]["public_host"] = public_case(host, 3)
    del host
    torch.cuda.empty_cache()
    shape = (8, 75, 128, 192) if args.quick else (8, 75, 2240, 2880)
    res["om4p125_daily_window"], ds = device_case("om4p125x8", *shape, max(3, reps // 2))
    del ds
    res["gpu_after"] = card()
    out = pathlib.Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
