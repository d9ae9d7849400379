"""The global steric, thermosteric and halosteric series from one pass against three single-height calls.

    python tools/global_variants_bench.py [--out FILE] [--quick]

Device-resident (OM4p25 x 12 and a window of OM4p125-shaped daily steps): ml_steric_global_variants against three
ml_steric_global launches, alternated in the same run, CUDA events, warm-up, best and median.  Host-resident (pinned
and pageable numpy) and chunked Datasets: steric_variants(ds, domain="global") against three
steric(ds, variant=v, domain="global") calls, wall time, host-to-device bytes and the largest difference between the
series.  Parity: the three masses of one whole step against the oracle.  One JSON document is written to --out.
"""

import argparse
import json
import pathlib
import statistics
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import momlevel_b200 as ml  # noqa: E402
from momlevel_b200 import core, synth  # noqa: E402
from momlevel_b200.labeled import ChunkedArray, DataArray  # noqa: E402

VARIANTS = ("steric", "thermosteric", "halosteric")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed_pair(fa, fb, reps):
    """Alternate a and b; CUDA events around each call.  Returns {name: [ms]}."""
    out = {"a": [], "b": []}
    for f in (fa, fb):  # warm-up: module load, tensor maps, attributes
        f()
        f()
    torch.cuda.synchronize()
    for _ in range(reps):
        for name, f in (("a", fa), ("b", fb)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            out[name].append(e0.elapsed_time(e1))
    return out


def device_case(label, nt, nz, ny, nx, reps):
    grid = synth.make_grid(nz, ny, nx, seed=123, device="cuda")
    T, S, V = synth.make_fields(grid, nt, seed=123, dtype=torch.float32)
    T, S, V = T.cuda(), S.cuda(), V.cuda()
    pres = grid["z_l"].cuda() * 1.0e4 + 101325.0
    Tr, Sr = T[0], S[0]

    def one_pass():
        return core.steric_global_variants(T, S, V, pres)

    def three():
        return (core.steric_global(T, S, V, pres), core.steric_global(T, Sr, V, pres, s_bcast=True),
                core.steric_global(Tr, S, V, pres, t_bcast=True))

    got, _ = one_pass()
    want = three()
    identical = all(torch.equal(got[v], w) for v, w in zip(VARIANTS, want))
    t = timed_pair(one_pass, three, reps)
    pts = nt * nz * ny * nx
    lvl = nz * ny * nx
    # algorithmic bytes: T and S once, plus per (tile, chunk) the reference slabs and the volume (fp32 each)
    chunks = -(-nt // 12)
    bytes_one = 2 * pts * 4 + chunks * 3 * lvl * 4
    bytes_three = 3 * 2 * pts * 4 - 2 * (pts - lvl) * 4 + 3 * chunks * lvl * 4  # the held operand is one slab
    rec = {"shape": [nt, nz, ny, nx], "points": pts, "bit_identical": identical,
           "one_pass_ms": {"best": min(t["a"]), "median": statistics.median(t["a"])},
           "three_launches_ms": {"best": min(t["b"]), "median": statistics.median(t["b"])},
           "one_pass_gpts_per_s": pts / min(t["a"]) / 1e6, "three_launches_gpts_per_s": pts / min(t["b"]) / 1e6,
           "one_pass_algorithmic_bytes": bytes_one, "three_launches_algorithmic_bytes": bytes_three,
           "one_pass_gb_per_s": bytes_one / min(t["a"]) / 1e6, "reps": reps}
    rec["speedup_best"] = min(t["b"]) / min(t["a"])
    print(label, json.dumps(rec), flush=True)
    del T, S, V
    torch.cuda.empty_cache()
    return rec


def _dataset(T, S, V, grid):
    nt = T.shape[0]
    ds = ml.Dataset()
    dims = ("time", "z_l", "yh", "xh")
    ds["thetao"] = DataArray(T, dims)
    ds["so"] = DataArray(S, dims)
    ds["volcello"] = DataArray(np.broadcast_to(V, (nt,) + V.shape), dims)
    ds["areacello"] = DataArray(grid["areacello"].numpy(), ("yh", "xh"))
    ds["z_l"] = DataArray(grid["z_l"].numpy(), ("z_l",))
    ds["z_i"] = DataArray(grid["z_i"].numpy(), ("z_i",))
    ds["deptho"] = DataArray(grid["deptho"].numpy(), ("yh", "xh"))
    ds["time"] = DataArray(np.arange(nt, dtype=np.float64), ("time",))
    return ds


def _chunked(ds, block):
    out = ds.copy()
    made = {}
    for name in ("thetao", "so", "volcello"):
        full = ds[name].data
        nt = full.shape[0]
        chunks = tuple(min(block, nt - a) for a in range(0, nt, block))

        def blocks(full=full, chunks=chunks):
            a = 0
            for n in chunks:
                yield full[a:a + n]
                a += n

        made[name] = ChunkedArray(full.shape, full.dtype, chunks, blocks)
        out[name] = DataArray(made[name], ds[name].dims)
    return out, made


def host_case(nt, nz, ny, nx, block):
    grid = synth.make_grid(nz, ny, nx, seed=7, device="cuda")
    T, S, V = (x.cpu() for x in synth.make_fields(grid, nt, seed=7, dtype=torch.float32))
    grid = {k: v.cpu() for k, v in grid.items()}
    torch.cuda.empty_cache()
    out = {"shape": [nt, nz, ny, nx], "field_bytes": 2 * T.numel() * 4}
    pinned = (T.pin_memory().numpy(), S.pin_memory().numpy())
    pageable = (T.numpy(), S.numpy())
    Vn = V.numpy()
    for kind, (Tn, Sn) in (("pinned", pinned), ("pageable", pageable), ("chunked", pageable)):
        ds = _dataset(Tn, Sn, Vn, grid)
        if kind == "chunked":
            ds, _ = _chunked(ds, block)

        def run_one():
            return ml.steric_variants(ds, domain="global")[0]

        def run_three():
            res = {}
            h2d = 0
            for v in VARIANTS:
                res[v] = ml.steric(ds, variant=v, domain="global")[0][v].values
                h2d += core.host_last_transfer()[0]
            return res, h2d

        run_one()  # warm-up: library, windows, pinned staging
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r1 = run_one()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        h2d_one = core.host_last_transfer()[0]
        r3, h2d_three = run_three()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        diff = max(float(np.max(np.abs(np.asarray(r1[v].values) - np.asarray(r3[v])))) for v in VARIANTS)
        out[kind] = {"steric_variants_s": t1 - t0, "three_steric_calls_s": t2 - t1, "steric_variants_h2d_bytes": h2d_one,
                     "three_steric_calls_h2d_bytes": h2d_three, "max_abs_series_diff_m": diff,
                     "speedup": (t2 - t1) / (t1 - t0)}
        print("host", kind, json.dumps(out[kind]), flush=True)
    return out


def parity(nz, ny, nx):
    """The three masses of one whole step (steric.py:135) against the oracle, float64 numpy."""
    from oracle import steric as osteric

    grid = synth.make_grid(nz, ny, nx, seed=5, device="cpu")
    T, S, V = synth.make_fields(grid, 2, seed=5, dtype=torch.float32)
    pres = grid["z_l"] * 1.0e4 + 101325.0
    got, sums = core.steric_global_variants(T.cuda(), S.cuda(), V.cuda(), pres.cuda())
    t, s, v = (x.numpy().astype(np.float64) for x in (T, S, V))
    area = grid["areacello"].numpy()
    oref = osteric.reference_state(t, s, np.broadcast_to(v, t.shape), area, grid["z_l"].numpy())
    rec = {"shape": [1, nz, ny, nx], "volo_rel_err": abs(float(sums[0]) / oref["volo"] - 1.0),
           "masso_rel_err": abs(float(sums[1]) / oref["masso"] - 1.0)}
    for name in VARIANTS:
        _, _, m = osteric.steric_global(t[1:], s[1:], grid["z_l"].numpy(), oref, variant=name)
        rec[f"{name}_mass_rel_err"] = abs(float(got[name][1]) / float(m[0]) - 1.0)
    print("parity", json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r03_global_variants.json"))
    ap.add_argument("--quick", action="store_true", help="small shapes: a rehearsal of the script, not a measurement")
    a = ap.parse_args()
    res = {"card": card(), "torch": torch.__version__}
    if a.quick:
        res["om4p25_x12"] = device_case("device", 12, 10, 64, 96, 3)
        res["host"] = host_case(6, 10, 64, 96, 2)
        res["parity"] = parity(6, 32, 64)
    else:
        res["om4p25_x12"] = device_case("OM4p25x12", 12, 75, 1080, 1440, 20)
        res["om4p125_daily_window"] = device_case("OM4p125x8", 8, 75, 2240, 2880, 10)
        res["host"] = host_case(12, 75, 1080, 1440, 3)
        res["parity"] = parity(75, 1080, 1440)
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({"card": res["card"]}))


if __name__ == "__main__":
    main()
