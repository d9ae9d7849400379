"""The time mean of a baseline period (setup_reference_state(period=...)) against an HBM copy and against the torch
composition a user has without it.

    python tools/mean_reference_bench.py [--out FILE] [--quick] [--reps N] [--chunked-steps N]

1. Device-resident OM4p25 x 12, fp32 T, S and volcello (12 B per point and step): ml_mean_state_accumulate as one
   first-and-last call with its outputs allocated beforehand, against a device-to-device copy of the same 12 B per
   point (the measured HBM copy bandwidth counts the bytes read and written), against the torch composition (fp64
   nansum of w * x and of w over time per field, then core.reference_state) and the public
   setup_reference_state(ds, period=...).  Alternated, CUDA events around each call after warm-up.  The means of the
   kernel and of the composition are compared (the composition sums in another order: a rounding difference).
2. An OM4p125-shaped (2880 x 2240 x 75) chunked period of daily steps, one step per block, blocks produced from host
   memory (one pageable buffer per field, re-yielded: block production costs nothing): wall time of
   setup_reference_state(period=...) and of a plain copy of the same blocks to the device in the same run, GB/s over
   the field bytes, peak RSS of the process.
The card's name, power limit and SM clocks are read in the same run.  --quick runs small shapes as a rehearsal: its
times are not a measurement.  One JSON document is written to --out (default profiles/r10_mean_reference.json).
"""

import argparse
import json
import pathlib
import resource
import statistics
import subprocess
import sys
import time

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import momlevel_b200 as ml  # noqa: E402
from momlevel_b200 import _lib, core, synth  # noqa: E402
from momlevel_b200.labeled import ChunkedArray, DataArray  # noqa: E402

DIMS = ("time", "z_l", "yh", "xh")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def timed(fns, reps):
    out = {k: [] for k in fns}
    for f in fns.values():
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
    return {k: {"best_ms": min(v), "median_ms": statistics.median(v)} for k, v in out.items()}


def fields(nt, nz, ny, nx, seed=1):
    """fp32 T, S, V [nt, nz, ny, nx] on the device, land NaN in every step and 2 % intermittent holes."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    land = torch.rand((1, 1, ny, nx), generator=g, device="cuda") < 0.3
    out = []
    for base, scale in ((10.0, 5.0), (35.0, 1.0), (1.0e9, 1.0e8)):
        x = base + scale * torch.randn((nt, nz, ny, nx), generator=g, device="cuda")
        x.masked_fill_(land, float("nan"))
        x.masked_fill_(torch.rand((nt, nz, ny, nx), generator=g, device="cuda") < 0.02, float("nan"))
        out.append(x)
    return out


def device_case(nt, nz, ny, nx, reps):
    T, S, V = fields(nt, nz, ny, nx)
    npts = T.numel()
    w = torch.tensor(np.resize([31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], nt).astype(np.float64), device="cuda")
    outs = tuple(torch.empty((nz, ny, nx), dtype=torch.float64, device="cuda") for _ in range(3))
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream

    def kernel():
        _lib.check(L.ml_mean_state_accumulate(_lib.F32, T.data_ptr(), S.data_ptr(), V.data_ptr(), _lib.F32, w.data_ptr(),
                                              nt, nz, ny * nx, None, 0, 3, *(o.data_ptr() for o in outs), st))

    src = torch.empty(3 * npts, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)

    def copy():
        dst.copy_(src)

    grid = synth.make_grid(nz, ny, nx, device="cuda")
    p = grid["z_l"].to(torch.float64) * 1.0e4 + 101325.0

    def composition():
        means = []
        for x in (T, S, V):
            x64 = x.to(torch.float64)
            ok = ~torch.isnan(x64)
            wb = w.view(-1, 1, 1, 1)
            means.append(torch.nansum(x64 * wb, 0) / (ok * wb).sum(0))
        return core.reference_state(*means, p)

    ds = synth.dataset_from_fields(grid, T, S, V[0])
    ds["volcello"] = DataArray(V, DIMS)

    def public():
        ml.reference.setup_reference_state(ds, period=slice(0, nt), period_weights=w.cpu().numpy())

    t = timed({"ml_mean_state_accumulate": kernel, "hbm_copy": copy, "torch_composition": composition,
               "setup_reference_state_period": public}, reps)
    kernel()
    means = []
    for x in (T, S, V):
        x64 = x.to(torch.float64)
        ok = ~torch.isnan(x64)
        wb = w.view(-1, 1, 1, 1)
        means.append(torch.nansum(x64 * wb, 0) / (ok * wb).sum(0))
    rel = [torch.abs(a - b) / torch.abs(b) for a, b in zip(outs, means)]
    diff = max(float(r[~torch.isnan(r)].max()) for r in rel)
    k_ms = t["ml_mean_state_accumulate"]["median_ms"]
    copy_gbs = 2 * 12 * npts / (t["hbm_copy"]["median_ms"] * 1e6)  # bytes read + written
    kernel_gbs = 12 * npts / (k_ms * 1e6)
    return {"shape": [nt, nz, ny, nx], "points": npts, "times": t,
            "input_bytes": 12 * npts, "output_bytes": 24 * nz * ny * nx,
            "hbm_copy_GBps": copy_gbs, "kernel_input_GBps": kernel_gbs,
            "kernel_over_copy_bandwidth": kernel_gbs / copy_gbs,
            "floor_ms_at_copy_bandwidth": 12 * npts / (copy_gbs * 1e6),
            "target_ms_at_0.85": 12 * npts / (0.85 * copy_gbs * 1e6),
            "max_rel_diff_kernel_vs_composition": diff}


def chunked_case(nt, nz, ny, nx):
    rng = np.random.default_rng(0)
    one = [(base + scale * rng.standard_normal((1, nz, ny, nx))).astype(np.float32)
           for base, scale in ((10.0, 5.0), (35.0, 1.0), (1.0e9, 1.0e8))]

    def chunked(a):
        return ChunkedArray((nt, nz, ny, nx), np.float32, (1,) * nt, lambda: (a for _ in range(nt)))

    grid = synth.make_grid(nz, ny, nx, device="cpu")
    ds = synth.dataset_from_fields(grid, torch.from_numpy(one[0]), torch.from_numpy(one[1]), torch.from_numpy(one[2][0]))
    for k, a in zip(("thetao", "so", "volcello"), one):
        ds[k] = DataArray(chunked(a), DIMS)
    nbytes = 3 * 4 * nt * nz * ny * nx
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ml.reference.setup_reference_state(ds, period=slice(0, nt))
    torch.cuda.synchronize()
    t_mean = time.perf_counter() - t0
    rss_mean = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss
    dev = [torch.empty((1, nz, ny, nx), dtype=torch.float32, device="cuda") for _ in range(3)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    its = [ds[k]._data.blocks() for k in ("thetao", "so", "volcello")]
    for _ in range(nt):
        for d, it in zip(dev, its):
            d.copy_(torch.from_numpy(next(it)))
    torch.cuda.synchronize()
    t_copy = time.perf_counter() - t0
    return {"shape": [nt, nz, ny, nx], "field_bytes": nbytes, "period_mean_s": t_mean,
            "period_mean_GBps": nbytes / t_mean / 1e9, "plain_copy_s": t_copy, "plain_copy_GBps": nbytes / t_copy / 1e9,
            "peak_rss_MiB_after_period_mean": rss_mean / 1024.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r10_mean_reference.json"))
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--chunked-steps", type=int, default=30)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "the benchmark needs a CUDA device"
    res = {"card": card(), "quick": a.quick}
    if a.quick:
        res["device_om4p25x12"] = device_case(3, 5, 40, 64, 3)
        res["chunked_om4p125"] = chunked_case(3, 5, 40, 64)
    else:
        res["device_om4p25x12"] = device_case(12, 75, 1080, 1440, a.reps)
        res["chunked_om4p125"] = chunked_case(a.chunked_steps, 75, 2240, 2880)
    res["card_after"] = card()
    pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    pathlib.Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
