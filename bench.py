"""bench.py -- steric grid-points/s on the OM4p25-shaped workload (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch: what ``momlevel.steric(dset)`` computes
for variant="steric", domain="local", Wright EOS on a 12-month 1440x1080x75 dataset --
the reference state (rho_ref + volo + masso from step 0) and the fused
EOS -> delta_rho -> clipped-dz -> column-integral in one pass, fp32 T/S resident in HBM, eta out.
Inputs (11.2 GB) are far larger than L2 (126 MB), so no flush is needed between steps.

Prints ONE JSON line (rank 0).  ``value`` = points of all ranks / max-over-ranks device time;
``e2e`` = the same metric through the host-buffer C-ABI entry (``ml_steric_local_host``:
pinned host -> device copies and the eta read-back inside the timed region; level rows cross
PCIe as they are or packed to the cells the reference reads, ``e2e.every_row_dense`` is the A/B,
``e2e.public_api_numpy_dataset`` the public ``steric(dset)`` call on pageable numpy fields);
``roofline`` is for the dominant kernel, timed with CUDA events on its stream;
``cpu_baseline`` = the numpy oracle (a port of the reference's path) on a bounded sample.
``--impl reference`` times only that CPU path, threaded over all host cores.
"""

import argparse
import json
import os
import pathlib
import statistics
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "steric grid-points/s (EOS+column integral)"
UNIT = "grid-points/s"
WORKLOADS = {
    # name -> (nt, nz, ny, nx)
    "om4p25": (12, 75, 1080, 1440),
    "spear1deg": (120, 75, 320, 360),
    "small": (12, 75, 120, 160),
}


def _positive(text):
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return n


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=_positive, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("ML_BENCH_WORKLOAD", "om4p25"), choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--force-direct", action="store_true", help="use the direct kernel family (A/B against TMA)")
    ap.add_argument("--configs", default=os.environ.get("ML_BENCH_CONFIGS", "3,4,5"),
                    help="BASELINE configs timed beside the headline (extras.configs); '' or --no-configs for none")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--no-selfcheck", action="store_true", help="skip the 200-step self-check (for ncu launch lists)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_BYTES = 48 << 20  # the dumped sample stays well under 64 MB for every workload
DUMP_SEED = 20261020


def dump_outputs(out_dir, eta, rho_ref, sums, v_ref):
    """Write the arrays one timed step returned, so that two builds can be compared output for output.

    ``sums.npy`` is {volo, masso}.  ``eta.npy`` ([nt][n]) holds ``n`` columns drawn with a fixed seed from those with
    a surface reference volume (elsewhere eta is NaN by definition) and sorted, so the sample depends only on the
    inputs.  When the call stored it, ``rho_ref.npy`` holds the reference density of the cells of these columns
    that have a reference volume, level by level.
    """
    import torch

    out_dir = pathlib.Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    nt, nz, ncol = eta.shape[0], v_ref.shape[0], eta[0].numel()
    wet = np.flatnonzero(~torch.isnan(v_ref.reshape(nz, ncol)[0]).cpu().numpy())
    n = min(wet.size, DUMP_BYTES // (8 * (nt + (nz if rho_ref is not None else 0))))
    cols = np.sort(np.random.default_rng(DUMP_SEED).choice(wet, size=n, replace=False))
    idx = torch.as_tensor(cols, device=eta.device)
    arrays = {"eta": eta.reshape(nt, ncol)[:, idx], "sums": sums}
    if rho_ref is not None:
        present = ~torch.isnan(v_ref.reshape(nz, ncol)[:, idx])
        arrays["rho_ref"] = rho_ref.reshape(nz, ncol)[:, idx][present]
    for name, x in arrays.items():
        np.save(out_dir / f"{name}.npy", x.double().cpu().numpy())
    return {"dir": str(out_dir), "files": sorted(f"{k}.npy" for k in arrays),
            "columns": f"{n} of the {wet.size} with a surface reference volume ({ncol} in all), seed {DUMP_SEED}"}


def config_of(args):
    nt, nz, ny, nx = WORKLOADS[args.workload]
    return {
        "workload": f"{args.workload}: {nx}x{ny}x{nz} z*, {nt} monthly steps, Wright EOS, variant=steric, domain=local"
                    " (reference state + fused column integral per step)",
        "grid": [nt, nz, ny, nx],
        "input_dtype": "f32",
        "l2_policy": "inputs (T+S per step batch) larger than L2; no flush",
        "sharding": "one independent 12-step batch (ensemble member) per GPU, no collective on the data path",
    }


# ------------------------------------------------------------------------------ clocks


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML, polled every ~5 ms).

    The timed region is tens of milliseconds, too short for `nvidia-smi -lms`; NVML is polled
    from a thread instead (the main thread sits in a CUDA synchronize, which releases the GIL).
    Falls back to one `nvidia-smi` query when NVML is not importable.
    """

    REASONS = {
        "hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4,
        "hw_power_brake_slowdown": 0x80,
    }

    def __init__(self, torch_device_index):
        self.samples, self.reasons, self.power = [], set(), []
        self.max_mhz = None
        self.stop = threading.Event()
        self.thread = None
        self.error = None
        try:
            import pynvml
            import torch

            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                pr = torch.cuda.get_device_properties(torch_device_index)
                busid = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
                self.handle = pynvml.nvmlDeviceGetHandleByPciBusId(busid.encode())
            except Exception:  # noqa: BLE001 -- older torch / masked devices: index order
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(torch_device_index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # noqa: BLE001 -- any NVML problem just disables the sampler
            self.nv = None
            self.error = f"{type(e).__name__}: {e}"

    def _poll(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                for name, bit in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0)
            except Exception as e:  # noqa: BLE001
                self.error = f"{type(e).__name__}: {e}"
                return
            time.sleep(0.004)

    def __enter__(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        if self.thread is not None:
            self.thread.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [f"unavailable: {self.error}"], "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_min_mhz": min(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "power_w_max": max(self.power), "samples": len(self.samples),
                "source": "NVML polled every ~5 ms from the first warm-up step to the end of the timed region"}


# ------------------------------------------------------------------------- CPU baseline


def reference_kernels():
    """Put the reference's own numpy EOS modules under the oracle's driver when an install of the reference is on
    the box (``pip install --no-deps --target baseline/_ref``, DESIGN.md section 1); returns ``(kind, files)``.

    The reference PACKAGE cannot be imported (xarray, xgcm, cftime are not installable here), so its driver
    (steric.py / reference.py / derived.py) stays the oracle's restatement either way.
    """
    from oracle import eos as oeos

    used = oeos.use_reference_modules(ROOT / "baseline" / "_ref")
    used = [str(pathlib.Path(u).relative_to(ROOT)) for u in used]
    return ("reference-numpy+port-driver" if used else "port"), used


def _oracle_slab(args_tuple):
    """One y-slab of the whole path on the host: reference state + local steric (numpy oracle)."""
    from oracle import steric as osteric

    T, S, V, area, depth, z_l, z_i = args_tuple
    T, S, V = (np.asarray(x, dtype=np.float64) for x in (T, S, V))  # the parity definition: fp64 upcast
    ref = osteric.reference_state(T, S, V[None], area, z_l)
    eta, _ = osteric.steric_local(T, S, z_l, z_i, depth, ref)
    return eta


def cpu_path(fields, rows_per_slab, nslabs, workers, row0=0):
    """Run the oracle over ``nslabs`` y-slabs on ``workers`` threads; returns (seconds, points, etas)."""
    from concurrent.futures import ThreadPoolExecutor

    T, S, V, area, depth, z_l, z_i = fields
    jobs = []
    for k in range(nslabs):
        ys = slice(row0 + k * rows_per_slab, row0 + (k + 1) * rows_per_slab)
        jobs.append((T[:, :, ys], S[:, :, ys], V[:, ys], area[ys], depth[ys], z_l, z_i))
    t0 = time.perf_counter()
    if workers == 1:
        etas = [_oracle_slab(j) for j in jobs]
    else:
        with ThreadPoolExecutor(max_workers=workers) as ex:
            etas = list(ex.map(_oracle_slab, jobs))
    dt = time.perf_counter() - t0
    points = sum(j[0].size for j in jobs)
    return dt, points, etas


def run_reference(args):
    """`--impl reference`: the reference's CPU path (numpy port) on all host cores, bounded sample."""
    import torch

    from momlevel_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kind, ref_files = reference_kernels()
    nt, nz, ny, nx = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    workers = min(cores, 64)
    rows = 4
    nslabs = min(max(workers, 1) * 2, ny // rows)
    # generate only the rows of the sample (the generator is seeded per step, not per row, so
    # the sample is a same-statistics slab rather than a bit-identical crop)
    grid = synth.make_grid(nz, rows * nslabs, nx, seed=123, device="cpu")
    T, S, V = synth.make_fields(grid, nt, seed=123, dtype=torch.float32)
    fields = (T.numpy(), S.numpy(), V.numpy(), grid["areacello"].numpy(), grid["deptho"].numpy(),
              grid["z_l"].numpy(), grid["z_i"].numpy())
    times = []
    points = 0
    for it in range(args.warmup + args.steps):
        dt, points, _ = cpu_path(fields, rows, nslabs, workers)
        if it >= args.warmup:
            times.append(dt)
    sec = sum(times) / len(times)
    value = points / sec
    sample = f"{nslabs} slabs of {rows}x{nx} columns x {nz} levels x {nt} steps = {points} points per step"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config_of(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": kind, "sample": sample,
                         "host_cpu_count": cores, "reference_files_used": ref_files},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "momlevel's steric path on the host: the reference's own eos/wright.py under the oracle's restatement of "
                "steric.py / reference.py / derived.py when baseline/_ref holds an install (kind says which), y-slabs on a "
                "thread pool; the package itself needs xarray, which is not installable here.  A RATE measured on a "
                "sample of the grid, not the whole grid",
    }
    print(json.dumps(line), flush=True)


def run_e2e(args, line, core, dist, dev, world, barrier, T, S, V, grid, z_i, depth, pres, eta, nt, ny, nx, points):
    """`e2e`: the same metric through ml_steric_local_host -- pinned host buffers in, host eta out."""
    import torch

    ok = 1
    try:
        Th = torch.empty(T.shape, dtype=T.dtype, pin_memory=True)
        Sh = torch.empty(S.shape, dtype=S.dtype, pin_memory=True)
        Vh = torch.empty(V.shape, dtype=V.dtype, pin_memory=True)
        eta_h = torch.empty((nt, ny, nx), dtype=torch.float64, pin_memory=True)
    except (RuntimeError, MemoryError):
        ok = 0
    flag = torch.tensor([ok], dtype=torch.int32, device=dev)
    if world > 1:  # all ranks take the same decision, or the timing collective below would hang
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if int(flag[0]) == 0:
        raise RuntimeError("could not pin the host buffers of the e2e leg on every rank")
    Th.copy_(T)
    Sh.copy_(S)
    Vh.copy_(V)
    z_h, d_h, p_h = z_i.cpu().numpy(), depth.cpu().numpy(), pres.cpu().numpy()
    n_e2e = max(1, min(args.steps, 5))

    # the ceiling the host-fed leg can be judged against: plain pinned cudaMemcpyAsync of 2 GB, all ranks at once
    n_probe = min(Th.numel(), 1 << 29)
    probe_dst = torch.empty(n_probe, dtype=Th.dtype, device=dev)
    probe_src = Th.view(-1)[:n_probe]
    probe_dst.copy_(probe_src, non_blocking=True)
    barrier()
    pa, pb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pa.record()
    for _ in range(3):
        probe_dst.copy_(probe_src, non_blocking=True)
    pb.record()
    torch.cuda.synchronize()
    probe = torch.tensor([pa.elapsed_time(pb) / 3], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(probe, op=dist.ReduceOp.MAX)
    h2d_peak_gbs = n_probe * Th.element_size() / (float(probe[0]) * 1e-3) / 1e9  # per rank, slowest rank
    del probe_dst

    # Level rows cross PCIe as they are or packed to the cells the reference reads.  The choice is the LIBRARY's
    # (ml_host_set_packing's default: rows taken from both ends until the packers and the copy engine meet, with
    # half the host's cores divided by the ranks that share them, LOCAL_WORLD_SIZE) -- what a caller of
    # momlevel_b200.steric(dset) gets; the A/B leg below sends every row as it is.
    pack_mode, pack_threads = 1, 0  # 0 = the library tunes the number of packing threads itself (PackTuner)
    core.host_packing(pack_mode, pack_threads)

    def e2e_step():
        return core.steric_local_host(Th, Sh, Vh, z_h, d_h, p_h, steps_per_window=1, eta_out=eta_h)

    e2e_step()  # (the library's first windows try its choices of packing threads; the timed calls run with the result)
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_step()
    torch.cuda.synchronize()
    lib_threads = core.host_last_pack_threads()
    dt = torch.tensor([(time.perf_counter() - t0) / n_e2e], dtype=torch.float64, device=dev)
    by_rank = None
    if world > 1:
        # what each rank saw (the figure of merit is the slowest): mean ms per call, packing threads of its last window,
        # share of rows it sent packed, host ms of its last call
        mine = torch.tensor([float(dt[0]) * 1e3, float(lib_threads), core.host_last_transfer()[1],
                             core.host_last_timings()["call_ms"]], dtype=torch.float64, device=dev)
        every = torch.empty(world * 4, dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(every, mine)
        by_rank = [[round(x, 2) for x in row] for row in every.view(world, 4).cpu().tolist()]
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    dense = Th.numel() * 4 + Sh.numel() * 4 + Vh.numel() * 4 + (z_h.size + d_h.size + p_h.size) * 8
    # what the library copied: level rows cross PCIe either as they are or as the cells the reference reads
    # (volcello present, steric.py:151-153), whichever side has time left -- the share differs from run to run
    h2d, packed_rows = core.host_last_transfer()
    host_ms = core.host_last_timings()
    d2h = eta_h.numel() * 8 + 16
    line["e2e"] = {"value": world * points / float(dt[0]), "unit": UNIT, "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h, "steps": n_e2e, "ms_per_step": float(dt[0]) * 1e3,
                   "api": "momlevel_b200.core.steric_local_host -> ml_steric_local_host (pinned host buffers)",
                   "host_input_bytes_per_step": dense, "level_rows_sent_packed": packed_rows,
                   "host_pack_mode": pack_mode, "host_pack_threads": lib_threads, "host_pack_policy": "library-tuned (ml_host_set_packing(1, 0)): threads of the last window", "host_pack_simd": core.host_pack_simd(),
                   "last_call_host_ms": host_ms}
    if by_rank is not None:
        line["e2e"]["by_rank_ms_threads_packed_lastcall"] = by_rank
    line["e2e"]["roofline"] = {
        "bound": "pcie_h2d", "h2d_bytes": h2d, "achieved_gbs": h2d / float(dt[0]) / 1e9,
        "peak_concurrent_h2d_gbs": h2d_peak_gbs, "frac": h2d / float(dt[0]) / 1e9 / h2d_peak_gbs,
        "dense_equivalent_gbs": dense / float(dt[0]) / 1e9,
        "dense_equivalent_frac": dense / float(dt[0]) / 1e9 / h2d_peak_gbs,
        "peak_source": f"plain pinned cudaMemcpyAsync of {n_probe * Th.element_size() >> 20} MiB on all {world} ranks at "
                       "once, slowest rank, measured in this run",
        "note": "frac counts the bytes that crossed PCIe per rank; dense_equivalent counts the caller's bytes (rows that "
                "travel packed to their present cells make it exceed the link rate)"}
    try:  # weak scaling of this leg against the committed one-GPU record (one batch per rank, one host for all ranks)
        base = json.loads((ROOT / "profiles" / "r02_bench_1gpu.json").read_text())["e2e"]["value"]
        line["e2e"]["efficiency_vs_n1"] = line["e2e"]["value"] / (world * float(base))
        line["e2e"]["n1_source"] = "profiles/r02_bench_1gpu.json (committed one-GPU run of this leg)"
    except (OSError, ValueError, KeyError, TypeError):
        pass
    # the device-resident and the host-streamed paths must agree
    err = (eta_h.to(dev) - eta).abs()
    line["e2e"]["max_abs_diff_vs_resident_m"] = float(torch.nan_to_num(err).max())
    # A/B: the other way of moving the rows (every row as it is when the timed setting packs, and the reverse)
    alt_mode = 0 if pack_mode else 1
    alt_key = "every_row_dense" if pack_mode else "rows_packed_where_cores_allow"
    core.host_packing(alt_mode, pack_threads)
    try:
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            e2e_step()
        torch.cuda.synchronize()
        dt0 = torch.tensor([(time.perf_counter() - t0) / n_e2e], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt0, op=dist.ReduceOp.MAX)
        line["e2e"][alt_key] = {"value": world * points / float(dt0[0]), "unit": UNIT,
                                "ms_per_step": float(dt0[0]) * 1e3,
                                "h2d_bytes_per_step": core.host_last_transfer()[0],
                                "level_rows_sent_packed": core.host_last_transfer()[1],
                                "max_abs_diff_vs_resident_m": float(torch.nan_to_num((eta_h.to(dev) - eta).abs()).max())}
    finally:
        core.host_packing(pack_mode, pack_threads)
    # BASELINE config 2 names all three variants: the same transfer feeding three integrations per window
    # (grid points counted once; three heights come back)
    try:
        outs = {"steric": eta_h, "thermosteric": torch.empty_like(eta_h, pin_memory=True),
                "halosteric": torch.empty_like(eta_h, pin_memory=True)}
        core.steric_local_host(Th, Sh, Vh, z_h, d_h, p_h, steps_per_window=1, variants=True, eta_out=outs)
        barrier()
        t0 = time.perf_counter()
        core.steric_local_host(Th, Sh, Vh, z_h, d_h, p_h, steps_per_window=1, variants=True, eta_out=outs)
        torch.cuda.synchronize()
        dt3 = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt3, op=dist.ReduceOp.MAX)
        line["e2e"]["all_three_variants"] = {"value": world * points / float(dt3[0]), "unit": UNIT,
                                             "ms_per_step": float(dt3[0]) * 1e3,
                                             "d2h_bytes_per_step": 3 * eta_h.numel() * 8 + 16,
                                             "api": "core.steric_local_host(variants=True) -> ml_steric_local_variants_host"}
    except (RuntimeError, MemoryError) as exc:  # the two extra pageable height fields are a few hundred MB
        line["e2e"]["all_three_variants"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
    # the call a user of the reference makes: steric(dset) on a Dataset backed by plain (pageable) numpy arrays,
    # validation, reference Dataset and result assembly included
    if world == 1 and not args.no_extras:
        try:
            import momlevel_b200 as ml
            from momlevel_b200 import synth

            cpu_grid = {k: v.cpu() for k, v in grid.items()}
            ds = synth.dataset_from_fields(cpu_grid, torch.from_numpy(Th.numpy().copy()),
                                           torch.from_numpy(Sh.numpy().copy()), torch.from_numpy(Vh.numpy().copy()))
            res, _ = ml.steric(ds)
            t0 = time.perf_counter()
            for _ in range(2):
                res, _ = ml.steric(ds)
                got = res["steric"].data
            dtp = (time.perf_counter() - t0) / 2
            nb, frac = core.host_last_transfer()
            line["e2e"]["public_api_numpy_dataset"] = {
                "value": points / dtp, "unit": UNIT, "ms_per_step": dtp * 1e3, "h2d_bytes_per_step": nb,
                "level_rows_sent_packed": frac, "api": "momlevel_b200.steric(dset), fields in pageable host memory",
                "max_abs_diff_vs_resident_m": float(torch.nan_to_num((got.to(dev) - eta).abs()).max())}
            del ds, res, got
        except Exception as exc:  # noqa: BLE001 -- an optional leg must not take the bench line down with it
            line["e2e"]["public_api_numpy_dataset"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
    return (Th.numpy(), Sh.numpy(), Vh.numpy(), grid["areacello"].cpu().numpy(), d_h, grid["z_l"].cpu().numpy(), z_h)


# ------------------------------------------------------------------------------ our arm


def run_ours(args):
    import torch
    import torch.distributed as dist

    import momlevel_b200 as ml
    from momlevel_b200 import core, synth

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    bound_cpus = 0
    if world > 1:
        from momlevel_b200 import distributed as mld

        bound_cpus = mld.bind_host_to_device(local_rank)  # pinned e2e buffers on the GPU's own NUMA node
        dist.init_process_group("nccl", device_id=dev)
    if args.force_direct:
        core.force_direct(True)
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_configs", str(ROOT / "tools" / "bench_configs.py"))
    bc = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bc)

    nt, nz, ny, nx = WORKLOADS[args.workload]
    ncol = ny * nx
    points = nt * nz * ncol
    grid = synth.make_grid(nz, ny, nx, seed=123, device=dev)
    T, S, V = synth.make_fields(grid, nt, seed=123 + rank, dtype=torch.float32)
    pres = (grid["z_l"] * 1.0e4 + 101325.0).contiguous()
    z_i, depth = grid["z_i"].contiguous(), grid["deptho"].contiguous()
    torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    k3_pairs = []

    def step(record=False):
        # what momlevel.steric(dset) launches: reference state (rho_ref, volo, masso) and the
        # column integral in one fused pass (ml_steric_local_selfref)
        if record:
            a, b = ev(), ev()
            a.record()
        # (the reference density itself is produced on first access of reference["rho"], like delta_rho;
        # volo / masso, which the result needs, come out of this pass)
        eta, rho_ref, sums = core.steric_local_selfref(T, S, V, z_i, depth, pres, want_rho_ref=False)
        if record:
            b.record()
            k3_pairs.append((a, b))
        return eta, rho_ref, sums

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are polled from the first warm-up step to the end of the timed region: the GPU runs the
    # same kernel back to back throughout, and the timed region alone (tens of ms) is too short
    # for more than a couple of NVML polls
    clk = ClockSampler(local_rank)
    clk.__enter__()
    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = core.launch_count()
    if True:
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(args.steps):
            eta, rho_ref, sums = step(record=True)
        e1.record()
        barrier()
    clk.__exit__(None, None, None)
    launches = core.launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    k3_ms = [a.elapsed_time(b) for a, b in k3_pairs]
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t[0]) / args.steps
    value = world * points / (ms_step * 1e-3)
    path = {1: "direct", 2: "tma"}.get(core.last_path(), "none")

    # roofline of the dominant kernel (k_steric_tma, self-reference mode): algorithmic bytes per
    # launch = T,S fp32 once + volcello(t=0) fp32 + deptho + eta (DESIGN.md; SURVEY 8d's 8.11 B per point
    # plus the reference volume)
    N = nz * ncol
    alg_bytes = nt * N * 8 + N * 4 + ncol * 8 * (nt + 1)
    k3_avg_ms = sum(k3_ms) / len(k3_ms)
    # share of the grid that carries water (upper interface above the sea floor and a reference volume)
    wet = (z_i[:-1].view(nz, 1, 1) < torch.nan_to_num(depth, nan=0.0).unsqueeze(0)) & ~torch.isnan(V)
    wet_fraction = float(wet.sum()) / float(N)
    del wet
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except (OSError, ValueError):
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = alg_bytes / (k3_avg_ms * 1e-3) / 1e9
    traffic = None  # dram__bytes_read + dram__bytes_write of one launch, from the committed ncu capture
    try:
        tr = json.loads((ROOT / "profiles" / "traffic.json").read_text()).get(args.workload)
        if tr and path == "tma":
            traffic = tr["dram_bytes_read"] + tr["dram_bytes_write"]
    except (OSError, ValueError, KeyError):
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "kernel": f"ml_steric_local_selfref ({path} family)", "kernel_ms": k3_avg_ms,
                "kernel_share_of_step": k3_avg_ms / (ms_total / args.steps),
                "algorithmic_bytes_per_launch": alg_bytes,
                # the other side of the ridge: 18 fp64 instructions per WET point (SASS count, DESIGN.md section 4;
                # cells with dz = 0 or no reference volume are skipped warp-wise once the tile is depth-sorted)
                # against the DFMA rate measured on this pool by tools/microbench.cu (18.1e12/s)
                "fp64": {"dfma_per_wet_point": 18, "wet_fraction": wet_fraction,
                         "achieved_tdfma_s": 18 * wet_fraction * points / (k3_avg_ms * 1e-3) / 1e12,
                         "peak_tdfma_s": 18.1, "frac": 18 * wet_fraction * points / (k3_avg_ms * 1e-3) / 18.1e12,
                         "peak_source": "profiles/r01_microbench_b200.txt (measured)"},
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": config_of(args), "roofline": roofline, "clocks": clk.summary(),
        "gpu_launches": launches * world, "kernel_family": path,
    }
    if world > 1:
        line["host_cpus_bound_per_rank"] = bound_cpus
    if rank == 0 and args.dump_outputs:
        line["dump_outputs"] = dump_outputs(args.dump_outputs, eta, rho_ref, sums, V)
    if rank == 0 and not args.no_cpu:
        # the headline's heights against the oracle on columns from every part of the grid (first / last / edge tiles
        # and a stride across the rest); the cpu_baseline leg below also compares the contiguous slab it times
        line["parity"] = bc.oracle_local_parity(T, S, V, None, grid, eta)
        line["parity"]["tolerance_m"] = 1e-9
    # the timed region above is tens of milliseconds; the same step 200 times under one event pair as a self-check
    if not args.no_selfcheck:
        clk2 = ClockSampler(local_rank)
        with clk2:
            e2, e3 = ev(), ev()
            e2.record()
            for _ in range(200):
                step()
            e3.record()
            torch.cuda.synchronize()
        line["selfcheck_200_steps"] = {
            "ms_per_step": e2.elapsed_time(e3) / 200, "value_this_rank": points / (e2.elapsed_time(e3) / 200 * 1e-3),
            "unit": UNIT, "clocks": clk2.summary(),
            "note": "0.4 s of back-to-back steps: long enough for the board's power management to act (sw_power_cap lowers "
                    "the SM clock), which the 20-step timed region above is not"}

    # ---- extras: the other variants / domains of the same dataset, a few steps each
    if not args.no_extras:
        def timed(fn, n=3):
            fn()
            torch.cuda.synchronize()
            a, b = ev(), ev()
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n

        extras = {}
        ms = timed(lambda: core.steric_local_selfref(T, S, V, z_i, depth, pres, want_rho_ref=True))
        extras["steric_local_selfref_with_rho_ref_stored_gpts"] = points / ms / 1e6
        rho_ref = core.steric_local_selfref(T, S, V, z_i, depth, pres, want_rho_ref=True)[1]
        ms = timed(lambda: core.steric_local(T, S, rho_ref, V, z_i, depth, pres))
        extras["steric_local_given_reference_gpts"] = points / ms / 1e6
        ms = timed(lambda: core.steric_local(T, S[0], rho_ref, V, z_i, depth, pres, s_bcast=True))
        extras["thermosteric_local_gpts"] = points / ms / 1e6
        ms = timed(lambda: core.steric_local(T[0], S, rho_ref, V, z_i, depth, pres, t_bcast=True))
        extras["halosteric_local_gpts"] = points / ms / 1e6
        ms = timed(lambda: core.steric_global(T, S, V, pres))
        extras["steric_global_gpts"] = points / ms / 1e6
        ms = timed(lambda: core.reference_state(T[0], S[0], V, pres))
        extras["reference_state_gpts"] = N / ms / 1e6
        ms = timed(lambda: core.steric_local(T, S, rho_ref, V, z_i, depth, pres, eos="linear"))
        extras["linear_local_gpts"] = points / ms / 1e6
        # BASELINE config 2 names all three variants: one call, one launch per height (grid points counted once)
        ms = timed(lambda: core.steric_local_variants(T, S, V, z_i, depth, pres))
        extras["all_three_variants_one_call_gpts"] = points / ms / 1e6
        half = nt // 2  # spice writes an fp64 field as large as both inputs; half the steps keeps HBM use bounded
        spice_out = torch.empty(T[:half].shape, dtype=torch.float64, device=dev)
        ms = timed(lambda: core.flament_spice(T[:half], S[:half], out=spice_out))
        extras["flament_spice_gpts"] = half * N / ms / 1e6
        del spice_out
        z_l = grid["z_l"].contiguous()  # the column diagnostics of SURVEY 8f: 8 B in + 8 B out per point, like spice
        ms = timed(lambda: core.calc_n2(T[:half], S[:half], z_l))
        extras["calc_n2_gpts"] = half * N / ms / 1e6
        ms = timed(lambda: core.calc_n2(T[:half], S[:half], z_l, adjust_negative=True))
        extras["calc_n2_adjusted_gpts"] = half * N / ms / 1e6
        # fields stored as fp64 (the reference's own test data; anything xarray arithmetic has touched): 16 B per point
        T64, S64, V64 = T[:half].double(), S[:half].double(), V.double()
        ms = timed(lambda: core.steric_local_selfref(T64, S64, V64, z_i, depth, pres, want_rho_ref=False))
        extras["steric_local_selfref_fp64_storage_gpts"] = half * N / ms / 1e6
        extras["steric_local_selfref_fp64_storage_hbm_frac"] = (half * N * 16 + N * 8 + ncol * 8 * (half + 1)) / (ms * 1e-3) / 1e9 / peak
        extras["steric_local_selfref_fp64_storage_family"] = {1: "direct", 2: "tma"}.get(core.last_path(), "none")
        del T64, S64, V64
        # a grid whose rows are not a multiple of 16 bytes (1441 x 1079 columns: odd): rank-1 tensor maps, one box per row
        rgrid = synth.make_grid(nz, ny - 1, nx + 1, seed=123, device=dev)
        rT, rS, rV = synth.make_fields(rgrid, nt, seed=123, dtype=torch.float32)
        rz, rd = rgrid["z_i"].contiguous(), rgrid["deptho"].contiguous()
        ms = timed(lambda: core.steric_local_selfref(rT, rS, rV, rz, rd, pres, want_rho_ref=False))
        extras["steric_local_selfref_ragged_rows_gpts"] = nt * nz * (ny - 1) * (nx + 1) / ms / 1e6
        extras["steric_local_selfref_ragged_rows_family"] = {1: "direct", 2: "tma"}.get(core.last_path(), "none")
        del rT, rS, rV, rgrid
        extras["steric_local_selfref_call_gpts"] = points / k3_avg_ms / 1e6
        # the public call with everything around the kernel: validation, variant select, result Datasets (wall clock,
        # synchronised on both sides; the first call checks the grid arrays and waits for that, the later ones queue
        # their work and return, and volo / masso of the last one are read back inside the timed region)
        dset = synth.dataset_from_fields(grid, T, S, V)
        ml.steric(dset)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            _, reference = ml.steric(dset)
        float(reference["rhoga"])
        torch.cuda.synchronize()
        extras["steric_public_api_wall_gpts"] = points / ((time.perf_counter() - t0) / 20) / 1e9
        t0 = time.perf_counter()
        _, reference = ml.steric(dset)
        float(reference["rhoga"])
        torch.cuda.synchronize()
        extras["steric_public_api_single_call_wall_gpts"] = points / (time.perf_counter() - t0) / 1e9
        del dset
        line["extras_Gpts_per_s"] = extras
        torch.cuda.empty_cache()

    # ---- e2e: host buffers through ml_steric_local_host, copies inside the timed region
    host_fields = None
    if not args.no_e2e:
        try:
            host_fields = run_e2e(args, line, core, dist, dev, world, barrier, T, S, V, grid, z_i, depth, pres, eta,
                                  nt, ny, nx, points)
        except (RuntimeError, MemoryError) as exc:  # e.g. not enough pinnable host memory for 8 ranks
            line["e2e"] = {"value": None, "unit": UNIT, "error": f"{type(exc).__name__}: {exc}"[:300]}
        if host_fields is not None:
            del T, S
            torch.cuda.empty_cache()

    # ---- cpu_baseline: the oracle on a bounded sample of the same workload (rank 0, N=1 only)
    if rank == 0 and world == 1 and not args.no_cpu:
        if host_fields is None:
            host_fields = (T.cpu().numpy(), S.cpu().numpy(), V.cpu().numpy(), grid["areacello"].cpu().numpy(),
                           depth.cpu().numpy(), grid["z_l"].cpu().numpy(), z_i.cpu().numpy())
        rows, nslabs = 8, 3
        row0 = max(0, ny // 2 - rows * nslabs // 2)
        kind, ref_files = reference_kernels()
        cpu_path(host_fields, rows, 1, 1, row0)  # warm-up
        sec, pts, etas = cpu_path(host_fields, rows, nslabs, 1, row0)
        got = eta[:, row0: row0 + rows * nslabs].cpu().numpy()
        want = np.concatenate(etas, axis=1)
        same_nan = bool(np.array_equal(np.isnan(got), np.isnan(want)))
        m = ~np.isnan(want)
        m[0, 0, 0] = m.any() or True  # never reduce over an empty set
        got, want = np.nan_to_num(got), np.nan_to_num(want)
        line["cpu_baseline"] = {
            "value": pts / sec, "unit": UNIT, "cores": 1, "kind": kind, "reference_files_used": ref_files,
            "sample": f"rows {row0}..{row0 + rows * nslabs} of {ny}: {rows * nslabs}x{nx} columns x {nz} levels x {nt} steps"
                      f" = {pts} points, numpy oracle on fp64-upcast inputs, single thread",
            "seconds": sec, "host_cpu_count": os.cpu_count(),
            "parity_max_abs_err_m": float(np.max(np.abs(got[m] - want[m]))), "parity_nan_pattern_equal": same_nan,
        }

    # ---- the other BASELINE configs (3: ensemble sharded by member x time block, 4: time-sharded global series with
    # its gather inside the timed region, 5: linear EOS + spice), each with its own roofline and oracle check
    which = [c for c in (args.configs or "").replace(" ", "").split(",") if c in ("3", "4", "5")]
    if which and not args.no_configs and args.workload == "om4p25":
        host_fields = eta = rho_ref = sums = V = None  # noqa: F841 -- release the headline's buffers first
        try:
            del T, S
        except NameError:  # the e2e leg has released them already
            pass
        import gc

        gc.collect()
        torch.cuda.empty_cache()
        launches1 = core.launch_count()
        try:
            line.setdefault("extras", {})["configs"] = bc.run_configs(which, rank, world, dev)
        except Exception as exc:  # noqa: BLE001 -- the headline line must still be printed
            if world > 1:
                raise
            line.setdefault("extras", {})["configs"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        line["extras"]["configs_gpu_launches_rank0"] = core.launch_count() - launches1

    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    # stdout carries the one JSON line; NCCL's version / debug banner (NCCL_DEBUG=VERSION on the GPU boxes) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
