#!/usr/bin/env python
"""Benchmark of the LEC hot path (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (``configs[3]`` of BASELINE.json, the largest single-GPU configuration): synthetic
ERA5 0.25 deg global-shape fields, 1440 x 721 x 37 levels, fp32, fixed box = all
longitudes x the 719 non-pole rows, hourly steps.  The full 744-step month is 572 GB, so
each GPU holds a resident time chunk of ``--chunk`` steps (+1 halo slot each side); one
bench "step" = one pass of the engine over that chunk (all 16 terms + 19 per-level families
for every time step of the chunk).  ``value`` = time steps/s over all GPUs with the inputs
resident in HBM; ``e2e`` = the same metric through ``lec_run_host`` with pinned HOST
buffers (H2D of every slot the pass needs -- five fields of the chunk's steps plus T of the two halo
slots, counted by the engine itself, ``lec_last_transfer`` -- and D2H of the results inside the timed
region); ``e2e.packed_int16`` = the same pass from int16-packed records (ERA5's on-disk form) through
``lec_run_host_raw``, decoded to fp64 on the device.
Time steps are independent, so N GPUs = N time shards (weak scaling) + ONE in-place NCCL
all-gather of the per-step results per pass (the finalize kernels write into this rank's slice of the
gather buffer).  The device-resident passes call the engine through ``torch.ops.lec_b200.run_device``
(the PyTorch C++ extension over the C ABI).  Extra keys of the line: ``e2e.plugin`` (the reference-facing
``lec_fixed`` call incl. all CSVs), ``fp64`` (float64 fields), ``c5`` (0.1 deg Semi-Lagrangian track boxes,
BASELINE.json configs[4]), ``clocks.power_w``.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "LEC timesteps/s (all terms), 0.25°×37-lvl ERA5 shape; % of HBM roofline"
UNIT = "timesteps/s"
NLON, NLAT, NLEV = 1440, 721, 37
BOX = dict(i0=0, i1=NLON - 1, j0=1, j1=NLAT - 2)          # pole rows excluded (cos(lat) = 0)
BOX_ROWS = BOX["j1"] - BOX["j0"] + 1
ALG_BYTES_PER_TIMESTEP = 5 * NLEV * BOX_ROWS * NLON * 4   # T,u,v,omega,Phi read once (SURVEY 8(d))


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chunk", type=int, default=48, help="resident time steps per GPU per pass")
    ap.add_argument("--e2e-chunk", type=int, default=12,
                    help="time steps per end-to-end pass (+2 halo slots); reduced if pinned host memory is short")
    ap.add_argument("--e2e-passes", type=int, default=3)
    ap.add_argument("--band-rows", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-e2e-packed", action="store_true", help="skip the int16-packed lec_run_host_raw variant")
    ap.add_argument("--fp64-chunk", type=int, default=24, help="time steps per pass of the float64-field line")
    ap.add_argument("--c5-steps", type=int, default=270, help="track steps per GPU of the C5 (0.1 deg track) line")
    ap.add_argument("--no-fp64", action="store_true")
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--no-plugin", action="store_true", help="skip the lec_fixed (plugin call) end-to-end line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed passes, write what the last one returned (terms, levels, flags; all ranks) "
                         "to DIR/<name>.npy as float64; the inputs are seeded, so two builds compare file for file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def row_kernel_name():
    """The row kernel the engine takes for the wide C4 rows (build default, LEC_ROW_KERNEL overrides)."""
    from lorenzcycletoolkit_b200 import engine as E
    return E.wide_row_kernel()


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def config_dict(chunk=48):
    """The workload, identical in both arms (the driver compares the two `config` objects)."""
    return {"workload": "synthetic ERA5 0.25deg global-shape 1440x721x37 fp32, fixed box 1440x719 "
                        "(pole rows excluded), hourly steps; BASELINE.json configs[3]",
            "box": [BOX["i0"], BOX["i1"], BOX["j0"], BOX["j1"]],
            "alg_bytes_per_timestep": ALG_BYTES_PER_TIMESTEP,
            "timesteps_per_pass_per_gpu": chunk,
            "l2": "inputs (>= 4.6 GB per pass) larger than L2; no flush needed"}


# --------------------------------------------------------------------------------------- #
class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def summary(self, t0, t1):
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons, pw = [], 0.0, set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [r for (t, r) in self.rows if t0 - 0.15 <= t <= t1 + 0.15] or [r for (_, r) in self.rows[-3:]]
        for r in rows:
            c = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(c[0])); mx = max(mx, float(c[1]))
            except (ValueError, IndexError):
                continue
            try:
                pw.append(float(c[2]))
            except (ValueError, IndexError):
                pass
            for n, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w": float(np.median(pw)) if pw else None}


# --------------------------------------------------------------------------------------- #
def cpu_port_baseline():
    """The numpy oracle on ONE full-size time step, one core (``kind: port``)."""
    import torch
    from oracle import cpu_bench as CB
    from lorenzcycletoolkit_b200 import synthetic as S
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))     # data synthesis only
    grid = S.era5_grid(NLON, NLAT)
    sub = dict(grid)
    for k in ("lat", "rlats", "coslats"):
        sub[k] = grid[k][1:NLAT - 1]
    fields = [x.numpy() for x in S.synth_fields(sub, 3, np.float32, "cpu")]
    P = CB.make_prepared(sub, fields, 0, BOX_ROWS)
    _, sec = CB.one_step(P)
    return {"value": 1.0 / sec, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"numpy oracle (restatement of the reference's xarray/numpy path), 1 full time step "
                      f"1440x719x37 fp32 in {sec:.1f} s, single process; the real reference cannot be "
                      f"imported in this image"}


def run_reference(args, rank):
    if rank != 0:
        return
    from oracle import cpu_bench as CB
    ncpu = os.cpu_count() or 1
    try:
        import psutil
        mem = psutil.virtual_memory().available
    except Exception:
        mem = 64 << 30
    total_steps = args.steps + args.warmup
    per_row = 55 * NLON * NLEV * 4                             # measured peak RSS ~ 55 one-slot field copies per row
    nproc = max(1, min(ncpu, 64))
    # the workload's own box (all 719 rows) whenever the run still ends within a few minutes (~10 s per
    # full step and process) and the host RAM holds one full step per process; else a latitude band
    if total_steps * 10.0 <= 300.0 and int(0.6 * mem / (BOX_ROWS * per_row)) >= 1:
        rows = BOX_ROWS
        nproc = max(1, min(nproc, int(0.6 * mem / (BOX_ROWS * per_row))))
    else:
        budget = 150.0 / max(total_steps, 1)                      # seconds per bench step
        rows = int(budget / (450e-9 * NLEV * NLON * 1.5))          # ~450 ns/point, 1.5x safety
        rows = min(rows, int(0.5 * mem / (nproc * per_row)))
        rows = max(8, min(BOX_ROWS, rows))
    times = CB.run_parallel(nproc, NLON, NLAT, rows, total_steps)
    timed = times[args.warmup:]
    total = float(np.sum(timed))
    # one band-step is rows/719 of a time step of the workload
    value = nproc * (rows / BOX_ROWS) * len(timed) / total
    sample = (f"numpy oracle, {nproc} processes x 1 time step each per bench step on "
              + ("the workload's full 1440x719x37 box" if rows == BOX_ROWS else
                 f"a {rows}-row latitude band (of {BOX_ROWS}) of the workload, scaled by rows")
              + "; real reference not importable here")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / len(timed), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "impl": "reference", "config": config_dict(args.chunk),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": nproc, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)



# --------------------------------------------------------------------------------------- #
def bench_fp64(args, grid, fields32, steps, dev, local_rank, world):
    """The same box with float64 FIELDS (what int16-packed ERA5 decodes to): device-resident, `--fp64-chunk`
    steps per pass.  Algorithmic bytes double (8 B per value)."""
    import torch
    import torch.distributed as dist
    from lorenzcycletoolkit_b200 import engine as E
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    n = min(args.fp64_chunk, len(steps))
    fields = [f[: n + 2].double() for f in fields32]
    eng = E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]),
                      f64(grid["coslats"]), grid["level"], np.float64, max_steps=n,
                      max_box_rows=BOX_ROWS, device=local_rank, band_rows=args.band_rows)
    st = steps[:n].copy()
    for _ in range(3):
        terms, levels, flags = eng.run_torch(fields, st)
    torch.cuda.synchronize(dev)
    assert int(flags.max().item()) == 0
    if world > 1:
        dist.barrier()
    eng.timing_reset()
    reps = max(3, args.steps // 2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.run_torch(fields, st)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    rows_ms = eng.last_timing()[0] / reps
    eng.close()
    del fields
    torch.cuda.empty_cache()
    peak, _ = measured_peak()
    alg = 2 * ALG_BYTES_PER_TIMESTEP
    ach = alg * n / (rows_ms * 1e-3) / 1e9
    return {"value": world * n * reps / (float(ms.item()) * 1e-3), "unit": UNIT, "dtype": "f64",
            "timesteps_per_pass_per_gpu": n, "passes": reps, "alg_bytes_per_timestep": alg,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "kernel_ms": rows_ms}}


C5_STEPS_TOTAL, C5_HALF, C5_NLEV = 2160, 75, 55          # BASELINE.json configs[4]: 0.1 deg, 55 levels, 151 x 151 boxes


def bench_c5(args, dev, rank, local_rank, world):
    """BASELINE.json configs[4] shape: 0.1 deg grid, 55 levels, a Semi-Lagrangian track of 2160 hourly steps with a
    15 x 15 deg (151 x 151 point) box per step, time-sharded: every GPU evaluates one `--c5-steps`-step segment
    of the track (2160 / 8 = 270 on an 8-GPU box) in ONE engine call.  Only the segment's extent +- margin is
    resident -- what the reference's slice_domain hands over (select_area.py:297-313) --, not the 7 GB/step
    global field.  The box moves 1 grid point per step in longitude and 1 every other step in latitude."""
    import torch
    import torch.distributed as dist
    from lorenzcycletoolkit_b200 import engine as E, synthetic as S
    n, half = args.c5_steps, C5_HALF
    side = 2 * half + 1
    nlon = (n + side + 12 + 3) // 4 * 4
    nlat = n // 2 + side + 12
    first = rank * n
    lon = (-150.0 + 0.1 * (first + np.arange(nlon))).astype(np.float32)
    lat = (-60.0 + 0.1 * (first // 2 + np.arange(nlat))).astype(np.float32)
    lev = np.linspace(1000.0, 100000.0, C5_NLEV)
    grid = dict(lon=lon, lat=lat, level=lev, rlons=np.deg2rad(lon), rlats=np.deg2rad(lat),
                coslats=np.cos(np.deg2rad(lat)))
    fields = S.synth_fields(grid, n + 2, np.float32, dev, t0=first)
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    eng = E.LecEngine(f64(lon), f64(lat), f64(grid["rlons"]), f64(grid["rlats"]), f64(grid["coslats"]), lev,
                      np.float32, max_steps=n, max_box_rows=side, device=local_rank)
    steps = E.time_stencil(3600.0 * np.arange(n + 2), E.make_steps(n + 2))[1:-1].copy()
    ci = half + 5 + np.arange(n)
    cj = half + 5 + np.arange(n) // 2
    steps["i0"], steps["i1"], steps["j0"], steps["j1"] = ci - half, ci + half, cj - half, cj + half
    for _ in range(3):
        terms, levels, flags = eng.run_torch(fields, steps)
    torch.cuda.synchronize(dev)
    assert int(flags.max().item()) == 0
    if world > 1:
        dist.barrier()
    eng.timing_reset()
    reps = max(5, args.steps)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        eng.run_torch(fields, steps)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    rows_ms, fin_ms, _ = eng.last_timing()
    rows_ms, fin_ms = rows_ms / reps, fin_ms / reps
    eng.close()
    del fields
    torch.cuda.empty_cache()
    peak, _ = measured_peak()
    alg = 5 * C5_NLEV * side * side * 4
    steps_per_s = world * n * reps / (float(ms.item()) * 1e-3)
    ach = alg * n / (rows_ms * 1e-3) / 1e9
    out = {"steps_per_s": steps_per_s, "unit": "track steps/s", "n_gpus": world, "steps_per_gpu_per_pass": n,
           "track_steps_total": C5_STEPS_TOTAL, "box": [side, side, C5_NLEV], "alg_bytes_per_step": alg,
           "frac": alg * steps_per_s / world / 1e9 / peak,
           "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "kernel_ms": rows_ms, "finalize_kernel_ms": fin_ms},
           "workload": "synthetic 0.1deg MPAS-A-regridded shape, 55 levels, Semi-Lagrangian 151x151 boxes, "
                       "one track segment per GPU; BASELINE.json configs[4]"}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f).get("c5", {})
        if tj.get("steps") == n:
            out["dram_over_alg"] = tj["dram_bytes_per_launch"] / (alg * n)
    return out


def bench_plugin(args, grid, nslots, dev, rank, local_rank, world):
    """End to end through the reference-facing plugin call: `lec_fixed(data, variable_list_df, ...)` on a C4-shaped
    dataset held in HOST memory (BoxData -> engine staging H2D -> kernels -> D2H -> the four term classes ->
    21 per-level CSV families + the results CSV written to tmpfs), wall clock.  Under torchrun the call shards
    the time steps over the ranks itself (strong scaling of this one job) and rank 0 writes."""
    import argparse as ap
    import logging
    import shutil
    import tempfile
    import pandas as pd
    import torch
    import torch.distributed as dist
    from lorenzcycletoolkit_b200 import synthetic as S
    from lorenzcycletoolkit_b200.frameworks import lec_fixed
    from lorenzcycletoolkit_b200.utils.preprocessing import LecDataset
    # the pole rows are outside the workload's box (cos(lat) = 0): the dataset is rows 1 .. 719, as slice_domain
    # would hand it over; every rank holds the same dataset
    sub = dict(grid)
    for k in ("lat", "rlats", "coslats"):
        sub[k] = grid[k][BOX["j0"]:BOX["j1"] + 1]
    fields = S.synth_fields(sub, nslots, np.float32, dev, t0=0)
    host = [torch.empty(f.shape, dtype=torch.float32, pin_memory=True) for f in fields]
    for h, d in zip(host, fields):
        h.copy_(d)
    torch.cuda.synchronize(dev)
    del fields
    torch.cuda.empty_cache()
    names = ["t", "u", "v", "w", "z"]
    data = LecDataset(variables={k: h.numpy() for k, h in zip(names, host)},
                      time=np.datetime64("2020-01-01T00", "ns") + np.arange(nslots) * np.timedelta64(1, "h"),
                      level=np.asarray(sub["level"]), lat=sub["lat"], lon=sub["lon"], rlats=sub["rlats"],
                      coslats=sub["coslats"], rlons=sub["rlons"],
                      names={"Time": "time", "Vertical Level": "level", "Latitude": "latitude", "Longitude": "longitude"})
    nl = pd.DataFrame({"Variable": ["t", "u", "v", "w", "z", "longitude", "latitude", "time", "level"],
                       "Units": ["K", "m/s", "m/s", "Pa/s", "m**2/s**2", "", "", "", "Pa"]},
                      index=["Air Temperature", "Eastward Wind Component", "Northward Wind Component", "Omega Velocity",
                             "Geopotential", "Longitude", "Latitude", "Time", "Vertical Level"])
    base = "/dev/shm" if os.path.isdir("/dev/shm") else None
    out = tempfile.mkdtemp(prefix=f"lec_bench_r{rank}_", dir=base)
    os.makedirs(os.path.join(out, "lv"))
    with open(os.path.join(out, "box"), "w") as f:
        f.write(f"min_lon;{float(grid['lon'][0])}\nmax_lon;{float(grid['lon'][-1])}\n"
                f"min_lat;{float(data.lat[0])}\nmax_lat;{float(data.lat[-1])}\n")
    a = ap.Namespace(infile="synthetic_C4.nc", fixed=True, track=False, choose=False, residuals=True,
                     box_limits=os.path.join(out, "box"), outname=None, plots=False, cdsapi=False, mpas=False)
    log = logging.getLogger("lec_bench")
    log.setLevel(logging.ERROR)
    best, split = None, None
    try:
        for rep in range(1 + args.e2e_passes):                 # first call = warm-up (CUDA context of the engine path)
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            df = lec_fixed(data, nl, out, os.path.join(out, "lv"), log, a, engine_options={"device": local_rank})
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            dt = float(dt.item())
            if rep > 0 and (best is None or dt < best):
                best, split = dt, dict(df.attrs.get("engine_ms", {}))
        assert np.isfinite(df["Az"].values).all() and len(df) == nslots
        files = len(os.listdir(os.path.join(out, "lv"))) if rank == 0 else 0
    finally:
        shutil.rmtree(out, ignore_errors=True)
    slot_bytes = NLEV * BOX_ROWS * NLON * 4
    return {"value": nslots / best, "unit": UNIT, "timesteps": nslots, "wall_s": best, "n_gpus": world,
            "scaling": "strong (one lec_fixed job sharded over the ranks)" if world > 1 else "single process",
            "h2d_bytes_per_step": int(5 * nslots * slot_bytes), "level_csv_files": files,
            "engine_call_ms": split.get("call_incl_copies") if split else None,
            "host_ms": (1e3 * best - split["call_incl_copies"]) if split else None,   # engine create/destroy, term classes, CSVs
            "api": "lorenzcycletoolkit_b200.frameworks.lec_fixed(data, variable_list_df, ...) -> BoxData -> "
                   "lec_run_host -> EnergyContents / ConversionTerms / BoundaryTerms / GenerationDissipationTerms "
                   "-> per-level CSVs + results CSV on tmpfs (best of %d calls, wall clock)" % args.e2e_passes}


def dump_outputs(d, g_res, flags, chunk, rank, world, dev):
    """``--dump-outputs``: the gathered results of the last timed pass as a caller receives them -- terms
    [steps, 16], levels [steps, 19, levels] and flags [steps] over the time steps of all ranks -- written by rank 0
    as float64 ``.npy`` (~0.3 MB per rank)."""
    import torch
    import torch.distributed as dist
    from lorenzcycletoolkit_b200 import engine as E
    if world > 1:
        gathered = torch.empty(world * chunk, dtype=flags.dtype, device=dev)
        dist.all_gather_into_tensor(gathered, flags)
        flags = gathered
    if rank != 0:
        return
    nt = chunk * E.NTERMS
    per_rank = g_res.view(world, -1)
    arrays = {"terms": per_rank[:, :nt].reshape(world * chunk, E.NTERMS),
              "levels": per_rank[:, nt:].reshape(world * chunk, E.NLEVEL_TERMS, NLEV),
              "flags": flags}
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, f"{name}.npy"), a.cpu().numpy().astype(np.float64))


# --------------------------------------------------------------------------------------- #
def run_b200(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from lorenzcycletoolkit_b200 import engine as E, synthetic as S

    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_base = cpu_port_baseline()            # before CUDA work: keeps the GPU timing clean

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))
    grid = S.era5_grid(NLON, NLAT)
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    chunk = args.chunk
    nslots = chunk + 2
    # time shard of this rank: steps [rank*chunk, (rank+1)*chunk) of the global hourly axis,
    # loaded with a one-slot halo on both sides (first/last slots are halos only)
    t_first = rank * chunk
    fields = S.synth_fields(grid, nslots, np.float32, dev, t0=t_first)
    eng = E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]),
                      f64(grid["coslats"]), grid["level"], np.float32, max_steps=chunk,
                      max_box_rows=BOX_ROWS, device=local_rank, band_rows=args.band_rows)
    steps = E.time_stencil(3600.0 * np.arange(nslots), E.make_steps(nslots))[1:-1].copy()
    for k, v in BOX.items():
        steps[k] = v
    # results: the finalize kernels write straight into this rank's slice of ONE gather buffer
    # ([terms | levels] per rank), one in-place all-gather per pass, nothing allocated inside the timed region
    nt, nl = chunk * E.NTERMS, chunk * E.NLEVEL_TERMS * NLEV
    g_res = torch.empty(world * (nt + nl), dtype=torch.float64, device=dev)
    mine = g_res[rank * (nt + nl):(rank + 1) * (nt + nl)]
    out = (mine[:nt].view(chunk, E.NTERMS), mine[nt:].view(chunk, E.NLEVEL_TERMS, NLEV),
           torch.zeros(chunk, dtype=torch.int32, device=dev))

    def one_pass():
        terms, levels, flags = eng.run_torch(fields, steps, out=out)
        if world > 1:
            dist.all_gather_into_tensor(g_res, mine)
        return terms, levels, flags

    def sync():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        terms, levels, flags = one_pass()
    sync()
    assert int(flags.max().item()) == 0, "synthetic data must not hit the NaN / sigma-floor paths"
    # nvidia-smi needs ~1 s to start sampling: keep the GPUs under the same load until rank 0 has a
    # first sample, so the clock record overlaps the timed region (extra warm-up passes, untimed).
    # Every rank runs the same passes: rank 0's decision is broadcast, because a pass contains
    # collectives at N > 1.
    t_wait = time.time()
    while True:
        one_pass()
        done = torch.tensor([1 if (sampler is None or sampler.rows or time.time() - t_wait > 5.0) else 0],
                            dtype=torch.int32, device=dev)
        if world > 1:
            dist.broadcast(done, src=0)
        if int(done.item()):
            break
    sync()
    eng.timing_reset()                     # accumulate the kernel durations of every timed pass
    launches0 = eng.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        one_pass()
    e1.record()
    sync()
    wall1 = time.time()
    # average kernel durations over the timed passes (CUDA events recorded by the engine around its
    # launches on torch's current stream)
    rows_ms, fin_ms, _ = eng.last_timing()
    rows_ms, fin_ms = rows_ms / args.steps, fin_ms / args.steps
    elapsed_ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    elapsed_ms = float(elapsed_ms.item())
    launches = eng.launch_count - launches0
    clocks = sampler.summary(wall0, wall1) if sampler else None
    value = world * chunk * args.steps / (elapsed_ms * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, g_res, out[2], chunk, rank, world, dev)

    # ---- the same box with float64 fields (the path int16-packed ERA5 takes) ------------------
    fp64_line = None if args.no_fp64 else bench_fp64(args, grid, fields, steps, dev, local_rank, world)

    # ---- end to end through lec_run_host with pinned host buffers --------------------------
    e2e = None
    if not args.no_e2e:
        ec = args.e2e_chunk
        try:                                  # keep the pinned buffers of all ranks below 35 % of the free host RAM
            import psutil
            avail = psutil.virtual_memory().available
            ec = max(2, min(ec, int(0.35 * avail / world / (5 * NLEV * NLAT * NLON * 4)) - 2))
        except Exception:
            pass
        ec = min(ec, chunk)
        host = [torch.empty((ec + 2, NLEV, NLAT, NLON), dtype=torch.float32, pin_memory=True) for _ in range(5)]
        for h, d in zip(host, fields):
            h.copy_(d[: ec + 2])
        torch.cuda.synchronize(dev)
        del fields
        torch.cuda.empty_cache()
        heng = E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]),
                           f64(grid["coslats"]), grid["level"], np.float32, max_steps=ec,
                           max_box_rows=BOX_ROWS, device=local_rank, band_rows=args.band_rows)
        hsteps = steps[:ec].copy()
        harr = [h.numpy() for h in host]
        heng.run_host(harr, hsteps)                              # warm-up (allocates the staging buffers)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_passes):
            ht, hl, hf = heng.run_host(harr, hsteps)
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        e2e = {"value": world * ec * args.e2e_passes / dt, "unit": UNIT,
               "h2d_bytes_per_step": int(heng.last_transfer()[0]),   # counted by the engine from its copies:
               "d2h_bytes_per_step": int(heng.last_transfer()[1]),   # 5 fields x ec slots + T of the 2 halo slots
               "timesteps_per_pass": ec, "passes": args.e2e_passes,
               "api": "LecEngine.run_host -> lec_run_host (pinned host buffers)"}
        heng.close()

        # ---- same, from int16-PACKED records (the way ERA5 NetCDF stores them): lec_run_host_raw ----
        # scale_factor + add_offset per field, decoded on the device to float64 as xarray would; the
        # engine then runs its fp64 path.  PCIe carries 2 bytes per value instead of 4.
        if not args.no_e2e_packed:
            packed, decode = [], []
            for h in host:
                lo, hi = float(h.min()), float(h.max())
                sc, off = (hi - lo) / 65000.0, 0.5 * (hi + lo)
                q = torch.empty(h.shape, dtype=torch.int16, pin_memory=True)
                for s_ in range(h.shape[0]):
                    q[s_].copy_(((h[s_].to(dev, non_blocking=True).double() - off) / sc).round().to(torch.int16))
                packed.append(q.numpy())
                decode.append(dict(scale=np.float64(sc), offset=np.float64(off)))
            torch.cuda.synchronize(dev)
            del host, harr
            torch.cuda.empty_cache()
            peng = E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]),
                               f64(grid["coslats"]), grid["level"], np.float64, max_steps=ec,
                               max_box_rows=BOX_ROWS, device=local_rank, band_rows=args.band_rows)
            ident = (np.arange(NLON), np.arange(NLAT), np.arange(NLEV))
            rec = np.arange(ec + 2)
            pt, _, pf = peng.run_host_raw(packed, *ident, rec, hsteps, decode=decode)        # warm-up
            # (bit parity of this path is a test, tests/test_raw_ingest_gpu.py; here only a sanity figure: the
            #  terms of the 16-bit quantised fields against the fp32 run, scaled by each term's magnitude)
            qerr = float(np.max(np.abs(pt - ht).max(axis=0) / np.abs(ht).max(axis=0)))
            assert int(pf.max()) == 0 and np.isfinite(pt).all()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(args.e2e_passes):
                peng.run_host_raw(packed, *ident, rec, hsteps, decode=decode)
            dtp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dtp, op=dist.ReduceOp.MAX)
            e2e["packed_int16"] = {"value": world * ec * args.e2e_passes / float(dtp.item()), "unit": UNIT,
                                   "h2d_bytes_per_step": int(peng.last_transfer()[0]),
                                   "d2h_bytes_per_step": int(peng.last_transfer()[1]),
                                   "quantisation_diff_vs_f32_run": qerr,
                                   "api": "LecEngine.run_host_raw -> lec_run_host_raw (pinned int16 records, "
                                          "scale_factor + add_offset decoded to fp64 on the device)"}
            peng.close()

    if "fields" in locals():
        del fields
    torch.cuda.empty_cache()
    # ---- end to end through the plugin call (lec_fixed on host arrays, CSVs included) -----------
    if e2e is not None and not args.no_plugin:
        e2e["engine"] = {k: e2e[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "api")}
        e2e["plugin"] = bench_plugin(args, grid, min(args.e2e_chunk, chunk) + 2, dev, rank, local_rank, world)
    # ---- C5: 0.1 deg Semi-Lagrangian track, one segment per GPU ---------------------------------
    c5_line = None if args.no_c5 else bench_c5(args, dev, rank, local_rank, world)

    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = ALG_BYTES_PER_TIMESTEP * chunk / (rows_ms * 1e-3) / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            if tj.get("chunk") == chunk:
                traffic = tj.get("dram_bytes_per_launch")
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": config_dict(chunk),
                "parallelism": f"time-sharded x{world}" + (", NCCL all-gather of per-step results" if world > 1 else ""),
                "arithmetic": "fp32 pointwise, fp64 reductions and finalize",
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                             "kernel": row_kernel_name(), "kernel_ms": rows_ms,
                             "finalize_kernel_ms": fin_ms,
                             "alg_bytes_per_launch": ALG_BYTES_PER_TIMESTEP * chunk},
                "cpu_baseline": cpu_base, "fp64": fp64_line, "c5": c5_line}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world == 1 and args.gpus > 1:
        # plain `python bench.py --gpus N`: relaunch under torchrun, one rank per GPU
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29517")] + sys.argv
        sys.exit(subprocess.call(cmd))
    run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
