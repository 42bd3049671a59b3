"""Track runs end to end through ``lec_run_host_raw``: staging windows on (``lec_set_host_windows``) against whole
slots, alternated in one process, on int16 big-endian interleaved records (NetCDF-3 record variables, pinned).

Shapes (0.1 deg, 55 levels, 151 x 151 boxes, hourly steps):
  c5_segment  bench.py's c5 segment: 270 steps over 436 x 298 columns (the segment's extent + margin)
  c5_extent   the whole config-5 track extent, 2320 x 1240 columns, crossed diagonally in --long-steps steps
Records repeat cyclically (slot s reads record s % --records): each slot's record crosses PCIe as in a real run, while
host memory holds only --records of them.

Modes, per repetition in this order:
  whole    windows off (whole slots)
  windows  windows on: each window's raw rows AND columns (the window's raw columns are one run: a crop)
  rows     windows on over a longitude map whose 4-column groups are rotated inside 16-column blocks, so no window's raw
           columns form one run: the whole raw rows of the window's row range cross PCIe (the fallback), with the
           same ingest work (every group of four raw columns stays consecutive and aligned).  This measures the DMA
           cost of short cropped rows against whole rows; its outputs are of permuted fields and are not compared.
Reports steps/s, measured and modelled (engine.track_windows) H2D bytes per step, and the device name, power limit
and SM clock read in the same run, to --out (JSON)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HALF, NLEV = 75, 55


def device_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                            "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_clock"], info["sm_clock_max"] = [x.strip() for x in q.split(",")]
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def case(name, nlon, nlat, nsteps, nrec, reps, rng):
    from lorenzcycletoolkit_b200 import engine as E
    side = 2 * HALF + 1
    lon = (-150.0 + 0.1 * np.arange(nlon)).astype(np.float32)
    lat = (-60.0 + 0.1 * np.arange(nlat)).astype(np.float32)
    lev = np.linspace(1000.0, 100000.0, NLEV)
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    rec = np.empty((nrec, 5, NLEV, nlat, nlon), dtype=">i2")
    for r in range(nrec):
        rec[r] = rng.integers(-3000, 3000, size=rec.shape[1:], dtype=np.int16)
    raws = [rec[:, f] for f in range(5)]
    pinned = E.pin_arrays(raws)
    decode = [{"scale": s, "offset": o, "float32": True}
              for s, o in ((0.01, 250.0), (0.01, 0.0), (0.01, 0.0), (1e-4, 0.0), (1.0, 5e4))]
    nslots = nsteps + 2
    steps = E.time_stencil(3600.0 * np.arange(nslots), E.make_steps(nslots))[1:-1].copy()
    ci = np.round(np.linspace(HALF + 5, nlon - HALF - 6, nsteps)).astype(np.int32)
    cj = np.round(np.linspace(HALF + 5, nlat - HALF - 6, nsteps)).astype(np.int32)
    steps["i0"], steps["i1"], steps["j0"], steps["j1"] = ci - HALF, ci + HALF, cj - HALF, cj + HALF
    slot_record = np.arange(nslots) % nrec
    ident = (np.arange(nlon, dtype=np.int32), np.arange(nlat, dtype=np.int32), np.arange(NLEV, dtype=np.int32))
    g = np.arange(nlon) // 4
    blk, grp = g // 4, g % 4
    rot = np.where((blk + 1) * 16 <= nlon, blk * 16 + ((grp + 1) % 4) * 4 + np.arange(nlon) % 4, np.arange(nlon))
    rows = (rot.astype(np.int32), ident[1], ident[2])
    eng = E.LecEngine(f64(lon), f64(lat), f64(np.deg2rad(lon)), f64(np.deg2rad(lat)), f64(np.cos(np.deg2rad(lat))),
                      lev, np.float32, max_steps=64, max_box_rows=side)
    modes = {"whole": (False, ident), "windows": (True, ident), "rows": (True, rows)}

    def run(mode):
        on, maps = modes[mode]
        eng.set_host_windows(on)
        t0 = time.perf_counter()
        out = eng.run_host_raw(raws, *maps, slot_record, steps, decode=decode, want_levels=True)
        return time.perf_counter() - t0, eng.last_transfer()[0], out
    ref = {}
    for m in modes:                                    # warm-up: staging buffers, raw buffers, module loads
        _, _, ref[m] = run(m)
    for n, (a, b) in enumerate(zip(ref["whole"], ref["windows"])):
        assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)), (name, n)
    res = {m: {"s": [], "h2d_bytes": None} for m in modes}
    for _ in range(reps):
        for m in modes:
            t, b, _ = run(m)
            res[m]["s"].append(t)
            res[m]["h2d_bytes"] = int(b)
    model = {}
    for m, (on, maps) in modes.items():
        if on:
            model[m] = E.track_windows(steps, (NLEV, nlat, nlon), np.float32, nslots=nslots, max_steps=64,
                                       raw=(*maps, nlon, 2))["h2d_bytes"]
    out = {"grid": [NLEV, nlat, nlon], "steps": nsteps, "box": [side, side, NLEV], "records_distinct": nrec, "pinned": bool(pinned),
           "record_bytes": int(5 * NLEV * nlat * nlon * 2), "modes": {}}
    for m, r in res.items():
        best = min(r["s"])
        out["modes"][m] = {"seconds": r["s"], "steps_per_s": nsteps / best, "steps_per_s_median": nsteps / float(np.median(r["s"])),
                           "h2d_bytes_per_step": r["h2d_bytes"] / nsteps,
                           "model_h2d_bytes_per_step": model[m] / nsteps if m in model else None}
        if m in model:
            assert r["h2d_bytes"] == model[m], (name, m, r["h2d_bytes"], model[m])
    w = out["modes"]
    out["h2d_ratio_whole_over_windows"] = w["whole"]["h2d_bytes_per_step"] / w["windows"]["h2d_bytes_per_step"]
    out["speedup_windows_over_whole"] = w["windows"]["steps_per_s"] / w["whole"]["steps_per_s"]
    out["speedup_windows_over_rows"] = w["windows"]["steps_per_s"] / w["rows"]["steps_per_s"]
    eng.close()
    print(name, json.dumps(out["modes"], indent=None), flush=True)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--records", type=int, default=16, help="distinct records held in host memory per shape")
    ap.add_argument("--long-steps", type=int, default=64, help="steps of the c5_extent track")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "track_e2e_b200.json"))
    args = ap.parse_args()
    import __graft_entry__ as G
    G.build()
    rng = np.random.default_rng(0)
    result = {"info": device_info(), "reps": args.reps,
              "c5_segment": case("c5_segment", 436, 298, 270, args.records, args.reps, rng),
              "c5_extent": case("c5_extent", 2320, 1240, args.long_steps, min(args.records, 8), args.reps, rng),
              "info_after": device_info()}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: result[k] for k in ("info", "info_after")}))
