"""Speed of the int16-packed device path (lec_run_device_packed) against the alternatives on the same data.

    python scripts/packed_probe.py [--steps 24] [--reps 5] [--c5-steps 270] [--out FILE]

C4 shape (ERA5 0.25 deg, 1440 x 721 x 37, fixed box 1440 x 719, hourly steps), int16 records packed from the seeded
synthetic fields of bench.py, in two decodings:
  fp64   ERA5 style: float64 scale_factor and add_offset, decoded to float64 (LEC_F64 handle)
  fp32   scale_factor only, decoded variable float32 (LEC_F32 handle)
and for each:
  packed     the row kernels read the int16 fields and decode on load (2 bytes per value resident)
  two_pass   decode the int16 fields into an fp scratch on the device (torch elementwise ops, the decode rule), then
             lec_run_device on the scratch: the way to use resident int16 data without this path
  resident   lec_run_device on fp fields that are already resident (4 / 8 bytes per value)
The C5 track shape (0.1 deg, 55 levels, 151 x 151 boxes moving 1 point per step) is measured packed (fp32 decode)
and resident fp32.  Rates are time steps per second over CUDA events around whole engine calls; "alg_GBps" is the
algorithmic bytes (five fields x box x levels at the STORED element size) over the row-kernel time.  Prints one
JSON object and writes it to --out.  Needs a CUDA device."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NLON, NLAT, NLEV = 1440, 721, 37
BOX = dict(i0=0, i1=NLON - 1, j0=1, j1=NLAT - 2)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def encode(fields, fp32):
    """int16 records + decode dicts: per field the range of the fields over all slots, 65000 codes."""
    import torch
    raws, decode = [], []
    for f in fields:
        lo, hi = float(f.min()), float(f.max())
        if fp32:
            scale, offset = max(abs(lo), abs(hi)) / 32000.0, None
            raw = torch.round(f.double() / scale)
        else:
            scale, offset = (hi - lo) / 65000.0, 0.5 * (hi + lo)
            raw = torch.round((f.double() - offset) / scale)
        raws.append(raw.to(torch.int16))
        decode.append(dict(scale=np.float64(scale), offset=None if offset is None else np.float64(offset),
                           fills=[-32767], float32=fp32))
    return raws, decode


def decode_into(raws, decode, out):
    """The decode rule with torch elementwise ops (the two-pass alternative's first pass)."""
    for r, d, o in zip(raws, decode, out):
        x = r.double() * d["scale"]
        if d["offset"] is not None:
            x = x + d["offset"]
        if d["float32"]:
            x = x.float().double()
        x = x.masked_fill(r == d["fills"][0], float("nan"))
        o.copy_(x)


def timed(fn, reps, eng=None):
    import torch
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    if eng is not None:
        eng.timing_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    rows_ms = eng.last_timing()[0] / reps if eng is not None else None
    return ms, rows_ms


def probe_c4(args, fields32, grid, steps):
    import torch
    from lorenzcycletoolkit_b200 import engine as E
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    n = len(steps)
    vals = 5 * (BOX["i1"] - BOX["i0"] + 1) * (BOX["j1"] - BOX["j0"] + 1) * NLEV
    out = {}
    for mode in ("fp64", "fp32"):
        fp32 = mode == "fp32"
        dt, tdt, esz = (np.float32, torch.float32, 4) if fp32 else (np.float64, torch.float64, 8)
        raws, decode = encode(fields32, fp32)
        pitch = (NLON + 7) // 8 * 8
        packed = []
        for r in raws:
            t = torch.zeros(r.shape[:3] + (pitch,), dtype=torch.int16, device=r.device)
            t[..., :NLON] = r
            packed.append(t)
        del raws
        eng = E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]), f64(grid["coslats"]),
                          grid["level"], dt, max_steps=n, max_box_rows=BOX["j1"] - BOX["j0"] + 1)
        res = {}
        ms, rows = timed(lambda: eng.run_torch_packed(packed, decode, steps), args.reps, eng)
        d = eng.last_dispatch()
        pt, _, pf = eng.run_torch_packed(packed, decode, steps)
        res["packed"] = dict(timesteps_per_s=n / (ms * 1e-3), row_kernel_ms_per_step=rows / n,
                             alg_GBps=vals * 2 * n / (rows * 1e-3) / 1e9, dispatch=d)
        scratch = [torch.empty(p.shape[:3] + (NLON,), dtype=tdt, device=p.device) for p in packed]
        views = [p[..., :NLON] for p in packed]

        def two_pass():
            decode_into(views, decode, scratch)
            return eng.run_torch(scratch, steps)
        ms, rows = timed(two_pass, args.reps, eng)
        tt, _, tf = two_pass()
        torch.cuda.synchronize()
        res["two_pass"] = dict(timesteps_per_s=n / (ms * 1e-3), row_kernel_ms_per_step=rows / n,
                               alg_GBps_fp_kernel=vals * esz * n / (rows * 1e-3) / 1e9)
        res["packed_equals_two_pass_bits"] = bool(torch.equal(pt.view(torch.int64), tt.view(torch.int64)))
        res["flags_max"] = int(max(pf.max().item(), tf.max().item()))
        # resident fp fields (no decode at all): the seeded fields themselves, upcast for fp64
        fp = [f.to(tdt) for f in fields32]
        ms, rows = timed(lambda: eng.run_torch(fp, steps), args.reps, eng)
        res["resident_fp"] = dict(timesteps_per_s=n / (ms * 1e-3), row_kernel_ms_per_step=rows / n,
                                  alg_GBps=vals * esz * n / (rows * 1e-3) / 1e9)
        res["packed_over_resident_fp_time"] = res["resident_fp"]["timesteps_per_s"] / res["packed"]["timesteps_per_s"]
        res["packed_over_two_pass_rate"] = res["packed"]["timesteps_per_s"] / res["two_pass"]["timesteps_per_s"]
        eng.close()
        del fp, scratch, packed, views
        torch.cuda.empty_cache()
        out[mode] = res
    return out


def probe_c5(args):
    import torch
    from lorenzcycletoolkit_b200 import engine as E, synthetic as S
    n, half, nlev = args.c5_steps, 75, 55
    side = 2 * half + 1
    nlon = (n + side + 12 + 3) // 4 * 4
    nlat = n // 2 + side + 12
    lon = (-150.0 + 0.1 * np.arange(nlon)).astype(np.float32)
    lat = (-60.0 + 0.1 * np.arange(nlat)).astype(np.float32)
    lev = np.linspace(1000.0, 100000.0, nlev)
    grid = dict(lon=lon, lat=lat, level=lev, rlons=np.deg2rad(lon), rlats=np.deg2rad(lat), coslats=np.cos(np.deg2rad(lat)))
    fields = S.synth_fields(grid, n + 2, np.float32, "cuda")
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    steps = E.time_stencil(3600.0 * np.arange(n + 2), E.make_steps(n + 2))[1:-1].copy()
    ci, cj = half + 5 + np.arange(n), half + 5 + np.arange(n) // 2
    steps["i0"], steps["i1"], steps["j0"], steps["j1"] = ci - half, ci + half, cj - half, cj + half
    raws, decode = encode(fields, True)
    pitch = (nlon + 7) // 8 * 8
    packed = []
    for r in raws:
        t = torch.zeros(r.shape[:3] + (pitch,), dtype=torch.int16, device=r.device)
        t[..., :nlon] = r
        packed.append(t)
    eng = E.LecEngine(f64(lon), f64(lat), f64(grid["rlons"]), f64(grid["rlats"]), f64(grid["coslats"]), lev,
                      np.float32, max_steps=n, max_box_rows=side)
    vals = 5 * nlev * side * side
    res = {"box": [side, side, nlev], "steps_per_call": n}
    ms, rows = timed(lambda: eng.run_torch_packed(packed, decode, steps), args.reps, eng)
    res["packed"] = dict(track_steps_per_s=n / (ms * 1e-3), alg_GBps=vals * 2 * n / (rows * 1e-3) / 1e9,
                         dispatch=eng.last_dispatch())
    ms, rows = timed(lambda: eng.run_torch(fields, steps), args.reps, eng)
    res["resident_fp32"] = dict(track_steps_per_s=n / (ms * 1e-3), alg_GBps=vals * 4 * n / (rows * 1e-3) / 1e9)
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=24, help="C4 time steps per engine call (+2 halo slots resident)")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c5-steps", type=int, default=270)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("packed_probe.py measures on a CUDA device; none is visible")
    from lorenzcycletoolkit_b200 import engine as E, synthetic as S
    grid = S.era5_grid()
    n = args.steps
    fields32 = S.synth_fields(grid, n + 2, np.float32, "cuda")
    steps = E.time_stencil(3600.0 * np.arange(n + 2), E.make_steps(n + 2))[1:-1].copy()
    for k, v in BOX.items():
        steps[k] = v
    per_step = {k: 5 * NLON * NLAT * NLEV * b for k, b in (("int16", 2), ("fp32", 4), ("fp64", 8))}
    out = {"gpu": gpu_info(), "c4": {"grid": [NLON, NLAT, NLEV], "box": [BOX["i1"] - BOX["i0"] + 1, BOX["j1"] - BOX["j0"] + 1],
                                      "steps_per_call": n,
                                      "bytes_per_timestep": per_step,
                                      "timesteps_in_180GB": {k: int(180e9 // v) for k, v in per_step.items()}}}
    out["c4"].update(probe_c4(args, fields32, grid, steps))
    del fields32
    torch.cuda.empty_cache()
    out["c5"] = probe_c5(args)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
