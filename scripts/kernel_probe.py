"""Row-kernel A/B on C4-shaped data: every variant named on the command line is run on the same resident
fields, timed with the engine's own CUDA events (isolated launches) and compared bit for bit with the first one.
  python scripts/kernel_probe.py [nsteps] [dtype f32|f64] variant ...     variant = direct | tile[:band[:comp]] (direct::1 = direct kernel with compensation)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lorenzcycletoolkit_b200 import engine as E, synthetic as S

nsteps = int(sys.argv[1]) if len(sys.argv) > 1 else 24
dt = np.float64 if (len(sys.argv) > 2 and sys.argv[2] == "f64") else np.float32
variants = sys.argv[3:] or ["direct", "tile"]
g = S.era5_grid()
f64 = lambda a: np.asarray(a, dtype=np.float64)
fields = S.synth_fields(g, nsteps + 2, dt, "cuda:0")
torch.cuda.synchronize()
steps = E.time_stencil(3600.0 * np.arange(nsteps + 2), E.make_steps(nsteps + 2))[1:-1]
steps["i0"], steps["i1"], steps["j0"], steps["j1"] = 0, 1439, 1, 719
B = 5 * 37 * 719 * 1440 * np.dtype(dt).itemsize
ref = None
for v in variants:
    parts = v.split(":")
    os.environ["LEC_ROW_KERNEL"] = parts[0]
    band = int(parts[1]) if len(parts) > 1 and parts[1] else 0
    os.environ["LEC_COMP"] = parts[2] if len(parts) > 2 else "0"                      # compensated fp32 linear sums on / off
    eng = E.LecEngine(f64(g["lon"]), f64(g["lat"]), f64(g["rlons"]), f64(g["rlats"]), f64(g["coslats"]), g["level"],
                      dt, max_steps=nsteps, max_box_rows=719, band_rows=band)
    best = 1e9
    for it in range(5):
        terms, levels, flags = eng.run_torch(fields, steps)
        torch.cuda.synchronize()
        a, b, c = eng.last_timing()
        best = min(best, a)
    out = (terms.cpu().numpy(), levels.cpu().numpy())
    same = "ref" if ref is None else ("bit-identical" if all(np.array_equal(x, y, equal_nan=True) for x, y in zip(out, ref))
                                        else f"DIFFERS max rel {max(np.max(np.abs(x - y) / (np.abs(y) + 1e-300)) for x, y in zip(out, ref)):.3e}")
    if ref is None:
        ref = out
    print(f"{v:14s} rows {best:8.3f} ms (last {a:.3f})  fin {b:.3f} ms  -> {B * nsteps / best / 1e6:7.0f} GB/s alg "
          f"({B * nsteps / best / 1e6 / 6535.7:.3f} of 6535.7)  flags {int(flags.max().item())}  {same}", flush=True)
    eng.close()
