"""Sustained A/B of row-kernel variants under the power cap: every variant runs 48-step launches back to back
for `seconds`, the variants are cycled `rounds` times in ONE process (same board, same thermal state), and the mean
kernel time per launch is reported per visit.  bench.py's device line is this measurement for the default variant.
  python scripts/kernel_sustained.py [seconds] [rounds] variant ...      variant = direct | tile"""
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lorenzcycletoolkit_b200 import engine as E, synthetic as S

seconds = float(sys.argv[1]) if len(sys.argv) > 1 else 3.0
rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 2
variants = sys.argv[3:] or ["direct", "tile"]
nsteps = 48
g = S.era5_grid()
f64 = lambda a: np.asarray(a, dtype=np.float64)
fields = S.synth_fields(g, nsteps + 2, np.float32, "cuda:0")
torch.cuda.synchronize()
steps = E.time_stencil(3600.0 * np.arange(nsteps + 2), E.make_steps(nsteps + 2))[1:-1]
steps["i0"], steps["i1"], steps["j0"], steps["j1"] = 0, 1439, 1, 719
B = 5 * 37 * 719 * 1440 * 4
engines = {}
for v in variants:
    os.environ["LEC_ROW_KERNEL"] = v
    engines[v] = E.LecEngine(f64(g["lon"]), f64(g["lat"]), f64(g["rlons"]), f64(g["rlats"]), f64(g["coslats"]), g["level"],
                             np.float32, max_steps=nsteps, max_box_rows=719)
for r in range(rounds):
    for v in variants:
        eng = engines[v]
        for _ in range(3):
            eng.run_torch(fields, steps)
        torch.cuda.synchronize()
        eng.timing_reset()
        n, t0 = 0, time.time()
        while time.time() - t0 < seconds:
            for _ in range(10):
                eng.run_torch(fields, steps)
            torch.cuda.synchronize()
            n += 10
        a, b, c = eng.last_timing()
        print(f"round {r} {v:10s} {n:4d} launches  rows {a / n:7.3f} ms  -> {B * nsteps / (a / n) / 1e6:6.0f} GB/s alg "
              f"({B * nsteps / (a / n) / 1e6 / 6535.7:.3f})", flush=True)
