"""``bench.py --dump-outputs``: the gather buffer of the timed pass is split into the arrays a caller receives."""
import numpy as np
import torch

import bench
from lorenzcycletoolkit_b200 import engine as E


def test_dump_outputs_splits_the_gather_buffer(tmp_path):
    chunk = 5
    nt, nl = chunk * E.NTERMS, chunk * E.NLEVEL_TERMS * bench.NLEV
    g_res = torch.arange(nt + nl, dtype=torch.float64)
    flags = torch.tensor([0, 1, 0, 2, 0], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path / "out"), g_res, flags, chunk, 0, 1, "cpu")
    terms, levels, fl = (np.load(tmp_path / "out" / f"{n}.npy") for n in ("terms", "levels", "flags"))
    assert terms.dtype == levels.dtype == fl.dtype == np.float64
    assert terms.shape == (chunk, E.NTERMS) and levels.shape == (chunk, E.NLEVEL_TERMS, bench.NLEV)
    assert np.array_equal(terms.ravel(), np.arange(nt)) and np.array_equal(levels.ravel(), np.arange(nt, nt + nl))
    assert np.array_equal(fl, [0, 1, 0, 2, 0])
