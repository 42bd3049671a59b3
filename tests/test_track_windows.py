"""CPU tests of the staging-window model ``engine.track_windows`` (the rule of ``lec_set_host_windows`` in
include/lec_b200.h) and of the new C symbol.  The GPU side, bits and measured bytes: test_track_windows_gpu.py."""
import ctypes
import os
import re

import numpy as np
import pytest

from lorenzcycletoolkit_b200 import engine as E

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _steps(boxes, slots=None):
    st = E.make_steps(len(boxes))
    n = len(boxes)
    idx = np.arange(n) if slots is None else np.asarray(slots)
    st["slot"], st["slot_m"], st["slot_p"] = idx, np.maximum(idx - 1, 0), np.minimum(idx + 1, n - 1)
    for k, (i0, i1, j0, j1) in enumerate(boxes):
        st["i0"][k], st["i1"][k], st["j0"][k], st["j1"][k] = i0, i1, j0, j1
    return st


def test_windows_are_unions_of_the_reading_boxes():
    boxes = [(5, 20, 3, 10), (9, 25, 4, 12), (13, 30, 6, 14)]
    m = E.track_windows(_steps(boxes), (2, 40, 50), np.float32)
    # T: slot 0 is read by steps 0 (centre) and 1 (slot_m); slot 1 by all three; slot 2 by steps 1 and 2
    assert m["t"].tolist() == [[4, 25, 3, 12], [4, 30, 3, 14], [8, 30, 4, 14]]
    # u, v, omega, Phi: the centre box alone, column origin rounded down to 4 (fp32)
    assert m["c"].tolist() == [[4, 20, 3, 10], [8, 25, 4, 12], [12, 30, 6, 14]]
    assert m["rows"] == 12 and m["pitch"] == 28           # slot 1: 27 columns -> 7 chunks of 4
    elem, L = 4, 2
    t_bytes = sum(L * (r[3] - r[2] + 1) * (r[1] - r[0] + 1) * elem for r in m["t"])
    c_bytes = sum(L * (r[3] - r[2] + 1) * (r[1] - r[0] + 1) * elem for r in m["c"])
    assert m["h2d_bytes"] == t_bytes + 4 * c_bytes
    m64 = E.track_windows(_steps(boxes), (2, 40, 50), np.float64)
    assert m64["c"][:, 0].tolist() == [4, 8, 12] and m64["t"][2, 0] == 8
    assert E.track_windows(_steps([(5, 20, 3, 10)] * 3), (2, 40, 50), np.float64)["c"][0, 0] == 4


def test_slots_no_step_reads_cost_nothing():
    st = _steps([(0, 9, 0, 9), (0, 9, 0, 9)], slots=[0, 5])
    st["slot_m"], st["slot_p"] = [0, 4], [1, 6]
    m = E.track_windows(st, (3, 10, 10), np.float32, nslots=8)
    assert [int(r[1] >= r[0]) for r in m["t"]] == [1, 1, 0, 0, 1, 1, 1, 0]
    one = 3 * 10 * 10 * 4
    # one chunk covering slots 0..6: T at the five slots some step reads, u.. at the two centres
    assert m["h2d_bytes"] == 5 * one + 4 * 2 * one


def test_raw_columns_cropped_when_one_run_else_whole_rows():
    boxes = [(2, 7, 1, 4)] * 2
    lev_map = np.array([3, 1, 2])                      # touched raw levels 1..3
    lat_map = np.arange(9, -1, -1)                     # north to south: rows 1..4 -> raw rows 5..8
    ident = (np.arange(12), lat_map, lev_map, 12, 2)
    m = E.track_windows(_steps(boxes), (3, 10, 12), np.float32, raw=ident)
    # x0 = 0 (rounded), 8 columns; 4 raw rows; 3 raw levels; int16
    per = 3 * 4 * 8 * 2
    assert m["h2d_bytes"] == 2 * per + 4 * 2 * per
    wrap = ((np.arange(12) + 5) % 12, lat_map, lev_map, 12, 2)     # raw columns 5..11, 0: the seam inside
    per_w = 3 * 4 * 12 * 2
    assert E.track_windows(_steps(boxes), (3, 10, 12), np.float32, raw=wrap)["h2d_bytes"] == 2 * per_w + 8 * per_w
    crop = (np.arange(12) + 3, lat_map, lev_map, 20, 4)            # fp32 records, rows of 20 raw columns
    assert E.track_windows(_steps(boxes), (3, 10, 12), np.float32, raw=crop)["h2d_bytes"] == 10 * 3 * 4 * 8 * 4


def test_chunk_replay_hands_t_over_between_chunks():
    """max_steps = 2: chunks {0, 1} (slots 0..2) and {2, 3} (slots 1..3): T slots 1 and 2 come from the first chunk's
    buffer, so only slot 3 crosses again; u.. cross at every chunk's centre range."""
    boxes = [(0, 3, 0, 3)] * 4
    m = E.track_windows(_steps(boxes), (1, 4, 4), np.float32, max_steps=2)
    one = 4 * 4 * 4
    assert m["h2d_bytes"] == (3 + 1) * one + 4 * (2 + 2) * one
    with pytest.raises(MemoryError):
        E.track_windows(_steps(boxes), (1, 4, 4), np.float32, stage_slots=2)


def test_track_windows_is_smaller_than_the_domain_on_a_c5_segment():
    """bench.py's c5 segment shape: 270 steps of 151 x 151 boxes over 436 x 298 x 55 (a straight track here)."""
    n, nlon, nlat = 270, 436, 298
    boxes = [(min(i, nlon - 151), min(i, nlon - 151) + 150, min(i // 2, nlat - 151), min(i // 2, nlat - 151) + 150)
             for i in range(n)]
    m = E.track_windows(_steps(boxes), (55, nlat, nlon), np.float32)
    whole = 5 * n * 55 * nlat * nlon * 4
    assert 4 < whole / m["h2d_bytes"] < 6
    assert m["rows"] == 152 and m["pitch"] == 156


def test_library_exports_lec_set_host_windows():
    import __graft_entry__ as G
    G.build()
    hdr = open(os.path.join(ROOT, "include", "lec_b200.h")).read()
    assert re.search(r"int lec_set_host_windows\(lec_handle \*h, int32_t on\);", hdr)
    lib = ctypes.CDLL(str(E.library_path()))
    assert hasattr(lib, "lec_set_host_windows")
    E.load_library()
    assert lib.lec_set_host_windows(None, 1) != 0          # no handle: LEC_ERR_INVALID


@pytest.mark.parametrize("case", ["ncep_track", "era5_packed"])
def test_level_plane_windows_equals_level_plane_slices(case, tmp_path, monkeypatch):
    """The plane-window gather of the 850-hPa diagnostics, raw-backed (decodes only the window points) and eager:
    the same values as slices of ``level_plane``, and the windows the engine's rule gives for a track."""
    import helpers as H
    from lorenzcycletoolkit_b200.utils import preprocessing as PP
    from test_preprocessing import INP, SAM, _args
    if case == "ncep_track":
        a = _args(track=True, trackfile=os.path.join(INP, "track_testdata_NCEP-R2"))
        nml = os.path.join(INP, "namelist_NCEP-R2")
    else:
        nc = str(tmp_path / "testdata_ERA5.nc")
        H.write_era5_like(nc, True, 160)
        a = _args(infile=nc, track=True, trackfile=os.path.join(INP, "track_testdata_ERA5"))
        nml = os.path.join(INP, "namelist_ERA5")
    lazy = PP.prepare_data(a, nml)
    monkeypatch.setenv("LEC_DEVICE_INGEST", "0")
    eager = PP.prepare_data(a, nml)
    assert lazy.raw is not None and eager.raw is None
    nt, nlat, nlon = len(lazy.time), len(lazy.lat), len(lazy.lon)
    rng = np.random.default_rng(1)
    boxes = [(t, int(x), int(x) + 2, int(y), int(y) + 1) for t, x, y in
             zip(range(nt), rng.integers(0, nlon - 3, nt), rng.integers(0, nlat - 2, nt))]
    boxes[0] = (0, 0, 0, 0, 0)
    boxes[-1] = (nt - 1, nlon - 1, nlon - 1, nlat - 1, nlat - 1)
    origins, rows, cols = E.diag_windows(E.diag_steps(boxes), nlon, nlat)
    assert (rows, cols) == (4, 5)
    for var in list(lazy.raw.fields)[:3]:
        k = len(lazy.level) // 2
        full = eager.level_plane(var, k)
        want = np.stack([full[t, y0:y0 + rows, x0:x0 + cols] for t, (x0, y0) in enumerate(origins)])
        for ds in (lazy, eager):
            got = ds.level_plane_windows(var, k, origins, rows, cols)
            assert got.dtype == want.dtype and np.array_equal(got, want, equal_nan=True), (case, var)
        sub = lazy.level_plane_windows(var, k, origins[2:4], rows, cols, times=[2, 3])
        assert np.array_equal(sub, want[2:4], equal_nan=True)
