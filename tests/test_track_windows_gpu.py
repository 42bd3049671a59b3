"""Staging windows of the host paths (``lec_set_host_windows``): with windows on, ``lec_run_host`` and
``lec_run_host_raw`` stage only the union of the boxes that read each slot, and every output -- 16 terms, 19
per-level families, 18 boundary pieces, flags -- keeps the bits of whole-slot staging, while ``last_transfer()[0]``
equals the bytes of ``engine.track_windows``.

Each comparison runs on ONE handle in the order: whole slots on the real fields (the reference), whole slots on
all-NaN fields (the staging buffers now hold NaN everywhere), windows on the real fields.  A window that missed a
value a kernel uses would read a NaN there.  The row-kernel instance is pinned by the environment (LEC_NARROW_G,
LEC_NARROW, LEC_ROW_KERNEL, LEC_COMP): windows fit more slots into the same staging bytes, so the two runs may cut
their kernel batches differently, and a batch chooses its instance from its own boxes."""
import numpy as np
import pytest

import helpers as H
from lorenzcycletoolkit_b200 import engine as E
from test_engine_synthetic_gpu import _dataset

pytestmark = pytest.mark.gpu

FAMILIES = {                      # environment of lec_create -> the row kernel every batch runs
    "tiled": {"LEC_NARROW": "0", "LEC_ROW_KERNEL": "tile"},
    "g4": {"LEC_NARROW_G": "4"},
    "g8": {"LEC_NARROW_G": "8"},
    "g16": {"LEC_NARROW_G": "16"},
    "direct": {"LEC_NARROW": "0", "LEC_ROW_KERNEL": "direct"},
}
EXPECT = {"tiled": ("tiled", 32), "g4": ("subwarp", 4), "g8": ("subwarp", 8), "g16": ("subwarp", 16),
          "direct": ("direct", 32)}
ARITH = {"f32": (np.float32, E.LEC_MATH_AUTO), "f32m64": (np.float32, E.LEC_MATH_F64), "f64": (np.float64, E.LEC_MATH_AUTO)}


@pytest.fixture
def family_env(monkeypatch):
    def set_family(name, comp="0"):
        for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
            monkeypatch.delenv(k, raising=False)
        for k, v in FAMILIES[name].items():
            monkeypatch.setenv(k, v)
        monkeypatch.setenv("LEC_COMP", comp)
    return set_family


def _coords(kind, nlon, nlat):
    if kind == "uniform":               # exactly uniform in fp64 radians too: no longitude tables (LONW 0)
        return (-60.0 + 0.5 * np.arange(nlon), -40.0 + 0.5 * np.arange(nlat)), {"coord_dtype": np.float64}
    if kind == "f32":                   # float32 radians: per-column trapezoid weights (LONW 1)
        return ((-60.0 + 0.25 * np.arange(nlon)).astype(np.float32), (-40.0 + 0.25 * np.arange(nlat)).astype(np.float32)), {}
    rng = np.random.default_rng(3)      # irregular: per-column weights and stencil (LONW 2)
    return (np.cumsum(rng.uniform(0.2, 0.3, nlon)) - 60, np.cumsum(rng.uniform(0.2, 0.3, nlat)) - 40), \
        {"coord_dtype": np.float64}


def _track(P, nt, boxes):
    steps = E.time_stencil(H.tsec_of(P), E.make_steps(nt))
    for it, (i0, i1, j0, j1) in enumerate(boxes):
        steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = i0, i1, j0, j1
    return steps


def _moving(nt, w, h, nlon, nlat, x0=1, y0=2, dx=3, dy=1):
    """Boxes of w x h points moving east-north-east, clamped to the grid."""
    out = []
    for t in range(nt):
        i0, j0 = min(x0 + dx * t, nlon - w), min(y0 + dy * t, nlat - h)
        out.append((i0, i0 + w - 1, j0, j0 + h - 1))
    return out


def _compare(eng, run, nan_run, model, tag):
    """run(): the call under test on ``eng``; nan_run(): the same call on all-NaN fields."""
    eng.set_host_windows(False)
    ref = _with_bnd(eng, run)
    _with_bnd(eng, nan_run)
    eng.set_host_windows(True)
    got = _with_bnd(eng, run)
    eng.set_host_windows(False)
    for n, (a, b) in enumerate(zip(ref, got)):
        assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), (tag, n)
    assert np.isfinite(got[0]).all(), tag
    if model is not None:
        assert eng.last_transfer()[0] == model["h2d_bytes"], (tag, eng.last_transfer()[0], model["h2d_bytes"])
    return got


def _with_bnd(eng, run):
    terms, levels, flags = run(want_boundary=True)
    return terms, levels, flags, eng.last_boundary.copy()


@pytest.mark.parametrize("coords", ["uniform", "f32", "irregular"])
@pytest.mark.parametrize("arith", list(ARITH))
@pytest.mark.parametrize("family", list(FAMILIES))
def test_every_row_kernel_family_keeps_its_bits(family, arith, coords, family_env):
    """Moving boxes through every row-kernel family the host paths can run, in fp32, fp32 with fp64 arithmetic and
    fp64, on uniform, float32-radian and irregular longitudes; boxes start on odd columns and change size."""
    dtype, math = ARITH[arith]
    family_env(family)
    nlon, nlat, nlev, nt = 120, 40, 4, 10
    (lon, lat), kw = _coords(coords, nlon, nlat)
    P, fields = _dataset(nlon, nlat, nlev, nt, dtype, lon=lon, lat=lat, dt_h=1, seed=7, **kw)
    boxes = _moving(nt, 61, 17, nlon, nlat, x0=3, dx=5)
    boxes[4] = (7, 40, 5, 30)                  # one box of another size
    steps = _track(P, nt, boxes)
    nans = [np.full_like(f, np.nan) for f in fields]
    model = E.track_windows(steps, (nlev, nlat, nlon), dtype)
    with H.make_engine(P, dtype, [1.0] * 5, math=math) as eng:
        _compare(eng, lambda **k: eng.run_host(fields, steps, **k), lambda **k: eng.run_host(nans, steps, **k), model,
                 (family, arith, coords))
        d = eng.last_dispatch()
    assert (d["kernel"], d["group"]) == EXPECT[family]
    assert model["h2d_bytes"] < 5 * nt * fields[0][0].nbytes


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_compensated_sums_keep_their_bits(dtype, family_env):
    """The compensated fp32 instances (LEC_COMP=1) of the tiled and sub-warp kernels."""
    nlon, nlat, nlev, nt = 120, 30, 3, 6
    P, fields = _dataset(nlon, nlat, nlev, nt, dtype, dt_h=1, seed=2)
    steps = _track(P, nt, _moving(nt, 70, 9, nlon, nlat, x0=2, dx=7))
    nans = [np.full_like(f, np.nan) for f in fields]
    for fam in ("tiled", "g16"):
        family_env(fam, comp="1")
        with H.make_engine(P, dtype, [1.0] * 5) as eng:
            _compare(eng, lambda **k: eng.run_host(fields, steps, **k), lambda **k: eng.run_host(nans, steps, **k),
                     E.track_windows(steps, (nlev, nlat, nlon), dtype), fam)


def _raw(fields, kind, lon_kind, rng):
    """File-layout records of ``fields``: rows north to south, two extra raw levels, the longitude map ``lon_kind``
    (identity, a crop of a wider raw row, or a wrap whose seam lies inside some windows); ``kind`` = f32 / f64
    records or int16 big-endian records interleaved field by field (NetCDF-3 record variables).  Returns raw arrays,
    maps, decode."""
    nt, nlev, nlat, nlon = fields[0].shape
    rlon = nlon + 9 if lon_kind == "crop" else nlon
    lon_map = {"identity": np.arange(nlon), "crop": np.arange(nlon) + 5,
               "wrap": (np.arange(nlon) + 47) % nlon}[lon_kind].astype(np.int32)
    lat_map = np.arange(nlat - 1, -1, -1, dtype=np.int32)
    lev_map = np.array([2, 0, 3, 1][:nlev] if nlev <= 4 else rng.permutation(nlev + 2)[:nlev], dtype=np.int32)
    nlev_r = nlev + 2
    sel = np.ix_(np.arange(nt), lev_map, lat_map, lon_map)
    if kind == "i16":
        inter = np.zeros((nt, 5, nlev_r, nlat, rlon), dtype=">i2")
        raws, decode = [], []
        for f, a in enumerate(fields):
            lo, hi = float(a.min()), float(a.max())
            scale, offset = (hi - lo) / 60000.0, 0.5 * (hi + lo)
            q = np.clip(np.round((a.astype(np.float64) - offset) / scale), -32000, 32000).astype(np.int16)
            view = inter[:, f]
            view[sel] = q
            raws.append(view)
            decode.append({"scale": scale, "offset": offset, "float32": a.dtype == np.float32})
        return raws, (lon_map, lat_map, lev_map), decode
    raws = []
    for a in fields:
        r = (rng.normal(size=(nt, nlev_r, nlat, rlon)) * 1e3).astype(a.dtype)
        r[sel] = a
        raws.append(r)
    return raws, (lon_map, lat_map, lev_map), None


@pytest.mark.parametrize("lon_kind", ["identity", "crop", "wrap"])
@pytest.mark.parametrize("kind,dtype", [("i16", np.float32), ("i16", np.float64), ("f32", np.float32),
                                        ("f64", np.float64)])
def test_raw_records_keep_their_bits(kind, dtype, lon_kind, family_env):
    """lec_run_host_raw through windows: int16 big-endian interleaved records into both handle types, fp32 and fp64
    records; identity, crop and wrap longitude maps; rows stored north to south.  The bytes follow the model (cropped
    raw columns where the window's raw columns are one run, whole raw rows where the wrap's seam cuts the window)."""
    rng = np.random.default_rng(21)
    nlon, nlat, nlev, nt = 96, 30, 4, 9
    P, fields = _dataset(nlon, nlat, nlev, nt, dtype, dt_h=1, seed=5)
    raws, maps, decode = _raw(fields, kind, lon_kind, rng)
    nan_raws = [np.full_like(r, -32768 if kind == "i16" else np.nan) for r in raws]
    nan_decode = None if decode is None else [dict(d, fills=[-32768]) for d in decode]
    steps = _track(P, nt, _moving(nt, 21, 11, nlon, nlat, x0=0, dx=9, dy=2))
    raw_desc = (*maps, raws[0].shape[-1], raws[0].dtype.itemsize)
    model = E.track_windows(steps, (nlev, nlat, nlon), dtype, raw=raw_desc)
    for fam in ("g8", "tiled"):
        family_env(fam)
        with H.make_engine(P, dtype, [1.0] * 5) as eng:
            rec = np.arange(nt)
            got = _compare(eng, lambda **k: eng.run_host_raw(raws, *maps, rec, steps, decode=decode, **k),
                           lambda **k: eng.run_host_raw(nan_raws, *maps, rec, steps, decode=nan_decode, **k),
                           model, (kind, lon_kind, fam))
            if kind != "i16":                       # the same values as engine-layout arrays, through windows too
                eng.set_host_windows(True)
                host = _with_bnd(eng, lambda **k: eng.run_host(fields, steps, **k))
                for a, b in zip(got, host):
                    assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
                assert eng.last_transfer()[0] == E.track_windows(steps, (nlev, nlat, nlon), dtype)["h2d_bytes"]
    if lon_kind == "wrap":
        assert any(r[1] >= r[0] and (maps[0][r[0]:r[1] + 1] == 0).any() and maps[0][r[0]] != 0 for r in model["t"])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("family", ["g8", "tiled", "direct"])
def test_edges_orders_neighbours_and_chunks(dtype, family, family_env):
    """Boxes on the grid's first and last rows and columns; shuffled, reversed and repeated step lists; time
    neighbours that are not adjacent slots; calls split into several greedy chunks (max_steps and a small staging
    of four steps, T slots handed over device to device); a fixed box with windows on."""
    family_env(family)
    rng = np.random.default_rng(4)
    nlon, nlat, nlev, nt = 75, 26, 3, 14
    P, fields = _dataset(nlon, nlat, nlev, nt, dtype, dt_h=1, seed=9)
    nans = [np.full_like(f, np.nan) for f in fields]
    boxes = _moving(nt, 23, 9, nlon, nlat, x0=0, y0=0, dx=5, dy=2)
    boxes[0], boxes[5], boxes[nt - 1] = (0, 10, 0, 6), (nlon - 12, nlon - 1, nlat - 7, nlat - 1), (0, nlon - 1, 0, nlat - 1)
    base = _track(P, nt, boxes)
    far = base.copy()                                   # neighbours three slots away
    far["slot_m"] = np.maximum(far["slot"] - 3, 0)
    far["slot_p"] = np.minimum(far["slot"] + 2, nt - 1)
    fixed = _track(P, nt, [(4, 60, 3, 20)] * nt)
    lists = {"in order": base, "shuffled": base[rng.permutation(nt)].copy(), "reversed": base[::-1].copy(),
             "repeats": base[np.r_[np.arange(nt), [5, 5, 0, nt - 1, 6]]].copy(), "far neighbours": far,
             "fixed": fixed}
    grid = (nlev, nlat, nlon)
    for name, st in lists.items():
        with H.make_engine(P, dtype, [1.0] * 5) as eng:
            _compare(eng, lambda **k: eng.run_host(fields, st, **k), lambda **k: eng.run_host(nans, st, **k),
                     E.track_windows(st, grid, dtype), name)
        with H.make_engine(P, dtype, [1.0] * 5, max_steps=4) as eng:       # chunks of <= 4 steps
            vecw = 2 if dtype == np.float64 else 4
            elem = np.dtype(dtype).itemsize
            slot_bytes = nlev * nlat * ((nlon + vecw - 1) // vecw * vecw) * elem
            m = E.track_windows(st, grid, dtype, max_steps=4)
            win_bytes = nlev * m["rows"] * m["pitch"] * elem
            # the whole-slot run allocates min(max_steps + 2, nslots) = 6 slots; windows fit more into those bytes
            m = E.track_windows(st, grid, dtype, max_steps=4, stage_slots=6 * slot_bytes // win_bytes)
            _compare(eng, lambda **k: eng.run_host(fields, st, **k), lambda **k: eng.run_host(nans, st, **k), m,
                     name + " / chunks")


def test_default_dispatcher_boxes_of_one_size():
    """The default dispatcher (nothing pinned) on C5-shaped boxes of one size: windows cut batches differently but
    every batch chooses the same instance."""
    nlon, nlat, nlev, nt = 200, 60, 5, 12
    P, fields = _dataset(nlon, nlat, nlev, nt, np.float32, dt_h=1, seed=1)
    steps = _track(P, nt, _moving(nt, 41, 41, nlon, nlat, x0=5, dx=11, dy=1))
    nans = [np.full_like(f, np.nan) for f in fields]
    with H.make_engine(P, np.float32, [1.0] * 5, max_steps=4) as eng:
        _compare(eng, lambda **k: eng.run_host(fields, steps, **k), lambda **k: eng.run_host(nans, steps, **k), None,
                 "default")


def test_windows_switch_and_errors():
    """lec_set_host_windows accepts 0 and 1 only; a box outside the grid is refused before anything is staged."""
    P, fields = _dataset(40, 20, 3, 4, np.float32, dt_h=1)
    steps = _track(P, 4, [(1, 10, 1, 8)] * 4)
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        assert eng._lib.lec_set_host_windows(eng._h, 2) == -1
        eng.set_host_windows(True)
        bad = steps.copy()
        bad["i1"][2] = 40
        with pytest.raises(IndexError):
            eng.run_host(fields, bad)
        bad = steps.copy()
        bad["i1"][1] = bad["i0"][1]
        with pytest.raises(ValueError):
            eng.run_host(fields, bad)
        t, _, _ = eng.run_host(fields, steps)
        assert np.isfinite(t).all()


# --------------------------------------------------------------------------------------- #
# 850-hPa diagnostics on plane windows (lec_diag850_host_windows)
def _diag_planes(rng, nt, nlat, nlon, dtype):
    lon = np.linspace(0, 2 * np.pi, nlon)[None, None, :]
    lat = np.linspace(-1, 1, nlat)[None, :, None]
    t = np.arange(nt)[:, None, None]
    u = 20 * np.cos(2 * lat) + 8 * np.sin(3 * lon + 0.3 * t) + rng.normal(0, 1, (nt, nlat, nlon))
    v = 6 * np.sin(2 * lon - 0.2 * t) * np.cos(lat) + rng.normal(0, 1, (nt, nlat, nlon))
    z = 1500 + 60 * np.cos(lon + 0.1 * t) * np.sin(2 * lat) + rng.normal(0, 2, (nt, nlat, nlon))
    return [np.ascontiguousarray(a, dtype=dtype) for a in (u, v, z)]


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_diag850_windows_have_the_bits_of_whole_planes(dtype):
    """Windows of the planes give the values and flat indices of the whole planes: NaNs (first NaN wins the index,
    values skip them), ties, an all-NaN box, the ``-z`` centre point (inside and outside the box), boxes of 1 and 2
    points on every domain edge and corner, and a window that misses a stencil point is refused."""
    rng = np.random.default_rng(8)
    nlat, nlon = 20, 24
    lon, lat = -60 + 2.5 * np.arange(nlon), -45 + 2.5 * np.arange(nlat)
    boxes = [(2, 15, 4, 12), (2, 15, 2, 12), (3, 20, 1, 18), (4, 7, 6, 9),
             (0, 0, 0, 0), (0, 1, 0, 1), (nlon - 1, nlon - 1, nlat - 1, nlat - 1), (nlon - 2, nlon - 1, nlat - 2, nlat - 1),
             (0, 0, 5, 6), (nlon - 1, nlon - 1, 3, 3), (7, 8, 0, 0), (10, 10, nlat - 1, nlat - 1), (0, nlon - 1, 0, nlat - 1)]
    centres = [(8, 8), (20, 3), (-1, -1), (5, 7), (0, 0), (3, 10), (nlon - 1, nlat - 1), (0, nlat - 1), (1, 5),
               (nlon - 1, 0), (8, 1), (10, nlat - 2), (12, 10)]
    nt = len(boxes)
    u, v, z = _diag_planes(rng, nt, nlat, nlon, dtype)
    z[0, 6, 9] = np.nan; z[0, 8, 3] = np.nan
    u[1, 5, 5] = np.nan
    z[2] = 1234.5
    u[3, 4:12, 2:10] = np.nan; v[3, 4:12, 2:10] = np.nan; z[3, 4:12, 2:10] = np.nan
    steps = E.diag_steps([(t,) + b for t, b in enumerate(boxes)], centres)
    scale, z_div = (1.0, 1.0, 9.80665), 9.80665
    ref = E.diag850_host(u, v, z, lon, lat, steps, scale=scale, z_div=z_div)
    origins, wy, wx = E.diag_windows(steps, nlon, nlat)
    cut = [np.stack([a[t, y0:y0 + wy, x0:x0 + wx] for t, (x0, y0) in enumerate(origins)]) for a in (u, v, z)]
    got = E.diag850_host_windows(*cut, origins, lon, lat, steps, scale=scale, z_div=z_div)
    for a, b in zip(ref, got):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8))
    assert np.isnan(ref[0][3][:4]).all() and ref[1][2, 2] == 0
    # the small boxes alone: small windows (the edge rule's three points), same bits
    small = steps[4:12].copy()
    small["slot"] = np.arange(8)
    small["ic"] = small["jc"] = -1                     # no centre point: the window is the grown box alone
    ref2 = E.diag850_host(*(a[4:12] for a in (u, v, z)), lon, lat, small, scale=scale, z_div=z_div)
    o2, wy2, wx2 = E.diag_windows(small, nlon, nlat)
    assert wy2 <= 4 and wx2 <= 4 and min(wy2, wx2) >= 3
    cut2 = [np.stack([a[4 + t, y0:y0 + wy2, x0:x0 + wx2] for t, (x0, y0) in enumerate(o2)]) for a in (u, v, z)]
    got2 = E.diag850_host_windows(*cut2, o2, lon, lat, small, scale=scale, z_div=z_div)
    for a, b in zip(ref2, got2):
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8), equal_nan=False)
    bad = o2.copy()
    bad[0] += 1                                         # step 0 (box at the corner) now misses column / row 0
    with pytest.raises(IndexError):
        E.diag850_host_windows(*cut2, bad, lon, lat, small)


# --------------------------------------------------------------------------------------- #
# The product route: `cli -t` with windows (the default of the moving framework) against whole slots and planes
_WRAPPER = """import functools, runpy, sys
import lorenzcycletoolkit_b200.cli as cli
cli.lec_moving = functools.partial(cli.lec_moving, engine_options={"host_windows": False})
sys.argv = [sys.argv[0]] + sys.argv[1:]
runpy.run_path(%r, run_name="__main__")
"""


@pytest.mark.parametrize("nproc", [1, 2])
def test_cli_track_writes_the_same_files_with_and_without_windows(tmp_path, nproc):
    """`lorenzcycletoolkit.py testdata_NCEP-R2.nc -r -t` (the moving framework stages windows for the LEC terms and
    the 850-hPa diagnostics) writes byte-identical files to the same run with engine_options={"host_windows":
    False}, in one process and under torchrun with two ranks (each rank windows its own time shard)."""
    import os
    import shutil
    from test_sharded_dropin_gpu import INP, SAM, _cli_run, _tree
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    wrapper = tmp_path / "whole_slots.py"
    wrapper.write_text(_WRAPPER % os.path.join(root, "lorenzcycletoolkit.py"))
    for name in ("windows", "whole"):
        d = tmp_path / name / "inputs"
        os.makedirs(d)
        shutil.copy(os.path.join(INP, "namelist_NCEP-R2"), d / "namelist")
        shutil.copy(os.path.join(INP, "track_testdata_NCEP-R2"), d / "track")
    argv = [os.path.join(SAM, "testdata_NCEP-R2.nc"), "-r", "-t"]
    _cli_run(str(tmp_path / "windows"), argv, nproc)
    import subprocess
    import sys
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, str(wrapper)] + argv, cwd=str(tmp_path / "whole"), env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    a, b = _tree(tmp_path / "windows" / "LEC_Results"), _tree(tmp_path / "whole" / "LEC_Results")
    assert sorted(a) == sorted(b) and len(a) >= 22
    for k in a:
        assert a[k] == b[k], k


def test_moving_framework_windows_by_default_and_on_request_off(monkeypatch):
    """BoxBatch turns windows on (engine_options={"host_windows": False} turns them off); BoxData (fixed boxes)
    keeps whole slots."""
    from lorenzcycletoolkit_b200.utils import box_data as B
    seen = []
    orig = E.LecEngine.set_host_windows
    monkeypatch.setattr(E.LecEngine, "set_host_windows", lambda self, on: (seen.append(bool(on)), orig(self, on))[1])
    P, fields = _dataset(40, 20, 3, 4, np.float32, dt_h=1)
    steps = _track(P, 4, [(1, 10, 1, 8)] * 4)
    for opts, want in (({"host_windows": True}, True), ({}, False)):
        seen.clear()
        B.run_time_sharded(P, np.float32, [1.0] * 5, fields, steps, 8, opts)
        assert seen == [want]
