"""GPU parity on synthetic datasets: the cases the bundled files cannot reach -- boxes that are
not 16-byte aligned, row lengths that defeat the 128-bit path, non-uniform axes, unit factors,
per-step boxes of different sizes, NaN / sigma-floor flags, error codes, bit-reproducibility and
time-shard invariance.  Same gates as test_engine_parity_gpu.py."""
import numpy as np
import pandas as pd
import pytest

from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E
import helpers as H

pytestmark = pytest.mark.gpu
TOL64, TOL32 = 1e-9, 1e-5
T0 = np.datetime64("2020-01-01T00")


def _dataset(nlon, nlat, nlev, nt, dtype, seed=0, lon=None, lat=None, level=None, dt_h=6, **kw):
    lon = np.linspace(-60, -60 + 2.5 * (nlon - 1), nlon) if lon is None else lon
    lat = np.linspace(-50, -50 + 2.5 * (nlat - 1), nlat) if lat is None else lat
    level = np.linspace(1e4, 1e5, nlev) if level is None else level
    time = T0 + np.arange(nt) * np.timedelta64(dt_h, "h")
    fields = H.smooth_fields(nt, nlev, nlat, nlon, dtype, seed, level=level, lat=lat)
    return H.prepared_from_arrays(fields, lon, lat, level, time, **kw), fields


def _run_fixed(P, fields, box, dtype, scale=None, **kw):
    with H.make_engine(P, dtype, scale or [1.0] * 5, **kw) as eng:
        return eng.run_host(fields, H.fixed_steps(P, *box))


def _check(terms, levels, df, lv, extra, tol):
    errs = H.compare_terms(terms, df, extra=extra)
    assert set(errs) == set(E.TERM_NAMES)
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, bad
    lerrs = H.compare_levels(levels, lv)
    bad = {k: v for k, v in lerrs.items() if not v <= tol}
    assert not bad, bad


# lec_run_host pads every row to whole 128-bit chunks, so all three widths take the vector kernels: what varies is the
# alignment of the box within its chunks, not of the rows (rows that are not 16-byte aligned, and with them the scalar
# kernel, only exist in caller-owned device fields: tests/test_dispatch_matrix_gpu.py)
@pytest.mark.parametrize("nlon", [48, 50, 37])
@pytest.mark.parametrize("dtype,tol", [(np.float64, TOL64), (np.float32, TOL32)])
def test_unaligned_boxes(nlon, dtype, tol):
    P, fields = _dataset(nlon, 21, 7, 5, dtype)
    for box in [(-57.5, 0.0, -45.0, -10.0), (-52.6, -20.1, -41.0, -22.0), (P.lon[3], P.lon[-1], P.lat[0], P.lat[-1]),
                (P.lon[1], P.lon[2], P.lat[5], P.lat[6])]:                       # incl. a 2x2 box
        df, lv, extra = O.lec_fixed(P, *box, mode="fp64")
        terms, levels, flags = _run_fixed(P, fields, box, dtype)
        assert not flags.any()
        _check(terms, levels, df, lv, extra, tol)


def test_wide_rows_cross_several_sweeps():
    """Rows longer than one 32-lane sweep (interior iterations) with an odd start column."""
    P, fields = _dataset(300, 9, 4, 4, np.float32, lon=np.linspace(-170, -170 + 1.0 * 299, 300),
                         lat=np.linspace(-20, 20, 9))
    box = (P.lon[5], P.lon[290], P.lat[1], P.lat[7])
    df, lv, extra = O.lec_fixed(P, *box, mode="fp64")
    terms, levels, _ = _run_fixed(P, fields, box, np.float32)
    _check(terms, levels, df, lv, extra, TOL32)
    terms, levels, _ = _run_fixed(P, [f.astype(np.float64) for f in fields], box, np.float64)
    df, lv, extra = O.lec_fixed(H.prepared_from_arrays([f.astype(np.float64) for f in fields], P.lon, P.lat, P.level, P.time),
                                *box, mode="fp64")
    _check(terms, levels, df, lv, extra, TOL64)


def test_non_uniform_axes_fp64():
    """Irregular longitudes, latitudes, levels and time steps: np.gradient's non-uniform branch on
    every axis, per-column longitude tables in the kernel."""
    rng = np.random.default_rng(3)
    lon = np.cumsum(rng.uniform(0.8, 1.6, 40)) - 70
    lat = np.cumsum(rng.uniform(0.8, 1.6, 17)) - 40
    level = np.array([1e3, 2e3, 5e3, 1e4, 2e4, 3e4, 5e4, 7e4, 8.5e4, 1e5])
    P, fields = _dataset(40, 17, 10, 6, np.float64, lon=lon, lat=lat, level=level, coord_dtype=np.float64)
    P.time = T0 + np.array([0, 3, 6, 12, 15, 24]) * np.timedelta64(1, "h")
    box = (lon[2], lon[37], lat[1], lat[15])
    df, lv, extra = O.lec_fixed(P, *box, mode="fp64")
    terms, levels, _ = _run_fixed(P, fields, box, np.float64)
    _check(terms, levels, df, lv, extra, TOL64)


def test_unit_factors_hpa_per_s_and_geopotential_height():
    """Namelist units other than SI (box_data.py:297-310) and geopotential height x g (:233-241)."""
    P, fields = _dataset(24, 11, 6, 4, np.float32)
    fields[3] = (fields[3] / 100).astype(np.float32)                  # omega in hPa/s
    fields[4] = (fields[4] / O.g).astype(np.float32)                  # geopotential height in m
    names = H.NAMES[:4] + ["Geopotential Height"]
    P = H.prepared_from_arrays(fields, P.lon, P.lat, P.level, P.time, units=("K", "m/s", "m/s", "hPa/s", "m"), names=names)
    box = (P.lon[2], P.lon[20], P.lat[1], P.lat[9])
    df, lv, extra = O.lec_fixed(P, *box, mode="fp64")
    terms, levels, _ = _run_fixed(P, fields, box, np.float32, scale=[1, 1, 1, 100.0, O.g])
    _check(terms, levels, df, lv, extra, TOL32)


def test_moving_boxes_of_different_sizes():
    P, fields = _dataset(64, 41, 6, 7, np.float64, lon=np.linspace(-80, -80 + 63 * 0.5, 64), lat=np.linspace(-40, -20, 41))
    times = pd.to_datetime(P.time)
    track = pd.DataFrame({"Lat": np.linspace(-33, -27, 7), "Lon": np.linspace(-70, -60, 7),
                          "length": [6, 7, 8, 9, 10, 8, 6], "width": [8, 9, 10, 12, 14, 10, 8]}, index=times)
    df, lv, boxes = O.lec_moving(P, track, mode="fp64")
    steps = H.moving_steps(P, track)
    for it, (_, idx) in enumerate(boxes):
        assert (steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it]) == idx
    rows = int((steps["j1"] - steps["j0"]).max() + 1)
    with H.make_engine(P, np.float64, [1.0] * 5, max_box_rows=rows) as eng:
        terms, levels, flags = eng.run_host(fields, steps)
    errs = H.compare_terms(terms, df)
    bad = {k: v for k, v in errs.items() if not v <= TOL64}
    assert not bad, bad
    lerrs = H.compare_levels(levels, lv)
    bad = {k: v for k, v in lerrs.items() if not v <= TOL64}
    assert not bad, bad


@pytest.mark.parametrize("dtype,tol", [(np.float64, TOL64), (np.float32, TOL32)])
def test_c5_shaped_track_boxes(dtype, tol):
    """BASELINE.json configs[4] shape at a size the oracle finishes in seconds: 0.1 deg grid, 15 x 15 deg
    = 151 x 151 point boxes that move every step (38 chunks of 128 bits: five sweeps of the 8-lane row
    groups, odd start columns, boxes touching neither / either domain edge)."""
    nlon, nlat = 260, 232
    lon = (-70.0 + 0.1 * np.arange(nlon)).astype(np.float32)
    lat = (-42.0 + 0.1 * np.arange(nlat)).astype(np.float32)
    P, fields = _dataset(nlon, nlat, 7, 5, dtype, lon=lon, lat=lat, dt_h=1, seed=21)
    times = pd.to_datetime(P.time)
    track = pd.DataFrame({"Lat": [-34.4, -33.9, -33.1, -31.0, -26.5], "Lon": [-62.45, -61.3, -59.0, -55.2, -51.6]},
                         index=times)
    df, lv, boxes = O.lec_moving(P, track, mode="fp64")
    steps = H.moving_steps(P, track)
    assert all(steps["i1"] - steps["i0"] == 150) and all(steps["j1"] - steps["j0"] == 150)
    assert steps["j0"][0] == 1 and steps["i0"][0] % 4 != 0 and steps["i1"][-1] == nlon - 1
    scale = [1.0] * 5
    with H.make_engine(P, dtype, scale, max_box_rows=151) as eng:
        terms, levels, flags = eng.run_host(fields, steps)
    assert not flags.any()
    errs = H.compare_terms(terms, df)
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, bad
    lerrs = H.compare_levels(levels, lv)
    bad = {k: v for k, v in lerrs.items() if not v <= tol}
    assert not bad, bad


def test_nan_and_sigma_floor_flags():
    P, fields = _dataset(24, 11, 6, 4, np.float64)
    box = (P.lon[2], P.lon[20], P.lat[1], P.lat[9])
    # (1) a missing value inside the box at step 2 only: that step (and its time neighbours through
    # dT/dt) is flagged, values outside the box never leak
    f2 = [f.copy() for f in fields]
    f2[1][2, 3, 5, 10] = np.nan
    f2[0][:, :, 0, 0] = np.nan                                          # outside the box
    terms, levels, flags = _run_fixed(P, f2, box, np.float64)
    assert flags[2] & E.FLAG_NONFINITE and not flags[0] & E.FLAG_NONFINITE
    assert np.isfinite(terms[0]).all() and np.isnan(terms[2]).any()
    # (2) neutral stratification at one level -> sigma <= 0.03 is floored exactly as thermodynamics.py:69
    f3 = [f.copy() for f in fields]
    x = (P.level / 1e5)[None, :, None, None]
    f3[0] = np.ascontiguousarray(np.broadcast_to(280.0 * x ** (2.0 / 7.0), f3[0].shape) + 0.01 * (f3[0] - 280.0))
    P3 = H.prepared_from_arrays(f3, P.lon, P.lat, P.level, P.time)
    df, lv, extra = O.lec_fixed(P3, *box, mode="fp64")
    assert (extra["box"].sigma_AA == 0.03).any()
    terms, levels, flags = _run_fixed(P3, f3, box, np.float64)
    assert (flags & E.FLAG_SIGMA_FLOOR).all()
    _check(terms, levels, df, lv, extra, 1e-8)


def test_error_codes():
    P, fields = _dataset(24, 11, 6, 4, np.float32)
    steps = H.fixed_steps(P, P.lon[2], P.lon[20], P.lat[1], P.lat[9])
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        bad = steps.copy(); bad["i1"] = bad["i0"]
        with pytest.raises(ValueError, match="fewer than 2"):
            eng.run_host(fields, bad)
        bad = steps.copy(); bad["j1"] = 99
        with pytest.raises(IndexError):
            eng.run_host(fields, bad)
        bad = steps.copy(); bad["slot_p"] = 7
        with pytest.raises(IndexError):
            eng.run_host(fields, bad)
        with pytest.raises(ValueError, match="engine dtype"):
            eng.run_host([f.astype(np.float64) for f in fields], steps)
        terms, _, _ = eng.run_host(fields, steps)                         # the handle survives errors
        assert np.isfinite(terms).all()
        # an empty step list is not an error: nothing launched, empty results (host and device API)
        import torch
        n0 = eng.launch_count
        t0, l0, f0 = eng.run_host(fields, steps[:0])
        assert t0.shape == (0, E.NTERMS) and l0.shape == (0, E.NLEVEL_TERMS, 6) and f0.shape == (0,)
        td, ld, fd = eng.run_torch([torch.from_numpy(f).cuda() for f in fields], steps[:0])
        torch.cuda.synchronize()
        assert td.shape == (0, E.NTERMS) and eng.launch_count == n0


def test_bit_reproducible_and_time_shard_invariant():
    """Same bits on every run, with a different kernel batching (max_steps) and when the time axis is
    split into shards that carry a one-slot halo (what sharding.py / bench.py do across GPUs)."""
    from lorenzcycletoolkit_b200 import sharding as S
    P, fields = _dataset(96, 21, 8, 9, np.float32)
    box = (P.lon[1], P.lon[90], P.lat[1], P.lat[19])
    gsteps = H.fixed_steps(P, *box)
    a = _run_fixed(P, fields, box, np.float32)
    b = _run_fixed(P, fields, box, np.float32, max_steps=2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    parts_t, parts_l = [], []
    shards = S.time_shards(len(gsteps), 3)
    for (s0, s1) in shards:
        lo, hi = S.shard_slots(s0, s1, len(gsteps))
        local = S.shard_steps(gsteps, s0, s1, lo)
        with H.make_engine(P, np.float32, [1.0] * 5) as eng:
            t, l, _ = eng.run_host([np.ascontiguousarray(f[lo:hi]) for f in fields], local)
        parts_t.append(t); parts_l.append(l)
    assert np.array_equal(np.concatenate(parts_t), a[0]) and np.array_equal(np.concatenate(parts_l), a[1])


def test_staged_chunks_cross_pcie_once():
    """lec_run_host in several staged chunks: results have the bits of the one-chunk call, and every
    field slot crosses PCIe once (T of a slot two chunks share is copied device-to-device; u, v, omega,
    Phi are not uploaded for slots that are only time neighbours)."""
    P, fields = _dataset(40, 17, 6, 11, np.float32)
    steps = H.fixed_steps(P, P.lon[1], P.lon[37], P.lat[1], P.lat[15])
    slot_bytes = fields[0][0].nbytes
    with H.make_engine(P, np.float32, [1.0] * 5, max_steps=64) as eng:
        a = eng.run_host(fields, steps)
        assert eng.last_transfer() == (5 * 11 * slot_bytes, a[0].nbytes + a[1].nbytes + a[2].nbytes)
    with H.make_engine(P, np.float32, [1.0] * 5, max_steps=3) as eng:
        b = eng.run_host(fields, steps)
        assert eng.last_transfer()[0] == 5 * 11 * slot_bytes
    with H.make_engine(P, np.float32, [1.0] * 5, host_stage_bytes=2 * 5 * 4 * slot_bytes) as eng:   # 4-slot windows
        c = eng.run_host(fields, steps)
        assert eng.last_transfer()[0] == 5 * 11 * slot_bytes
    for x in (b, c):
        assert np.array_equal(a[0], x[0]) and np.array_equal(a[1], x[1]) and np.array_equal(a[2], x[2])
    # an interior window: the two halo slots bring T only
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        d = eng.run_host(fields, steps[3:7])
        assert eng.last_transfer()[0] == (5 * 4 + 2) * slot_bytes
    assert np.array_equal(d[0], a[0][3:7]) and np.array_equal(d[1], a[1][3:7])


def test_device_api_matches_host_api():
    import torch
    P, fields = _dataset(48, 21, 7, 5, np.float32)
    box = (P.lon[2], P.lon[40], P.lat[1], P.lat[19])
    steps = H.fixed_steps(P, *box)
    ht, hl, hf = _run_fixed(P, fields, box, np.float32)
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        dev = [torch.from_numpy(f).cuda() for f in fields]
        t, l, f = eng.run_torch(dev, steps)
        torch.cuda.synchronize()
        assert eng.launch_count == 4
        rows_ms, fin_ms, call_ms = eng.last_timing()
        assert rows_ms > 0 and fin_ms > 0 and call_ms >= rows_ms
    assert np.array_equal(t.cpu().numpy(), ht) and np.array_equal(l.cpu().numpy(), hl)


def test_torch_extension_route_equals_ctypes_route(monkeypatch):
    """``run_torch`` goes through ``torch.ops.lec_b200.run_device`` (csrc/lec_torch_ext.cpp) when the extension is
    built, through ctypes otherwise: same library call, same bits, same exceptions; the operator runs on torch's
    CURRENT stream and writes into caller-provided tensors."""
    import torch
    P, fields = _dataset(48, 21, 7, 5, np.float32)
    steps = H.fixed_steps(P, P.lon[2], P.lon[40], P.lat[1], P.lat[19])
    dev = [torch.from_numpy(f).cuda() for f in fields]
    out = {}
    for route in ("ext", "ctypes"):
        monkeypatch.setattr(E, "_torch_ext", None if route == "ext" else False)
        with H.make_engine(P, np.float32, [1.0] * 5) as eng:
            assert E.load_torch_extension() == (route == "ext")
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                n = len(steps)
                pre = (torch.full((n, E.NTERMS), -1.0, dtype=torch.float64, device="cuda"),
                       torch.empty((n, E.NLEVEL_TERMS, 7), dtype=torch.float64, device="cuda"),
                       torch.ones(n, dtype=torch.int32, device="cuda"))
                t, l, f = eng.run_torch(dev, steps, out=pre)
                assert t is pre[0] and eng.launch_count == 4
            side.synchronize()
            out[route] = (t.cpu().numpy(), l.cpu().numpy(), f.cpu().numpy())
            bad = steps.copy()
            bad["i1"] = 48                          # outside the grid
            with pytest.raises(IndexError):
                eng.run_torch(dev, bad)
    monkeypatch.setattr(E, "_torch_ext", None)
    for a, b in zip(out["ext"], out["ctypes"]):
        assert np.array_equal(a, b)
    assert np.isfinite(out["ext"][0]).all() and not out["ext"][2].any()


@pytest.mark.parametrize("seed", range(12))
def test_random_configurations(seed):
    """Seeded random grids, boxes and series lengths down to the degenerate minima the reference
    accepts (2 levels, 2 time steps, 2 x 2 boxes), fp32 and fp64, uniform and irregular axes."""
    rng = np.random.default_rng(1000 + seed)
    nlon, nlat = int(rng.integers(6, 70)), int(rng.integers(5, 30))
    nlev, nt = int(rng.integers(2, 12)), int(rng.integers(2, 7))
    dtype = np.float64 if seed % 2 else np.float32
    if rng.random() < 0.5:
        lon = np.cumsum(rng.uniform(0.5, 2.0, nlon)) - 100
        lat = np.cumsum(rng.uniform(0.5, 2.0, nlat)) - 60
        level = np.sort(rng.uniform(1e3, 1e5, nlev))
        level[-1] = 1e5
        cd = np.float64
    else:
        step = float(rng.choice([0.25, 0.5, 1.0, 2.5]))
        lon = -120 + step * np.arange(nlon)
        lat = -45 + step * np.arange(nlat)
        level = np.linspace(1e4, 1e5, nlev)
        cd = np.float32
    P, fields = _dataset(nlon, nlat, nlev, nt, dtype, seed=seed, lon=lon, lat=lat, level=level, coord_dtype=cd)
    i0 = int(rng.integers(0, nlon - 1)); i1 = int(rng.integers(i0 + 1, nlon))
    j0 = int(rng.integers(0, nlat - 1)); j1 = int(rng.integers(j0 + 1, nlat))
    box = (float(P.lon[i0]), float(P.lon[i1]), float(P.lat[j0]), float(P.lat[j1]))
    df, lv, extra = O.lec_fixed(P, *box, mode="fp64")
    terms, levels, flags = _run_fixed(P, fields, box, dtype)
    assert not (flags & E.FLAG_NONFINITE).any()
    _check(terms, levels, df, lv, extra, TOL64 if dtype == np.float64 else TOL32)



@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("coords", ["f32", "irregular"])
def test_tiled_kernel_has_the_bits_of_the_direct_kernel(dtype, coords, monkeypatch):
    """The TMA-tiled row kernel sweeps a row with the same lane <-> column mapping, accumulation order and
    butterfly as the direct-load kernel, so terms and per-level integrands must be IDENTICAL -- on rows of
    several sweep iterations, an odd start column, a box height that is no multiple of the tile height, boxes
    that touch the grid edges (TMA out-of-bounds fill) and per-step boxes of different sizes, NaNs outside and
    inside the box included."""
    nlon, nlat, nlev, nt = 700, 61, 5, 6
    if coords == "f32":
        lon = (-150.0 + 0.25 * np.arange(nlon)).astype(np.float32)          # float32 radians: per-column weights
        lat = (-7.0 + 0.25 * np.arange(nlat)).astype(np.float32)
        kw = {}
    else:
        rng = np.random.default_rng(5)
        lon = np.cumsum(rng.uniform(0.2, 0.3, nlon)) - 100
        lat = np.cumsum(rng.uniform(0.2, 0.3, nlat)) - 8
        kw = {"coord_dtype": np.float64}
    P, fields = _dataset(nlon, nlat, nlev, nt, dtype, lon=lon, lat=lat, dt_h=1, seed=11, **kw)
    fields[0][2, 1, 3, 5] = np.nan           # inside some boxes
    fields[1][:, :, 0, :] = np.nan           # first grid row: outside every box below except the full-height one
    steps = E.time_stencil(H.tsec_of(P), E.make_steps(nt))
    boxes = [(5, 690, 1, 59), (0, 699, 1, 60), (3, 699, 7, 40), (130, 640, 2, 3), (1, 517, 1, 60), (0, 699, 0, 60)]
    for it, (i0, i1, j0, j1) in enumerate(boxes):
        steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = i0, i1, j0, j1
    out = {}
    for kernel in ("direct", "tile"):
        monkeypatch.setenv("LEC_ROW_KERNEL", kernel)
        monkeypatch.setenv("LEC_NARROW", "0")
        with H.make_engine(P, dtype, [1.0] * 5) as eng:
            out[kernel] = eng.run_host(fields, steps)
            # the same box for every step takes the banded tile order
            same = steps.copy()
            same["i0"], same["i1"], same["j0"], same["j1"] = 2, 697, 1, 59
            out[kernel + "/banded"] = eng.run_host(fields, same)
    for a, b in ((out["direct"], out["tile"]), (out["direct/banded"], out["tile/banded"])):
        for x, y in zip(a, b):
            assert np.array_equal(x, y, equal_nan=True)
    assert np.isnan(out["tile"][0]).any() and np.isfinite(out["tile"][0][3]).all()


def test_sub_warp_kernel_reports_nans_only_for_the_boxes_that_hold_them():
    """Track boxes take the sub-warp kernel with 8-lane row groups: moving boxes of different sizes (odd start
    columns, heights that are no multiple of a warp's four rows, boxes on the grid edges), a NaN inside one box and a
    NaN row outside every box but the last.  Only the steps whose box holds a NaN may report one."""
    nlon, nlat, nlev, nt = 260, 232, 5, 6
    lon = (-70.0 + 0.1 * np.arange(nlon)).astype(np.float32)
    lat = (-42.0 + 0.1 * np.arange(nlat)).astype(np.float32)
    P, fields = _dataset(nlon, nlat, nlev, nt, np.float32, lon=lon, lat=lat, dt_h=1, seed=23)
    fields[0][2, 1, 50, 170] = np.nan         # inside box 2 only
    fields[2][:, :, 0, :] = np.nan            # first grid row: outside every box but the last
    steps = E.time_stencil(H.tsec_of(P), E.make_steps(nt))
    boxes = [(5, 155, 1, 151), (1, 151, 3, 153), (30, 180, 33, 97), (109, 259, 81, 231), (7, 67, 100, 160), (0, 150, 0, 150)]
    for it, (i0, i1, j0, j1) in enumerate(boxes):
        steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = i0, i1, j0, j1
    with H.make_engine(P, np.float32, [1.0] * 5, max_box_rows=151) as eng:
        terms = eng.run_host(fields, steps)[0]
        d = eng.last_dispatch()
    assert d["kernel"] == "subwarp" and d["group"] == 8, d
    assert np.isnan(terms[2]).any() and np.isnan(terms[5]).any() and np.isfinite(terms[[0, 1, 3, 4]]).all()
