"""Shared test plumbing: feed the CUDA engine from the oracle's prepared dataset and
compare the two.  Test infrastructure only (imports ``oracle``)."""
import os

import numpy as np

from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

FIELD_ORDER = ["Air Temperature", "Eastward Wind Component", "Northward Wind Component",
               "Omega Velocity", "Geopotential"]


def load_prepared(nc, namelist="namelist_NCEP-R2", track=None):
    raw = O.read_netcdf3(os.path.join(GOLDEN, "samples", nc))
    nl = O.read_namelist(os.path.join(GOLDEN, "inputs", namelist))
    tr = O.read_track(os.path.join(GOLDEN, "inputs", track)) if track else None
    return O.process_data(raw, nl, tr), tr


def engine_inputs(P, dtype):
    """Five [t][k][j][i] arrays in engine order + unit scales (box_data.py:297-310, :233-241)."""
    fields, scale = [], []
    for name in FIELD_ORDER:
        if name == "Geopotential" and name not in P.fields:
            arr, s = P.fields["Geopotential Height"], O._UNIT_TO_SI[P.units["Geopotential Height"]] * O.g
        else:
            arr, s = P.fields[name], O._UNIT_TO_SI[P.units[name]]
        fields.append(np.ascontiguousarray(arr, dtype=dtype))
        scale.append(s)
    return fields, scale


def make_engine(P, dtype, scale, max_steps=64, **kw):
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    return E.LecEngine(f64(P.lon), f64(P.lat), f64(P.rlons), f64(P.rlats), f64(P.coslats), f64(P.level),
                       dtype, scale, max_steps=max_steps, **kw)


def tsec_of(P):
    return ((P.time - P.time.min()) / np.timedelta64(1, "s")).astype(np.float64)


def fixed_steps(P, west, east, south, north):
    n = len(P.time)
    steps = E.time_stencil(tsec_of(P), E.make_steps(n))
    steps["i0"], steps["i1"] = E.nearest_index(P.lon, west), E.nearest_index(P.lon, east)
    steps["j0"], steps["j1"] = E.nearest_index(P.lat, south), E.nearest_index(P.lat, north)
    return steps


def moving_steps(P, track):
    import pandas as pd
    n = len(P.time)
    steps = E.time_stencil(tsec_of(P), E.make_steps(n))
    for it, t in enumerate(pd.to_datetime(P.time)):
        lim = O.get_limits(track, t)
        steps["i0"][it], steps["i1"][it] = E.nearest_index(P.lon, lim["min_lon"]), E.nearest_index(P.lon, lim["max_lon"])
        steps["j0"][it], steps["j1"][it] = E.nearest_index(P.lat, lim["min_lat"]), E.nearest_index(P.lat, lim["max_lat"])
    return steps


def series_err(a, b):
    """max_t |a-b| / max_t |b| (SURVEY.md section 7, test plan)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    den = np.max(np.abs(b))
    return float(np.max(np.abs(a - b)) / den) if den > 0 else float(np.max(np.abs(a - b)))


def compare_terms(terms, df, names=None, extra=None):
    """Series-scaled error per term between engine ``terms[n,16]`` and an oracle frame."""
    out = {}
    for i, name in enumerate(E.TERM_NAMES):
        if names is not None and name not in names:
            continue
        if name in df.columns:
            ref = df[name].values
        elif extra is not None and name in extra:
            ref = np.asarray(extra[name])
        else:
            continue
        out[name] = series_err(terms[:, i], ref)
    return out


def compare_levels(levels, lv):
    out = {}
    for i, name in enumerate(E.LEVEL_TERM_NAMES):
        ref = np.asarray(lv[name], dtype=np.float64)
        out[name] = series_err(levels[:, i, :], ref)
    return out


# --------------------------------------------------------------------------------------- #
# synthetic datasets (oracle side)
NAMES = ["Air Temperature", "Eastward Wind Component", "Northward Wind Component", "Omega Velocity", "Geopotential"]


def prepared_from_arrays(fields, lon, lat, level, time, units=("K", "m/s", "m/s", "Pa/s", "m**2/s**2"),
                         names=None, coord_dtype=np.float32):
    """Oracle dataset from five [t][k][j][i] arrays; radians/cos computed in the coordinate dtype
    exactly as process_data does (preprocessing.py:288-290)."""
    P = O.Prepared()
    names = names or NAMES
    P.fields = dict(zip(names, fields))
    P.units = dict(zip(names, units))
    P.time = np.asarray(time)
    P.level = np.asarray(level, dtype=np.float64)
    P.lat = np.asarray(lat, dtype=coord_dtype)
    P.lon = np.asarray(lon, dtype=coord_dtype)
    P.rlats, P.coslats, P.rlons = np.deg2rad(P.lat), np.cos(np.deg2rad(P.lat)), np.deg2rad(P.lon)
    return P


def smooth_fields(nt, nlev, nlat, nlon, dtype, seed=0, level=None, lat=None):
    """Small seeded test fields with realistic magnitudes (stable stratification)."""
    rng = np.random.default_rng(seed)
    p = np.linspace(1.0, 10.0, nlev)[:, None, None] * 1e4 if level is None else np.asarray(level)[:, None, None]
    x = p / 1e5
    phi = np.linspace(-0.9, 0.9, nlat)[None, :, None] if lat is None else np.deg2rad(np.asarray(lat, dtype=np.float64))[None, :, None]
    lam = np.linspace(0, 2 * np.pi, nlon, endpoint=False)[None, None, :]
    out = []
    base = [288.0 - 60.0 * (1 - x ** 0.19) + 15 * (np.cos(phi) ** 2 - 0.5), 10 * np.cos(phi) * x, 0 * x, 0 * x,
            9.80665 * 44330.0 * (1 - x ** 0.19)]
    amp, noise = [3.0, 8.0, 6.0, 0.2, 300.0], [0.5, 1.0, 1.0, 0.02, 20.0]
    for f in range(5):
        arr = np.empty((nt, nlev, nlat, nlon))
        for t in range(nt):
            wave = sum(amp[f] / m * np.cos(m * lam + 0.3 * t * m + f + 2 * m * x) * np.cos(phi) ** 2 for m in (1, 2, 3))
            arr[t] = base[f] + wave + noise[f] * rng.standard_normal((nlev, nlat, nlon))
        out.append(np.ascontiguousarray(arr.astype(dtype)))
    return out


def write_era5_like(path, packed, nlon):
    """A small NetCDF-3 file with ERA5's on-disk conventions (see tests/test_era5_conventions_gpu.py)."""
    import pandas as pd
    from scipy.io import netcdf_file
    from lorenzcycletoolkit_b200.synthetic import ERA5_LEVELS_HPA
    lon = (-65.0 + 0.25 * np.arange(nlon)).astype(np.float32)
    lat = (-5.0 - 0.25 * np.arange(141)).astype(np.float32)            # north -> south, as ERA5 stores it
    lev = np.array(ERA5_LEVELS_HPA[::-1], dtype=np.int32)              # 1000 ... 1 hPa
    nt = 5
    fields = smooth_fields(nt, len(lev), len(lat), nlon, np.float32, seed=7,
                             level=lev.astype(np.float64) * 100.0, lat=lat)
    with netcdf_file(path, "w") as f:
        f.createDimension("time", nt); f.createDimension("level", len(lev))
        f.createDimension("latitude", len(lat)); f.createDimension("longitude", nlon)
        t = f.createVariable("time", "i4", ("time",)); t.units = "hours since 1900-01-01 00:00:00.0"
        t[:] = int((pd.Timestamp("2005-08-09") - pd.Timestamp("1900-01-01")) / pd.Timedelta("1h")) + np.arange(nt)
        v = f.createVariable("level", "i4", ("level",)); v.units = "millibars"; v[:] = lev
        v = f.createVariable("latitude", "f4", ("latitude",)); v.units = "degrees_north"; v[:] = lat
        v = f.createVariable("longitude", "f4", ("longitude",)); v.units = "degrees_east"; v[:] = lon
        for name, arr in zip("TUVWZ", fields):
            if packed:
                lo, hi = float(arr.min()), float(arr.max())
                scale, offset = (hi - lo) / 65000.0, 0.5 * (hi + lo)
                var = f.createVariable(name, "i2", ("time", "level", "latitude", "longitude"))
                var.scale_factor, var.add_offset, var._FillValue = scale, offset, np.int16(-32767)
                var[:] = np.round((arr - offset) / scale).astype(np.int16)
            else:
                var = f.createVariable(name, "f4", ("time", "level", "latitude", "longitude"))
                var[:] = arr


def write_era5_unheld_fill(path, nlon):
    """:func:`write_era5_like`'s int16 file with a ``_FillValue`` no int16 can hold (40000) and stored 32767 values
    (the value that fill saturates to in int16) spread over T and Z: no record is missing."""
    src = path + ".src.nc"
    write_era5_like(src, True, nlon)

    def plant(name, data):
        if name in ("T", "Z"):
            data.reshape(-1)[::97] = 32767
        return data
    write_netcdf3_copy(src, path, plant, attrs={v: {"_FillValue": np.int32(40000)} for v in "TUVWZ"})


def write_netcdf3_copy(src, dst, edit=None, extra=None, attrs=None):
    """Copy a NetCDF-3 classic file variable by variable, letting ``edit(name, array)`` change the data
    (e.g. plant ``_FillValue`` entries; the variable takes the dtype of the array it returns); dimensions, dtypes and
    attributes are kept, ``attrs``: ``name -> {attribute: value}`` set on top.  ``extra``: new variables,
    ``name -> (dims, array, attrs)``."""
    from scipy.io import netcdf_file
    with netcdf_file(src, mmap=False) as f, netcdf_file(dst, "w") as g:
        for k in f._attributes:
            setattr(g, k, getattr(f, k))
        for name, size in f.dimensions.items():
            g.createDimension(name, size)
        for name, v in f.variables.items():
            data = np.array(v.data)
            data = data.astype(data.dtype.newbyteorder("="))
            out = edit(name, data) if edit else None
            data = data if out is None else out
            var = g.createVariable(name, data.dtype if data.dtype.kind != "S" else "c", v.dimensions)
            for a, x in dict({a: getattr(v, a) for a in v._attributes}, **(attrs or {}).get(name, {})).items():
                setattr(var, a, x)
            var[:] = data
        for name, (dims, arr, attrs) in (extra or {}).items():
            var = g.createVariable(name, np.asarray(arr).dtype, dims)
            for k, v in attrs.items():
                setattr(var, k, v)
            var[:] = arr


# --------------------------------------------------------------------------------------- #
# one step of the oracle on any box, and the per-level boundary pieces
BOUNDARY_TERMS = ["BAz", "BAe", "BKz", "BKe", "BΦZ", "BΦE"]


def boundary_pieces(pieces):
    """The dict ``O.boundary_terms(..., pieces=)`` fills, as the engine's ``[..][6][3][nlev]`` array."""
    return np.stack([np.asarray(pieces[n], dtype=np.float64) for n in BOUNDARY_TERMS], axis=-3)


def oracle_step(P, box, it, dTdt):
    """One step evaluated as ``O.lec_moving`` does (a ``BoxState`` of time ``it`` on the box of grid indices
    ``box = (i0, i1, j0, j1)``, ``dTdt`` the global ``np.gradient`` dT/dt), for a ``P`` already in the arithmetic
    of the comparison (``O.to_mode(P, "fp64")``).  Returns (16 terms by name, per-level families by name,
    boundary pieces ``[6][3][nlev]``, raw): ``raw`` holds the same 19 families as computed, before the reference's
    ``_handle_nans`` (they differ only where a family has a missing level), and under ``"sigma"`` the static
    stability before its 0.03 floor."""
    i0, i1, j0, j1 = box
    b = O.BoxState(P, P.lon[i0], P.lon[i1], P.lat[j0], P.lat[j1], fixed=False, dTdt=dTdt[it], tsel=it)
    assert b.idx == tuple(box), (b.idx, box)
    lv, raw, terms, pieces = {}, {}, {}, {}
    terms.update(O.energy_contents(b, lv, raw))
    terms.update(O.conversion_terms(b, lv, raw))
    terms.update(O.boundary_terms(b, pieces=pieces))
    terms.update(O.generation_terms(b, lv, raw))
    f64 = lambda d: {k: np.asarray(v, dtype=np.float64) for k, v in d.items()}
    return ({k: float(v) for k, v in terms.items()}, f64(lv), boundary_pieces(pieces),
            dict(f64(raw), sigma=np.asarray(b.sigma_prefloor, dtype=np.float64)))


# --------------------------------------------------------------------------------------- #
# int16-packed fields (lec_run_device_packed) and device-side boundary pieces
FILL = -32767


def _is_torch(a):
    return not isinstance(a, np.ndarray) and hasattr(a, "is_cuda")


def encode(fields, spec, bounds=None):
    """int16 records of float fields + the decode dicts of LecEngine.run_torch_packed.  ``fields``: numpy arrays, or
    torch tensors, encoded where they live by the same float64 operations (fields too large for the host).
    ``bounds``: per field the (min, max) of the whole series when ``fields`` hold one slice of it at a time."""
    raws, decode = [], []
    for n, (a, sp) in enumerate(zip(fields, spec)):
        dev = _is_torch(a)
        a = a.double() if dev else np.asarray(a, dtype=np.float64)
        lo, hi = (float(a.min()), float(a.max())) if bounds is None else (float(bounds[n][0]), float(bounds[n][1]))
        if sp["offset"]:
            scale, offset = (hi - lo) / 65000.0, 0.5 * (hi + lo)
        else:
            scale, offset = max(abs(lo), abs(hi)) / 32000.0, None
        q = (a - (offset or 0.0)) / scale
        raw = q.round().short() if dev else np.round(q).astype(np.int16)      # both round half to even
        fills = [FILL, -32768][:sp["nfill"]]
        raws.append(raw)
        decode.append(dict(scale=np.float64(scale), offset=None if offset is None else np.float64(offset),
                           fills=fills, float32=sp["float32"]))
    return raws, decode


def decode(raw, dec, dtype):
    """The decode rule in numpy (or in torch for a device tensor): multiply, then add, as separate float64
    operations."""
    dev = _is_torch(raw)
    x = raw.double() if dev else raw.astype(np.float64)
    if dec["scale"] is not None:
        x = x * np.float64(dec["scale"])
    if dec["offset"] is not None:
        x = x + np.float64(dec["offset"])
    if dec["float32"]:
        x = x.float().double() if dev else x.astype(np.float32).astype(np.float64)
    for fv in dec["fills"]:
        x[raw == fv] = np.nan
    if dev:
        return x if np.dtype(dtype) == np.float64 else x.float()
    return x.astype(dtype)


def padded(raw, pitch):
    """Device int16 [slot][level][lat][pitch]; the pad columns hold fill values."""
    import torch
    buf = np.full(raw.shape[:3] + (pitch,), FILL, dtype=np.int16)
    buf[..., :raw.shape[3]] = raw
    return torch.from_numpy(buf).cuda()


def with_boundary(eng, n, fn):
    """Run ``fn()`` (a LecEngine.run_torch* call) with the per-level boundary pieces armed on a device buffer;
    returns (fn's results as numpy arrays..., pieces ``[n][18][nlev]``)."""
    import ctypes as C
    import torch
    bnd = torch.empty((n, E.NBOUNDARY_PIECES, eng.nlev), dtype=torch.float64, device="cuda")
    eng._check(eng._lib.lec_set_boundary_levels(eng._h, C.c_void_p(bnd.data_ptr())), "lec_set_boundary_levels")
    try:
        out = fn()
    finally:
        eng._lib.lec_set_boundary_levels(eng._h, None)
    torch.cuda.synchronize()
    return tuple(x.cpu().numpy() for x in out) + (bnd.cpu().numpy(),)


def check_refs(out, refs, tol):
    """Steps of one box against their oracle results (``oracle_step``): all 16 terms, 19 per-level families and 18
    boundary pieces, series-scaled over the steps.  ``out`` = (terms, levels, flags, pieces [n][6][3][nlev]).
    Returns the worst error."""
    terms, levels, flags, bnd = out
    assert not flags.any(), flags
    assert np.isfinite(terms).all() and np.isfinite(levels).all() and np.isfinite(bnd).all()
    errs = {name: series_err(terms[:, i], [r[0][name] for r in refs]) for i, name in enumerate(E.TERM_NAMES)}
    errs.update({"lv:" + name: series_err(levels[:, i], np.stack([np.broadcast_to(r[1][name], levels.shape[2:])
                                                                   for r in refs]))
                 for i, name in enumerate(E.LEVEL_TERM_NAMES)})
    errs.update({f"bnd:{name}.{part}": series_err(bnd[:, n, part], np.stack([r[2][n, part] for r in refs]))
                 for n, name in enumerate(BOUNDARY_TERMS) for part in range(3)})
    assert len(errs) == 16 + 19 + 18
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, bad
    return max(errs.values())


def staged_slots(steps, window, max_steps):
    """The greedy chunks of ``lec_run_host*`` over a staging window of ``window`` slots, replayed: returns (T slots that
    cross PCIe, slots of u / v / omega / Phi that cross PCIe per field, whether a chunk took T slots device to device
    from a previous window that starts at an earlier slot).  A chunk stages T over its whole slot range, minus the
    slots the previous chunk's window holds, and the other fields over the range of its centre slots."""
    n, s0, chunk, prev_lo, prev_hi = len(steps), 0, 0, 0, -1
    t_slots = c_slots = 0
    shifted = False
    while s0 < n:
        lo, hi, s1 = 1 << 30, -1, s0
        while s1 < n and s1 - s0 < max_steps:
            sl = [int(steps[k][s1]) for k in ("slot", "slot_m", "slot_p")]
            if max(hi, *sl) - min(lo, *sl) + 1 > window:
                break
            lo, hi, s1 = min(lo, *sl), max(hi, *sl), s1 + 1
        assert s1 > s0, "a step needs more slots than the window holds"
        t_lo = lo
        if chunk >= 1 and prev_lo <= lo <= prev_hi:
            t_lo = min(prev_hi, hi) + 1
            shifted |= lo > prev_lo
        t_slots += max(0, hi - t_lo + 1)
        centre = steps["slot"][s0:s1]
        c_slots += int(centre.max() - centre.min() + 1)
        prev_lo, prev_hi, s0, chunk = lo, hi, s1, chunk + 1
    return t_slots, c_slots, shifted


def same_bits(a, b):
    for x, y in zip(a, b):
        assert x.shape == y.shape and np.array_equal(x.view(np.uint8), y.view(np.uint8))
