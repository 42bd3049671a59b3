"""numpy restatement of the LorenzCycleToolkit hot path (CPU oracle).

TEST INFRASTRUCTURE ONLY -- never imported by ``lorenzcycletoolkit_b200``.

The reference (daniloceano/LorenzCycleToolkit v1.1.11) is pure Python on top of
xarray 2024.2.0 / numpy 2.0.0 / MetPy 1.6.2 / Pint 0.24.3 / pandas 2.2.2, none
of which (except numpy/pandas) exist in this image, so the reference itself
cannot be imported.  This module restates its arithmetic with plain numpy, one
function per reference function, keeping the *operation order and dtype
propagation* of the reference so that it reproduces the reference's own bundled
outputs (``tests/golden/samples``; pinned by ``tests/test_oracle_golden.py``):

  parity pins: Catarina_NCEP-R2 fixed results (22 columns x 36 steps),
  per-level CSVs of Reg1-Representative fixed / track-15x15 on the 5-step
  ``testdata_NCEP-R2.nc`` subset.  Unpinned (formula from source only):
  B-Phi-Z, B-Phi-E, Dz/De, NaN path, 850-hPa diagnostics.

Third-party semantics restated here (SURVEY.md Appendix B):
  * ``DataArray.integrate``      -> :func:`trapz`      (xarray duck_array_ops.trapz)
  * ``DataArray.differentiate``  -> ``np.gradient(f, x, axis, edge_order=1)``
  * ``.sel(method="nearest")``   -> pandas ``Index.get_indexer(method="nearest")``
  * ``.sel(dim=slice(a, b))``    -> inclusive label slice on a sorted index
  * ``interpolate_na(dim=level)``-> :func:`interpolate_na_level`
  * MetPy constants / ``potential_temperature``

Two dtype modes:
  ``mode="ref"``  keep the stored dtypes (float32 files stay float32 wherever
                  numpy's NEP-50 promotion keeps them so, as in the reference);
  ``mode="fp64"`` upcast the stored field values and the derived coordinate
                  arrays (rlats/coslats/rlons *as computed in the stored dtype*)
                  to float64 first, then run the identical arithmetic.

Array convention: fields are ``[time][level][lat][lon]`` (fixed framework) or
``[level][lat][lon]`` (one step of the moving framework); every function below
uses negative axes (lon=-1, lat=-2, level=-3) so both work.
"""

from __future__ import annotations

import warnings

import numpy as np
import pandas as pd

# --------------------------------------------------------------------------- #
# MetPy 1.6.2 constants (metpy/constants/default.py), Python floats = "weak"
# scalars under NEP 50, exactly as pint Quantities wrapping Python floats.
# --------------------------------------------------------------------------- #
g = 9.80665
Re = 6371008.7714
_R = 8.314462618
_Md = 28.96546e-3
Rd = _R / _Md                                  # 287.04749097718457
_gamma = 1.4
Cp_d = _gamma * Rd / (_gamma - 1)              # 1004.6662184201462
kappa = Rd / Cp_d                              # 0.28571428571428564
P0 = 100000.0                                  # 1000 hPa in Pa

LEVEL_TERMS = [
    "Az", "Ae", "Kz", "Ke", "Ge", "Gz", "Cz", "Cz_1", "Cz_2", "Ca", "Ca_1", "Ca_2",
    "Ce", "Ce_1", "Ce_2", "Ck", "Ck_1", "Ck_2", "Ck_3", "Ck_4", "Ck_5",
]  # lec_fixed_framework.py:172-194 / lec_moving_framework.py:583-605


# --------------------------------------------------------------------------- #
# xarray / pandas primitives
# --------------------------------------------------------------------------- #
def trapz(y, x, axis):
    """xarray ``duck_array_ops.trapz`` (used by ``DataArray.integrate``;
    call sites calc_averages.py:43,76 and every ``.integrate(level)``)."""
    y = np.asarray(y)
    x = np.asarray(x)
    if axis < 0:
        axis = y.ndim + axis
    x_sl1 = (slice(1, None),) + (None,) * (y.ndim - axis - 1)
    x_sl2 = (slice(None, -1),) + (None,) * (y.ndim - axis - 1)
    slice1 = (slice(None),) * axis + (slice(1, None),)
    slice2 = (slice(None),) * axis + (slice(None, -1),)
    dx = x[x_sl1] - x[x_sl2]
    integrand = dx * 0.5 * (y[tuple(slice1)] + y[tuple(slice2)])
    return np.sum(integrand, axis=axis)


def differentiate(f, x, axis):
    """``DataArray.differentiate(coord, edge_order=1)`` == ``np.gradient``."""
    return np.gradient(f, x, axis=axis, edge_order=1)


def nearest_index(coord, value):
    """``coord.sel({dim: value}, method="nearest")`` (box_data.py:133-135):
    pandas nearest indexer; ties go to the larger coordinate."""
    idx = pd.Index(np.asarray(coord))
    return int(idx.get_indexer([value], method="nearest")[0])


def label_slice(coord, lo, hi):
    """``.sel(dim=slice(lo, hi))`` on an increasing index: inclusive bounds."""
    coord = np.asarray(coord)
    i0 = int(np.searchsorted(coord, lo, side="left"))
    i1 = int(np.searchsorted(coord, hi, side="right"))
    return i0, i1  # python half-open [i0, i1)


def interpolate_na_level(arr, levels, axis):
    """``interpolate_na(dim=level)``: linear in the coordinate, interior gaps
    only; slices with no NaN or only NaN are returned unchanged."""
    arr = np.array(arr, dtype=np.result_type(arr.dtype, np.float32), copy=True)
    x = np.asarray(levels, dtype=np.float64)
    moved = np.moveaxis(arr, axis, -1)
    flat = moved.reshape(-1, moved.shape[-1])
    for row in flat:
        nans = np.isnan(row)
        n = int(nans.sum())
        if n == 0 or n == row.size:
            continue
        row[:] = np.interp(x, x[~nans], row[~nans], left=np.nan, right=np.nan)
    return arr


def handle_nans(function, levels, axis):
    """``_handle_nans`` (energy_contents.py:190-208 and its three copies).

    Returns ``(function, levels)`` because dropping levels changes the
    coordinate used by the following ``integrate``.
    """
    function = np.asarray(function)
    levels = np.asarray(levels)
    if np.isnan(function).any():
        function = interpolate_na_level(function, levels, axis)
        if np.isnan(function).any():
            ax = axis if axis >= 0 else function.ndim + axis
            other = tuple(a for a in range(function.ndim) if a != ax)
            keep = ~np.isnan(function).any(axis=other) if other else ~np.isnan(function)
            function = np.compress(keep, function, axis=ax)
            levels = levels[keep]
    return function, levels


# --------------------------------------------------------------------------- #
# NetCDF-3 reading with xarray's decode semantics (what xr.open_dataset does
# implicitly; preprocessing.py:73-74)
# --------------------------------------------------------------------------- #
def _decode_time(values, units):
    unit, _, ref = units.partition(" since ")
    unit = unit.strip().lower()
    ref = ref.strip().replace("T", " ")
    ref64 = np.datetime64(pd.Timestamp(ref).to_datetime64(), "ns")
    per = {"seconds": 1, "second": 1, "minutes": 60, "minute": 60, "hours": 3600,
           "hour": 3600, "days": 86400, "day": 86400}[unit]
    ns = np.round(np.asarray(values, dtype=np.float64) * per * 1e9).astype("int64")
    return ref64 + ns.astype("timedelta64[ns]")


def read_netcdf3(path):
    """Open a NetCDF-3 classic file the way ``xr.open_dataset`` would decode it:
    ``_FillValue``/``missing_value`` -> NaN, ``scale_factor``/``add_offset``
    unpacking, CF time decoding; float32 stays float32."""
    from scipy.io import netcdf_file

    out = {"vars": {}, "dims": {}, "attrs": {}}
    with netcdf_file(path, mmap=False) as f:
        for name, v in f.variables.items():
            data = np.array(v.data)
            if data.dtype.byteorder == ">":
                data = data.astype(data.dtype.newbyteorder("="))
            attrs = {a: getattr(v, a) for a in v._attributes}
            attrs = {k: (val.decode() if isinstance(val, bytes) else val) for k, val in attrs.items()}
            fills = [attrs[k] for k in ("_FillValue", "missing_value") if k in attrs]
            scale, offset = attrs.get("scale_factor"), attrs.get("add_offset")
            if data.dtype.kind in "iu" and (scale is not None or offset is not None):
                small = data.dtype.itemsize <= 2 and offset is None
                fdt = np.float32 if small else np.float64
                raw = data
                data = raw.astype(fdt)
                for fv in fills:
                    data[raw == fv] = np.nan
                if scale is not None:
                    data *= scale
                if offset is not None:
                    data += offset
            elif data.dtype.kind == "f":
                for fv in fills:
                    data[data == fv] = np.nan
            units = attrs.get("units", "")
            if isinstance(units, str) and " since " in units and data.ndim == 1:
                data = _decode_time(data, units)
            out["vars"][name] = data
            out["dims"][name] = tuple(v.dimensions)
            out["attrs"][name] = attrs
    return out


def read_namelist(path):
    """``pd.read_csv(namelist, sep=";", index_col=0, header=0)``
    (validation.py:167, lorenzcycletoolkit.py:175)."""
    return pd.read_csv(path, sep=";", index_col=0, header=0)


def read_track(path):
    """Track file (``time;Lat;Lon[;length;width;...]``, time ``%Y-%m-%d-%H%M``;
    preprocessing.py:176-182)."""
    tr = pd.read_csv(path, delimiter=";", index_col="time")
    tr.index = pd.to_datetime(tr.index, format="%Y-%m-%d-%H%M")
    return tr


_UNIT_TO_SI = {  # pint factors for the units that occur in inputs/namelist_*
    "K": 1.0, "m/s": 1.0, "Pa/s": 1.0, "m**2/s**2": 1.0, "m": 1.0, "gpm": 1.0,
    "hPa/s": 100.0,
}


# --------------------------------------------------------------------------- #
# preprocessing.py:149-371 (process_data) and select_area.py:254-338
# --------------------------------------------------------------------------- #
class Prepared:
    """The preprocessed dataset handed to the frameworks (the layout contract
    of SURVEY.md section 3.5): dims sorted lon/level/lat ascending, levels in Pa
    >= 1000 Pa, extra coords rlats/coslats/rlons in the coordinate dtype."""

    def __init__(self):
        self.fields = {}      # canonical name -> array [t][k][j][i]
        self.units = {}       # canonical name -> namelist unit string
        self.time = None      # datetime64[ns]
        self.level = None     # Pa
        self.lat = self.lon = None
        self.rlats = self.coslats = self.rlons = None
        self.names = {}       # Time / Vertical Level / Latitude / Longitude -> var name


_FIELD_ROWS = ["Air Temperature", "Eastward Wind Component", "Northward Wind Component",
               "Omega Velocity", "Geopotential", "Geopotential Height"]


def process_data(raw, namelist, track=None):
    """``process_data`` (preprocessing.py:149-371)."""
    tname = namelist.loc["Time"]["Variable"]
    lon_n = namelist.loc["Longitude"]["Variable"]
    lat_n = namelist.loc["Latitude"]["Variable"]
    lev_n = namelist.loc["Vertical Level"]["Variable"]
    V = raw["vars"]
    time, lon, lat, lev = V[tname], V[lon_n], V[lat_n], V[lev_n]

    fields, units = {}, {}
    for row in _FIELD_ROWS:
        if row in namelist.index:
            var = namelist.loc[row]["Variable"]
            dims = raw["dims"][var]
            arr = V[var]
            order = [dims.index(d) for d in (tname, lev_n, lat_n, lon_n)]
            fields[row] = np.transpose(arr, order)
            units[row] = namelist.loc[row]["Units"]

    # :168-274 keep only data times equal to track times
    if track is not None:
        dt_data = int((time[1] - time[0]) / np.timedelta64(1, "h"))
        dt_track = int((track.index[1] - track.index[0]) / np.timedelta64(1, "h"))
        if dt_data > dt_track:
            raise ValueError("Data time step is higher than track time step")
        if track.index[0] < time[0] or track.index[-1] > time[-1]:
            raise ValueError("Track time limits do not match with data time limits")
        sel = pd.Index(time).get_indexer(track.index.values)
        if (sel < 0).any():
            raise KeyError("track time not in data")
        time = time[sel]
        fields = {k: a[sel] for k, a in fields.items()}

    # :275-281 longitude to [-180, 180)
    if lon.min() < -180 or lon.max() > 180:
        lon = (lon + 180) % 360 - 180
        o = np.argsort(lon, kind="stable")
        lon = lon[o]
        fields = {k: a[..., o] for k, a in fields.items()}

    # :288-290 radians coordinates in the coordinate's own dtype
    rlats = np.deg2rad(lat)
    coslats = np.cos(np.deg2rad(lat))
    rlons = np.deg2rad(lon)

    # :301-314 level -> Pa
    lunits = raw["attrs"][lev_n].get("units", "hPa")
    fac = {"hPa": 100.0, "millibars": 100.0, "mbar": 100.0, "mb": 100.0, "Pa": None}[str(lunits)]
    lev = lev * fac if fac is not None else lev

    # :358-362 sort lon, level, lat ascending
    o = np.argsort(lon, kind="stable")
    lon, rlons = lon[o], rlons[o]
    fields = {k: a[..., o] for k, a in fields.items()}
    o = np.argsort(lev, kind="stable")
    lev = lev[o]
    fields = {k: a[:, o] for k, a in fields.items()}
    o = np.argsort(lat, kind="stable")
    lat, rlats, coslats = lat[o], rlats[o], coslats[o]
    fields = {k: a[:, :, o] for k, a in fields.items()}

    # :364-365 keep levels in [1000 Pa, max]
    k0, k1 = label_slice(lev, 1000, float(lev.max()))
    lev = lev[k0:k1]
    fields = {k: a[:, k0:k1] for k, a in fields.items()}

    P = Prepared()
    P.fields, P.units = {k: np.ascontiguousarray(a) for k, a in fields.items()}, units
    P.time, P.level, P.lat, P.lon = time, lev, lat, lon
    P.rlats, P.coslats, P.rlons = rlats, coslats, rlons
    P.names = {"Time": tname, "Vertical Level": lev_n, "Latitude": lat_n, "Longitude": lon_n}
    return P


def crop(P, j0, j1, i0, i1):
    """Label slice of every field and coordinate (half-open index ranges)."""
    Q = Prepared()
    Q.fields = {k: a[:, :, j0:j1, i0:i1] for k, a in P.fields.items()}
    Q.units, Q.time, Q.level, Q.names = P.units, P.time, P.level, P.names
    Q.lat, Q.rlats, Q.coslats = P.lat[j0:j1], P.rlats[j0:j1], P.coslats[j0:j1]
    Q.lon, Q.rlons = P.lon[i0:i1], P.rlons[i0:i1]
    return Q


def slice_domain_fixed(P, min_lon, max_lon, min_lat, max_lat):
    """``slice_domain`` fixed branch (select_area.py:272-295,331-336): crop to
    the nearest grid values of the four limits (of ``inputs/box_limits``)."""
    W = P.lon[nearest_index(P.lon, float(min_lon))]
    E = P.lon[nearest_index(P.lon, float(max_lon))]
    S = P.lat[nearest_index(P.lat, float(min_lat))]
    N = P.lat[nearest_index(P.lat, float(max_lat))]
    j0, j1 = label_slice(P.lat, float(S), float(N))
    i0, i1 = label_slice(P.lon, float(W), float(E))
    return crop(P, j0, j1, i0, i1)


def slice_domain_track(P, track):
    """``slice_domain`` track branch (select_area.py:297-313,331-336)."""
    dx = P.lon[1] - P.lon[0]
    dy = P.lat[1] - P.lat[0]
    if "width" in track.columns:
        mw, ml = track["width"].max(), track["length"].max()
    else:
        mw, ml = 15, 15
    W = track["Lon"].min() - (mw / 2) - dx
    E = track["Lon"].max() + (mw / 2) + dx
    S = track["Lat"].min() - (ml / 2) - dy
    N = track["Lat"].max() + (ml / 2) + dy
    j0, j1 = label_slice(P.lat, S, N)
    i0, i1 = label_slice(P.lon, W, E)
    return crop(P, j0, j1, i0, i1)


def to_mode(P, mode):
    """``mode="fp64"``: upcast stored values and the stored-dtype coordinate
    arrays to float64 (never recompute radians from degrees in double)."""
    if mode == "ref":
        return P
    assert mode == "fp64"
    Q = Prepared()
    Q.fields = {k: a.astype(np.float64) for k, a in P.fields.items()}
    Q.units, Q.time, Q.names = P.units, P.time, P.names
    Q.level = P.level.astype(np.float64)
    for n in ("lat", "lon", "rlats", "coslats", "rlons"):
        setattr(Q, n, getattr(P, n).astype(np.float64))
    return Q


# --------------------------------------------------------------------------- #
# calc_averages.py
# --------------------------------------------------------------------------- #
def CalcZonalAverage(f, rlons, xlength):
    """calc_averages.py:25-43."""
    return trapz(f, rlons, -1) / xlength


def CalcAreaAverage(f, rlats, coslats, rlons=None, xlength=None):
    """calc_averages.py:46-78.  ``f`` has a trailing lon axis only when
    ``xlength`` is given (then the zonal mean is taken first); ``ylength`` is
    recomputed from the box rlats exactly as at :75."""
    ZA = CalcZonalAverage(f, rlons, xlength) if xlength is not None else f
    ylength = np.sin(rlats[-1]) - np.sin(rlats[0])
    return trapz(ZA * coslats, rlats, -1) / ylength


# --------------------------------------------------------------------------- #
# thermodynamics.py
# --------------------------------------------------------------------------- #
def StaticStability(T, p, rlats, coslats, rlons, xlength, ylength):
    """thermodynamics.py:26-73.  ``p`` broadcastable along the level axis."""
    sigma_AA = static_stability_prefloor(T, p, rlats, coslats, rlons, xlength, ylength)
    return np.where(sigma_AA > 0.03, sigma_AA, 0.03)


def static_stability_prefloor(T, p, rlats, coslats, rlons, xlength, ylength):
    """:func:`StaticStability` before its floor: the value the floor tests (NaN where a level is missing)."""
    pk = p.reshape((-1, 1, 1))
    FirstTerm = g * T / Cp_d
    SecondTerm = pk * g / Rd
    ThirdTerm = differentiate(T, p, -3)
    function = FirstTerm - (SecondTerm * ThirdTerm)
    sigma_ZA = trapz(function, rlons, -1) / xlength
    return trapz(sigma_ZA * coslats, rlats, -1) / ylength


def AdiabaticHeating(T, p, omega, u, v, lat_deg, lon_deg, coslats, dTdt):
    """thermodynamics.py:76-124 (``dTdt`` already evaluated by the caller:
    box-local ``np.gradient`` over all file times in fixed mode, the global
    track-time derivative cropped to the box in moving mode)."""
    dTdlambda = differentiate(T, lon_deg, -1)
    dTdphi = differentiate(T, lat_deg, -2)
    dx = np.deg2rad(differentiate(lon_deg, lon_deg, 0))[None, :] * coslats[:, None] * Re   # [lat][lon]
    dy = (np.deg2rad(differentiate(lat_deg, lat_deg, 0)) * Re)[:, None]                    # [lat][1]
    AdvHTemp = -1 * ((u * dTdlambda / dx) + (v * dTdphi / dy))
    pk = p.reshape((-1, 1, 1))
    theta = T / (pk / P0) ** kappa
    sigma = -1 * (T / theta) * differentiate(theta, p, -3)
    ResT = dTdt - AdvHTemp - (sigma * omega)
    return ResT * Cp_d


# --------------------------------------------------------------------------- #
# box_data.py
# --------------------------------------------------------------------------- #
class BoxState:
    """``BoxData`` (box_data.py:57-310).  ``P`` holds either all times
    (``[t][k][j][i]``, fixed) or one time step (``[k][j][i]``, moving)."""

    def __init__(self, P, west, east, south, north, fixed=True, dTdt=None, tsel=None):
        lon, lat = P.lon, P.lat
        iw, ie = nearest_index(lon, west), nearest_index(lon, east)
        js, jn = nearest_index(lat, south), nearest_index(lat, north)
        self.idx = (iw, ie, js, jn)
        # :128-131 (0-d arrays in the coordinate dtype)
        self.xlength = np.asarray(P.rlons[ie] - P.rlons[iw])
        self.ylength = np.asarray(np.sin(P.rlats[jn]) - np.sin(P.rlats[js]))
        # inclusive label slices :304-309
        j0, j1 = label_slice(lat, lat[js], lat[jn])
        i0, i1 = label_slice(lon, lon[iw], lon[ie])
        self.sl = (j0, j1, i0, i1)
        self.lat, self.lon = lat[j0:j1], lon[i0:i1]
        self.rlats, self.coslats, self.rlons = P.rlats[j0:j1], P.coslats[j0:j1], P.rlons[i0:i1]
        self.p = P.level
        self.time = P.time

        def ext(name):
            a = P.fields[name]
            if tsel is not None:
                a = a[tsel]
            fac = _UNIT_TO_SI[P.units[name]]
            a = a[..., j0:j1, i0:i1]
            return a if fac == 1.0 else a * fac

        self.tair = ext("Air Temperature")
        self.u = ext("Eastward Wind Component")
        self.v = ext("Northward Wind Component")
        self.omega = ext("Omega Velocity")
        if "Geopotential" in P.fields:
            self.geopt = ext("Geopotential")
        else:
            self.geopt = ext("Geopotential Height") * g          # :233-241

        for n in ("tair", "u", "v", "omega", "geopt"):
            self._means(n)

        # :243-295
        if fixed:
            tsec = (P.time - P.time.min()) / np.timedelta64(1, "s")
            dTdt_box = differentiate(self.tair, tsec, 0)
        else:
            dTdt_box = dTdt[..., j0:j1, i0:i1]
        self.Q = AdiabaticHeating(self.tair, self.p, self.omega, self.u, self.v,
                                  self.lat, self.lon, self.coslats, dTdt_box)
        self._means("Q")
        # sigma_prefloor: what the 0.03 floor tests, so a caller can predict when the floor applies
        self.sigma_prefloor = static_stability_prefloor(self.tair, self.p, self.rlats, self.coslats,
                                                        self.rlons, self.xlength, self.ylength)
        self.sigma_AA = np.where(self.sigma_prefloor > 0.03, self.sigma_prefloor, 0.03)

    def _means(self, n):
        f = getattr(self, n)
        ZA = CalcZonalAverage(f, self.rlons, self.xlength)
        AA = CalcAreaAverage(ZA, self.rlats, self.coslats)
        setattr(self, n + "_ZA", ZA)
        setattr(self, n + "_AA", AA)
        setattr(self, n + "_ZE", f - ZA[..., None])
        setattr(self, n + "_AE", ZA - AA[..., None])

    # shorthands used by the term functions -------------------------------- #
    def AAz(self, f):                       # CalcAreaAverage(f, ylength)
        return CalcAreaAverage(f, self.rlats, self.coslats)

    def AA(self, f):                        # CalcAreaAverage(f, ylength, xlength=xlength)
        return CalcAreaAverage(f, self.rlats, self.coslats, self.rlons, self.xlength)

    def ZA(self, f):
        return CalcZonalAverage(f, self.rlons, self.xlength)


# --------------------------------------------------------------------------- #
# src/analysis/*.py
# --------------------------------------------------------------------------- #
def _integrate_levels(function, levels):
    function, levels = handle_nans(function, levels, -1)
    return function, trapz(function, levels, -1)


class _Families:
    """Records the per-level families of one term function: ``lv`` receives them as the reference saves them (after
    ``_handle_nans`` for the integrated ones), ``raw`` (optional) as they were computed, before ``_handle_nans``."""

    def __init__(self, lv, raw):
        self.lv, self.raw = lv, raw

    def keep(self, name, f):                # a family that is saved but not integrated
        self.lv[name] = f
        if self.raw is not None:
            self.raw[name] = f
        return f

    def integrate(self, name, f, levels):   # returns the trapezoid over the kept levels
        if self.raw is not None:
            self.raw[name] = f
        self.lv[name], I = _integrate_levels(f, levels)
        return I


def energy_contents(b, lv, raw=None):
    """energy_contents.py:99-165.  ``raw``: optional dict of the per-level families before ``_handle_nans``."""
    s = b.sigma_AA
    F = _Families(lv, raw)
    out = {}
    out["Az"] = F.integrate("Az", b.AAz(b.tair_AE ** 2) / (2 * s), b.p)
    out["Ae"] = F.integrate("Ae", b.AA(b.tair_ZE ** 2) / (2 * s), b.p)
    out["Kz"] = F.integrate("Kz", b.AAz(b.u_ZA ** 2 + b.v_ZA ** 2), b.p) / (2 * g)
    out["Ke"] = F.integrate("Ke", b.AA(b.u_ZE ** 2 + b.v_ZE ** 2), b.p) / (2 * g)
    return out


def conversion_terms(b, lv, raw=None):
    """conversion_terms.py:103-245 (order of the calls as in the frameworks).  ``raw``: as in
    :func:`energy_contents`."""
    s = b.sigma_AA
    p = b.p
    F = _Families(lv, raw)
    out = {}
    # calc_cz :168-192
    term1 = F.keep("Cz_1", Rd / (p * g))
    term2 = F.keep("Cz_2", b.AAz(b.omega_AE * b.tair_AE))
    out["Cz"] = F.integrate("Cz", -(term1 * term2), p)
    # calc_ca :103-140
    DelPhi_tairAE = differentiate(b.tair_AE * b.coslats, b.rlats, -1)
    t1 = (b.v_ZE * b.tair_ZE * DelPhi_tairAE[..., None]) / (2 * Re * s)[..., None, None]
    t1 = F.keep("Ca_1", b.AA(t1))
    DelPres_tairAE = differentiate(b.tair_AE, p, -2)
    t2 = (b.omega_ZE * b.tair_ZE) * DelPres_tairAE[..., None]
    t2 = F.keep("Ca_2", b.AA(t2) / s)
    out["Ca"] = F.integrate("Ca", -(t1 + t2), p)
    # calc_ck :194-245
    tan_lats = np.tan(b.rlats)
    DelPhi_uZA_cosphi = differentiate(b.u_ZA / b.coslats, b.rlats, -1)
    k1 = (b.coslats[:, None] * b.u_ZE * b.v_ZE / Re) * DelPhi_uZA_cosphi[..., None]
    k1 = F.keep("Ck_1", b.AA(k1))
    DelPhi_vZA = differentiate(b.v_ZA, b.rlats, -1)
    k2 = ((b.v_ZE ** 2) / Re) * DelPhi_vZA[..., None]
    k2 = F.keep("Ck_2", b.AA(k2))
    k3 = (tan_lats[:, None] * (b.u_ZE ** 2) * b.v_ZA[..., None]) / Re
    k3 = F.keep("Ck_3", b.AA(k3))
    DelPres_uZAp = differentiate(b.u_ZA, p, -2)
    k4 = b.omega_ZE * b.u_ZE * DelPres_uZAp[..., None]
    k4 = F.keep("Ck_4", b.AA(k4))
    DelPres_vZAp = differentiate(b.u_ZA, p, -2)            # sic: u_ZA (:225-229)
    k5 = b.omega_ZE * b.v_ZE * DelPres_vZAp[..., None]
    k5 = F.keep("Ck_5", b.AA(k5))
    out["Ck"] = F.integrate("Ck", k1 + k2 + k3 + k4 + k5, p) / g
    # calc_ce :142-166
    F.keep("Ce_1", term1)
    e2 = F.keep("Ce_2", b.AA(b.omega_ZE * b.tair_ZE))
    out["Ce"] = F.integrate("Ce", -(term1 * e2), p)
    return out


def boundary_terms(b, legacy_0d=False, pieces=None):
    """boundary_terms.py:122-418.

    ``legacy_0d``: evaluate ``c1, c2`` in float64 from the coordinate-dtype
    ``xlength, ylength`` (numpy 1.x value-based casting of Python-float x 0-d
    float32 array -- how the bundled goldens were produced, SURVEY.md C.1);
    default is the pinned numpy 2.0 NEP-50 behaviour (float32 on fp32 files).

    ``pieces``: a dict that receives, per term, the three per-level arrays the engine returns through
    ``lec_set_boundary_levels`` (lec_b200.h), stacked as ``[3][level]`` (``[time][3][level]`` for a fixed box):
    part 0 the E-W flux after ``Yphi``, part 1 the N-S difference, part 2 the vertical-flux integrand, all taken
    before ``_handle_nans``, so that ``term = c1 * trapz_p(part 0) + c2 * trapz_p(part 1) - (part 2[-1] - part 2[0])``.
    """
    s = b.sigma_AA
    p = b.p
    if legacy_0d:
        xl, yl = float(b.xlength), float(b.ylength)
    else:
        xl, yl = b.xlength, b.ylength
    c1 = -1 / (Re * xl * yl)
    c2 = -1 / (Re * yl)
    sk = s[..., None]                 # [.., k, 1] against [.., k, j]
    sk2 = s[..., None, None]          # against [.., k, j, i]
    E, W, N, S = -1, 0, -1, 0         # box edges (label == first/last of the box slice)
    T_AE, T_ZE = b.tair_AE, b.tair_ZE
    T_AE3 = T_AE[..., None]
    cos = b.coslats

    def Yphi(f):                      # .integrate("rlats") without cos
        return trapz(f, b.rlats, -1)

    def vint(f):                      # _handle_nans then integrate over level
        f, lev = handle_nans(f, p, -1)
        return trapz(f, lev, -1)

    def BT(f):                        # isel(level=-1) - isel(level=0) after _handle_nans
        f, _ = handle_nans(f, p, -1)
        return f[..., -1] - f[..., 0]

    def term(name, ew, ns, vert):     # ew, ns, vert: the per-level E-W, N-S and vertical pieces
        if pieces is not None:
            pieces[name] = np.stack([ew, ns, vert], axis=-2)
        return vint(ew) * c1 + vint(ns) * c2 - BT(vert)

    out = {}
    # calc_baz :125-181
    t1 = ((2 * T_AE3 * T_ZE * b.u) + (T_AE3 ** 2 * b.u)) / (2 * sk2)
    t1 = Yphi(t1[..., E] - t1[..., W])
    t2 = b.ZA(b.v_ZE * T_ZE) * 2 * T_AE
    t2 = (t2 + ((T_AE ** 2) * b.v_ZA)) * cos
    t2 = (t2[..., N] - t2[..., S]) / (2 * s)
    t3a = b.ZA(2 * b.omega_ZE * T_ZE) * T_AE
    t3b = b.omega_ZA * T_AE ** 2
    t3 = b.AAz(t3a + t3b) / (2 * s)
    out["BAz"] = term("BAz", t1, t2, t3)
    # calc_bae :183-230
    t1 = b.u * (T_ZE ** 2)
    t1 = t1[..., E] - t1[..., W]
    t1 = Yphi(t1 / (2 * sk))
    t2 = b.ZA(b.v * T_ZE ** 2) * cos
    t2 = t2 / (2 * sk)
    t2 = t2[..., N] - t2[..., S]
    t3 = b.AA((b.omega * T_ZE ** 2) / (2 * sk2))
    out["BAe"] = term("BAe", t1, t2, t3)
    # calc_bkz :232-280
    Kstar = b.u ** 2 + b.v ** 2 - b.u_ZE ** 2 - b.v_ZE ** 2
    t1 = b.u * Kstar
    t1 = t1[..., E] - t1[..., W]
    t1 = Yphi(t1 / (2 * g))
    t2 = b.ZA(Kstar * b.v * cos[:, None])
    t2 = t2[..., N] - t2[..., S]
    t2 = t2 / (2 * g)
    t3 = b.AA(Kstar * b.omega) / (2 * g)
    out["BKz"] = term("BKz", t1, t2, t3)
    # calc_bke :282-326
    Kp = b.u_ZE ** 2 + b.v_ZE ** 2
    t1 = b.u * Kp
    t1 = t1[..., E] - t1[..., W]
    t1 = Yphi(t1 / (2 * g))
    t2 = b.ZA(Kp * b.v * cos[:, None])
    t2 = t2[..., N] - t2[..., S]
    t2 = t2 / (2 * g)
    t3 = b.AA(Kp * b.omega) / (2 * g)
    out["BKe"] = term("BKe", t1, t2, t3)
    # calc_boz :328-370 (no E-W difference, sic)
    t1 = (b.v_ZA * b.geopt_AE) / g
    t1 = Yphi(t1)
    t2 = (b.v_ZA * b.geopt_AE) * cos / g
    t2 = t2[..., N] - t2[..., S]
    t3 = b.AAz(b.omega_AE * b.geopt_AE) / g
    out["BΦZ"] = term("BΦZ", t1, t2, t3)
    # calc_boe :372-418 (v_ZE*geopt_AE and BPhiZ's N-S term, sic)
    t1 = (b.v_ZE * b.geopt_AE[..., None]) / g
    t1 = t1[..., E] - t1[..., W]
    t1 = Yphi(t1)
    t2 = (b.v_ZA * b.geopt_AE) * cos / g
    t2 = t2[..., N] - t2[..., S]
    t3 = b.AA(b.omega_ZE * b.geopt_ZE) / g
    out["BΦE"] = term("BΦE", t1, t2, t3)
    return out


def generation_terms(b, lv, raw=None):
    """generation_and_dissipation_terms.py:122-152 (Gz, Ge).  ``raw``: as in :func:`energy_contents`."""
    s = b.sigma_AA
    F = _Families(lv, raw)
    out = {}
    out["Gz"] = F.integrate("Gz", b.AAz(b.Q_AE * b.tair_AE) / (Cp_d * s), b.p)
    out["Ge"] = F.integrate("Ge", b.AA(b.Q_ZE * b.tair_ZE) / (Cp_d * s), b.p)
    return out


def dissipation_terms(b, ust):
    """generation_and_dissipation_terms.py:154-188 ("still needs to be fully implemented and tested"; never run
    by a bundled case: UNPINNED).  ``ust`` = the box slice of the "Friction Velocity" field, [t][j][i]; the same
    field serves as both stress components (box_data.py:189-195).  Dz as written; De with the zonal mean its area
    average needs (as written, CalcAreaAverage(term, ylength) of a (t, lat, lon) array returns (t, lon))."""
    ust_ZA = b.ZA(ust)
    ust_ZE = ust - ust_ZA[..., None]
    u0_ZA, v0_ZA = b.u_ZA[:, 0], b.v_ZA[:, 0]                       # isel(level=0): first level of the sorted axis
    Dz = b.AAz(u0_ZA * ust_ZA + v0_ZA * ust_ZA) / g
    De = b.AA(b.u_ZE[:, 0] * ust_ZE + b.v_ZE[:, 0] * ust_ZE) / g
    return {"Dz": Dz, "De": De}


# --------------------------------------------------------------------------- #
# calc_budget_and_residual.py
# --------------------------------------------------------------------------- #
def calc_budget_diff(df, dates):
    """calc_budget_and_residual.py:32-56."""
    dt = float((dates[1] - dates[0]) / np.timedelta64(1, "s"))
    for term in ["Az", "Ae", "Kz", "Ke"]:
        df[f"∂{term}/∂t (finite diff.)"] = np.gradient(df[term], dt)
    return df


def calc_residuals(df):
    """calc_budget_and_residual.py:131-154."""
    df["RGz"] = df["∂Az/∂t (finite diff.)"] + df["Cz"] + df["Ca"] - df["BAz"]
    df["RKz"] = df["∂Kz/∂t (finite diff.)"] - df["Cz"] - df["Ck"] - df["BKz"]
    df["RGe"] = df["∂Ae/∂t (finite diff.)"] - df["Ca"] + df["Ce"] - df["BAe"]
    df["RKe"] = df["∂Ke/∂t (finite diff.)"] - df["Ce"] + df["Ck"] - df["BKe"]
    return df


# --------------------------------------------------------------------------- #
# frameworks
# --------------------------------------------------------------------------- #
FIXED_COLUMNS = ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe", "Gz", "Ge"]
MOVING_COLUMNS = ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe",
                  "BΦZ", "BΦE", "Gz", "Ge"]


def lec_fixed(P, min_lon, max_lon, min_lat, max_lat, mode="ref", legacy_0d=False):
    """``lec_fixed`` body (lec_fixed_framework.py:199-303), ``-r`` flavour.

    ``P`` is the output of :func:`process_data` + :func:`slice_domain_fixed`.
    Returns ``(df, levels, extra)``: the results DataFrame (reference column
    order), the per-level dict ``name -> [t][k]`` (or ``[k]`` for Cz_1/Ce_1)
    and the B-Phi terms the reference computes and then drops.
    """
    P = to_mode(P, mode)
    b = BoxState(P, min_lon, max_lon, min_lat, max_lat, fixed=True)
    lv = {}
    terms = {}
    terms.update(energy_contents(b, lv))
    terms.update(conversion_terms(b, lv))
    bt = boundary_terms(b, legacy_0d=legacy_0d)
    terms.update(bt)
    terms.update(generation_terms(b, lv))
    df = pd.DataFrame(index=P.time.astype("datetime64[ns]"))
    for c in FIXED_COLUMNS:
        df[c] = np.asarray(terms[c], dtype=np.float64)
    df = calc_budget_diff(df, P.time)
    df = calc_residuals(df)
    extra = {"BΦZ": bt["BΦZ"], "BΦE": bt["BΦE"], "box": b}
    return df, lv, extra


# --------------------------------------------------------------------------- #
# MetPy 1.6.2 ``vorticity`` on a latitude / longitude grid (lec_moving_framework.py:660-663), restated from
# the published source (metpy/calc/kinematics.py: vorticity, vector_derivative; metpy/calc/tools.py:
# parse_grid_arguments, nominal_lat_lon_grid_deltas, first_derivative; metpy/xarray.py: grid_deltas).  MetPy
# and pyproj are not importable in this image: PARITY UNPINNED (no reference output carries these columns).
#   dx = a * diff(lon [rad])                                  "nominal" spacing on the equator
#   dy = geodesic distance between (0, lat_j) and (0, lat_j+1)  = meridian arc on the ellipsoid
#   parallel_scale k = sqrt(1 - e^2 sin^2 phi) / cos phi,  meridional_scale h = (1 - e^2 sin^2 phi)^(3/2) / (1 - e^2)
#       (PROJ pj_factors of the geographic "projection" x = lambda, y = phi; ellipsoid of CRS('+proj=latlon'):
#        PROJ's default GRS80)
#   dv/dx = k * d(v)/dx + u * (h / k) * d(k)/dy ,   du/dy = h * d(u)/dy + v * (k / h) * d(h)/dx ,
#   zeta = dv/dx - du/dy, every derivative MetPy's 3-point first_derivative (second-order one-sided at the ends).
GRS80_A = 6378137.0
GRS80_F = 1.0 / 298.257222101
GRS80_E2 = GRS80_F * (2.0 - GRS80_F)
_GL8_X = np.array([-0.9602898564975363, -0.7966664774136267, -0.5255324099163290, -0.1834346424956498,
                   0.1834346424956498, 0.5255324099163290, 0.7966664774136267, 0.9602898564975363])
_GL8_W = np.array([0.1012285362903763, 0.2223810344533745, 0.3137066458778873, 0.3626837833783620,
                   0.3626837833783620, 0.3137066458778873, 0.2223810344533745, 0.1012285362903763])


def metpy_latlon_factors(lon_deg, lat_deg):
    """``(dx[nlon-1], dy[nlat-1], parallel_scale[nlat], meridional_scale[nlat])`` of a 1-D lat / lon grid in
    float64 from the stored coordinate values (``nominal_lat_lon_grid_deltas`` + ``Proj.get_factors``).  The
    meridian arc (what ``Geod.inv`` returns along a meridian, signed by the forward azimuth) is integrated with
    an 8-point Gauss-Legendre rule per interval: exact to rounding for grid spacings of a few degrees."""
    lon = np.asarray(lon_deg, dtype=np.float64) * (np.pi / 180.0)
    phi = np.asarray(lat_deg, dtype=np.float64) * (np.pi / 180.0)
    dx = GRS80_A * np.diff(lon)
    half = 0.5 * (phi[1:] - phi[:-1])
    mid = 0.5 * (phi[1:] + phi[:-1])
    x = mid[:, None] + half[:, None] * _GL8_X[None, :]
    M = GRS80_A * (1.0 - GRS80_E2) / (1.0 - GRS80_E2 * np.sin(x) ** 2) ** 1.5
    dy = half * np.sum(M * _GL8_W[None, :], axis=1)
    t = 1.0 - GRS80_E2 * np.sin(phi) ** 2
    return dx, dy, np.sqrt(t) / np.cos(phi), t * np.sqrt(t) / (1.0 - GRS80_E2)


def metpy_first_derivative(f, delta, axis):
    """``metpy.calc.first_derivative(f, delta=delta, axis=axis)``: 3-point differences on unevenly spaced
    points, centred in the interior, one-sided (still 3 points) at both ends."""
    f = np.moveaxis(np.asarray(f, dtype=np.float64), axis, -1)
    d = np.asarray(delta, dtype=np.float64)
    d0, d1 = d[:-1], d[1:]
    comb = d0 + d1
    center = (-d1 / (comb * d0) * f[..., :-2] + (d1 - d0) / (d0 * d1) * f[..., 1:-1] + d0 / (comb * d1) * f[..., 2:])
    d0, d1 = d[:1], d[1:2]
    comb = d0 + d1
    big = comb + d0
    left = -big / (comb * d0) * f[..., :1] + comb / (d0 * d1) * f[..., 1:2] - d0 / (comb * d1) * f[..., 2:3]
    d0, d1 = d[-2:-1], d[-1:]
    comb = d0 + d1
    big = comb + d1
    right = d1 / (comb * d0) * f[..., -3:-2] - comb / (d0 * d1) * f[..., -2:-1] + big / (comb * d1) * f[..., -1:]
    return np.moveaxis(np.concatenate((left, center, right), axis=-1), -1, axis)


def metpy_vorticity(u, v, lon_deg, lat_deg):
    """``metpy.calc.vorticity(u, v)`` for ``[...][lat][lon]`` arrays on a 1-D lat / lon grid (m/s -> 1/s)."""
    u = np.asarray(u, dtype=np.float64)
    v = np.asarray(v, dtype=np.float64)
    dx, dy, ps, ms = metpy_latlon_factors(lon_deg, lat_deg)
    P = np.broadcast_to(ps[:, None], u.shape[-2:])
    Mm = np.broadcast_to(ms[:, None], u.shape[-2:])
    dudy = metpy_first_derivative(u, dy, -2)
    dvdx = metpy_first_derivative(v, dx, -1)
    dpdy = metpy_first_derivative(P, dy, -2)
    dmdx = metpy_first_derivative(Mm, dx, -1)
    dx_correction = Mm / P * dpdy
    dy_correction = P / Mm * dmdx
    dudy = Mm * dudy + v * dy_correction
    dvdx = P * dvdx + u * dx_correction
    return dvdx - dudy


def diag850(u, v, z, lon_deg, lat_deg, boxes, scale=(1.0, 1.0, 1.0), z_div=1.0, centres=None):
    """850-hPa track diagnostics (lec_moving_framework.py:650-663 wind speed and MetPy vorticity over the
    pre-sliced domain; :269-417 get_position; tools.py:95-128 find_extremum_coordinates), float64.
    ``u, v, z``: [slot][lat][lon] planes of the 850-hPa level; ``boxes``: (slot, i0, i1, j0, j1) per step,
    inclusive label-slice indices; ``centres``: optional (ic, jc) per step -- the grid point nearest to the
    track centre, where ``-z`` takes the vorticity (:317-324).
    Returns values[n, 5] (zeta nanmin, zeta nanmax, hgt nanmin, wind nanmax, zeta at the centre or NaN) and the
    flat argmin/argmax indices[n, 4] of the box in the same order."""
    u = np.asarray(u, dtype=np.float64) * scale[0]
    v = np.asarray(v, dtype=np.float64) * scale[1]
    hgt = np.asarray(z, dtype=np.float64) * scale[2] / z_div
    zeta = metpy_vorticity(u, v, lon_deg, lat_deg)
    wspd = np.sqrt(u * u + v * v)
    vals = np.full((len(boxes), 5), np.nan); idx = np.empty((len(boxes), 4), dtype=np.int32)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)          # all-NaN boxes
        for n, (s, i0, i1, j0, j1) in enumerate(boxes):
            zb, hb, wb = (a[s, j0:j1 + 1, i0:i1 + 1] for a in (zeta, hgt, wspd))
            vals[n, :4] = np.nanmin(zb), np.nanmax(zb), np.nanmin(hb), np.nanmax(wb)
            idx[n] = zb.argmin(), zb.argmax(), hb.argmin(), wb.argmax()
            if centres is not None and centres[n][0] >= 0:
                vals[n, 4] = zeta[s, centres[n][1], centres[n][0]]
    return vals, idx


def get_limits(track, t):
    """``get_limits`` track branch (lec_moving_framework.py:199-266)."""
    closest = int(np.argmin(np.abs(track.index - t)))
    row = track.iloc[closest]
    clat, clon = row["Lat"], row["Lon"]
    width = row.get("width", 15)
    length = row.get("length", 15)
    return {
        "central_lat": clat, "central_lon": clon, "length": length, "width": width,
        "min_lon": clon - (width / 2), "max_lon": clon + (width / 2),
        "min_lat": clat - (length / 2), "max_lat": clat + (length / 2),
    }


def lec_moving(P, track, mode="ref", legacy_0d=False, residuals=True):
    """``lec_moving`` (lec_moving_framework.py:546-750) + the global dTdt of
    ``run_lec_analysis`` (lorenzcycletoolkit.py:184-186).

    ``P`` is the output of :func:`process_data` (with the track) +
    :func:`slice_domain_track`.
    """
    P = to_mode(P, mode)
    tsec = (P.time - P.time.min()) / np.timedelta64(1, "s")
    dTdt = differentiate(P.fields["Air Temperature"], tsec, 0)
    rows, lvs, boxes = [], [], []
    times = pd.to_datetime(P.time)
    for it, t in enumerate(times):
        lim = get_limits(track, t)
        b = BoxState(P, lim["min_lon"], lim["max_lon"], lim["min_lat"], lim["max_lat"],
                     fixed=False, dTdt=dTdt[it], tsel=it)
        lv = {}
        terms = {}
        terms.update(energy_contents(b, lv))
        terms.update(conversion_terms(b, lv))
        terms.update(boundary_terms(b, legacy_0d=legacy_0d))
        terms.update(generation_terms(b, lv))
        rows.append({c: float(terms[c]) for c in MOVING_COLUMNS})
        lvs.append(lv)
        boxes.append((lim, b.idx))
    df = pd.DataFrame(rows, index=times, dtype=float)[MOVING_COLUMNS]
    df = calc_budget_diff(df, P.time)
    if residuals:
        df = calc_residuals(df)
    def _stack(k):
        rows = [np.asarray(lv[k]) for lv in lvs]
        if len({r.shape for r in rows}) == 1:
            return np.stack(rows)
        return rows          # ragged: _handle_nans dropped different levels at different steps
    levels = {k: _stack(k) for k in lvs[0]}
    return df, levels, boxes
