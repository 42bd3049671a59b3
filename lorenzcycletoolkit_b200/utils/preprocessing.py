"""Host plumbing in front of the CUDA engine: the semantics of the reference's
``src/utils/preprocessing.py`` (``get_data`` :35, ``process_data`` :149, ``prepare_data``
:374) and of ``slice_domain`` (``src/utils/select_area.py:254-338``), on a numpy-backed
dataset instead of ``xarray`` (xarray/netCDF4 are not importable in this image).

The result of :func:`prepare_data` is the layout contract of the engine (SURVEY.md 3.5):
C-contiguous ``[time][level ascending, Pa][lat ascending][lon ascending]`` fields, levels
>= 1000 Pa, and ``rlats / coslats / rlons`` computed in the coordinate's own dtype.
"""

from __future__ import annotations

import logging
from dataclasses import dataclass, field

import numpy as np
import pandas as pd

FIELD_ROWS = ("Air Temperature", "Geopotential", "Geopotential Height", "Omega Velocity",
              "Eastward Wind Component", "Northward Wind Component")
# rows only the (host-side, unfinished in the reference) Dz / De terms read: a namelist that names one switches
# the loader to its eager host layout
EXTRA_ROWS = ("Friction Velocity",)

_LEVEL_TO_PA = {"pa": 1.0, "pascal": 1.0, "pascals": 1.0, "hpa": 100.0, "millibar": 100.0,
                "millibars": 100.0, "mbar": 100.0, "mb": 100.0}

_SECONDS = {"second": 1.0, "seconds": 1.0, "sec": 1.0, "s": 1.0, "minute": 60.0, "minutes": 60.0,
            "hour": 3600.0, "hours": 3600.0, "hr": 3600.0, "h": 3600.0, "day": 86400.0, "days": 86400.0}


@dataclass
class RawStore:
    """Fields still in FILE layout plus what the host pipeline has decided about them so far: every
    transform of ``process_data`` / ``slice_domain`` only edits the index maps, the records themselves
    go to the GPU as stored (``lec_run_host_raw`` decodes and re-orders them there)."""
    fields: dict                     # var -> raw [record][level][lat][lon] (int16/float32/float64, any byte order)
    decode: dict                     # var -> dict(scale=, offset=, fills=[...], float32=bool)
    rec: np.ndarray                  # dataset time index  -> raw record
    lev: np.ndarray                  # dataset level index -> raw level
    lat: np.ndarray
    lon: np.ndarray

    def select(self, axis, sel):
        maps = {"rec": self.rec, "lev": self.lev, "lat": self.lat, "lon": self.lon}
        maps[axis] = np.atleast_1d(maps[axis][sel])
        return RawStore(self.fields, self.decode, **maps)

    def dtype_of(self, var):
        return decoded_dtype(self.fields[var].dtype, self.decode[var])

    def materialise(self, var, level=None):
        """The array the eager pipeline would hold for ``var`` (one dataset level if ``level`` is given)."""
        lev = self.lev if level is None else self.lev[level:level + 1]
        out = apply_decode(self.fields[var][np.ix_(self.rec, lev, self.lat, self.lon)], self.decode[var])
        return out if level is None else out[:, 0]

    def plane_windows(self, var, level, times, origins, rows, cols):
        """``materialise(var, level)[t, y0:y0 + rows, x0:x0 + cols]`` for each ``t`` of ``times`` with its origin
        ``(x0, y0)`` of ``origins``, decoding only those points: ``[len(times)][rows][cols]``."""
        raw = self.fields[var]
        out = [apply_decode(raw[np.ix_(self.rec[[t]], self.lev[[level]], self.lat[y0:y0 + rows],
                                       self.lon[x0:x0 + cols])], self.decode[var])[0, 0]
               for t, (x0, y0) in zip(times, origins)]
        return np.stack(out) if out else np.zeros((0, rows, cols))


def decode_rule(stored_dtype, attrs):
    """The CF decode of a variable stored as ``stored_dtype`` with attributes ``attrs`` (what ``xr.open_dataset``
    applies, preprocessing.py:35-147): ``dict(scale=, offset=, fills=[...], float32=)`` as :class:`RawStore` and
    ``LecEngine.run_host_raw`` take it, or None for a variable that is not decoded (a plain integer or a
    non-numeric one).  Integers with a ``scale_factor`` and/or ``add_offset`` are unpacked, to float32 when the
    stored type has at most 2 bytes and there is no offset, else to float64; stored floats are only masked.
    ``_FillValue`` / ``missing_value`` entries are kept as values of the stored type, and only those the type holds
    exactly: no stored value equals one it cannot hold (the device compares in the stored type too)."""
    dt = np.dtype(stored_dtype).newbyteorder("=")
    scale, offset = attrs.get("scale_factor"), attrs.get("add_offset")
    if dt.kind not in "iuf" or (dt.kind != "f" and scale is None and offset is None):
        return None
    if dt.kind == "f":
        scale = offset = None
    fills = []
    with np.errstate(invalid="ignore", over="ignore"):
        for fv in (x for k in ("_FillValue", "missing_value") if k in attrs for x in np.atleast_1d(attrs[k]).ravel()):
            held = fv.astype(dt)
            if held == fv:
                fills.append(held)
    return dict(scale=None if scale is None else np.float64(scale), offset=None if offset is None else np.float64(offset),
                fills=fills, float32=dt.kind != "f" and dt.itemsize <= 2 and offset is None)


def decoded_dtype(stored_dtype, rule):
    """The dtype :func:`apply_decode` gives a variable stored as ``stored_dtype`` under ``rule``."""
    if rule is None or stored_dtype.kind == "f":
        return stored_dtype.newbyteorder("=")
    return np.dtype(np.float32 if rule["float32"] else np.float64)


def apply_decode(raw, rule):
    """``raw`` decoded by ``rule`` (:func:`decode_rule`) on the host, a new native-endian array: fill values to NaN,
    then an in-place multiply by the scale and an in-place add of the offset in the decoded dtype -- xarray's
    operations, which ``lec_ingest_kernel`` reproduces bit for bit."""
    out = raw.astype(decoded_dtype(raw.dtype, rule))
    if rule is not None:
        for fv in rule["fills"]:
            out[raw == fv] = np.nan
        if rule["scale"] is not None:
            out *= rule["scale"]
        if rule["offset"] is not None:
            out += rule["offset"]
    return out


def raw_store(fields, order):
    """A :class:`RawStore` over ``fields`` = ``{var: (array as stored, dims, decode_rule)}``, or None when the
    device cannot decode them and the host path has to: every field stored in ``order`` (the engine's dimension
    order), one shape and one dtype for all, that dtype int16 / float32 / float64 in either byte order, at most two
    fill values, integers packed (a scale or an offset) and floats not."""
    arrays = [a for a, _, _ in fields.values()]
    first = arrays[0]
    if not all(dims == order and rule is not None and len(rule["fills"]) <= 2 and a.dtype == first.dtype and
               a.shape == first.shape and (a.dtype.kind == "i") == (rule["scale"] is not None or rule["offset"] is not None)
               for a, dims, rule in fields.values()):
        return None
    if first.dtype.newbyteorder("=") not in (np.dtype(np.int16), np.dtype(np.float32), np.dtype(np.float64)):
        return None
    nrec, nlev, nlat, nlon = first.shape
    return RawStore({v: a for v, (a, _, _) in fields.items()}, {v: rule for v, (_, _, rule) in fields.items()},
                    np.arange(nrec), np.arange(nlev), np.arange(nlat), np.arange(nlon))


def _engine_order(var, data, dims, order, surface=False):
    """``data`` with dimensions ``dims`` transposed to ``order``; with ``surface``, a field without a level dimension
    goes to (time, lat, lon)."""
    want = (order[0], order[2], order[3]) if surface and len(dims) == 3 else order
    if sorted(dims) != sorted(want):
        raise ValueError(f"{var} has dimensions {dims}, expected a permutation of {want}")
    return np.transpose(data, [dims.index(d) for d in want])


def packed_device_fields(store: RawStore, names, device="cuda"):
    """Five int16 fields of a raw-backed dataset made resident on the GPU, still packed (2 bytes per value), for
    ``LecEngine.run_torch_packed``: ``[time][level][lat][pitch]`` in the dataset's order (the store's record, level,
    row and column maps applied), native byte order, rows padded with zeros to a pitch of a multiple of 8 elements.
    A one-time load: one host gather and byte swap per time slot and field, then one copy to the device.  Returns
    ``(tensors, decode)``; ``decode`` is the per-field rule of ``store.decode``.  Fields that are not int16, or whose
    packing the decode rule cannot express (more than two fill values, a fill value that is not an int16 value, a
    scale or offset that is not finite), raise ``ValueError``."""
    import torch
    nlon = len(store.lon)
    pitch = (nlon + 7) // 8 * 8
    decode = []
    for v in names:
        raw, dec = store.fields[v], store.decode[v]
        if raw.dtype.kind != "i" or raw.dtype.itemsize != 2:
            raise ValueError(f"{v} is stored as {raw.dtype}, not int16: packed device fields need int16 records")
        fills = list(dec.get("fills", ()))
        if len(fills) > 2 or not all(np.isfinite(float(x)) and float(x) == int(x) and -32768 <= int(x) <= 32767
                                     for x in fills):
            raise ValueError(f"{v}: fill values {fills} cannot be matched against int16 records")
        for k in ("scale", "offset"):
            if dec.get(k) is not None and not np.isfinite(float(dec[k])):
                raise ValueError(f"{v}: {k} {dec[k]} is not finite")
        decode.append(dict(dec))
    out = []
    for v in names:
        raw = store.fields[v]
        t = torch.zeros((len(store.rec), len(store.lev), len(store.lat), pitch), dtype=torch.int16, device=device)
        host = np.zeros((len(store.lev), len(store.lat), pitch), dtype=np.int16)
        for s, r in enumerate(store.rec):
            host[:, :, :nlon] = raw[r][np.ix_(store.lev, store.lat, store.lon)]     # gather + byte swap to native
            t[s].copy_(torch.from_numpy(host))
        out.append(t)
    return out, decode


class _LazyVariables(dict):
    """``LecDataset.variables`` of a raw-backed dataset: decoded and re-ordered on first access."""

    def __init__(self, store):
        super().__init__()
        self.store = store

    def __missing__(self, key):
        if key not in self.store.fields:
            raise KeyError(key)
        self[key] = self.store.materialise(key)
        return self[key]

    def __contains__(self, key):
        return key in self.store.fields

    def keys(self):
        return self.store.fields.keys()

    def __iter__(self):
        return iter(self.store.fields)

    def __len__(self):
        return len(self.store.fields)

    def items(self):
        return [(k, self[k]) for k in self.store.fields]


@dataclass
class LecDataset:
    """A small stand-in for the ``xr.Dataset`` the reference passes around: variables are
    numpy arrays ``[time][level][lat][lon]`` keyed by their file names, coordinates are 1-D
    arrays, ``names`` maps the namelist's coordinate rows to variable names."""
    variables: dict = field(default_factory=dict)
    time: np.ndarray = None          # datetime64[ns]
    level: np.ndarray = None
    lat: np.ndarray = None
    lon: np.ndarray = None
    rlats: np.ndarray = None
    coslats: np.ndarray = None
    rlons: np.ndarray = None
    names: dict = field(default_factory=dict)     # Time / Vertical Level / Latitude / Longitude
    attrs: dict = field(default_factory=dict)     # per-variable attribute dicts
    raw: RawStore = None                          # set while the fields are still in file layout

    def __getitem__(self, key):
        if key in self.variables:
            return self.variables[key]
        for row, attr in (("Time", "time"), ("Vertical Level", "level"), ("Latitude", "lat"), ("Longitude", "lon")):
            if key == self.names.get(row):
                return getattr(self, attr)
        raise KeyError(key)

    def __contains__(self, key):
        try:
            self[key]
            return True
        except KeyError:
            return False

    def compute(self):
        return self

    def _replace(self, **kw):
        d = LecDataset(**{k: getattr(self, k) for k in self.__dataclass_fields__})
        for k, v in kw.items():
            setattr(d, k, v)
        return d

    def isel(self, time=None, level=None, lat=None, lon=None):
        """Positional selection with slices or index arrays (kept 4-D)."""
        out = self._replace(variables=self.variables if self.raw is not None else dict(self.variables))
        for axis, (sel, coords) in enumerate(((time, ("time",)), (level, ("level",)),
                                              (lat, ("lat", "rlats", "coslats")), (lon, ("lon", "rlons")))):
            if sel is None:
                continue
            for c in coords:
                if getattr(out, c) is not None:
                    setattr(out, c, np.atleast_1d(getattr(out, c)[sel]) if out.raw is not None else getattr(out, c)[sel])
            if out.raw is not None:          # only the index map moves
                out.raw = out.raw.select(("rec", "lev", "lat", "lon")[axis], sel)
                out.variables = _LazyVariables(out.raw)
                continue
            def pick(v):                     # 4-D fields (time, level, lat, lon); surface fields (time, lat, lon)
                if v.ndim == 4:
                    ax = axis
                elif axis == 1:
                    return v                 # a surface field has no level axis
                else:
                    ax = axis if axis == 0 else axis - 1
                idx = [slice(None)] * v.ndim
                idx[ax] = sel
                return v[tuple(idx)]
            out.variables = {k: pick(v) for k, v in out.variables.items()}
        return out

    def level_plane_windows(self, var, k, origins, rows, cols, times=None):
        """``level_plane(var, k)[t, y0:y0 + rows, x0:x0 + cols]`` for every time ``t`` (or those of ``times``) with its
        window origin ``(x0, y0)``: ``[n][rows][cols]``.  A raw-backed dataset decodes only those points."""
        times = np.arange(len(origins)) if times is None else np.asarray(times)
        if self.raw is not None and var not in dict.keys(self.variables):
            return self.raw.plane_windows(var, k, times, origins, rows, cols)
        a = self[var]
        return np.stack([np.asarray(a[t, k, y0:y0 + rows, x0:x0 + cols]) for t, (x0, y0) in zip(times, origins)]) \
            if len(times) else np.zeros((0, rows, cols))

    def level_plane(self, var, k):
        """``self[var][:, k]`` without materialising the other levels of a raw-backed dataset."""
        if self.raw is not None and var not in dict.keys(self.variables):
            return self.raw.materialise(var, level=k)
        return np.asarray(self[var])[:, k]

    def load(self):
        """Decode and re-order every field on the host now (the eager layout); drops the raw backing."""
        if self.raw is not None:
            self.variables = {k: np.ascontiguousarray(self.variables[k]) for k in self.raw.fields}
            self.raw = None
        return self


# --------------------------------------------------------------------------------------- #
_STANDARD_CALENDARS = ("standard", "gregorian", "proleptic_gregorian")


def _decode_cf_time(values, units, calendar=None):
    """CF ``<unit> since <reference>`` -> datetime64[ns], standard calendars only (xarray would go through
    cftime for noleap / 360_day / julian axes; decoding those as Gregorian would silently shift the
    track-time selection and the dT/dt spacing, so they are refused)."""
    if calendar is not None and str(calendar).strip().lower() not in _STANDARD_CALENDARS:
        raise ValueError(f"time axis uses the '{calendar}' calendar; only {_STANDARD_CALENDARS} are supported")
    unit, _, ref = units.partition(" since ")
    try:
        per = _SECONDS[unit.strip().lower()]
    except KeyError:
        raise ValueError(f"time units '{units}': unknown unit '{unit.strip()}' "
                         f"(known: {sorted(set(_SECONDS))})") from None
    ref64 = np.datetime64(pd.Timestamp(ref.strip().replace("T", " ")).to_datetime64(), "ns")
    ns = np.round(np.asarray(values, dtype=np.float64) * per * 1e9).astype("int64")
    return ref64 + ns.astype("timedelta64[ns]")


def open_netcdf3(path, variable_list_df, lazy=None):
    """``xr.open_dataset`` for NetCDF-3 classic files (``get_data``, preprocessing.py:35-147):
    ``_FillValue``/``missing_value`` -> NaN, ``scale_factor``/``add_offset`` unpacking (float32
    unless an offset or a wide integer type forces float64), CF time decoding; float32 stays
    float32.  Only the variables the namelist names are read.

    ``lazy`` (default: on unless ``LEC_DEVICE_INGEST=0``): when every field is stored as
    ``[time][level][lat][lon]`` in one of int16 / float32 / float64, the fields are NOT decoded here --
    the dataset keeps the records as stored (:class:`RawStore`) and the GPU decodes them."""
    import os
    from scipy.io import netcdf_file
    if lazy is None:
        lazy = os.environ.get("LEC_DEVICE_INGEST", "1") != "0"

    names = {row: variable_list_df.loc[row]["Variable"] for row in ("Time", "Vertical Level", "Latitude", "Longitude")}
    wanted = [variable_list_df.loc[r]["Variable"] for r in FIELD_ROWS if r in variable_list_df.index]
    extra = [variable_list_df.loc[r]["Variable"] for r in EXTRA_ROWS if r in variable_list_df.index]
    if extra:
        lazy = False
    ds = LecDataset(names=names)
    with netcdf_file(path, mmap=False) as f:
        missing = [v for v in list(names.values()) + wanted if v not in f.variables]
        if missing:
            raise KeyError(f"variables {missing} named by the namelist are not in {path} "
                           f"(file has {sorted(f.variables)})")

        def read(name):          # (data as stored, big-endian, dims, attributes, decode rule)
            v = f.variables[name]
            at = {a: (x.decode() if isinstance(x, bytes) else x) for a, x in ((a, getattr(v, a)) for a in v._attributes)}
            return v.data, tuple(v.dimensions), at, decode_rule(v.data.dtype, at)

        def decode(name):
            data, _, at, rule = read(name)
            return apply_decode(data, rule), at

        t, t_at = decode(names["Time"])
        units = t_at.get("units", "")
        ds.time = _decode_cf_time(t, units, t_at.get("calendar")) if " since " in str(units) else t
        ds.level, ds.attrs[names["Vertical Level"]] = decode(names["Vertical Level"])
        ds.lat, ds.lon = decode(names["Latitude"])[0], decode(names["Longitude"])[0]
        order = (names["Time"], names["Vertical Level"], names["Latitude"], names["Longitude"])
        fields = {var: read(var) for var in wanted}
        store = raw_store({var: (a, dims, rule) for var, (a, dims, _, rule) in fields.items()}, order) if lazy else None
        if store is not None:
            ds.raw, ds.variables = store, _LazyVariables(store)
            ds.attrs.update({var: at for var, (_, _, at, _) in fields.items()})
            return ds
        for var in wanted + extra:           # extra rows: (time, level, lat, lon) or a surface field (time, lat, lon)
            if var not in f.variables:
                raise KeyError(f"variable {var} named by the namelist is not in {path}")
            data, dims, ds.attrs[var], rule = fields[var] if var in fields else read(var)
            ds.variables[var] = _engine_order(var, apply_decode(data, rule), dims, order, surface=var in extra)
    return ds


class _NcVar:
    """What :func:`from_xarray` reads of a variable: ``values`` (as stored, no mask / scale applied), ``dims``, ``attrs``."""

    def __init__(self, values, dims, attrs):
        self.values, self.dims, self.attrs = values, tuple(dims), dict(attrs)


def open_netcdf4(path, variable_list_df, lazy=None):
    """NetCDF-4 (HDF5) input -- what current CDS ERA5 downloads are, ``xr.open_dataset`` in the reference
    (preprocessing.py:74) -- through ``netCDF4`` or ``h5py`` when one of them is importable (neither ships with
    this image; both are optional).  Variables are read AS STORED (no mask-and-scale), so int16-packed fields
    stay raw-backed and are decoded on the GPU like NetCDF-3 records (:func:`from_xarray` does the rest, packed
    coordinates included)."""
    import os
    if lazy is None:
        lazy = os.environ.get("LEC_DEVICE_INGEST", "1") != "0"
    names = [variable_list_df.loc[row]["Variable"] for row in ("Time", "Vertical Level", "Latitude", "Longitude")]
    wanted = names + [variable_list_df.loc[r]["Variable"] for r in FIELD_ROWS + EXTRA_ROWS if r in variable_list_df.index]

    def plain(x):
        x = x.decode() if isinstance(x, bytes) else x
        return x.item() if isinstance(x, np.generic) else x
    ds = {}
    try:
        import netCDF4
    except ImportError:
        netCDF4 = None
    if netCDF4 is not None:
        with netCDF4.Dataset(path, "r") as f:
            f.set_auto_maskandscale(False)
            missing = [v for v in wanted if v not in f.variables]
            if missing:
                raise KeyError(f"variables {missing} named by the namelist are not in {path} (file has {sorted(f.variables)})")
            for v in wanted:
                var = f.variables[v]
                ds[v] = _NcVar(np.asarray(var[...]), var.dimensions, {a: plain(var.getncattr(a)) for a in var.ncattrs()})
    else:
        try:
            import h5py
        except ImportError:
            raise RuntimeError(
                f"{path} is a NetCDF-4 / HDF5 file; reading it needs the `netCDF4` or `h5py` package (neither is "
                "installed).  Convert it with `nccopy -k classic`, or open it with xarray yourself and pass the "
                "dataset through lorenzcycletoolkit_b200.utils.preprocessing.from_xarray") from None
        with h5py.File(path, "r") as f:
            missing = [v for v in wanted if v not in f]
            if missing:
                raise KeyError(f"variables {missing} named by the namelist are not in {path} (file has {sorted(f)})")
            for v in wanted:
                var = f[v]
                dims = [d.label or (var.dims[i][0].name.split("/")[-1] if len(var.dims[i]) else f"dim{i}")
                        for i, d in enumerate(var.dims)]
                attrs = {a: plain(x) for a, x in var.attrs.items()
                         if a not in ("DIMENSION_LIST", "REFERENCE_LIST", "CLASS", "NAME", "_Netcdf4Dimid", "_Netcdf4Coordinates")}
                ds[v] = _NcVar(np.asarray(var[...]), dims, attrs)
    tv = ds[names[0]]
    units = str(tv.attrs.get("units", ""))
    if " since " in units:
        tv.values = _decode_cf_time(tv.values, units, tv.attrs.get("calendar"))
    return from_xarray(ds, variable_list_df, lazy=lazy)


def open_dataset(path, variable_list_df, lazy=None):
    """``xr.open_dataset(infile)`` of the reference (preprocessing.py:73-74) by file signature: NetCDF-3 classic /
    64-bit offset through scipy, NetCDF-4 (HDF5) through netCDF4 / h5py."""
    with open(path, "rb") as f:
        magic = f.read(8)
    if magic[:3] == b"CDF":
        return open_netcdf3(path, variable_list_df, lazy=lazy)
    if magic == b"\x89HDF\r\n\x1a\n":
        return open_netcdf4(path, variable_list_df, lazy=lazy)
    raise ValueError(f"{path}: neither a NetCDF-3 (CDF) nor a NetCDF-4 / HDF5 file")


def from_xarray(ds, variable_list_df, lazy=True):
    """Adaptor for the reference's own loader: an ``xr.Dataset`` (``xr.open_dataset(infile)`` as in
    ``get_data``, preprocessing.py:35-147, or opened with ``mask_and_scale=False`` to keep packed int16
    records) -> :class:`LecDataset`, ready for :func:`process_data` / :func:`slice_domain`.  Duck-typed: only
    ``ds[name].values / .dims / .attrs`` are used, so xarray itself is not imported here.  Fields stored as
    ``(time, level, lat, lon)`` in one of int16 / float32 / float64 stay raw-backed (``lazy``); anything
    else is decoded and transposed on the host."""
    names = {row: variable_list_df.loc[row]["Variable"] for row in ("Time", "Vertical Level", "Latitude", "Longitude")}
    wanted = [variable_list_df.loc[r]["Variable"] for r in FIELD_ROWS if r in variable_list_df.index]
    extra = [variable_list_df.loc[r]["Variable"] for r in EXTRA_ROWS if r in variable_list_df.index]
    out = LecDataset(names=names)

    def read(name):                       # (values as stored, dims, attributes, decode rule)
        a, at = np.asarray(ds[name].values), dict(ds[name].attrs)
        return a, tuple(ds[name].dims), at, decode_rule(a.dtype, at)
    t = np.asarray(ds[names["Time"]].values)
    out.time = t.astype("datetime64[ns]") if np.issubdtype(t.dtype, np.datetime64) else t
    for row, attr in (("Vertical Level", "level"), ("Latitude", "lat"), ("Longitude", "lon")):
        a, _, at, rule = read(names[row])
        setattr(out, attr, apply_decode(a, rule))
    out.attrs[names["Vertical Level"]] = dict(ds[names["Vertical Level"]].attrs)
    order = (names["Time"], names["Vertical Level"], names["Latitude"], names["Longitude"])
    fields = {var: read(var) for var in wanted}
    for var, (_, _, at, _) in fields.items():
        out.attrs[var] = at
    store = raw_store({var: (a, dims, rule) for var, (a, dims, _, rule) in fields.items()}, order) \
        if lazy and not extra else None
    if store is not None:
        def contiguous_records(a):        # the ABI wants every record C-contiguous
            return a if a.strides[1:] == np.empty(a.shape[1:], a.dtype).strides and a.strides[0] > 0 else np.ascontiguousarray(a)
        store.fields = {v: contiguous_records(a) for v, a in store.fields.items()}
        out.raw, out.variables = store, _LazyVariables(store)
        return out
    for var in wanted + extra:            # extra rows: (time, level, lat, lon) or a surface field (time, lat, lon)
        a, dims, out.attrs[var], rule = fields[var] if var in fields else read(var)
        out.variables[var] = _engine_order(var, apply_decode(a, rule), dims, order, surface=var in extra)
    return out


def read_namelist(path):
    """``pd.read_csv(namelist, sep=";", index_col=0, header=0)`` (lorenzcycletoolkit.py:175)."""
    df = pd.read_csv(path, sep=";", index_col=0, header=0)
    for row in ("Air Temperature", "Omega Velocity", "Eastward Wind Component", "Northward Wind Component",
                "Longitude", "Latitude", "Time", "Vertical Level"):
        if row not in df.index:
            raise ValueError(f"namelist {path} has no '{row}' row")
    if "Geopotential" not in df.index and "Geopotential Height" not in df.index:
        raise ValueError(f"namelist {path} needs a 'Geopotential' or 'Geopotential Height' row")
    return df


def read_track(path):
    """Track file ``time;Lat;Lon[;length;width;...]`` with ``%Y-%m-%d-%H%M`` times
    (preprocessing.py:176-182; validation.py:28-164 rejects any other date format)."""
    tr = pd.read_csv(path, delimiter=";", index_col="time")
    for col in ("Lat", "Lon"):
        if col not in tr.columns:
            raise ValueError(f"track file {path} has no '{col}' column")
    try:
        tr.index = pd.to_datetime(tr.index, format="%Y-%m-%d-%H%M")
    except ValueError as e:
        raise ValueError(f"track file {path}: times must look like 2005-08-08-0600") from e
    return tr


def read_box_limits(path):
    """``inputs/box_limits``: four ``key;value`` rows (lec_fixed_framework.py:59-154)."""
    df = pd.read_csv(path, header=None, delimiter=";", index_col=0)
    missing = [k for k in ("min_lon", "max_lon", "min_lat", "max_lat") if k not in df.index]
    if missing:
        raise ValueError(f"Box limits file missing required fields: {missing}. Found: {list(df.index)}")
    lim = {k: float(df.loc[k].iloc[0]) for k in ("min_lon", "max_lon", "min_lat", "max_lat")}
    if lim["min_lon"] > lim["max_lon"]:
        raise ValueError(f"Invalid box_limits: min_lon ({lim['min_lon']}) > max_lon ({lim['max_lon']}). Check {path}")
    if lim["min_lat"] > lim["max_lat"]:
        raise ValueError(f"Invalid box_limits: min_lat ({lim['min_lat']}) > max_lat ({lim['max_lat']}). Check {path}")
    return lim


# --------------------------------------------------------------------------------------- #
def _label_slice(coord, lo, hi):
    """``.sel(dim=slice(lo, hi))`` on an increasing index: inclusive at both ends."""
    return slice(int(np.searchsorted(coord, lo, side="left")), int(np.searchsorted(coord, hi, side="right")))


def process_data(data: LecDataset, args, variable_list_df, app_logger=None) -> LecDataset:
    """``process_data`` (preprocessing.py:149-371)."""
    log = app_logger or logging.getLogger("lorenzcycletoolkit")
    time = data.time
    if getattr(args, "track", False):
        log.debug("📅 Selecting only data matching the track dates... ")
        track = read_track(args.trackfile)
        data_dt = int((time[1] - time[0]) / np.timedelta64(1, "h"))
        track_dt = int((track.index[1] - track.index[0]) / np.timedelta64(1, "h"))
        if data_dt > track_dt:
            raise ValueError(f"Data time step ({data_dt}h) is higher than track time step ({track_dt}h). "
                             "Cannot select track timesteps that don't exist in data.")
        if track.index[0] < time[0]:
            raise ValueError(f"Track initial timestamp ({track.index[0]}) is earlier than data initial "
                             f"timestamp ({time[0]}).")
        if track.index[-1] > time[-1]:
            raise ValueError(f"Track final timestamp ({track.index[-1]}) is later than data final "
                             f"timestamp ({time[-1]}).")
        if getattr(args, "cdsapi", False):
            track = track[track.index.hour % data_dt == 0]
        sel = pd.Index(time).get_indexer(track.index.values)
        if (sel < 0).any():
            raise KeyError(f"track times {list(track.index[sel < 0])} are not in the data")
        data = data.isel(time=sel)

    lon = data.lon
    if lon.min() < -180 or lon.max() > 180:                      # tools.py:76-92
        lon = (lon + 180) % 360 - 180
        order = np.argsort(lon, kind="stable")
        data = data._replace(lon=lon).isel(lon=order)

    # radians in the coordinate's own dtype (:288-290)
    data = data._replace(rlats=np.deg2rad(data.lat), coslats=np.cos(np.deg2rad(data.lat)),
                         rlons=np.deg2rad(data.lon))

    lev_name = data.names["Vertical Level"]
    units = data.attrs.get(lev_name, {}).get("units")
    if units is None:
        log.warning(f"⚠️  Vertical level coordinate '{lev_name}' has no units attribute. Assuming hPa (hectopascals).")
        units = "hPa"
    fac = _LEVEL_TO_PA.get(str(units).strip().lower())
    if fac is None:
        raise ValueError(f"Cannot convert vertical level units to Pa. Check if '{lev_name}' has valid pressure units.")
    data = data._replace(level=data.level * fac if fac != 1.0 else data.level)

    data = data.isel(lon=np.argsort(data.lon, kind="stable"))
    data = data.isel(level=np.argsort(data.level, kind="stable"))
    data = data.isel(lat=np.argsort(data.lat, kind="stable"))
    data = data.isel(level=_label_slice(data.level, 1000, float(data.level.max())))   # :364-365
    if data.raw is None:
        data.variables = {k: np.ascontiguousarray(v) for k, v in data.variables.items()}
    return data


def slice_domain(data: LecDataset, args, variable_list_df, box_limits_file="inputs/box_limits") -> LecDataset:
    """``slice_domain`` (select_area.py:254-338).  Fixed: crop to the nearest grid values of the
    limits in ``inputs/box_limits`` (the reference hard-codes that path even when ``--box_limits``
    points elsewhere); track: track extent +- (max width / 2 + one grid step)."""
    from ..engine import nearest_index

    if getattr(args, "fixed", False):
        lim = read_box_limits(box_limits_file)
        W = data.lon[nearest_index(data.lon, lim["min_lon"])]
        E = data.lon[nearest_index(data.lon, lim["max_lon"])]
        S = data.lat[nearest_index(data.lat, lim["min_lat"])]
        N = data.lat[nearest_index(data.lat, lim["max_lat"])]
    elif getattr(args, "track", False):
        dx, dy = data.lon[1] - data.lon[0], data.lat[1] - data.lat[0]
        track = read_track(args.trackfile if getattr(args, "trackfile", None) else "inputs/track")
        if "width" in track.columns:
            mw, ml = track["width"].max(), track["length"].max()
        else:
            mw, ml = 15, 15
        W, E = track["Lon"].min() - mw / 2 - dx, track["Lon"].max() + mw / 2 + dx
        S, N = track["Lat"].min() - ml / 2 - dy, track["Lat"].max() + ml / 2 + dy
    else:
        raise NotImplementedError("the interactive --choose framework needs a display (out of scope)")
    out = data.isel(lat=_label_slice(data.lat, S, N), lon=_label_slice(data.lon, W, E))
    if out.raw is None:
        out.variables = {k: np.ascontiguousarray(v) for k, v in out.variables.items()}
    return out


def prepare_data(args, varlist="inputs/namelist", app_logger=None, box_limits_file="inputs/box_limits") -> LecDataset:
    """``prepare_data`` (preprocessing.py:374-413): namelist -> open -> process -> pre-crop."""
    log = app_logger or logging.getLogger("lorenzcycletoolkit")
    variable_list_df = read_namelist(varlist)
    data = open_dataset(args.infile, variable_list_df)
    data = process_data(data, args, variable_list_df, log)
    sliced = slice_domain(data, args, variable_list_df, box_limits_file)
    log.debug("✅ Data prepared.")
    return sliced
