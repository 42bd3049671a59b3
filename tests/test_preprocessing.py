"""CPU tests of the host plumbing (product code) against the oracle's restatement and the
reference's input formats."""
import argparse
import os

import numpy as np
import pytest

from oracle import lec_oracle as O
import helpers as H
from lorenzcycletoolkit_b200.utils import preprocessing as PP
from lorenzcycletoolkit_b200.utils import calc_budget_and_residual as CB

INP = os.path.join(H.GOLDEN, "inputs")
SAM = os.path.join(H.GOLDEN, "samples")


def _args(**kw):
    d = dict(infile=os.path.join(SAM, "testdata_NCEP-R2.nc"), fixed=False, track=False, choose=False,
             residuals=True, cdsapi=False, mpas=False, trackfile=None, box_limits=None)
    d.update(kw)
    return argparse.Namespace(**d)


def _same(P, d):
    assert np.array_equal(P.lon, d.lon) and np.array_equal(P.lat, d.lat) and np.array_equal(P.level, d.level)
    assert np.array_equal(P.rlons, d.rlons) and np.array_equal(P.rlats, d.rlats) and np.array_equal(P.coslats, d.coslats)
    assert d.rlons.dtype == P.rlons.dtype == np.float32
    assert np.array_equal(P.time, d.time)
    for row, var in (("Air Temperature", "TMP_2_ISBL"), ("Omega Velocity", "V_VEL_2_ISBL"),
                     ("Geopotential Height", "HGT_2_ISBL")):
        assert np.array_equal(P.fields[row], d[var], equal_nan=True)
        assert d[var].flags.c_contiguous


def test_prepare_fixed_equals_oracle():
    a = _args(fixed=True, box_limits=os.path.join(INP, "box_limits_Reg1"))
    d = PP.prepare_data(a, os.path.join(INP, "namelist_NCEP-R2"), box_limits_file=a.box_limits)
    P, _ = H.load_prepared("testdata_NCEP-R2.nc")
    _same(O.slice_domain_fixed(P, -60, -30, -42.5, -17.5), d)


def test_prepare_track_equals_oracle():
    a = _args(track=True, trackfile=os.path.join(INP, "track_testdata_NCEP-R2"))
    d = PP.prepare_data(a, os.path.join(INP, "namelist_NCEP-R2"))
    P, tr = H.load_prepared("testdata_NCEP-R2.nc", track="track_testdata_NCEP-R2")
    _same(O.slice_domain_track(P, tr), d)


def test_catarina_lon_wrap_and_level_sort():
    a = _args(infile=os.path.join(SAM, "Catarina_NCEP-R2.nc"), fixed=True)
    nl = PP.read_namelist(os.path.join(INP, "namelist_NCEP-R2"))
    raw = PP.open_netcdf3(a.infile, nl)
    assert raw.lon.max() > 180                       # file stores 0..360
    d = PP.process_data(raw, a, nl)
    assert d.lon.min() >= -180 and d.lon.max() < 180 and np.all(np.diff(d.lon) > 0)
    assert np.all(np.diff(d.level) > 0) and d.level[0] == 1000.0 and d.level[-1] == 100000.0


@pytest.mark.parametrize("case", ["ncep_fixed", "ncep_track", "catarina", "era5_f32", "era5_packed", "era5_unheld_fill"])
def test_raw_backed_dataset_equals_host_prepared(case, tmp_path, monkeypatch):
    """Default loading keeps the fields in file layout (RawStore: only index maps move through
    process_data / slice_domain); what it materialises on access has the bits of the eager host pipeline
    (LEC_DEVICE_INGEST=0), also when the fill value is one the int16 records cannot hold."""
    nml = os.path.join(INP, "namelist_NCEP-R2")
    if case == "ncep_fixed":
        a = _args(fixed=True, box_limits=os.path.join(INP, "box_limits_Reg1"))
    elif case == "ncep_track":
        a = _args(track=True, trackfile=os.path.join(INP, "track_testdata_NCEP-R2"))
    elif case == "catarina":
        a = _args(infile=os.path.join(SAM, "Catarina_NCEP-R2.nc"), fixed=True, box_limits=os.path.join(INP, "box_limits_Reg1"))
    else:
        nc = str(tmp_path / "testdata_ERA5.nc")
        if case == "era5_unheld_fill":
            H.write_era5_unheld_fill(nc, 160)
        else:
            H.write_era5_like(nc, case == "era5_packed", 160)
        a = _args(infile=nc, track=True, trackfile=os.path.join(INP, "track_testdata_ERA5"))
        nml = os.path.join(INP, "namelist_ERA5")
    kw = dict(box_limits_file=a.box_limits) if a.box_limits else {}
    lazy = PP.prepare_data(a, nml, **kw)
    monkeypatch.setenv("LEC_DEVICE_INGEST", "0")
    eager = PP.prepare_data(a, nml, **kw)
    assert lazy.raw is not None and eager.raw is None
    for c in ("time", "level", "lat", "lon", "rlats", "coslats", "rlons"):
        x, y = getattr(lazy, c), getattr(eager, c)
        assert x.dtype == y.dtype and np.array_equal(x, y), c
    assert set(lazy.variables.keys()) == set(eager.variables.keys())
    for var in eager.variables:
        x, y = lazy[var], eager[var]
        assert x.dtype == y.dtype and x.shape == y.shape and np.array_equal(x, y, equal_nan=True), var
        k = len(eager.level) // 2
        assert np.array_equal(lazy.level_plane(var, k), y[:, k], equal_nan=True)
        assert lazy.raw.dtype_of(var) == y.dtype
    assert lazy.load().raw is None and isinstance(lazy.variables, dict)


class _FakeDataArray:
    def __init__(self, values, dims=(), attrs=None):
        self.values, self.dims, self.attrs = values, dims, dict(attrs or {})


def _plant_float_fills(name, data):
    if name in ("T", "U"):
        data.reshape(-1)[::53] = -999.0 if name == "T" else 1e20
    return data


def _pack_coordinates(name, data):
    if name == "latitude":                   # -5 - 0.25 k: decoded with the offset, to float64
        return np.round((data + 5.0) / 0.25).astype(np.int16)
    if name == "longitude":                  # -65 + 0.25 i: scale only, to float32
        return np.round(data / np.float32(0.25)).astype(np.int16)
    return None


_PACKED_COORDS = {"latitude": {"scale_factor": 0.25, "add_offset": -5.0}, "longitude": {"scale_factor": np.float32(0.25)}}


def _era5_case(tmp_path, case):
    """The ERA5-like file and namelist of a :func:`test_from_xarray_adaptor_equals_file_loader` case."""
    nc, nlf = str(tmp_path / "testdata_ERA5.nc"), os.path.join(INP, "namelist_ERA5")
    H.write_era5_like(nc + ".src", case not in (False, "float_fills"), 160)
    edit, attrs, extra = None, None, None
    if case == "float_fills":
        edit, attrs = _plant_float_fills, {v: {"_FillValue": np.float32(-999.0), "missing_value": np.float32(1e20)}
                                           for v in "TUVWZ"}
    elif case == "unsigned":                 # values NetCDF-3 can store as int16 and from_xarray gets as uint16
        edit = lambda name, data: np.abs(data) if name in list("TUVWZ") else None
    elif case == "extra_rows":
        ust = np.round(np.random.default_rng(3).uniform(0, 3, size=(5, 141, 160)) / 1e-4).astype(np.int16)
        ust.reshape(-1)[::53] = -32767
        extra = {"UST": (("time", "latitude", "longitude"), ust, {"scale_factor": 1e-4, "_FillValue": np.int16(-32767)})}
        nlf = str(tmp_path / "namelist")
        with open(nlf, "w") as f:
            f.write(open(os.path.join(INP, "namelist_ERA5")).read().rstrip("\n") + "\nFriction Velocity;;UST;m/s\n")
    elif case == "packed_coords":
        edit, attrs = _pack_coordinates, _PACKED_COORDS
    H.write_netcdf3_copy(nc + ".src", nc, edit, extra, attrs)
    return nc, PP.read_namelist(nlf)


@pytest.mark.parametrize("case", [False, True, "float_fills", "unsigned", "extra_rows", "packed_coords"])
def test_from_xarray_adaptor_equals_file_loader(tmp_path, case):
    """from_xarray on a duck-typed Dataset (``ds[name].values/.dims/.attrs``: what xr.open_dataset(...,
    mask_and_scale=False, decode_times=True) exposes) gives the dataset open_netcdf3 gives, raw-backed or not,
    and one whose field is stored (time, lat, level, lon) is transposed on the host.  Cases: float32 (False) or
    int16-packed (True) fields; float32 fields with _FillValue and missing_value entries; packed fields held as
    uint16; a packed Friction Velocity row with fill values; int16-packed latitude and longitude."""
    from scipy.io import netcdf_file
    nc, nl = _era5_case(tmp_path, case)
    ref = PP.open_netcdf3(nc, nl)
    with netcdf_file(nc, mmap=False) as f:
        ds = {}
        for name, v in f.variables.items():
            at = {a: (getattr(v, a).decode() if isinstance(getattr(v, a), bytes) else getattr(v, a)) for a in v._attributes}
            ds[name] = _FakeDataArray(np.array(v.data).astype(v.data.dtype.newbyteorder("=")), tuple(v.dimensions), at)
    ds["time"] = _FakeDataArray(ref.time, ("time",))                       # decode_times=True
    if case == "unsigned":
        for name in "TUVWZ":
            ds[name].values = ds[name].values.astype(np.uint16)
    a = _args(infile=nc, track=True, trackfile=os.path.join(INP, "track_testdata_ERA5"))
    want = PP.slice_domain(PP.process_data(ref, a, nl), a, nl)
    if case == "float_fills":
        assert np.isnan(want["T"]).any() and np.isnan(want["U"]).any()
    if case == "extra_rows":
        assert want["UST"].dtype == np.float32 and np.isnan(want["UST"]).any()
    for lazy in (True, False):
        d = PP.from_xarray(ds, nl, lazy=lazy)
        assert (d.raw is not None) == (lazy and case not in ("unsigned", "extra_rows"))
        got = PP.slice_domain(PP.process_data(d, a, nl), a, nl)
        for c in ("time", "level", "lat", "lon", "rlats", "coslats", "rlons"):
            assert getattr(got, c).dtype == getattr(want, c).dtype and np.array_equal(getattr(got, c), getattr(want, c)), c
        assert set(got.variables.keys()) == set(want.variables.keys())
        for var in want.variables.keys():
            assert got[var].dtype == want[var].dtype and np.array_equal(got[var], want[var], equal_nan=True), var
    ds["T"] = _FakeDataArray(np.ascontiguousarray(np.swapaxes(ds["T"].values, 1, 2)),
                             ("time", "latitude", "level", "longitude"), ds["T"].attrs)
    d = PP.from_xarray(ds, nl)
    assert d.raw is None
    got = PP.slice_domain(PP.process_data(d, a, nl), a, nl)
    assert np.array_equal(got["T"], want["T"], equal_nan=True)


def test_input_format_errors(tmp_path):
    bad = tmp_path / "box"
    bad.write_text("min_lon;-30\nmax_lon;-60\nmin_lat;-40\nmax_lat;-20\n")
    with pytest.raises(ValueError, match="min_lon"):
        PP.read_box_limits(bad)
    bad.write_text("min_lon;-30\nmax_lon;-20\n")
    with pytest.raises(ValueError, match="missing required fields"):
        PP.read_box_limits(bad)
    trk = tmp_path / "track"
    trk.write_text("time;Lat;Lon\n2005-08-08 00:00:00;-22.5;-45\n")
    with pytest.raises(ValueError):
        PP.read_track(trk)
    tr = PP.read_track(os.path.join(INP, "track_testdata_NCEP-R2"))
    assert str(tr.index[1]) == "2005-08-08 06:00:00"


def test_track_outside_data_is_rejected():
    a = _args(track=True, trackfile=os.path.join(INP, "track_Reg1-Representative"))
    with pytest.raises(ValueError, match="later than data final timestamp"):
        PP.prepare_data(a, os.path.join(INP, "namelist_NCEP-R2"))


def test_budget_and_residual_columns():
    import pandas as pd
    t = np.datetime64("2020-01-01") + np.arange(4) * np.timedelta64(6, "h")
    df = pd.DataFrame({k: np.arange(4.0) * (i + 1) for i, k in enumerate(
        ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe", "Gz", "Ge"])}, index=t)
    df = CB.calc_residuals(CB.calc_budget_diff(df, t))
    assert list(df.columns[-8:]) == ["∂Az/∂t (finite diff.)", "∂Ae/∂t (finite diff.)", "∂Kz/∂t (finite diff.)",
                                     "∂Ke/∂t (finite diff.)", "RGz", "RKz", "RGe", "RKe"]
    assert np.allclose(df["∂Az/∂t (finite diff.)"], 1 / 21600.0)
    odf = O.calc_residuals(O.calc_budget_diff(df[df.columns[:14]].copy(), t))
    assert np.array_equal(df.values, odf.values)


def test_netcdf4_input_through_an_optional_reader(tmp_path, monkeypatch):
    """A NetCDF-4 (HDF5) file is routed by its signature to netCDF4 / h5py (neither ships with this image: a stand-in
    module with netCDF4's API serves the bundled NetCDF-3 contents) and yields the dataset the NetCDF-3 path yields,
    also from a copy whose latitude and longitude are int16-packed; without a reader the error says what to install."""
    import argparse
    import sys
    import types
    from scipy.io import netcdf_file
    from lorenzcycletoolkit_b200.utils import preprocessing as PP
    src = os.path.join(SAM, "testdata_NCEP-R2.nc")
    nlf = os.path.join(INP, "namelist_NCEP-R2")
    box = os.path.join(INP, "box_limits_Reg1")
    fake = tmp_path / "testdata_nc4.nc"
    fake.write_bytes(b"\x89HDF\r\n\x1a\n" + b"\0" * 64)
    args = argparse.Namespace(infile=str(fake), fixed=True, track=False, choose=False, residuals=True, box_limits=box,
                              cdsapi=False, mpas=False)
    monkeypatch.setitem(sys.modules, "netCDF4", None)          # import netCDF4 -> ImportError
    monkeypatch.setitem(sys.modules, "h5py", None)
    with pytest.raises(RuntimeError, match="netCDF4.*h5py"):
        PP.prepare_data(args, nlf, box_limits_file=box)

    class Var:
        def __init__(self, v):
            self._v = v
            self.dimensions = tuple(v.dimensions)

        def __getitem__(self, key):
            a = np.array(self._v.data)
            return a.astype(a.dtype.newbyteorder("="))

        def ncattrs(self):
            return list(self._v._attributes)

        def getncattr(self, a):
            return getattr(self._v, a)

    served = [src]

    class Dataset:
        def __init__(self, path, mode="r"):
            assert path == str(fake)
            self._f = netcdf_file(served[0], mmap=False)
            self.variables = {k: Var(v) for k, v in self._f.variables.items()}
            self.auto = True

        def set_auto_maskandscale(self, flag):
            self.auto = flag

        def __enter__(self):
            return self

        def __exit__(self, *exc):
            assert self.auto is False
            self._f.close()

    mod = types.ModuleType("netCDF4")
    mod.Dataset = Dataset
    monkeypatch.setitem(sys.modules, "netCDF4", mod)
    packed = str(tmp_path / "packed_coords.nc")      # latitude: scale only (float32), longitude: with an offset (float64)
    H.write_netcdf3_copy(src, packed, lambda name, data: np.round(data / 2.5).astype(np.int16) if name == "lat_2" else
                         np.round((data + 100.0) / 2.5).astype(np.int16) if name == "lon_2" else None,
                         attrs={"lat_2": {"scale_factor": np.float32(2.5)}, "lon_2": {"scale_factor": 2.5, "add_offset": -100.0}})
    for served[0], dtypes in ((src, (np.float32, np.float32)), (packed, (np.float32, np.float64))):
        args.infile = str(fake)
        got = PP.prepare_data(args, nlf, box_limits_file=box)
        args.infile = served[0]
        want = PP.prepare_data(args, nlf, box_limits_file=box)
        assert got.raw is not None and want.raw is not None          # both stay raw-backed (decoded on the GPU)
        assert (want.lat.dtype, want.lon.dtype) == dtypes
        for k in ("time", "level", "lat", "lon", "rlats", "coslats", "rlons"):
            assert getattr(got, k).dtype == getattr(want, k).dtype and np.array_equal(getattr(got, k), getattr(want, k)), k
        for var in ("TMP_2_ISBL", "V_VEL_2_ISBL"):
            assert np.array_equal(np.asarray(got[var]), np.asarray(want[var]))
