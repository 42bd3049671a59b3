"""ctypes binding of the C ABI in ``include/lec_b200.h`` (``liblec_b200.so``).

This is the only compute path of the package: there is no CPU fallback.  If the
shared library has not been built (``python __graft_entry__.py``) importing
:class:`LecEngine` works, but constructing one raises ``RuntimeError``; on a
machine without a CUDA device ``lec_create`` fails with ``LEC_ERR_CUDA``.

Host helpers that need no GPU (``nearest_index``, ``gradient_coefs``) restate the
pandas / numpy semantics the reference relies on (SURVEY.md Appendix B.2, B.5).
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

LEC_F32, LEC_F64 = 0, 1
LEC_MATH_AUTO, LEC_MATH_F64 = 0, 1
NTERMS = 16
NLEVEL_TERMS = 19
NBOUNDARY_PIECES = 18        # [BAz BAe BKz BKe BΦZ BΦE] x [E-W, N-S, vertical flux] per level
BOUNDARY_TERMS = ["BAz", "BAe", "BKz", "BKe", "BΦZ", "BΦE"]
FLAG_NONFINITE, FLAG_SIGMA_FLOOR = 1, 2

TERM_NAMES = ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce",
              "BAz", "BAe", "BKz", "BKe", "BΦZ", "BΦE", "Gz", "Ge"]
LEVEL_TERM_NAMES = ["Az", "Ae", "Kz", "Ke", "Ge", "Gz", "Cz", "Cz_2", "Ca", "Ca_1", "Ca_2",
                    "Ce", "Ce_2", "Ck", "Ck_1", "Ck_2", "Ck_3", "Ck_4", "Ck_5"]

STEP_DTYPE = np.dtype([("slot", "i4"), ("slot_m", "i4"), ("slot_p", "i4"),
                       ("i0", "i4"), ("i1", "i4"), ("j0", "i4"), ("j1", "i4"), ("reserved", "i4"),
                       ("ct_m", "f8"), ("ct_0", "f8"), ("ct_p", "f8")], align=True)
assert STEP_DTYPE.itemsize == 56

_ERRORS = {-1: ValueError, -3: ValueError, -4: IndexError, -5: MemoryError}

_LIB_PATH = Path(__file__).resolve().parent / "_lib" / "liblec_b200.so"
_lib = None


class _GridDesc(C.Structure):
    _fields_ = [("nlon", C.c_int32), ("nlat", C.c_int32), ("nlev", C.c_int32),
                ("lon_deg", C.POINTER(C.c_double)), ("lat_deg", C.POINTER(C.c_double)),
                ("rlon", C.POINTER(C.c_double)), ("rlat", C.POINTER(C.c_double)),
                ("coslat", C.POINTER(C.c_double)), ("plev", C.POINTER(C.c_double)),
                ("dtype", C.c_int32), ("math", C.c_int32),
                ("field_scale", C.c_double * 5),
                ("max_steps", C.c_int32), ("max_box_rows", C.c_int32),
                ("device", C.c_int32), ("band_rows", C.c_int32),
                ("host_stage_bytes", C.c_int64)]


class _RawDesc(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("nlon", C.c_int32), ("nlat", C.c_int32), ("nlev", C.c_int32),
                ("lon_map", C.POINTER(C.c_int32)), ("lat_map", C.POINTER(C.c_int32)), ("lev_map", C.POINTER(C.c_int32)),
                ("scale", C.c_double * 5), ("offset", C.c_double * 5),
                ("use_scale", C.c_int32 * 5), ("use_offset", C.c_int32 * 5), ("round_f32", C.c_int32 * 5),
                ("nfill", C.c_int32 * 5), ("fill", (C.c_double * 2) * 5),
                ("big_endian", C.c_int32), ("reserved", C.c_int32), ("record_stride", C.c_int64 * 5)]


class _PackedDesc(C.Structure):
    _fields_ = [("pitch", C.c_int32), ("reserved", C.c_int32),
                ("scale", C.c_double * 5), ("offset", C.c_double * 5),
                ("use_scale", C.c_int32 * 5), ("use_offset", C.c_int32 * 5), ("round_f32", C.c_int32 * 5),
                ("nfill", C.c_int32 * 5), ("fill", (C.c_double * 2) * 5)]


class _Dispatch(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("kernel", "vec", "group", "lonw", "comp", "math64", "tile_rows",
                                         "tiles_per_band", "nbands", "packed")]


ROW_KERNELS = ("direct", "subwarp", "tiled")      # lec_dispatch.kernel (LEC_ROWS_*)

LEC_RAW_F32, LEC_RAW_F64, LEC_RAW_I16 = 0, 1, 2
_RAW_DTYPES = {np.dtype(np.float32): LEC_RAW_F32, np.dtype(np.float64): LEC_RAW_F64, np.dtype(np.int16): LEC_RAW_I16}


class _DiagGrid(C.Structure):
    _fields_ = [("nlon", C.c_int32), ("nlat", C.c_int32), ("dtype", C.c_int32), ("device", C.c_int32),
                ("dx", C.POINTER(C.c_double)), ("dy", C.POINTER(C.c_double)),
                ("parallel_scale", C.POINTER(C.c_double)), ("meridional_scale", C.POINTER(C.c_double)),
                ("scale", C.c_double * 3), ("z_div", C.c_double)]


DIAG_STEP_DTYPE = np.dtype([("slot", "i4"), ("i0", "i4"), ("i1", "i4"), ("j0", "i4"), ("j1", "i4"),
                            ("ic", "i4"), ("jc", "i4"), ("reserved", "i4")])
DIAG_NAMES = ("zeta_min", "zeta_max", "hgt_min", "wind_max")
NDIAG_VALUES = 5          # the four extrema + zeta at the track centre


def diag_steps(boxes, centres=None):
    """:data:`DIAG_STEP_DTYPE` array from ``(slot, i0, i1, j0, j1)`` tuples; ``centres``: optional ``(ic, jc)`` per
    step (domain indices of the grid point nearest to the track centre), default none (-1)."""
    st = np.zeros(len(boxes), dtype=DIAG_STEP_DTYPE)
    st["ic"] = st["jc"] = -1
    for n, b in enumerate(boxes):
        st["slot"][n], st["i0"][n], st["i1"][n], st["j0"][n], st["j1"][n] = b
        if centres is not None:
            st["ic"][n], st["jc"][n] = centres[n]
    return st


def library_path() -> Path:
    return Path(os.environ.get("LEC_B200_LIB", _LIB_PATH))


_TORCH_EXT_PATH = Path(__file__).resolve().parent / "_lib" / "lec_torch_ext.so"
_torch_ext = None          # None = not tried, False = absent / disabled, True = torch.ops.lec_b200 is registered


def load_torch_extension() -> bool:
    """Register ``torch.ops.lec_b200.run_device`` (csrc/lec_torch_ext.cpp: the thin PyTorch C++ extension over the
    C ABI, built by ``__graft_entry__.build()``).  Returns False when the extension has not been built or
    ``LEC_TORCH_EXT=0``; :meth:`LecEngine.run_torch` then calls ``lec_run_device`` through ctypes -- the same CUDA
    library either way.  An override library (``LEC_B200_LIB``) keeps the ctypes route: the extension is linked to
    the in-tree ``liblec_b200.so``."""
    global _torch_ext
    if _torch_ext is None:
        _torch_ext = False
        if os.environ.get("LEC_TORCH_EXT", "1") != "0" and "LEC_B200_LIB" not in os.environ and _TORCH_EXT_PATH.exists():
            import torch
            load_library()                        # liblec_b200.so first: the extension resolves its symbols from it
            try:
                torch.ops.load_library(str(_TORCH_EXT_PATH))
                _torch_ext = True
            except (OSError, RuntimeError) as e:   # e.g. built against another torch: keep the ctypes binding
                import warnings
                warnings.warn(f"lec_torch_ext.so could not be loaded ({e}); run_torch uses the ctypes binding")
    return _torch_ext


def load_library():
    """Load ``liblec_b200.so`` and declare every symbol of ``include/lec_b200.h``."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not path.exists():
        raise RuntimeError(
            f"{path} is missing: the CUDA engine has not been built "
            "(run `python __graft_entry__.py` in the repo root). There is no CPU fallback.")
    lib = C.CDLL(str(path))
    vp, dp, ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32)
    lib.lec_create.argtypes = [C.POINTER(vp), C.POINTER(_GridDesc)]
    lib.lec_create.restype = C.c_int
    lib.lec_destroy.argtypes = [vp]
    lib.lec_destroy.restype = C.c_int
    lib.lec_run_device.argtypes = [vp, C.POINTER(vp), C.c_int32, vp, C.c_int32, vp, vp, vp, vp]
    lib.lec_run_device.restype = C.c_int
    lib.lec_run_device_packed.argtypes = [vp, C.POINTER(_PackedDesc), C.POINTER(vp), C.c_int32, vp, C.c_int32, vp, vp, vp,
                                          vp]
    lib.lec_run_device_packed.restype = C.c_int
    lib.lec_run_host.argtypes = [vp, C.POINTER(vp), C.c_int32, vp, C.c_int32, vp, vp, vp]
    lib.lec_run_host.restype = C.c_int
    lib.lec_run_host_raw.argtypes = [vp, C.POINTER(_RawDesc), C.POINTER(vp), C.c_int32, vp, C.c_int32, vp, C.c_int32,
                                     vp, vp, vp]
    lib.lec_run_host_raw.restype = C.c_int
    lib.lec_gradient_coefs.argtypes = [dp, C.c_int32, dp, dp, dp]
    lib.lec_gradient_coefs.restype = C.c_int
    lib.lec_nearest_index.argtypes = [dp, C.c_int32, C.c_double]
    lib.lec_nearest_index.restype = C.c_int32
    lib.lec_last_timing.argtypes = [vp, C.POINTER(C.c_float)]
    lib.lec_last_timing.restype = C.c_int
    lib.lec_timing_reset.argtypes = [vp]
    lib.lec_timing_reset.restype = C.c_int
    lib.lec_last_transfer.argtypes = [vp, C.POINTER(C.c_int64)]
    lib.lec_last_transfer.restype = C.c_int
    lib.lec_set_boundary_levels.argtypes = [vp, vp]
    lib.lec_set_boundary_levels.restype = C.c_int
    lib.lec_pin_host.argtypes = [vp, C.c_int64]
    lib.lec_pin_host.restype = C.c_int
    lib.lec_unpin_host.argtypes = [vp]
    lib.lec_unpin_host.restype = C.c_int
    lib.lec_launch_count.argtypes = [vp]
    lib.lec_launch_count.restype = C.c_int64
    lib.lec_last_dispatch.argtypes = [vp, C.POINTER(_Dispatch)]
    lib.lec_last_dispatch.restype = C.c_int
    lib.lec_diag850_host.argtypes = [C.POINTER(_DiagGrid), vp, vp, vp, C.c_int32, vp, C.c_int32, vp, vp]
    lib.lec_diag850_host.restype = C.c_int
    lib.lec_diag850_device.argtypes = [C.POINTER(_DiagGrid), vp, vp, vp, C.c_int32, vp, C.c_int32, vp, vp, vp]
    lib.lec_diag850_device.restype = C.c_int
    lib.lec_strerror.argtypes = [C.c_int]
    lib.lec_strerror.restype = C.c_char_p
    lib.lec_last_error.argtypes = [vp]
    lib.lec_last_error.restype = C.c_char_p
    lib.lec_version.argtypes = []
    lib.lec_version.restype = C.c_char_p
    _lib = lib
    return lib


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def nearest_index(coord, value) -> int:
    """``coord.sel(value, method="nearest")`` index (pandas nearest; ties -> larger)."""
    c = _f64(coord)
    return int(load_library().lec_nearest_index(_dptr(c), c.size, float(value)))


def gradient_coefs(x):
    """``np.gradient(f, x, edge_order=1)`` as three coefficient arrays (a, b, c)."""
    x = _f64(x)
    a, b, c = (np.empty_like(x) for _ in range(3))
    rc = load_library().lec_gradient_coefs(_dptr(x), x.size, _dptr(a), _dptr(b), _dptr(c))
    if rc != 0:
        raise ValueError("gradient needs at least two coordinate values")
    return a, b, c


def diag850_host(u, v, z, lon_deg, lat_deg, steps, scale=(1.0, 1.0, 1.0), z_div=1.0, device=0):
    """850-hPa track diagnostics on the GPU (``lec_diag850_host``): ``u, v, z`` are ``[slot][lat][lon]``
    planes of the 850-hPa level (one float dtype), ``steps`` a :data:`DIAG_STEP_DTYPE` array of
    label-sliced boxes (:func:`diag_steps`).  Vorticity is MetPy's on the lat / lon grid
    (``utils.geodesy.latlon_grid_metrics``).  Returns ``(values[n, 5], flat_index[n, 4])``: the extrema in
    :data:`DIAG_NAMES` order with NaNs skipped and zeta at the step's centre point (NaN if none), and numpy
    ``argmin`` / ``argmax`` of the box (row-major)."""
    from .utils.geodesy import latlon_grid_metrics
    lib = load_library()
    dt = np.float32 if all(np.asarray(a).dtype == np.float32 for a in (u, v, z)) else np.float64
    planes = [np.ascontiguousarray(a, dtype=dt) for a in (u, v, z)]
    if planes[0].ndim != 3 or any(a.shape != planes[0].shape for a in planes):
        raise ValueError("u, v, z must be [slot][lat][lon] planes of one shape")
    nslots, nlat, nlon = planes[0].shape
    if np.size(lon_deg) != nlon or np.size(lat_deg) != nlat:
        raise ValueError("coordinate sizes do not match the planes")
    if nlon < 3 or nlat < 3:
        raise ValueError("the 850-hPa diagnostics need at least three grid points along each axis "
                         "(3-point derivatives)")
    dx, dy, ps, ms = (_f64(a) for a in latlon_grid_metrics(lon_deg, lat_deg))
    g = _DiagGrid()
    g.nlon, g.nlat, g.dtype, g.device = nlon, nlat, (LEC_F32 if dt == np.float32 else LEC_F64), int(device)
    g.dx, g.dy, g.parallel_scale, g.meridional_scale = _dptr(dx), _dptr(dy), _dptr(ps), _dptr(ms)
    for i in range(3):
        g.scale[i] = float(scale[i])
    g.z_div = float(z_div)
    st = np.ascontiguousarray(steps, dtype=DIAG_STEP_DTYPE)
    vals = np.empty((st.size, NDIAG_VALUES), dtype=np.float64)
    idx = np.empty((st.size, len(DIAG_NAMES)), dtype=np.int32)
    rc = lib.lec_diag850_host(C.byref(g), planes[0].ctypes.data, planes[1].ctypes.data, planes[2].ctypes.data,
                              nslots, st.ctypes.data, st.size, vals.ctypes.data, idx.ctypes.data)
    if rc != 0:
        msg = f"lec_diag850_host: {lib.lec_strerror(rc).decode()}"
        extra = lib.lec_last_error(None).decode()
        raise _ERRORS.get(rc, RuntimeError)(msg + (f" ({extra})" if extra and rc == -2 else ""))
    return vals, idx


_PINNED = {}          # start address -> (bytes, weakref to the owner of the memory)


def pin_arrays(arrays, limit_bytes=None):
    """Page-lock the host range that holds ``arrays`` (``lec_pin_host`` = ``cudaHostRegister``) so that
    ``lec_run_host*`` copies from them at the pinned PCIe rate.  The arrays may be strided views of one buffer (the
    interleaved record variables of a NetCDF-3 file): the smallest range covering all of them is registered once and
    released when the first array's base object is collected.  Returns True if the range is (now) pinned; a range
    that cannot be registered, or is larger than ``limit_bytes`` (default: a quarter of the host RAM), stays
    pageable and False is returned."""
    import weakref
    if os.environ.get("LEC_PIN_RAW", "1") == "0":
        return False

    def span(a):
        if a.size == 0:
            return a.ctypes.data, a.ctypes.data
        hi = a.ctypes.data + a.itemsize + sum((n - 1) * abs(st) for n, st in zip(a.shape, a.strides))
        return a.ctypes.data, hi
    spans = [span(np.asarray(a)) for a in arrays]
    lo, hi = min(s[0] for s in spans), max(s[1] for s in spans)
    if lo in _PINNED and _PINNED[lo][0] >= hi - lo:
        return True
    if limit_bytes is None:
        try:
            limit_bytes = os.sysconf("SC_PAGE_SIZE") * os.sysconf("SC_PHYS_PAGES") // 4
        except (ValueError, OSError):
            limit_bytes = 16 << 30
    if hi - lo > limit_bytes or hi <= lo:
        return False
    lib = load_library()
    if lib.lec_pin_host(C.c_void_p(lo), hi - lo) != 0:
        return False
    owner = np.asarray(arrays[0])
    while isinstance(owner.base, np.ndarray):
        owner = owner.base

    def release(addr=lo):
        if _PINNED.pop(addr, None) is not None:
            lib.lec_unpin_host(C.c_void_p(addr))
    try:
        ref = weakref.finalize(owner, release)
    except TypeError:
        ref = None
    _PINNED[lo] = (hi - lo, ref)
    return True


def _set_decode(d, decode, strict=False):
    """Fill the decode fields (scale, offset, use_*, round_f32, nfill, fill) that ``lec_raw_desc`` and
    ``lec_packed_desc`` share from per-field dicts ``scale``, ``offset``, ``fills``, ``float32``.  ``strict``: more than
    two fill values, or one that is not an int16 value, is an error (otherwise the first two are used)."""
    for f, dec in enumerate(decode or [{}] * 5):
        d.scale[f] = float(dec.get("scale", 1.0) if dec.get("scale") is not None else 1.0)
        d.offset[f] = float(dec.get("offset", 0.0) if dec.get("offset") is not None else 0.0)
        d.use_scale[f] = int(dec.get("scale") is not None)
        d.use_offset[f] = int(dec.get("offset") is not None)
        d.round_f32[f] = int(bool(dec.get("float32", False)))
        fills = list(dec.get("fills", ()))
        if strict and (len(fills) > 2 or any(not (float(v) == int(v) and -32768 <= int(v) <= 32767)
                                             for v in fills if np.isfinite(float(v)))
                       or not all(np.isfinite(float(v)) for v in fills)):
            raise ValueError(f"field {f}: int16 decoding takes at most two fill values, each an int16 value (got {fills})")
        fills = fills[:2]
        d.nfill[f] = len(fills)
        for n, fv in enumerate(fills):
            d.fill[f][n] = float(fv)


def make_steps(nsteps: int) -> np.ndarray:
    return np.zeros(nsteps, dtype=STEP_DTYPE)


def time_stencil(tsec, steps, first_slot=0, slots=None):
    """Fill slot/slot_m/slot_p and the dT/dt coefficients of ``steps`` for a time
    axis ``tsec`` (seconds): ``np.gradient`` over that axis, as
    ``DataArray.differentiate(time, datetime_unit="s")`` does
    (thermodynamics.py:109-110, lorenzcycletoolkit.py:184-186)."""
    tsec = _f64(tsec)
    n = tsec.size
    a, b, c = gradient_coefs(tsec)
    idx = np.arange(n) if slots is None else np.asarray(slots)
    steps["slot"] = idx + first_slot
    steps["slot_m"] = np.maximum(idx - 1, 0) + first_slot
    steps["slot_p"] = np.minimum(idx + 1, n - 1) + first_slot
    steps["ct_m"], steps["ct_0"], steps["ct_p"] = a[idx], b[idx], c[idx]
    return steps


class LecEngine:
    """One handle of the CUDA engine for one prepared grid."""

    def __init__(self, lon_deg, lat_deg, rlon, rlat, coslat, plev, dtype, field_scale=None,
                 max_steps=64, max_box_rows=0, device=0, math=LEC_MATH_AUTO, band_rows=0,
                 host_stage_bytes=0):
        self._lib = load_library()
        self._h = C.c_void_p()
        self._keep = [_f64(a) for a in (lon_deg, lat_deg, rlon, rlat, coslat, plev)]
        lon, lat, rl, rp, cl, pl = self._keep
        if rl.size != lon.size or rp.size != lat.size or cl.size != lat.size:
            raise ValueError("coordinate arrays disagree in length")
        self.nlon, self.nlat, self.nlev = lon.size, lat.size, pl.size
        self.np_dtype = np.dtype(dtype)
        if self.np_dtype not in (np.dtype(np.float32), np.dtype(np.float64)):
            raise ValueError("fields must be float32 or float64")
        d = _GridDesc()
        d.nlon, d.nlat, d.nlev = self.nlon, self.nlat, self.nlev
        d.lon_deg, d.lat_deg, d.rlon, d.rlat, d.coslat, d.plev = (_dptr(a) for a in self._keep)
        d.dtype = LEC_F64 if self.np_dtype == np.float64 else LEC_F32
        d.math = math
        scale = [1.0] * 5 if field_scale is None else [float(s) for s in field_scale]
        d.field_scale = (C.c_double * 5)(*scale)
        d.max_steps, d.max_box_rows, d.device = int(max_steps), int(max_box_rows), int(device)
        d.band_rows, d.host_stage_bytes = int(band_rows), int(host_stage_bytes)
        self.device = int(device)
        self.max_steps = int(max_steps)
        self.last_boundary = None
        rc = self._lib.lec_create(C.byref(self._h), C.byref(d))
        if rc != 0:
            msg = self._message(rc)
            self.close()
            raise _ERRORS.get(rc, RuntimeError)(f"lec_create: {msg}")

    # ------------------------------------------------------------------ #
    def _message(self, rc):
        msg = self._lib.lec_strerror(rc).decode()
        if self._h:
            extra = self._lib.lec_last_error(self._h).decode()
            if extra:
                msg += f" ({extra})"
        return msg

    def _check(self, rc, what):
        if rc != 0:
            raise _ERRORS.get(rc, RuntimeError)(f"{what}: {self._message(rc)}")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.lec_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # ------------------------------------------------------------------ #
    def _steps_arg(self, steps):
        steps = np.ascontiguousarray(steps, dtype=STEP_DTYPE)
        return steps, steps.ctypes.data_as(C.c_void_p)

    def _boundary_begin(self, n, want):
        """Arm ``lec_set_boundary_levels`` with a fresh ``[n][6][3][nlev]`` host array (or disarm it)."""
        self.last_boundary = np.empty((n, 6, 3, self.nlev), dtype=np.float64) if want else None
        self._check(self._lib.lec_set_boundary_levels(
            self._h, self.last_boundary.ctypes.data if want else None), "lec_set_boundary_levels")

    def run_host(self, fields, steps, want_levels=True, want_boundary=False):
        """``lec_run_host``: ``fields`` = five C-contiguous host arrays
        ``[slot][level][lat][lon]`` (T, u, v, omega, Phi) of the engine dtype.
        Returns ``(terms[nsteps,16], levels[nsteps,19,nlev] | None, flags[nsteps])``; with
        ``want_boundary`` the per-level boundary pieces ``[nsteps][6][3][nlev]`` are left in
        ``self.last_boundary``."""
        if len(fields) != 5:
            raise ValueError("need five fields: T, u, v, omega, Phi")
        arrs = []
        for a in fields:
            a = np.asarray(a)
            if a.dtype != self.np_dtype or not a.flags.c_contiguous:
                raise ValueError("fields must be C-contiguous arrays of the engine dtype")
            if a.ndim != 4 or a.shape[1:] != (self.nlev, self.nlat, self.nlon):
                raise ValueError(f"field shape {a.shape} does not match the grid")
            arrs.append(a)
        nslots = arrs[0].shape[0]
        if any(a.shape[0] != nslots for a in arrs):
            raise ValueError("fields disagree in the number of time slots")
        steps, sp = self._steps_arg(steps)
        n = steps.size
        terms = np.empty((n, NTERMS), dtype=np.float64)
        levels = np.empty((n, NLEVEL_TERMS, self.nlev), dtype=np.float64) if want_levels else None
        flags = np.zeros(n, dtype=np.int32)
        ptrs = (C.c_void_p * 5)(*[a.ctypes.data for a in arrs])
        self._boundary_begin(n, want_boundary)
        try:
            rc = self._lib.lec_run_host(self._h, ptrs, nslots, sp, n, terms.ctypes.data,
                                        levels.ctypes.data if want_levels else None, flags.ctypes.data)
        finally:
            self._lib.lec_set_boundary_levels(self._h, None)
        self._check(rc, "lec_run_host")
        return terms, levels, flags

    def run_host_raw(self, raw_fields, lon_map, lat_map, lev_map, slot_record, steps, decode=None, want_levels=True,
                     want_boundary=False):
        """``lec_run_host_raw``: ``raw_fields`` = five C-contiguous host arrays ``[record][level][lat][lon]`` in
        FILE layout (one of int16 / float32 / float64), ``*_map`` the engine-index -> raw-index maps,
        ``slot_record`` the record of each engine time slot, ``decode`` = per field a dict with optional
        ``scale``, ``offset``, ``fills`` (<= 2 values) and ``float32`` (decoded variable is float32).
        Same results as :meth:`run_host` on the host-prepared arrays."""
        if len(raw_fields) != 5:
            raise ValueError("need five fields: T, u, v, omega, Phi")
        arrs = [np.asarray(a) for a in raw_fields]
        dt = arrs[0].dtype
        native = dt.newbyteorder("=")

        def record_contiguous(a):      # every record C-contiguous; records may be strided (NetCDF-3 interleaving)
            return a.ndim == 4 and a.strides[1:] == (a.shape[2] * a.shape[3] * a.itemsize, a.shape[3] * a.itemsize,
                                                      a.itemsize) and a.strides[0] > 0
        if native not in _RAW_DTYPES or any(a.dtype != dt or a.shape != arrs[0].shape or not record_contiguous(a)
                                            for a in arrs):
            raise ValueError("raw fields must be [record][level][lat][lon] arrays (contiguous records) of one of "
                             "int16/float32/float64")
        maps = [np.ascontiguousarray(m, dtype=np.int32) for m in (lon_map, lat_map, lev_map)]
        if (maps[0].size, maps[1].size, maps[2].size) != (self.nlon, self.nlat, self.nlev):
            raise ValueError("index maps do not match the engine grid")
        slot_record = np.ascontiguousarray(slot_record, dtype=np.int32)
        d = _RawDesc()
        d.dtype = _RAW_DTYPES[native]
        d.big_endian = int(dt.byteorder == ">" or (dt.byteorder == "=" and not np.little_endian))
        nrec, d.nlev, d.nlat, d.nlon = arrs[0].shape
        for f, a in enumerate(arrs):
            d.record_stride[f] = int(a.strides[0])
        ip = C.POINTER(C.c_int32)
        d.lon_map, d.lat_map, d.lev_map = (m.ctypes.data_as(ip) for m in maps)
        _set_decode(d, decode)
        steps, sp = self._steps_arg(steps)
        n = steps.size
        terms = np.empty((n, NTERMS), dtype=np.float64)
        levels = np.empty((n, NLEVEL_TERMS, self.nlev), dtype=np.float64) if want_levels else None
        flags = np.zeros(n, dtype=np.int32)
        ptrs = (C.c_void_p * 5)(*[a.ctypes.data for a in arrs])
        self._boundary_begin(n, want_boundary)
        try:
            rc = self._lib.lec_run_host_raw(self._h, C.byref(d), ptrs, nrec, slot_record.ctypes.data, slot_record.size,
                                            sp, n, terms.ctypes.data, levels.ctypes.data if want_levels else None,
                                            flags.ctypes.data)
        finally:
            self._lib.lec_set_boundary_levels(self._h, None)
        self._check(rc, "lec_run_host_raw")
        return terms, levels, flags

    def run_device(self, field_ptrs, nslots, steps, out_terms_ptr, out_levels_ptr=None,
                   out_flags_ptr=None, stream=None):
        """``lec_run_device`` on raw device pointers (ints); asynchronous on ``stream``."""
        steps, sp = self._steps_arg(steps)
        ptrs = (C.c_void_p * 5)(*[int(p) for p in field_ptrs])
        rc = self._lib.lec_run_device(self._h, ptrs, int(nslots), sp, steps.size,
                                      C.c_void_p(int(out_terms_ptr)),
                                      C.c_void_p(int(out_levels_ptr)) if out_levels_ptr else None,
                                      C.c_void_p(int(out_flags_ptr)) if out_flags_ptr else None,
                                      C.c_void_p(int(stream)) if stream else None)
        self._check(rc, "lec_run_device")

    def run_torch(self, fields, steps, want_levels=True, out=None):
        """Convenience over :meth:`run_device` for five CUDA ``torch`` tensors; runs on
        torch's current stream and returns CUDA tensors (no synchronisation).  ``out`` = preallocated
        ``(terms [n,16] f64, levels [n,19,nlev] f64, flags [n] i32)`` to write into (e.g. views of a gather buffer)."""
        import torch
        dt = torch.float64 if self.np_dtype == np.float64 else torch.float32
        for t in fields:
            if not t.is_cuda or t.dtype != dt or not t.is_contiguous():
                raise ValueError("fields must be contiguous CUDA tensors of the engine dtype")
            if t.device.index != self.device:
                raise ValueError("fields live on another device than the engine")
            if tuple(t.shape[1:]) != (self.nlev, self.nlat, self.nlon):
                raise ValueError(f"field shape {tuple(t.shape)} does not match the grid")
        n = len(steps)
        dev = fields[0].device
        if out is not None:
            terms, levels, flags = out
            if (tuple(terms.shape) != (n, NTERMS) or terms.dtype != torch.float64 or not terms.is_contiguous()
                    or tuple(levels.shape) != (n, NLEVEL_TERMS, self.nlev) or levels.dtype != torch.float64
                    or not levels.is_contiguous() or tuple(flags.shape) != (n,) or flags.dtype != torch.int32):
                raise ValueError("out = (terms [n,16] f64, levels [n,19,nlev] f64, flags [n] i32), contiguous")
        else:
            terms = torch.empty((n, NTERMS), dtype=torch.float64, device=dev)
            levels = torch.empty((n, NLEVEL_TERMS, self.nlev), dtype=torch.float64, device=dev) if want_levels else None
            flags = torch.zeros(n, dtype=torch.int32, device=dev)
        if load_torch_extension():
            # the PyTorch C++ extension: argument checks, torch's current stream and lec_run_device, in C++
            st, _ = self._steps_arg(steps)
            rc = torch.ops.lec_b200.run_device(int(self._h.value), list(fields), torch.from_numpy(st.view(np.uint8)),
                                               terms, levels, flags)
            self._check(int(rc), "lec_run_device")
            return terms, levels, flags
        stream = torch.cuda.current_stream(dev).cuda_stream
        self.run_device([t.data_ptr() for t in fields], fields[0].shape[0], steps, terms.data_ptr(),
                        levels.data_ptr() if levels is not None else None, flags.data_ptr(), stream)
        return terms, levels, flags

    def run_device_packed(self, field_ptrs, nslots, pitch, decode, steps, out_terms_ptr, out_levels_ptr=None,
                          out_flags_ptr=None, stream=None):
        """``lec_run_device_packed`` on raw device pointers (ints) to int16 fields ``[slot][level][lat][pitch]``;
        ``decode`` = per field a dict as in :meth:`run_host_raw`; asynchronous on ``stream``."""
        d = _PackedDesc()
        d.pitch = int(pitch)
        _set_decode(d, decode, strict=True)
        steps, sp = self._steps_arg(steps)
        ptrs = (C.c_void_p * 5)(*[int(p) for p in field_ptrs])
        rc = self._lib.lec_run_device_packed(self._h, C.byref(d), ptrs, int(nslots), sp, steps.size,
                                             C.c_void_p(int(out_terms_ptr)),
                                             C.c_void_p(int(out_levels_ptr)) if out_levels_ptr else None,
                                             C.c_void_p(int(out_flags_ptr)) if out_flags_ptr else None,
                                             C.c_void_p(int(stream)) if stream else None)
        self._check(rc, "lec_run_device_packed")

    def run_torch_packed(self, fields, decode, steps, want_levels=True, out=None):
        """:meth:`run_torch` for five int16 CUDA tensors that stay packed in device memory (2 bytes per value):
        ``[slot][level][lat][n]`` with contiguous rows ``pitch = stride(2)`` elements apart, a multiple of 8, and
        ``nlon <= n <= pitch`` (the padded rows :func:`~lorenzcycletoolkit_b200.utils.preprocessing.packed_device_fields`
        returns, or a ``[..., :nlon]`` view of them).  ``decode``: per field a dict ``scale``, ``offset``, ``fills``
        (at most two int16 values), ``float32`` as in :meth:`run_host_raw`; the kernels decode every value they load
        by the rule of the raw-record ingest, so the results have the bits of :meth:`run_torch` on the decoded fields.
        Runs on torch's current stream; no synchronisation."""
        import torch
        if len(fields) != 5:
            raise ValueError("need five fields: T, u, v, omega, Phi")
        f0 = fields[0]
        for t in fields:
            if not t.is_cuda or t.dtype != torch.int16:
                raise ValueError("packed fields must be int16 CUDA tensors")
            if t.device.index != self.device:
                raise ValueError("fields live on another device than the engine")
            if t.dim() != 4 or tuple(t.shape[1:3]) != (self.nlev, self.nlat) or not self.nlon <= t.shape[3] <= t.stride(2):
                raise ValueError(f"field shape {tuple(t.shape)} does not match the grid")
            if (t.stride(3) != 1 or t.stride(2) % 8 or t.stride(1) != t.shape[2] * t.stride(2)
                    or t.stride(0) != t.shape[1] * t.stride(1) or t.shape != f0.shape or t.stride() != f0.stride()):
                raise ValueError("packed fields need contiguous rows with a pitch (row stride) that is a multiple of 8, "
                                 "one shape and layout for all five")
        n = len(steps)
        dev = f0.device
        if out is not None:
            terms, levels, flags = out
        else:
            terms = torch.empty((n, NTERMS), dtype=torch.float64, device=dev)
            levels = torch.empty((n, NLEVEL_TERMS, self.nlev), dtype=torch.float64, device=dev) if want_levels else None
            flags = torch.zeros(n, dtype=torch.int32, device=dev)
        if load_torch_extension():
            d = _PackedDesc()
            _set_decode(d, decode, strict=True)
            st, _ = self._steps_arg(steps)
            raw = np.frombuffer(bytes(d), dtype=np.uint8).copy()
            rc = torch.ops.lec_b200.run_device_packed(int(self._h.value), list(fields), torch.from_numpy(raw),
                                                      torch.from_numpy(st.view(np.uint8)), terms, levels, flags)
            self._check(int(rc), "lec_run_device_packed")
            return terms, levels, flags
        stream = torch.cuda.current_stream(dev).cuda_stream
        self.run_device_packed([t.data_ptr() for t in fields], f0.shape[0], f0.stride(2), decode, steps, terms.data_ptr(),
                               levels.data_ptr() if levels is not None else None, flags.data_ptr(), stream)
        return terms, levels, flags

    def last_timing(self):
        """Device milliseconds of the last run: (row-moment kernels, finalize kernels, whole call)."""
        out = (C.c_float * 3)()
        self._check(self._lib.lec_last_timing(self._h, out), "lec_last_timing")
        return float(out[0]), float(out[1]), float(out[2])

    def timing_reset(self):
        """From now on :meth:`last_timing` returns the kernel times summed over every run since this call."""
        self._check(self._lib.lec_timing_reset(self._h), "lec_timing_reset")

    def last_transfer(self):
        """(host->device, device->host) bytes the last :meth:`run_host` moved over PCIe."""
        out = (C.c_int64 * 2)()
        self._check(self._lib.lec_last_transfer(self._h, out), "lec_last_transfer")
        return int(out[0]), int(out[1])

    def last_dispatch(self) -> dict:
        """Row kernel of the last kernel batch (``lec_last_dispatch``): ``kernel`` (one of :data:`ROW_KERNELS`),
        ``vec``, ``group``, ``lonw``, ``comp``, ``math64``, ``tile_rows``, ``tiles_per_band``, ``nbands``, ``packed``
        (int16 fields: :meth:`run_torch_packed`)."""
        d = _Dispatch()
        self._check(self._lib.lec_last_dispatch(self._h, C.byref(d)), "lec_last_dispatch")
        out = {n: int(getattr(d, n)) for n, _ in _Dispatch._fields_}
        out["kernel"] = ROW_KERNELS[out["kernel"]]
        out["comp"], out["math64"], out["packed"] = bool(out["comp"]), bool(out["math64"]), bool(out["packed"])
        return out

    @property
    def launch_count(self) -> int:
        return int(self._lib.lec_launch_count(self._h))


def version() -> str:
    return load_library().lec_version().decode()


def wide_row_kernel() -> str:
    """Name of the row kernel wide boxes (more than 200 chunks of 128 bits per row) take: the build default named by
    ``lec_version`` unless ``LEC_ROW_KERNEL`` overrides it."""
    choice = os.environ.get("LEC_ROW_KERNEL") or ("tile" if "rows=tile" in version() else "direct")
    return "lec_row_moments_tile_kernel" if choice == "tile" else "lec_row_moments_kernel"
