"""lec_run_device_packed: int16 fields resident in device memory, decoded by the row kernels.

The decode rule is the raw-record ingest's (x = double(raw) * scale + offset as two float64 roundings, through float32
where the decoded variable is float32, NaN for a fill value), so a packed run must have the bits of ``lec_run_device``
on the same fields decoded by that rule -- here decoded in numpy.  Each cell also asserts that both runs took the same
row kernel (kernel, group, lonw, comp, math64; tile rows as the int16 ring shapes them) and that the packed one says
so (``packed``).  Fields carry fill values around each fixed box, in its alignment columns and in the pad columns past
``nlon``: none may reach a result."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E
from lorenzcycletoolkit_b200.utils import preprocessing as PP
import helpers as H

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ARITH = {"f32": (np.float32, E.LEC_MATH_AUTO, 4), "m64": (np.float32, E.LEC_MATH_F64, 4),
         "f64": (np.float64, E.LEC_MATH_AUTO, 2)}
LONW = {"exact": 0, "f32": 1, "irregular": 2}
FILL = H.FILL
T0 = np.datetime64("2020-01-01T00")
NT, NLEV = 4, 4
WIDE = (816, 131)


@pytest.fixture(autouse=True)
def _default_dispatcher(monkeypatch):
    for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
        monkeypatch.delenv(k, raising=False)


def _decode_spec(arith):
    """ERA5 style (float64 scale and offset: decoded to float64) on every field; the fp64 handle also gets two fields
    packed with a scale only, whose decoded variable is float32 (rounded once), and one with two fill values."""
    spec = [dict(offset=True, float32=False, nfill=1) for _ in range(5)]
    if arith == "f64":
        spec[3] = dict(offset=False, float32=True, nfill=1)
        spec[4] = dict(offset=False, float32=True, nfill=2)
    return spec


_DATA = {}


def _dataset(coords, nlon, nlat):
    """float fields on a grid whose longitude tables take LONW = LONW[coords] (as test_dispatch_matrix_gpu)."""
    key = (coords, nlon, nlat)
    if key not in _DATA:
        i = np.arange(nlon, dtype=np.float64)
        lat = -40.0 + 0.5 * np.arange(nlat)
        if coords == "exact":
            lon, cd = -100.0 + 0.5 * i, np.float64
        elif coords == "f32":
            lon, cd = -100.0 + 0.25 * i, np.float32
        else:
            lon, cd = -100.0 + np.cumsum(np.random.default_rng(5).uniform(0.2, 0.3, nlon)), np.float64
        time = T0 + np.arange(NT) * np.timedelta64(6, "h")
        level = np.linspace(2e4, 1e5, NLEV)
        fields = H.smooth_fields(NT, NLEV, nlat, nlon, np.float32, seed=nlon, level=level, lat=lat)
        P = H.prepared_from_arrays(fields, lon, lat, level, time, coord_dtype=cd)
        if coords == "exact":
            P.rlons = (i - 200.0) * 2.0 ** -7
        _DATA[key] = (P, fields)
    return _DATA[key]


def _plant_fills(raws, box, vecw, inside=None):
    """Fill values on the ring around ``box``, in the columns of its first and last chunk, and (``inside``) at one
    point of the box."""
    i0, i1, j0, j1 = box
    out = [r.copy() for r in raws]
    nlat, nlon = out[0].shape[2:]
    lo, hi = i0 // vecw * vecw, min(nlon - 1, (i1 // vecw + 1) * vecw - 1)
    cols = [c for c in sorted({i0 - 1, i1 + 1, *range(lo, i0), *range(i1 + 1, hi + 1)}) if 0 <= c < nlon]
    for r in out:
        r[:, :, j0:j1 + 1, cols] = FILL
        for j in (j0 - 1, j1 + 1):
            if 0 <= j < nlat:
                r[:, :, j, max(0, min(lo, i0 - 1)):hi + 2] = FILL
    if inside is not None:
        out[inside[0]][1, 2, (j0 + j1) // 2, (i0 + i1) // 2] = FILL
    return out


def _steps(P, boxes):
    steps = E.time_stencil(H.tsec_of(P), E.make_steps(len(P.time)))
    for it, b in enumerate(boxes):
        steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = b
    return steps


def _pair(P, raws, decode, boxes, arith, band_rows=0, pitch_extra=0):
    """(packed results, packed dispatch), (decoded results, decoded dispatch) on one engine configuration."""
    dtype, math, _ = ARITH[arith]
    steps = _steps(P, boxes)
    nlon = raws[0].shape[3]
    pitch = (nlon + 7) // 8 * 8 + pitch_extra
    dec_t = [torch.from_numpy(np.ascontiguousarray(H.decode(r, d, dtype))).cuda() for r, d in zip(raws, decode)]
    pk_t = [H.padded(r, pitch) for r in raws]
    with H.make_engine(P, dtype, [1.0] * 5, math=math, band_rows=band_rows) as eng:
        a = H.with_boundary(eng, len(steps), lambda: eng.run_torch_packed(pk_t, decode, steps))
        da = eng.last_dispatch()
        b = H.with_boundary(eng, len(steps), lambda: eng.run_torch(dec_t, steps))
        db = eng.last_dispatch()
    return (a, da), (b, db)


def _packed_tile_rows(arith):
    return {"f32": 11, "m64": 7, "f64": 11}[arith]


def _cell(key, boxes, arith, inside=None, **kw):
    P, fields = _dataset(*key)
    vecw = ARITH[arith][2]
    raws, decode = H.encode(fields, _decode_spec(arith))
    if len(set(boxes)) == 1:
        raws = _plant_fills(raws, boxes[0], vecw, inside)
    (a, da), (b, db) = _pair(P, raws, decode, boxes, arith, **kw)
    assert da["packed"] and not db["packed"]
    for k in ("kernel", "group", "lonw", "comp", "math64", "vec"):
        assert da[k] == db[k], (k, da, db)
    assert da["kernel"] in ("tiled", "subwarp"), da
    if da["kernel"] == "tiled":
        assert da["tile_rows"] == _packed_tile_rows(arith), da
    else:
        assert da["tile_rows"] == db["tile_rows"], (da, db)
    if inside is None:
        assert not a[2].any() and np.isfinite(a[0]).all() and np.isfinite(a[1]).all(), a[2]
        H.same_bits(a, b)
    else:
        for x, y in zip(a, b):
            assert np.array_equal(x, y, equal_nan=True)
    return a, da


def _box(chunks, vecw, i0, j0, j1):
    return (i0, (i0 // vecw + chunks - 1) * vecw + 1, j0, j1)


@pytest.mark.parametrize("coords", ["exact", "f32", "irregular"])
@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("chunks", [4, 5, 112, 113, 200, 201])
def test_width_thresholds_have_the_bits_of_the_decoded_fields(chunks, arith, coords):
    vecw = ARITH[arith][2]
    box = _box(chunks, vecw, vecw + 1, 1, 129)
    _, d = _cell((coords,) + WIDE, [box] * NT, arith)
    assert d["lonw"] == (LONW[coords] if d["kernel"] == "tiled" else (0 if coords == "exact" else 2))
    assert d["group"] == (32 if chunks > 200 else 16 if chunks > 112 else 8 if chunks > 4 else 4)


@pytest.mark.parametrize("chunks,rows,comp", [(200, 128, True), (201, 128, True), (128, 128, False), (129, 128, True),
                                              (201, 129, False)])
def test_compensated_sums_thresholds(chunks, rows, comp):
    box = _box(chunks, 4, 5, 1, rows)
    _, d = _cell(("f32",) + WIDE, [box] * NT, "f32")
    assert d["comp"] == comp


@pytest.mark.parametrize("kernel", ["subwarp", "tiled"])
@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("corner", ["first", "last"])
def test_boxes_on_the_first_and_last_column_and_row(kernel, arith, corner):
    vecw = ARITH[arith][2]
    nlon, nlat = WIDE
    if corner == "last":
        last = (nlon - 1) // vecw
        i0 = (last - 199) * vecw + 1 if kernel == "subwarp" else 1
        box = (i0, nlon - 1, 2, nlat - 1)
    else:
        box = (0, 199 * vecw + 1 if kernel == "subwarp" else nlon - 2, 0, nlat - 3)
    _, d = _cell(("f32",) + WIDE, [box] * NT, arith, pitch_extra=8)
    assert d["kernel"] == kernel


@pytest.mark.parametrize("arith", ["f32", "f64"])
@pytest.mark.parametrize("i0", range(8))
def test_every_shift_of_the_first_chunk_in_the_tiled_boxes(i0, arith):
    """The tiled kernel's int16 boxes start at the first chunk's column rounded down to a multiple of 8, so the chunk
    sits (c0 * VEC) & 7 columns into them: 0 or 4 for fp32, 0, 2, 4 or 6 for fp64.  First columns 0 ... 7 reach them
    all, on fixed boxes and on moving boxes whose first column changes every step."""
    _, d = _cell(("f32",) + WIDE, [(i0, 813, 2, 60)] * NT, arith)
    assert d["kernel"] == "tiled"
    moving = [((i0 + 3 * t) % 8, 811 - t, 2 + t, 60 + t) for t in range(NT)]
    _, d = _cell(("f32",) + WIDE, moving, arith)
    assert d["kernel"] == "tiled"


@pytest.mark.parametrize("kernel", ["subwarp", "tiled"])
@pytest.mark.parametrize("arith", ["f32", "f64"])
def test_banded_fixed_box_and_moving_boxes(kernel, arith):
    vecw = ARITH[arith][2]
    chunks = 60 if kernel == "subwarp" else 201
    fixed = _box(chunks, vecw, 3, 2, 62)
    _, d = _cell(("f32",) + WIDE, [fixed] * NT, arith, band_rows=22)
    assert d["nbands"] > 1 and d["kernel"] == kernel
    moving = [_box(chunks, vecw, 1 + t, 2 + 7 * t, 62 + 7 * t) for t in range(NT)]
    _, d = _cell(("f32",) + WIDE, moving, arith, band_rows=22)
    assert d["nbands"] > 1 and d["kernel"] == kernel


@pytest.mark.parametrize("kernel", ["subwarp", "tiled"])
@pytest.mark.parametrize("arith", ["f32", "f64"])
@pytest.mark.parametrize("field", [0, 1, 4])
def test_a_fill_inside_the_box_raises_the_nonfinite_flag(kernel, arith, field):
    vecw = ARITH[arith][2]
    box = _box(60 if kernel == "subwarp" else 204, vecw, 3, 2, 40)
    a, _ = _cell(("f32",) + WIDE, [box] * NT, arith, inside=(field,))
    assert a[2][1] & E.FLAG_NONFINITE
    if field != 0:                   # T of slot 1 is also the time neighbour of steps 0 and 2
        assert not (np.delete(a[2], 1) & E.FLAG_NONFINITE).any()


def test_the_direct_kernel_switch_does_not_apply(monkeypatch):
    monkeypatch.setenv("LEC_ROW_KERNEL", "direct")
    P, fields = _dataset("f32", *WIDE)
    raws, decode = H.encode(fields, _decode_spec("f32"))
    for chunks, kernel in ((60, "subwarp"), (201, "tiled")):
        box = _box(chunks, 4, 5, 1, 40)
        steps = _steps(P, [box] * NT)
        with H.make_engine(P, np.float32, [1.0] * 5) as eng:
            eng.run_torch_packed([H.padded(r, 816) for r in raws], decode, steps)
            d = eng.last_dispatch()
        assert d["kernel"] == kernel and d["packed"], d


def test_the_torch_operator_and_the_ctypes_route_agree(monkeypatch):
    P, fields = _dataset("f32", *WIDE)
    raws, decode = H.encode(fields, _decode_spec("f32"))
    tens = [H.padded(r, 824) for r in raws]
    outs = []
    for ext in (True, False):
        if E.load_torch_extension() != ext:
            monkeypatch.setattr(E, "_torch_ext", ext)
        assert E.load_torch_extension() == ext
        with H.make_engine(P, np.float32, [1.0] * 5) as eng:
            for box in (_box(60, 4, 5, 1, 40), _box(201, 4, 5, 1, 40)):
                outs.append(tuple(x.cpu().numpy() for x in eng.run_torch_packed(tens, decode, _steps(P, [box] * NT))))
    assert len(outs) == 4
    H.same_bits(outs[0], outs[2])
    H.same_bits(outs[1], outs[3])


def test_a_view_of_the_first_nlon_columns_is_accepted():
    P, fields = _dataset("f32", 810, 40)
    raws, decode = H.encode(fields, _decode_spec("f32"))
    box = _box(202, 4, 1, 1, 38)
    steps = _steps(P, [box] * NT)
    full = [H.padded(r, 816) for r in raws]
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        a = tuple(x.cpu().numpy() for x in eng.run_torch_packed(full, decode, steps))
        b = tuple(x.cpu().numpy() for x in eng.run_torch_packed([t[..., :810] for t in full], decode, steps))
    H.same_bits(a, b)


def test_invalid_arguments_are_rejected():
    P, fields = _dataset("f32", 810, 40)
    raws, decode = H.encode(fields, _decode_spec("f32"))
    steps = _steps(P, [_box(202, 4, 1, 1, 38)] * NT)
    good = [H.padded(r, 816) for r in raws]
    terms = torch.empty((NT, E.NTERMS), dtype=torch.float64, device="cuda")
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        ptrs = [t.data_ptr() for t in good]
        for pitch in (808, 812, 820):          # below nlon / not a multiple of 8
            with pytest.raises(ValueError, match="invalid argument"):
                eng.run_device_packed(ptrs, NT, pitch, decode, steps, terms.data_ptr())
        with pytest.raises(ValueError, match="invalid argument"):     # base 2 bytes past 16-byte alignment
            eng.run_device_packed([p + 2 for p in ptrs], NT, 816, decode, steps, terms.data_ptr())
        with pytest.raises(ValueError, match="fill"):                 # three fill values
            eng.run_device_packed(ptrs, NT, 816, [dict(decode[0], fills=[1, 2, 3])] + decode[1:], steps,
                                  terms.data_ptr())
        d = E._PackedDesc()
        d.pitch = 816
        E._set_decode(d, decode)
        d.nfill[2] = 3                                                # the C ABI checks it too
        arr = (C.c_void_p * 5)(*ptrs)
        st, sp = eng._steps_arg(steps)
        assert eng._lib.lec_run_device_packed(eng._h, C.byref(d), arr, NT, sp, NT, C.c_void_p(terms.data_ptr()),
                                              None, None, None) == -1
        with pytest.raises(ValueError, match="int16"):
            eng.run_torch_packed([t.to(torch.int32) for t in good], decode, steps)
        with pytest.raises(ValueError, match="pitch"):
            eng.run_torch_packed([torch.zeros((NT, NLEV, 40, 812), dtype=torch.int16, device="cuda")] * 5, decode,
                                 steps)
        n0 = eng.launch_count
        eng.run_device_packed(ptrs, NT, 816, decode, steps[:0], terms.data_ptr())
        assert eng.launch_count == n0


def test_era5_records_have_the_bits_of_the_raw_record_path(tmp_path):
    """The int16 ERA5-convention file (latitude north to south, levels surface first): its RawStore made resident with
    packed_device_fields gives the bits of lec_run_host_raw on the same records."""
    nc = str(tmp_path / "era5.nc")
    H.write_era5_like(nc, True, 161)
    nl = PP.read_namelist(os.path.join(H.GOLDEN, "inputs", "namelist_ERA5"))
    ds = PP.open_netcdf3(nc, nl)
    assert ds.raw is not None
    store = ds.raw.select("lat", slice(None, None, -1)).select("lev", slice(None, None, -1))
    names = list("TUVWZ")
    lat, lon = ds.lat[::-1], ds.lon
    lev = np.asarray(ds.level[::-1], dtype=np.float64) * 100.0
    rl, rp = np.deg2rad(lon), np.deg2rad(lat)
    tens, decode = PP.packed_device_fields(store, names)
    assert tens[0].dtype == torch.int16 and tens[0].stride(2) == 168
    nt = len(store.rec)
    tsec = np.arange(nt) * 3600.0
    for box in ((3, 63, 5, 65), (0, 160, 0, 140)):
        steps = E.time_stencil(tsec, E.make_steps(nt))
        steps["i0"], steps["i1"], steps["j0"], steps["j1"] = box
        with E.LecEngine(lon, lat, rl, rp, np.cos(rp), lev, np.float64, [1.0] * 5, max_steps=nt) as eng:
            a = tuple(x.cpu().numpy() for x in eng.run_torch_packed(tens, decode, steps))
            b = eng.run_host_raw([store.fields[v] for v in names], store.lon, store.lat, store.lev, store.rec, steps,
                                 decode=[store.decode[v] for v in names])
        H.same_bits(a, b)


def test_non_int16_records_are_refused(tmp_path):
    nc = str(tmp_path / "era5.nc")
    H.write_era5_like(nc, False, 160)
    nl = PP.read_namelist(os.path.join(H.GOLDEN, "inputs", "namelist_ERA5"))
    ds = PP.open_netcdf3(nc, nl)
    with pytest.raises(ValueError, match="not int16"):
        PP.packed_device_fields(ds.raw, list("TUVWZ"))


def _packed_prepared(P, names, fp32):
    """int16 encodings of the prepared fields ``names`` and P with those fields replaced by their decoded values."""
    spec = [dict(offset=not fp32, float32=fp32, nfill=1)] * len(names)
    raws, decode = H.encode([P.fields[n] for n in names], spec)
    Q = O.Prepared()
    Q.__dict__.update(P.__dict__)
    Q.fields = dict(P.fields)
    for n, r, d in zip(names, raws, decode):
        Q.fields[n] = H.decode(r, d, np.float64)
    return raws, decode, Q


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 1e-5)])
def test_catarina_fixed_box_matches_the_oracle(dtype, tol):
    P, _ = H.load_prepared("Catarina_NCEP-R2.nc")
    box = (-55, -36, -35, -20)
    P = O.slice_domain_fixed(P, *box)
    names = [n if n in P.fields else "Geopotential Height" for n in H.FIELD_ORDER]
    raws, decode, Q = _packed_prepared(P, names, fp32=dtype == np.float32)
    df, _, extra = O.lec_fixed(Q, *box, mode="fp64")
    _, scale = H.engine_inputs(Q, dtype)
    pitch = (raws[0].shape[3] + 7) // 8 * 8
    with H.make_engine(Q, dtype, scale) as eng:
        terms, _, flags = eng.run_torch_packed([H.padded(r, pitch) for r in raws], decode, H.fixed_steps(Q, *box))
        assert eng.last_dispatch()["packed"]
    errs = H.compare_terms(terms.cpu().numpy(), df, extra=extra)
    assert max(errs.values()) <= tol, errs


@pytest.mark.parametrize("dtype,tol", [(np.float64, 1e-9), (np.float32, 1e-5)])
def test_testdata_track_matches_the_oracle(dtype, tol):
    P, track = H.load_prepared("testdata_NCEP-R2.nc", track="track_testdata_NCEP-R2")
    P = O.slice_domain_track(P, track)
    names = [n if n in P.fields else "Geopotential Height" for n in H.FIELD_ORDER]
    raws, decode, Q = _packed_prepared(P, names, fp32=dtype == np.float32)
    df, _, _ = O.lec_moving(Q, track, mode="fp64")
    _, scale = H.engine_inputs(Q, dtype)
    pitch = (raws[0].shape[3] + 7) // 8 * 8
    steps = H.moving_steps(Q, track)
    with H.make_engine(Q, dtype, scale, max_box_rows=int((steps["j1"] - steps["j0"]).max()) + 1) as eng:
        terms, _, flags = eng.run_torch_packed([H.padded(r, pitch) for r in raws], decode, steps)
    errs = H.compare_terms(terms.cpu().numpy(), df)
    assert len(errs) >= 14 and max(errs.values()) <= tol, errs
