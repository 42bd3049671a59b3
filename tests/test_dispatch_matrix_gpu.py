"""Every row kernel the dispatcher of ``run_batch`` (csrc/lec_engine.cu) can choose, against the fp64 oracle.

Each case first asserts the template instance it was built for (``LecEngine.last_dispatch()``), then compares all
16 terms and the 19 per-level families with ``O.lec_fixed`` / ``O.lec_moving(mode="fp64")`` under the gates of the
other parity files (1e-9 for fp64 arithmetic, 1e-5 for fp32).  The cells (a chunk is 128 bits of a row: 4 fp32
or 2 fp64 columns; a box row covers ``i1 // vecw - i0 // vecw + 1`` chunks):

  sub-warp kernel, G = 4 / 8 / 16 lanes per row    <= 4 / 5-112 / 113-200 chunks, 16-byte aligned rows
  TMA-tiled kernel                                  201+ chunks (R = 15 rows per tile, 11 with COMP or fp64
                                                    fields, 7 for fp32 fields with fp64 arithmetic)
  compensated fp32 linear sums (COMP)               129+ chunks and <= 128 rows
  longitude tables LONW = 0 / 1 / 2                 exactly uniform / per-column weights / irregular stencil
  scalar direct kernel (VEC = 1)                    caller-owned device rows that are not 16-byte aligned
  vector direct kernel                              LEC_ROW_KERNEL=direct (opt-in)
  latitude-banded block order                       lec_grid_desc.band_rows > 0, fixed and moving boxes

Cells of 16-byte aligned rows run through ``lec_run_host`` (rows padded to whole chunks) and through
``lec_run_device`` on the caller's tensors (pitch = nlon) and must give the same bits: the lane <-> column
mapping depends on ``i0 // vecw`` only.  Fixed boxes carry NaNs on the ring around the box (columns i0-1, i1+1,
rows j0-1, j1+1) and in the columns that share the box's first and last chunk; no kernel may read them into a
result.  The last test asserts that the module reached every cell, so that a retuned threshold shows up as a
failure instead of as a case that silently moved to another kernel."""
import functools

import numpy as np
import pandas as pd
import pytest

from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E
import helpers as H

pytestmark = pytest.mark.gpu
TOL = {"f32": 1e-5, "m64": 1e-9, "f64": 1e-9}
# arithmetic -> (field dtype, lec_grid_desc.math, columns per chunk)
ARITH = {"f32": (np.float32, E.LEC_MATH_AUTO, 4), "m64": (np.float32, E.LEC_MATH_F64, 4),
         "f64": (np.float64, E.LEC_MATH_AUTO, 2)}
LONW = {"exact": 0, "f32": 1, "irregular": 2}            # lon_mode() of each coordinate set
T0 = np.datetime64("2020-01-01T00")
NT, NLEV = 4, 4
RECORDS = []                                            # (dispatch record + case facts) of every run


@pytest.fixture(autouse=True)
def _default_dispatcher(monkeypatch):
    for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
        monkeypatch.delenv(k, raising=False)


@functools.lru_cache(maxsize=None)
def _dataset(coords, nlon, nlat):
    """float32-valued fields (the fp64 cells run them upcast, so one oracle result serves every arithmetic) on a
    grid whose longitude tables take LONW = ``LONW[coords]`` under fp32 and fp64 arithmetic alike."""
    i = np.arange(nlon, dtype=np.float64)
    lat = -40.0 + 0.5 * np.arange(nlat)
    if coords == "exact":          # exactly uniform in fp64: degrees i / 2 (stencil) and radians i / 128 (weights);
        lon, cd = -100.0 + 0.5 * i, np.float64      # the oracle takes trapezoid weights from rlons, derivatives from lon
    elif coords == "f32":          # float32 radians: trapezoid weights spread by ~3e-5, stencil exact
        lon, cd = -100.0 + 0.25 * i, np.float32
    else:
        lon, cd = -100.0 + np.cumsum(np.random.default_rng(5).uniform(0.2, 0.3, nlon)), np.float64
    time = T0 + np.arange(NT) * np.timedelta64(6, "h")
    level = np.linspace(2e4, 1e5, NLEV)
    fields = H.smooth_fields(NT, NLEV, nlat, nlon, np.float32, seed=nlon, level=level, lat=lat)
    P = H.prepared_from_arrays(fields, lon, lat, level, time, coord_dtype=cd)
    if coords == "exact":
        P.rlons = (i - 200.0) * 2.0 ** -7
    return P, fields


_REF = {}


def _reference(key, P, boxes):
    """Oracle results of one dataset and one box per step, cached: several cells share a box."""
    k = (key, tuple(boxes))
    if k not in _REF:
        if len(set(boxes)) == 1:
            i0, i1, j0, j1 = boxes[0]
            df, lv, extra = O.lec_fixed(P, float(P.lon[i0]), float(P.lon[i1]), float(P.lat[j0]), float(P.lat[j1]),
                                        mode="fp64")
            assert extra["box"].idx == boxes[0]
            extra = {n: extra[n] for n in ("BΦZ", "BΦE")}
        else:                      # a track whose limits fall on the grid points of each box
            lon, lat = np.asarray(P.lon, np.float64), np.asarray(P.lat, np.float64)
            track = pd.DataFrame({"Lat": [(lat[b[2]] + lat[b[3]]) / 2 for b in boxes],
                                  "Lon": [(lon[b[0]] + lon[b[1]]) / 2 for b in boxes],
                                  "length": [lat[b[3]] - lat[b[2]] for b in boxes],
                                  "width": [lon[b[1]] - lon[b[0]] for b in boxes]}, index=pd.to_datetime(P.time))
            df, lv, got = O.lec_moving(P, track, mode="fp64")
            assert [idx for _, idx in got] == list(boxes)
            extra = None
        _REF[k] = (df, lv, extra)
    return _REF[k]


def _nan_ring(fields, box, vecw):
    """Copies of ``fields`` with NaN on every slot and level where a kernel must not look for ``box``."""
    i0, i1, j0, j1 = box
    out = [f.copy() for f in fields]
    nlat, nlon = out[0].shape[2:]
    lo, hi = i0 // vecw * vecw, min(nlon - 1, (i1 // vecw + 1) * vecw - 1)      # first / last column of its chunks
    cols = [c for c in sorted({i0 - 1, i1 + 1, *range(lo, i0), *range(i1 + 1, hi + 1)}) if 0 <= c < nlon]
    for f in out:
        f[:, :, j0:j1 + 1, cols] = np.nan
        for j in (j0 - 1, j1 + 1):
            if 0 <= j < nlat:
                f[:, :, j, max(0, min(lo, i0 - 1)):hi + 2] = np.nan
    return out


def _device(a, misaligned):
    import torch
    t = torch.from_numpy(a)
    if not misaligned:
        return t.cuda()
    buf = torch.empty(a.size + 1, dtype=t.dtype, device="cuda")     # base pointer one whole element past alignment
    x = buf[1:].view(a.shape)
    x.copy_(t)
    assert x.is_contiguous() and x.data_ptr() % 16 != 0
    return x


def _run(P, fields, boxes, arith, route, band_rows=0, misaligned=False):
    dtype, math, _ = ARITH[arith]
    arrs = [np.ascontiguousarray(f, dtype=dtype) for f in fields]
    steps = E.time_stencil(H.tsec_of(P), E.make_steps(len(P.time)))
    for it, b in enumerate(boxes):
        steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = b
    with H.make_engine(P, dtype, [1.0] * 5, math=math, band_rows=band_rows) as eng:
        if route == "host":
            out = eng.run_host(arrs, steps)
        else:
            out = tuple(x.cpu().numpy() for x in eng.run_torch([_device(a, misaligned) for a in arrs], steps))
        return out, eng.last_dispatch()


def _check(out, ref, tol):
    terms, levels, flags = out
    assert not flags.any(), flags
    assert np.isfinite(terms).all() and np.isfinite(levels).all()
    df, lv, extra = ref
    errs = H.compare_terms(terms, df, extra=extra)
    assert set(errs) == set(E.TERM_NAMES)
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, bad
    lerrs = H.compare_levels(levels, lv)
    assert set(lerrs) == set(E.LEVEL_TERM_NAMES)
    bad = {k: v for k, v in lerrs.items() if not v <= tol}
    assert not bad, bad


def _cell(key, boxes, arith, want, routes=("host", "torch"), **kw):
    """Run one box per step through each route: assert the dispatch ``want``, the oracle within the gate of the
    arithmetic, and the same bits on every route.  Returns the results and the dispatch record of the last route."""
    P, fields = _dataset(*key)
    vecw = ARITH[arith][2]
    ref = _reference(key, P, boxes)
    if len(set(boxes)) == 1:
        fields = _nan_ring(fields, boxes[0], vecw)
    outs = []
    for route in routes:
        out, d = _run(P, fields, boxes, arith, route, **kw)
        RECORDS.append(dict(d, arith=arith, fields="f64" if arith == "f64" else "f32", nlon=key[1], route=route,
                            chunks=max(b[1] // vecw - b[0] // vecw + 1 for b in boxes),
                            rows=max(b[3] - b[2] + 1 for b in boxes), misaligned=kw.get("misaligned", False),
                            banded=d["nbands"] > 1, moving=len(set(boxes)) > 1))
        assert {k: d[k] for k in want} == want, d
        _check(out, ref, TOL[arith])
        outs.append(out)
    for o in outs[1:]:
        for x, y in zip(outs[0], o):
            assert np.array_equal(x, y)
    return outs[-1], d


def _box(chunks, vecw, i0, j0, j1):
    """Columns i0 ... i1 over exactly ``chunks`` chunks, i1 one column into its chunk (padding columns after it)."""
    return (i0, (i0 // vecw + chunks - 1) * vecw + 1, j0, j1)


def _tile_rows(arith, comp=False):
    return {"f32": 11 if comp else 15, "m64": 7, "f64": 11}[arith]


WIDE = (816, 131)        # fp32: 204 chunks per row, fp64: 408; rows 1 ... 129 leave a ring row on either side


def _want_width(chunks, arith, coords, comp=False):
    vecw = ARITH[arith][2]
    if chunks > 200:
        return dict(kernel="tiled", vec=vecw, group=32, lonw=LONW[coords], comp=comp, math64=arith != "f32",
                    tile_rows=_tile_rows(arith, comp))
    return dict(kernel="subwarp", vec=vecw, group=4 if chunks <= 4 else 8 if chunks <= 112 else 16,
                lonw=0 if coords == "exact" else 2, comp=comp, math64=arith != "f32")


# ---------------------------------------------------------------------------------------------------------------- #
WIDTHS = [4, 5, 112, 113, 200, 201]


@pytest.mark.parametrize("coords", ["exact", "f32", "irregular"])
@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("chunks", WIDTHS)
def test_width_thresholds(chunks, arith, coords):
    """Both sides of every group-width threshold (4/5, 112/113 chunks) and of the tiled kernel (200/201), an odd
    first column, 129 rows (no COMP)."""
    vecw = ARITH[arith][2]
    box = _box(chunks, vecw, vecw + 1, 1, 129)
    _cell((coords,) + WIDE, [box] * NT, arith, _want_width(chunks, arith, coords))


@pytest.mark.parametrize("kernel", ["subwarp", "tiled"])
@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
def test_box_on_the_last_column_and_row(kernel, arith):
    vecw = ARITH[arith][2]
    nlon, nlat = WIDE
    last = (nlon - 1) // vecw
    i0 = (last - 199) * vecw + 1 if kernel == "subwarp" else 1          # 200 chunks / the whole row
    box = (i0, nlon - 1, 2, nlat - 1)
    chunks = last - i0 // vecw + 1
    assert (chunks == 200) == (kernel == "subwarp")
    _cell(("f32",) + WIDE, [box] * NT, arith, _want_width(chunks, arith, "f32"))


COMP_CASES = [(200, 128, True), (201, 128, True), (128, 128, False), (129, 128, True)]


@pytest.mark.parametrize("chunks,rows,comp", COMP_CASES)
def test_compensated_sums_thresholds(chunks, rows, comp):
    """COMP in the sub-warp and the tiled kernel: 128 / 129 chunks at 128 rows (129 rows: test_width_thresholds)."""
    box = _box(chunks, 4, 5, 1, rows)
    _cell(("f32",) + WIDE, [box] * NT, "f32", _want_width(chunks, "f32", "f32", comp=comp))


VECTOR_DIRECT = [("f32", "exact"), ("f32", "f32"), ("f32", "irregular"), ("m64", "f32"), ("f64", "f32")]


@pytest.mark.parametrize("arith,coords", VECTOR_DIRECT)
def test_vector_direct_kernel(arith, coords, monkeypatch):
    """``LEC_ROW_KERNEL=direct``: wide boxes through the direct-load warp-per-row kernel instead of the TMA ring."""
    monkeypatch.setenv("LEC_ROW_KERNEL", "direct")
    vecw = ARITH[arith][2]
    box = _box(201, vecw, vecw + 1, 1, 129)
    _cell((coords,) + WIDE, [box] * NT, arith, dict(kernel="direct", vec=vecw, group=32, lonw=LONW[coords],
                                                    comp=False, math64=arith != "f32", tile_rows=2))


@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("chunks", [5, 201])
def test_direct_kernel_on_a_misaligned_base(chunks, arith):
    """Caller-owned fields whose base pointer is one element past 16-byte alignment (rows of whole chunks): the
    scalar direct kernel, for narrow and wide boxes."""
    vecw = ARITH[arith][2]
    box = _box(chunks, vecw, vecw + 1, 1, 129)
    _cell(("f32",) + WIDE, [box] * NT, arith, dict(kernel="direct", vec=1, group=32, lonw=1, comp=False,
                                                   math64=arith != "f32"),
          routes=("torch",), misaligned=True)


SCALAR_GRIDS = [("f32", "f32", 301), ("f32", "f32", 302), ("f32", "f32", 303), ("f32", "exact", 301),
                ("f32", "irregular", 301), ("m64", "f32", 301), ("f64", "f32", 301), ("f64", "f32", 303)]


@pytest.mark.parametrize("shape", ["narrow", "wide", "edge"])
@pytest.mark.parametrize("arith,coords,nlon", SCALAR_GRIDS)
def test_scalar_direct_kernel(arith, coords, nlon, shape):
    """``lec_run_device`` on rows of nlon % 4 = 1, 2, 3 (fp32) and odd nlon (fp64) columns: the rows of the
    caller's tensors are not 16-byte aligned, so the VEC = 1 branch of lec_row_body.inc runs.  (``lec_run_host``
    pads the same grid to whole chunks and takes the vector kernels: another lane <-> column mapping, so the two
    routes agree to the gate, not to the bit.)"""
    nlat = 41
    box = {"narrow": (5, 14, 3, 12), "wide": (1, 290, 1, 38), "edge": (150, nlon - 1, 20, nlat - 1)}[shape]
    _cell((coords, nlon, nlat), [box] * NT, arith, dict(kernel="direct", vec=1, group=32, lonw=LONW[coords],
                                                       comp=False, math64=arith != "f32"), routes=("torch",))


# ---------------------------------------------------------------------------------------------------------------- #
BAND_GRID = ("exact", 406, 70)        # 406 % 4 == 2: fp32 device rows are not 16-byte aligned (scalar kernel)
# family -> (arithmetic, route, env, fixed box, moving boxes of one height: 61 rows, no multiple of any band below)
BAND_FAMILIES = {
    "subwarp": ("f32", "host", {}, (3, 150, 3, 63), [(3, 150, 3, 63), (6, 153, 5, 65), (1, 148, 4, 64), (8, 155, 6, 66)]),
    "tiled": ("f64", "host", {}, (1, 401, 3, 63), [(1, 401, 3, 63), (0, 400, 5, 65), (4, 404, 4, 64), (2, 402, 6, 66)]),
    "direct": ("f32", "torch", {}, (3, 150, 3, 63), [(3, 150, 3, 63), (6, 153, 5, 65), (1, 148, 4, 64), (8, 155, 6, 66)]),
}
BAND_CASES = [(f, m) for f in BAND_FAMILIES for m in ("fixed", "moving")]


@pytest.mark.parametrize("family,motion", BAND_CASES)
def test_banded_order(family, motion, monkeypatch):
    """``band_rows`` > 0: a request that is no multiple of the family's rows per tile (rounded down to one), a box
    height that is no multiple of the band; several bands, and the bits of the step-major order."""
    arith, route, env, fixed, moving = BAND_FAMILIES[family]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    boxes = [fixed] * NT if motion == "fixed" else moving
    base, d0 = _cell(BAND_GRID, boxes, arith, dict(kernel=family, nbands=1), routes=(route,))
    tr = d0["tile_rows"]
    req = tr * max(1, (61 // tr) // 2) + 1
    out, d = _cell(BAND_GRID, boxes, arith, dict(kernel=family, tile_rows=tr), routes=(route,), band_rows=req)
    band = d["tiles_per_band"] * tr
    assert d["nbands"] > 1 and band == req - 1 and 61 % band != 0, d
    for x, y in zip(base, out):
        assert np.array_equal(x, y)


# ---------------------------------------------------------------------------------------------------------------- #
def _cells_required():
    req = []
    for arith, fl in (("f32", "f32"), ("m64", "f32"), ("f64", "f64")):
        req += [dict(kernel="subwarp", group=g, arith=arith, vec=ARITH[arith][2]) for g in (4, 8, 16)]
        req += [dict(kernel="tiled", arith=arith, tile_rows=_tile_rows(arith))]
        req += [dict(kernel="direct", vec=1, arith=arith), dict(kernel="direct", vec=ARITH[arith][2], arith=arith)]
        req += [dict(kernel="direct", vec=1, misaligned=True, fields=fl)]
    req += [dict(kernel="direct", vec=1, fields="f32", route="torch", nlon=n) for n in (301, 302, 303)]
    req += [dict(kernel="direct", vec=1, fields="f64", route="torch", nlon=n) for n in (301, 303)]
    # thresholds, fp32: group width, tiled kernel, COMP by width and by height
    req += [dict(arith="f32", chunks=c, kernel=k, group=g, comp=False)
            for c, k, g in ((4, "subwarp", 4), (5, "subwarp", 8), (112, "subwarp", 8), (113, "subwarp", 16),
                            (200, "subwarp", 16), (201, "tiled", 32))]
    req += [dict(arith="f32", kernel=k, chunks=c, rows=r, comp=comp)
            for k, c, r, comp in (("subwarp", 128, 128, False), ("subwarp", 129, 128, True), ("subwarp", 200, 128, True),
                                  ("subwarp", 200, 129, False), ("tiled", 201, 128, True), ("tiled", 201, 129, False))]
    req += [dict(kernel="tiled", arith="f32", comp=True, tile_rows=11)]
    for kernel, lonws in (("direct", (0, 1, 2)), ("subwarp", (0, 2)), ("tiled", (0, 1, 2))):
        req += [dict(kernel=kernel, lonw=w) for w in lonws]
        req += [dict(kernel=kernel, banded=True, moving=m) for m in (False, True)]
    return req


N_CASES = (len(WIDTHS) * 9 + 6 + len(COMP_CASES) + len(VECTOR_DIRECT) + 6 + len(SCALAR_GRIDS) * 3
           + len(BAND_CASES))


def test_every_dispatch_cell_was_reached(request):
    """The cells the cases above reached contain the whole matrix: a threshold that moves makes this fail."""
    mine = [it for it in request.session.items if it.module is request.module and it is not request.node]
    if len(mine) < N_CASES:
        pytest.skip("needs the whole module: the dispatch records of every case")
    missing = [r for r in _cells_required() if not any(all(x.get(k) == v for k, v in r.items()) for x in RECORDS)]
    assert not missing, missing
