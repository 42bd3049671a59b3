"""The host paths in front of the row kernels: ``lec_run_host_raw`` (the raw-record ingest kernel, then the staging
windows), and ``lec_run_host`` on the grids it sends through the same ingest with identity maps.

``lec_ingest_kernel`` (csrc/lec_ingest.cuh) decodes four engine columns per thread.  Its three branches:
  vector   the four raw columns are consecutive and the first is aligned to four elements: one 8-, 16- or 32-byte
           load (int16: one 8-byte load unpacked into four lanes; fp64: two 16-byte loads);
  element  four element loads (a seam, a reversed axis, a misaligned crop or row);
  tail     the last, partial group of a row (``nlon % 4`` columns), written element by element.
``_kinds`` models that predicate in numpy, so each case below knows which branches it ran.

A. Load paths: every raw type and handle type (int16 decoded to fp32 and to fp64, into either handle; fp32 and fp64
   records), native and big-endian interleaved records, six longitude maps (identity, crops on and off a multiple of
   4, wraps by a multiple of 4 and not, a reversed axis), every ``nlon % 4`` of fp32 handles and even / odd ``nlon``
   of fp64 handles; levels scrambled with extra raw levels, rows north to south, a row sub-range (the strided 3-D
   copy) with the crops.  A whole-grid box and an interior box at every slot.  References: ``run_host`` on the
   numpy-decoded arrays (always), ``run_torch_packed`` on the same int16 values (an independent decode in the row
   kernels), ``run_torch`` on the decoded fields where the engine rows are unpadded, the fp64 oracle at 1e-9 on fp64
   handles.  A last test fails unless every (raw type, byte order, branch) cell was reached.
B. Decode rules and fills: every int16 combination of scale / offset / float32 rounding into both handle types, fp32
   and fp64 records; no fill, one, two equal and two distinct fill values (the int16 extremes -32768 and 32767); fills
   in each lane of a vector group, in a tail group, on the first and last column, row and touched raw level, in
   native and big-endian records.  Probe boxes around each fill: the box whose edge is the fill's column (row) is
   non-finite, the box one column (row) further is finite and has the reference's bits.
D. bench.py's ``e2e`` and ``e2e.packed_int16`` configurations at C4 size, through one, 11-slot and 3-slot staging
   windows (the staging windows on small grids are in tests/test_raw_ingest_gpu.py)."""
import functools
import gc
import time

import numpy as np
import pytest

import bench
import helpers as H
from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E, synthetic as S
from test_engine_synthetic_gpu import _dataset
from test_production_scale_gpu import BENCH_BOX, C4_SLOT, DISPATCH_KEYS, GIB, ROW_KEYS, _bench_steps, _need, _run, \
    _solo_env

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(autouse=True)
def _default_dispatcher_and_report(monkeypatch, request):
    for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
        monkeypatch.delenv(k, raising=False)
    t0 = time.perf_counter()
    yield
    gc.collect()
    if torch.cuda.is_available():
        torch.cuda.empty_cache()
    if request.node.name.startswith("test_e2e"):
        print(f"\n{request.node.name}: {time.perf_counter() - t0:.1f} s")


VECTOR, ELEMENT, TAIL = 0, 1, 2
KIND_NAMES = ("vector", "element", "tail")


def _kinds(lon_map, lat_map, lev_map, rlon):
    """Branch of every 4-column group of every engine row, ``[level][row][group]``, as ``lec_ingest_kernel`` takes it:
    tail when fewer than four columns are left; vector when the four raw columns are consecutive and the first one's
    index in the raw staging buffer (levels ``kr_lo..``, rows ``jr_lo..`` of one record; a cudaMalloc base) is a
    multiple of 4; element otherwise."""
    lon_map, lat_map, lev_map = (np.asarray(m, dtype=np.int64) for m in (lon_map, lat_map, lev_map))
    n = lon_map.size
    nj = int(lat_map.max() - lat_map.min() + 1)
    rows = (lev_map[:, None] - lev_map.min()) * nj + (lat_map[None, :] - lat_map.min())
    out = np.empty((lev_map.size, lat_map.size, (n + 3) // 4), dtype=np.int8)
    for g, i4 in enumerate(range(0, n, 4)):
        r = lon_map[i4:i4 + 4]
        if r.size < 4:
            out[:, :, g] = TAIL
        elif not np.array_equal(r, r[0] + np.arange(4)):
            out[:, :, g] = ELEMENT
        else:
            out[:, :, g] = np.where((rows * rlon + r[0]) % 4 == 0, VECTOR, ELEMENT)
    return out


def _records(rng, vals, lon_map, rlon, lat_map, rnlat, lev_map, rnlev, rec_of_slot, nrec, order):
    """Five raw record arrays ``[record][level][lat][lon]`` holding the engine-layout ``vals`` where the maps say and
    junk elsewhere; ``order == "big"``: big-endian, the records of the five variables interleaved in one buffer."""
    dt = vals[0].dtype
    shape = (nrec, rnlev, rnlat, rlon)
    if order == "big":
        buf = np.empty((nrec, 5) + shape[1:], dtype=dt.newbyteorder(">"))
        raws = [buf[:, f] for f in range(5)]
    else:
        raws = [np.empty(shape, dtype=dt) for _ in range(5)]
    idx = np.ix_(np.asarray(rec_of_slot), np.asarray(lev_map), np.asarray(lat_map), np.asarray(lon_map))
    for r, v in zip(raws, vals):
        if dt == np.int16:
            r[...] = rng.integers(-30000, 30000, size=shape, dtype=np.int16)
        else:
            r[...] = rng.normal(size=shape) * 1e3
        r[idx] = v
    return raws


def _same(got, ref, what):
    """(terms, levels, flags, pieces): NaN at the same places, every other bit equal."""
    for name, x, y in zip(("terms", "levels", "flags", "pieces"), got, ref):
        assert x.shape == y.shape, (what, name)
        if x.dtype.kind == "f":
            nx, ny = np.isnan(x), np.isnan(y)
            assert np.array_equal(nx, ny), f"{what}: {name} NaN at other places"
            x, y = np.where(nx, 0.0, x), np.where(ny, 0.0, y)
        bad = np.flatnonzero((x.view(np.uint8) != y.view(np.uint8)).reshape(x.shape[0], -1).any(axis=1))
        assert bad.size == 0, f"{what}: {name} differ in steps {bad.tolist()}"


def _host(eng, fields, steps):
    out = eng.run_host(fields, steps, want_boundary=True)
    return out + (eng.last_boundary.copy(),)


def _host_raw(eng, raws, maps, slot_record, steps, decode):
    out = eng.run_host_raw(raws, *maps, slot_record, steps, decode=decode, want_boundary=True)
    return out + (eng.last_boundary.copy(),)


def _pitch(n, dtype):
    """Row length of the engine's own staging: whole 16-byte chunks."""
    per = 16 // np.dtype(dtype).itemsize
    return (n + per - 1) // per * per


# ---------------------------------------------------------------------------------------------------------------- #
# A. load paths
NLAT_A, NLEV_A, NT_A = 7, 3, 4
RAWS = {     # name -> (raw dtype, handle dtype, int16 packing as helpers.encode takes it)
    "i16_f32": (np.int16, np.float32, dict(offset=False, float32=True, nfill=0)),
    "i16_f64": (np.int16, np.float64, dict(offset=True, float32=False, nfill=0)),
    "i16f32_in_f64": (np.int16, np.float64, dict(offset=False, float32=True, nfill=0)),
    "i16f64_in_f32": (np.int16, np.float32, dict(offset=True, float32=False, nfill=0)),
    "f32": (np.float32, np.float32, None),
    "f64": (np.float64, np.float64, None),
}
LON_MAPS = ("identity", "crop4", "crop5", "wrap8", "wrap7", "reversed")
WIDTHS = {np.float32: (32, 33, 34, 35), np.float64: (34, 35)}
ORDERS = ("little", "big")
CASES_A = [(raw, order, lonm, n) for raw, (_, hdt, _) in RAWS.items() for order in ORDERS for lonm in LON_MAPS
           for n in WIDTHS[hdt]]
CELLS = set()            # (raw dtype, byte order, branch) the cases reached, by the model
PACKED_COMPARED = set()  # raw names whose run_torch_packed reference ran the row kernel instance of run_host_raw


def _lon_map(kind, n):
    """Engine column -> raw column, and the raw row length."""
    i = np.arange(n)
    return {"identity": (i, n), "crop4": (8 + i, n + 12), "crop5": (5 + i, n + 12), "wrap8": ((i + 8) % n, n),
            "wrap7": ((i + 7) % n, n), "reversed": (n - 1 - i, n)}[kind]


def _lat_map(kind, nlat):
    """Rows stored north to south; with the crops a row sub-range of a taller record (the strided 3-D copy)."""
    if kind in ("crop4", "crop5"):
        return nlat + 1 - np.arange(nlat), nlat + 3
    return nlat - 1 - np.arange(nlat), nlat


def _lev_map(rng, nlev, extra=2):
    """Levels in any order, with extra raw levels (some inside the touched range, which crosses PCIe too)."""
    return np.argsort(rng.permutation(nlev + extra))[:nlev], nlev + extra


@functools.lru_cache(maxsize=None)
def _data_a(raw, n):
    """(decoded dataset, raw values in engine layout, decoded engine-layout arrays, decode dicts) of one raw type and
    width; the layout of the records does not change them."""
    rdt, hdt, spec = RAWS[raw]
    P, fields = _dataset(n, NLAT_A, NLEV_A, NT_A, np.float64, seed=n)
    if spec is None:
        vals, decode = [f.astype(rdt) for f in fields], None
        decoded = [v.astype(hdt) for v in vals]
    else:
        vals, decode = H.encode(fields, [spec] * 5)
        decoded = [H.decode(q, d, hdt) for q, d in zip(vals, decode)]
    return H.prepared_from_arrays(decoded, P.lon, P.lat, P.level, P.time), vals, decoded, decode


def _steps_a(P, n):
    """The whole grid at every slot (every decoded value enters a result), then an interior box at every slot."""
    nt = len(P.time)
    out = []
    for box in ((0, n - 1, 0, NLAT_A - 1), (2, n - 4, 1, NLAT_A - 2)):
        st = E.time_stencil(H.tsec_of(P), E.make_steps(nt))
        st["i0"], st["i1"], st["j0"], st["j1"] = box
        out.append(st)
    return np.concatenate(out)


@functools.lru_cache(maxsize=None)
def _oracle_a(raw, n):
    P = _data_a(raw, n)[0]
    Q = O.to_mode(P, "fp64")
    dTdt = O.differentiate(Q.fields["Air Temperature"], H.tsec_of(Q), 0)
    return [H.oracle_step(Q, tuple(int(s[k]) for k in ("i0", "i1", "j0", "j1")), int(s["slot"]), dTdt)
            for s in _steps_a(P, n)]


@pytest.mark.parametrize("raw,order,lonm,n", CASES_A)
def test_ingest_load_paths(raw, order, lonm, n):
    rdt, hdt, spec = RAWS[raw]
    P, vals, decoded, decode = _data_a(raw, n)
    rng = np.random.default_rng(1000 * n + 10 * LON_MAPS.index(lonm) + ORDERS.index(order))
    lon_map, rlon = _lon_map(lonm, n)
    lat_map, rnlat = _lat_map(lonm, NLAT_A)
    lev_map, rnlev = _lev_map(rng, NLEV_A)
    rec = 1 + np.arange(NT_A)                      # a time selection: record 0 and the last one are not read
    raws = _records(rng, vals, lon_map, rlon, lat_map, rnlat, lev_map, rnlev, rec, NT_A + 2, order)
    kinds = _kinds(lon_map, lat_map, lev_map, rlon)
    CELLS.update((np.dtype(rdt).name, order, KIND_NAMES[k]) for k in np.unique(kinds))
    steps = _steps_a(P, n)
    with H.make_engine(P, hdt, [1.0] * 5) as eng:
        got = _host_raw(eng, raws, (lon_map, lat_map, lev_map), rec, steps, decode)
        d = eng.last_dispatch()
        assert not got[2].any()
        _same(got, _host(eng, decoded, steps), "run_host on the decoded arrays")
        if spec is not None:          # the row kernels' own int16 decode, rows padded to a multiple of 8
            pk = _run(eng, [H.padded(v, (n + 7) // 8 * 8) for v in vals], steps, decode)
            dp = eng.last_dispatch()
            if {k: dp[k] for k in ROW_KEYS} == {k: d[k] for k in ROW_KEYS}:
                _same(got, pk, "run_torch_packed on the int16 values")
                PACKED_COMPARED.add(raw)
        if _pitch(n, hdt) == n:       # unpadded rows: the device-resident fields are the staging layout
            tr = _run(eng, [torch.from_numpy(x).cuda() for x in decoded], steps)
            dt = eng.last_dispatch()
            assert {k: dt[k] for k in DISPATCH_KEYS} == {k: d[k] for k in DISPATCH_KEYS}, (dt, d)
            _same(got, tr, "run_torch on the decoded fields")
    if hdt == np.float64:
        H.check_refs(got, _oracle_a(raw, n), 1e-9)


def test_every_ingest_cell_was_reached(request):
    """The load-path cases reached, by the model of the branch predicate, every cell of
    {int16, float32, float64} x {little-endian, big-endian interleaved} x {vector, element, tail}, and the int16 cases
    met run_torch_packed's bits under the same row-kernel instance for every int16 raw type."""
    mine = [it for it in request.session.items if it.module is request.module
            and getattr(it, "originalname", None) == "test_ingest_load_paths"]
    if len(mine) < len(CASES_A):
        pytest.skip("needs every case of test_ingest_load_paths")
    required = {(t, o, k) for t in ("int16", "float32", "float64") for o in ORDERS for k in KIND_NAMES}
    assert not required - CELLS, sorted(required - CELLS)
    assert PACKED_COMPARED == {r for r, (rdt, _, _) in RAWS.items() if rdt == np.int16}, PACKED_COMPARED


# ---------------------------------------------------------------------------------------------------------------- #
# B. decode rules and fill placement
NB, NLAT_B, NLEV_B = 35, 9, 4
LON_B = 8 + np.arange(NB)                 # a crop on a multiple of 4 of 48-column rows: vector groups, then the tail
RLON_B = NB + 13
LAT_B = NLAT_B - 1 - np.arange(NLAT_B)
LEV_B = np.array([4, 1, 3, 2])            # raw levels 1..4 of 6 touched, in another order
UNITS_B = [1.0, 1.0, 1.0, 1e-3, 10.0]     # omega stored in mPa/s, Phi in 10 m^2/s^2: every field fits int16 unscaled
K_FIRST, K_LAST = int(np.argmin(LEV_B)), int(np.argmax(LEV_B))
FILLS_B = [      # (where, field, level, row, column)
    ("lane 0", 0, 2, 4, 12), ("lane 1", 1, 0, 3, 17), ("lane 2", 2, 3, 5, 22), ("lane 3", 3, 1, 4, 27),
    ("tail group", 4, 2, 6, 33), ("first column", 0, 1, 2, 0), ("last column", 1, 2, 7, 34),
    ("first raw level", 2, K_FIRST, 1, 9), ("last raw level", 0, K_LAST, 6, 30), ("first row", 3, 0, 0, 5),
    ("last row", 4, 3, NLAT_B - 1, 20),
]
NT_B = 2 * len(FILLS_B) + 1               # fill p at slot 2p + 1: no step reads two of them
FILL_VALUES = {np.int16: (-32768, 32767), np.float32: (-9999.0, float(np.float32(9.969209968386869e36))),
               np.float64: (-9999.0, 9.969209968386869e36)}
NFILLS = {"none": [], "one": [0], "equal": [0, 0], "distinct": [0, 1]}     # indices into FILL_VALUES
I16_RULES = [(s, o, r) for s in (True, False) for o in (True, False) for r in (True, False)]
CASES_B = ([("int16", rule, hdt, nf, order) for rule in I16_RULES for hdt in ("f32", "f64") for nf in NFILLS
            for order in ORDERS] +
           [(rt, None, rt, nf, order) for rt in ("f32", "f64") for nf in NFILLS for order in ORDERS])
DT = {"f32": np.float32, "f64": np.float64}


def test_fill_positions_are_where_they_claim():
    """The lanes, the tail group and the edges of FILLS_B, by the branch model."""
    kinds = _kinds(LON_B, LAT_B, LEV_B, RLON_B)
    for where, f, k, j, c in FILLS_B:
        if where.startswith("lane"):
            assert kinds[k, j, c // 4] == VECTOR and c % 4 == int(where[-1]), where
    assert kinds[FILLS_B[4][2], FILLS_B[4][3], FILLS_B[4][4] // 4] == TAIL
    assert {c for _, _, _, _, c in FILLS_B} >= {0, NB - 1} and {j for _, _, _, j, _ in FILLS_B} >= {0, NLAT_B - 1}
    assert LEV_B[K_FIRST] == LEV_B.min() and LEV_B[K_LAST] == LEV_B.max()


def _probe_pairs(j, c):
    """Boxes around (row j, column c): pairs (box with the point on its edge, the same box one column / row away)."""
    rows = (max(0, min(j - 1, NLAT_B - 3)), max(0, min(j - 1, NLAT_B - 3)) + 2)
    cols = (max(0, min(c - 1, NB - 3)), max(0, min(c - 1, NB - 3)) + 2)
    pairs = []
    if c + 3 <= NB - 1:
        pairs.append(((c, c + 2) + rows, (c + 1, c + 3) + rows))              # west edge
    if c - 3 >= 0:
        pairs.append(((c - 2, c) + rows, (c - 3, c - 1) + rows))              # east edge
    if j + 3 <= NLAT_B - 1:
        pairs.append((cols + (j, j + 2), cols + (j + 1, j + 3)))              # south edge
    if j - 3 >= 0:
        pairs.append((cols + (j - 2, j), cols + (j - 3, j - 1)))              # north edge
    return pairs


def _box_has_nan(decoded, st):
    i0, i1, j0, j1 = (int(st[k]) for k in ("i0", "i1", "j0", "j1"))
    sl = [int(st["slot_m"]), int(st["slot"]), int(st["slot_p"])]
    return any(np.isnan(a[sl if f == 0 else sl[1:2], :, j0:j1 + 1, i0:i1 + 1]).any() for f, a in enumerate(decoded))


@functools.lru_cache(maxsize=None)
def _dataset_b():
    P, fields = _dataset(NB, NLAT_B, NLEV_B, NT_B, np.float64, seed=5)
    return P, [f / u for f, u in zip(fields, UNITS_B)]


@pytest.mark.parametrize("rtype,rule,htype,nfill,order", CASES_B)
def test_decode_rules_and_fills(rtype, rule, htype, nfill, order):
    P, stored = _dataset_b()
    hdt = DT[htype]
    rdt = np.int16 if rtype == "int16" else DT[rtype]
    a, b = FILL_VALUES[rdt]
    fills = [(a, b)[i] for i in NFILLS[nfill]]
    if rdt == np.int16:
        use_scale, use_offset, round32 = rule
        vals, decode = [], []
        for x in stored:
            lo, hi = float(x.min()), float(x.max())
            off = 0.5 * (lo + hi) if use_offset else 0.0
            scale = ((hi - lo) / 65000.0 if use_offset else max(abs(lo), abs(hi)) / 32000.0) if use_scale else 1.0
            q = np.round((x - off) / scale)
            assert np.abs(q).max() <= 32500
            vals.append(q.astype(np.int16))
            decode.append(dict(scale=np.float64(scale) if use_scale else None,
                               offset=np.float64(off) if use_offset else None, fills=fills, float32=round32))
    else:
        vals = [x.astype(rdt) for x in stored]
        decode = [dict(scale=None, offset=None, fills=fills, float32=False)] * 5
    for p, (_, f, k, j, c) in enumerate(FILLS_B):       # the two values alternate; they are fills if `fills` says so
        vals[f][2 * p + 1, k, j, c] = (a, b)[p % 2]
    decoded = [H.decode(v, d, hdt) for v, d in zip(vals, decode)]
    rng = np.random.default_rng(77)
    rec = np.arange(NT_B)
    raws = _records(rng, vals, LON_B, RLON_B, LAT_B, NLAT_B, LEV_B, 6, rec, NT_B, order)

    whole = E.time_stencil(H.tsec_of(P), E.make_steps(NT_B))
    whole["i0"], whole["i1"], whole["j0"], whole["j1"] = 0, NB - 1, 0, NLAT_B - 1
    inner = whole.copy()
    inner["i0"], inner["i1"], inner["j0"], inner["j1"] = 1, NB - 2, 1, NLAT_B - 2
    probes, pairs = [], []           # pairs: (fill index, step of the box on the fill, step of the box next to it)
    for p, (_, f, k, j, c) in enumerate(FILLS_B):
        for incl, excl in _probe_pairs(j, c):
            for box in (incl, excl):
                st = whole[2 * p + 1:2 * p + 2].copy()
                st["i0"], st["i1"], st["j0"], st["j1"] = box
                probes.append(st)
            pairs.append((p, 2 * NT_B + len(probes) - 2, 2 * NT_B + len(probes) - 1))
    steps = np.concatenate([whole, inner] + probes)

    fill_at = [(a, b)[p % 2] in fills for p in range(len(FILLS_B))]
    assert sum(fill_at) == {"none": 0, "one": 6, "equal": 6, "distinct": len(FILLS_B)}[nfill]
    for p, si, se in pairs:          # the design: the first box of a pair holds the fill, the second none
        assert _box_has_nan(decoded, steps[si]) == fill_at[p] and not _box_has_nan(decoded, steps[se])

    with H.make_engine(P, hdt, UNITS_B) as eng:
        got = _host_raw(eng, raws, (LON_B, LAT_B, LEV_B), rec, steps, decode)
        ref = _host(eng, decoded, steps)
    _same(got, ref, "run_host on the decoded arrays")
    terms, levels, flags, pieces = got
    for p, si, se in pairs:
        where = FILLS_B[p][0]
        if fill_at[p]:
            assert flags[si] & E.FLAG_NONFINITE, (where, steps[si])
        assert not flags[se] & E.FLAG_NONFINITE, (where, steps[se])
        assert np.isfinite(terms[se]).all() and np.isfinite(levels[se]).all() and np.isfinite(pieces[se]).all(), where


# ---------------------------------------------------------------------------------------------------------------- #
# D. bench.py's e2e configurations at scale
E2E_CHUNK = 12                            # bench.py's --e2e-chunk default
E2E_SLOTS = E2E_CHUNK + 2
WINDOWS = (E2E_SLOTS, 11, 3)              # one window; bench's automatic budget on an idle B200 (fp64); 3 slots
PACKING_E2E = [dict(offset=True, float32=False, nfill=0)] * 5      # bench.py's: scale_factor + add_offset, to fp64


def _need_host(nbytes):
    with open("/proc/meminfo") as f:
        avail = next(int(line.split()[1]) * 1024 for line in f if line.startswith("MemAvailable:"))
    if avail < nbytes:
        pytest.skip(f"needs {nbytes / GIB:.1f} GiB of available host memory, {avail / GIB:.1f} GiB are available")


def _c4_engine(grid, dtype, window=0):
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    slot = bench.NLEV * len(grid["lat"]) * len(grid["lon"]) * np.dtype(dtype).itemsize
    return E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]),
                       f64(grid["coslats"]), grid["level"], dtype, max_steps=E2E_CHUNK, max_box_rows=bench.BOX_ROWS,
                       host_stage_bytes=2 * 5 * window * slot)


def _host_windows(monkeypatch, grid, dtype, ref, d, run, slot_field_bytes):
    """``run(eng)`` through each window of WINDOWS, on handles forced to the reference's row-kernel instance: the
    reference's bits step by step, and the bytes the maps imply (T of every slot once, the other four fields at the
    12 centre slots; T slots a previous window holds are copied device to device)."""
    with monkeypatch.context() as m:
        for k, v in _solo_env(d).items():
            m.setenv(k, v)
        for w in WINDOWS:
            t0 = time.perf_counter()
            with _c4_engine(grid, dtype, w) as eng:
                got = run(eng)
                got = got + (eng.last_boundary.copy(),)
                dh = eng.last_dispatch()
                h2d = eng.last_transfer()[0]
            print(f"window {w}: {time.perf_counter() - t0:.1f} s")
            assert {k: dh[k] for k in DISPATCH_KEYS} == {k: d[k] for k in DISPATCH_KEYS}, (w, dh, d)
            _same(got, ref, f"{w}-slot windows")
            assert h2d == (E2E_SLOTS + 4 * E2E_CHUNK) * slot_field_bytes, (w, h2d)
            del got


def test_e2e_fp32_host_arrays(monkeypatch):
    """bench.py's ``e2e`` line: 12 C4 steps from 14 pinned fp32 host slots through ``lec_run_host`` (rows of 1440
    columns: plain H2D copies, no ingest), against ``run_torch`` on the same fields resident on the device."""
    nbytes = 5 * E2E_SLOTS * C4_SLOT * 4
    _need(2 * nbytes + 4 * GIB)
    _need_host(nbytes + 4 * GIB)
    grid = S.era5_grid(bench.NLON, bench.NLAT)
    steps = _bench_steps(E2E_SLOTS, BENCH_BOX)
    fields = S.synth_fields(grid, E2E_SLOTS, np.float32, "cuda:0", t0=0)
    with _c4_engine(grid, np.float32) as eng:
        ref = _run(eng, fields, steps)
        d = eng.last_dispatch()
    assert not ref[2].any()
    host = [torch.empty(tuple(f.shape), dtype=torch.float32, pin_memory=True) for f in fields]
    for h, f in zip(host, fields):
        h.copy_(f)
    del fields
    torch.cuda.empty_cache()
    arrs = [h.numpy() for h in host]
    _host_windows(monkeypatch, grid, np.float32, ref, d, lambda eng: eng.run_host(arrs, steps, want_boundary=True),
                  bench.NLEV * bench.NLAT * bench.NLON * 4)
    del arrs, host


def test_e2e_packed_int16_records(monkeypatch):
    """bench.py's ``e2e.packed_int16`` line: the same 14 slots as int16 records (scale + offset from each field's
    extremes over the 14 slots, encoded on the device slot by slot, decoded to fp64) through ``lec_run_host_raw`` with
    identity maps (77 MB raw slot-fields, 307 MB fp64 slots); then the same records as a file in 0..360 longitudes
    with the pole rows cropped, as ``process_data`` / ``slice_domain`` map them (longitude wrapped by 720 columns,
    rows 1..719: the strided 3-D copy of each 721-row record).  Reference: ``run_torch`` on the decoded fields."""
    nlat3 = bench.NLAT - 2
    dec_bytes = 5 * E2E_SLOTS * C4_SLOT * 8
    _need(max(dec_bytes + dec_bytes // 5, 2 * dec_bytes) + 4 * GIB)     # decoded fields + one rolled; one window
    _need_host(5 * E2E_SLOTS * C4_SLOT * 2 + 4 * GIB)
    grid = S.era5_grid(bench.NLON, bench.NLAT)
    one, lo, hi = None, [None] * 5, [None] * 5
    for s in range(E2E_SLOTS):               # pass 1: each field's extremes over the slots
        one = S.synth_fields(grid, 1, np.float32, "cuda:0", t0=s, out=one)
        for f in range(5):
            lo[f] = one[f].min() if lo[f] is None else torch.minimum(lo[f], one[f].min())
            hi[f] = one[f].max() if hi[f] is None else torch.maximum(hi[f], one[f].max())
    bounds = [(float(x), float(y)) for x, y in zip(lo, hi)]
    q = [torch.empty((E2E_SLOTS, bench.NLEV, bench.NLAT, bench.NLON), dtype=torch.int16, pin_memory=True)
         for _ in range(5)]
    for s in range(E2E_SLOTS):               # pass 2: encoded on the device, one slot at a time
        one = S.synth_fields(grid, 1, np.float32, "cuda:0", t0=s, out=one)
        raws, decode = H.encode([x[0] for x in one], PACKING_E2E, bounds=bounds)
        for f in range(5):
            q[f][s].copy_(raws[f])
    del one, raws
    assert all(dc["fills"] == [] and dc["offset"] is not None and not dc["float32"] for dc in decode)

    dec = [torch.empty(tuple(x.shape), dtype=torch.float64, device="cuda:0") for x in q]
    for f in range(5):
        for s in range(E2E_SLOTS):
            dec[f][s].copy_(H.decode(q[f][s].cuda(), decode[f], np.float64))
    steps = _bench_steps(E2E_SLOTS, BENCH_BOX)
    with _c4_engine(grid, np.float64) as eng:
        ref2 = _run(eng, dec, steps)
        d2 = eng.last_dispatch()
    grid3 = dict(grid)
    for k in ("lat", "rlats", "coslats"):
        grid3[k] = grid[k][1:bench.NLAT - 1]
    for f in range(5):                       # engine column i = raw column (i + 720) % 1440, engine row j = raw row j + 1
        dec[f] = torch.roll(dec[f][:, :, 1:bench.NLAT - 1], -bench.NLON // 2, dims=3)
    steps3 = _bench_steps(E2E_SLOTS, (0, bench.NLON - 1, 0, nlat3 - 1))
    with _c4_engine(grid3, np.float64) as eng:
        ref3 = _run(eng, dec, steps3)
        d3 = eng.last_dispatch()
    del dec
    torch.cuda.empty_cache()
    assert not ref2[2].any() and not ref3[2].any()

    qn = [x.numpy() for x in q]
    rec = np.arange(E2E_SLOTS)
    ident = (np.arange(bench.NLON), np.arange(bench.NLAT), np.arange(bench.NLEV))
    _host_windows(monkeypatch, grid, np.float64, ref2, d2,
                  lambda eng: eng.run_host_raw(qn, *ident, rec, steps, decode=decode, want_boundary=True),
                  bench.NLEV * bench.NLAT * bench.NLON * 2)
    wrap = ((np.arange(bench.NLON) + bench.NLON // 2) % bench.NLON, np.arange(1, bench.NLAT - 1), np.arange(bench.NLEV))
    _host_windows(monkeypatch, grid3, np.float64, ref3, d3,
                  lambda eng: eng.run_host_raw(qn, *wrap, rec, steps3, decode=decode, want_boundary=True),
                  bench.NLEV * nlat3 * bench.NLON * 2)
    del qn, q
