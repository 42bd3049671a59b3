"""Batches of unlike boxes: every step against the fp64 oracle and against its own solo run.

The C ABI gives every step of a ``lec_run_*`` call its own box (track files may give each step its own length and
width), but ``run_batch`` (csrc/lec_engine.cu) launches ONE row-kernel instance per kernel batch, chosen from the
batch's extremes: the widest box picks the family and group width, widest and tallest together pick COMP, the tallest
sets the tiles per band.  Every other step then runs inside an instance chosen for another step's box: a one-chunk
row in a tiled launch (one sweep iteration), a 2-row box in a 15-, 11- or 7-row tile, a 2-column box in a 16-lane
group.  Each test below compares every step with the oracle (``helpers.oracle_step``: the moving framework's per-step
``BoxState``) in all three outputs -- 16 terms, 19 per-level families, 18 per-level boundary pieces -- under the
suite's gates (series-scaled over the steps of one box, 1e-9 for fp64 arithmetic, 1e-5 for fp32).

A step's row records depend only on its own box and on the instance it ran under (lane <-> column mapping, summation
order and butterfly are fixed per instance; finalize works one step at a time), so a step run inside any batch must
also have the BITS of the same step run alone on a fresh handle whose dispatcher switches (``LEC_NARROW``,
``LEC_NARROW_G``, ``LEC_COMP``) force the same instance."""
import functools

import numpy as np
import pytest

from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E, synthetic as S
import helpers as H

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOL = {"f32": 1e-5, "m64": 1e-9, "f64": 1e-9}
ARITH = {"f32": (np.float32, E.LEC_MATH_AUTO, 4), "m64": (np.float32, E.LEC_MATH_F64, 4),
         "f64": (np.float64, E.LEC_MATH_AUTO, 2)}
LONW = {"exact": 0, "f32": 1, "irregular": 2}
DISPATCH_KEYS = ("kernel", "vec", "group", "lonw", "comp", "math64", "tile_rows")
T0 = np.datetime64("2020-01-01T00")
NT, NLEV = 3, 4
WIDE = (816, 131)            # fp32: 204 chunks per row, fp64: 408


@pytest.fixture(autouse=True)
def _default_dispatcher(monkeypatch):
    for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
        monkeypatch.delenv(k, raising=False)


@functools.lru_cache(maxsize=None)
def _dataset(coords):
    """float32-valued fields on the WIDE grid (as test_dispatch_matrix_gpu), their fp64 oracle dataset and the global
    dT/dt of the moving framework."""
    nlon, nlat = WIDE
    i = np.arange(nlon, dtype=np.float64)
    lat = -40.0 + 0.5 * np.arange(nlat)
    if coords == "exact":
        lon, cd = -100.0 + 0.5 * i, np.float64
    elif coords == "f32":
        lon, cd = -100.0 + 0.25 * i, np.float32
    else:
        lon, cd = -100.0 + np.cumsum(np.random.default_rng(5).uniform(0.2, 0.3, nlon)), np.float64
    time_ = T0 + np.arange(NT) * np.timedelta64(6, "h")
    level = np.linspace(2e4, 1e5, NLEV)
    fields = H.smooth_fields(NT, NLEV, nlat, nlon, np.float32, seed=nlon + 1, level=level, lat=lat)
    P = H.prepared_from_arrays(fields, lon, lat, level, time_, coord_dtype=cd)
    if coords == "exact":
        P.rlons = (i - 200.0) * 2.0 ** -7
    Q = O.to_mode(P, "fp64")
    dTdt = O.differentiate(Q.fields["Air Temperature"], H.tsec_of(Q), 0)
    return P, fields, Q, dTdt


@functools.lru_cache(maxsize=None)
def _device(coords, dtype):
    return tuple(torch.from_numpy(np.ascontiguousarray(f, dtype=dtype)).cuda() for f in _dataset(coords)[1])


@functools.lru_cache(maxsize=None)
def _oracle(coords, box, it):
    _, _, Q, dTdt = _dataset(coords)
    return H.oracle_step(Q, box, it, dTdt)


def _box(chunks, vecw, i0, j0, j1):
    return (i0, (i0 // vecw + chunks - 1) * vecw + 1, j0, j1)


# pilot -> (chunks, rows j0 ... j1): the box that decides the instance of the batch
PILOTS = {"tiled": (201, (1, 129)), "g16": (150, (3, 62)), "g8": (60, (1, 129))}


def _want(pilot, arith, coords):
    vecw, m64 = ARITH[arith][2], arith != "f32"
    if pilot == "tiled":        # 129 rows: no COMP
        return dict(kernel="tiled", vec=vecw, group=32, lonw=LONW[coords], comp=False, math64=m64,
                    tile_rows={"f32": 15, "m64": 7, "f64": 11}[arith])
    g = 16 if pilot == "g16" else 8
    return dict(kernel="subwarp", vec=vecw, group=g, lonw=0 if coords == "exact" else 2,
                comp=pilot == "g16" and not m64, math64=m64, tile_rows=32 // g)    # 150 chunks x 60 rows: COMP


def _boxes(pilot, arith):
    """The pilot, then small boxes that ride in its instance; the last one holds the grid's last column and row."""
    vecw = ARITH[arith][2]
    nlon, nlat = WIDE
    chunks, (j0, j1) = PILOTS[pilot]
    p = _box(chunks, vecw, vecw + 1, j0, j1)
    R = _want(pilot, arith, "f32")["tile_rows"]
    boxes = [p,
             (2 * vecw, 2 * vecw + 1, 10, 11),                       # 2 x 2 inside one chunk
             (vecw - 1, vecw, 20, 31),                               # 2 columns across a chunk boundary
             (7 * vecw + (vecw > 2), 8 * vecw - 1, 40, 49),          # one chunk (odd first column in fp32)
             (p[0], p[1], 50, 51),                                   # 2 rows at the pilot's width
             (0, 2 * vecw + 1, 0, 5)]                                # column 0, row 0
    boxes += [(3 * vecw + 1, 5 * vecw + 2, 60, 60 + h - 1) for h in sorted({max(2, R - 1), R, R + 1})]
    return boxes + [(nlon - 6, nlon - 1, nlat - 6, nlat - 1)]


def _items(boxes):
    """(box, time index) of every step: each box at every time slot, time-major, so the last step is the last box
    in the last slot."""
    return [(b, it) for it in range(NT) for b in boxes]


def _steps(P, items):
    st = E.time_stencil(H.tsec_of(P), E.make_steps(NT))
    steps = E.make_steps(len(items))
    for n, (b, it) in enumerate(items):
        steps[n] = st[it]                          # slot, slot_m, slot_p, ct_*: time slots shared between steps
        steps["i0"][n], steps["i1"][n], steps["j0"][n], steps["j1"][n] = b
    return steps


def _engine(coords, arith, **kw):
    P = _dataset(coords)[0]
    dtype, math, _ = ARITH[arith]
    return H.make_engine(P, dtype, [1.0] * 5, math=math, **kw)


def _run_torch(eng, coords, arith, steps):
    """(terms, levels, flags, pieces [n][6][3][nlev]) of run_torch on the device-resident fields."""
    dev = _device(coords, ARITH[arith][0])
    t, lv, f, b = H.with_boundary(eng, len(steps), lambda: eng.run_torch(list(dev), steps))
    return t, lv, f, b.reshape(len(steps), 6, 3, eng.nlev)


def _run_host(eng, coords, arith, steps):
    arrs = [np.ascontiguousarray(f, dtype=ARITH[arith][0]) for f in _dataset(coords)[1]]
    t, lv, f = eng.run_host(arrs, steps, want_boundary=True)
    return t, lv, f, eng.last_boundary


def _fp32_out_of_reach(box):
    """A 2-row box wider than 32 chunks: its area eddies [X]_j - [[X]] are tiny against the zonal eddies, so fp32
    arithmetic cannot reach 1e-5 of them (DESIGN.md section 5).  Measured alone on a B200: 2 rows x 801 columns
    1.4e-5 (BKe) with the compensated sums the dispatcher gives it, 2.3e-5 without.  Such steps are held to the bits
    of their solo run under fp32 arithmetic and to the oracle under fp64 arithmetic."""
    return box[3] - box[2] + 1 == 2 and box[1] // 4 - box[0] // 4 + 1 > 32


def _check_oracle(out, items, coords, arith):
    """Every step against the oracle at the gate of ``arith``, each box its own series."""
    tol = TOL[arith]
    for box in dict.fromkeys(b for b, _ in items):
        if arith == "f32" and _fp32_out_of_reach(box):
            continue
        idx = [n for n, (b, _) in enumerate(items) if b == box]
        try:
            H.check_refs(tuple(x[idx] for x in out), [_oracle(coords, *items[n]) for n in idx], tol)
        except AssertionError as e:
            raise AssertionError(f"box {box}: {e}") from None


def _solo_env(d):
    """Dispatcher switches that make a one-step batch take the instance ``d``."""
    env = {"LEC_COMP": "1" if d["comp"] else "0"}
    if d["kernel"] == "tiled":
        env["LEC_NARROW"] = "0"
    else:
        env["LEC_NARROW_G"] = str(d["group"])
    return env


def _check_solo(out, steps, d, coords, arith, monkeypatch):
    """Each step of ``out`` has the bits of the same step run alone, on a fresh handle, under the instance ``d``."""
    with monkeypatch.context() as m:
        for k, v in _solo_env(d).items():
            m.setenv(k, v)
        for n in range(len(steps)):
            with _engine(coords, arith, max_steps=1) as eng:
                solo = _run_torch(eng, coords, arith, steps[n:n + 1])
                ds = eng.last_dispatch()
            assert {k: ds[k] for k in DISPATCH_KEYS} == {k: d[k] for k in DISPATCH_KEYS}, (n, ds, d)
            H.same_bits([x[n:n + 1] for x in out], solo)


# ---------------------------------------------------------------------------------------------------------------- #
@pytest.mark.parametrize("coords", ["exact", "f32", "irregular"])
@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("pilot", ["tiled", "g16", "g8"])
def test_small_boxes_in_the_pilots_instance(pilot, arith, coords, monkeypatch):
    """(a) The pilot box sets the instance; 2 x 2, 2-column, one-chunk, 2-row, tile_rows - 1 / + 0 / + 1 row and
    grid-corner boxes ride in it.  run_host and run_torch give the same bits, every step meets the oracle and has
    the bits of its solo run (the 2-row box at the pilot's width: see _fp32_out_of_reach)."""
    items = _items(_boxes(pilot, arith))
    P = _dataset(coords)[0]
    steps = _steps(P, items)
    with _engine(coords, arith) as eng:
        host = _run_host(eng, coords, arith, steps)
        d = eng.last_dispatch()
    assert {k: d[k] for k in DISPATCH_KEYS} == _want(pilot, arith, coords), d
    with _engine(coords, arith) as eng:
        dev = _run_torch(eng, coords, arith, steps)
        assert eng.last_dispatch() == d
    H.same_bits(host, dev)
    _check_oracle(host, items, coords, arith)
    _check_solo(host, steps, d, coords, arith, monkeypatch)


@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("pilot", ["tiled", "g16", "g8"])
def test_order_and_duplicates(pilot, arith):
    """(b) The steps of (a) reversed, with one step repeated: the same permutation of the results, bit for bit."""
    coords = "irregular"
    items = _items(_boxes(pilot, arith))
    P = _dataset(coords)[0]
    perm = list(range(len(items)))[::-1] + [3, len(items) - 1]
    with _engine(coords, arith) as eng:
        a = _run_torch(eng, coords, arith, _steps(P, items))
        b = _run_torch(eng, coords, arith, _steps(P, [items[n] for n in perm]))
    H.same_bits([x[perm] for x in a], b)


def _split_items(arith):
    """Consecutive kernel batches of 2 steps switch instance: tiled, G = 16, G = 8, tiled, ..."""
    vecw = ARITH[arith][2]
    tiled, g16, g8 = (_box(PILOTS[k][0], vecw, vecw + 1, *PILOTS[k][1]) for k in ("tiled", "g16", "g8"))
    boxes = [tiled, (tiled[0], tiled[1], 50, 51), g16, (7 * vecw + (vecw > 2), 8 * vecw - 1, 40, 49), g8,
             (2 * vecw, 2 * vecw + 1, 10, 11)]
    # time slots 0 and 2 alternate, so that a 2-slot staging window holds one step only
    return [(b, (n + k) % 2 * 2) for k in range(2) for n, b in enumerate(boxes)]


@pytest.mark.parametrize("max_steps", [1, 2, 4])
@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
def test_split_batches_that_switch_instances(arith, max_steps):
    """(c) A call cut into kernel batches of ``max_steps`` steps whose instances differ: run_torch with the pieces
    armed has the bits of the per-slice calls (terms, levels, flags and pieces land at each batch's offsets), and
    run_host through 2-slot staging windows (several staged chunks) meets the oracle."""
    coords = "f32"
    items = _split_items(arith)
    P = _dataset(coords)[0]
    steps = _steps(P, items)
    with _engine(coords, arith, max_steps=max_steps) as eng:
        whole = _run_torch(eng, coords, arith, steps)
        parts, kernels = [], []
        for s0 in range(0, len(steps), max_steps):
            parts.append(_run_torch(eng, coords, arith, steps[s0:s0 + max_steps]))
            d = eng.last_dispatch()
            kernels.append((d["kernel"], d["group"]))
    if max_steps == 2:
        assert kernels == [("tiled", 32), ("subwarp", 16), ("subwarp", 8)] * 2, kernels
    H.same_bits(whole, [np.concatenate(x) for x in zip(*parts)])
    slot_bytes = NLEV * WIDE[1] * WIDE[0] * np.dtype(ARITH[arith][0]).itemsize
    with _engine(coords, arith, max_steps=max_steps, host_stage_bytes=2 * 5 * 2 * slot_bytes) as eng:
        host = _run_host(eng, coords, arith, steps)
    _check_oracle(host, items, coords, arith)


@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
def test_a_reused_handle_reads_no_stale_records(arith):
    """(d) Tall boxes, then short ones on the same handle: the second call has the bits of a fresh handle."""
    coords = "exact"
    vecw = ARITH[arith][2]
    P = _dataset(coords)[0]
    tall = _items([_box(201, vecw, 1, 0, 130), _box(60, vecw, vecw + 1, 1, 129), (0, 2 * vecw + 1, 0, 130)])
    short = _items([(vecw + 1, _box(201, vecw, vecw + 1, 0, 1)[1], 50, 51), (2 * vecw, 2 * vecw + 1, 10, 11),
                    (3 * vecw + 1, 5 * vecw + 2, 60, 62)])
    with _engine(coords, arith) as eng:
        _run_torch(eng, coords, arith, _steps(P, tall))
        again = _run_torch(eng, coords, arith, _steps(P, short))
    with _engine(coords, arith) as eng:
        fresh = _run_torch(eng, coords, arith, _steps(P, short))
    H.same_bits(again, fresh)
    _check_oracle(fresh, short, coords, arith)


# ---------------------------------------------------------------------------------------------------------------- #
@functools.lru_cache(maxsize=None)
def _packed(coords, arith):
    """int16 encodings of the dataset (ERA5 style: scale and offset, one fill value), the device tensors, the decode
    dicts and the numpy-decoded fields on the device."""
    raws, dec = H.encode(_dataset(coords)[1], [dict(offset=True, float32=False, nfill=1)] * 5)
    pitch = (WIDE[0] + 7) // 8 * 8
    decoded = [torch.from_numpy(np.ascontiguousarray(H.decode(r, d, ARITH[arith][0]))).cuda() for r, d in zip(raws, dec)]
    return [H.padded(r, pitch) for r in raws], dec, decoded


def _packed_pair(coords, arith, items):
    P = _dataset(coords)[0]
    steps = _steps(P, items)
    pk, dec, decoded = _packed(coords, arith)
    with _engine(coords, arith) as eng:
        a = H.with_boundary(eng, len(steps), lambda: eng.run_torch_packed(pk, dec, steps))
        da = eng.last_dispatch()
        b = H.with_boundary(eng, len(steps), lambda: eng.run_torch(decoded, steps))
        db = eng.last_dispatch()
    assert da["packed"] and not db["packed"]
    for k in ("kernel", "vec", "group", "lonw", "comp", "math64"):
        assert da[k] == db[k], (k, da, db)
    assert not a[2].any() and np.isfinite(a[0]).all() and np.isfinite(a[3]).all()
    H.same_bits(a, b)
    return da


@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("pilot", ["tiled", "g16", "g8"])
def test_packed_batches_have_the_bits_of_the_decoded_fields(pilot, arith):
    """(e) The batches of (a) through run_torch_packed: the bits of run_torch on the numpy-decoded fields."""
    da = _packed_pair("f32", arith, _items(_boxes(pilot, arith)))
    assert da["kernel"] == _want(pilot, arith, "f32")["kernel"]


@pytest.mark.parametrize("arith", ["f32", "f64"])
def test_packed_small_boxes_at_every_int16_shift_in_a_tiled_launch(arith):
    """(e) Boxes of one chunk whose first column is 0 ... 7 modulo 8 (the in-box shift of the 8-column-aligned int16
    TMA boxes and the first column within the chunk), inside a tiled launch.  Where the first column is the last of
    its chunk, the box is that column and the next."""
    vecw = ARITH[arith][2]
    boxes = [_box(201, vecw, vecw + 1, 1, 40)]
    for s in range(8):
        i0 = 64 + 8 * s + s
        i1 = i0 // vecw * vecw + vecw - 1
        boxes.append((i0, i1 if i1 > i0 else i0 + 1, 2 + 5 * s, 4 + 6 * s))
    da = _packed_pair("f32", arith, _items(boxes))
    assert da["kernel"] == "tiled"


# ---------------------------------------------------------------------------------------------------------------- #
C4_BAND = (0, 1439, 400, 423)          # 24 rows of the full-width C4 grid: 360 chunks, the shape COMP exists for
C4_NARROW = (700, 707, 300, 499)       # 8 columns x 200 rows: makes the batch's tallest box 200 rows


def _c4_mixed():
    """The C4 grid, 3 fp32 slots on the device, the engine coordinates, the steps and the oracle of each step."""
    grid = S.era5_grid()
    dev = S.synth_fields(grid, 3, np.float32, "cuda:0")
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    coords = [f64(grid[k]) for k in ("lon", "lat", "rlons", "rlats", "coslats")]
    items = [(C4_BAND, 0), (C4_NARROW, 1), (C4_BAND, 1)]
    ref = {}
    for box in (C4_BAND, C4_NARROW):      # the oracle on the box's crop (the box is the whole crop)
        i0, i1, j0, j1 = box
        host = [d[:, :, j0:j1 + 1, i0:i1 + 1].cpu().numpy() for d in dev]
        P = H.prepared_from_arrays(host, grid["lon"][i0:i1 + 1], grid["lat"][j0:j1 + 1], grid["level"],
                                   T0 + np.arange(3) * np.timedelta64(1, "h"))
        Q = O.to_mode(P, "fp64")
        dTdt = O.differentiate(Q.fields["Air Temperature"], H.tsec_of(Q), 0)
        for b, it in items:
            if b == box:
                ref[(b, it)] = H.oracle_step(Q, (0, i1 - i0, 0, j1 - j0), it, dTdt)
    return grid, dev, coords, items, ref


@pytest.fixture(scope="module")
def c4_mixed():
    data = _c4_mixed()
    yield data
    del data
    torch.cuda.empty_cache()


def test_a_band_batched_with_a_tall_box_meets_the_gate_without_compensated_sums(c4_mixed):
    """(f) A 24-row full-width band next to an 8 x 200 box in one batch.  COMP is decided from the batch's widest and
    tallest boxes, so the band runs with plain fp32 linear sums here (alone it would get COMP); both band steps
    still meet the 1e-5 gate in every term, per-level family and boundary piece.  Measured on a B200: 8.2e-6 (the
    N-S piece of BAe) in this batch, 8.4e-6 alone with COMP."""
    grid, dev, coords, items, ref = c4_mixed
    stencil = E.time_stencil(3600.0 * np.arange(3), E.make_steps(3))
    steps = E.make_steps(len(items))
    for n, (b, it) in enumerate(items):
        steps[n] = stencil[it]
        steps["i0"][n], steps["i1"][n], steps["j0"][n], steps["j1"][n] = b
    with E.LecEngine(*coords, grid["level"], np.float32, max_steps=3, max_box_rows=200) as eng:
        t, lv, f, b = H.with_boundary(eng, 3, lambda: eng.run_torch(dev, steps))
        d = eng.last_dispatch()
    assert d["kernel"] == "tiled" and not d["comp"] and d["tile_rows"] == 15, d
    out = (t, lv, f, b.reshape(3, 6, 3, -1))
    worst = {}
    for box in (C4_BAND, C4_NARROW):
        idx = [n for n, (bx, _) in enumerate(items) if bx == box]
        sub = tuple(x[idx] for x in out)
        refs = [ref[items[n]] for n in idx]
        worst[box] = H.check_refs(sub, refs, 1e-5)
    print(f"C4 band in a mixed batch: worst error {worst[C4_BAND]:.2e} (COMP {d['comp']}); "
          f"8 x 200 box {worst[C4_NARROW]:.2e}")

