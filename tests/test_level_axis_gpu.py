"""The engine along the level axis, against the fp64 oracle: level counts from 2 to 137, missing values and the way
they spread, and the 0.03 floor of the static stability.

A. Level counts.  ``lec_fin_integrate_kernel`` runs 64 threads, each handling levels k, k + 64, ...; the other
   suites run at most 55 levels.  L = 2, 3, 37 (ERA5's 1 ... 1000 hPa set), 64, 65, 137, each on an exactly uniform
   and an irregular level axis, through every row-kernel family (tiled, sub-warp G = 4 / 8 / 16, vector direct,
   scalar direct) in fp64 arithmetic, and in fp32 and LEC_MATH_F64 arithmetic at 65 and 137 levels.  All 16 terms,
   19 per-level families and 18 per-level boundary pieces against ``helpers.oracle_step`` (1e-9 / 1e-5).

B. Propagation.  The host's NaN path (``analysis/_base.py``) works on the per-level families and boundary pieces
   the engine returns, so WHICH (step, family, level) entries come out NaN is part of the interface.  One missing
   value per case (field, level, column or row of the box, time slot, uniform or irregular levels); every step
   must give the NaN masks of the oracle's families taken before ``_handle_nans`` (``raw``) and of its pieces, the
   finite entries within the gate, the NaN mask of the 16 terms as the trapezoids of those families give it, and
   the flags exactly: NONFINITE iff a family or piece is non-finite, SIGMA_FLOOR iff some stability before the floor
   is <= 0.03 or NaN.

C. The sigma floor at the top, the bottom (one-sided d[T]/dp) and an interior level.

D. The product path (``lec_fixed`` / ``lec_moving`` with the host NaN path) against ``O.lec_fixed`` /
   ``O.lec_moving``, including a step with every level missing."""
import functools

import numpy as np
import pandas as pd
import pytest

from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E, synthetic as S
import helpers as H

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TOL = {"f32": 1e-5, "m64": 1e-9, "f64": 1e-9}
ARITH = {"f32": (np.float32, E.LEC_MATH_AUTO, 4), "m64": (np.float32, E.LEC_MATH_F64, 4),
         "f64": (np.float64, E.LEC_MATH_AUTO, 2)}
T0 = np.datetime64("2020-01-01T00")
NT = 3
RECORDS = []                       # (family, L, arith, dispatch record) of every level-count case


@pytest.fixture(autouse=True)
def _default_dispatcher(monkeypatch):
    for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
        monkeypatch.delenv(k, raising=False)


def _levels(L, kind):
    """Pa, ascending.  ``uniform``: integer steps, so every difference is exactly equal in float64 (np.gradient's
    uniform branch); ``irregular``: ERA5's 37 levels, or a geometric sequence."""
    if kind == "uniform":
        return 1000.0 + (99000 // (L - 1)) * np.arange(L, dtype=np.float64)
    if L == 37:
        return np.sort(np.asarray(S.ERA5_LEVELS_HPA, dtype=np.float64)) * 100.0
    return np.geomspace(5000.0, 100000.0, L)


def _prepared(L, kind, nlon, nlat, seed):
    """float32-valued fields (the fp64 cells run them upcast, so one oracle result serves every arithmetic)."""
    level = _levels(L, kind)
    assert (np.all(np.diff(level) == np.diff(level)[0])) == (kind == "uniform" or L == 2)
    lon = -100.0 + 0.25 * np.arange(nlon)
    lat = -40.0 + 0.5 * np.arange(nlat)
    time_ = T0 + np.arange(NT) * np.timedelta64(6, "h")
    fields = H.smooth_fields(NT, L, nlat, nlon, np.float32, seed=seed, level=level, lat=lat)
    return H.prepared_from_arrays(fields, lon, lat, level, time_), fields


def _oracle_of(P):
    Q = O.to_mode(P, "fp64")
    return Q, O.differentiate(Q.fields["Air Temperature"], H.tsec_of(Q), 0)


def _steps(P, boxes):
    steps = E.time_stencil(H.tsec_of(P), E.make_steps(NT))
    for it, b in enumerate(boxes):
        steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = b
    return steps


def _run(P, fields, boxes, arith, route):
    """(terms, levels, flags, pieces [n][6][3][L]) and the dispatch record of one run."""
    dtype, math, _ = ARITH[arith]
    arrs = [np.ascontiguousarray(f, dtype=dtype) for f in fields]
    steps = _steps(P, boxes)
    with H.make_engine(P, dtype, [1.0] * 5, math=math) as eng:
        if route == "host":
            t, lv, f = eng.run_host(arrs, steps, want_boundary=True)
            out = (t, lv, f, eng.last_boundary)
        else:
            dev = [torch.from_numpy(a).cuda() for a in arrs]
            t, lv, f, b = H.with_boundary(eng, len(steps), lambda: eng.run_torch(dev, steps))
            out = (t, lv, f, b.reshape(len(steps), 6, 3, eng.nlev))
        return out, eng.last_dispatch()


# ---------------------------------------------------------------------------------------------------------------- #
# A. level counts
LEVEL_COUNTS = [2, 3, 37, 64, 65, 137]
GRID_A = (803, 10)                 # nlon % 4 = 3: caller-owned device rows are not 16-byte aligned (scalar kernel)
ROWS_A = (1, 8)
# family -> (route, LEC_ROW_KERNEL, columns i0, i1 per arithmetic): chunks of 128 bits per row decide the family
FAMILIES = {
    "g4": ("host", None, {"f32": (3, 8), "f64": (3, 8)}),              # 3 / 4 chunks
    "g8": ("host", None, {"f32": (1, 200), "f64": (1, 200)}),          # 51 / 101
    "g16": ("host", None, {"f32": (1, 600), "f64": (1, 300)}),         # 151 / 151
    "tiled": ("host", None, {"f32": (1, 801), "f64": (1, 801)}),       # 201 / 401
    "direct": ("host", "direct", {"f32": (1, 801), "f64": (1, 801)}),
    "scalar": ("torch", None, {"f32": (1, 200), "f64": (1, 200)}),
}


def _want(family, arith):
    vecw = ARITH[arith][2]
    if family.startswith("g"):
        return dict(kernel="subwarp", vec=vecw, group=int(family[1:]))
    if family == "tiled":
        return dict(kernel="tiled", vec=vecw, group=32)
    return dict(kernel="direct", vec=1 if family == "scalar" else vecw, group=32)


@functools.lru_cache(maxsize=2)
def _dataset_a(L, kind):
    P, fields = _prepared(L, kind, *GRID_A, seed=L)
    return (P, fields) + _oracle_of(P)


@functools.lru_cache(maxsize=None)
def _oracle_a(L, kind, box):
    _, _, Q, dTdt = _dataset_a(L, kind)
    return [H.oracle_step(Q, box, it, dTdt) for it in range(NT)]


A_CASES = ([(L, kind, "f64", fam) for L in LEVEL_COUNTS for kind in ("uniform", "irregular") for fam in FAMILIES]
           + [(L, kind, arith, fam) for L in (65, 137) for kind in ("uniform", "irregular") for arith in ("f32", "m64")
              for fam in FAMILIES])


@pytest.mark.parametrize("L,kind,arith,family", A_CASES)
def test_level_count(L, kind, arith, family, monkeypatch):
    route, env, cols = FAMILIES[family]
    if env:
        monkeypatch.setenv("LEC_ROW_KERNEL", env)
    P, fields = _dataset_a(L, kind)[:2]
    box = cols["f64" if arith == "f64" else "f32"] + ROWS_A
    out, d = _run(P, fields, [box] * NT, arith, route)
    RECORDS.append(dict(d, family=family, L=L, arith=arith))
    want = _want(family, arith)
    assert {k: d[k] for k in want} == want, d
    assert out[1].shape == (NT, 19, L) and out[3].shape == (NT, 6, 3, L)
    H.check_refs(out, _oracle_a(L, kind, box), TOL[arith])


def test_every_level_count_cell_was_reached(request):
    """Every family ran above 64 levels (one integrate thread per two levels) in every arithmetic."""
    mine = [it for it in request.session.items if it.module is request.module and it.name.startswith("test_level_count")]
    if len(mine) < len(A_CASES):
        pytest.skip("needs the whole module: the dispatch records of every level-count case")
    missing = [(fam, L, arith) for fam in FAMILIES for L in (65, 137) for arith in ARITH
               if not any(r["family"] == fam and r["L"] == L and r["arith"] == arith
                          and all(r[k] == v for k, v in _want(fam, arith).items()) for r in RECORDS)]
    assert not missing, missing


# ---------------------------------------------------------------------------------------------------------------- #
# B. propagation of a missing value; C. the sigma floor
def _raw_terms(raw, pieces, p, c1, c2):
    """The 16 terms as the device integrates them: trapezoids over every level of the families before
    ``_handle_nans`` (a missing level leaves the term NaN), boundary terms from the pieces."""
    vint = lambda f: O.trapz(f, p, -1)
    out = {"Az": vint(raw["Az"]), "Ae": vint(raw["Ae"]), "Kz": vint(raw["Kz"]) / (2 * O.g),
           "Ke": vint(raw["Ke"]) / (2 * O.g), "Cz": vint(raw["Cz"]), "Ca": vint(raw["Ca"]),
           "Ck": vint(raw["Ck"]) / O.g, "Ce": vint(raw["Ce"]), "Gz": vint(raw["Gz"]), "Ge": vint(raw["Ge"])}
    for n, name in enumerate(H.BOUNDARY_TERMS):
        ew, ns, vert = pieces[n]
        out[name] = c1 * vint(ew) + c2 * vint(ns) - (vert[-1] - vert[0])
    return np.array([out[name] for name in E.TERM_NAMES])


def _box_consts(Q, box):
    i0, i1, j0, j1 = box
    xl = Q.rlons[i1] - Q.rlons[i0]
    yl = np.sin(Q.rlats[j1]) - np.sin(Q.rlats[j0])
    return -1 / (O.Re * xl * yl), -1 / (O.Re * yl)


def _masked_err(a, b):
    """Series-scaled error over the entries where both are finite (the masks are compared separately)."""
    m = np.isfinite(b)
    if not m.any():
        return 0.0
    den = np.max(np.abs(b[m]))
    d = np.max(np.abs(a[m] - b[m]))
    return float(d / den) if den > 0 else float(d)


def check_propagation(out, refs, Q, boxes, tol, floored_values=True):
    """Every step against the oracle's families before ``_handle_nans``: identical NaN masks of the 19 x L families,
    the 18 x L pieces and the 16 terms, finite entries within ``tol`` (series-scaled over the steps), exact flags.
    ``floored_values=False`` leaves the values of the levels whose sigma was floored out of the per-level
    comparison (their masks stay in): dividing by 0.03 instead of ~2.4 makes such a level the largest entry of its
    family, so the series' error becomes that level's own relative error, which fp32 arithmetic does not hold to
    1e-5 where the level's area eddies are small (measured on a B200: 1.1e-4 in a vertical-flux piece)."""
    terms, levels, flags, bnd = out
    n, L = levels.shape[0], levels.shape[2]
    fam = np.stack([np.stack([np.broadcast_to(r[3][name], (L,)) for name in E.LEVEL_TERM_NAMES]) for r in refs])
    pcs = np.stack([r[2] for r in refs]).reshape(n, 18, L)
    bnd = bnd.reshape(n, 18, L)
    rterms = np.stack([_raw_terms(r[3], r[2], Q.level, *_box_consts(Q, b)) for r, b in zip(refs, boxes)])
    floored = np.stack([~(r[3]["sigma"] > 0.03) for r in refs])[:, None, :]        # [step][1][level]
    bad = []
    for what, a, b in (("families", levels, fam), ("pieces", bnd, pcs), ("terms", terms, rterms)):
        if not np.array_equal(np.isfinite(a), np.isfinite(b)):
            diff = np.argwhere(np.isfinite(a) != np.isfinite(b))
            bad.append(f"{what} NaN mask differs at (step, entry, level) {diff[:6].tolist()}")
        if not floored_values and what != "terms":
            b = np.where(floored, np.nan, b)
        for e in range(a.shape[1]):
            err = _masked_err(a[:, e], b[:, e])
            if not err <= tol:
                bad.append(f"{what}[{e}] {err:.3g}")
    want = np.zeros(n, dtype=np.int32)
    for s, r in enumerate(refs):
        if not (np.isfinite(fam[s]).all() and np.isfinite(pcs[s]).all()):
            want[s] |= E.FLAG_NONFINITE
        if not (r[3]["sigma"] > 0.03).all():
            want[s] |= E.FLAG_SIGMA_FLOOR
    if not np.array_equal(flags, want):
        bad.append(f"flags {flags.tolist()} != {want.tolist()}")
    assert not bad, bad
    return want


GRID_B = (16, 10)
LB = 7
BOX_B = (2, 12, 2, 7)
FIELDS = {"T": 0, "u": 1, "v": 2, "w": 3, "Phi": 4}
LEVEL_AT = {"k0": 0, "k1": 1, "mid": 3, "kL-2": LB - 2, "kL-1": LB - 1}
POS_AT = {"interior": (5, 7), "west": (5, BOX_B[0]), "east": (4, BOX_B[1]), "south": (BOX_B[2], 6),
          "north": (BOX_B[3], 8)}                                   # (row, column)


@functools.lru_cache(maxsize=None)
def _base_b(kind, nlon=GRID_B[0]):
    return _prepared(LB, kind, nlon, GRID_B[1], seed=11)


def _planted(kind, plants, nlon=GRID_B[0]):
    """Copies of the fields with NaN at every (field, slot, level, row, column) of ``plants``; the prepared dataset
    over them, its fp64 oracle dataset and dT/dt."""
    P0, fields = _base_b(kind, nlon)
    fields = [f.copy() for f in fields]
    for f, t, k, j, i in plants:
        fields[f][t, k, j, i] = np.nan
    P = H.prepared_from_arrays(fields, P0.lon, P0.lat, P0.level, P0.time)
    return (P, fields) + _oracle_of(P)


_REF_B = {}


def _case(kind, plants, boxes, arith, route="host", nlon=GRID_B[0]):
    """Run one planted dataset through the engine and check it against the oracle (cached per dataset and boxes:
    the fp32 and fp64 cells share it).  Returns the expected flags."""
    key = (kind, tuple(plants), tuple(boxes), nlon)
    if key not in _REF_B:
        P, fields, Q, dTdt = _planted(kind, plants, nlon)
        _REF_B[key] = (P, fields, Q, [H.oracle_step(Q, b, it, dTdt) for it, b in enumerate(boxes)])
    P, fields, Q, refs = _REF_B[key]
    out, d = _run(P, fields, boxes, arith, route)
    try:
        return check_propagation(out, refs, Q, boxes, TOL[arith], floored_values=arith != "f32"), d
    except AssertionError as e:
        raise AssertionError(f"{kind} levels, NaN at (field, slot, level, row, column) {plants}, {arith}: {e}") \
            from None


@pytest.mark.parametrize("arith", ["f64", "f32"])
@pytest.mark.parametrize("kind", ["uniform", "irregular"])
@pytest.mark.parametrize("field", list(FIELDS))
def test_missing_value_propagation(field, kind, arith):
    """Field x level {0, 1, interior, L-2, L-1} x box position {interior, west / east column, south / north row} x
    slot {first, interior, last}, in the default (sub-warp) kernel."""
    seen = 0
    for k in LEVEL_AT.values():
        for j, i in POS_AT.values():
            for t in range(NT):
                want, d = _case(kind, [(FIELDS[field], t, k, j, i)], [BOX_B] * NT, arith)
                assert d["kernel"] == "subwarp", d
                seen |= int(np.bitwise_or.reduce(want))
    # a missing T reaches sigma (floor) and a family; a missing Phi reaches only the boundary pieces
    assert seen & E.FLAG_NONFINITE
    assert bool(seen & E.FLAG_SIGMA_FLOOR) == (field == "T"), seen


GRID_WIDE_B = 405                  # odd: fp64 device rows are not 16-byte aligned (scalar kernel through run_torch)
BOX_WIDE_B = (1, 401, 2, 7)        # 201 chunks of fp64: the tiled kernel


@pytest.mark.parametrize("family", ["tiled", "direct", "scalar"])
@pytest.mark.parametrize("kind", ["uniform", "irregular"])
def test_missing_value_propagation_wide_kernels(family, kind, monkeypatch):
    """Field x edge level x edge column through the tiled, vector direct and scalar direct kernels (fp64)."""
    route = "torch" if family == "scalar" else "host"
    if family == "direct":
        monkeypatch.setenv("LEC_ROW_KERNEL", "direct")
    want_d = dict(kernel="tiled" if family == "tiled" else "direct", vec=1 if family == "scalar" else 2)
    for f in FIELDS.values():
        for k in (0, LB - 1):
            for i in (BOX_WIDE_B[0], BOX_WIDE_B[1]):
                _, d = _case(kind, [(f, 1, k, 4, i)], [BOX_WIDE_B] * NT, "f64", route, nlon=GRID_WIDE_B)
                assert {x: d[x] for x in want_d} == want_d, d


MOVING_B = [(2, 12, 2, 7), (4, 14, 3, 8), (2, 12, 2, 7)]


@pytest.mark.parametrize("arith", ["f64", "f32"])
@pytest.mark.parametrize("kind", ["uniform", "irregular"])
def test_missing_value_in_one_moving_box(kind, arith):
    """A moving box: the value missing in slot 1 lies inside step 1's box and outside the boxes of steps 0 and 2,
    which read slot 1 through dT/dt; only step 1 may see it."""
    for f in FIELDS.values():
        for k in (0, 3, LB - 1):
            for j, i in ((5, 14), (8, 6), (8, 13)):
                want, _ = _case(kind, [(f, 1, k, j, i)], MOVING_B, arith)
                assert want[0] == 0 and want[2] == 0 and want[1] & E.FLAG_NONFINITE, want


@pytest.mark.parametrize("kind", ["uniform", "irregular"])
def test_two_missing_levels_and_slots(kind):
    """Missing values at two adjacent interior levels of one slot, and at the first and last slot."""
    for plants in ([(1, 1, 2, 4, 6), (1, 1, 3, 5, 8)], [(0, 0, 3, 4, 6), (0, NT - 1, 3, 4, 6)],
                   [(2, 0, 0, 3, 3), (3, NT - 1, LB - 1, 6, 11)]):
        for arith in ("f64", "f32"):
            _case(kind, plants, [BOX_B] * NT, arith)


def test_ck5_on_a_uniform_level_axis():
    """u missing at an interior level: on an exactly uniform level axis np.gradient's centred difference does not
    read [u] of that level, so the reference's Ck_5 (co-factor [w'v']) stays finite there; on an irregular axis it is
    NaN.  The engine must give both."""
    k = LEVEL_AT["mid"]
    for kind, finite in (("uniform", True), ("irregular", False)):
        for arith in ("f64", "f32"):
            _case(kind, [(FIELDS["u"], 1, k, 4, 7)], [BOX_B] * NT, arith)
        refs = _REF_B[(kind, ((1, 1, k, 4, 7),), (BOX_B,) * NT, GRID_B[0])][3]
        assert np.isfinite(refs[1][3]["Ck_5"][k]) == finite
        assert not np.isfinite(refs[1][3]["Ck_4"][k])


def _neutral(kind, k, target):
    """Fields whose layer at level ``k`` is scaled, per slot, so that the box's static stability before the floor
    is ``target`` there (it is linear in that layer's T)."""
    P0, fields = _base_b(kind)
    i0, i1, j0, j1 = BOX_B
    T = fields[0].astype(np.float64)
    Q = O.to_mode(P0, "fp64")
    b = O.BoxState(Q, Q.lon[i0], Q.lon[i1], Q.lat[j0], Q.lat[j1], fixed=True)
    s1 = b.sigma_prefloor[:, k]

    def sigma_at(scale):
        Tt = T[..., j0:j1 + 1, i0:i1 + 1].copy()
        Tt[:, k] *= scale
        return O.static_stability_prefloor(Tt, Q.level, b.rlats, b.coslats, b.rlons, b.xlength, b.ylength)[:, k]

    s0 = sigma_at(0.5)
    f = 0.5 + 0.5 * (target - s0) / (s1 - s0)
    out = [x.copy() for x in fields]
    out[0][:, k] = (T[:, k] * f[:, None, None]).astype(np.float32)
    return out


@pytest.mark.parametrize("arith", ["f64", "f32"])
@pytest.mark.parametrize("kind", ["uniform", "irregular"])
@pytest.mark.parametrize("where", ["top", "bottom", "interior"])
@pytest.mark.parametrize("target", [-0.5, 0.01])
def test_sigma_floor_at_the_edges(where, kind, arith, target):
    """An unstable (or nearly neutral) layer at the top or the bottom level, where d[T]/dp is one-sided, or at an
    interior level: sigma floors to 0.03 there (and wherever the changed layer takes a neighbour's d[T]/dp below
    the floor too), the flags are exactly SIGMA_FLOOR, and every output matches the oracle."""
    k = {"top": 0, "bottom": LB - 1, "interior": 3}[where]
    fields = _neutral(kind, k, target)
    P0 = _base_b(kind)[0]
    P = H.prepared_from_arrays(fields, P0.lon, P0.lat, P0.level, P0.time)
    Q, dTdt = _oracle_of(P)
    refs = [H.oracle_step(Q, BOX_B, it, dTdt) for it in range(NT)]
    for r in refs:
        assert not r[3]["sigma"][k] > 0.03, r[3]["sigma"]
    out, _ = _run(P, fields, [BOX_B] * NT, arith, "host")
    want = check_propagation(out, refs, Q, [BOX_B] * NT, TOL[arith])
    assert (want == E.FLAG_SIGMA_FLOOR).all()


# ---------------------------------------------------------------------------------------------------------------- #
# D. the product path: lec_fixed / lec_moving on an in-memory LecDataset (as bench.py's plugin line builds it)
NT_D, GRID_D = 4, (16, 12)
LEVELS_D = {"uniform": np.arange(25000.0, 100001.0, 15000.0),                 # 850 hPa: the moving framework's plane
            "irregular": np.array([20000.0, 30000.0, 50000.0, 70000.0, 85000.0, 92500.0, 100000.0])}
BOX_D = (2, 13, 2, 9)
NAMES_D = ["t", "u", "v", "w", "z"]


def _nl():
    return pd.DataFrame({"Variable": NAMES_D + ["longitude", "latitude", "time", "level"],
                         "Units": ["K", "m/s", "m/s", "Pa/s", "m**2/s**2", "", "", "", "Pa"]},
                        index=H.NAMES + ["Longitude", "Latitude", "Time", "Vertical Level"])


def _fields_d(kind, plants):
    level = LEVELS_D[kind]
    nlon, nlat = GRID_D
    lon, lat = -60.0 + 0.5 * np.arange(nlon), -35.0 + 0.5 * np.arange(nlat)
    fields = H.smooth_fields(NT_D, len(level), nlat, nlon, np.float32, seed=21, level=level, lat=lat)
    for f, t, k, j, i in plants:
        fields[f][t, k, j, i] = np.nan
    time_ = np.datetime64("2020-01-01T00", "ns") + np.arange(NT_D) * np.timedelta64(1, "h")
    return H.prepared_from_arrays(fields, lon, lat, level, time_)


def _read_levels(path):
    """Rows of a per-level CSV after its header, as (index, values): rows may differ in length (levels dropped)."""
    rows = []
    for line in open(path, encoding="utf-8").read().splitlines()[1:]:
        cells = line.split(",")
        rows.append((cells[0], np.array([float(x) if x else np.nan for x in cells[1:]])))
    return rows


def _product(kind, plants, tmp_path, moving, oracle=True):
    """The product's frame and per-level files, and the oracle's frame and families, for one planted dataset."""
    from lorenzcycletoolkit_b200.frameworks import lec_fixed, lec_moving
    from lorenzcycletoolkit_b200.utils.preprocessing import LecDataset
    import argparse
    import logging
    P = _fields_d(kind, plants)
    data = LecDataset(variables=dict(zip(NAMES_D, (P.fields[n] for n in H.NAMES))), time=P.time, level=P.level,
                      lat=P.lat, lon=P.lon, rlats=P.rlats, coslats=P.coslats, rlons=P.rlons,
                      names={"Time": "time", "Vertical Level": "level", "Latitude": "latitude", "Longitude": "longitude"})
    lon, lat = np.asarray(P.lon, np.float64), np.asarray(P.lat, np.float64)
    i0, i1, j0, j1 = BOX_D
    out = tmp_path / f"{kind}_{'m' if moving else 'f'}_{abs(hash(tuple(plants)))}"
    lv_dir = out / "lv"
    lv_dir.mkdir(parents=True)
    log = logging.getLogger("lec_level_axis")
    if not moving:
        (out / "box").write_text(f"min_lon;{lon[i0]}\nmax_lon;{lon[i1]}\nmin_lat;{lat[j0]}\nmax_lat;{lat[j1]}\n")
        args = argparse.Namespace(infile="synthetic.nc", fixed=True, track=False, choose=False, residuals=True,
                                  box_limits=str(out / "box"), outname=None, plots=False, cdsapi=False, mpas=False)
        df = lec_fixed(data, _nl(), str(out), str(lv_dir), log, args)
        odf, olv, _ = O.lec_fixed(P, lon[i0], lon[i1], lat[j0], lat[j1], mode="fp64") if oracle else (None, None, None)
    else:
        # the box moves one column east per step, its limits on grid points
        track = pd.DataFrame({"Lat": [(lat[j0] + lat[j1]) / 2] * NT_D,
                              "Lon": [(lon[i0 + s - 1] + lon[i1 + s - 1]) / 2 for s in range(NT_D)],
                              "length": [lat[j1] - lat[j0]] * NT_D, "width": [lon[i1] - lon[i0]] * NT_D},
                             index=pd.to_datetime(P.time))
        trk = out / "track"
        track.to_csv(trk, sep=";", index_label="time", date_format="%Y-%m-%d-%H%M")
        args = argparse.Namespace(infile="synthetic.nc", fixed=False, track=True, choose=False, residuals=True,
                                  trackfile=str(trk), cdsapi=False, mpas=False, zeta=False, plots=False)
        df = lec_moving(data, _nl(), None, str(out), str(out), str(lv_dir), log, args)
        odf, olv, _ = O.lec_moving(P, O.read_track(str(trk)), mode="fp64") if oracle else (None, None, None)
    return df, lv_dir, odf, olv


def _check_product(df, lv_dir, odf, olv, moving):
    """Frame and every per-level CSV against the oracle: NaN masks equal, finite values within 1e-5."""
    assert list(df.columns) == list(odf.columns)
    for c in odf.columns:
        a, b = df[c].values, odf[c].values
        assert np.array_equal(np.isnan(a), np.isnan(b)), (c, a, b)
        ok = ~np.isnan(b)
        if ok.any():
            assert H.series_err(a[ok], b[ok]) <= 1e-5, (c, H.series_err(a[ok], b[ok]))
    for name in O.LEVEL_TERMS:
        rows = _read_levels(lv_dir / f"{name}_level.csv")
        want = olv[name]
        if name in ("Cz_1", "Ce_1") and not moving:
            rows = rows[1:]                                   # a row of levels, then the values
            want = [want]
        got = [r[1] for r in rows]
        want = [np.asarray(w, dtype=np.float64) for w in want]
        assert [g.shape for g in got] == [w.shape for w in want], (name, [g.shape for g in got])
        for g, w in zip(got, want):
            assert np.array_equal(np.isnan(g), np.isnan(w)), (name, g, w)
        g, w = np.concatenate(got), np.concatenate(want)
        ok = ~np.isnan(w)
        if ok.any():
            assert H.series_err(g[ok], w[ok]) <= 1e-5, (name, H.series_err(g[ok], w[ok]))


PRODUCT_CASES = {
    # name -> (level axis, [(field, slot, level, row, column)]; None = the whole plane)
    "phi_only": ("irregular", [(4, 1, 3, 5, 6)]),
    "top_level_one_time": ("irregular", [(3, 1, 0, None, None)]),
    "two_adjacent_levels": ("uniform", [(1, 2, 2, None, None), (1, 2, 3, None, None)]),
    "first_and_last_slot": ("irregular", [(0, 0, 3, 5, 6), (0, NT_D - 1, 2, 4, 9)]),
    "u_on_uniform_levels": ("uniform", [(1, 1, 2, 5, 7)]),
}


def _plants(spec):
    nlon, nlat = GRID_D
    out = []
    for f, t, k, j, i in spec:
        out += [(f, t, k, jj, ii) for jj in range(nlat) for ii in range(nlon)] if j is None else [(f, t, k, j, i)]
    return out


@pytest.mark.parametrize("moving", [False, True], ids=["fixed", "moving"])
@pytest.mark.parametrize("case", list(PRODUCT_CASES))
def test_product_path(case, moving, tmp_path):
    kind, spec = PRODUCT_CASES[case]
    plants = _plants(spec)
    df, lv_dir, odf, olv = _product(kind, plants, tmp_path, moving)
    _check_product(df, lv_dir, odf, olv, moving)
    L = len(LEVELS_D[kind])
    if case == "phi_only":
        # Phi reaches only the boundary terms: every other column keeps the device value of the clean dataset
        cdf = _product(kind, [], tmp_path, moving, oracle=False)[0]
        for c in df.columns:
            if "Φ" not in c:
                assert np.array_equal(df[c].values, cdf[c].values), c
        if moving:
            assert not np.array_equal(df["BΦZ"].values, cdf["BΦZ"].values)
    if case == "top_level_one_time":
        # omega's top level is missing at one time: fixed mode drops it from the omega families at every time,
        # moving mode only at that step
        lens = [r[1].size for r in _read_levels(lv_dir / "Ce_level.csv")]
        assert lens == ([L - 1] * NT_D if not moving else [L, L - 1, L, L])
    if case == "u_on_uniform_levels":
        rows = _read_levels(lv_dir / "Ck_5_level.csv")
        assert np.isfinite(rows[1][1][2]) and not np.isfinite(_read_levels(lv_dir / "Ck_4_level.csv")[1][1][2])


def test_moving_step_with_every_level_missing(tmp_path):
    """omega missing on every level of one step: the host's NaN path drops every level of the vertical-flux pieces,
    and returns NaN for their bottom-minus-top part (xarray's ``isel(level=-1)`` on an empty level axis would raise);
    the other steps are untouched."""
    plants = _plants([(3, 2, k, None, None) for k in range(len(LEVELS_D["irregular"]))])
    df = _product("irregular", plants, tmp_path, True, oracle=False)[0]
    cdf = _product("irregular", [], tmp_path, True, oracle=False)[0]
    for name in ("BAz", "BAe", "BKz", "BKe", "BΦZ", "BΦE"):
        assert np.isnan(df[name].values[2]), name
    for c in ("Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "Gz", "Ge") + tuple(H.BOUNDARY_TERMS):
        assert np.array_equal(df[c].values[[0, 1, 3]], cdf[c].values[[0, 1, 3]]), c
