"""The numpy oracle against the reference's own bundled outputs (SURVEY.md Appendix C).

These pins are what gives the oracle its authority: the reference itself cannot be imported
in this image.  Tolerances are the ones established in the survey session."""
import os

import numpy as np
import pandas as pd
import pytest

from oracle import lec_oracle as O
import helpers as H

S = os.path.join(H.GOLDEN, "samples")


@pytest.fixture(scope="module")
def catarina():
    P, _ = H.load_prepared("Catarina_NCEP-R2.nc")
    box = (-55, -36, -35, -20)          # samples/Catarina_NCEP-R2_fixed/log.txt:3
    return O.slice_domain_fixed(P, *box), box


def test_catarina_fixed_all_columns(catarina):
    """Pin 1: all 22 columns x 36 steps of the bundled results CSV, ref-dtype mode with the
    legacy (numpy 1.x) float64 c1/c2 the goldens were produced with."""
    P, box = catarina
    df, _, _ = O.lec_fixed(P, *box, mode="ref", legacy_0d=True)
    g = pd.read_csv(os.path.join(S, "Catarina_NCEP-R2_fixed", "Catarina_NCEP-R2_fixed_results.csv"), index_col=0)
    assert list(g.columns) == list(df.columns)
    assert len(g) == len(df) == 36
    tol = {c: 1e-12 for c in g.columns}
    tol.update({"Ck": 1e-9, "RKz": 1e-8, "RKe": 1e-9})        # Ck integrand is float32 in the reference
    for c in g.columns:
        rel = np.max(np.abs(df[c].values - g[c].values) / np.abs(g[c].values))
        assert rel <= tol[c], (c, rel)


def test_catarina_nep50_boundary_terms(catarina):
    """With NEP-50 float32 c1/c2 (pinned numpy 2.0) the boundary terms move by <= 1e-4."""
    P, box = catarina
    df, _, _ = O.lec_fixed(P, *box, mode="ref", legacy_0d=False)
    g = pd.read_csv(os.path.join(S, "Catarina_NCEP-R2_fixed", "Catarina_NCEP-R2_fixed_results.csv"), index_col=0)
    for c in ["BAz", "BAe", "BKz", "BKe"]:
        assert H.series_err(df[c].values, g[c].values) <= 1e-4


def test_catarina_fp64_mode_close_to_reference(catarina):
    """fp64-upcast arithmetic vs the reference's own float32-propagating output (Appendix C.3)."""
    P, box = catarina
    df, _, _ = O.lec_fixed(P, *box, mode="fp64")
    g = pd.read_csv(os.path.join(S, "Catarina_NCEP-R2_fixed", "Catarina_NCEP-R2_fixed_results.csv"), index_col=0)
    for c in ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe", "Gz", "Ge"]:
        assert H.series_err(df[c].values, g[c].values) <= 5e-3, c


def _golden_levels(folder, term, nrows):
    g = pd.read_csv(os.path.join(S, folder, f"{term}_lv_ISBL3.csv"), index_col=0)
    cols = np.array([float(c) for c in g.columns])
    g.columns = list(cols / 100.0 if cols.max() > 2000 else cols)      # newer files label levels in Pa
    return g.iloc[:nrows]


def test_testdata_fixed_per_level_pins():
    """Pin 2: testdata_NCEP-R2.nc is the 5-step/5-level subset of Reg1-Representative; levels
    700-1000 hPa (centred d/dp in both) must match the bundled per-level CSVs."""
    P, _ = H.load_prepared("testdata_NCEP-R2.nc")
    box = (-60, -30, -42.5, -17.5)       # inputs/box_limits_Reg1
    P = O.slice_domain_fixed(P, *box)
    _, lv, _ = O.lec_fixed(P, *box, mode="ref")
    lev_hpa = P.level / 100.0
    cols = [float(x) for x in lev_hpa if x >= 700]
    kidx = [int(np.where(lev_hpa == c)[0][0]) for c in cols]
    checks = {"Kz": (5, 5e-7), "Ke": (5, 5e-7), "Az": (5, 5e-7), "Ae": (5, 5e-7), "Ce": (5, 5e-7),
              "Ck": (5, 2e-6), "Ge": (4, 1e-11), "Gz": (4, 2e-5)}    # row 5 of G*: one-sided dT/dt in the subset
    for term, (nrows, tol) in checks.items():
        g = _golden_levels("Reg1-Representative_NCEP-R2_fixed", term, nrows)
        ours = np.asarray(lv[term], dtype=np.float64)[:nrows][:, kidx]
        ref = g[cols].values
        rel = np.max(np.abs(ours - ref) / np.abs(ref))
        assert rel <= tol, (term, rel)
    # per-level Cz / Ca goldens carry the opposite sign (Jan-2024 version skew): compare magnitudes
    for term in ("Cz", "Ca"):
        g = _golden_levels("Reg1-Representative_NCEP-R2_fixed", term, 5)
        ours = np.asarray(lv[term], dtype=np.float64)[:, kidx]
        ref = g[cols].values
        assert np.max(np.abs(np.abs(ours) - np.abs(ref)) / np.abs(ref)) <= 2e-5, term


def test_testdata_track_pins():
    """Pin 3: moving box selection, per-level energy arithmetic and the moving-mode Q."""
    P, tr = H.load_prepared("testdata_NCEP-R2.nc", track="track_testdata_NCEP-R2")
    P = O.slice_domain_track(P, tr)
    _, lv, boxes = O.lec_moving(P, tr, mode="ref")
    for lim, (iw, ie, js, jn) in boxes:
        assert (P.lon[iw], P.lon[ie], P.lat[js], P.lat[jn]) == (-52.5, -37.5, -30.0, -15.0)
    lev_hpa = P.level / 100.0
    cols = [float(x) for x in lev_hpa if x >= 700]
    kidx = [int(np.where(lev_hpa == c)[0][0]) for c in cols]
    checks = {"Kz": (3, 2e-7), "Ke": (3, 2e-7), "Az": (3, 1e-12), "Ae": (3, 1e-12), "Ce": (3, 1e-12),
              "Ge": (2, 1e-10), "Gz": (2, 1e-10)}
    for term, (nrows, tol) in checks.items():
        g = _golden_levels("Reg1-Representative_NCEP-R2_track-15x15", term, nrows)
        ours = np.asarray(lv[term], dtype=np.float64)[:nrows][:, kidx]
        ref = g[cols].values
        rel = np.max(np.abs(ours - ref) / np.abs(ref))
        assert rel <= tol, (term, rel)


def test_preprocessing_contract():
    """process_data semantics (preprocessing.py:275-365): lon wrapped to [-180,180) and sorted,
    levels ascending in Pa, lat ascending, radians in the coordinate dtype."""
    P, _ = H.load_prepared("Catarina_NCEP-R2.nc")
    assert P.lon.dtype == np.float32 and P.rlons.dtype == np.float32 and P.coslats.dtype == np.float32
    assert np.all(np.diff(P.lon) > 0) and P.lon.min() >= -180 and P.lon.max() < 180
    assert np.all(np.diff(P.lat) > 0) and np.all(np.diff(P.level) > 0)
    assert P.level.min() >= 1000.0 and P.level.max() == 100000.0
    assert P.fields["Air Temperature"].shape == (36, 17, len(P.lat), len(P.lon))


def test_handle_nans_interpolates_then_drops():
    lev = np.array([100., 200., 300., 400.])
    f = np.array([[1., np.nan, 3., 4.], [np.nan, 2., 3., 4.]])
    out, l2 = O.handle_nans(f, lev, -1)
    # interior gap filled linearly; the leading NaN cannot be extrapolated -> level 100 dropped for all rows
    assert np.array_equal(l2, lev[1:])
    assert np.allclose(out, [[2., 3., 4.], [2., 3., 4.]])


def test_stationary_track_reproduces_the_pinned_fixed_run(catarina):
    """The moving framework's integrated columns have no reference output of their own (SURVEY.md 8(c)).  They are
    pinned indirectly: a track that never moves, whose 19 x 15 degree box is the Catarina fixed box, must give the
    fixed framework's numbers -- the same 12 terms that pin 1 checks against the reference's own CSV -- although the
    moving path takes a different route through the oracle (per-step BoxState on [level][lat][lon], dT/dt from the
    global ``np.gradient`` over the time axis, box limits from ``get_limits``)."""
    P, box = catarina
    times = pd.to_datetime(P.time)
    track = pd.DataFrame({"Lat": -27.5, "Lon": -45.5, "length": 15.0, "width": 19.0}, index=times)
    lim = O.get_limits(track, times[3])
    assert (lim["min_lon"], lim["max_lon"], lim["min_lat"], lim["max_lat"]) == tuple(float(b) for b in box)
    fixed, flv, extra = O.lec_fixed(P, *box, mode="fp64")
    moving, mlv, boxes = O.lec_moving(P, track, mode="fp64")
    assert all(idx == boxes[0][1] for _, idx in boxes)
    for c in fixed.columns:
        assert c in moving.columns
        a, b = moving[c].values, fixed[c].values
        assert np.max(np.abs(a - b)) <= 1e-12 * np.max(np.abs(b)), c
    for name, want in (("BΦZ", extra["BΦZ"]), ("BΦE", extra["BΦE"])):       # computed by both, written by the moving one
        assert np.max(np.abs(moving[name].values - np.asarray(want))) <= 1e-12 * np.max(np.abs(want)), name
    for name in ("Az", "Ae", "Kz", "Ke", "Ge", "Gz", "Ck", "Ca", "Ce", "Cz"):
        f, m = np.asarray(flv[name]), np.asarray(mlv[name])
        assert f.shape == m.shape and np.max(np.abs(f - m)) <= 1e-12 * np.max(np.abs(f)), name


def test_boundary_pieces_reassemble_the_boundary_terms(catarina):
    """The per-level pieces ``boundary_terms(pieces=)`` exposes (the engine's ``lec_set_boundary_levels`` output)
    rebuild the six boundary terms: c1 * trapz_p(E-W) + c2 * trapz_p(N-S) - (vertical at the last level - at the
    first).  Fixed box: one [time][3][level] array per term."""
    P, box = catarina
    b = O.BoxState(O.to_mode(P, "fp64"), *box, fixed=True)
    pieces = {}
    out = O.boundary_terms(b, pieces=pieces)
    assert set(pieces) == set(H.BOUNDARY_TERMS)
    nt, nlev = len(P.time), len(P.level)
    c1 = -1 / (O.Re * b.xlength * b.ylength)
    c2 = -1 / (O.Re * b.ylength)
    arr = H.boundary_pieces(pieces)
    assert arr.shape == (nt, 6, 3, nlev) and np.isfinite(arr).all()
    np.testing.assert_array_equal(arr[:, 5, 1], arr[:, 4, 1])              # BΦE takes BΦZ's N-S piece (sic)
    for n, name in enumerate(H.BOUNDARY_TERMS):
        ew, ns, vert = arr[:, n, 0], arr[:, n, 1], arr[:, n, 2]
        want = c1 * O.trapz(ew, b.p, -1) + c2 * O.trapz(ns, b.p, -1) - (vert[:, -1] - vert[:, 0])
        assert H.series_err(want, out[name]) <= 1e-12, name
        assert np.abs(ew).max() > 0 and np.abs(ns).max() > 0 and np.abs(vert).max() > 0, name
