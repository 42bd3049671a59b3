"""The oracle's ``raw=`` hook: the per-level families of ``energy_contents``, ``conversion_terms`` and
``generation_terms`` before the reference's ``_handle_nans``, and the static stability before its 0.03 floor.  The
GPU suite compares the engine's NaN pattern with these (tests/test_level_axis_gpu.py), so the hook must not move a
single bit of the oracle's results."""
import numpy as np

from oracle import lec_oracle as O
import helpers as H

T0 = np.datetime64("2020-01-01T00")


def _box(level, plants=()):
    nt, nlat, nlon = 4, 9, 12
    fields = H.smooth_fields(nt, len(level), nlat, nlon, np.float32, seed=3, level=level)
    for f, t, k, j, i in plants:
        fields[f][t, k, j, i] = np.nan
    P = H.prepared_from_arrays(fields, -50 + 0.5 * np.arange(nlon), -20 + 0.5 * np.arange(nlat), level,
                               T0 + np.arange(nt) * np.timedelta64(6, "h"))
    Q = O.to_mode(P, "fp64")
    return O.BoxState(Q, Q.lon[1], Q.lon[10], Q.lat[1], Q.lat[7], fixed=True)


def _families(b, raw):
    lv, terms = {}, {}
    for fn in (O.energy_contents, O.conversion_terms, O.generation_terms):
        terms.update(fn(b, lv) if raw is None else fn(b, lv, raw))
    return terms, lv


def test_raw_families_equal_the_saved_ones_without_missing_values():
    for level in (np.linspace(1e4, 1e5, 6), np.geomspace(5e3, 1e5, 7)):
        b = _box(level)
        raw = {}
        t0, lv0 = _families(b, None)
        t1, lv1 = _families(b, raw)
        assert set(t0) == set(t1) and all(np.array_equal(t0[k], t1[k]) for k in t0)
        assert list(lv0) == list(lv1) == list(raw) and len(raw) == 21
        for k in raw:
            assert np.array_equal(lv0[k], lv1[k]) and np.array_equal(raw[k], lv1[k]), k
        assert (b.sigma_prefloor > 0.03).all() and np.array_equal(b.sigma_prefloor, b.sigma_AA)


def test_raw_families_keep_the_missing_levels():
    """u missing at an interior level k of one slot: the integrated families are NaN there before ``_handle_nans``
    and interpolated after it; Ck_5's d[u]/dp is np.gradient's, so on an exactly uniform level axis (centred
    difference without the centre) it stays finite at k, on an irregular one it is NaN."""
    k = 3
    for level, ck5_finite in ((np.linspace(1e4, 1e5, 6), True), (np.geomspace(5e3, 1e5, 7), False)):
        b = _box(level, [(1, 2, k, 4, 5)])
        raw = {}
        _, lv = _families(b, raw)
        assert np.isnan(raw["Ck"][2, k]) and np.isfinite(lv["Ck"][2]).all()
        assert np.isnan(raw["Kz"][2, k]) and np.isfinite(lv["Kz"][2]).all()
        assert np.isfinite(raw["Ck"][[0, 1, 3]]).all()
        assert np.isnan(raw["Ck_4"][2, k]) and np.isfinite(raw["Ck_5"][2, k]) == ck5_finite
        assert np.isfinite(b.sigma_prefloor).all()


def test_prefloor_sigma_of_a_missing_temperature():
    """T missing at level k: sigma before the floor is NaN at k (g T / cp) and at k +- 1 (d T / dp reads level k);
    the floor turns those into 0.03."""
    k = 2
    b = _box(np.geomspace(5e3, 1e5, 7), [(0, 1, k, 4, 5)])
    low = ~(b.sigma_prefloor[1] > 0.03)
    assert low.tolist() == [i in (k - 1, k, k + 1) for i in range(7)]
    assert np.isnan(b.sigma_prefloor[1, k - 1:k + 2]).all() and (b.sigma_AA[1, k - 1:k + 2] == 0.03).all()
    assert np.array_equal(np.where(b.sigma_prefloor > 0.03, b.sigma_prefloor, 0.03), b.sigma_AA)
