"""GPU tests of the drop-in host API (BoxData, term classes, lec_fixed, lec_moving, CLI): the
reference's own smoke tests (tests/test_R2_fixed.py, tests/test_R2_track.py) with numeric
assertions against the bundled goldens and the oracle added."""
import argparse
import logging
import os
import shutil

import numpy as np
import pandas as pd
import pytest

from oracle import lec_oracle as O
import helpers as H
from lorenzcycletoolkit_b200 import cli
from lorenzcycletoolkit_b200.utils import preprocessing as PP

pytestmark = pytest.mark.gpu
INP = os.path.join(H.GOLDEN, "inputs")
SAM = os.path.join(H.GOLDEN, "samples")


def _workdir(tmp_path, box=None, track=None):
    # contents only (copyfile, not copy): the staged inputs stay writable when the checkout is read-only
    os.makedirs(tmp_path / "inputs")
    shutil.copyfile(os.path.join(INP, "namelist_NCEP-R2"), tmp_path / "inputs" / "namelist")
    if box:
        shutil.copyfile(os.path.join(INP, box), tmp_path / "inputs" / "box_limits")
    if track:
        shutil.copyfile(os.path.join(INP, track), tmp_path / "inputs" / "track")


def test_cli_fixed_catarina_matches_bundled_results(tmp_path, monkeypatch):
    """End-to-end known-answer test: the CLI on samples/Catarina_NCEP-R2.nc reproduces the
    reference's own Catarina_NCEP-R2_fixed_results.csv (fp32 file -> the reference's float32
    propagation bounds the agreement, SURVEY.md Appendix C.3)."""
    _workdir(tmp_path)
    (tmp_path / "inputs" / "box_limits").write_text("min_lon;-55\nmax_lon;-36\nmin_lat;-35\nmax_lat;-20\n")
    monkeypatch.chdir(tmp_path)
    cli.main([os.path.join(SAM, "Catarina_NCEP-R2.nc"), "-r", "-f"])
    out = tmp_path / "LEC_Results" / "Catarina_NCEP-R2_fixed"
    df = pd.read_csv(out / "Catarina_NCEP-R2_fixed_results.csv", index_col=0)
    g = pd.read_csv(os.path.join(SAM, "Catarina_NCEP-R2_fixed", "Catarina_NCEP-R2_fixed_results.csv"), index_col=0)
    assert list(df.columns) == list(g.columns)
    assert list(df.index) == list(g.index)
    for c in ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe", "Gz", "Ge"]:
        assert H.series_err(df[c].values, g[c].values) <= 5e-3, c
    # 21 per-level files with header + one row per time step
    files = sorted(os.listdir(out / "results_vertical_levels"))
    assert len(files) == 21
    az = pd.read_csv(out / "results_vertical_levels" / "Az_lv_ISBL3.csv", index_col=0)
    assert az.shape == (36, 17) and float(az.columns[0]) == 1000.0
    gaz = pd.read_csv(os.path.join(SAM, "Catarina_NCEP-R2_fixed", "Az_lv_ISBL3.csv"), index_col=0)
    assert H.series_err(az.values, gaz.values) <= 1e-3
    assert os.path.exists(out / "log.Catarina_NCEP-R2")


def test_lec_fixed_against_oracle_fp64_semantics(tmp_path):
    """lec_fixed on testdata_NCEP-R2.nc / box_limits_Reg1 (the reference's tests/test_R2_fixed.py
    case) against the oracle evaluated in fp64 on the same fp32 values: 1e-5 (fp32-input mode)."""
    nl = PP.read_namelist(os.path.join(INP, "namelist_NCEP-R2"))
    args = argparse.Namespace(infile=os.path.join(SAM, "testdata_NCEP-R2.nc"), fixed=True, track=False,
                              choose=False, residuals=True, box_limits=os.path.join(INP, "box_limits_Reg1"),
                              outname=None, plots=False, cdsapi=False, mpas=False)
    data = PP.prepare_data(args, os.path.join(INP, "namelist_NCEP-R2"), box_limits_file=args.box_limits)
    lv_dir = tmp_path / "lv"
    os.makedirs(lv_dir)
    from lorenzcycletoolkit_b200.frameworks import lec_fixed
    df = lec_fixed(data, nl, str(tmp_path), str(lv_dir), logging.getLogger("t"), args)
    P, _ = H.load_prepared("testdata_NCEP-R2.nc")
    box = (-60, -30, -42.5, -17.5)
    P = O.slice_domain_fixed(P, *box)
    odf, _, _ = O.lec_fixed(P, *box, mode="fp64")
    assert list(df.columns) == list(odf.columns)
    for c in odf.columns:
        assert H.series_err(df[c].values, odf[c].values) <= 1e-5, c


def test_cli_track_matches_oracle_and_writes_reference_files(tmp_path, monkeypatch):
    """The reference's tests/test_R2_track.py case with numbers: results CSV vs the oracle's
    moving framework, trackfile columns, per-level rows labelled per step."""
    _workdir(tmp_path, track="track_testdata_NCEP-R2")
    monkeypatch.chdir(tmp_path)
    cli.main([os.path.join(SAM, "testdata_NCEP-R2.nc"), "-r", "-t"])
    out = tmp_path / "LEC_Results" / "testdata_NCEP-R2_track"
    df = pd.read_csv(out / "testdata_NCEP-R2_track_results.csv", index_col=0)
    P, tr = H.load_prepared("testdata_NCEP-R2.nc", track="track_testdata_NCEP-R2")
    P = O.slice_domain_track(P, tr)
    odf, _, _ = O.lec_moving(P, tr, mode="fp64")
    assert list(df.columns) == list(odf.columns)
    for c in odf.columns:
        assert H.series_err(df[c].values, odf[c].values) <= 1e-5, c
    tf = pd.read_csv(out / "testdata_NCEP-R2_track_trackfile", sep=";")
    assert list(tf.columns[:9]) == ["time", "Lat", "Lon", "length", "width", "min_lon", "max_lon", "min_lat", "max_lat"]
    assert {"min_max_zeta_850", "min_hgt_850", "max_wind_850"} <= set(tf.columns)
    assert len(tf) == 5 and tf["time"][1] == "2005-08-08-0600"
    # 850-hPa diagnostics (lec_diag850 kernel) against the numpy restatement on the same pre-sliced domain
    k = int(np.where(np.asarray(P.level) == 85000.0)[0][0])
    boxes = []
    for n in range(5):
        (j0, j1), (i0, i1) = O.label_slice(P.lat, tf["min_lat"][n], tf["max_lat"][n]), O.label_slice(P.lon, tf["min_lon"][n], tf["max_lon"][n])
        boxes.append((n, i0, i1 - 1, j0, j1 - 1))
    F = P.fields
    ovals, oidx = O.diag850(F["Eastward Wind Component"][:, k], F["Northward Wind Component"][:, k],
                            F["Geopotential Height"][:, k], P.lon, P.lat, boxes)
    nx = boxes[0][2] - boxes[0][1] + 1
    assert np.allclose(tf["min_max_zeta_850"], ovals[:, 0], rtol=1e-12) and np.allclose(tf["min_hgt_850"], ovals[:, 2], rtol=1e-12)
    assert np.allclose(tf["max_wind_850"], ovals[:, 3], rtol=1e-12)
    assert np.array_equal(tf["max_wind_850_lat"], [P.lat[boxes[n][3] + oidx[n, 3] // nx] for n in range(5)])
    assert np.array_equal(tf["min_max_zeta_850_lon"], [P.lon[boxes[n][1] + oidx[n, 0] % nx] for n in range(5)])
    ke = pd.read_csv(out / "results_vertical_levels" / "Ke_lv_ISBL3.csv", index_col=0)
    assert list(ke.index) == [t.strftime("%Y-%m-%d %H:%M:%S") for t in pd.to_datetime(P.time)]


def test_cli_track_zeta_flag_takes_vorticity_at_the_track_centre(tmp_path, monkeypatch):
    """``-z`` with a track that has no min_max_zeta_850 column: the reference takes izeta_850 at the grid point
    nearest to (central_lat, central_lon) (lec_moving_framework.py:317-324); a column in the track file wins
    over everything, NaN included (:313-314); positions always come from the box extrema."""
    _workdir(tmp_path, track="track_testdata_NCEP-R2")
    monkeypatch.chdir(tmp_path)
    cli.main([os.path.join(SAM, "testdata_NCEP-R2.nc"), "-r", "-t", "-z"])
    out = tmp_path / "LEC_Results" / "testdata_NCEP-R2_track"
    tf = pd.read_csv(out / "testdata_NCEP-R2_track_trackfile", sep=";")
    P, tr = H.load_prepared("testdata_NCEP-R2.nc", track="track_testdata_NCEP-R2")
    P = O.slice_domain_track(P, tr)
    k = int(np.where(np.asarray(P.level) == 85000.0)[0][0])
    boxes, centres = [], []
    for n in range(5):
        (j0, j1), (i0, i1) = O.label_slice(P.lat, tf["min_lat"][n], tf["max_lat"][n]), O.label_slice(P.lon, tf["min_lon"][n], tf["max_lon"][n])
        boxes.append((n, i0, i1 - 1, j0, j1 - 1))
        centres.append((O.nearest_index(P.lon, tf["Lon"][n]), O.nearest_index(P.lat, tf["Lat"][n])))
    F = P.fields
    ovals, oidx = O.diag850(F["Eastward Wind Component"][:, k], F["Northward Wind Component"][:, k],
                            F["Geopotential Height"][:, k], P.lon, P.lat, boxes, centres=centres)
    assert np.allclose(tf["min_max_zeta_850"], ovals[:, 4], rtol=1e-12)
    assert not np.allclose(tf["min_max_zeta_850"], ovals[:, 0], rtol=1e-3)         # not the box minimum
    nx = boxes[0][2] - boxes[0][1] + 1
    assert np.array_equal(tf["min_max_zeta_850_lon"], [P.lon[boxes[n][1] + oidx[n, 0] % nx] for n in range(5)])
    # a track file that carries the column wins, with or without -z
    trk = tmp_path / "inputs" / "track"
    rows = trk.read_text().strip().splitlines()
    trk.write_text("\n".join([rows[0] + ";min_max_zeta_850"] + [r + f";{-1e-5 * (n + 1)}" for n, r in enumerate(rows[1:])]) + "\n")
    cli.main([os.path.join(SAM, "testdata_NCEP-R2.nc"), "-r", "-t", "-z"])
    tf2 = pd.read_csv(out / "testdata_NCEP-R2_track_trackfile", sep=";")
    assert np.allclose(tf2["min_max_zeta_850"], [-1e-5 * (n + 1) for n in range(5)], rtol=1e-12)


def test_batched_level_files_equal_per_step_appends(tmp_path):
    """One CSV write per file for the whole track (compute_and_store_terms_batch) leaves the files the
    reference's 21-appends-per-step loop would leave, byte for byte, and the same term lists."""
    import filecmp
    import logging
    from lorenzcycletoolkit_b200.utils.box_data import BoxBatch
    from lorenzcycletoolkit_b200.frameworks import lec_moving_framework as MF
    from lorenzcycletoolkit_b200.frameworks.lec_fixed_framework import create_level_files
    nl = PP.read_namelist(os.path.join(INP, "namelist_NCEP-R2"))
    args = argparse.Namespace(infile=os.path.join(SAM, "testdata_NCEP-R2.nc"), fixed=False, track=True,
                              choose=False, residuals=True, trackfile=os.path.join(INP, "track_testdata_NCEP-R2"),
                              cdsapi=False, mpas=False)
    data = PP.prepare_data(args, os.path.join(INP, "namelist_NCEP-R2"))
    lim = dict(min_lon=-52.5, max_lon=-37.5, min_lat=-30.0, max_lat=-15.0)
    log = logging.getLogger("lorenzcycletoolkit")
    out = {}
    for mode in ("step", "batch"):
        d = tmp_path / mode
        os.makedirs(d)
        create_level_files(str(d), "time", nl.loc["Vertical Level"]["Variable"], data.level)
        batch = BoxBatch(data, nl, [lim] * len(data.time), args, None, str(d))
        terms = MF.create_terms_dict(args)
        if mode == "step":
            for it in range(len(data.time)):
                terms = MF.compute_and_store_terms(batch.step(it), terms, log)
        else:
            terms = MF.compute_and_store_terms_batch(batch, terms, log)
        out[mode] = terms
    files = sorted(os.listdir(tmp_path / "step"))
    assert len(files) >= 19 and files == sorted(os.listdir(tmp_path / "batch"))
    match, mismatch, errors = filecmp.cmpfiles(tmp_path / "step", tmp_path / "batch", files, shallow=False)
    assert not mismatch and not errors
    assert out["step"] == out["batch"]


def test_boxdata_single_step_with_explicit_dTdt():
    """BoxData(idata, ..., dTdt=idTdt) -- the per-step call of the reference's moving loop --
    agrees with the batched evaluation."""
    from lorenzcycletoolkit_b200.utils.box_data import BoxData, BoxBatch
    nl = PP.read_namelist(os.path.join(INP, "namelist_NCEP-R2"))
    args = argparse.Namespace(infile=os.path.join(SAM, "testdata_NCEP-R2.nc"), fixed=False, track=True,
                              choose=False, residuals=True, trackfile=os.path.join(INP, "track_testdata_NCEP-R2"),
                              cdsapi=False, mpas=False)
    data = PP.prepare_data(args, os.path.join(INP, "namelist_NCEP-R2"))
    lim = dict(min_lon=-52.5, max_lon=-37.5, min_lat=-30.0, max_lat=-15.0)
    batch = BoxBatch(data, nl, [lim] * len(data.time), args, None, None)
    T = data["TMP_2_ISBL"].astype(np.float64)
    tsec = ((data.time - data.time.min()) / np.timedelta64(1, "s")).astype(np.float64)
    dTdt = np.gradient(T, tsec, axis=0)
    it = 2
    one = BoxData(data.isel(time=slice(it, it + 1)), nl, -52.5, -37.5, -30.0, -15.0, args, None, None, dTdt=dTdt[it])
    assert np.allclose(one.terms[0], batch.terms[it], rtol=2e-6, atol=0)


def test_dissipation_terms_from_friction_velocity(tmp_path):
    """Without -r the fixed framework evaluates Dz / De from a "Friction Velocity" namelist row
    (generation_and_dissipation_terms.py:154-188, unfinished in the reference: formula from the source, UNPINNED).
    A surface field (time, lat, lon) rides through the loader's wrap / sort / crop with the 4-D fields."""
    import shutil
    from lorenzcycletoolkit_b200.frameworks import lec_fixed
    rng = np.random.default_rng(3)
    src = os.path.join(SAM, "Catarina_NCEP-R2.nc")
    ust = rng.uniform(0.1, 0.6, size=(36, 7, 8)).astype(np.float32)          # file order: lat north -> south, lon 0..360
    path = str(tmp_path / "Catarina_ust.nc")
    H.write_netcdf3_copy(src, path, extra={"UST": (("initial_time0_hours", "lat_2", "lon_2"), ust, {"units": "m/s"})})
    nlf = tmp_path / "namelist"
    nlf.write_text(open(os.path.join(INP, "namelist_NCEP-R2")).read().rstrip("\n") + "\nFriction Velocity;friction_velocity;UST;m/s\n")
    boxf = tmp_path / "box"
    boxf.write_text("min_lon;-55\nmax_lon;-36\nmin_lat;-35\nmax_lat;-20\n")
    nl = PP.read_namelist(str(nlf))
    args = argparse.Namespace(infile=path, fixed=True, track=False, choose=False, residuals=False,
                              box_limits=str(boxf), outname=None, plots=False, cdsapi=False, mpas=False)
    data = PP.prepare_data(args, str(nlf), box_limits_file=args.box_limits)
    assert data["UST"].shape == (36,) + data["TMP_2_ISBL"].shape[2:]
    os.makedirs(tmp_path / "lv")
    df = lec_fixed(data, nl, str(tmp_path), str(tmp_path / "lv"), logging.getLogger("t"), args)
    assert list(df.columns[:16]) == ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe",
                                     "Gz", "Ge", "Dz", "De"]
    # oracle: the same box state, the friction field wrapped / sorted / cropped as process_data does
    P, _ = H.load_prepared("Catarina_NCEP-R2.nc")
    box = (-55, -36, -35, -20)
    lat_f = np.array([-20.0, -22.5, -25.0, -27.5, -30.0, -32.5, -35.0])
    lon_f = (np.array([305.0, 307.5, 310.0, 312.5, 315.0, 317.5, 320.0, 322.5]) + 180) % 360 - 180
    u = ust[:, np.argsort(lat_f)][:, :, np.argsort(lon_f)].astype(np.float64)
    P = O.to_mode(O.slice_domain_fixed(P, *box), "fp64")
    b = O.BoxState(P, *box, fixed=True)
    j0, j1, i0, i1 = b.sl
    od = O.dissipation_terms(b, u[:, j0:j1, i0:i1])
    assert H.series_err(df["Dz"].values, od["Dz"]) <= 1e-6 and H.series_err(df["De"].values, od["De"]) <= 1e-6
    # with -r the columns are absent, and without the namelist row the call says what is missing
    nl2 = PP.read_namelist(os.path.join(INP, "namelist_NCEP-R2"))
    data2 = PP.prepare_data(args, os.path.join(INP, "namelist_NCEP-R2"), box_limits_file=args.box_limits)
    with pytest.raises(ValueError, match="Friction Velocity"):
        lec_fixed(data2, nl2, str(tmp_path), str(tmp_path / "lv"), logging.getLogger("t"), args)


def test_cli_stationary_track_equals_cli_fixed(tmp_path, monkeypatch):
    """`-t` with a track that never moves over the Catarina box against `-f` on the same box: the moving framework
    (track-time selection, domain slicing around the track, per-step boxes from get_limits, global dT/dt, BoxBatch)
    and the fixed one (box file, domain = the box, BoxData) must agree on every column both write -- the columns the
    bundled Catarina results pin for the fixed run."""
    P, _ = H.load_prepared("Catarina_NCEP-R2.nc")
    _workdir(tmp_path)
    (tmp_path / "inputs" / "box_limits").write_text("min_lon;-55\nmax_lon;-36\nmin_lat;-35\nmax_lat;-20\n")
    with open(tmp_path / "inputs" / "track", "w") as f:
        f.write("time;Lat;Lon;length;width\n")
        for t in pd.to_datetime(P.time):
            f.write(f"{t.strftime('%Y-%m-%d-%H%M')};-27.5;-45.5;15;19\n")
    monkeypatch.chdir(tmp_path)
    nc = os.path.join(SAM, "Catarina_NCEP-R2.nc")
    cli.main([nc, "-r", "-f"])
    cli.main([nc, "-r", "-t"])
    fixed = pd.read_csv(tmp_path / "LEC_Results" / "Catarina_NCEP-R2_fixed" / "Catarina_NCEP-R2_fixed_results.csv", index_col=0)
    track = pd.read_csv(tmp_path / "LEC_Results" / "Catarina_NCEP-R2_track" / "Catarina_NCEP-R2_track_results.csv", index_col=0)
    assert len(fixed) == len(track) == 36
    tf = pd.read_csv(tmp_path / "LEC_Results" / "Catarina_NCEP-R2_track" / "Catarina_NCEP-R2_track_trackfile", sep=";")
    assert (tf["min_lon"] == -55).all() and (tf["max_lon"] == -36).all() and (tf["min_lat"] == -35).all() and (tf["max_lat"] == -20).all()
    for c in fixed.columns:
        assert c in track.columns, c
        assert H.series_err(track[c].values, fixed[c].values) <= 1e-5, c
