"""The reference's own four CLI tests (tests/test_R2_fixed.py, test_R2_track.py, test_ERA5_fixed.py,
test_ERA5_track.py), call for call, against the ROOT module ``lorenzcycletoolkit`` of this repo: same imports,
same argv (including -p and -v), same sequence create_arg_parser -> setup_results_directory ->
initialize_logging -> prepare_data -> run_lec_analysis.  The reference's tests only check that nothing
raises; here the written results are compared with the oracle as well.  samples/testdata_ERA5.nc is missing
from the reference checkout, so a synthetic file with ERA5's on-disk conventions stands in for it."""
import os
import shutil
import sys

import numpy as np
import pandas as pd
import pytest

from oracle import lec_oracle as O
import helpers as H

pytestmark = pytest.mark.gpu
INP = os.path.join(H.GOLDEN, "inputs")
SAM = os.path.join(H.GOLDEN, "samples")


def _reference_flow(monkeypatch, argv, method):
    sys.path.insert(0, H.ROOT if hasattr(H, "ROOT") else os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from lorenzcycletoolkit import (create_arg_parser, initialize_logging, prepare_data, run_lec_analysis,
                                    setup_results_directory)
    monkeypatch.setattr("sys.argv", argv)
    args = create_arg_parser().parse_args()
    assert args.residuals and args.plots and args.verbosity and args.infile == argv[1]
    results_subdirectory, figures_directory, results_subdirectory_vertical_levels = setup_results_directory(args, method)
    app_logger = initialize_logging(results_subdirectory, args)
    app_logger.info("Starting LEC analysis")
    app_logger.info(f"Command line arguments: {args}")
    data = prepare_data(args, "inputs/namelist", app_logger)
    run_lec_analysis(data, args, results_subdirectory, figures_directory, results_subdirectory_vertical_levels, app_logger)
    return results_subdirectory


def _stage(tmp_path, monkeypatch, namelist, sample=None):
    # contents only (copyfile, not copy): the staged inputs stay writable when the checkout is read-only, so the
    # tests can put box_limits_Reg1 over box_limits as the reference's tests do
    os.makedirs(tmp_path / "inputs")
    os.makedirs(tmp_path / "samples")
    for f in os.listdir(INP):
        shutil.copyfile(os.path.join(INP, f), tmp_path / "inputs" / f)
    if sample:
        shutil.copyfile(os.path.join(SAM, sample), tmp_path / "samples" / sample)
    monkeypatch.chdir(tmp_path)
    shutil.copy(f"inputs/{namelist}", "inputs/namelist")


def _compare(results_subdirectory, stem, odf, tol):
    df = pd.read_csv(os.path.join(results_subdirectory, f"{stem}_results.csv"), index_col=0)
    assert list(df.columns) == list(odf.columns) and len(df) == len(odf)
    for c in odf.columns:
        assert H.series_err(df[c].values, odf[c].values) <= tol, c
    assert len(os.listdir(os.path.join(results_subdirectory, "results_vertical_levels"))) == 21


def test_R2_fixed(tmp_path, monkeypatch):
    _stage(tmp_path, monkeypatch, "namelist_NCEP-R2", "testdata_NCEP-R2.nc")
    shutil.copy("inputs/box_limits_Reg1", "inputs/box_limits")
    out = _reference_flow(monkeypatch, ["lorenzcycletoolkit.py", "samples/testdata_NCEP-R2.nc", "-r", "-f", "-p", "-v"], "fixed")
    P, _ = H.load_prepared("testdata_NCEP-R2.nc")
    box = (-60, -30, -42.5, -17.5)
    odf, _, _ = O.lec_fixed(O.slice_domain_fixed(P, *box), *box, mode="fp64")
    _compare(out, "testdata_NCEP-R2_fixed", odf, 1e-5)


def test_R2_track(tmp_path, monkeypatch):
    _stage(tmp_path, monkeypatch, "namelist_NCEP-R2", "testdata_NCEP-R2.nc")
    shutil.copy("inputs/track_testdata_NCEP-R2", "inputs/track")
    out = _reference_flow(monkeypatch, ["lorenzcycletoolkit.py", "samples/testdata_NCEP-R2.nc", "-r", "-t", "-p", "-v"], "track")
    P, tr = H.load_prepared("testdata_NCEP-R2.nc", track="track_testdata_NCEP-R2")
    odf, _, _ = O.lec_moving(O.slice_domain_track(P, tr), tr, mode="fp64")
    _compare(out, "testdata_NCEP-R2_track", odf, 1e-5)
    assert os.path.exists(os.path.join(out, "testdata_NCEP-R2_track_trackfile"))


def _era5_oracle(nc, track=None):
    raw = O.read_netcdf3(nc)
    nl = O.read_namelist(os.path.join(INP, "namelist_ERA5"))
    return O.process_data(raw, nl, track)


def test_ERA5_fixed(tmp_path, monkeypatch):
    _stage(tmp_path, monkeypatch, "namelist_ERA5")
    H.write_era5_like("samples/testdata_ERA5.nc", True, 160)
    shutil.copy("inputs/box_limits_Reg1", "inputs/box_limits")
    out = _reference_flow(monkeypatch, ["lorenzcycletoolkit.py", "samples/testdata_ERA5.nc", "-r", "-f", "-p", "-v"], "fixed")
    box = (-60, -30, -42.5, -17.5)
    P = O.slice_domain_fixed(_era5_oracle("samples/testdata_ERA5.nc"), *box)
    odf, _, _ = O.lec_fixed(P, *box, mode="fp64")
    _compare(out, "testdata_ERA5_fixed", odf, 1e-9)          # packed int16 -> float64 fields: fp64 gate


def test_ERA5_track(tmp_path, monkeypatch):
    _stage(tmp_path, monkeypatch, "namelist_ERA5")
    H.write_era5_like("samples/testdata_ERA5.nc", False, 161)       # float32 fields, odd row length
    shutil.copy("inputs/track_testdata_ERA5", "inputs/track")
    out = _reference_flow(monkeypatch, ["lorenzcycletoolkit.py", "samples/testdata_ERA5.nc", "-r", "-t", "-p", "-v"], "track")
    tr = O.read_track(os.path.join(INP, "track_testdata_ERA5"))
    P = O.slice_domain_track(_era5_oracle("samples/testdata_ERA5.nc", tr), tr)
    odf, _, _ = O.lec_moving(P, tr, mode="fp64")
    _compare(out, "testdata_ERA5_track", odf, 1e-5)
