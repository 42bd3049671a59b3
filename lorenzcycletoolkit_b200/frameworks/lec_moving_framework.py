"""Semi-Lagrangian moving-box driver (reference: ``src/frameworks/lec_moving_framework.py:35-841``).

The reference loops over time steps in Python and builds one ``BoxData`` (about 150 xarray
expressions) per step.  Here the per-step boxes are collected first (``get_limits``) and the
whole track is evaluated by ONE engine call (``BoxBatch``); the per-step term objects, the
per-level CSV rows, the results CSV and the ``*_trackfile`` are then written exactly as before."""

from __future__ import annotations

import logging
import os
from pathlib import Path

import numpy as np
import pandas as pd

from ..sharding import is_rank0 as _is_rank0
from ..analysis import BoundaryTerms, ConversionTerms, EnergyContents, GenerationDissipationTerms
from ..utils.box_data import BoxBatch, unit_factor, G
from ..utils.calc_budget_and_residual import calc_budget_diff, calc_residuals
from ..utils.preprocessing import read_track, _label_slice
from .lec_fixed_framework import create_level_files

RE = 6371008.7714


def create_terms_dict(args):
    """lec_moving_framework.py:35-55."""
    terms = ["Az", "Ae", "Kz", "Ke", "Cz", "Ca", "Ck", "Ce", "BAz", "BAe", "BKz", "BKe", "BΦZ", "BΦE"]
    terms += ["Gz", "Ge"] if args.residuals else ["Gz", "Ge", "Dz", "De"]
    return {t: [] for t in terms}


def handle_track_file(data, times, LonIndexer, LatIndexer, TimeIndexer, args, app_logger):
    """Read the track and check that it lies inside the data (lec_moving_framework.py:58-160)."""
    trackfile = args.trackfile
    try:
        track = read_track(trackfile)
    except FileNotFoundError:
        app_logger.error(f"❌ Track file {trackfile} not found.")
        raise
    lon, lat = np.asarray(data.lon), np.asarray(data.lat)
    if track["Lon"].min() < lon.min() or track["Lon"].max() > lon.max():
        raise ValueError("Track longitude limits are outside the data domain")
    if track["Lat"].min() < lat.min() or track["Lat"].max() > lat.max():
        raise ValueError("Track latitude limits are outside the data domain")
    t = pd.to_datetime(times)
    if track.index.min() > t.max() or track.index.max() < t.min():
        raise ValueError("Track time limits do not overlap the data time limits")
    return track


def get_limits(args, t, data850, track=None):
    """Box of one time step (lec_moving_framework.py:199-266): the track row nearest in time,
    centre +- width/2 (default 15 x 15 degrees)."""
    if not getattr(args, "track", False):
        raise NotImplementedError("the interactive --choose framework needs a display (out of scope)")
    closest = int(np.argmin(np.abs(track.index - t)))
    row = track.iloc[closest]
    central_lat, central_lon = row["Lat"], row["Lon"]
    width, length = row.get("width", 15), row.get("length", 15)
    return {"datestr": pd.to_datetime(t).strftime("%Y-%m-%d-%H%M"),
            "central_lat": central_lat, "central_lon": central_lon, "length": length, "width": width,
            "min_lon": central_lon - width / 2, "max_lon": central_lon + width / 2,
            "min_lat": central_lat - length / 2, "max_lat": central_lat + length / 2}


def diagnostics_850(data, variable_list_df, limits_list, device=None, windows=True):
    """850-hPa wind speed, relative vorticity (MetPy's ``vorticity`` on the lat / lon grid) and geopotential
    height (lec_moving_framework.py:650-663), their extrema inside every step's label-sliced box
    (get_position, :269-417) and the vorticity at the grid point nearest to the track centre (the ``-z``
    branch, :317-324), for ALL time steps in one ``lec_diag850_host`` call on the GPU (the reference recomputes
    the domain-wide fields per step inside its time loop).
    Returns per step ``(values[5], flat_index[4], lat_of_box, lon_of_box)``: ``engine.DIAG_NAMES`` order, then
    zeta at the centre.  ``windows``: gather and copy only each step's window of the three planes
    (``lec_diag850_host_windows``, same bits), else the whole planes (``lec_diag850_host``)."""
    from .. import engine as E
    k = int(np.argmin(np.abs(np.asarray(data.level, dtype=np.float64) - 85000.0)))
    if float(data.level[k]) != 85000.0:
        raise KeyError("85000 Pa level not found (the moving framework needs 850 hPa)")

    lat, lon = np.asarray(data.lat), np.asarray(data.lon)
    rows_z = ["Geopotential", G] if "Geopotential" in variable_list_df.index else ["Geopotential Height", 1.0]
    z_div = rows_z[1]
    names = ["Eastward Wind Component", "Northward Wind Component", rows_z[0]]
    su, sv, sz = (unit_factor(variable_list_df.loc[row]["Units"], row) for row in names)

    def planes(a, b, origins=None, shape=None):
        """u, v, z of times a..b-1: whole planes, or the windows of ``origins`` (one per time)."""
        out = []
        for row in names:
            var = variable_list_df.loc[row]["Variable"]
            out.append(data.level_plane(var, k)[a:b] if origins is None else
                       data.level_plane_windows(var, k, origins, *shape, times=np.arange(a, b)))
        return out
    steps = np.zeros(len(limits_list), dtype=E.DIAG_STEP_DTYPE)
    boxes = []
    for it, lim in enumerate(limits_list):
        js, is_ = _label_slice(lat, lim["min_lat"], lim["max_lat"]), _label_slice(lon, lim["min_lon"], lim["max_lon"])
        if js.stop <= js.start or is_.stop <= is_.start:
            raise ValueError(f"the box of step {it} selects no grid point")
        # izeta_850.sel(latitude=central_lat, longitude=central_lon, method="nearest") (:319-323)
        steps[it] = (it, is_.start, is_.stop - 1, js.start, js.stop - 1,
                     E.nearest_index(lon, lim["central_lon"]), E.nearest_index(lat, lim["central_lat"]), 0)
        boxes.append((lat[js], lon[is_]))
    rank, world, dist = 0, 1, None
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
    except ImportError:
        pass
    if device is None:
        import torch
        device = int(os.environ.get("LOCAL_RANK", rank)) % max(torch.cuda.device_count(), 1) if world > 1 else \
            int(os.environ.get("LOCAL_RANK", 0))
    def run(st, a, b):                 # steps of times a..b-1, slot = time - a
        if not windows:
            return E.diag850_host(*planes(a, b), lon, lat, st, scale=(su, sv, sz), z_div=z_div, device=device)
        origins, wy, wx = E.diag_windows(st, len(lon), len(lat))
        return E.diag850_host_windows(*planes(a, b, origins, (wy, wx)), origins, lon, lat, st, scale=(su, sv, sz),
                                      z_div=z_div, device=device)

    if world == 1:
        vals, idx = run(steps, 0, len(steps))
    else:
        # time-sharded like the LEC terms: this rank's steps (no halo: the diagnostics are per-time), then one
        # all-gather of the 4 values + 4 indices per step
        import torch
        from .. import sharding as S
        shards = S.time_shards(len(steps), world)
        a, b = shards[rank]
        local = np.zeros((b - a, 9))
        if b > a:
            st = steps[a:b].copy()
            st["slot"] -= a
            lv, li = run(st, a, b)
            local[:, :5], local[:, 5:] = lv, li
        t = torch.from_numpy(local)
        if dist.get_backend() == "nccl":
            t = t.cuda(device)
        full = S.gather_results(t, shards).cpu().numpy()
        vals, idx = np.ascontiguousarray(full[:, :5]), full[:, 5:].astype(np.int32)
    return [(vals[it], idx[it], boxes[it][0], boxes[it][1]) for it in range(len(limits_list))]


def get_position(track, limits, d850, args):
    """Extrema inside the (unsnapped, label-sliced) box (lec_moving_framework.py:269-417) from one step's
    entry of :func:`diagnostics_850`.  As in the reference: a ``min_max_zeta_850`` column of the track wins
    unconditionally; without it ``-z`` takes the vorticity at the grid point nearest to the track centre, else
    the box minimum (southern hemisphere) / maximum; ``min_hgt_850`` / ``max_wind_850`` of the track win when
    not NaN; positions always come from the computed fields.  The data time must be a track time (KeyError
    otherwise, ``track.loc[datestr]`` at :291)."""
    vals, idx, blat, blon = d850
    zeta_min, zeta_max, hgt_min, wind_max, zeta_centre = (float(x) for x in vals)
    row = None
    if track is not None:
        ts = pd.to_datetime(limits["datestr"], format="%Y-%m-%d-%H%M")
        if ts not in track.index:
            raise KeyError(f"{limits['datestr']}: the data time is not in the track file")
        row = track.loc[ts]

    def from_track(col):
        return row is not None and col in track.columns and not pd.isna(row[col])

    if row is not None and "min_max_zeta_850" in track.columns:
        min_max_zeta = float(row["min_max_zeta_850"])
    elif row is not None and getattr(args, "zeta", False):
        min_max_zeta = zeta_centre
    else:
        min_max_zeta = zeta_min if limits["min_lat"] < 0 else zeta_max
    min_hgt = float(row["min_hgt_850"]) if from_track("min_hgt_850") else hgt_min
    max_wind = float(row["max_wind_850"]) if from_track("max_wind_850") else wind_max

    def where(flat):
        j, i = divmod(int(flat), len(blon))
        return blat[j], blon[i]

    zlat, zlon = where(idx[0] if blat.min() < 0 else idx[1])
    hlat, hlon = where(idx[2])
    wlat, wlon = where(idx[3])
    return {"min_max_zeta_850_lat": zlat, "min_max_zeta_850_lon": zlon, "min_max_zeta_850": min_max_zeta,
            "min_hgt_850_lat": hlat, "min_hgt_850_lon": hlon, "min_hgt_850": min_hgt,
            "max_wind_850_lat": wlat, "max_wind_850_lon": wlon, "max_wind_850": max_wind}


def compute_and_store_terms(box_obj, terms_dict, app_logger):
    """One step's 16 scalars appended to the lists (lec_moving_framework.py:430-495)."""
    try:
        ec = EnergyContents(box_obj, "moving", app_logger)
        for n, f in (("Az", ec.calc_az), ("Ae", ec.calc_ae), ("Kz", ec.calc_kz), ("Ke", ec.calc_ke)):
            terms_dict[n].append(f())
        ct = ConversionTerms(box_obj, "moving", app_logger)
        for n, f in (("Cz", ct.calc_cz), ("Ca", ct.calc_ca), ("Ck", ct.calc_ck), ("Ce", ct.calc_ce)):
            terms_dict[n].append(f())
        bt = BoundaryTerms(box_obj, "moving", app_logger)
        for n, f in (("BAz", bt.calc_baz), ("BAe", bt.calc_bae), ("BKz", bt.calc_bkz), ("BKe", bt.calc_bke),
                     ("BΦZ", bt.calc_boz), ("BΦE", bt.calc_boe)):
            terms_dict[n].append(f())
        gd = GenerationDissipationTerms(box_obj, "moving", app_logger)
        terms_dict["Gz"].append(gd.calc_gz())
        terms_dict["Ge"].append(gd.calc_ge())
        if "Dz" in terms_dict:
            terms_dict["Dz"].append(gd.calc_dz())
            terms_dict["De"].append(gd.calc_de())
    except Exception:
        app_logger.exception("❌ An exception occurred while computing the LEC terms of a step")
        raise
    return terms_dict


def compute_and_store_terms_batch(batch, terms_dict, app_logger):
    """All steps at once: the term classes see the whole :class:`BoxBatch`, return one value per step and
    append every step's per-level row with ONE write per CSV file (the reference appends to 21 files per
    step, energy_contents.py:210-226 and its copies) -- same file contents, row for row."""
    batch.batched = True
    try:
        one = {k: [] for k in terms_dict}
        compute_and_store_terms(batch, one, app_logger)
        for k, v in one.items():
            terms_dict[k].extend(np.asarray(v[0], dtype=np.float64).reshape(-1).tolist())
    finally:
        batch.batched = False
    return terms_dict


def finalize_results(times, terms_dict, args, results_subdirectory, out_track, app_logger, write=True):
    """Results CSV + trackfile (lec_moving_framework.py:498-543)."""
    df = pd.DataFrame(terms_dict, index=pd.to_datetime(times), dtype=float)
    app_logger.info("📈 Estimating budget terms...")
    df = calc_budget_diff(df, np.asarray(times), app_logger)
    if args.residuals:
        app_logger.info("🧮 Computing residuals...")
        df = calc_residuals(df, app_logger)
    method = "track" if args.track else "choose"
    infile_name = os.path.basename(args.infile).split(".nc")[0]
    results_file = os.path.join(results_subdirectory, f"{infile_name}_{method}_results.csv")
    if not write:
        return results_file, df
    df.to_csv(results_file)
    app_logger.info(f"💾 Results saved to {results_file}")
    out_track = out_track.rename(columns={"datestr": "time", "central_lat": "Lat", "central_lon": "Lon"})
    output_trackfile = os.path.join(results_subdirectory, f"{infile_name}_{method}_trackfile")
    out_track.to_csv(output_trackfile, index=False, sep=";")
    app_logger.info(f"📍 System track saved to {output_trackfile}")
    return results_file, df


def lec_moving(data, variable_list_df, dTdt, results_subdirectory, figures_directory,
               results_subdirectory_vertical_levels, app_logger, args, engine_options=None):
    """``dTdt`` is accepted for signature compatibility and ignored: the row kernel evaluates the
    same centred time difference of T over the track-selected times (lorenzcycletoolkit.py:184-186)
    from the adjacent time slots of the resident field."""
    app_logger = app_logger or logging.getLogger("lorenzcycletoolkit")
    app_logger.info("📊 Computing energetics using moving framework")
    LonIndexer = variable_list_df.loc["Longitude"]["Variable"]
    LatIndexer = variable_list_df.loc["Latitude"]["Variable"]
    TimeName = variable_list_df.loc["Time"]["Variable"]
    VerticalCoordIndexer = variable_list_df.loc["Vertical Level"]["Variable"]
    write = _is_rank0()          # under torchrun every rank computes its time shard; rank 0 writes the files
    if write:
        create_level_files(results_subdirectory_vertical_levels, TimeName, VerticalCoordIndexer, data.level)
    else:
        results_subdirectory_vertical_levels = None
    times = pd.to_datetime(np.asarray(data.time))
    if len(times) == 0:
        raise ValueError("Mismatch between trackfile and data! Check that the track times exist in the file.")
    track = handle_track_file(data, times, LonIndexer, LatIndexer, TimeName, args, app_logger)

    limits_list = [get_limits(args, t, None, track) for t in times]
    # staging windows (lec_set_host_windows, lec_diag850_host_windows): the run's host->device bytes follow the box,
    # not the domain; engine_options={"host_windows": False} stages whole slots / planes (the same bits)
    windows = bool((engine_options or {}).get("host_windows", True))
    d850 = diagnostics_850(data, variable_list_df, limits_list, windows=windows)
    rows = []
    for it, t in enumerate(times):
        limits = limits_list[it]
        position = get_position(track, limits, d850[it], args)
        app_logger.info(f"🗺️ {t}: box center=({limits['central_lat']:.2f}, {limits['central_lon']:.2f}), "
                        f"size={limits['length']}°x{limits['width']}°")
        rows.append({**limits, **position})
    out_track = pd.DataFrame(rows)

    try:
        batch = BoxBatch(data, variable_list_df, limits_list, args, results_subdirectory,
                         results_subdirectory_vertical_levels, engine_options=engine_options)
    except Exception:
        app_logger.exception("❌ An exception occurred while creating BoxData object")
        raise
    _, _, call_ms = batch.timing_ms
    app_logger.info(f"🚀 B200 engine: {len(times)} steps in {call_ms:.2f} ms")
    terms_dict = create_terms_dict(args)
    if batch.has_nonfinite:
        # the reference's NaN path (_handle_nans) interpolates / drops levels per time step
        for it in range(len(times)):
            terms_dict = compute_and_store_terms(batch.step(it), terms_dict, app_logger)
    else:
        terms_dict = compute_and_store_terms_batch(batch, terms_dict, app_logger)
    results_file, df = finalize_results(times, terms_dict, args, results_subdirectory, out_track, app_logger,
                                        write=write)
    return df
