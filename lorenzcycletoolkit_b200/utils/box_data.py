"""``BoxData`` drop-in (reference: ``src/utils/box_data.py:57-310``).

The reference's ``BoxData`` slices the box and materialises ~50 full-size arrays (zonal /
area means and eddies of T, u, v, omega, Phi, Q, plus sigma) that the four term classes then
combine.  Here the constructor snaps the box exactly as the reference does and hands the
prepared fields to the CUDA engine (``lec_run_host``), which returns every term and every
per-level integrand of every time step in one pass; the term classes in
``lorenzcycletoolkit_b200.analysis`` read those results.  There is no CPU path.
"""

from __future__ import annotations

import numpy as np

from .. import engine as E

G = 9.80665     # metpy.constants.g (box_data.py:233-241: Phi = hgt * g)
RE = 6371008.7714   # metpy.constants.Re

_UNIT_TO_SI = {  # pint factors of the units that occur in the reference's inputs/namelist_*
    "K": 1.0, "kelvin": 1.0, "m/s": 1.0, "m s-1": 1.0, "m s**-1": 1.0, "Pa/s": 1.0, "Pa s-1": 1.0,
    "Pa s**-1": 1.0, "hPa/s": 100.0, "m**2/s**2": 1.0, "m2 s-2": 1.0, "m**2 s**-2": 1.0, "m2/s2": 1.0,
    "m": 1.0, "gpm": 1.0, "dam": 10.0,
}

ENGINE_FIELDS = ("Air Temperature", "Eastward Wind Component", "Northward Wind Component",
                 "Omega Velocity", "Geopotential")


def unit_factor(unit, name):
    try:
        return _UNIT_TO_SI[str(unit).strip()]
    except KeyError:
        raise ValueError(f"Unit error in {name}: cannot convert '{unit}' to SI") from None


def engine_fields(data, variable_list_df):
    """The five engine fields (T, u, v, omega, Phi) of a prepared dataset as C-contiguous
    arrays of one float dtype, plus the namelist-unit -> SI factors (box_data.py:297-310;
    geopotential height is multiplied by g, :233-241)."""
    arrs, scale = [], []
    for row in ENGINE_FIELDS:
        if row == "Geopotential" and row not in variable_list_df.index:
            row_used, extra = "Geopotential Height", G
        else:
            row_used, extra = row, 1.0
        var = variable_list_df.loc[row_used]["Variable"]
        arrs.append(np.asarray(data[var]))
        scale.append(unit_factor(variable_list_df.loc[row_used]["Units"], row_used) * extra)
    dt = np.float32 if all(a.dtype == np.float32 for a in arrs) else np.float64
    return [np.ascontiguousarray(a, dtype=dt) for a in arrs], scale, np.dtype(dt)


class RawInput:
    """The five engine fields of a raw-backed dataset: records as stored + index maps + decode rules
    (``lec_run_host_raw``); slicing the time axis only slices the slot -> record map."""

    def __init__(self, fields, decode, rec, lev, lat, lon):
        self.fields, self.decode, self.rec, self.lev, self.lat, self.lon = fields, decode, rec, lev, lat, lon

    def __getitem__(self, sel):
        return RawInput(self.fields, self.decode, self.rec[sel], self.lev, self.lat, self.lon)

    def run(self, eng, steps, want_boundary=False):
        E.pin_arrays(self.fields)          # the loader's pageable record arrays: page-locked once (LEC_PIN_RAW=0: never)
        return eng.run_host_raw(self.fields, self.lon, self.lat, self.lev, self.rec, steps, decode=self.decode,
                                want_boundary=want_boundary)


def engine_raw(data, variable_list_df):
    """:func:`engine_fields` for a dataset whose fields are still in file layout (``data.raw``): returns
    ``(RawInput, scale, dtype)`` or None when the dataset is host-prepared."""
    store = getattr(data, "raw", None)
    if store is None:
        return None
    names, scale = [], []
    for row in ENGINE_FIELDS:
        if row == "Geopotential" and row not in variable_list_df.index:
            row_used, extra = "Geopotential Height", G
        else:
            row_used, extra = row, 1.0
        names.append(variable_list_df.loc[row_used]["Variable"])
        scale.append(unit_factor(variable_list_df.loc[row_used]["Units"], row_used) * extra)
    dts = [store.dtype_of(v) for v in names]
    dt = np.dtype(np.float32) if all(d == np.float32 for d in dts) else np.dtype(np.float64)
    raw = RawInput([store.fields[v] for v in names], [store.decode[v] for v in names],
                   store.rec, store.lev, store.lat, store.lon)
    return raw, scale, dt


def make_engine(data, dtype, scale, max_steps, max_box_rows=0, **opts):
    f64 = lambda a: np.asarray(a, dtype=np.float64)     # stored-dtype values upcast, never recomputed
    return E.LecEngine(f64(data.lon), f64(data.lat), f64(data.rlons), f64(data.rlats), f64(data.coslats),
                       f64(data.level), dtype, scale, max_steps=max_steps, max_box_rows=max_box_rows, **opts)


def run_time_sharded(data, dtype, scale, fields, steps, max_box_rows, opts):
    """Evaluate ``steps`` on this process's GPU, or -- when ``torch.distributed`` is initialised
    (``torchrun``) -- this rank's contiguous time shard (+ one halo slot each side, taken from the
    input) followed by ONE all-gather of the per-step results (SURVEY.md 8(e)).  Every rank returns
    the full ``(terms, levels, flags, timing, boundary_pieces)``; only the device index differs per rank."""
    import os
    rank, world = 0, 1
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
    except ImportError:
        dist = None
    opts = dict(opts)
    windows = bool(opts.pop("host_windows", False))      # lec_set_host_windows: each rank windows its own shard

    def run(eng, f, st):
        eng.set_host_windows(windows)
        if isinstance(f, RawInput):
            out = f.run(eng, st, want_boundary=True)
        else:
            out = eng.run_host(f, st, want_boundary=True)
        return out + (eng.last_boundary,)

    if world == 1:
        with make_engine(data, dtype, scale, max_steps=min(len(steps), 256), max_box_rows=max_box_rows, **opts) as eng:
            terms, levels, flags, bnd = run(eng, fields, steps)
            return terms, levels, flags, eng.last_timing(), bnd

    import torch
    from .. import sharding as S
    ngpu = torch.cuda.device_count()
    opts.setdefault("device", int(os.environ.get("LOCAL_RANK", rank)) % max(ngpu, 1))
    n = len(steps)
    shards = S.time_shards(n, world)
    a, b = shards[rank]
    nlev = len(data.level)
    terms = np.zeros((0, E.NTERMS)); levels = np.zeros((0, E.NLEVEL_TERMS, nlev)); flags = np.zeros(0, np.int32)
    bnd = np.zeros((0, 6, 3, nlev))
    timing = (0.0, 0.0, 0.0)
    if b > a:
        lo = int(min(steps["slot"][a:b].min(), steps["slot_m"][a:b].min(), steps["slot_p"][a:b].min()))
        hi = int(max(steps["slot"][a:b].max(), steps["slot_m"][a:b].max(), steps["slot_p"][a:b].max())) + 1
        local = S.shard_steps(steps, a, b, lo)
        with make_engine(data, dtype, scale, max_steps=min(b - a, 256), max_box_rows=max_box_rows, **opts) as eng:
            if isinstance(fields, RawInput):
                terms, levels, flags, bnd = run(eng, fields[lo:hi], local)
            else:
                terms, levels, flags, bnd = run(eng, [np.ascontiguousarray(f[lo:hi]) for f in fields], local)
            timing = eng.last_timing()
    # one collective for everything: [terms | levels | boundary pieces | flags] per step (NCCL on the GPU,
    # gloo on the host)
    m = len(terms)                      # 0 on a rank whose shard is empty (more ranks than time steps / shard size)
    nl, nb = E.NLEVEL_TERMS * nlev, E.NBOUNDARY_PIECES * nlev
    packed = np.concatenate([terms.reshape(m, E.NTERMS), levels.reshape(m, nl), bnd.reshape(m, nb),
                             flags.reshape(m, 1).astype(np.float64)], axis=1)
    t = torch.from_numpy(np.ascontiguousarray(packed))
    if dist.get_backend() == "nccl":
        t = t.cuda(opts["device"])
    full = S.gather_results(t, shards).cpu().numpy()
    return (np.ascontiguousarray(full[:, :E.NTERMS]),
            np.ascontiguousarray(full[:, E.NTERMS:E.NTERMS + nl]).reshape(n, E.NLEVEL_TERMS, nlev),
            full[:, -1].astype(np.int32), timing,
            np.ascontiguousarray(full[:, E.NTERMS + nl:E.NTERMS + nl + nb]).reshape(n, 6, 3, nlev))


def boundary_constants(data, i0, i1, j0, j1):
    """``c1 = -1 / (Re xlength ylength)``, ``c2 = -1 / (Re ylength)`` (boundary_terms.py:122-123) of a snapped
    box, in float64 from the stored-dtype radians, as the engine evaluates them."""
    rl, rp = np.asarray(data.rlons, dtype=np.float64), np.asarray(data.rlats, dtype=np.float64)
    xlen = rl[i1] - rl[i0]
    ylen = np.sin(rp[j1]) - np.sin(rp[j0])
    return np.array([-1.0 / (RE * xlen * ylen), -1.0 / (RE * ylen)])


def time_seconds(time):
    """``differentiate(time, datetime_unit="s")``: float64 seconds since the first time."""
    time = np.asarray(time)
    if np.issubdtype(time.dtype, np.datetime64):
        return ((time - time.min()) / np.timedelta64(1, "s")).astype(np.float64)
    return time.astype(np.float64) - float(time.min())


class BoxData:
    """Box state of the LEC computation for a fixed box over all times (``args.fixed``) or for
    one time step of the moving framework (``dTdt`` given), evaluated on the GPU."""

    def __init__(self, data, variable_list_df, western_limit, eastern_limit, southern_limit,
                 northern_limit, args, results_subdirectory, results_subdirectory_vertical_levels,
                 dTdt=None, engine_options=None):
        self.args = args
        self.results_subdirectory = results_subdirectory
        self.results_subdirectory_vertical_levels = results_subdirectory_vertical_levels
        self.LonIndexer = variable_list_df.loc["Longitude"]["Variable"]
        self.LatIndexer = variable_list_df.loc["Latitude"]["Variable"]
        self.TimeName = variable_list_df.loc["Time"]["Variable"]
        self.VerticalCoordIndexer = variable_list_df.loc["Vertical Level"]["Variable"]
        self.PressureData = np.asarray(data.level, dtype=np.float64)
        self.times = np.atleast_1d(np.asarray(data.time))
        self.data, self.variable_list_df = data, variable_list_df     # Dz / De read one level of u, v on the host

        # box_data.py:115-135: nearest snap (ties -> larger coordinate), lengths in the coord dtype
        self.idx = (E.nearest_index(data.lon, western_limit), E.nearest_index(data.lon, eastern_limit),
                    E.nearest_index(data.lat, southern_limit), E.nearest_index(data.lat, northern_limit))
        i0, i1, j0, j1 = self.idx
        self.western_limit, self.eastern_limit = data.lon[i0], data.lon[i1]
        self.southern_limit, self.northern_limit = data.lat[j0], data.lat[j1]
        self.xlength = data.rlons[i1] - data.rlons[i0]
        self.ylength = np.sin(data.rlats[j1]) - np.sin(data.rlats[j0])
        if i1 - i0 < 1 or j1 - j0 < 1:
            raise ValueError("the box must span at least two grid points in longitude and latitude")

        raw = engine_raw(data, variable_list_df) if dTdt is None else None
        if raw is not None:
            fields, scale, dtype = raw
            nt = len(fields.rec)
        else:
            fields, scale, dtype = engine_fields(data, variable_list_df)
            fields = [f if f.ndim == 4 else f[None] for f in fields]
            nt = fields[0].shape[0]
        opts = dict(engine_options or {})
        if dTdt is None:
            # fixed framework: d/dt over ALL file times (thermodynamics.py:109-110)
            if nt < 2:
                raise ValueError("the fixed framework needs at least two time steps (np.gradient over time)")
            steps = E.time_stencil(time_seconds(self.times), E.make_steps(nt))
        else:
            # one step of the moving framework with an explicit dT/dt field
            # (lec_moving_framework.py:719-730).  The engine differentiates T itself, so the given
            # tendency is encoded as a second time slot T + dTdt * tau, exactly representable in fp64.
            if nt != 1:
                raise ValueError("dTdt is only accepted together with a single-time dataset")
            tau = 65536.0
            fields = [np.ascontiguousarray(f, dtype=np.float64) for f in fields]
            dtype = np.dtype(np.float64)
            tend = np.asarray(dTdt, dtype=np.float64).reshape(fields[0].shape[1:]) / scale[0]
            fields[0] = np.ascontiguousarray(np.stack([fields[0][0], fields[0][0] + tend * tau]))
            for f in range(1, 5):
                fields[f] = np.ascontiguousarray(np.stack([fields[f][0], fields[f][0]]))
            steps = E.make_steps(1)
            steps["slot"], steps["slot_m"], steps["slot_p"] = 0, 0, 1
            steps["ct_m"], steps["ct_0"], steps["ct_p"] = 0.0, -1.0 / tau, 1.0 / tau
        steps["i0"], steps["i1"], steps["j0"], steps["j1"] = i0, i1, j0, j1
        self.terms, self.levels, self.flags, self.timing_ms, self.boundary_levels = run_time_sharded(
            data, dtype, scale, fields, steps, j1 - j0 + 1, opts)
        self.dtype = dtype
        self.c12 = np.tile(boundary_constants(data, i0, i1, j0, j1), (len(self.terms), 1))

    # ---- views the term classes use --------------------------------------------------- #
    def term(self, name):
        return self.terms[:, E.TERM_NAMES.index(name)]

    def level_term(self, name):
        return self.levels[:, E.LEVEL_TERM_NAMES.index(name), :]

    def boundary_pieces(self, name):
        """``[step][3][level]``: E-W, N-S and vertical-flux pieces of boundary term ``name`` per level."""
        return self.boundary_levels[:, E.BOUNDARY_TERMS.index(name)]

    @property
    def has_nonfinite(self):
        return bool((self.flags & E.FLAG_NONFINITE).any())


class BoxBatch(BoxData):
    """All steps of the moving framework in ONE engine call: one box per step
    (lec_moving_framework.py:639-740 evaluates one ``BoxData`` per time step in a Python loop).
    ``limits`` is a list of dicts with min_lon / max_lon / min_lat / max_lat (``get_limits``)."""

    def __init__(self, data, variable_list_df, limits, args, results_subdirectory,
                 results_subdirectory_vertical_levels, engine_options=None):
        self.args = args
        self.results_subdirectory = results_subdirectory
        self.results_subdirectory_vertical_levels = results_subdirectory_vertical_levels
        self.LonIndexer = variable_list_df.loc["Longitude"]["Variable"]
        self.LatIndexer = variable_list_df.loc["Latitude"]["Variable"]
        self.TimeName = variable_list_df.loc["Time"]["Variable"]
        self.VerticalCoordIndexer = variable_list_df.loc["Vertical Level"]["Variable"]
        self.PressureData = np.asarray(data.level, dtype=np.float64)
        self.times = np.asarray(data.time)
        nt = len(self.times)
        if nt != len(limits):
            raise ValueError("one box per time step is required")
        if nt < 2:
            raise ValueError("the moving framework needs at least two time steps (dT/dt over the track times)")
        fields, scale, dtype = engine_raw(data, variable_list_df) or engine_fields(data, variable_list_df)
        # global dT/dt over the track-selected times (lorenzcycletoolkit.py:184-186)
        steps = E.time_stencil(time_seconds(self.times), E.make_steps(nt))
        self.boxes = []
        for it, lim in enumerate(limits):
            i0, i1 = E.nearest_index(data.lon, lim["min_lon"]), E.nearest_index(data.lon, lim["max_lon"])
            j0, j1 = E.nearest_index(data.lat, lim["min_lat"]), E.nearest_index(data.lat, lim["max_lat"])
            if i1 - i0 < 1 or j1 - j0 < 1:
                raise ValueError(f"box of step {it} spans fewer than two grid points")
            steps["i0"][it], steps["i1"][it], steps["j0"][it], steps["j1"][it] = i0, i1, j0, j1
            self.boxes.append((i0, i1, j0, j1))
        rows = int(max(b[3] - b[2] + 1 for b in self.boxes))
        # moving boxes stage only each slot's window (engine_options={"host_windows": False}: whole slots)
        opts = dict(engine_options or {})
        opts.setdefault("host_windows", True)
        self.terms, self.levels, self.flags, self.timing_ms, self.boundary_levels = run_time_sharded(
            data, dtype, scale, fields, steps, rows, opts)
        self.dtype = dtype
        self.idx = None
        self.c12 = np.array([boundary_constants(data, *b) for b in self.boxes])

    def step(self, it):
        """The single-step view the term classes see in the moving framework."""
        return _StepView(self, it)


class _StepView:
    def __init__(self, batch, it):
        self._b = batch
        for k in ("args", "results_subdirectory", "results_subdirectory_vertical_levels", "LonIndexer",
                  "LatIndexer", "TimeName", "VerticalCoordIndexer", "PressureData", "dtype"):
            setattr(self, k, getattr(batch, k))
        self.times = batch.times[it:it + 1]
        self.terms = batch.terms[it:it + 1]
        self.levels = batch.levels[it:it + 1]
        self.flags = batch.flags[it:it + 1]
        self.boundary_levels = batch.boundary_levels[it:it + 1]
        self.c12 = batch.c12[it:it + 1]
        self.idx = batch.boxes[it]

    term = BoxData.term
    level_term = BoxData.level_term
    boundary_pieces = BoxData.boundary_pieces
    has_nonfinite = BoxData.has_nonfinite
