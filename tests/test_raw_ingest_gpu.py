"""lec_run_host_raw: fields still in FILE layout (latitude north-to-south, longitudes 0..360, levels in any
order with extra ones above 10 hPa, int16-packed or float, a time selection) against lec_run_host on the
arrays the host pipeline would have prepared -- bit-identical results, fewer PCIe bytes."""
import os

import numpy as np
import pytest

import helpers as H
from lorenzcycletoolkit_b200 import engine as E
from lorenzcycletoolkit_b200.utils import preprocessing as PP
from test_engine_synthetic_gpu import _dataset

pytestmark = pytest.mark.gpu


def _raw_layout(rng, fields, extra_levels=2, roll=7):
    """Scramble engine-layout fields into a file layout; returns raw arrays and the engine->raw maps."""
    nt, nlev, nlat, nlon = fields[0].shape
    lev_perm = rng.permutation(nlev + extra_levels)            # raw level order
    lev_map = np.array([int(np.where(lev_perm == k)[0][0]) for k in range(nlev)], dtype=np.int32)
    lat_map = np.arange(nlat - 1, -1, -1, dtype=np.int32)      # stored north -> south
    lon_map = ((np.arange(nlon) + roll) % nlon).astype(np.int32)
    raws = []
    for f in fields:
        raw = (rng.normal(size=(nt, nlev + extra_levels, nlat, nlon)) * 1e3).astype(f.dtype)    # junk in unused levels
        raw[:, lev_map[:, None, None], lat_map[None, :, None], lon_map[None, None, :]] = f
        raws.append(np.ascontiguousarray(raw))
    return raws, lon_map, lat_map, lev_map


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_float_records_any_layout(dtype):
    rng = np.random.default_rng(11)
    P, fields = _dataset(48, 19, 6, 7, dtype)
    steps = H.fixed_steps(P, P.lon[2], P.lon[44], P.lat[1], P.lat[17])
    raws, lon_map, lat_map, lev_map = _raw_layout(rng, fields)
    raws[0][2, lev_map[3], lat_map[5], lon_map[9]] = -9999.0       # a fill value inside the box
    ref_fields = [f.copy() for f in fields]
    ref_fields[0][2, 3, 5, 9] = np.nan
    with H.make_engine(P, dtype, [1.0] * 5) as eng:
        a = eng.run_host(ref_fields, steps)
        h2d_a = eng.last_transfer()[0]
        b = eng.run_host_raw(raws, lon_map, lat_map, lev_map, np.arange(7), steps,
                             decode=[dict(fills=[-9999.0])] + [{}] * 4)
        h2d_b = eng.last_transfer()[0]
    assert (a[2][1:4] & E.FLAG_NONFINITE).all()
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)
    nk = int(lev_map.max() - lev_map.min() + 1)      # the raw level RANGE the maps touch crosses PCIe
    assert h2d_b * 6 == h2d_a * nk


def test_time_selection_and_crop():
    """Engine grid = a crop of the raw grid (rows and columns), slots = every other record."""
    rng = np.random.default_rng(12)
    P, fields = _dataset(40, 15, 5, 6, np.float32)
    nt, nlev, nlat, nlon = fields[0].shape
    big = [rng.normal(size=(2 * nt, nlev, nlat + 9, nlon + 12)).astype(np.float32) for _ in range(5)]
    j0, i0 = 4, 5
    for b, f in zip(big, fields):
        b[::2, :, j0:j0 + nlat, i0:i0 + nlon] = f
    steps = H.fixed_steps(P, P.lon[1], P.lon[37], P.lat[1], P.lat[13])
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        a = eng.run_host(fields, steps)
        b = eng.run_host_raw(big, i0 + np.arange(nlon), j0 + np.arange(nlat), np.arange(nlev), 2 * np.arange(nt), steps)
        # only the touched rows cross PCIe (whole rows of them)
        assert eng.last_transfer()[0] == 5 * nt * nlev * nlat * (nlon + 12) * 4
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


@pytest.mark.parametrize("with_offset", [True, False])
def test_packed_int16(with_offset):
    """ERA5-style packing: decoded like xarray (float64 with an add_offset, float32 without), a quarter /
    half of the PCIe bytes of the decoded arrays."""
    rng = np.random.default_rng(13)
    P, fields = _dataset(36, 17, 6, 5, np.float64)
    steps = H.fixed_steps(P, P.lon[1], P.lon[33], P.lat[1], P.lat[15])
    packed, decode, decoded = [], [], []
    for f in fields:
        lo, hi = f.min(), f.max()
        scale = np.float64((hi - lo) / 65000.0)
        offset = np.float64(0.5 * (hi + lo)) if with_offset else None
        q = np.round((f - (offset if with_offset else 0.0)) / scale)
        if not with_offset:
            scale = np.float64(np.abs(f).max() / 32000.0)
            q = np.round(f / scale)
        q = q.astype(np.int16)
        packed.append(q)
        if with_offset:
            d = q.astype(np.float64); d *= scale; d += offset
        else:
            d = q.astype(np.float32); d *= scale
        decoded.append(d)
        decode.append(dict(scale=scale, offset=offset, float32=not with_offset))
    dt = np.float64 if with_offset else np.float32
    raws, lon_map, lat_map, lev_map = _raw_layout(rng, packed, extra_levels=1, roll=18)
    raws[3][1, lev_map[2], lat_map[6], lon_map[10]] = -32767
    decoded[3][1, 2, 6, 10] = np.nan
    decode[3]["fills"] = [-32767]
    with H.make_engine(P, dt, [1.0] * 5) as eng:
        a = eng.run_host(decoded, steps)
        h2d_a = eng.last_transfer()[0]
        b = eng.run_host_raw(raws, lon_map, lat_map, lev_map, np.arange(5), steps, decode=decode)
        h2d_b = eng.last_transfer()[0]
    for x, y in zip(a, b):
        assert np.array_equal(x, y, equal_nan=True)
    nk = int(lev_map.max() - lev_map.min() + 1)
    assert h2d_b * np.dtype(dt).itemsize * 6 == h2d_a * 2 * nk      # int16 records, raw level range nk for 6 engine levels


@pytest.mark.parametrize("dtype", [np.int16, np.float32, np.float64])
def test_big_endian_interleaved_records(dtype):
    """NetCDF-3 classic layout: big-endian values, the records of the five variables interleaved in one
    buffer (record r of T, of u, ... then record r + 1) -- consumed in place."""
    rng = np.random.default_rng(14)
    fdt = np.float32 if dtype == np.int16 else dtype
    P, fields = _dataset(32, 13, 5, 6, fdt)
    steps = H.fixed_steps(P, P.lon[1], P.lon[30], P.lat[1], P.lat[11])
    nt, nlev, nlat, nlon = fields[0].shape
    if dtype == np.int16:
        scales = [np.float64(np.abs(f).max() / 32000.0) for f in fields]
        native = [np.round(f / s).astype(np.int16) for f, s in zip(fields, scales)]
        ref = []
        for q, s in zip(native, scales):
            d = q.astype(np.float32); d *= s; ref.append(d)
        decode = [dict(scale=s, float32=True) for s in scales]
    else:
        native, ref, decode = fields, fields, None
    be = np.dtype(dtype).newbyteorder(">")
    file_buf = np.empty((nt, 5, nlev, nlat, nlon), dtype=be)           # [record][variable][level][lat][lon]
    for f in range(5):
        file_buf[:, f] = native[f]
    raws = [file_buf[:, f] for f in range(5)]
    assert not raws[0].flags.c_contiguous
    ident = (np.arange(nlon), np.arange(nlat), np.arange(nlev))
    with H.make_engine(P, fdt, [1.0] * 5) as eng:
        a = eng.run_host(ref, steps)
        b = eng.run_host_raw(raws, *ident, np.arange(nt), steps, decode=decode)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_fill_value_the_records_cannot_hold(tmp_path):
    """int16 records with _FillValue = 40000, which no int16 equals, and stored 32767 values (what 40000 saturates to in
    int16): lec_run_host_raw on the raw-backed dataset has the bits of lec_run_host on what it materialises, where the
    32767 values are values, not missing."""
    nc = str(tmp_path / "era5.nc")
    H.write_era5_unheld_fill(nc, 160)
    ds = PP.open_netcdf3(nc, PP.read_namelist(os.path.join(H.GOLDEN, "inputs", "namelist_ERA5")))
    store = ds.raw.select("lat", slice(None, None, -1)).select("lev", slice(None, None, -1))
    names = list("TUVWZ")
    assert (store.fields["T"] == 32767).any() and not np.isnan(store.materialise("T")).any()
    lat, lon = ds.lat[::-1], ds.lon
    lev = np.asarray(ds.level[::-1], dtype=np.float64) * 100.0
    rl, rp = np.deg2rad(lon), np.deg2rad(lat)
    nt = len(store.rec)
    steps = E.time_stencil(np.arange(nt) * 3600.0, E.make_steps(nt))
    steps["i0"], steps["i1"], steps["j0"], steps["j1"] = 0, 159, 0, 140
    with E.LecEngine(lon, lat, rl, rp, np.cos(rp), lev, np.float64, [1.0] * 5, max_steps=nt) as eng:
        a = eng.run_host([np.ascontiguousarray(store.materialise(v)) for v in names], steps)
        b = eng.run_host_raw([store.fields[v] for v in names], store.lon, store.lat, store.lev, store.rec, steps,
                             decode=[store.decode[v] for v in names])
    H.same_bits(a, b)


def test_raw_records_in_staged_chunks():
    """Several staged chunks (small windows): the two raw staging buffers and the ingest stream are reused
    across chunks and calls; T halo slots come device-to-device from the previous chunk.  Every result has the bits of
    the one-window call, for any step order, records in any order (one serving two slots), windows that split the
    pass mid-way, and a reused handle whose maps change; the H2D bytes are those of the slots the chunks stage."""
    rng = np.random.default_rng(15)
    P, fields = _dataset(40, 17, 6, 13, np.float32)
    steps = H.fixed_steps(P, P.lon[1], P.lon[37], P.lat[1], P.lat[15])
    raws, lon_map, lat_map, lev_map = _raw_layout(rng, fields, extra_levels=0)
    slot_bytes = fields[0][0].nbytes
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        a = eng.run_host(fields, steps)
    with H.make_engine(P, np.float32, [1.0] * 5, max_steps=3) as eng:
        for _ in range(2):
            b = eng.run_host_raw(raws, lon_map, lat_map, lev_map, np.arange(13), steps)
            assert eng.last_transfer()[0] == 5 * 13 * slot_bytes
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
        c = eng.run_host(fields, steps)                    # the two host paths share the staging buffers
        assert np.array_equal(a[0], c[0])
    with H.make_engine(P, np.float32, [1.0] * 5, host_stage_bytes=2 * 5 * 4 * slot_bytes) as eng:
        d = eng.run_host_raw(raws, lon_map, lat_map, lev_map, np.arange(13), steps[::-1].copy())   # steps in reverse order
        assert np.array_equal(d[0], a[0][::-1]) and np.array_equal(d[1], a[1][::-1])

    def same(b, ref, idx, what):
        for x, y in zip(ref, b):
            assert np.array_equal(x[idx], y), what

    def h2d(st, window, nk, nj):           # T at every slot that crosses PCIe, the other four at the centre slots
        t_slots, c_slots, _ = H.staged_slots(st, window, 64)
        return (t_slots + 4 * c_slots) * nk * nj * 40 * 4

    # Step lists shuffled, reversed and with repeats, through 3-slot windows and 8-slot ones (in order, the pass splits
    # after 7 steps and the second window starts inside the first, at a later slot: its first T slots come device to
    # device from the other buffer)
    lists = {"in order": np.arange(13), "shuffled": rng.permutation(13), "reversed": np.arange(13)[::-1],
             "repeats": np.r_[np.arange(13), [5, 5, 0, 12, 6]]}
    for w in (3, 8):
        assert H.staged_slots(steps, w, 64)[2]
        with H.make_engine(P, np.float32, [1.0] * 5, host_stage_bytes=2 * 5 * w * slot_bytes) as eng:
            for name, idx in lists.items():
                st = steps[idx].copy()
                same(eng.run_host_raw(raws, lon_map, lat_map, lev_map, np.arange(13), st), a, idx, (w, name))
                assert eng.last_transfer()[0] == h2d(st, w, 6, 17), (w, name)

    # Records in another order, one of them serving slots 4 and 9
    fields2 = [f.copy() for f in fields]
    for f in fields2:
        f[9] = f[4]
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        a2 = eng.run_host(fields2, steps)
    slot_record = np.empty(13, dtype=np.int32)
    slot_record[np.arange(13) != 9] = rng.permutation(12)
    slot_record[9] = slot_record[4]
    raws2 = [np.empty((12,) + r.shape[1:], dtype=r.dtype) for r in raws]
    keep = np.arange(13) != 9
    for r2, r in zip(raws2, raws):
        r2[slot_record[keep]] = r[keep]
    with H.make_engine(P, np.float32, [1.0] * 5, host_stage_bytes=2 * 5 * 3 * slot_bytes) as eng:
        same(eng.run_host_raw(raws2, lon_map, lat_map, lev_map, slot_record, steps), a2, slice(None), "slot_record")

    # One handle, three layouts of the same fields: a wider raw level range and a row sub-range (the raw staging
    # buffers grow; 3-D copies), then other longitude maps (the device copy of the maps is replaced)
    def place(lon_m, lat_m, lev_m, nlev_r, nlat_r):
        out = []
        for f in fields:
            r = (rng.normal(size=(13, nlev_r, nlat_r, 40)) * 1e3).astype(np.float32)
            r[np.ix_(np.arange(13), lev_m, lat_m, lon_m)] = f
            out.append(r)
        return out
    lev_b, lat_b, lon_c = np.array([7, 0, 5, 2, 3, 6]), 1 + lat_map, (np.arange(40) + 18) % 40
    layouts = [(raws, (lon_map, lat_map, lev_map), 6), (place(lon_map, lat_b, lev_b, 9, 19), (lon_map, lat_b, lev_b), 8),
               (place(lon_c, lat_b, lev_b, 9, 19), (lon_c, lat_b, lev_b), 8)]
    with H.make_engine(P, np.float32, [1.0] * 5, host_stage_bytes=2 * 5 * 3 * slot_bytes) as eng:
        for n, (raws_, maps, nk) in enumerate(layouts):
            same(eng.run_host_raw(raws_, *maps, np.arange(13), steps), a, slice(None), f"layout {n}")
            assert eng.last_transfer()[0] == h2d(steps, 3, nk, 17), n


def test_raw_errors():
    P, fields = _dataset(24, 11, 4, 3, np.float32)
    steps = H.fixed_steps(P, P.lon[1], P.lon[20], P.lat[1], P.lat[9])
    ident = (np.arange(24), np.arange(11), np.arange(4))
    with H.make_engine(P, np.float32, [1.0] * 5) as eng:
        with pytest.raises(IndexError):
            eng.run_host_raw(fields, np.arange(24) + 1, ident[1], ident[2], np.arange(3), steps)
        with pytest.raises(IndexError):
            eng.run_host_raw(fields, *ident, [0, 1, 3], steps)
        with pytest.raises(ValueError):
            eng.run_host_raw([f.astype(np.float64) for f in fields], *ident, np.arange(3), steps)
        with pytest.raises(ValueError):
            eng.run_host_raw(fields, ident[0][:-1], ident[1], ident[2], np.arange(3), steps)
        t, _, _ = eng.run_host_raw(fields, *ident, np.arange(3), steps)
        assert np.array_equal(t, eng.run_host(fields, steps)[0])
        with pytest.raises(ValueError, match=r"invalid argument \(at most two fill values per field\)"):
            eng.run_host_raw(fields, *ident, np.arange(3), steps, decode=[dict(fills=[1.0, 2.0, 3.0])] + [{}] * 4)
        packed = [np.zeros(f.shape, dtype=np.int16) for f in fields]
        scaled = [dict(scale=np.float64(0.01), float32=True)] * 5
        with pytest.raises(ValueError, match=r"invalid argument \(a fill value is not an int16 value\)"):
            eng.run_host_raw(packed, *ident, np.arange(3), steps, decode=[dict(scaled[0], fills=[40000.0])] + scaled[1:])
