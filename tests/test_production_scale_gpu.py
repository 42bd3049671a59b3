"""The row kernels at the scale bench.py measures them, and with time neighbours 2^31 elements apart.

The inputs come from bench.py's own constants and generators (``NLON``, ``NLAT``, ``BOX``, ``BOX_ROWS``, ``C5_HALF``,
``C5_NLEV``; ``synthetic.era5_grid`` / ``synth_fields`` with the bench's ``t0``), so these tests check the configuration
that is timed: the 48-step fp32 and the 24-step fp64 C4 chunk, 64 int16-packed C4 steps (66 slots, more than 2^31
elements per field) and the 270-step C5 track segment in one call.

Reference of every step: the bits of the same step run alone on a fresh handle over a 3-slot copy
``[T(slot_m), T(slot), T(slot_p)]`` (u, v, omega, Phi at the centre slot, NaN in the two slots no kernel may read),
under the same row-kernel instance (``last_dispatch``).  A step's row records depend only on its box, the values of
its slots and the instance -- not on the block order, the batch size or where the slots lie in the buffer -- so a
difference is a wrong address, a wrong slot or state leaking between steps.  Where stated, steps also meet the fp64
oracle at the gates of DESIGN.md section 5 in all 16 terms, 19 per-level families and 18 per-level boundary pieces.

Each test reads the free device memory first and skips, naming both numbers, when it is short of what the test needs
(the GPU may be shared); every large tensor is released before the next test."""
import gc
import time

import numpy as np
import pytest

import bench
from oracle import lec_oracle as O
from lorenzcycletoolkit_b200 import engine as E, synthetic as S
import helpers as H

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

GIB = 1 << 30
C4_SLOT = bench.NLEV * bench.NLAT * bench.NLON        # elements of one C4 time slot (the kernels' slot stride)
T0 = np.datetime64("2020-01-01T00")
DISPATCH_KEYS = ("kernel", "vec", "group", "lonw", "comp", "math64", "tile_rows", "packed")
ROW_KEYS = ("kernel", "vec", "group", "lonw", "comp", "math64")   # int16 fields vs their decoded values: ring shapes differ
ARITH = {"f32": (np.float32, E.LEC_MATH_AUTO), "m64": (np.float32, E.LEC_MATH_F64), "f64": (np.float64, E.LEC_MATH_AUTO)}
PACKING = [dict(offset=True, float32=False, nfill=1)] * 5     # ERA5's: scale_factor, add_offset, one _FillValue


@pytest.fixture(autouse=True)
def _default_dispatcher_and_report(monkeypatch, request):
    for k in ("LEC_ROW_KERNEL", "LEC_NARROW", "LEC_NARROW_G", "LEC_COMP"):
        monkeypatch.delenv(k, raising=False)
    cuda = torch.cuda.is_available()
    if cuda:
        torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    yield
    gc.collect()
    if cuda:
        torch.cuda.empty_cache()
        print(f"\n{request.node.name}: {time.perf_counter() - t0:.1f} s, peak of torch's device allocations "
              f"{torch.cuda.max_memory_allocated() / GIB:.1f} GiB")


def _need(nbytes):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / GIB:.1f} GiB of free device memory, {free / GIB:.1f} GiB are free")


def _c4_grid():
    return S.era5_grid(bench.NLON, bench.NLAT)


def _engine(grid, arith, max_steps, max_box_rows):
    dtype, math = ARITH[arith]
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    return E.LecEngine(f64(grid["lon"]), f64(grid["lat"]), f64(grid["rlons"]), f64(grid["rlats"]), f64(grid["coslats"]),
                       grid["level"], dtype, max_steps=max_steps, max_box_rows=max_box_rows, math=math)


def _run(eng, fields, steps, decode=None):
    """(terms, levels, flags, pieces [n][6][3][nlev]) of run_torch, or of run_torch_packed with ``decode``."""
    if decode is None:
        fn = lambda: eng.run_torch(list(fields), steps)
    else:
        fn = lambda: eng.run_torch_packed(list(fields), decode, steps)
    t, lv, f, b = H.with_boundary(eng, len(steps), fn)
    return t, lv, f, b.reshape(len(steps), 6, 3, eng.nlev)


def _bench_steps(nslots, box):
    """bench.py's steps: the hourly np.gradient stencil of ``nslots`` slots without the two halo slots."""
    steps = E.time_stencil(3600.0 * np.arange(nslots), E.make_steps(nslots))[1:-1].copy()
    steps["i0"], steps["i1"], steps["j0"], steps["j1"] = box
    return steps


BENCH_BOX = (bench.BOX["i0"], bench.BOX["i1"], bench.BOX["j0"], bench.BOX["j1"])


# ---------------------------------------------------------------------------------------------------------------- #
# solo runs and the oracle on a 3-slot copy
def _solo_env(d):
    """Dispatcher switches that make a one-step batch take the instance ``d`` (a misaligned base, which selects the
    scalar direct kernel, is carried by the copy itself)."""
    env = {"LEC_COMP": "1" if d["comp"] else "0"}
    if d["kernel"] == "subwarp":
        env["LEC_NARROW_G"] = str(d["group"])
    else:
        env["LEC_NARROW"] = "0"
        env["LEC_ROW_KERNEL"] = "tile" if d["kernel"] == "tiled" else "direct"
    return env


def _three_slots(fields, step, decode=None, arith=None, misaligned=False):
    """The slots one step reads, copied: T at (slot_m, slot, slot_p), u, v, omega, Phi at slot between two NaN slots
    (int16 fields decoded by ``helpers.decode``'s rule); and the step renumbered onto them."""
    sl = [int(step["slot_m"]), int(step["slot"]), int(step["slot_p"])]
    out = []
    for f, a in enumerate(fields):
        src = a[sl] if f == 0 else a[sl[1]:sl[1] + 1]
        if decode is not None:
            src = H.decode(src, decode[f], ARITH[arith][0])
        shape = (3,) + tuple(src.shape[1:])
        x = torch.empty(int(np.prod(shape)) + int(misaligned), dtype=src.dtype, device=src.device)[int(misaligned):]
        x = x.view(shape)
        if f == 0:
            x.copy_(src)
        else:
            x.fill_(float("nan"))
            x[1].copy_(src[0])
        out.append(x)
    st = np.array([step]).copy()
    st["slot_m"], st["slot"], st["slot_p"] = 0, 1, 2
    return out, st


def _check_solo(out, d, grid, arith, max_box_rows, fields, steps, monkeypatch, only=None, decode=None,
                misaligned=False, keys=DISPATCH_KEYS):
    """Every step of ``out`` (or those in ``only``) has the bits of its solo run under the instance ``d``; with
    ``decode``, the solo runs read the decoded values of the int16 ``fields``."""
    with monkeypatch.context() as m:
        for k, v in _solo_env(d).items():
            m.setenv(k, v)
        for n in range(len(steps)) if only is None else only:
            three, st = _three_slots(fields, steps[n], decode, arith, misaligned)
            with _engine(grid, arith, 1, max_box_rows) as eng:
                solo = _run(eng, three, st)
                ds = eng.last_dispatch()
            del three
            assert {k: ds[k] for k in keys} == {k: d[k] for k in keys}, (n, ds, d)
            try:
                H.same_bits([x[n:n + 1] for x in out], solo)
            except AssertionError:
                raise AssertionError(f"step {n} (slots {steps['slot_m'][n]}, {steps['slot'][n]}, {steps['slot_p'][n]}) "
                                     f"does not have the bits of its solo run") from None


def _oracle(grid, fields, step):
    """The fp64 oracle of one interior hourly step on the crop of its box and 3 slots (the box is the whole crop, as
    the reference slices it)."""
    i0, i1, j0, j1 = (int(step[k]) for k in ("i0", "i1", "j0", "j1"))
    sl = [int(step["slot_m"]), int(step["slot"]), int(step["slot_p"])]
    assert sl[0] == sl[1] - 1 and sl[2] == sl[1] + 1
    host = [f[sl][:, :, j0:j1 + 1, i0:i1 + 1].cpu().numpy() for f in fields]
    P = H.prepared_from_arrays(host, grid["lon"][i0:i1 + 1], grid["lat"][j0:j1 + 1], grid["level"],
                               T0 + np.arange(3) * np.timedelta64(1, "h"))
    del host
    Q = O.to_mode(P, "fp64")
    dTdt = O.differentiate(Q.fields["Air Temperature"], H.tsec_of(Q), 0)
    return H.oracle_step(Q, (0, i1 - i0, 0, j1 - j0), 1, dTdt)


def _check_oracle(out, n, ref, tol):
    worst = H.check_refs(tuple(x[n:n + 1] for x in out), [ref], tol)
    print(f"step {n} against the oracle: worst of 53 outputs {worst:.2e} (gate {tol:g})")


# ---------------------------------------------------------------------------------------------------------------- #
# 1. far time neighbours
FAR = 56                 # real slots 0, FAR - 1 and FAR of a 57-slot C4 buffer; the slots between hold a constant
FAR_INSTANCES = {        # name -> (dispatcher switches, base one element off, int16 fields, (kernel, group))
    "direct": ({"LEC_ROW_KERNEL": "direct", "LEC_NARROW": "0"}, False, False, ("direct", 32)),
    "scalar": ({"LEC_ROW_KERNEL": "direct", "LEC_NARROW": "0"}, True, False, ("direct", 32)),
    "g4": ({"LEC_NARROW_G": "4"}, False, False, ("subwarp", 4)),
    "g8": ({"LEC_NARROW_G": "8"}, False, False, ("subwarp", 8)),
    "g16": ({"LEC_NARROW_G": "16"}, False, False, ("subwarp", 16)),
    "tiled": ({"LEC_NARROW": "0"}, False, False, ("tiled", 32)),
    "i16_g8": ({"LEC_NARROW_G": "8"}, False, True, ("subwarp", 8)),
    "i16_tiled": ({"LEC_NARROW": "0"}, False, True, ("tiled", 32)),
}


def _far_step(slots, it):
    """The step at position ``it`` of an hourly axis of the buffer slots ``slots``: time_stencil's coefficients, slot
    numbers of the buffer."""
    st = E.time_stencil(3600.0 * np.asarray(slots, dtype=np.float64), E.make_steps(len(slots)))[it:it + 1].copy()
    for k in ("slot", "slot_m", "slot_p"):
        st[k] = np.asarray(slots)[st[k]]
    st["i0"], st["i1"], st["j0"], st["j1"] = BENCH_BOX
    return st


def test_far_neighbour_offsets_do_not_fit_32_bits():
    """Why the far-neighbour cases exist: T(slot_m) of a step FAR slots after it lies FAR * 38,414,880 elements away,
    past 2^31; taken as a 32-bit offset it would wrap to +2,143,734,016, i.e. about 2.14 G elements past T(slot) and
    outside the 57-slot buffer.  FAR - 1 slots is the largest distance a 32-bit offset can hold."""
    assert C4_SLOT == 38_414_880
    assert (FAR - 1) * C4_SLOT < 2 ** 31 <= FAR * C4_SLOT
    assert (-FAR * C4_SLOT + 2 ** 31) % 2 ** 32 - 2 ** 31 == 2_143_734_016


@pytest.mark.parametrize("arith", ["f32", "m64", "f64"])
@pytest.mark.parametrize("inst", list(FAR_INSTANCES))
def test_far_time_neighbours(inst, arith, monkeypatch):
    """One C4 buffer passed as all five fields (read-only aliasing): slots 0, 55 and 56 hold synthetic T, the others
    a constant, so a wrong slot gives other bits.  Steps whose neighbours lie 55 slots away (offsets just below
    2^31 elements) have the bits of their solo runs in every instance.  Steps whose neighbours lie 56 slots away
    have them in the tiled kernel, which addresses slots as TMA coordinates; the direct and sub-warp kernels, which
    address them as 32-bit element offsets, refuse the batch with LEC_ERR_INVALID and never return wrong bits."""
    env, misaligned, packed, (kernel, group) = FAR_INSTANCES[inst]
    dtype = ARITH[arith][0]
    esz = 2 if packed else np.dtype(dtype).itemsize
    _need((FAR + 1) * C4_SLOT * esz + 15 * C4_SLOT * np.dtype(dtype).itemsize + 3 * GIB)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    grid = _c4_grid()
    real = torch.cat([S.synth_fields(grid, 1, np.float32, "cuda:0", t0=t)[0] for t in (0, FAR - 1, FAR)])
    if packed:
        raws, dec = H.encode([real], PACKING[:1])
        decode, real = [dec[0]] * 5, raws[0]
        buf = torch.zeros((FAR + 1,) + tuple(real.shape[1:]), dtype=torch.int16, device="cuda:0")
    else:
        decode, real = None, real.to(torch.float64 if dtype == np.float64 else torch.float32)
        n = (FAR + 1) * C4_SLOT
        buf = torch.empty(n + int(misaligned), dtype=real.dtype, device="cuda:0")[int(misaligned):]
        buf = buf.view((FAR + 1,) + tuple(real.shape[1:])).fill_(250.0)
        assert (buf.data_ptr() % 16 != 0) == misaligned
    buf[[0, FAR - 1, FAR]] = real
    del real
    fields = [buf] * 5
    near = np.concatenate([_far_step([0, FAR - 1, FAR], 1), _far_step([0, FAR - 1], 0)])   # 55 slots away
    far = np.concatenate([_far_step([0, FAR], 1), _far_step([0, FAR], 0)])                  # 56 slots away
    assert list(far["slot"]) == [FAR, 0] and list(far["slot_m"]) == [0, 0] and list(far["slot_p"]) == [FAR, FAR]
    with _engine(grid, arith, 2, bench.BOX_ROWS) as eng:
        out = _run(eng, fields, near, decode)
        d = eng.last_dispatch()
        assert (d["kernel"], d["group"], d["vec"] == 1, d["packed"]) == (kernel, group, misaligned, packed), d
        assert not out[2].any()
        _check_solo(out, d, grid, arith, bench.BOX_ROWS, fields, near, monkeypatch, decode=decode,
                    misaligned=misaligned, keys=ROW_KEYS if packed else DISPATCH_KEYS)
        if kernel == "tiled":
            out = _run(eng, fields, far, decode)
            assert eng.last_dispatch() == d
        else:
            with pytest.raises(ValueError, match="2\\^31 or more elements from slot"):
                _run(eng, fields, far, decode)
            return
    _check_solo(out, d, grid, arith, bench.BOX_ROWS, fields, far, monkeypatch, decode=decode,
                keys=ROW_KEYS if packed else DISPATCH_KEYS)


# ---------------------------------------------------------------------------------------------------------------- #
# 2. the C4 bench chunk, fp32 and fp64
@pytest.mark.parametrize("arith", ["f32", "f64"])
def test_c4_bench_chunk(arith, monkeypatch):
    """run_b200's chunk (48 steps, 50 slots, fp32) and bench_fp64's (24 steps, 26 slots: the fp32 fields' first slots
    upcast), built as bench.py builds them, in the latitude-banded block order the engine chooses for them: every
    step has the bits of its solo run.  The fp32 chunk's last step (slot 48, next to the highest addresses) also
    meets the oracle at 1e-5."""
    chunk = 48 if arith == "f32" else 24          # bench.py's --chunk and --fp64-chunk defaults
    nslots = chunk + 2
    esz = np.dtype(ARITH[arith][0]).itemsize
    _need(5 * nslots * C4_SLOT * esz + 15 * C4_SLOT * esz + 4 * GIB)
    grid = _c4_grid()
    fields = S.synth_fields(grid, nslots, np.float32, "cuda:0", t0=0)
    if arith == "f64":
        for f in range(5):
            fields[f] = fields[f].double()
            torch.cuda.empty_cache()
    steps = _bench_steps(nslots, BENCH_BOX)
    with _engine(grid, arith, chunk, bench.BOX_ROWS) as eng:
        out = _run(eng, fields, steps)
        d = eng.last_dispatch()
    assert d["kernel"] == "tiled" and d["nbands"] > 1, d
    assert not out[2].any()
    _check_solo(out, d, grid, arith, bench.BOX_ROWS, fields, steps, monkeypatch)
    if arith == "f32":
        _check_oracle(out, chunk - 1, _oracle(grid, fields, steps[chunk - 1]), 1e-5)
    del fields


# ---------------------------------------------------------------------------------------------------------------- #
# 3. int16 residency past 2^31 elements per field
NARROW_BOX = (601, 751, 300, 450)       # 151 x 151 on the C4 grid: the sub-warp kernel


@pytest.mark.parametrize("arith", ["f32", "f64"])
def test_int16_c4_residency_past_2_31_elements(arith, monkeypatch):
    """64 resident int16 C4 steps (66 slots, 2.5 G elements and 5 GB per field), encoded by ``helpers.encode`` with
    scale and offset from each field's extremes over all slots, rows at ``packed_device_fields``'s pitch.  The full
    bench box (tiled kernel) and a 151 x 151 box (sub-warp kernel), 64 steps per call: every step has the bits of
    its solo run on the decoded fields."""
    nsteps = 64
    nslots = nsteps + 2
    assert nslots * C4_SLOT > 2 ** 31
    pitch = (bench.NLON + 7) // 8 * 8
    slot16 = bench.NLEV * bench.NLAT * pitch
    esz = np.dtype(ARITH[arith][0]).itemsize
    _need(5 * nslots * slot16 * 2 + 15 * C4_SLOT * (esz + 2) + 4 * GIB)
    grid = _c4_grid()
    one = None
    lo, hi = [None] * 5, [None] * 5
    for s in range(nslots):                 # pass 1: each field's extremes over the slots
        one = S.synth_fields(grid, 1, np.float32, "cuda:0", t0=s, out=one)
        for f in range(5):
            a, b = one[f].min(), one[f].max()
            lo[f] = a if lo[f] is None else torch.minimum(lo[f], a)
            hi[f] = b if hi[f] is None else torch.maximum(hi[f], b)
    bounds = [(float(a), float(b)) for a, b in zip(lo, hi)]
    packed = [torch.full((nslots, bench.NLEV, bench.NLAT, pitch), H.FILL, dtype=torch.int16, device="cuda:0")
              for _ in range(5)]
    for s in range(nslots):                 # pass 2: the same slots again, encoded
        one = S.synth_fields(grid, 1, np.float32, "cuda:0", t0=s, out=one)
        raws, decode = H.encode([x[0] for x in one], PACKING, bounds=bounds)
        for f in range(5):
            packed[f][s, :, :, :bench.NLON].copy_(raws[f])
        if s == 0:                          # the device encode and decode are numpy's, bit for bit (T of slot 0)
            host = one[0][0].cpu().numpy()
            raw_np, dec_np = H.encode([host], PACKING[:1], bounds=bounds[:1])
            assert dec_np[0] == decode[0] and np.array_equal(raw_np[0], raws[0].cpu().numpy())
            assert np.array_equal(H.decode(raw_np[0], dec_np[0], ARITH[arith][0]).view(np.uint8),
                                  H.decode(raws[0], decode[0], ARITH[arith][0]).cpu().numpy().view(np.uint8))
            del host, raw_np
    del one, raws
    fields = [p[..., :bench.NLON] for p in packed]
    with _engine(grid, arith, nsteps, bench.BOX_ROWS) as eng:
        for box, kernel in ((BENCH_BOX, "tiled"), (NARROW_BOX, "subwarp")):
            steps = _bench_steps(nslots, box)
            out = _run(eng, fields, steps, decode)
            d = eng.last_dispatch()
            assert d["kernel"] == kernel and d["packed"], d
            assert not out[2].any()
            _check_solo(out, d, grid, arith, bench.BOX_ROWS, fields, steps, monkeypatch, decode=decode, keys=ROW_KEYS)
    del fields, packed


# ---------------------------------------------------------------------------------------------------------------- #
# 4. the C5 bench line
def _c5_inputs(n):
    """bench_c5's domain, fields and steps for rank 0: ``n`` moving 151 x 151 x 55 boxes over ``n + 2`` slots."""
    half = bench.C5_HALF
    side = 2 * half + 1
    nlon = (n + side + 12 + 3) // 4 * 4
    nlat = n // 2 + side + 12
    lon = (-150.0 + 0.1 * np.arange(nlon)).astype(np.float32)
    lat = (-60.0 + 0.1 * np.arange(nlat)).astype(np.float32)
    lev = np.linspace(1000.0, 100000.0, bench.C5_NLEV)
    grid = dict(lon=lon, lat=lat, level=lev, rlons=np.deg2rad(lon), rlats=np.deg2rad(lat), coslats=np.cos(np.deg2rad(lat)))
    fields = S.synth_fields(grid, n + 2, np.float32, "cuda:0", t0=0)
    steps = E.time_stencil(3600.0 * np.arange(n + 2), E.make_steps(n + 2))[1:-1].copy()
    ci = half + 5 + np.arange(n)
    cj = half + 5 + np.arange(n) // 2
    steps["i0"], steps["i1"], steps["j0"], steps["j1"] = ci - half, ci + half, cj - half, cj + half
    return grid, fields, steps


C5_STEPS = 270            # bench.py's --c5-steps default


def test_c5_bench_line(monkeypatch):
    """bench_c5's call: 270 moving 151 x 151 x 55 boxes over 272 slots of a 436 x 298 x 55 domain (1.94 G elements per
    field) in one call.  Every step has the bits of its solo run; the first, a middle and the last step and one whose
    box starts at column 3 mod 4 (the last column of a chunk) meet the oracle at 1e-5."""
    side = 2 * bench.C5_HALF + 1
    nlon = (C5_STEPS + side + 12 + 3) // 4 * 4
    nlat = C5_STEPS // 2 + side + 12
    _need(5 * (C5_STEPS + 2) * bench.C5_NLEV * nlat * nlon * 4 + 4 * GIB)
    grid, fields, steps = _c5_inputs(C5_STEPS)
    assert (len(grid["lon"]), len(grid["lat"]), fields[0].numel()) == (436, 298, 272 * 55 * 298 * 436)
    with _engine(grid, "f32", C5_STEPS, side) as eng:
        out = _run(eng, fields, steps)
        d = eng.last_dispatch()
    assert d["kernel"] == "subwarp" and d["group"] == 8, d
    assert not out[2].any()
    _check_solo(out, d, grid, "f32", side, fields, steps, monkeypatch)
    odd = int(np.flatnonzero(steps["i0"] % 4 == 3)[0])
    for n in sorted({0, odd, C5_STEPS // 2, C5_STEPS - 1}):
        _check_oracle(out, n, _oracle(grid, fields, steps[n]), 1e-5)
    del fields
