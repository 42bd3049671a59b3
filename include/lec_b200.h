/*
 * lec_b200.h -- C ABI of the B200-native Lorenz Energy Cycle engine.
 *
 * The reference (daniloceano/LorenzCycleToolkit v1.1.11) is pure Python and has
 * no FFI layer; the boundary that this library replaces is the arithmetic of
 *
 *   src/utils/box_data.py:78-310        BoxData (box slice, ZA/AA/ZE/AE, sigma, Q)
 *   src/utils/calc_averages.py:25-78    CalcZonalAverage / CalcAreaAverage
 *   src/utils/thermodynamics.py:26-124  StaticStability / AdiabaticHEating
 *   src/analysis/energy_contents.py:99-165              Az Ae Kz Ke
 *   src/analysis/conversion_terms.py:103-245            Cz Ca Ck Ce (+15 per-level families)
 *   src/analysis/boundary_terms.py:122-418              BAz BAe BKz BKe BPhiZ BPhiE
 *   src/analysis/generation_and_dissipation_terms.py:122-152   Gz Ge
 *   src/frameworks/lec_fixed_framework.py:199-279       (one BoxData for all times)
 *   src/frameworks/lec_moving_framework.py:639-740      (one BoxData per time step)
 *
 * i.e. everything between "a preprocessed [time][level][lat][lon] dataset in
 * memory" and "per-time-step scalars + per-level rows".  One lec_run_* call
 * evaluates all terms for a batch of time steps, each with its own box.
 *
 * Conventions: plain pointers and sizes; the caller owns every buffer it
 * passes; the engine owns its scratch; every function returns 0 (LEC_OK) or a
 * negative error code and never throws; lec_run_device is asynchronous on the
 * given CUDA stream, lec_run_host returns after the results are in host memory.
 * One handle per thread AND per stream: the engine's scratch (row records, finalize
 * buffers, timing events) is single-buffered per handle, so a handle must not have two
 * lec_run_* calls in flight on different streams (use one handle per stream; handles are
 * independent).  There is no CPU fallback: without a CUDA device lec_create fails with
 * LEC_ERR_CUDA.
 */
#ifndef LEC_B200_H
#define LEC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LEC_OK               0
#define LEC_ERR_INVALID     -1   /* bad argument                                              */
#define LEC_ERR_CUDA        -2   /* CUDA runtime failure (see lec_last_error)                  */
#define LEC_ERR_DEGENERATE  -3   /* an axis of the box has < 2 points (np.gradient would raise)*/
#define LEC_ERR_BOUNDS      -4   /* box or time slot outside the prepared domain               */
#define LEC_ERR_NOMEM       -5

#define LEC_F32 0
#define LEC_F64 1

/* Arithmetic of the row-moment kernel (lec_grid_desc.math). */
#define LEC_MATH_AUTO 0   /* storage type: fp32 pointwise + fp64 reductions for fp32 fields */
#define LEC_MATH_F64  1   /* fp64 pointwise arithmetic whatever the storage type            */

/* Field order of every `fields[5]` argument. */
#define LEC_FIELD_T      0   /* air temperature                 [K]        */
#define LEC_FIELD_U      1   /* eastward wind                   [m/s]      */
#define LEC_FIELD_V      2   /* northward wind                  [m/s]      */
#define LEC_FIELD_OMEGA  3   /* pressure vertical velocity      [Pa/s]     */
#define LEC_FIELD_PHI    4   /* geopotential (or height*scale)  [m^2/s^2]  */

/* Per-step scalar outputs, out_terms[step][LEC_NTERMS] (lec_moving column order,
 * lec_moving_framework.py:45-55; lec_fixed drops the two B-Phi columns). */
#define LEC_NTERMS 16
enum lec_term {
  LEC_AZ = 0, LEC_AE, LEC_KZ, LEC_KE, LEC_CZ, LEC_CA, LEC_CK, LEC_CE,
  LEC_BAZ, LEC_BAE, LEC_BKZ, LEC_BKE, LEC_BPHIZ, LEC_BPHIE, LEC_GZ, LEC_GE
};

/* Per-level outputs, out_levels[step][LEC_NLEVEL_TERMS][nlev]: the integrands the
 * reference writes with _save_vertical_levels (energy_contents.py:210,
 * conversion_terms.py:287, generation_and_dissipation_terms.py:230).  Cz_1/Ce_1
 * (= Rd/(p g)) depend on pressure only and are left to the host. */
#define LEC_NLEVEL_TERMS 19
enum lec_level_term {
  LEC_LV_AZ = 0, LEC_LV_AE, LEC_LV_KZ, LEC_LV_KE, LEC_LV_GE, LEC_LV_GZ,
  LEC_LV_CZ, LEC_LV_CZ_2, LEC_LV_CA, LEC_LV_CA_1, LEC_LV_CA_2,
  LEC_LV_CE, LEC_LV_CE_2, LEC_LV_CK, LEC_LV_CK_1, LEC_LV_CK_2,
  LEC_LV_CK_3, LEC_LV_CK_4, LEC_LV_CK_5
};

/* out_flags[step] bits */
#define LEC_FLAG_NONFINITE   1   /* a per-level integrand is NaN/Inf (reference _handle_nans path) */
#define LEC_FLAG_SIGMA_FLOOR 2   /* sigma <= 0.03 (or NaN) replaced by 0.03 (thermodynamics.py:69)  */

/*
 * The prepared domain (output of preprocessing.py:149-371 + select_area.py:254-338):
 * C-contiguous [time][level ascending Pa][lat ascending][lon ascending].
 * Coordinates are the STORED-dtype values upcast to double (rlat/rlon/coslat as
 * computed by np.deg2rad / np.cos in the coordinate dtype, preprocessing.py:288-290).
 */
typedef struct lec_grid_desc {
  int32_t nlon, nlat, nlev;
  const double *lon_deg;      /* [nlon] */
  const double *lat_deg;      /* [nlat] */
  const double *rlon;         /* [nlon] */
  const double *rlat;         /* [nlat] */
  const double *coslat;       /* [nlat] */
  const double *plev;         /* [nlev], Pa */
  int32_t dtype;              /* LEC_F32 | LEC_F64: element type of the field buffers */
  int32_t math;               /* LEC_MATH_AUTO | LEC_MATH_F64 */
  double field_scale[5];      /* namelist-unit -> SI factor per field (box_data.py:297-310;
                                 g for geopotential height, :233-241) */
  int32_t max_steps;          /* scratch is sized for this many steps per kernel batch; longer
                                 runs are split into batches internally */
  int32_t max_box_rows;       /* largest box height in rows (0 = nlat) */
  int32_t device;             /* CUDA device ordinal */
  int32_t band_rows;          /* latitude rows per L2 band of the fixed-box sweep; 0 = auto */
  int64_t host_stage_bytes;   /* device bytes lec_run_host may use for staging; 0 = auto */
} lec_grid_desc;

/*
 * One time step of work.  `slot*` index the time axis of the field buffers.
 * dT/dt (thermodynamics.py:109-110 / lorenzcycletoolkit.py:184-186) is
 *   ct_m * T[slot_m] + ct_0 * T[slot] + ct_p * T[slot_p]
 * with the np.gradient coefficients of the time axis the reference differentiates
 * over (lec_gradient_coefs gives them); this is what lets a time shard carry a
 * one-slot halo.  The box is inclusive index bounds on the prepared grid
 * (box_data.py:115-135 nearest snap; lec_nearest_index reproduces it).
 * slot_m and slot_p may be any slots of the buffer, with one limit: in a kernel
 * batch that runs the direct or the sub-warp row kernel (LEC_ROWS_DIRECT /
 * LEC_ROWS_SUBWARP), |slot_m - slot| and |slot_p - slot| times the elements of
 * one slot (nlev * nlat * row length) must stay below 2^31; such a batch fails
 * with LEC_ERR_INVALID and a lec_last_error text.  The tiled kernel
 * (LEC_ROWS_TILED, wide boxes) has no such limit.
 */
typedef struct lec_step {
  int32_t slot, slot_m, slot_p;
  int32_t i0, i1, j0, j1;
  int32_t reserved;
  double ct_m, ct_0, ct_p;
} lec_step;

typedef struct lec_handle lec_handle;

int lec_create(lec_handle **out, const lec_grid_desc *desc);
int lec_destroy(lec_handle *h);

/* Fields and outputs in DEVICE memory; asynchronous on `stream` (a cudaStream_t
 * passed as void*; NULL = legacy default stream).  `steps` is a host array.
 * out_terms [nsteps][LEC_NTERMS], out_levels [nsteps][LEC_NLEVEL_TERMS][nlev]
 * (may be NULL), out_flags [nsteps] (may be NULL).  nsteps = 0 is not an error: nothing is launched. */
int lec_run_device(lec_handle *h, const void *const fields[5], int32_t nslots,
                   const lec_step *steps, int32_t nsteps,
                   double *out_terms, double *out_levels, int32_t *out_flags,
                   void *stream);

/* Same with HOST buffers: stages the fields to the device in time chunks on two
 * streams (copy of chunk n+1 overlaps compute of chunk n), copies the results
 * back and synchronises.  This is the call the Python drop-ins use. */
int lec_run_host(lec_handle *h, const void *const fields[5], int32_t nslots,
                 const lec_step *steps, int32_t nsteps,
                 double *out_terms, double *out_levels, int32_t *out_flags);

/* Host helpers that restate third-party semantics the reference relies on. */

/* np.gradient(f, x, edge_order=1) as coefficients: out[i] = a[i] f[i-1] + b[i] f[i] + c[i] f[i+1]
 * (uniform branch iff np.diff(x) is exactly constant).  Needs n >= 2. */
int lec_gradient_coefs(const double *x, int32_t n, double *a, double *b, double *c);

/* pandas Index.get_indexer([value], method="nearest") on an increasing index
 * (ties -> larger coordinate), i.e. xarray .sel(method="nearest"). */
int32_t lec_nearest_index(const double *coord, int32_t n, double value);

/* ---- raw-record ingest (SURVEY.md 8(f) rank 2) ------------------------------------------------------
 * lec_run_host for fields still in FILE layout: replaces the host-side decode of get_data
 * (src/utils/preprocessing.py:35-147: scale_factor / add_offset / _FillValue) and the full-dataset
 * re-sorts of process_data (:149-371: longitude wrap + sort, latitude / level sort, levels < 10 hPa
 * dropped, track-time selection) and of slice_domain (src/utils/select_area.py:254-338).  The raw records
 * cross PCIe as stored and a device pass writes the engine layout; results have the bits of lec_run_host
 * on the host-prepared arrays. */
#define LEC_RAW_F32 0
#define LEC_RAW_F64 1
#define LEC_RAW_I16 2

typedef struct lec_raw_desc {
  int32_t dtype;                 /* LEC_RAW_*: element type of the raw records */
  int32_t nlon, nlat, nlev;      /* one raw record is [nlev][nlat][nlon], C order, as stored */
  const int32_t *lon_map;        /* [grid nlon] engine column i <- raw column lon_map[i] */
  const int32_t *lat_map;        /* [grid nlat] engine row j    <- raw row lat_map[j] */
  const int32_t *lev_map;        /* [grid nlev] engine level k  <- raw level lev_map[k] */
  double scale[5], offset[5];    /* packed decode per field: double(raw) * scale (+ offset) */
  int32_t use_scale[5], use_offset[5];
  int32_t round_f32[5];          /* decoded variable is float32 (rounded once), else float64 */
  int32_t nfill[5];              /* 0..2 fill values per field; raw == fill -> NaN */
  double fill[5][2];
  int32_t big_endian;            /* 1: records are big-endian (NetCDF-3 classic), swapped on the device */
  int32_t reserved;
  int64_t record_stride[5];      /* bytes between consecutive records of field f; 0 = contiguous records
                                    (NetCDF-3 interleaves the records of its record variables) */
} lec_raw_desc;

/* raw[f] points at [nrecords] records of field f; slot_record[nslots] names the record of each engine
 * time slot (the track-time selection).  Everything else as lec_run_host.  The handle's dtype must be
 * LEC_F32 for LEC_RAW_F32, LEC_F64 for LEC_RAW_F64, either for LEC_RAW_I16. */
int lec_run_host_raw(lec_handle *h, const lec_raw_desc *raw_desc, const void *const raw[5], int32_t nrecords,
                     const int32_t *slot_record, int32_t nslots, const lec_step *steps, int32_t nsteps,
                     double *out_terms, double *out_levels, int32_t *out_flags);

/* ---- int16-packed fields resident in device memory ----------------------------------------------------
 * lec_run_device for fields stored the way ERA5 and most reanalysis files store them: int16 with a per-field
 * scale_factor / add_offset (2 bytes per value instead of the 4 or 8 of the decoded fields).  The row kernels decode
 * every value they load by the rule of lec_run_host_raw:
 *   x = double(raw);  x = x * scale (use_scale);  x = x + offset (use_offset)  (two roundings, no FMA)
 *   x = double(float(x)) (round_f32);  raw == fill[0] (nfill >= 1) or raw == fill[1] (nfill >= 2) -> NaN
 * and the value is x in the handle's dtype (LEC_F32 / LEC_F64); arithmetic as lec_run_device (desc.math), so the
 * results have the bits of lec_run_device on the decoded fields.  Device data is native-endian.
 * fields[f]: int16 [nslots][nlev][nlat][pitch], C order, 16-byte aligned; the pitch - nlon pad columns are never
 * read into a result.  Everything else (steps, outputs, stream, batches of max_steps, lec_set_boundary_levels,
 * timing, nsteps = 0) as lec_run_device.  LEC_ERR_INVALID for a pitch below nlon or not a multiple of 8, a
 * misaligned field, nfill outside 0..2 or a fill value that is not an int16 value.  The row kernel is the TMA-tiled
 * one for wide boxes and the sub-warp one for narrow boxes whatever LEC_ROW_KERNEL says;
 * lec_last_dispatch reports it with packed = 1. */
typedef struct lec_packed_desc {
  int32_t pitch;                 /* row length of the packed fields in elements: >= nlon, multiple of 8 (16 B) */
  int32_t reserved;
  double scale[5], offset[5];
  int32_t use_scale[5], use_offset[5];
  int32_t round_f32[5];
  int32_t nfill[5];
  double fill[5][2];
} lec_packed_desc;

int lec_run_device_packed(lec_handle *h, const lec_packed_desc *pd, const int16_t *const fields[5], int32_t nslots,
                          const lec_step *steps, int32_t nsteps, double *out_terms, double *out_levels,
                          int32_t *out_flags, void *stream);

/* Optional extra output of every following lec_run_* on this handle: the 18 per-level boundary pieces
 *   out[step][LEC_NBOUNDARY_PIECES][nlev],  piece = 3 * term + part,
 *   term in BAz BAe BKz BKe BPhiZ BPhiE, part 0 = east-minus-west flux integrated over latitude,
 *   1 = north-minus-south flux, 2 = vertical flux,
 * i.e. the (time, level) arrays src/analysis/boundary_terms.py hands to _handle_nans (:142,157,169 and
 * the same three places of each term, :420-438) before `.integrate(level)` / `isel(level=-1) - isel(level=0)`;
 * term = c1 * trapz_p(part 0) + c2 * trapz_p(part 1) - (part 2 at the last level - part 2 at the first),
 * c1 = -1 / (Re xlength ylength), c2 = -1 / (Re ylength) (:122-123).  The host applies the reference's
 * interpolate / drop-level NaN rule to them when out_flags reports LEC_FLAG_NONFINITE.
 * `out` is a DEVICE pointer for lec_run_device and a HOST pointer for lec_run_host*; NULL switches the
 * output off again.  The buffer must hold nsteps * 18 * nlev doubles of the following call. */
#define LEC_NBOUNDARY_PIECES 18
int lec_set_boundary_levels(lec_handle *h, double *out);

/* 1: the following lec_run_host / lec_run_host_raw calls on this handle stage only each slot's window;
 * 0 (default): whole slots.  Results keep their bits; only the bytes staged (lec_last_transfer) change.
 * For a track run, whose prepared domain spans the whole track, the bytes follow the box instead of the domain.
 * The windows of one call, computed once from all its steps:
 *   - window of a slot: the union of the boxes (i0..i1 x j0..j1) of the steps that read it -- for T as centre slot or
 *     time neighbour (slot, slot_m, slot_p), for u, v, omega and Phi as centre slot only.  The row kernels need no
 *     value outside a box (the j-1 / j+1 rows and lon neighbours they use lie inside it), so there is no margin.
 *   - column origin x0: rounded down to a multiple of 4 (LEC_F32) or 2 (LEC_F64) columns, so that the row kernels'
 *     128-bit chunks and summation order are those of the grid.
 *   - a slot is stored as its T window; all slots of the call share one buffer shape (the largest T window, rows
 *     padded to whole 128-bit chunks), so a larger staging window (host_stage_bytes) fits in the same bytes.
 * lec_last_transfer then counts, per (slot, field) that a greedy chunk stages (as without windows: T over the
 * chunk's slot range minus the slots the previous chunk holds, the other four over its centre slot range; slots
 * no step reads are skipped):
 *   lec_run_host      nlev * (y1 - y0 + 1) * (x1 - x0 + 1) elements of the handle's dtype;
 *   lec_run_host_raw  (max - min + 1 of lev_map: the raw level range, untouched levels inside it included)
 *                     * (max - min + 1 of lat_map[y0..y1]) * w raw elements, where w = x1 - x0 + 1 when
 *                     lon_map[x0..x1] is one increasing run of raw columns, else the raw row length: whole raw
 *                     rows, e.g. when a longitude wrap's seam falls inside the window (the whole globe's row for
 *                     a global file, where the two runs either side of the seam would do).
 * LEC_ERR_INVALID unless on is 0 or 1. */
int lec_set_host_windows(lec_handle *h, int32_t on);

/* Page-lock (cudaHostRegister) / release a host range the caller keeps alive, so that the lec_run_host* copies
 * out of it run at the pinned PCIe rate instead of through the driver's pageable staging.  For the record arrays a
 * NetCDF reader returns (the reference's loader, src/utils/preprocessing.py:35-147, hands over pageable numpy
 * memory).  Handle-free; LEC_ERR_CUDA (text: lec_last_error(NULL)) if the range cannot be registered -- the
 * copies then simply stay pageable. */
int lec_pin_host(void *ptr, int64_t bytes);
int lec_unpin_host(void *ptr);

/* Device time of the last lec_run_* on this handle, milliseconds:
 * [0] row-moment kernel(s), [1] finalize kernel(s), [2] whole call incl. copies. */
int lec_last_timing(lec_handle *h, float out_ms[3]);

/* Start accumulating: after this call lec_last_timing returns the SUMS [0], [1] over every
 * lec_run_* since the reset (at most 4096 kernel batches), [2] stays the last call. */
int lec_timing_reset(lec_handle *h);

/* Number of kernel launches issued by this handle so far. */
int64_t lec_launch_count(lec_handle *h);

/* Row-moment kernel that the last kernel batch of the last lec_run_* call on this handle launched (a call
 * with more steps than max_steps runs several batches; each chooses again).  Read-only: it reports what
 * the dispatcher chose and changes nothing.  LEC_ERR_INVALID before the first batch. */
#define LEC_ROWS_DIRECT          0   /* direct loads, one warp per row                                 */
#define LEC_ROWS_SUBWARP         1   /* direct loads, a group of `group` lanes per row (narrow boxes)  */
#define LEC_ROWS_TILED           2   /* TMA ring of tile_rows-row tiles, one warp per row (wide boxes)  */
typedef struct lec_dispatch {
  int32_t kernel;           /* LEC_ROWS_* */
  int32_t vec;              /* elements per lane load: 4 (fp32) / 2 (fp64) on 16-byte aligned rows, 1 scalar */
  int32_t group;            /* lanes per row: 4, 8 or 16 for the sub-warp kernel, else 32 */
  int32_t lonw;             /* longitude tables: 0 uniform, 1 per-column weights, 2 weights and stencil */
  int32_t comp;             /* 1: compensated fp32 linear sums */
  int32_t math64;           /* 1: fp64 pointwise arithmetic (fp64 fields or LEC_MATH_F64) */
  int32_t tile_rows;        /* box rows per tile (tiled kernel), per CTA otherwise */
  int32_t tiles_per_band;   /* tiles per latitude band of the block order */
  int32_t nbands;           /* latitude bands (1: step-major order) */
  int32_t packed;           /* 1: int16 fields decoded by the row kernel (lec_run_device_packed) */
} lec_dispatch;
int lec_last_dispatch(const lec_handle *h, lec_dispatch *out);

/* Bytes the last lec_run_host moved over PCIe: out[0] host->device (fields: T for every slot a step
 * or its time neighbours touch, u/v/omega/Phi for the centre slots only; slots shared by two staged
 * chunks are copied device-to-device and not counted; with lec_set_host_windows, the windows' bytes),
 * out[1] device->host (results). */
int lec_last_transfer(lec_handle *h, int64_t out_bytes[2]);

/* ---- 850-hPa track diagnostics (SURVEY.md 8(f) rank 1) --------------------------------------------
 * Replaces, for a batch of time steps, the per-step wind_speed / vorticity of the moving framework
 * (src/frameworks/lec_moving_framework.py:650-663), the box extrema of get_position (:269-417, incl. the
 * vorticity at the track centre of the -z branch, :317-324) and the arg-reductions of
 * find_extremum_coordinates (src/utils/tools.py:95-128).  Handle-free: the planes are the 850-hPa level of
 * u, v and geopotential (height), [slot][lat][lon], dtype LEC_F32 / LEC_F64.
 * Vorticity is MetPy 1.6.2's `vorticity` on a latitude / longitude grid: "nominal" grid deltas dx (on the
 * equator) and dy (meridian arcs), the map factors parallel_scale / meridional_scale of the ellipsoid, and
 * MetPy's 3-point `first_derivative` over the DOMAIN axes; evaluated in fp64 in numpy's operation order. */
typedef struct lec_diag_step {
  int32_t slot;            /* time slot of the planes */
  int32_t i0, i1, j0, j1;  /* label-sliced box, inclusive domain indices */
  int32_t ic, jc;          /* domain indices of the grid point nearest to the track centre; -1 = none */
  int32_t reserved;
} lec_diag_step;

typedef struct lec_diag_grid {
  int32_t nlon, nlat, dtype, device;
  const double *dx;               /* [nlon-1] nominal zonal grid deltas, metres  (a * diff(lon in radians)) */
  const double *dy;               /* [nlat-1] meridional grid deltas, metres (signed meridian arcs) */
  const double *parallel_scale;   /* [nlat] */
  const double *meridional_scale; /* [nlat] */
  double scale[3];                /* unit factors of u, v and the height field */
  double z_div;                   /* height = field * scale[2] / z_div (g for geopotential, else 1) */
} lec_diag_grid;

enum lec_diag { LEC_DIAG_ZETA_MIN = 0, LEC_DIAG_ZETA_MAX, LEC_DIAG_HGT_MIN, LEC_DIAG_WIND_MAX, LEC_NDIAG };
#define LEC_NDIAG_VALUES 5      /* the four extrema + zeta at the track centre */

/* out_val[nsteps][LEC_NDIAG_VALUES]: extrema with NaNs skipped (nanmin / nanmax; NaN if the box is all NaN),
 * then zeta at (jc, ic) (NaN when not requested);
 * out_idx[nsteps][LEC_NDIAG]: numpy argmin / argmax of the box (row-major flat index, first occurrence,
 * the first NaN wins).  Errors: LEC_ERR_BOUNDS for a box outside the domain, LEC_ERR_DEGENERATE for a
 * domain axis with fewer than 3 points (first_derivative needs three); CUDA error text through
 * lec_last_error(NULL). */
int lec_diag850_device(const lec_diag_grid *grid, const void *u, const void *v, const void *z, int32_t nslots,
                       const lec_diag_step *steps, int32_t nsteps, double *out_val, int32_t *out_idx,
                       void *cuda_stream);          /* u, v, z, out_* in device memory; steps on the host */
int lec_diag850_host(const lec_diag_grid *grid, const void *u, const void *v, const void *z, int32_t nslots,
                     const lec_diag_step *steps, int32_t nsteps, double *out_val, int32_t *out_idx);
/* lec_diag850_host on WINDOWS of the planes: u, v, z are [nslots][win_rows][win_cols] host arrays, plane s holding the
 * domain points of columns origin[2 s] .. + win_cols - 1 and rows origin[2 s + 1] .. + win_rows - 1.  Box and centre
 * indices of the steps stay domain indices; the results are those of lec_diag850_host on the whole planes, bit for
 * bit.  The window a step needs: its box (and its centre point, when ic, jc >= 0) grown by one point a side and
 * clamped to the domain, and where that meets a domain edge, at least three points along that axis (MetPy's
 * one-sided first_derivative reads points 0..2 and n-3..n-1).  LEC_ERR_BOUNDS if a step reads outside its window. */
int lec_diag850_host_windows(const lec_diag_grid *grid, const void *u, const void *v, const void *z, int32_t nslots,
                             int32_t win_rows, int32_t win_cols, const int32_t *origin, const lec_diag_step *steps,
                             int32_t nsteps, double *out_val, int32_t *out_idx);

const char *lec_strerror(int code);
const char *lec_last_error(lec_handle *h);   /* CUDA error text after LEC_ERR_CUDA (NULL: handle-free calls of this thread) */
const char *lec_version(void);

#ifdef __cplusplus
}
#endif
#endif /* LEC_B200_H */
