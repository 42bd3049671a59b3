// C ABI of the B200 LEC engine (include/lec_b200.h): handle, grid tables, launches,
// host staging.  No torch types, no CPU fallback.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/lec_b200.h"
#include "lec_common.cuh"
#include "lec_finalize.cuh"
#include "lec_row_moments.cuh"
#include "lec_row_tile.cuh"
#include "lec_row_narrow.cuh"
#include "lec_diag850.cuh"
#include "lec_ingest.cuh"

using namespace lec;

struct lec_handle {
  lec_grid_desc desc{};
  int device = 0;
  GridDev g{};
  int pitch = 0;                                 // row length of the engine's own staging (lec_run_host*)
  double* d_tables = nullptr;
  float* d_tables32 = nullptr;
  int use_tile = 1;                             // LEC_ROW_KERNEL=tile|direct: TMA-tiled row kernel for wide boxes
  int num_sms = 148;
  long long h2d_bytes = 0, d2h_bytes = 0;      // PCIe traffic of the last lec_run_host
  int comp_mode = -1;                           // LEC_COMP=0|1: force the compensated fp32 linear sums off / on (-1: by box shape)
  int use_narrow = 1;                           // LEC_NARROW=0: never use the sub-warp kernel for narrow boxes
  int force_narrow_g = 0;                       // LEC_NARROW_G=4|8|16: force the group width (measurements)
  double* d_rec = nullptr;
  double* d_fin = nullptr;             // finalize scratch [max_steps][nlev][kLevStride]
  StepDev* d_steps = nullptr;          // [2][max_steps], alternating per kernel batch
  StepDev* h_steps = nullptr;          // pinned, same shape
  cudaEvent_t ev_steps[2] = {nullptr, nullptr};   // "step table half uploaded"
  bool steps_pending[2] = {false, false};
  int batch_parity = 0;
  int max_steps = 0, max_ny = 0;
  size_t elem = 4;
  std::vector<double> lon_deg, lat_deg, rlon, rlat, coslat, plev;
  // host-staging path
  void* stage[2][5] = {{nullptr}};
  size_t stage_cap = 0;                       // bytes of each stage[b][f]: stage_cap / (bytes of one staged slot) slots
  int host_windows = 0;                       // lec_set_host_windows
  void* raw_stage[2] = {nullptr, nullptr};   // raw sub-volumes (lec_run_host_raw): copy of n+1 overlaps ingest of n
  size_t raw_stage_bytes = 0;
  cudaStream_t s_ingest = nullptr;
  cudaEvent_t ev_raw_ready[2] = {nullptr, nullptr}, ev_raw_free[2] = {nullptr, nullptr}, ev_ingested = nullptr;
  long long raw_seq = 0;
  int* d_maps = nullptr;               // lon_map | lat_map | lev_map
  double* d_out_terms = nullptr;
  double* d_out_levels = nullptr;
  int* d_out_flags = nullptr;
  long long out_cap = 0;
  double* bnd_user = nullptr;          // lec_set_boundary_levels: device (run_device) or host (run_host*) pointer
  double* d_out_bnd = nullptr;         // device staging of the boundary pieces for run_host*
  long long bnd_cap = 0;
  cudaStream_t s_copy = nullptr, s_comp = nullptr;
  cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
  // timing
  std::vector<cudaEvent_t> ev_pool;
  int ev_used = 0;
  cudaEvent_t ev_call0 = nullptr, ev_call1 = nullptr;
  bool call_timed = false;
  bool accumulate_timing = false;
  long long launches = 0;
  lec_dispatch dispatch{};                      // row kernel of the last kernel batch (lec_last_dispatch)
  bool dispatched = false;
  std::string err;
};

namespace {

const char* kVersion = "lec_b200 0.2 (sm_100a; rows=tile)";

#define CK(call)                                                                   \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e__);                \
      return LEC_ERR_CUDA;                                                         \
    }                                                                              \
  } while (0)

// np.gradient interior coefficients at point i of a (possibly non-uniform) axis.  The kernels apply them in
// difference form, a (f[i-1] - f[i]) + c (f[i+1] - f[i]), which reads f[i]; numpy's branch for a wholly uniform
// axis, (f[i+1] - f[i-1]) / 2h, never does, so a missing f[i] makes the kernels' derivative NaN where numpy's is
// finite.  In the row kernels (d/dt, d/dlon, d/dlat, and d/dp in the stability term of Q) the derivative's
// co-factor holds the same missing value, so the NaN cannot reach an output.  F2's d[u]/dp is the exception
// (Ck_5 multiplies it by [w'v']): there the finalize kernel takes numpy's form on a uniform level axis (p_2h).
inline void grad_interior(const double* x, int i, double& a, double& b, double& c) {
  const double hs = x[i] - x[i - 1], hd = x[i + 1] - x[i];
  if (hs == hd) {
    a = -1.0 / (2.0 * hs); b = 0.0; c = 1.0 / (2.0 * hs);
  } else {
    a = -hd / (hs * (hd + hs)); b = (hd - hs) / (hd * hs); c = hs / (hd * (hd + hs));
  }
}

// 0: uniform longitudes, 1: per-column weights + uniform stencil, 2: per-column weights and stencil.
// fp64 arithmetic needs exact uniformity to skip a table; for fp32 arithmetic a 1e-6 relative spread is
// below the rounding of the values themselves.
int lon_mode(const lec_handle* h) {
  const bool m64 = h->desc.dtype == LEC_F64 || h->desc.math == LEC_MATH_F64;
  const int need = m64 ? 2 : 1;
  if (h->g.lon_uniform >= need) return 0;
  return h->g.stencil_uniform >= need ? 1 : 2;
}

template <typename FT, typename CT, int VEC, bool COMP>
void launch_direct_c(const RowParams& rp, int lonw, long long grid, cudaStream_t st) {
  if (lonw == 0) lec_row_moments_kernel<FT, CT, VEC, 0, COMP><<<(unsigned)grid, kRowThreads, 0, st>>>(rp);
  else if (lonw == 1) lec_row_moments_kernel<FT, CT, VEC, 1, COMP><<<(unsigned)grid, kRowThreads, 0, st>>>(rp);
  else lec_row_moments_kernel<FT, CT, VEC, 2, COMP><<<(unsigned)grid, kRowThreads, 0, st>>>(rp);
}

template <typename FT, typename CT, int VEC, bool COMP, typename ST>
void launch_narrow_c(const RowParams& rp, bool table, int G, long long grid, cudaStream_t st) {
#define LEC_NARROW(LW, GG) lec_row_moments_narrow_kernel<FT, CT, VEC, LW, GG, COMP, ST><<<(unsigned)grid, kNarrowThreads, 0, st>>>(rp)
  if (table) { if (G == 16) LEC_NARROW(2, 16); else if (G == 8) LEC_NARROW(2, 8); else LEC_NARROW(2, 4); }
  else { if (G == 16) LEC_NARROW(0, 16); else if (G == 8) LEC_NARROW(0, 8); else LEC_NARROW(0, 4); }
#undef LEC_NARROW
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// 4-D tensor map over a [slot][level][lat][lon] field (or [slot][level][window row][window column]) of `esize`-byte elements (fp64 / fp32 / int16) with a
// (bx x by) box in (lon, lat).
bool make_map(CUtensorMap* m, const void* base, int esize, int nlon, int nlat, int nlev, int nslots, int bx, int by) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return false;
  const cuuint64_t e = (cuuint64_t)esize;
  const cuuint64_t dims[4] = {(cuuint64_t)nlon, (cuuint64_t)nlat, (cuuint64_t)nlev, (cuuint64_t)nslots};
  const cuuint64_t strides[3] = {nlon * e, (cuuint64_t)nlat * nlon * e, (cuuint64_t)nlev * nlat * nlon * e};
  const cuuint32_t box[4] = {(cuuint32_t)bx, (cuuint32_t)by, 1, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  // (int16 fields: the driver has no signed 16-bit type; TMA copies the bits unchanged, zero fill included)
  const CUtensorMapDataType dt = esize == 8 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT64
                                 : esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT16;
  return enc(m, dt, 4, const_cast<void*>(base),
             dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Ring shapes of the tiled kernel, rows (= consumer warps) x stages: the one place the tile height is chosen
// (run_batch records it in lec_dispatch::tile_rows, launch_rows instantiates it).  R consumer warps + 1 producer warp;
// the per-SMSP register file allows 168 registers per thread up to 12 warps per CTA and 128 up to 16.  Stages sized
// to fill the 227 KB of shared memory.
//   fp32 arithmetic                 15 rows x 3 stages  (128 registers, no spills)
//   fp32 with compensated sums      11 rows x 4 stages  (six more live registers)
//   fp64 fields                     11 rows x 4 stages  (158-168 registers)
//   fp32 fields, fp64 arithmetic     7 rows x 6 stages  (four values per lane in fp64: > 168 registers)
// Over int16 fields a stage holds about half (fp32) or a quarter (fp64) of the bytes, so the ring gets more stages (at
// most 8: the barriers share the 128 bytes behind it).  fp32 arithmetic takes 11 rows, not 15: 15 consumer warps
// leave 128 registers and the decode's fp64 temporaries spill there (16-56 B).
//   fp32 arithmetic, plain or compensated  11 rows x 7 stages  (196 KB)
//   fp64 decode                            11 rows x 8 stages  (122 KB)
//   fp32 decode, fp64 arithmetic            7 rows x 8 stages  (142 KB)
struct RingShape { int rows, stages; };
constexpr RingShape ring_shape(bool f64, bool m64, bool comp, bool i16) {
  if (i16) return f64 ? RingShape{11, 8} : m64 ? RingShape{7, 8} : RingShape{11, 7};
  if (f64) return {11, 4};
  if (m64) return {7, 6};
  if (comp) return {11, 4};
  return {15, 3};
}

template <typename FT, typename CT, bool COMP, typename ST>
cudaError_t launch_tile_c(const TmaMaps& maps, const RowParams& rp, int lonw, int grid, cudaStream_t st) {
  constexpr RingShape shape = ring_shape(sizeof(FT) == 8, sizeof(CT) == 8, COMP, sizeof(ST) != sizeof(FT));
  constexpr int R = shape.rows, S = shape.stages;
  using G = TileGeom<FT, R, S, ST>;
  cudaError_t e = cudaSuccess;
#define LEC_TILE_LAUNCH(LW, TB, SMEM)                                                                             \
  do {                                                                                                            \
    e = cudaFuncSetAttribute(lec_row_moments_tile_kernel<FT, CT, LW, R, S, COMP, TB, ST>,                          \
                             cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);                                  \
    if (e == cudaSuccess) lec_row_moments_tile_kernel<FT, CT, LW, R, S, COMP, TB, ST><<<grid, G::threads, SMEM, st>>>(maps, rp); \
  } while (0)
  // fp32 per-column weights (LONW == 1): table in shared memory when it fits behind the ring
  const int tab_bytes = (sizeof(ST) == sizeof(FT) ? (rp.g.nlon + 3) & ~3 : rp.pk.ntab) * 4;
  if (lonw == 0) LEC_TILE_LAUNCH(0, false, G::smem_bytes);
  else if (lonw == 1) {
    if (sizeof(CT) == 4 && sizeof(FT) == 4 && G::smem_bytes + tab_bytes <= 227 * 1024) LEC_TILE_LAUNCH(1, true, G::smem_bytes + tab_bytes);
    else LEC_TILE_LAUNCH(1, false, G::smem_bytes);
  } else LEC_TILE_LAUNCH(2, false, G::smem_bytes);
#undef LEC_TILE_LAUNCH
  return e != cudaSuccess ? e : cudaGetLastError();
}

// The row-kernel instance that `d` names, over fields of FT stored as ST (int16 when d.packed).
template <typename FT, typename CT, bool COMP, typename ST>
cudaError_t launch_rows_c(const lec_dispatch& d, const RowParams& rp, const TmaMaps& maps, long long grid, int num_sms,
                          cudaStream_t st) {
  constexpr int VEC = 16 / sizeof(FT);
  if (d.kernel == LEC_ROWS_TILED) {
    const int pgrid = (int)std::min<long long>(grid, (long long)num_sms);      // persistent: one CTA per SM
    return launch_tile_c<FT, CT, COMP, ST>(maps, rp, d.lonw, pgrid, st);
  }
  if (d.kernel == LEC_ROWS_SUBWARP) launch_narrow_c<FT, CT, VEC, COMP, ST>(rp, d.lonw != 0, d.group, grid, st);
  else if constexpr (sizeof(ST) != sizeof(FT)) return cudaErrorInvalidValue;     // no direct kernel reads int16 fields
  else if (d.vec == 1) launch_direct_c<FT, CT, 1, COMP>(rp, d.lonw, grid, st);
  else launch_direct_c<FT, CT, VEC, COMP>(rp, d.lonw, grid, st);
  return cudaGetLastError();
}

// COMP (compensated linear sums) only exists for fp32 arithmetic.
template <typename FT, typename CT, typename ST>
cudaError_t launch_rows_t(const lec_dispatch& d, const RowParams& rp, const TmaMaps& maps, long long grid, int num_sms,
                          cudaStream_t st) {
  if constexpr (sizeof(CT) == 4) {
    if (d.comp) return launch_rows_c<FT, CT, true, ST>(d, rp, maps, grid, num_sms, st);
  }
  return launch_rows_c<FT, CT, false, ST>(d, rp, maps, grid, num_sms, st);
}

// Launches the row kernel of one batch: the instance `d` (filled by run_batch) names, over the handle's field dtype.
cudaError_t launch_rows(const lec_handle* h, const lec_dispatch& d, const RowParams& rp, const TmaMaps& maps,
                        long long grid, cudaStream_t st) {
  const int sms = h->num_sms;
  if (h->desc.dtype == LEC_F64) {
    return d.packed ? launch_rows_t<double, double, short>(d, rp, maps, grid, sms, st)
                    : launch_rows_t<double, double, double>(d, rp, maps, grid, sms, st);
  }
  if (d.math64) {
    return d.packed ? launch_rows_t<float, double, short>(d, rp, maps, grid, sms, st)
                    : launch_rows_t<float, double, float>(d, rp, maps, grid, sms, st);
  }
  return d.packed ? launch_rows_t<float, float, short>(d, rp, maps, grid, sms, st)
                  : launch_rows_t<float, float, float>(d, rp, maps, grid, sms, st);
}

cudaEvent_t next_event(lec_handle* h) {
  if (h->ev_used == (int)h->ev_pool.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    h->ev_pool.push_back(e);
  }
  return h->ev_pool[h->ev_used++];
}

// The slot and box checks of one step (build_step; lec_run_host* before they compute windows from the steps).
int check_step(const lec_handle* h, const lec_step& s, int nslots) {
  if (s.slot < 0 || s.slot >= nslots || s.slot_m < 0 || s.slot_m >= nslots || s.slot_p < 0 ||
      s.slot_p >= nslots)
    return LEC_ERR_BOUNDS;
  if (s.i0 < 0 || s.i1 >= h->desc.nlon || s.j0 < 0 || s.j1 >= h->desc.nlat) return LEC_ERR_BOUNDS;
  if (s.i1 - s.i0 < 1 || s.j1 - s.j0 < 1) return LEC_ERR_DEGENERATE;
  return LEC_OK;
}

// Validate one step and build its device form.
int build_step(const lec_handle* h, const lec_step& s, int nslots, StepDev& d) {
  if (const int rc = check_step(h, s, nslots)) return rc;
  if (s.j1 - s.j0 + 1 > h->max_ny) return LEC_ERR_BOUNDS;
  const double* x = h->lon_deg.data();
  const double* y = h->lat_deg.data();
  const double* rl = h->rlon.data();
  const double* rp = h->rlat.data();
  d.slot = s.slot; d.slot_m = s.slot_m; d.slot_p = s.slot_p;
  d.i0 = s.i0; d.i1 = s.i1; d.j0 = s.j0; d.j1 = s.j1; d.rec_base = 0;
  d.ox = d.oy = d.oxm = d.oym = d.oxp = d.oyp = 0;       // window origins and T offsets: run_batch
  d.d_m = d.d_p = 0;
  // every constant factor of Q = cp (dT/dt + u dT/dx + v dT/dy - S omega) is folded on the host
  const double q0 = kCp * h->g.scale[0], qv = q0 * h->g.scale[2];
  d.ct_m = q0 * s.ct_m; d.ct_p = q0 * s.ct_p; d.ct_s = q0 * (s.ct_m + s.ct_0 + s.ct_p);
  // one-sided np.gradient at the box edges; gradient(lon, lon) is exactly 1 there
  const double unit = kDeg2Rad * kRe;
  d.cxW = 1.0 / ((x[s.i0 + 1] - x[s.i0]) * unit);
  d.cxE = 1.0 / ((x[s.i1] - x[s.i1 - 1]) * unit);
  d.cyS = qv / ((y[s.j0 + 1] - y[s.j0]) * unit);
  d.cyN = qv / ((y[s.j1] - y[s.j1 - 1]) * unit);
  d.wW = 0.5 * (rl[s.i0 + 1] - rl[s.i0]);
  d.wE = 0.5 * (rl[s.i1] - rl[s.i1 - 1]);
  const double xlen = rl[s.i1] - rl[s.i0];                       // box_data.py:128
  const double ylen = std::sin(rp[s.j1]) - std::sin(rp[s.j0]);   // box_data.py:129-131
  d.inv_xlen = 1.0 / xlen; d.inv_ylen = 1.0 / ylen;
  d.c1 = -1.0 / (kRe * xlen * ylen);                             // boundary_terms.py:122
  d.c2 = -1.0 / (kRe * ylen);                                    // boundary_terms.py:123
  d.f_ct_m = (float)d.ct_m; d.f_ct_p = (float)d.ct_p; d.f_ct_s = (float)d.ct_s;
  d.f_cxW = (float)d.cxW; d.f_cxE = (float)d.cxE; d.f_cyS = (float)d.cyS; d.f_cyN = (float)d.cyN;
  d.f_wW = (float)d.wW; d.f_wE = (float)d.wE;
  d.f_wWn = h->g.wl_u != 0.0 ? (float)(d.wW / h->g.wl_u) : 0.f;
  d.f_wEn = h->g.wl_u != 0.0 ? (float)(d.wE / h->g.wl_u) : 0.f;
  d.f_pad = 0.f;
  return LEC_OK;
}

// The decode a lec_raw_desc or lec_packed_desc states (members of the same names), checked once for both entry points,
// as IngestParams' decode members; what a field does not use is folded as PackedDev folds it (fills: kNoFill).
template <typename Desc>
int read_decode(lec_handle* h, const Desc& d, bool i16, IngestParams (&dec)[5]) {
  for (int f = 0; f < 5; ++f) {
    IngestParams& e = dec[f];
    if (d.nfill[f] < 0 || d.nfill[f] > 2) { h->err = "at most two fill values per field"; return LEC_ERR_INVALID; }
    for (int n = 0; n < d.nfill[f]; ++n)
      if (const double v = d.fill[f][n]; i16 && !(v >= -32768.0 && v <= 32767.0 && v == std::floor(v))) { h->err = "a fill value is not an int16 value"; return LEC_ERR_INVALID; }
    e.nfill = d.nfill[f]; e.fill0 = e.nfill > 0 ? d.fill[f][0] : kNoFill; e.fill1 = e.nfill > 1 ? d.fill[f][1] : kNoFill;
    e.use_scale = i16 && d.use_scale[f]; e.use_offset = i16 && d.use_offset[f]; e.round32 = i16 && d.round_f32[f];
    e.scale = e.use_scale ? d.scale[f] : 1.0; e.offset = e.use_offset ? d.offset[f] : -0.0;
  }
  return LEC_OK;
}

}  // namespace

extern "C" {

const char* lec_version(void) { return kVersion; }

const char* lec_strerror(int code) {
  switch (code) {
    case LEC_OK: return "ok";
    case LEC_ERR_INVALID: return "invalid argument";
    case LEC_ERR_CUDA: return "CUDA runtime failure";
    case LEC_ERR_DEGENERATE: return "box axis has fewer than 2 points";
    case LEC_ERR_BOUNDS: return "box or time slot outside the prepared domain";
    case LEC_ERR_NOMEM: return "out of memory";
    default: return "unknown error";
  }
}

static thread_local std::string g_free_err;   // error text of the handle-free entry points

const char* lec_last_error(lec_handle* h) { return h ? h->err.c_str() : g_free_err.c_str(); }

int64_t lec_launch_count(lec_handle* h) { return h ? h->launches : 0; }

int lec_last_dispatch(const lec_handle* h, lec_dispatch* out) {
  if (!h || !out || !h->dispatched) return LEC_ERR_INVALID;
  *out = h->dispatch;
  return LEC_OK;
}

int lec_last_transfer(lec_handle* h, int64_t out_bytes[2]) {
  if (!h || !out_bytes) return LEC_ERR_INVALID;
  out_bytes[0] = h->h2d_bytes; out_bytes[1] = h->d2h_bytes;
  return LEC_OK;
}

int lec_gradient_coefs(const double* x, int32_t n, double* a, double* b, double* c) {
  if (!x || !a || !b || !c || n < 2) return LEC_ERR_INVALID;
  bool uniform = true;
  const double h0 = x[1] - x[0];
  for (int i = 1; i + 1 < n; ++i)
    if (x[i + 1] - x[i] != h0) { uniform = false; break; }
  for (int i = 1; i + 1 < n; ++i) {
    if (uniform) { a[i] = -1.0 / (2.0 * h0); b[i] = 0.0; c[i] = 1.0 / (2.0 * h0); }
    else {
      const double hs = x[i] - x[i - 1], hd = x[i + 1] - x[i];
      a[i] = -hd / (hs * (hd + hs)); b[i] = (hd - hs) / (hd * hs); c[i] = hs / (hd * (hd + hs));
    }
  }
  a[0] = 0.0; b[0] = -1.0 / (x[1] - x[0]); c[0] = 1.0 / (x[1] - x[0]);
  a[n - 1] = -1.0 / (x[n - 1] - x[n - 2]); b[n - 1] = 1.0 / (x[n - 1] - x[n - 2]); c[n - 1] = 0.0;
  return LEC_OK;
}

int32_t lec_nearest_index(const double* coord, int32_t n, double value) {
  if (!coord || n < 1 || std::isnan(value)) return -1;
  // pandas Index._get_nearest_indexer: left = pad, right = backfill,
  // left if left_distance < right_distance (or right missing) else right.
  const double* ub = std::upper_bound(coord, coord + n, value);   // first > value
  const int left = int(ub - coord) - 1;                           // last <= value
  const double* lb = std::lower_bound(coord, coord + n, value);   // first >= value
  const int right = (lb == coord + n) ? -1 : int(lb - coord);
  if (left < 0) return right;
  if (right < 0) return left;
  const double dl = std::fabs(coord[left] - value), dr = std::fabs(coord[right] - value);
  return (dl < dr) ? left : right;
}

int lec_destroy(lec_handle* h) {
  if (!h) return LEC_OK;
  cudaSetDevice(h->device);
  cudaFree(h->d_tables); cudaFree(h->d_tables32); cudaFree(h->d_rec); cudaFree(h->d_fin); cudaFree(h->d_steps);
  if (h->h_steps) cudaFreeHost(h->h_steps);
  for (int b = 0; b < 2; ++b)
    for (int f = 0; f < 5; ++f) cudaFree(h->stage[b][f]);
  cudaFree(h->d_out_terms); cudaFree(h->d_out_levels); cudaFree(h->d_out_flags); cudaFree(h->d_out_bnd);
  cudaFree(h->raw_stage[0]); cudaFree(h->raw_stage[1]); cudaFree(h->d_maps);
  for (int b = 0; b < 2; ++b) {
    if (h->ev_copied[b]) cudaEventDestroy(h->ev_copied[b]);
    if (h->ev_done[b]) cudaEventDestroy(h->ev_done[b]);
  }
  for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
  for (int b = 0; b < 2; ++b) if (h->ev_steps[b]) cudaEventDestroy(h->ev_steps[b]);
  if (h->ev_call0) cudaEventDestroy(h->ev_call0);
  if (h->ev_call1) cudaEventDestroy(h->ev_call1);
  if (h->s_copy) cudaStreamDestroy(h->s_copy);
  if (h->s_comp) cudaStreamDestroy(h->s_comp);
  if (h->s_ingest) cudaStreamDestroy(h->s_ingest);
  for (int b = 0; b < 2; ++b) {
    if (h->ev_raw_ready[b]) cudaEventDestroy(h->ev_raw_ready[b]);
    if (h->ev_raw_free[b]) cudaEventDestroy(h->ev_raw_free[b]);
  }
  if (h->ev_ingested) cudaEventDestroy(h->ev_ingested);
  delete h;
  return LEC_OK;
}

int lec_create(lec_handle** out, const lec_grid_desc* desc) {
  if (!out || !desc) return LEC_ERR_INVALID;
  *out = nullptr;
  const int nlon = desc->nlon, nlat = desc->nlat, L = desc->nlev;
  if (nlon < 2 || nlat < 2 || L < 2) return LEC_ERR_DEGENERATE;
  if (!desc->lon_deg || !desc->lat_deg || !desc->rlon || !desc->rlat || !desc->coslat || !desc->plev)
    return LEC_ERR_INVALID;
  if (desc->dtype != LEC_F32 && desc->dtype != LEC_F64) return LEC_ERR_INVALID;
  if (desc->max_steps < 1 || desc->max_box_rows < 0 || desc->max_box_rows > nlat) return LEC_ERR_INVALID;
  for (int i = 0; i + 1 < nlon; ++i) if (!(desc->lon_deg[i + 1] > desc->lon_deg[i])) return LEC_ERR_INVALID;
  for (int j = 0; j + 1 < nlat; ++j) if (!(desc->lat_deg[j + 1] > desc->lat_deg[j])) return LEC_ERR_INVALID;
  for (int k = 0; k + 1 < L; ++k) if (!(desc->plev[k + 1] > desc->plev[k])) return LEC_ERR_INVALID;

  lec_handle* h = new (std::nothrow) lec_handle;
  if (!h) return LEC_ERR_NOMEM;
  *out = h;   // returned even on failure so lec_last_error works; caller still destroys
  h->desc = *desc;
  h->device = desc->device;
  h->elem = desc->dtype == LEC_F64 ? 8 : 4;
  h->max_steps = desc->max_steps;
  if (const char* e = std::getenv("LEC_NARROW")) h->use_narrow = std::atoi(e) != 0;
  if (const char* e = std::getenv("LEC_COMP")) h->comp_mode = std::atoi(e) != 0;
  if (const char* e = std::getenv("LEC_NARROW_G")) {
    const int gq = std::atoi(e);
    if (gq == 16 || gq == 8 || gq == 4) h->force_narrow_g = gq;
  }
  if (const char* e = std::getenv("LEC_ROW_KERNEL")) {
    if (std::strcmp(e, "tile") == 0) h->use_tile = 1;
    else if (std::strcmp(e, "direct") == 0) h->use_tile = 0;
  }
  h->max_ny = desc->max_box_rows ? desc->max_box_rows : nlat;
  h->lon_deg.assign(desc->lon_deg, desc->lon_deg + nlon);
  h->rlon.assign(desc->rlon, desc->rlon + nlon);
  h->lat_deg.assign(desc->lat_deg, desc->lat_deg + nlat);
  h->rlat.assign(desc->rlat, desc->rlat + nlat);
  h->coslat.assign(desc->coslat, desc->coslat + nlat);
  h->plev.assign(desc->plev, desc->plev + L);
  h->desc.lon_deg = h->lon_deg.data(); h->desc.lat_deg = h->lat_deg.data();
  h->desc.rlon = h->rlon.data(); h->desc.rlat = h->rlat.data();
  h->desc.coslat = h->coslat.data(); h->desc.plev = h->plev.data();

  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (h->device < 0 || h->device >= ndev) { h->err = "no such CUDA device"; return LEC_ERR_CUDA; }
  CK(cudaSetDevice(h->device));
  CK(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device));

  // ---- host tables --------------------------------------------------------------------------
  const double unit = kDeg2Rad * kRe;
  std::vector<double> tab;
  auto reserve = [&](int n) { size_t o = tab.size(); tab.resize(o + ((n + 1) & ~1), 0.0); return o; };
  const size_t o_wl = reserve(nlon + 4), o_cxa = reserve(nlon + 4), o_cxc = reserve(nlon + 4);   // read up to the padded pitch
  const size_t o_rlat = reserve(nlat), o_cos = reserve(nlat), o_tan = reserve(nlat), o_cya = reserve(nlat),
               o_cyc = reserve(nlat), o_fya = reserve(nlat), o_fyc = reserve(nlat), o_fxj = reserve(nlat);
  double scl[5];
  for (int f = 0; f < 5; ++f) scl[f] = desc->field_scale[f] == 0.0 ? 1.0 : desc->field_scale[f];
  for (int f = 0; f < 5; ++f) h->g.scale[f] = scl[f];     // build_step needs them before g is complete
  const double q0 = kCp * scl[0];                          // cp * (unit factor of T)
  const size_t o_p = reserve(L), o_pa = reserve(L), o_pc = reserve(L), o_sm = reserve(L), o_sp = reserve(L),
               o_ss = reserve(L);
  const double* x = h->lon_deg.data();
  const double* y = h->lat_deg.data();
  for (int i = 1; i + 1 < nlon; ++i) {
    double a, b, c;
    grad_interior(x, i, a, b, c);
    const double gl = a * x[i - 1] + b * x[i] + c * x[i + 1];          // np.gradient(lon, lon)
    const double fold = 1.0 / (gl * kDeg2Rad * kRe);                   // 1/(deg2rad(.) Re); cos(lat) per row
    tab[o_cxa + i] = a * fold; tab[o_cxc + i] = c * fold;
    tab[o_wl + i] = 0.5 * (h->rlon[i + 1] - h->rlon[i - 1]);
  }
  // uniformity of the interior longitude tables: 2 exact, 1 to 1e-6 relative, 0 neither -- separately
  // for the lon stencil (degree axis: exactly uniform on the usual float32 grids) and for stencil +
  // trapezoid weights (float32 radians: weights differ by ~3e-5)
  int uni = 0, uni_st = 0;
  double m_wl = 0.0, m_a = 0.0, m_c = 0.0;
  if (nlon >= 3) {
    for (int i = 1; i + 1 < nlon; ++i) { m_wl += tab[o_wl + i]; m_a += tab[o_cxa + i]; m_c += tab[o_cxc + i]; }
    m_wl /= (nlon - 2); m_a /= (nlon - 2); m_c /= (nlon - 2);
    double dev_w = 0.0, dev_s = 0.0;
    bool exact_w = true, exact_s = true;
    for (int i = 1; i + 1 < nlon; ++i) {
      dev_w = std::max(dev_w, std::fabs(tab[o_wl + i] / m_wl - 1.0));
      dev_s = std::max(dev_s, std::fabs(tab[o_cxa + i] / m_a - 1.0));
      dev_s = std::max(dev_s, std::fabs(tab[o_cxc + i] / m_c - 1.0));
      exact_w = exact_w && tab[o_wl + i] == tab[o_wl + 1];
      exact_s = exact_s && tab[o_cxa + i] == tab[o_cxa + 1] && tab[o_cxc + i] == tab[o_cxc + 1];
    }
    uni_st = exact_s ? 2 : (dev_s < 1e-6 ? 1 : 0);
    uni = (exact_s && exact_w) ? 2 : (std::max(dev_s, dev_w) < 1e-6 ? 1 : 0);
    if (exact_w) m_wl = tab[o_wl + 1];
    if (exact_s) { m_a = tab[o_cxa + 1]; m_c = tab[o_cxc + 1]; }
  }
  for (int j = 0; j < nlat; ++j) {
    tab[o_rlat + j] = h->rlat[j]; tab[o_cos + j] = h->coslat[j]; tab[o_tan + j] = std::tan(h->rlat[j]);
    tab[o_fxj + j] = q0 * scl[1] / h->coslat[j];           // multiplies the lon stencil: cp sT sU / cos(lat)
    if (j >= 1 && j + 1 < nlat) {
      double a, b, c;
      grad_interior(y, j, a, b, c);
      const double gp = a * y[j - 1] + b * y[j] + c * y[j + 1];
      const double fold = 1.0 / (gp * unit);
      tab[o_cya + j] = q0 * scl[2] * a * fold; tab[o_cyc + j] = q0 * scl[2] * c * fold;   // cp sT sV / dy
      grad_interior(h->rlat.data(), j, a, b, c);
      tab[o_fya + j] = a; tab[o_fyc + j] = c;
    }
  }
  double p_2h = 2.0 * (h->plev[1] - h->plev[0]);
  for (int k = 1; k + 1 < L; ++k)
    if (h->plev[k + 1] - h->plev[k] != h->plev[1] - h->plev[0]) p_2h = 0.0;
  {
    std::vector<double> a(L), b(L), c(L), E(L);
    lec_gradient_coefs(h->plev.data(), L, a.data(), b.data(), c.data());
    // per-point non-uniform rule in the interior (identical to numpy's uniform branch where hs == hd, but for
    // the centre read: see grad_interior)
    for (int k = 1; k + 1 < L; ++k) grad_interior(h->plev.data(), k, a[k], b[k], c[k]);
    for (int k = 0; k < L; ++k) E[k] = std::pow(h->plev[k] / kP0, kKappa);   // T / theta
    for (int k = 0; k < L; ++k) {
      tab[o_p + k] = h->plev[k]; tab[o_pa + k] = a[k]; tab[o_pc + k] = c[k];
      const double sm = (k > 0) ? -E[k] * a[k] / E[k - 1] : 0.0;
      const double sp = (k + 1 < L) ? -E[k] * c[k] / E[k + 1] : 0.0;
      const double qs = -q0 * scl[3];                     // -cp sT sW: Q has -S omega
      tab[o_sm + k] = qs * sm; tab[o_sp + k] = qs * sp; tab[o_ss + k] = qs * (sm + sp - b[k]);
    }
  }
  CK(cudaMalloc(&h->d_tables, tab.size() * sizeof(double)));
  CK(cudaMemcpy(h->d_tables, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
  GridDev& g = h->g;
  g.nlon = nlon; g.nlat = nlat; g.nlev = L;
  g.wl = h->d_tables + o_wl; g.cxa = h->d_tables + o_cxa; g.cxc = h->d_tables + o_cxc;
  g.rlat = h->d_tables + o_rlat; g.coslat = h->d_tables + o_cos; g.tanlat = h->d_tables + o_tan;
  g.cya = h->d_tables + o_cya; g.cyc = h->d_tables + o_cyc; g.fya = h->d_tables + o_fya; g.fyc = h->d_tables + o_fyc;
  g.fxj = h->d_tables + o_fxj;
  g.plev = h->d_tables + o_p; g.pa = h->d_tables + o_pa; g.pc = h->d_tables + o_pc; g.p_2h = p_2h;
  g.sm = h->d_tables + o_sm; g.sp = h->d_tables + o_sp; g.ss = h->d_tables + o_ss;
  g.lon_uniform = uni; g.stencil_uniform = uni_st;
  g.wl_u = m_wl; g.cxa_u = m_a; g.cxc_u = m_c;
  {
    const size_t n4 = (size_t)((nlon + 3) & ~3), l4 = (size_t)((nlat + 3) & ~3), k4 = (size_t)((L + 3) & ~3);
    std::vector<float> t32(3 * n4 + 3 * l4 + 3 * k4, 0.f);
    for (int i = 0; i < nlon; ++i) {
      t32[i] = (float)tab[o_wl + i]; t32[n4 + i] = (float)tab[o_cxa + i]; t32[2 * n4 + i] = (float)tab[o_cxc + i];
    }
    float* lat32 = t32.data() + 3 * n4;
    for (int j = 0; j < nlat; ++j) {
      lat32[j] = (float)tab[o_cya + j]; lat32[l4 + j] = (float)tab[o_cyc + j]; lat32[2 * l4 + j] = (float)tab[o_fxj + j];
    }
    float* lev32 = lat32 + 3 * l4;
    for (int k = 0; k < L; ++k) {
      lev32[k] = (float)tab[o_sm + k]; lev32[k4 + k] = (float)tab[o_sp + k]; lev32[2 * k4 + k] = (float)tab[o_ss + k];
    }
    CK(cudaMalloc(&h->d_tables32, t32.size() * sizeof(float)));
    CK(cudaMemcpy(h->d_tables32, t32.data(), t32.size() * sizeof(float), cudaMemcpyHostToDevice));
    g.wl32 = h->d_tables32; g.cxa32 = h->d_tables32 + n4; g.cxc32 = h->d_tables32 + 2 * n4;
    g.cya32 = h->d_tables32 + 3 * n4; g.cyc32 = g.cya32 + l4; g.fxj32 = g.cya32 + 2 * l4;
    g.sm32 = g.cya32 + 3 * l4; g.sp32 = g.sm32 + k4; g.ss32 = g.sm32 + 2 * k4;
    g.cxa_u32 = (float)m_a; g.cxc_u32 = (float)m_c;
  }
  for (int f = 0; f < 5; ++f) g.scale[f] = desc->field_scale[f] == 0.0 ? 1.0 : desc->field_scale[f];
  {
    const int vecw = desc->dtype == LEC_F64 ? 2 : 4;
    h->pitch = (nlon + vecw - 1) / vecw * vecw;
  }

  const size_t rec_bytes = (size_t)h->max_steps * L * h->max_ny * LEC_NREC * sizeof(double);
  if (cudaMalloc(&h->d_rec, rec_bytes) != cudaSuccess) { cudaGetLastError(); h->err = "row-record scratch"; return LEC_ERR_NOMEM; }
  CK(cudaMalloc(&h->d_fin, sizeof(double) * (size_t)h->max_steps * L * kLevStride));
  CK(cudaMalloc(&h->d_steps, sizeof(StepDev) * 2 * h->max_steps));
  CK(cudaMallocHost(&h->h_steps, sizeof(StepDev) * 2 * h->max_steps));
  for (int b = 0; b < 2; ++b) CK(cudaEventCreateWithFlags(&h->ev_steps[b], cudaEventDisableTiming));
  CK(cudaEventCreate(&h->ev_call0));
  CK(cudaEventCreate(&h->ev_call1));
  return LEC_OK;
}

// Window of every staged slot of a kernel batch (lec_set_host_windows): the shared shape and each slot's origin,
// indexed by the batch's slot numbers.
struct WinView { int rows, pitch; const int* ox; const int* oy; };

// One kernel batch (<= max_steps steps) on `st`.  pitch: row length of the fields in elements (0: the grid's);
// pk: the fields are int16, decoded by the row kernel (lec_run_device_packed); win: the fields are staged windows.
static int run_batch(lec_handle* h, const void* const fields[5], int nslots, const lec_step* steps, int n,
                     double* out_terms, double* out_levels, int* out_flags, double* out_bnd, cudaStream_t st,
                     int pitch = 0, const PackedDev* pk = nullptr, const WinView* win = nullptr) {
  // nlon below is the ROW LENGTH of the field buffers: the grid's for caller-owned fp device fields, the padded
  // pitch of the engine's own staging or of caller-owned int16 fields (box indices are checked against the grid
  // in build_step); with windows, the rows of a slot are win->rows rows of win->pitch elements
  const int L = h->desc.nlev, nlon = win ? win->pitch : pitch > 0 ? pitch : h->desc.nlon;
  const int nrows = win ? win->rows : h->desc.nlat;
  GridDev gd = h->g;
  gd.nlon = pitch > 0 ? pitch : h->desc.nlon;       // (the tiled kernel's shared weight table: global columns)
  int max_rows = 0, max_cols = 0;
  bool same_box = true, same_rows = true;
  const int par = h->batch_parity;
  h->batch_parity ^= 1;
  StepDev* hs = h->h_steps + (size_t)par * h->max_steps;
  StepDev* ds = h->d_steps + (size_t)par * h->max_steps;
  if (h->steps_pending[par]) { CK(cudaEventSynchronize(h->ev_steps[par])); h->steps_pending[par] = false; }
  for (int s = 0; s < n; ++s) {
    const int rc = build_step(h, steps[s], nslots, hs[s]);
    if (rc != LEC_OK) return rc;
    if (win) {
      StepDev& d = hs[s];
      d.ox = win->ox[d.slot]; d.oy = win->oy[d.slot];
      d.oxm = win->ox[d.slot_m]; d.oym = win->oy[d.slot_m];
      d.oxp = win->ox[d.slot_p]; d.oyp = win->oy[d.slot_p];
    }
    max_rows = std::max(max_rows, steps[s].j1 - steps[s].j0 + 1);
    max_cols = std::max(max_cols, steps[s].i1 - steps[s].i0 + 1);
    same_box = same_box && steps[s].i0 == steps[0].i0 && steps[s].i1 == steps[0].i1 &&
               steps[s].j0 == steps[0].j0 && steps[s].j1 == steps[0].j1;
    same_rows = same_rows && steps[s].j1 - steps[s].j0 == steps[0].j1 - steps[0].j0;
  }
  // latitude banding (fixed box, several steps): sweep time inside a band of box rows so T(t+-1) stays in L2
  int band_rows = h->desc.band_rows;
  if (band_rows <= 0) {
    // (counted at the handle's element size for int16 fields too: they take the block order of lec_run_device on the
    //  decoded fields; a budget for 2-byte values has not been measured)
    const double band_budget = 18e6;   // bytes of all five fields per band-step
    band_rows = int(band_budget / (5.0 * L * max_cols * h->elem));
  }
  const int vecw = h->desc.dtype == LEC_F64 ? 2 : 4;
  bool vec = nlon % vecw == 0;
  for (int f = 0; f < 5; ++f) vec = vec && (reinterpret_cast<uintptr_t>(fields[f]) % 16 == 0);
  // narrow boxes (track mode): a row is swept by a group of 16 / 8 / 4 lanes, 32/G rows per warp
  int max_chunks = 0;
  for (int s = 0; s < n; ++s) max_chunks = std::max(max_chunks, steps[s].i1 / vecw - steps[s].i0 / vecw + 1);
  // (measured, scripts/c5_probe.py: 8-lane groups win up to ~100 chunks -- 2873 vs 1527 GB/s on the
  //  151-column C5 box --, 16-lane groups by 5 % at 151 chunks, the warp-per-row kernels beyond)
  int narrow_g = (vec && h->use_narrow && max_chunks <= 200) ? (max_chunks > 112 ? 16 : max_chunks > 4 ? 8 : 4) : 0;
  if (h->force_narrow_g && vec) narrow_g = h->force_narrow_g;
  // Compensated fp32 linear sums (lec_lin_add): needed when a lane adds many chunks (long rows) while the
  // box is short in latitude, i.e. when the area eddies [X]_j - [[X]] are small against the zonal eddies
  // whose partial sums carry the rounding error (a 24-row band of the C4 grid gave Cz_2 / Ca_2 1.7e-5
  // without it).  Tall boxes and short rows run the plain sums (7 % fewer FP instructions).
  int comp_mode = h->comp_mode;
  const bool comp = comp_mode == 1 || (comp_mode < 0 && max_chunks > 32 * 4 && max_rows <= 128);
  // wide boxes: the TMA-tiled kernel (rows 16-byte aligned, a tensor-map encoder in the driver); int16 fields have
  // no other wide-box kernel (the caller's pitch makes every row 16-byte aligned)
  const bool want_tile = (h->use_tile || pk) && vec && !narrow_g && encode_tiled_fn() != nullptr;
  if (pk && !narrow_g && !want_tile) { h->err = "int16 fields need the TMA-tiled row kernel: no tensor-map encoder"; return LEC_ERR_CUDA; }
  // The row-kernel instance of this batch, decided here once: launch_rows instantiates it and lec_last_dispatch
  // reports it.  COMP only exists for fp32 arithmetic; the sub-warp kernel has no per-column-weight variant (any
  // table is the full one).
  const bool math64 = h->desc.dtype == LEC_F64 || h->desc.math == LEC_MATH_F64;
  const int lonw = lon_mode(h);
  lec_dispatch d{};
  d.kernel = want_tile ? LEC_ROWS_TILED : narrow_g ? LEC_ROWS_SUBWARP : LEC_ROWS_DIRECT;
  d.vec = vec ? vecw : 1;
  d.group = d.kernel == LEC_ROWS_SUBWARP ? narrow_g : 32;
  d.lonw = d.kernel == LEC_ROWS_SUBWARP && lonw != 0 ? 2 : lonw;
  d.comp = comp && !math64;
  d.math64 = math64;
  d.tile_rows = d.kernel == LEC_ROWS_TILED ? ring_shape(h->desc.dtype == LEC_F64, math64, d.comp, pk).rows
                : d.kernel == LEC_ROWS_SUBWARP ? kNarrowWarps * (32 / narrow_g) : kRowsPerCta;
  d.packed = pk != nullptr;
  if (d.kernel != LEC_ROWS_TILED) {
    // The direct and sub-warp kernels address T(slot_m) and T(slot_p) as 32-bit element offsets from T(slot) (64-bit
    // bases instead spill in the sub-warp kernel's fp64-arithmetic instances); the tiled kernel takes slots as TMA
    // coordinates and has no such limit.
    const long long stride = (long long)L * nrows * nlon;
    for (int s = 0; s < n; ++s) {
      StepDev& q = hs[s];
      const long long dm = (long long)(q.slot_m - q.slot) * stride + (long long)(q.oy - q.oym) * nlon + (q.ox - q.oxm);
      const long long dp = (long long)(q.slot_p - q.slot) * stride + (long long)(q.oy - q.oyp) * nlon + (q.ox - q.oxp);
      if (dm <= -(1LL << 31) || dm >= (1LL << 31) || dp <= -(1LL << 31) || dp >= (1LL << 31)) {
        h->err = "slot_m / slot_p lie 2^31 or more elements from slot, which the direct and sub-warp row kernels "
                 "cannot address (the tiled kernel can)";
        return LEC_ERR_INVALID;
      }
      q.d_m = (int)dm; q.d_p = (int)dp;
    }
  }
  const int tile_rows = d.tile_rows;
  band_rows = std::max(tile_rows, band_rows / tile_rows * tile_rows);
  // (moving boxes of one height were tried with the banded order too: 3.06 TB/s against 3.28 unbanded on the C5
  //  track -- a whole 151 x 151 x 55 step is 35 MB, so step-major order already keeps T(t+-1) in L2)
  // moving boxes of one height are banded only on request (lec_grid_desc::band_rows > 0): measured slower than
  // step-major order on the C5 track (2.19-2.25 vs 2.07 ms for bands of 8-64 rows; a whole step is 35 MB, L2-resident)
  const bool bandable = same_box || (same_rows && h->desc.band_rows > 0);
  if (!bandable || n < 3 || band_rows >= max_rows) band_rows = (max_rows + tile_rows - 1) / tile_rows * tile_rows;
  RowParams rp{};
  for (int f = 0; f < 5; ++f) rp.field[f] = fields[f];
  rp.g = gd; rp.steps = ds; rp.rec = h->d_rec; rp.nsteps = n; rp.max_ny = h->max_ny;
  rp.tiles_per_band = band_rows / tile_rows;
  rp.dv_tiles = FastDiv::make((unsigned)rp.tiles_per_band);
  rp.dv_lev = FastDiv::make((unsigned)L);
  rp.dv_steps = FastDiv::make((unsigned)n);
  rp.nbands = (max_rows + band_rows - 1) / band_rows;
  rp.slot_stride = (long long)L * nrows * nlon;
  rp.lev_stride = (long long)nrows * nlon;
  rp.row_stride = nlon;
  if (rp.slot_stride >= (1LL << 31)) { h->err = "one time slot holds 2^31 or more elements"; return LEC_ERR_INVALID; }
  const long long grid = (long long)rp.nbands * n * L * rp.tiles_per_band;
  if (grid > 0x7fffffffLL) return LEC_ERR_INVALID;
  rp.grid = grid;
  if (pk) rp.pk = *pk;
  d.tiles_per_band = rp.tiles_per_band; d.nbands = rp.nbands;
  h->dispatch = d;
  h->dispatched = true;
  CK(cudaMemcpyAsync(ds, hs, sizeof(StepDev) * n, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(h->ev_steps[par], st));
  h->steps_pending[par] = true;

  cudaEvent_t e0 = next_event(h), e1 = next_event(h), e2 = next_event(h);
  if (!e0 || !e1 || !e2) { h->err = "cudaEventCreate"; return LEC_ERR_CUDA; }
  CK(cudaEventRecord(e0, st));
  TmaMaps maps;
  if (d.kernel == LEC_ROWS_TILED) {
    const bool f64 = h->desc.dtype == LEC_F64;
    const int C = f64 ? 64 : 128, V = f64 ? 2 : 4, R = d.tile_rows;
    // box widths of TileGeom: int16 boxes have 8 more columns and a 16-byte halo on each side (aligned box starts)
    const int esz = pk ? 2 : f64 ? 8 : 4, PW = pk ? C + 8 : C, HV = pk ? 8 : V;
    bool ok = make_map(&maps.t_halo, fields[0], esz, nlon, nrows, L, nslots, PW + 2 * HV, R + 2) &&
              make_map(&maps.t_plain, fields[0], esz, nlon, nrows, L, nslots, PW, R) &&
              make_map(&maps.u, fields[1], esz, nlon, nrows, L, nslots, PW, R) &&
              make_map(&maps.v, fields[2], esz, nlon, nrows, L, nslots, PW, R) &&
              make_map(&maps.w, fields[3], esz, nlon, nrows, L, nslots, PW, R) &&
              make_map(&maps.f, fields[4], esz, nlon, nrows, L, nslots, PW, R);
    if (!ok) { h->err = "cuTensorMapEncodeTiled failed"; return LEC_ERR_CUDA; }
  }
  const cudaError_t le = launch_rows(h, d, rp, maps, grid, st);
  if (le != cudaSuccess) {
    h->err = std::string(d.kernel == LEC_ROWS_TILED ? "tiled row kernel launch: " : "cudaGetLastError(): ") + cudaGetErrorString(le);
    return LEC_ERR_CUDA;
  }
  CK(cudaEventRecord(e1, st));
  FinParams fp{};
  fp.g = gd; fp.steps = ds; fp.rec = h->d_rec; fp.max_ny = h->max_ny;
  fp.out_terms = out_terms; fp.out_levels = out_levels; fp.out_flags = out_flags; fp.out_bnd = out_bnd;
  fp.fin = h->d_fin; fp.nsteps = n;
  const int fgrid = (n * L + kFinThreads / 32 - 1) / (kFinThreads / 32);
  lec_fin_means_kernel<<<fgrid, kFinThreads, 0, st>>>(fp);
  lec_fin_sums_kernel<<<fgrid, kFinThreads, 0, st>>>(fp);
  lec_fin_integrate_kernel<<<n, 64, 0, st>>>(fp);
  CK(cudaGetLastError());
  CK(cudaEventRecord(e2, st));
  h->launches += 4;
  return LEC_OK;
}

// lec_run_device and lec_run_device_packed after their argument checks
static int run_device_impl(lec_handle* h, const void* const fields[5], int32_t nslots, const lec_step* steps,
                           int32_t nsteps, double* out_terms, double* out_levels, int32_t* out_flags, void* stream,
                           int pitch = 0, const PackedDev* pk = nullptr) {
  CK(cudaSetDevice(h->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int L = h->desc.nlev;
  if (!h->accumulate_timing || h->ev_used > 3 * 4096) h->ev_used = 0;
  h->call_timed = true;
  CK(cudaEventRecord(h->ev_call0, st));
  for (int s0 = 0; s0 < nsteps; s0 += h->max_steps) {
    const int n = std::min(h->max_steps, nsteps - s0);
    const int rc = run_batch(h, fields, nslots, steps + s0, n, out_terms + (size_t)s0 * LEC_NTERMS,
                             out_levels ? out_levels + (size_t)s0 * LEC_NLEVEL_TERMS * L : nullptr,
                             out_flags ? out_flags + s0 : nullptr,
                             h->bnd_user ? h->bnd_user + (size_t)s0 * kNB * L : nullptr, st, pitch, pk);
    if (rc != LEC_OK) return rc;
  }
  CK(cudaEventRecord(h->ev_call1, st));
  return LEC_OK;
}

int lec_run_device(lec_handle* h, const void* const fields[5], int32_t nslots, const lec_step* steps,
                   int32_t nsteps, double* out_terms, double* out_levels, int32_t* out_flags, void* stream) {
  if (h && nsteps == 0) return LEC_OK;      // an empty batch: nothing to launch, the (empty) outputs may be NULL
  if (!h || !fields || !steps || nsteps < 0 || nslots < 1 || !out_terms) return LEC_ERR_INVALID;
  for (int f = 0; f < 5; ++f) if (!fields[f]) return LEC_ERR_INVALID;
  return run_device_impl(h, fields, nslots, steps, nsteps, out_terms, out_levels, out_flags, stream);
}

int lec_run_device_packed(lec_handle* h, const lec_packed_desc* pd, const int16_t* const fields[5], int32_t nslots,
                          const lec_step* steps, int32_t nsteps, double* out_terms, double* out_levels,
                          int32_t* out_flags, void* stream) {
  if (h && nsteps == 0) return LEC_OK;
  if (!h || !pd || !fields || !steps || nsteps < 0 || nslots < 1 || !out_terms) return LEC_ERR_INVALID;
  if (pd->pitch < h->desc.nlon || pd->pitch % 8 != 0) {
    h->err = "pitch must be at least nlon and a multiple of 8 elements (16-byte rows)";
    return LEC_ERR_INVALID;
  }
  IngestParams dec[5];
  if (const int rc = read_decode(h, *pd, true, dec)) return rc;
  PackedDev pk{};
  const void* ptrs[5];
  for (int f = 0; f < 5; ++f) {
    if (!fields[f] || reinterpret_cast<uintptr_t>(fields[f]) % 16 != 0) {
      h->err = "int16 fields must be 16-byte aligned device pointers";
      return LEC_ERR_INVALID;
    }
    pk.scale[f] = dec[f].scale; pk.offset[f] = dec[f].offset; pk.round32[f] = dec[f].round32;
    pk.fill0[f] = (int)dec[f].fill0; pk.fill1[f] = (int)dec[f].fill1;
    ptrs[f] = fields[f];
  }
  pk.ntab = (h->desc.nlon + 3) & ~3;
  return run_device_impl(h, ptrs, nslots, steps, nsteps, out_terms, out_levels, out_flags, stream, pd->pitch, &pk);
}

// Where lec_run_host* takes its slots from: engine-layout host arrays, or raw records + index maps.
struct HostSource {
  const void* const* fields = nullptr;
  const lec_raw_desc* raw = nullptr;
  IngestParams dec[5] = {};                            // read_decode of raw; none for engine-layout arrays
  const int32_t* slot_record = nullptr;
  int nrecords = 0;
  int jr_lo = 0, jr_hi = 0, kr_lo = 0, kr_hi = 0;     // raw rows / levels the maps touch
};

// lec_set_host_windows: the window of every slot of one lec_run_host* call.  A rectangle of global columns x0..x1 and
// rows y0..y1 (x1 < x0: the slot is not read), and for raw records the part of a record it is decoded from: raw rows
// jr0 .. jr0 + nj - 1 of every touched level, raw columns rc0 .. rc0 + rw - 1.
struct Rect { int x0 = 0, x1 = -1, y0 = 0, y1 = -1; int jr0 = 0, nj = 0, rc0 = 0, rw = 0; };
struct HostWindows {
  int rows = 0, pitch = 0;                 // the shape all slots share
  std::vector<Rect> t, c;                  // per slot: T (= the slot's window: its origin), u / v / omega / Phi
  std::vector<int> ox, oy;                 // per slot: origin of the window
};

// The windows of a call (header: lec_set_host_windows).  The row kernels read, around a box, the T rows j - 1 / j + 1
// of its interior rows and the lon neighbours of its interior columns -- all inside the box -- and load (tiled kernel:
// the halo rows and the 16-byte lon-halo vector of every tile; every kernel: the pad columns of a box's edge chunks)
// values outside it that never reach a result.  So a window is the union of the boxes, its column origin rounded down
// to a 128-bit chunk so that window chunks are grid chunks (the lane <-> column map, and with it every sum, keeps its
// order).
static void host_windows(const lec_handle* h, const HostSource& src, int nslots, const lec_step* steps, int nsteps,
                         HostWindows& w) {
  const int vecw = h->desc.dtype == LEC_F64 ? 2 : 4;
  w.t.assign(nslots, Rect{}); w.c.assign(nslots, Rect{});
  auto grow = [](Rect& r, const lec_step& s) {
    if (r.x1 < r.x0) { r.x0 = s.i0; r.x1 = s.i1; r.y0 = s.j0; r.y1 = s.j1; return; }
    r.x0 = std::min(r.x0, s.i0); r.x1 = std::max(r.x1, s.i1); r.y0 = std::min(r.y0, s.j0); r.y1 = std::max(r.y1, s.j1);
  };
  for (int n = 0; n < nsteps; ++n) {
    const lec_step& s = steps[n];
    grow(w.c[s.slot], s); grow(w.t[s.slot], s); grow(w.t[s.slot_m], s); grow(w.t[s.slot_p], s);
  }
  w.rows = w.pitch = 0;
  w.ox.assign(nslots, 0); w.oy.assign(nslots, 0);
  for (int sl = 0; sl < nslots; ++sl) {
    for (Rect* r : {&w.t[sl], &w.c[sl]}) {
      if (r->x1 < r->x0) continue;
      r->x0 -= r->x0 % vecw;
      if (src.raw) {                      // raw rows of the window rows; raw columns if they are one increasing run
        const int* lat = src.raw->lat_map + r->y0;
        const int* lon = src.raw->lon_map + r->x0;
        int lo = lat[0], hi = lat[0];
        for (int j = 1; j <= r->y1 - r->y0; ++j) { lo = std::min(lo, lat[j]); hi = std::max(hi, lat[j]); }
        r->jr0 = lo; r->nj = hi - lo + 1;
        bool run = true;
        for (int i = 1; i <= r->x1 - r->x0 && run; ++i) run = lon[i] == lon[0] + i;
        r->rc0 = run ? lon[0] : 0; r->rw = run ? r->x1 - r->x0 + 1 : src.raw->nlon;
      }
    }
    const Rect& t = w.t[sl];
    if (t.x1 < t.x0) continue;
    w.ox[sl] = t.x0; w.oy[sl] = t.y0;
    w.rows = std::max(w.rows, t.y1 - t.y0 + 1);
    w.pitch = std::max(w.pitch, (t.x1 - t.x0 + vecw) / vecw * vecw);
  }
}

// The ingest kernel over ip (raw element type of r, the handle's field type) on s_ingest.
static void launch_ingest(const lec_handle* h, const lec_raw_desc& r, const IngestParams& ip, dim3 grid) {
  const bool f64 = h->desc.dtype == LEC_F64;
  if (r.dtype == LEC_RAW_I16) {
    if (f64) lec_ingest_kernel<short, double><<<grid, kIngestThreads, 0, h->s_ingest>>>(ip);
    else lec_ingest_kernel<short, float><<<grid, kIngestThreads, 0, h->s_ingest>>>(ip);
  } else if (r.dtype == LEC_RAW_F32) {
    lec_ingest_kernel<float, float><<<grid, kIngestThreads, 0, h->s_ingest>>>(ip);
  } else {
    lec_ingest_kernel<double, double><<<grid, kIngestThreads, 0, h->s_ingest>>>(ip);
  }
}

// stage_field with windows: the rectangle of field f of every slot in [s_lo, s_hi] that has one, into that slot's
// window (slot s at position s - win_lo of stage[b][f]), on s_copy.  Engine-layout arrays: one 3-D copy per slot.  Raw
// records: one 3-D copy of the rectangle's raw rows (and raw columns, when they are one run) of every touched level,
// then the ingest kernel over the rectangle.
static int stage_field_windows(lec_handle* h, const HostSource& src, const HostWindows& w, int f, int b, int win_lo,
                               int s_lo, int s_hi, size_t slot_bytes) {
  const int L = h->desc.nlev;
  const size_t elem = h->elem;
  const std::vector<Rect>& rects = f == 0 ? w.t : w.c;
  for (int s = s_lo; s <= s_hi; ++s) {
    const Rect& q = rects[s];
    if (q.x1 < q.x0) continue;
    const int nx = q.x1 - q.x0 + 1, ny = q.y1 - q.y0 + 1;
    char* slot_dst = static_cast<char*>(h->stage[b][f]) + (size_t)(s - win_lo) * slot_bytes;
    if (!src.raw) {
      cudaMemcpy3DParms cp{};
      cp.srcPtr = make_cudaPitchedPtr(const_cast<void*>(src.fields[f]), h->desc.nlon * elem, h->desc.nlon * elem, h->desc.nlat);
      cp.srcPos = make_cudaPos(q.x0 * elem, q.y0, (size_t)s * L);
      cp.dstPtr = make_cudaPitchedPtr(slot_dst, w.pitch * elem, w.pitch * elem, w.rows);
      cp.dstPos = make_cudaPos((q.x0 - w.ox[s]) * elem, q.y0 - w.oy[s], 0);
      cp.extent = make_cudaExtent(nx * elem, ny, L);
      cp.kind = cudaMemcpyHostToDevice;
      CK(cudaMemcpy3DAsync(&cp, h->s_copy));
      h->h2d_bytes += (long long)L * ny * nx * (long long)elem;
      continue;
    }
    const lec_raw_desc& r = *src.raw;
    const size_t relem = r.dtype == LEC_RAW_I16 ? 2 : r.dtype == LEC_RAW_F32 ? 4 : 8;
    const int nk = src.kr_hi - src.kr_lo + 1;
    const size_t row_bytes = (size_t)r.nlon * relem, rec_bytes = row_bytes * r.nlat * r.nlev;
    const size_t rec_stride = r.record_stride[f] > 0 ? (size_t)r.record_stride[f] : rec_bytes;
    const char* rec = static_cast<const char*>(src.fields[f]) + (size_t)src.slot_record[s] * rec_stride;
    const int rb = int(h->raw_seq & 1);
    if (h->raw_seq >= 2) CK(cudaStreamWaitEvent(h->s_copy, h->ev_raw_free[rb], 0));   // its last ingest has read it
    ++h->raw_seq;
    cudaMemcpy3DParms cp{};
    cp.srcPtr = make_cudaPitchedPtr(const_cast<char*>(rec), row_bytes, row_bytes, r.nlat);
    cp.srcPos = make_cudaPos(q.rc0 * relem, q.jr0, src.kr_lo);
    cp.dstPtr = make_cudaPitchedPtr(h->raw_stage[rb], q.rw * relem, q.rw * relem, q.nj);
    cp.dstPos = make_cudaPos(0, 0, 0);
    cp.extent = make_cudaExtent(q.rw * relem, q.nj, nk);
    cp.kind = cudaMemcpyHostToDevice;
    CK(cudaMemcpy3DAsync(&cp, h->s_copy));
    h->h2d_bytes += (long long)nk * q.nj * q.rw * (long long)relem;
    CK(cudaEventRecord(h->ev_raw_ready[rb], h->s_copy));
    CK(cudaStreamWaitEvent(h->s_ingest, h->ev_raw_ready[rb], 0));
    IngestParams ip = src.dec[f];
    // the maps from the rectangle's origin on; the source pointer is shifted so that raw column rc0 is its element 0
    ip.lon_map = h->d_maps + q.x0; ip.lat_map = h->d_maps + h->desc.nlon + q.y0;
    ip.lev_map = h->d_maps + h->desc.nlon + h->desc.nlat;
    ip.nlon = nx; ip.nlat = w.rows; ip.nlev = L; ip.pitch = w.pitch;      // (nlat: rows per level of the window)
    ip.rlon = q.rw; ip.nj_raw = q.nj; ip.jr_lo = q.jr0; ip.kr_lo = src.kr_lo;
    ip.big_endian = r.big_endian != 0;
    ip.src = static_cast<const char*>(h->raw_stage[rb]) - (ptrdiff_t)q.rc0 * (ptrdiff_t)relem;
    ip.dst = slot_dst + ((size_t)(q.y0 - w.oy[s]) * w.pitch + (q.x0 - w.ox[s])) * elem;
    launch_ingest(h, r, ip, dim3((nx + 4 * kIngestThreads - 1) / (4 * kIngestThreads), ny, L));
    CK(cudaEventRecord(h->ev_raw_free[rb], h->s_ingest));
    CK(cudaGetLastError());
    ++h->launches;
  }
  return LEC_OK;
}

// Bring engine slots [s_lo, s_hi] of field f into stage[b][f] (slot s at position s - win_lo), on s_copy.
static int stage_field(lec_handle* h, const HostSource& src, int f, int b, int win_lo, int s_lo, int s_hi,
                       size_t slot_bytes) {
  if (s_hi < s_lo) return LEC_OK;
  char* dst = static_cast<char*>(h->stage[b][f]) + (size_t)(s_lo - win_lo) * slot_bytes;
  if (!src.raw) {
    CK(cudaMemcpyAsync(dst, static_cast<const char*>(src.fields[f]) + (size_t)s_lo * slot_bytes,
                       (size_t)(s_hi - s_lo + 1) * slot_bytes, cudaMemcpyHostToDevice, h->s_copy));
    h->h2d_bytes += (long long)(s_hi - s_lo + 1) * (long long)slot_bytes;
    return LEC_OK;
  }
  const lec_raw_desc& r = *src.raw;
  const size_t relem = r.dtype == LEC_RAW_I16 ? 2 : r.dtype == LEC_RAW_F32 ? 4 : 8;
  const int nj = src.jr_hi - src.jr_lo + 1, nk = src.kr_hi - src.kr_lo + 1;
  const size_t row_bytes = (size_t)r.nlon * relem, rec_bytes = row_bytes * r.nlat * r.nlev;
  IngestParams ip = src.dec[f];
  ip.lon_map = h->d_maps; ip.lat_map = h->d_maps + h->desc.nlon; ip.lev_map = ip.lat_map + h->desc.nlat;
  ip.nlon = h->desc.nlon; ip.nlat = h->desc.nlat; ip.nlev = h->desc.nlev; ip.pitch = h->pitch;
  ip.rlon = r.nlon; ip.nj_raw = nj; ip.jr_lo = src.jr_lo; ip.kr_lo = src.kr_lo;
  ip.big_endian = r.big_endian != 0;
  const size_t rec_stride = r.record_stride[f] > 0 ? (size_t)r.record_stride[f] : rec_bytes;
  const dim3 grid((h->desc.nlon + 4 * kIngestThreads - 1) / (4 * kIngestThreads), h->desc.nlat, h->desc.nlev);
  for (int s = s_lo; s <= s_hi; ++s) {
    const char* rec = static_cast<const char*>(src.fields[f]) + (size_t)src.slot_record[s] * rec_stride;
    const int rb = int(h->raw_seq & 1);
    if (h->raw_seq >= 2) CK(cudaStreamWaitEvent(h->s_copy, h->ev_raw_free[rb], 0));   // its last ingest has read it
    ++h->raw_seq;
    if (nj == r.nlat) {        // whole planes: the level range is one contiguous block
      CK(cudaMemcpyAsync(h->raw_stage[rb], rec + (size_t)src.kr_lo * row_bytes * r.nlat, (size_t)nk * nj * row_bytes,
                         cudaMemcpyHostToDevice, h->s_copy));
    } else {                   // row range of every level: one strided 3-D copy
      cudaMemcpy3DParms cp{};
      cp.srcPtr = make_cudaPitchedPtr(const_cast<char*>(rec), row_bytes, row_bytes, r.nlat);
      cp.srcPos = make_cudaPos(0, src.jr_lo, src.kr_lo);
      cp.dstPtr = make_cudaPitchedPtr(h->raw_stage[rb], row_bytes, row_bytes, nj);
      cp.dstPos = make_cudaPos(0, 0, 0);
      cp.extent = make_cudaExtent(row_bytes, nj, nk);
      cp.kind = cudaMemcpyHostToDevice;
      CK(cudaMemcpy3DAsync(&cp, h->s_copy));
    }
    h->h2d_bytes += (long long)nk * nj * (long long)row_bytes;
    CK(cudaEventRecord(h->ev_raw_ready[rb], h->s_copy));
    CK(cudaStreamWaitEvent(h->s_ingest, h->ev_raw_ready[rb], 0));
    ip.src = h->raw_stage[rb];
    ip.dst = dst + (size_t)(s - s_lo) * slot_bytes;
    launch_ingest(h, r, ip, grid);
    CK(cudaEventRecord(h->ev_raw_free[rb], h->s_ingest));
    CK(cudaGetLastError());
    ++h->launches;
  }
  return LEC_OK;
}

static int run_host_impl(lec_handle* h, HostSource& src, int32_t nslots, const lec_step* steps, int32_t nsteps,
                         double* out_terms, double* out_levels, int32_t* out_flags) {
  CK(cudaSetDevice(h->device));
  const int L = h->desc.nlev;
  // The engine's own slots have rows padded to whole 128-bit chunks, so the vector / sub-warp kernels run
  // for every grid width.  Engine-layout host arrays whose rows are not such a multiple take the ingest
  // route too (identity maps): a contiguous H2D copy per slot, then a device pass that re-pitches it.
  // With windows (lec_set_host_windows) a staged slot is one window of every level instead, for both sources.
  HostWindows win;
  const bool windows = h->host_windows != 0;
  if (windows) {                       // the windows come from every step: check them first (as build_step does)
    for (int s = 0; s < nsteps; ++s)
      if (const int rc = check_step(h, steps[s], nslots)) { h->err = "step " + std::to_string(s) + ": bad slot or box"; return rc; }
    host_windows(h, src, nslots, steps, nsteps, win);
  }
  const size_t slot_bytes = windows ? (size_t)L * win.rows * win.pitch * h->elem
                                    : (size_t)L * h->desc.nlat * h->pitch * h->elem;
  lec_raw_desc ident;
  std::vector<int32_t> iota;
  if (!src.raw && h->pitch != h->desc.nlon && !windows) {
    const int m = std::max(std::max(h->desc.nlon, h->desc.nlat), std::max(L, (int)nslots));
    iota.resize(m);
    for (int i = 0; i < m; ++i) iota[i] = i;
    std::memset(&ident, 0, sizeof ident);
    ident.dtype = h->desc.dtype == LEC_F64 ? LEC_RAW_F64 : LEC_RAW_F32;
    ident.nlon = h->desc.nlon; ident.nlat = h->desc.nlat; ident.nlev = L;
    ident.lon_map = ident.lat_map = ident.lev_map = iota.data();
    src.raw = &ident; src.slot_record = iota.data(); src.nrecords = nslots;
    src.jr_lo = 0; src.jr_hi = h->desc.nlat - 1; src.kr_lo = 0; src.kr_hi = L - 1;
  }
  if (!h->s_copy) {
    CK(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      CK(cudaEventCreateWithFlags(&h->ev_copied[b], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&h->ev_done[b], cudaEventDisableTiming));
    }
  }
  if (src.raw) {
    const lec_raw_desc& r = *src.raw;
    const size_t relem = r.dtype == LEC_RAW_I16 ? 2 : r.dtype == LEC_RAW_F32 ? 4 : 8;
    size_t need = (size_t)(src.kr_hi - src.kr_lo + 1) * (src.jr_hi - src.jr_lo + 1) * r.nlon * relem;
    if (windows) {                     // the largest window part of a record
      need = 0;
      for (const std::vector<Rect>* rs : {&win.t, &win.c})
        for (const Rect& q : *rs)
          if (q.x0 <= q.x1) need = std::max(need, (size_t)(src.kr_hi - src.kr_lo + 1) * q.nj * q.rw * relem);
    }
    if (!h->s_ingest) {
      CK(cudaStreamCreateWithFlags(&h->s_ingest, cudaStreamNonBlocking));
      for (int b = 0; b < 2; ++b) {
        CK(cudaEventCreateWithFlags(&h->ev_raw_ready[b], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&h->ev_raw_free[b], cudaEventDisableTiming));
      }
      CK(cudaEventCreateWithFlags(&h->ev_ingested, cudaEventDisableTiming));
    }
    if (h->raw_stage_bytes < need) {
      CK(cudaStreamSynchronize(h->s_ingest));
      for (int b = 0; b < 2; ++b) {
        cudaFree(h->raw_stage[b]); h->raw_stage[b] = nullptr;
      }
      h->raw_stage_bytes = 0; h->raw_seq = 0;
      for (int b = 0; b < 2; ++b)
        if (cudaMalloc(&h->raw_stage[b], need) != cudaSuccess) { cudaGetLastError(); h->err = "raw staging buffer"; return LEC_ERR_NOMEM; }
      h->raw_stage_bytes = need;
    }
    const int nmap = h->desc.nlon + h->desc.nlat + L;
    if (!h->d_maps) CK(cudaMalloc(&h->d_maps, sizeof(int) * nmap));
    // (pageable source: the copies return once the driver has staged the maps)
    CK(cudaMemcpyAsync(h->d_maps, r.lon_map, sizeof(int) * h->desc.nlon, cudaMemcpyHostToDevice, h->s_copy));
    CK(cudaMemcpyAsync(h->d_maps + h->desc.nlon, r.lat_map, sizeof(int) * h->desc.nlat, cudaMemcpyHostToDevice, h->s_copy));
    CK(cudaMemcpyAsync(h->d_maps + h->desc.nlon + h->desc.nlat, r.lev_map, sizeof(int) * L, cudaMemcpyHostToDevice, h->s_copy));
  }
  // Staging window: as many slots as this call can use (nslots, max_steps + 2 halo slots) within the byte
  // budget.  A reused handle whose earlier call was shorter gets a larger window here -- the window of the
  // first call must not cap the later ones (a 1- or 2-slot window cannot hold slot_m, slot, slot_p).
  // (Windows make a staged slot smaller, so the same buffers hold more of them: the window counts in slots of this
  // call's size.)
  long long stage_slots = (long long)(h->stage_cap / slot_bytes);
  if (stage_slots < std::min<long long>((long long)h->max_steps + 2, nslots)) {
    long long budget = h->desc.host_stage_bytes;
    if (budget <= 0) {
      size_t fr = 0, tot = 0;
      CK(cudaMemGetInfo(&fr, &tot));
      fr += h->stage_cap * 10;                                  // what the old window gives back
      budget = (long long)std::min<size_t>(fr / 4, (size_t)32 << 30);
    }
    long long slots = budget / (long long)(2 * 5 * slot_bytes);
    slots = std::min<long long>(slots, (long long)h->max_steps + 2);
    slots = std::min<long long>(slots, nslots);
    if (slots < 1) { h->err = "host_stage_bytes too small for one slot"; return LEC_ERR_NOMEM; }
    if (slots > stage_slots) {
      if (h->stage[0][0]) {            // nothing of an earlier call may still read or write the old window
        CK(cudaStreamSynchronize(h->s_copy));
        CK(cudaStreamSynchronize(h->s_comp));
        if (h->s_ingest) CK(cudaStreamSynchronize(h->s_ingest));
      }
      for (int b = 0; b < 2; ++b)
        for (int f = 0; f < 5; ++f) { cudaFree(h->stage[b][f]); h->stage[b][f] = nullptr; }
      h->stage_cap = 0;
      for (int b = 0; b < 2; ++b)
        for (int f = 0; f < 5; ++f)
          if (cudaMalloc(&h->stage[b][f], (size_t)slots * slot_bytes) != cudaSuccess) {
            cudaGetLastError(); h->err = "staging buffers"; return LEC_ERR_NOMEM;
          }
      h->stage_cap = (size_t)slots * slot_bytes;
      stage_slots = slots;
    }
  }
  if (h->out_cap < nsteps) {
    cudaFree(h->d_out_terms); cudaFree(h->d_out_levels); cudaFree(h->d_out_flags);
    h->d_out_terms = h->d_out_levels = nullptr; h->d_out_flags = nullptr; h->out_cap = 0;
    CK(cudaMalloc(&h->d_out_terms, sizeof(double) * LEC_NTERMS * nsteps));
    CK(cudaMalloc(&h->d_out_levels, sizeof(double) * LEC_NLEVEL_TERMS * L * nsteps));
    CK(cudaMalloc(&h->d_out_flags, sizeof(int) * nsteps));
    h->out_cap = nsteps;
  }
  if (h->bnd_user && h->bnd_cap < nsteps) {
    cudaFree(h->d_out_bnd); h->d_out_bnd = nullptr; h->bnd_cap = 0;
    CK(cudaMalloc(&h->d_out_bnd, sizeof(double) * kNB * L * nsteps));
    h->bnd_cap = nsteps;
  }
  if (!h->accumulate_timing || h->ev_used > 3 * 4096) h->ev_used = 0;
  h->call_timed = true;
  CK(cudaEventRecord(h->ev_call0, h->s_copy));

  std::vector<lec_step> local;
  int s0 = 0, chunk = 0, prev_lo = 0, prev_hi = -1;
  h->h2d_bytes = h->d2h_bytes = 0;
  while (s0 < nsteps) {
    // greedy chunk: as many steps as share a slot window of <= stage_slots
    int lo = 1 << 30, hi = -1, s1 = s0;
    while (s1 < nsteps && s1 - s0 < h->max_steps) {
      const lec_step& s = steps[s1];
      if (s.slot < 0 || s.slot >= nslots || s.slot_m < 0 || s.slot_m >= nslots || s.slot_p < 0 || s.slot_p >= nslots)
        return LEC_ERR_BOUNDS;
      const int nlo = std::min(std::min(lo, s.slot), std::min(s.slot_m, s.slot_p));
      const int nhi = std::max(std::max(hi, s.slot), std::max(s.slot_m, s.slot_p));
      if (nhi - nlo + 1 > stage_slots) break;
      lo = nlo; hi = nhi; ++s1;
    }
    if (s1 == s0) { h->err = "one step needs more slots than the staging window holds"; return LEC_ERR_NOMEM; }
    const int b = chunk & 1;
    // the buffer is free once the batch that last used it has finished
    if (chunk >= 2) {
      CK(cudaStreamWaitEvent(h->s_copy, h->ev_done[b], 0));
      if (src.raw) CK(cudaStreamWaitEvent(h->s_ingest, h->ev_done[b], 0));
    }
    // T needs the whole window (centre slots and their time neighbours); the slots the previous chunk
    // already brought over are copied device-to-device from its buffer instead of crossing PCIe again
    int t_lo = lo;
    if (chunk >= 1 && lo >= prev_lo && lo <= prev_hi) {
      const int ov_hi = std::min(prev_hi, hi);
      CK(cudaMemcpyAsync(h->stage[b][0], static_cast<const char*>(h->stage[b ^ 1][0]) + (size_t)(lo - prev_lo) * slot_bytes,
                         (size_t)(ov_hi - lo + 1) * slot_bytes, cudaMemcpyDeviceToDevice, h->s_copy));
      t_lo = ov_hi + 1;
    }
    auto stage = [&](int f, int s_lo, int s_hi) {
      return windows ? stage_field_windows(h, src, win, f, b, lo, s_lo, s_hi, slot_bytes)
                     : stage_field(h, src, f, b, lo, s_lo, s_hi, slot_bytes);
    };
    { const int rc = stage(0, t_lo, hi); if (rc != LEC_OK) return rc; }
    // u, v, omega, Phi are read at the centre slots only
    int c_lo = 1 << 30, c_hi = -1;
    for (int s = s0; s < s1; ++s) { c_lo = std::min(c_lo, steps[s].slot); c_hi = std::max(c_hi, steps[s].slot); }
    for (int f = 1; f < 5; ++f) {
      const int rc = stage(f, c_lo, c_hi);
      if (rc != LEC_OK) return rc;
    }
    prev_lo = lo; prev_hi = hi;
    if (src.raw) {             // the copy stream joins the ingest stream: the chunk is staged when both are done
      CK(cudaEventRecord(h->ev_ingested, h->s_ingest));
      CK(cudaStreamWaitEvent(h->s_copy, h->ev_ingested, 0));
    }
    CK(cudaEventRecord(h->ev_copied[b], h->s_copy));
    CK(cudaStreamWaitEvent(h->s_comp, h->ev_copied[b], 0));
    local.assign(steps + s0, steps + s1);
    for (lec_step& s : local) { s.slot -= lo; s.slot_m -= lo; s.slot_p -= lo; }
    const WinView wv{win.rows, win.pitch, windows ? win.ox.data() + lo : nullptr, windows ? win.oy.data() + lo : nullptr};
    const int rc = run_batch(h, h->stage[b], hi - lo + 1, local.data(), s1 - s0,
                             h->d_out_terms + (size_t)s0 * LEC_NTERMS,
                             h->d_out_levels + (size_t)s0 * LEC_NLEVEL_TERMS * L, h->d_out_flags + s0,
                             h->bnd_user ? h->d_out_bnd + (size_t)s0 * kNB * L : nullptr, h->s_comp, h->pitch,
                             nullptr, windows ? &wv : nullptr);
    if (rc != LEC_OK) return rc;
    CK(cudaEventRecord(h->ev_done[b], h->s_comp));
    s0 = s1; ++chunk;
  }
  CK(cudaMemcpyAsync(out_terms, h->d_out_terms, sizeof(double) * LEC_NTERMS * nsteps, cudaMemcpyDeviceToHost, h->s_comp));
  if (out_levels)
    CK(cudaMemcpyAsync(out_levels, h->d_out_levels, sizeof(double) * LEC_NLEVEL_TERMS * L * nsteps,
                       cudaMemcpyDeviceToHost, h->s_comp));
  if (out_flags)
    CK(cudaMemcpyAsync(out_flags, h->d_out_flags, sizeof(int) * nsteps, cudaMemcpyDeviceToHost, h->s_comp));
  if (h->bnd_user)
    CK(cudaMemcpyAsync(h->bnd_user, h->d_out_bnd, sizeof(double) * kNB * L * nsteps, cudaMemcpyDeviceToHost, h->s_comp));
  h->d2h_bytes = (h->bnd_user ? (long long)sizeof(double) * kNB * L * nsteps : 0) +
                 (long long)sizeof(double) * LEC_NTERMS * nsteps +
                 (out_levels ? (long long)sizeof(double) * LEC_NLEVEL_TERMS * L * nsteps : 0) +
                 (out_flags ? (long long)sizeof(int) * nsteps : 0);
  CK(cudaEventRecord(h->ev_call1, h->s_comp));
  CK(cudaStreamSynchronize(h->s_comp));
  CK(cudaStreamSynchronize(h->s_copy));
  return LEC_OK;
}

int lec_run_host(lec_handle* h, const void* const fields[5], int32_t nslots, const lec_step* steps,
                 int32_t nsteps, double* out_terms, double* out_levels, int32_t* out_flags) {
  if (h && nsteps == 0) { h->h2d_bytes = h->d2h_bytes = 0; return LEC_OK; }
  if (!h || !fields || !steps || nsteps < 0 || nslots < 1 || !out_terms) return LEC_ERR_INVALID;
  for (int f = 0; f < 5; ++f) if (!fields[f]) return LEC_ERR_INVALID;
  HostSource src;
  src.fields = fields;
  return run_host_impl(h, src, nslots, steps, nsteps, out_terms, out_levels, out_flags);
}

int lec_run_host_raw(lec_handle* h, const lec_raw_desc* rd, const void* const raw[5], int32_t nrecords,
                     const int32_t* slot_record, int32_t nslots, const lec_step* steps, int32_t nsteps,
                     double* out_terms, double* out_levels, int32_t* out_flags) {
  if (h && nsteps == 0) { h->h2d_bytes = h->d2h_bytes = 0; return LEC_OK; }
  if (!h || !rd || !raw || !slot_record || !steps || nsteps < 0 || nslots < 1 || nrecords < 1 || !out_terms ||
      !rd->lon_map || !rd->lat_map || !rd->lev_map || rd->nlon < 1 || rd->nlat < 1 || rd->nlev < 1)
    return LEC_ERR_INVALID;
  for (int f = 0; f < 5; ++f) if (!raw[f] || rd->record_stride[f] < 0) return LEC_ERR_INVALID;
  if (rd->dtype != LEC_RAW_F32 && rd->dtype != LEC_RAW_F64 && rd->dtype != LEC_RAW_I16) return LEC_ERR_INVALID;
  if ((rd->dtype == LEC_RAW_F32 && h->desc.dtype != LEC_F32) || (rd->dtype == LEC_RAW_F64 && h->desc.dtype != LEC_F64)) {
    h->err = "raw float records need a handle of the same float type";
    return LEC_ERR_INVALID;
  }
  HostSource src;
  if (const int rc = read_decode(h, *rd, rd->dtype == LEC_RAW_I16, src.dec)) return rc;
  src.fields = raw; src.raw = rd; src.slot_record = slot_record; src.nrecords = nrecords;
  auto range = [](const int32_t* m, int n, int limit, int& lo, int& hi) {
    lo = 1 << 30; hi = -1;
    for (int i = 0; i < n; ++i) { if (m[i] < 0 || m[i] >= limit) return false; lo = std::min(lo, (int)m[i]); hi = std::max(hi, (int)m[i]); }
    return true;
  };
  int ilo, ihi;
  if (!range(rd->lon_map, h->desc.nlon, rd->nlon, ilo, ihi) || !range(rd->lat_map, h->desc.nlat, rd->nlat, src.jr_lo, src.jr_hi) ||
      !range(rd->lev_map, h->desc.nlev, rd->nlev, src.kr_lo, src.kr_hi))
    return LEC_ERR_BOUNDS;
  for (int s = 0; s < nslots; ++s) if (slot_record[s] < 0 || slot_record[s] >= nrecords) return LEC_ERR_BOUNDS;
  return run_host_impl(h, src, nslots, steps, nsteps, out_terms, out_levels, out_flags);
}

int lec_pin_host(void* ptr, int64_t bytes) {
  if (!ptr || bytes <= 0) return LEC_ERR_INVALID;
  const cudaError_t e = cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterPortable);
  if (e != cudaSuccess) {
    cudaGetLastError();
    g_free_err = std::string("cudaHostRegister: ") + cudaGetErrorString(e);
    return LEC_ERR_CUDA;
  }
  return LEC_OK;
}

int lec_unpin_host(void* ptr) {
  if (!ptr) return LEC_ERR_INVALID;
  const cudaError_t e = cudaHostUnregister(ptr);
  if (e != cudaSuccess) {
    cudaGetLastError();
    g_free_err = std::string("cudaHostUnregister: ") + cudaGetErrorString(e);
    return LEC_ERR_CUDA;
  }
  return LEC_OK;
}

int lec_set_host_windows(lec_handle* h, int32_t on) {
  if (!h || (on != 0 && on != 1)) return LEC_ERR_INVALID;
  h->host_windows = on;
  return LEC_OK;
}

int lec_set_boundary_levels(lec_handle* h, double* out) {
  if (!h) return LEC_ERR_INVALID;
  h->bnd_user = out;
  return LEC_OK;
}

int lec_timing_reset(lec_handle* h) {
  if (!h) return LEC_ERR_INVALID;
  h->ev_used = 0;
  h->accumulate_timing = true;
  return LEC_OK;
}

int lec_last_timing(lec_handle* h, float out_ms[3]) {
  if (!h || !out_ms) return LEC_ERR_INVALID;
  out_ms[0] = out_ms[1] = out_ms[2] = 0.f;
  if (!h->call_timed) return LEC_OK;
  CK(cudaSetDevice(h->device));
  CK(cudaEventSynchronize(h->ev_call1));
  for (int i = 0; i + 2 < h->ev_used; i += 3) {
    float a = 0.f, b = 0.f;
    CK(cudaEventElapsedTime(&a, h->ev_pool[i], h->ev_pool[i + 1]));
    CK(cudaEventElapsedTime(&b, h->ev_pool[i + 1], h->ev_pool[i + 2]));
    out_ms[0] += a; out_ms[1] += b;
  }
  // the whole-call events may sit on different streams (host path): elapsed time is still defined
  CK(cudaEventElapsedTime(&out_ms[2], h->ev_call0, h->ev_call1));
  return LEC_OK;
}

// ---- 850-hPa track diagnostics (handle-free) ---------------------------------------------------------
namespace {

#define CKF(call)                                                                  \
  do {                                                                             \
    cudaError_t e__ = (call);                                                      \
    if (e__ != cudaSuccess) {                                                      \
      g_free_err = std::string(#call) + ": " + cudaGetErrorString(e__);            \
      rc = LEC_ERR_CUDA;                                                           \
      goto done;                                                                   \
    }                                                                              \
  } while (0)

// MetPy first_derivative(f, delta=d) as a 3-point stencil per index: out[i] = A f[s] + B f[s+1] + C f[s+2],
// s = clamp(i - 1, 0, n - 3); coefficients written exactly as metpy/calc/tools.py writes them (signs folded:
// x - c f == x + (-c) f bit for bit).
struct DiagAxisHost {
  std::vector<double> A, B, C;
  DiagAxisHost(const double* d, int n) : A(n), B(n), C(n) {          // d[n-1] grid deltas
    for (int i = 1; i + 1 < n; ++i) {
      const double d0 = d[i - 1], d1 = d[i], comb = d0 + d1;
      A[i] = -d1 / (comb * d0); B[i] = (d1 - d0) / (d0 * d1); C[i] = d0 / (comb * d1);
    }
    {
      const double d0 = d[0], d1 = d[1], comb = d0 + d1, big = comb + d0;
      A[0] = -big / (comb * d0); B[0] = comb / (d0 * d1); C[0] = -(d0 / (comb * d1));
    }
    {
      const double d0 = d[n - 3], d1 = d[n - 2], comb = d0 + d1, big = comb + d1;
      A[n - 1] = d1 / (comb * d0); B[n - 1] = -(comb / (d0 * d1)); C[n - 1] = big / (comb * d1);
    }
  }
};

// win_rows / win_cols / origin: the planes are windows of the domain, origin[2 s] = (column, row) of slot s's
// window (lec_diag850_host_windows); origin NULL: whole-domain planes.
int diag850_run(const lec_diag_grid* g, const void* u, const void* v, const void* z, int32_t nslots,
                const lec_diag_step* steps, int32_t nsteps, double* out_val, int32_t* out_idx, cudaStream_t st,
                bool host_io, int win_rows = 0, int win_cols = 0, const int32_t* origin = nullptr) {
  if (!g || !u || !v || !z || !steps || !out_val || !out_idx || nsteps < 0 || nslots < 1 || !g->dx || !g->dy ||
      !g->parallel_scale || !g->meridional_scale || (g->dtype != LEC_F32 && g->dtype != LEC_F64))
    return LEC_ERR_INVALID;
  if (g->nlon < 3 || g->nlat < 3) return LEC_ERR_DEGENERATE;
  if (nsteps == 0) return LEC_OK;
  for (int s = 0; s < nsteps; ++s) {
    const lec_diag_step& q = steps[s];
    if (q.slot < 0 || q.slot >= nslots || q.i0 < 0 || q.i1 >= g->nlon || q.i0 > q.i1 || q.j0 < 0 || q.j1 >= g->nlat ||
        q.j0 > q.j1 || q.ic >= g->nlon || q.jc >= g->nlat)
      return LEC_ERR_BOUNDS;
  }
  if (origin) {        // every value the kernel reads must lie inside the step's window (header: the window rule)
    if (win_rows < 1 || win_cols < 1) return LEC_ERR_INVALID;
    for (int s = 0; s < nsteps; ++s) {
      const lec_diag_step& q = steps[s];
      const int ox = origin[2 * q.slot], oy = origin[2 * q.slot + 1];
      // columns / rows the 3-point stencils of the box points (and of the centre point) read
      auto span = [](int a, int b, int n, int& lo, int& hi) {
        lo = std::min(std::max(a - 1, 0), n - 3); hi = std::max(std::min(b + 1, n - 1), 2);
      };
      int xl, xh, yl, yh;
      span(q.ic >= 0 && q.jc >= 0 ? std::min(q.i0, q.ic) : q.i0, q.ic >= 0 && q.jc >= 0 ? std::max(q.i1, q.ic) : q.i1,
           g->nlon, xl, xh);
      span(q.ic >= 0 && q.jc >= 0 ? std::min(q.j0, q.jc) : q.j0, q.ic >= 0 && q.jc >= 0 ? std::max(q.j1, q.jc) : q.j1,
           g->nlat, yl, yh);
      if (xl < ox || xh >= ox + win_cols || yl < oy || yh >= oy + win_rows) {
        g_free_err = "a step reads outside its window";
        return LEC_ERR_BOUNDS;
      }
    }
  }
  int rc = LEC_OK;
  const int nx = g->nlon, ny = g->nlat;
  const size_t elem = g->dtype == LEC_F64 ? 8 : 4;
  const int ld = origin ? win_cols : nx;
  const long long plane = origin ? (long long)win_rows * win_cols : (long long)ny * nx;
  const size_t plane_bytes = (size_t)nslots * plane * elem;
  DiagAxisHost ax(g->dx, nx), ay(g->dy, ny);
  // one table upload: [ax.A ax.B ax.C | ay.A ay.B ay.C | k | h | (h/k) dk/dy | k/h] then the steps
  std::vector<double> tab;
  tab.insert(tab.end(), ax.A.begin(), ax.A.end()); tab.insert(tab.end(), ax.B.begin(), ax.B.end());
  tab.insert(tab.end(), ax.C.begin(), ax.C.end());
  tab.insert(tab.end(), ay.A.begin(), ay.A.end()); tab.insert(tab.end(), ay.B.begin(), ay.B.end());
  tab.insert(tab.end(), ay.C.begin(), ay.C.end());
  tab.insert(tab.end(), g->parallel_scale, g->parallel_scale + ny);
  tab.insert(tab.end(), g->meridional_scale, g->meridional_scale + ny);
  for (int j = 0; j < ny; ++j) {       // dx_correction = meridional_scale / parallel_scale * first_derivative(parallel_scale, dy)
    const int sj = std::min(std::max(j - 1, 0), ny - 3);
    const double* k = g->parallel_scale;
    const double dkdy = ((ay.A[j] * k[sj]) + (ay.B[j] * k[sj + 1])) + (ay.C[j] * k[sj + 2]);
    tab.push_back(g->meridional_scale[j] / g->parallel_scale[j] * dkdy);
  }
  for (int j = 0; j < ny; ++j) tab.push_back(g->parallel_scale[j] / g->meridional_scale[j]);
  double* d_tab = nullptr; DiagStepDev* d_steps = nullptr; double* d_val = nullptr; int* d_idx = nullptr;
  void* d_f[3] = {nullptr, nullptr, nullptr};
  const void* src[3] = {u, v, z};
  std::vector<DiagStepDev> hs(nsteps);
  for (int s = 0; s < nsteps; ++s)
    hs[s] = DiagStepDev{steps[s].slot, steps[s].i0, steps[s].i1, steps[s].j0, steps[s].j1, steps[s].ic, steps[s].jc,
                        origin ? origin[2 * steps[s].slot] : 0, origin ? origin[2 * steps[s].slot + 1] : 0};
  DiagParams p{};
  CKF(cudaSetDevice(g->device));
  CKF(cudaMalloc(&d_tab, tab.size() * sizeof(double)));
  CKF(cudaMalloc(&d_steps, sizeof(DiagStepDev) * nsteps));
  CKF(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice, st));
  CKF(cudaMemcpyAsync(d_steps, hs.data(), sizeof(DiagStepDev) * nsteps, cudaMemcpyHostToDevice, st));
  if (host_io) {
    for (int f = 0; f < 3; ++f) {
      CKF(cudaMalloc(&d_f[f], plane_bytes));
      CKF(cudaMemcpyAsync(d_f[f], src[f], plane_bytes, cudaMemcpyHostToDevice, st));
    }
    CKF(cudaMalloc(&d_val, sizeof(double) * LEC_NDIAG_VALUES * nsteps));
    CKF(cudaMalloc(&d_idx, sizeof(int) * LEC_NDIAG * nsteps));
  }
  p.u = host_io ? d_f[0] : u; p.v = host_io ? d_f[1] : v; p.z = host_io ? d_f[2] : z;
  p.ax = DiagAxis{d_tab, d_tab + nx, d_tab + 2 * nx, nx};
  p.ay = DiagAxis{d_tab + 3 * nx, d_tab + 3 * nx + ny, d_tab + 3 * nx + 2 * ny, ny};
  p.ps = d_tab + 3 * nx + 3 * ny; p.ms = p.ps + ny; p.dxcorr = p.ms + ny; p.pm = p.dxcorr + ny;
  p.su = g->scale[0]; p.sv = g->scale[1]; p.sz = g->scale[2]; p.zdiv = g->z_div;
  p.steps = d_steps; p.out_val = host_io ? d_val : out_val; p.out_idx = host_io ? d_idx : out_idx;
  p.nlon = nx; p.nlat = ny; p.ld = ld; p.plane = plane;
  if (g->dtype == LEC_F64) lec_diag850_kernel<double><<<nsteps, kDiagThreads, 0, st>>>(p);
  else lec_diag850_kernel<float><<<nsteps, kDiagThreads, 0, st>>>(p);
  CKF(cudaGetLastError());
  if (host_io) {
    CKF(cudaMemcpyAsync(out_val, d_val, sizeof(double) * LEC_NDIAG_VALUES * nsteps, cudaMemcpyDeviceToHost, st));
    CKF(cudaMemcpyAsync(out_idx, d_idx, sizeof(int) * LEC_NDIAG * nsteps, cudaMemcpyDeviceToHost, st));
  }
  CKF(cudaStreamSynchronize(st));     // the tables and the step list are freed below
done:
  cudaFree(d_tab); cudaFree(d_steps); cudaFree(d_val); cudaFree(d_idx);
  for (int f = 0; f < 3; ++f) cudaFree(d_f[f]);
  return rc;
}

}  // namespace

int lec_diag850_device(const lec_diag_grid* grid, const void* u, const void* v, const void* z, int32_t nslots,
                       const lec_diag_step* steps, int32_t nsteps, double* out_val, int32_t* out_idx, void* cuda_stream) {
  return diag850_run(grid, u, v, z, nslots, steps, nsteps, out_val, out_idx, static_cast<cudaStream_t>(cuda_stream), false);
}

int lec_diag850_host(const lec_diag_grid* grid, const void* u, const void* v, const void* z, int32_t nslots,
                     const lec_diag_step* steps, int32_t nsteps, double* out_val, int32_t* out_idx) {
  return diag850_run(grid, u, v, z, nslots, steps, nsteps, out_val, out_idx, nullptr, true);
}

int lec_diag850_host_windows(const lec_diag_grid* grid, const void* u, const void* v, const void* z, int32_t nslots,
                             int32_t win_rows, int32_t win_cols, const int32_t* origin, const lec_diag_step* steps,
                             int32_t nsteps, double* out_val, int32_t* out_idx) {
  if (!origin) return LEC_ERR_INVALID;
  return diag850_run(grid, u, v, z, nslots, steps, nsteps, out_val, out_idx, nullptr, true, win_rows, win_cols, origin);
}

}  // extern "C"
