// Kernel A of the LEC engine: the only HBM-heavy kernel.
//
// One warp owns one box row (step, level, lat) and sweeps it along longitude in
// 128-bit chunks.  In a SINGLE pass over T, u, v, omega, Phi it evaluates
//   * the diabatic-heating residual Q pointwise (thermodynamics.py:76-124): centred
//     differences in lon/lat/p/t on T written in difference form a(T[-1]-T)+c(T[+1]-T)
//     so fp32 arithmetic does not cancel; every constant factor (cp, 1/dx, 1/dy, unit
//     scales, 1/cos(lat)) is folded into per-row coefficients, leaving 21 flops per point,
//   * the 22 shifted zonal trapezoid moments of lec_common.cuh (the zonal means and every
//     eddy product of box_data.py:157-231 / src/analysis/*.py follow from them exactly),
//   * the raw west/east edge values needed by boundary_terms.py.
// Shifted single-pass moments (shift = first box value of the row) replace the
// reference's "mean first, anomalies second" two passes: the central moments are
// recovered in fp64 by the finalize kernel, so no rounded mean ever biases the anomalies.
// Only the first and last sweep iteration of a row can touch the box edges (masked
// columns, half trapezoid weights, one-sided d/dlon); the iterations in between run a
// branch-free body.  Lanes reduce with a 23-shuffle fp64 halving butterfly; the sum order
// is fixed, so results are bit-reproducible across launches, shards and GPUs.
#pragma once
#include "lec_common.cuh"
#include "lec_pair.cuh"

namespace lec {

constexpr int kRowsPerCta = 2;                // warps per CTA, one row each (adjacent rows share L1 lines)
constexpr int kRowThreads = kRowsPerCta * 32;

// Division of a 31-bit numerator by a run-time constant as one wide multiply and a shift (the block / tile index is
// decoded by every warp: three hardware-emulated 32-bit divides are ~60 instructions).  Host side: make().
struct FastDiv {
  unsigned mul;   // floor(2^(31 + L) / d) + 1,  L = ceil(log2 d)
  unsigned shr;   // 31 + L
  unsigned d;
  static FastDiv make(unsigned d) {
    FastDiv f;
    unsigned L = 0;
    while ((1ull << L) < d) ++L;
    f.mul = (unsigned)(((1ull << (31 + L)) / d) + 1ull);
    f.shr = 31 + L;
    f.d = d;
    return f;
  }
  // n < 2^31 (the hosts guarantee grid < 2^31): exact
  __device__ __forceinline__ unsigned div(unsigned n) const { return (unsigned)(((unsigned long long)n * mul) >> shr); }
  __device__ __forceinline__ unsigned divmod(unsigned n, unsigned& rem) const {
    const unsigned q = div(n);
    rem = n - q * d;
    return q;
  }
};

// Decode of int16 fields resident in device memory (lec_run_device_packed), per field: the rule of lec_ingest_kernel
// with the switches folded into the constants (no scale: 1.0; no offset: -0.0, which adds exactly nothing, signed
// zeros included) and the fill values as raw integers (kNoFill never matches an int16).
constexpr int kNoFill = 0x10000;
struct PackedDev {
  double scale[5], offset[5];
  int fill0[5], fill1[5];
  int round32[5];          // fp64 fields: the decoded variable is float32 (rounded once)
  int ntab;                // longitude-table entries of the tiled kernel's shared copy (the row pitch may be longer)
};

struct RowParams {
  const void* field[5];
  GridDev g;
  const StepDev* steps;
  double* rec;
  int nsteps;
  int max_ny;            // record rows reserved per (step, level)
  int nbands;            // (read by the host only)
  int tiles_per_band;    // CTA row-tiles per latitude band
  FastDiv dv_tiles, dv_lev, dv_steps;   // block / tile index -> (band, step, level, row tile)
  long long slot_stride; // elements per slot = nlev * lev_stride
  long long lev_stride;  // elements per level of a slot: rows * row_stride (the window's rows, or nlat)
  int row_stride;        // elements per row (the window's pitch, or the fields' row length)
  long long grid;        // number of CTAs
  PackedDev pk;          // int16 instances only
};

// TMA bulk prefetch of a byte range into L2 (no destination, no completion tracking).
__device__ __forceinline__ void prefetch_l2_range(const void* p, long long lo_byte, long long hi_byte) {
  // the instruction wants a 16-byte aligned address and size: shrink the range to whole
  // 16-byte units of the ABSOLUTE address (it is only a hint; never reach outside the row)
  const unsigned long long a0 = reinterpret_cast<unsigned long long>(p) + (unsigned long long)lo_byte;
  const unsigned long long a1 = reinterpret_cast<unsigned long long>(p) + (unsigned long long)hi_byte;
  const unsigned long long lo = (a0 + 15ULL) & ~15ULL, hi = a1 & ~15ULL;
  if (hi <= lo) return;
  const unsigned n = unsigned(hi - lo);
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(lo), "r"(n) : "memory");
}

template <typename FT, int VEC> struct VecLoad;
template <> struct VecLoad<float, 4> {
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  static __device__ __forceinline__ void ld_stream(const float* p, float (&v)[4]) {
    float4 t = __ldcs(reinterpret_cast<const float4*>(p)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
};
template <> struct VecLoad<double, 2> {
  static __device__ __forceinline__ void ld(const double* p, double (&v)[2]) {
    double2 t = __ldg(reinterpret_cast<const double2*>(p)); v[0] = t.x; v[1] = t.y; }
  static __device__ __forceinline__ void ld_stream(const double* p, double (&v)[2]) {
    double2 t = __ldcs(reinterpret_cast<const double2*>(p)); v[0] = t.x; v[1] = t.y; }
};
template <typename FT> struct VecLoad<FT, 1> {
  static __device__ __forceinline__ void ld(const FT* p, FT (&v)[1]) { v[0] = __ldg(p); }
  static __device__ __forceinline__ void ld_stream(const FT* p, FT (&v)[1]) { v[0] = __ldcs(p); }
};

// One int16 element of field F decoded to FT: x = double(raw) * scale + offset (two roundings, no FMA), rounded
// through float32 where the decoded variable is float32, NaN for a fill value -- lec_ingest_kernel's rule, so the
// row kernels see the bits lec_run_device sees on the decoded fields.  (A float32 FT rounds once anyway.)
// NAN_OR: how a float32 value becomes NaN -- a select, or an integer OR into x (the same bits); which of the two
// builds without spills depends on the kernel (ptxas: the sub-warp kernel wants the select, the tiled one the OR).
template <typename FT, int F, bool NAN_OR = false>
__device__ __forceinline__ FT unpack_i16(short raw, const PackedDev& pk) {
  const double x = __dadd_rn(__dmul_rn(double(raw), pk.scale[F]), pk.offset[F]);
  const bool fill = int(raw) == pk.fill0[F] || int(raw) == pk.fill1[F];
  if constexpr (sizeof(FT) == 8) {
    return fill ? __longlong_as_double(0x7ff8000000000000LL) : pk.round32[F] ? double(float(x)) : x;
  } else if constexpr (NAN_OR) {
    // a fill sets the exponent and quiet bit of x: a NaN, whose float32 conversion is the canonical NaN
    return float(__hiloint2double(__double2hiint(x) | (fill ? 0x7ff80000 : 0), __double2loint(x)));
  } else {
    return fill ? __int_as_float(0x7fffffff) : float(x);    // = float(NaN)
  }
}

template <typename FT, int VEC, int F, bool NAN_OR = false>
__device__ __forceinline__ void unpack_i16_vec(unsigned lo, unsigned hi, FT (&v)[VEC], const PackedDev& pk) {
  v[0] = unpack_i16<FT, F, NAN_OR>(short(lo & 0xffffu), pk);
  v[1] = unpack_i16<FT, F, NAN_OR>(short(lo >> 16), pk);
  if constexpr (VEC == 4) {
    v[2] = unpack_i16<FT, F, NAN_OR>(short(hi & 0xffffu), pk);
    v[3] = unpack_i16<FT, F, NAN_OR>(short(hi >> 16), pk);
  }
}

// Global loads of the row kernels by stored element type ST: the float types load as stored (VecLoad); int16 loads
// the lane's VEC values (8 bytes for fp32, 4 for fp64) and decodes them.  F = field (LEC_FIELD_*).
template <typename ST, typename FT, int VEC>
struct RowLoad {
  template <int F> static __device__ __forceinline__ void ld(const ST* p, FT (&v)[VEC], const PackedDev&) { VecLoad<FT, VEC>::ld(p, v); }
  template <int F> static __device__ __forceinline__ FT one(const ST* p, const PackedDev&) { return __ldg(p); }
};
template <typename FT, int VEC>
struct RowLoad<short, FT, VEC> {
  static_assert(VEC == 4 || VEC == 2, "int16 rows are read in the chunks of the vector kernels");
  template <int F> static __device__ __forceinline__ void ld(const short* p, FT (&v)[VEC], const PackedDev& pk) {
    if constexpr (VEC == 4) {
      const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
      unpack_i16_vec<FT, VEC, F>(t.x, t.y, v, pk);
    } else {
      unpack_i16_vec<FT, VEC, F>(__ldg(reinterpret_cast<const unsigned*>(p)), 0u, v, pk);
    }
  }
  template <int F> static __device__ __forceinline__ FT one(const short* p, const PackedDev& pk) { return unpack_i16<FT, F>(__ldg(p), pk); }
};

__device__ __forceinline__ double shfl_xor_f64(double v, int m) {
  return __shfl_xor_sync(0xffffffffu, v, m);
}

// Halving butterfly: N values per lane -> lane L ends with the full-warp sum of value
// bitrev5(L) (zero for indices >= N).  23 shuffles for N = 22 instead of 110.
template <int N>
__device__ __forceinline__ double butterfly_reduce(double (&v)[N], int lane) {
  static_assert(N <= 32, "at most one value per lane");
  double a[32];
#pragma unroll
  for (int i = 0; i < 32; ++i) a[i] = (i < N) ? v[i] : 0.0;
  int n = 32;
#pragma unroll
  for (int bit = 16; bit >= 1; bit >>= 1) {
    n >>= 1;
    const bool hi = (lane & bit) != 0;
#pragma unroll
    for (int i = 0; i < n; ++i) {
      // statically skip pairs that are known to be all-zero padding
      const int live = (N + (32 / (2 * n)) - 1) / (32 / (2 * n));   // live values before this step
      if (2 * i < live) {
        const double keep = hi ? a[2 * i + 1] : a[2 * i];
        const double send = hi ? a[2 * i] : a[2 * i + 1];
        a[i] = keep + shfl_xor_f64(send, bit);
      } else {
        a[i] = 0.0;
      }
    }
  }
  return a[0];
}

__device__ __forceinline__ int bitrev5(int x) {
  return ((x & 1) << 4) | ((x & 2) << 2) | (x & 4) | ((x & 8) >> 2) | ((x & 16) >> 4);
}

// Per-row constants of the pointwise Q, every factor folded (rounded once to CT).
template <typename CT>
struct RowCoefS {
  CT ct_m, ct_p, ct_s;     // cp * sT * time stencil
  CT cy_m, cy_p;           // cp * sT * sV * lat stencil / dy
  CT s_m, s_p, s_s;        // -cp * sT * sW * static-stability stencil
  CT fx;                   // cp * sT * sU / cos(lat): multiplies the lon stencil
};

constexpr int R_NLIN = 6;   // the linear sums S_a .. S_q carry a compensation term in fp32 arithmetic

// s += x with the rounding error of the addition collected in c (FastTwoSum: exact when |s| >= |x|, i.e.
// whenever the error matters).  COMP is chosen per launch: the compensation matters when a lane adds many
// chunks (long rows) while the terms are built from small differences of zonal means (a box of few rows);
// fp64 arithmetic needs none.
template <typename CT, bool COMP>
__device__ __forceinline__ void lec_lin_add(CT& s, CT& c, CT x) {
  if constexpr (sizeof(CT) == 4 && COMP) {
    const CT t = s + x;
    c += x - (t - s);
    s = t;
  } else {
    s += x;
  }
}

// 22 moment updates of one grid point (weight already applied to the W* operands).
template <typename CT, bool COMP>
__device__ __forceinline__ void accumulate_s(CT (&S)[R_NSUM], CT (&Cc)[R_NLIN], CT Wa, CT Wb, CT Wc, CT Ww, CT Wf, CT Wq,
                                           CT a, CT b, CT c, CT w, CT f, CT q) {
  lec_lin_add<CT, COMP>(S[R_A], Cc[R_A], Wa); lec_lin_add<CT, COMP>(S[R_B], Cc[R_B], Wb); lec_lin_add<CT, COMP>(S[R_C], Cc[R_C], Wc);
  lec_lin_add<CT, COMP>(S[R_W], Cc[R_W], Ww); lec_lin_add<CT, COMP>(S[R_F], Cc[R_F], Wf); lec_lin_add<CT, COMP>(S[R_Q], Cc[R_Q], Wq);
  const CT pbb = Wb * b, pcc = Wc * c, pca = Wc * a, pwa = Ww * a;
  S[R_AA] += Wa * a; S[R_BB] += pbb; S[R_CC] += pcc; S[R_BC] += Wb * c;
  S[R_CA] += pca; S[R_WA] += pwa; S[R_WB] += Ww * b; S[R_WC] += Ww * c;
  S[R_WF] += Ww * f; S[R_QA] += Wa * q;
  S[R_CAA] += pca * a; S[R_WAA] += pwa * a; S[R_BBC] += pbb * c; S[R_CCC] += pcc * c;
  S[R_BBW] += pbb * w; S[R_CCW] += pcc * w;
}

// same, with the four shared products (Wb b, Wc c, Wc a, Ww a) computed by the caller (packed)
template <typename CT, bool COMP>
__device__ __forceinline__ void accumulate_pp(CT (&S)[R_NSUM], CT (&Cc)[R_NLIN], CT Wa, CT Wb, CT Wc, CT Ww, CT Wf, CT Wq,
                                              CT a, CT b, CT c, CT w, CT f, CT q, CT pbb, CT pcc, CT pca, CT pwa) {
  lec_lin_add<CT, COMP>(S[R_A], Cc[R_A], Wa); lec_lin_add<CT, COMP>(S[R_B], Cc[R_B], Wb); lec_lin_add<CT, COMP>(S[R_C], Cc[R_C], Wc);
  lec_lin_add<CT, COMP>(S[R_W], Cc[R_W], Ww); lec_lin_add<CT, COMP>(S[R_F], Cc[R_F], Wf); lec_lin_add<CT, COMP>(S[R_Q], Cc[R_Q], Wq);
  S[R_AA] += Wa * a; S[R_BB] += pbb; S[R_CC] += pcc; S[R_BC] += Wb * c;
  S[R_CA] += pca; S[R_WA] += pwa; S[R_WB] += Ww * b; S[R_WC] += Ww * c;
  S[R_WF] += Ww * f; S[R_QA] += Wa * q;
  S[R_CAA] += pca * a; S[R_WAA] += pwa * a; S[R_BBC] += pbb * c; S[R_CCC] += pcc * c;
  S[R_BBW] += pbb * w; S[R_CCW] += pcc * w;
}

// Row-level coefficients of one box row (step st, level k, row j): every constant factor was folded on the
// host (lec_engine.cu); fp32 arithmetic reads the fp32 copies of the tables, so the set-up has no
// double -> float conversions.  Edge columns: one-sided lon stencil; trapezoid weights relative to the
// uniform weight when LONW == 0.
template <typename CT, int LONW>
struct RowSetup {
  RowCoefS<CT> rc;
  CT cxa_u, cxc_u, cxW, cxE, wW, wE;
  double fxd;
  __device__ __forceinline__ void init(const RowParams& p, const StepDev* __restrict__ st, int j, int k, int j0, int j1) {
    if constexpr (sizeof(CT) == 4) {
      rc.ct_m = st->f_ct_m; rc.ct_p = st->f_ct_p; rc.ct_s = st->f_ct_s;
      rc.cy_m = (j == j0) ? 0.f : (j == j1) ? -st->f_cyN : __ldg(p.g.cya32 + j);
      rc.cy_p = (j == j1) ? 0.f : (j == j0) ? st->f_cyS : __ldg(p.g.cyc32 + j);
      rc.s_m = __ldg(p.g.sm32 + k); rc.s_p = __ldg(p.g.sp32 + k); rc.s_s = __ldg(p.g.ss32 + k);
      rc.fx = __ldg(p.g.fxj32 + j);
      fxd = 0.0;
      cxa_u = rc.fx * p.g.cxa_u32; cxc_u = rc.fx * p.g.cxc_u32;
      cxW = rc.fx * st->f_cxW; cxE = rc.fx * st->f_cxE;
      wW = (LONW == 0) ? st->f_wWn : st->f_wW; wE = (LONW == 0) ? st->f_wEn : st->f_wE;
    } else {
      rc.ct_m = st->ct_m; rc.ct_p = st->ct_p; rc.ct_s = st->ct_s;
      rc.cy_m = (j == j0) ? 0.0 : (j == j1) ? -st->cyN : p.g.cya[j];
      rc.cy_p = (j == j1) ? 0.0 : (j == j0) ? st->cyS : p.g.cyc[j];
      rc.s_m = p.g.sm[k]; rc.s_p = p.g.sp[k]; rc.s_s = p.g.ss[k];
      fxd = p.g.fxj[j];
      rc.fx = fxd;
      cxa_u = fxd * p.g.cxa_u; cxc_u = fxd * p.g.cxc_u;
      cxW = fxd * st->cxW; cxE = fxd * st->cxE;
      const double wnorm = (LONW == 0) ? 1.0 / p.g.wl_u : 1.0;
      wW = st->wW * wnorm; wE = st->wE * wnorm;
    }
  }
};

// LONW: 0 = uniform longitudes (weight applied once after the reduction), 1 = per-column trapezoid
// weights with a uniform lon stencil, 2 = per-column weights and stencil (irregular longitudes).
// CTAs per SM: 8 (16 warps), 6 (12 warps) for fp64 arithmetic and compensated fp32 sums
template <typename FT, typename CT, int VEC, int LONW, bool COMP>
__global__ void __launch_bounds__(kRowThreads, sizeof(CT) == 8 || COMP ? 6 : 8)
lec_row_moments_kernel(const RowParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA order: band-major, then step, level, row-tile.  Sweeping time inside a latitude
  // band keeps T(t+1) (first touched as the time neighbour of step t) in L2 until it is
  // the centre of step t+1 and the t-1 neighbour of step t+2.  (grid < 2^31: 32-bit divides)
  const unsigned bid = blockIdx.x;
  unsigned ujt, uk, us;
  const unsigned q1 = p.dv_tiles.divmod(bid, ujt);
  const unsigned q2 = p.dv_lev.divmod(q1, uk);
  const int band = int(p.dv_steps.divmod(q2, us));
  const int jt = int(ujt), k = int(uk), s = int(us);

  const StepDev* __restrict__ st = p.steps + s;
  const int i0 = st->i0, i1 = st->i1, j0 = st->j0, j1 = st->j1;
  const int jrel = (band * p.tiles_per_band + jt) * kRowsPerCta + warp;
  if (jrel > j1 - j0) return;                 // warp-uniform; no block barriers below
  const int j = j0 + jrel;
  const int nlon = p.row_stride, nlev = p.g.nlev;

  // One 64-bit base per field (the centre row, shifted by the window origin so that global columns index it); the six
  // T neighbours are 32-bit element offsets from the T base, so a load address is one IMAD.WIDE (the host checks the
  // offsets fit 31 bits).
  const long long plane = p.lev_stride;
  const long long row_c = ((long long)st->slot * nlev + k) * plane + (long long)(j - st->oy) * nlon - st->ox;
  const FT* __restrict__ Tc_row = static_cast<const FT*>(p.field[0]) + row_c;
  const FT* __restrict__ U_row = static_cast<const FT*>(p.field[1]) + row_c;
  const FT* __restrict__ V_row = static_cast<const FT*>(p.field[2]) + row_c;
  const FT* __restrict__ W_row = static_cast<const FT*>(p.field[3]) + row_c;
  const FT* __restrict__ F_row = static_cast<const FT*>(p.field[4]) + row_c;
  const int d_m = st->d_m, d_p = st->d_p;
  const int d_km = (k > 0) ? -int(plane) : 0, d_kp = (k < nlev - 1) ? int(plane) : 0;
  const int d_jm = (j > j0) ? -nlon : 0, d_jp = (j < j1) ? nlon : 0;

  // L2 prefetch of the rows that come from DRAM (u, v, omega, Phi of this step and T of the
  // next time slot; T of this slot was fetched as the time neighbour one step earlier; +9 % measured)
  if (lane < 5) {
    const FT* base = (lane == 0) ? Tc_row + d_p : static_cast<const FT*>(p.field[lane]) + row_c;
    prefetch_l2_range(base, (long long)i0 * sizeof(FT), (long long)(i1 + 1) * sizeof(FT));
  }

  RowSetup<CT, LONW> rs;
  rs.init(p, st, j, k, j0, j1);
  const RowCoefS<CT>& rc = rs.rc;
  const CT cxa_u = rs.cxa_u, cxc_u = rs.cxc_u, cxW = rs.cxW, cxE = rs.cxE, wW = rs.wW, wE = rs.wE;
  [[maybe_unused]] const double fxd = rs.fxd;
  const bool box_aligned = (i0 % VEC == 0) && ((i1 + 1) % VEC == 0);   // no partly-masked chunk in the row

  // shifts: raw first-in-box values of the row (broadcast loads)
  const FT shT = __ldg(Tc_row + i0), shU = __ldg(U_row + i0), shV = __ldg(V_row + i0),
           shW = __ldg(W_row + i0), shF = __ldg(F_row + i0);
  const CT cshT = CT(shT), cshU = CT(shU), cshV = CT(shV), cshW = CT(shW), cshF = CT(shF);

  CT S[R_NSUM], Cc[R_NLIN];
#pragma unroll
  for (int n = 0; n < R_NSUM; ++n) S[n] = CT(0);
#pragma unroll
  for (int n = 0; n < R_NLIN; ++n) Cc[n] = CT(0);

  double* __restrict__ rec = p.rec + (((long long)s * nlev + k) * p.max_ny + jrel) * LEC_NREC;

  const int c0 = i0 / VEC, c1 = i1 / VEC;
  const int niter = (c1 - c0 + 32) / 32;

  // one IMAD.WIDE per address: base (64-bit, in registers) + 32-bit element index x sizeof
  auto at = [](const FT* base, int idx) -> const FT* {
    unsigned long long a;
    asm("mad.wide.s32 %0, %1, %2, %3;" : "=l"(a) : "r"(idx), "r"((int)sizeof(FT)), "l"(base));
    return reinterpret_cast<const FT*>(a);
  };
  // The first and the last sweep iteration of a row are peeled: only they can touch the box edges or hold
  // lanes past the row end, so the iterations in between run a body without masks, clamps and selects.
  {
    const int it = 0;
#define LEC_BODY_EDGE 1
#include "lec_row_iter_direct.inc"
#undef LEC_BODY_EDGE
  }
  for (int it = 1; it < niter - 1; ++it) {
#define LEC_BODY_EDGE 0
#include "lec_row_iter_direct.inc"
#undef LEC_BODY_EDGE
  }
  if (niter > 1) {
    const int it = niter - 1;
#define LEC_BODY_EDGE 1
#include "lec_row_iter_direct.inc"
#undef LEC_BODY_EDGE
  }

  double Sd[R_NSUM];
#pragma unroll
  for (int n = 0; n < R_NSUM; ++n) Sd[n] = double(S[n]);
  if constexpr (sizeof(CT) == 4 && COMP) {
#pragma unroll
    for (int n = 0; n < R_NLIN; ++n) Sd[n] += double(Cc[n]);
  }
  double tot = butterfly_reduce<R_NSUM>(Sd, lane);
  if (LONW == 0) tot *= p.g.wl_u;
  const int idx = bitrev5(lane);
  if (idx < R_NSUM) rec[idx] = tot;
  if (lane == 1) {   // raw (unscaled) shifts; the finalize kernel applies the unit scales
    rec[R_SH_T] = double(shT); rec[R_SH_U] = double(shU); rec[R_SH_V] = double(shV);
    rec[R_SH_W] = double(shW); rec[R_SH_F] = double(shF);
  }
}

}  // namespace lec
