// Shared definitions of the B200 Lorenz Energy Cycle engine (device + host).
//
// Data layout in HBM (DESIGN.md section 3):
//   fields      5 x [slot][level][lat][lon]   storage dtype (fp32 | fp64), C-contiguous
//   row records [step][level][row][LEC_NREC]  fp64, written by the row-moment kernel,
//               read by the finalize kernel
//   results     [step][LEC_NTERMS], [step][LEC_NLEVEL_TERMS][level]   fp64
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace lec {

// MetPy 1.6.2 constants (metpy/constants/default.py), as used by
// src/utils/thermodynamics.py:22 and src/analysis/*.py of the reference.
constexpr double kG = 9.80665;
constexpr double kRe = 6371008.7714;
constexpr double kRd = 8.314462618 / 28.96546e-3;
constexpr double kCp = 1.4 * kRd / (1.4 - 1.0);
constexpr double kKappa = kRd / kCp;
constexpr double kP0 = 100000.0;
constexpr double kDeg2Rad = 3.14159265358979323846 / 180.0;

// ---- row record (one per step, level and box row) -------------------------
// Shifted zonal trapezoid sums  S_xy = sum_i w_i x_i y_i  with x = X - shift_X
// (a=T, b=u, c=v, w=omega, f=Phi; q=Q unshifted) -- 22 values, then the five
// shifts (= the raw west edge values), then the raw east edge values of u, v, T.
enum RecIdx {
  R_A = 0, R_B, R_C, R_W, R_F, R_Q,
  R_AA, R_BB, R_CC, R_BC, R_CA, R_WA, R_WB, R_WC, R_WF, R_QA,
  R_CAA, R_WAA, R_BBC, R_CCC, R_BBW, R_CCW,
  R_NSUM,                                    // = 22
  R_SH_T = R_NSUM, R_SH_U, R_SH_V, R_SH_W, R_SH_F,
  R_UE, R_VE, R_TE,                          // (the west edge values ARE the shifts: first box value of the row)
  R_COUNT                                    // = 30
};
constexpr int LEC_NREC = 30;                 // an even count (16-byte rows)
static_assert(R_COUNT <= LEC_NREC, "record too small");

// One time step of work, device form (built on the host from lec_step).
struct StepDev {
  int slot, slot_m, slot_p;
  int i0, i1, j0, j1;
  int rec_base;            // first record row of this step: rec + (rec_base * nlev * max_ny ...)
  double ct_m, ct_p, ct_s; // cp sT dT/dt = ct_m (T_m - T) + ct_p (T_p - T) + ct_s T,  ct_s ~ ct_m+ct_0+ct_p
  double cxW, cxE;         // one-sided d/dlon at the box edges, folded with 1/(deg2rad(1) Re)
  double wW, wE;           // trapezoid weights (rlon) of the two edge columns
  double cyS, cyN;         // one-sided d/dlat at the box edges, folded with cp sT sV / dy
  double inv_xlen, inv_ylen, c1, c2;
  // fp32 copies for the fp32-arithmetic row kernels (no double -> float conversions in the row set-up);
  // f_wWn / f_wEn are the edge weights relative to the uniform interior weight (LONW == 0)
  float f_ct_m, f_ct_p, f_ct_s, f_cxW, f_cxE, f_wW, f_wE, f_wWn, f_wEn, f_cyS, f_cyN, f_pad;
  // Fields are addressed in the coordinates of each slot's window (lec_set_host_windows; origin 0 and window = grid
  // otherwise): global column i, row j of slot s sit at window column i - ox(s), row j - oy(s).  Box indices and the
  // grid tables stay global.  ox, oy: window origin of the centre slot; oxm, oym / oxp, oyp: of slot_m / slot_p (the
  // tiled kernel's TMA coordinates); d_m, d_p: element offset of T(slot_m) / T(slot_p) from T(slot) at the same
  // global point (the direct and sub-warp kernels; the host checks that they fit 31 bits).
  int ox, oy, oxm, oym, oxp, oyp;
  int d_m, d_p;
};

// Grid tables resident on the device (all fp64; built once in lec_create).
struct GridDev {
  int nlon, nlat, nlev;
  // longitude [nlon]
  const double* wl;        // interior trapezoid weight 0.5 (rlon[i+1] - rlon[i-1])
  const double* cxa;       // interior d/dlon stencil: cxa (T[i-1]-T[i]) + cxc (T[i+1]-T[i]),
  const double* cxc;       //   folded with 1/(deg2rad(gradient(lon)) Re)
  const float* wl32;       // fp32 copies of the three longitude tables (fp32 arithmetic)
  const float* cxa32;
  const float* cxc32;
  const float* cya32;      // fp32 copies of the per-row / per-level coefficient tables
  const float* cyc32;
  const float* fxj32;
  const float* sm32;
  const float* sp32;
  const float* ss32;
  float cxa_u32, cxc_u32;
  // latitude [nlat]
  const double* rlat;
  const double* coslat;
  const double* tanlat;
  const double* cya;       // interior d/dlat stencil folded with cp sT sV / dy_j
  const double* cyc;
  const double* fxj;       // cp sT sU / cos(lat_j): row factor of the d/dlon stencil
  const double* fya;       // np.gradient coefficients w.r.t. rlat (interior rows)
  const double* fyc;
  // level [nlev]
  const double* plev;
  const double* pa;        // np.gradient coefficients w.r.t. p incl. the one-sided ends
  const double* pc;
  double p_2h;             // 2 h when the whole level axis is exactly uniform (np.gradient's uniform branch), else 0
  const double* sm;        // -cp sT sW S,  S = sm (T[k-1]-T) + sp (T[k+1]-T) + ss T  (stability term of Q)
  const double* sp;
  const double* ss;
  int lon_uniform;         // trapezoid weights AND lon stencil -- 2: exactly constant; 1: constant to 1e-6
                           // (enough for fp32 arithmetic); 0: tables needed.  Scalars below = constants
  int stencil_uniform;     // the same classification for the lon stencil alone (degree axis)
  double wl_u, cxa_u, cxc_u;
  double scale[5];         // namelist unit -> SI factor per field
};

}  // namespace lec
