// Kernel B of the LEC engine: from row records to the Lorenz terms of one time step.
//
// One CTA per step.  Everything here is O(levels x box rows) fp64 work on the records
// written by lec_row_moments_kernel:
//   phase 1  area means [X] of the six zonal means, per level (calc_averages.py:46-78)
//            and sigma (thermodynamics.py:26-73, by linearity in T, floor 0.03)
//   phase 2  per level: cos(lat)-weighted meridional trapezoids of every integrand of
//            energy_contents.py / conversion_terms.py / boundary_terms.py /
//            generation_and_dissipation_terms.py, the plain-latitude trapezoids of the
//            east-minus-west fluxes, and the north/south edge rows
//   phase 3  per level integrands (the reference's per-level CSV families)
//   phase 4  trapezoidal integration over pressure, bottom-minus-top fluxes -> 16 scalars
#pragma once
#include "lec_common.cuh"
#include "lec_row_moments.cuh"   // butterfly_reduce, bitrev5

namespace lec {

constexpr int kFinThreads = 256;

// per-level meridional sums (phase 2)
enum SumIdx {
  SQ_AZ = 0, SQ_AE, SQ_KZ, SQ_KE, SQ_CZ2, SQ_CE2, SQ_CA1, SQ_CA2, SQ_CK1, SQ_CK2, SQ_CK3, SQ_CK4, SQ_CK5,
  SQ_GZ, SQ_GE, SQ_BAZ3, SQ_BAE3, SQ_BKZ3, SQ_BKE3, SQ_BOZ3, SQ_BOE3,
  Y_BAZ1, Y_BAE1, Y_BKZ1, Y_BKE1, Y_BOZ1, Y_BOE1,
  SQ_NSUM                                         // = 27
};
enum EdgeIdx { N_BAZ2 = 0, N_BAE2, N_BKZ2, N_BKE2, N_BOZ2, N_NEDGE };   // x2: north, south
// boundary pieces per level (phase 3): [term][E-W, N-S, vertical flux]
constexpr int kNB = 6 * 3;
constexpr int kLevStride = 6 /*AA*/ + 1 /*sigma*/ + SQ_NSUM + 2 * N_NEDGE + kNB;

struct FinParams {
  GridDev g;
  const StepDev* steps;
  const double* rec;
  int max_ny;
  double* fin;           // finalize scratch [nsteps][nlev][kLevStride]
  int nsteps;
  double* out_terms;     // [nsteps][16]
  double* out_levels;    // [nsteps][19][nlev] or nullptr
  int* out_flags;        // [nsteps] or nullptr
  double* out_bnd;       // [nsteps][18][nlev] or nullptr: per-level boundary pieces (lec_set_boundary_levels)
};

struct RowQ {
  double Tm, um, vm, wm, Fm, Qm;
  double TT, uu, vv, uv, vT, wT, wu, wv, wF, QT;
  double vTTc, wTTc, uuv, vvv, uuw, vvw;
  double uW, vW, TW, uE, vE, TE;
};

// A lane reads ITS OWN record (rows are 240 bytes apart: every load instruction of a warp touches 32 sectors), so
// the number of load instructions is what the finalize kernels pay for: 128-bit loads, and only the values needed.
static_assert(LEC_NREC % 2 == 0 && R_SH_T % 2 == 0, "records are read as 16-byte pairs");
template <int FIRST, int N>
__device__ __forceinline__ void rec_load(const double* r, double (&v)[N]) {
  static_assert(FIRST % 2 == 0 && N % 2 == 0, "whole 16-byte pairs");
#pragma unroll
  for (int i = 0; i < N; i += 2) {
    const double2 t = __ldg(reinterpret_cast<const double2*>(r + FIRST + i));
    v[i] = t.x; v[i + 1] = t.y;
  }
}
// zonal means of fields 0 .. NF-1 of another row / level: unit scale x (shift + shifted mean)
template <int NF>
__device__ __forceinline__ void rec_means(const double* r, double ix, const double* sc, double (&m)[NF]) {
  constexpr int NP = (NF + 1) / 2 * 2;
  double a[NP], sh[NP];
  rec_load<R_A, NP>(r, a);
  rec_load<R_SH_T, NP>(r, sh);
#pragma unroll
  for (int f = 0; f < NF; ++f) m[f] = sc[f] * (sh[f] + a[f] * ix);
}

// central zonal moments (SI units) from the raw shifted sums of one record
__device__ __forceinline__ void derive_row(const double* __restrict__ rg, double ix, const double* sc, RowQ& q) {
  double r[LEC_NREC];
  rec_load<0, LEC_NREC>(rg, r);
  const double sT = sc[0], sU = sc[1], sV = sc[2], sW = sc[3], sF = sc[4];
  const double ma = r[R_A] * ix * sT, mb = r[R_B] * ix * sU, mc = r[R_C] * ix * sV, mw = r[R_W] * ix * sW,
               mf = r[R_F] * ix * sF, mq = r[R_Q] * ix;
  q.Tm = r[R_SH_T] * sT + ma; q.um = r[R_SH_U] * sU + mb; q.vm = r[R_SH_V] * sV + mc;
  q.wm = r[R_SH_W] * sW + mw; q.Fm = r[R_SH_F] * sF + mf; q.Qm = mq;
  const double Saa = r[R_AA] * ix * (sT * sT), Sbb = r[R_BB] * ix * (sU * sU), Scc = r[R_CC] * ix * (sV * sV),
               Sbc = r[R_BC] * ix * (sU * sV), Sca = r[R_CA] * ix * (sV * sT), Swa = r[R_WA] * ix * (sW * sT),
               Swb = r[R_WB] * ix * (sW * sU), Swc = r[R_WC] * ix * (sW * sV);
  q.TT = Saa - ma * ma; q.uu = Sbb - mb * mb; q.vv = Scc - mc * mc; q.uv = Sbc - mb * mc;
  q.vT = Sca - mc * ma; q.wT = Swa - mw * ma; q.wu = Swb - mw * mb; q.wv = Swc - mw * mc;
  q.wF = r[R_WF] * ix * (sW * sF) - mw * mf;
  q.QT = r[R_QA] * ix * sT - mq * ma;
  // ZA(x'y'z') = Sxyz - mx Syz - my Sxz - mz Sxy + 2 mx my mz
  q.vTTc = r[R_CAA] * ix * (sV * sT * sT) - mc * Saa - 2.0 * ma * Sca + 2.0 * mc * ma * ma;
  q.wTTc = r[R_WAA] * ix * (sW * sT * sT) - mw * Saa - 2.0 * ma * Swa + 2.0 * mw * ma * ma;
  q.uuv = r[R_BBC] * ix * (sU * sU * sV) - mc * Sbb - 2.0 * mb * Sbc + 2.0 * mb * mb * mc;
  q.vvv = r[R_CCC] * ix * (sV * sV * sV) - 3.0 * mc * Scc + 2.0 * mc * mc * mc;
  q.uuw = r[R_BBW] * ix * (sU * sU * sW) - mw * Sbb - 2.0 * mb * Swb + 2.0 * mb * mb * mw;
  q.vvw = r[R_CCW] * ix * (sV * sV * sW) - mw * Scc - 2.0 * mc * Swc + 2.0 * mc * mc * mw;
  q.uW = r[R_SH_U] * sU; q.vW = r[R_SH_V] * sV; q.TW = r[R_SH_T] * sT;   // the shifts are the first box value of the row
  q.uE = r[R_UE] * sU; q.vE = r[R_VE] * sV; q.TE = r[R_TE] * sT;
}

// Scratch of the finalize kernels, per (step, level): [AA(6) | sigma | 27 sums | 2x5 edge rows | 18 boundary pieces]
struct FinCommon {
  int s, k, L, j0, j1, ny;
  double ix, iy;
};

#define LEC_FIN_PROLOGUE(SK)                                                                         \
  const int L = p.g.nlev;                                                                            \
  [[maybe_unused]] const int s = (SK) / L, k = (SK) - s * L;                                                          \
  const StepDev st = p.steps[s];                                                                     \
  [[maybe_unused]] const int j0 = st.j0, j1 = st.j1, ny = j1 - j0 + 1;                                                \
  [[maybe_unused]] const double ix = st.inv_xlen, iy = st.inv_ylen;                                                   \
  [[maybe_unused]] const double sc[5] = {p.g.scale[0], p.g.scale[1], p.g.scale[2], p.g.scale[3], p.g.scale[4]};       \
  [[maybe_unused]] const double* __restrict__ rlat = p.g.rlat;                                                        \
  [[maybe_unused]] const double* __restrict__ coslat = p.g.coslat;                                                    \
  [[maybe_unused]] const double* __restrict__ plev = p.g.plev;                                                        \
  [[maybe_unused]] const double* rec_s = p.rec + (long long)s * L * p.max_ny * LEC_NREC;                              \
  double* fin_s = p.fin + (long long)s * L * kLevStride;                                             \
  [[maybe_unused]] double* AA = fin_s;                       /* [L][6]   */                                           \
  [[maybe_unused]] double* sig = AA + 6 * L;                 /* [L]      */                                           \
  [[maybe_unused]] double* sums = sig + L;                   /* [L][27]  */                                           \
  [[maybe_unused]] double* edges = sums + SQ_NSUM * L;       /* [L][2][5] */                                          \
  [[maybe_unused]] double* bnd = edges + 2 * N_NEDGE * L;    /* [L][6][3] */                                          \
  [[maybe_unused]] auto wphi = [&](int j) -> double {                                                                 \
    const double lo = (j > j0) ? rlat[j] - rlat[j - 1] : 0.0;                                        \
    const double hi = (j < j1) ? rlat[j + 1] - rlat[j] : 0.0;                                        \
    return 0.5 * (lo + hi);                                                                          \
  };                                                                                                 \


// F1: one warp per (step, level): area means [X] of the six zonal means (calc_averages.py:46-78)
__global__ void __launch_bounds__(kFinThreads)
lec_fin_means_kernel(const FinParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sk = blockIdx.x * (kFinThreads / 32) + warp;
  if (sk >= p.nsteps * p.g.nlev) return;
  LEC_FIN_PROLOGUE(sk)
  double a[6] = {0, 0, 0, 0, 0, 0};
  for (int jr = lane; jr < ny; jr += 32) {
    const int j = j0 + jr;
    const double* r = rec_s + ((long long)k * p.max_ny + jr) * LEC_NREC;
    const double cw = wphi(j) * coslat[j];
    double sm[6], sh[6];
    rec_load<R_A, 6>(r, sm);
    rec_load<R_SH_T, 6>(r, sh);
#pragma unroll
    for (int f = 0; f < 5; ++f) a[f] += cw * (sc[f] * (sh[f] + sm[f] * ix));
    a[5] += cw * (sm[5] * ix);
  }
  const double tot = butterfly_reduce<6>(a, lane);
  const int idx = bitrev5(lane);
  if (idx < 6) AA[6 * k + idx] = tot * iy;
  if (k == 0 && lane == 0 && p.out_flags) p.out_flags[s] = 0;
}

// F2: one warp per (step, level): sigma and the meridional sums of every integrand
__global__ void __launch_bounds__(kFinThreads)
lec_fin_sums_kernel(const FinParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sk = blockIdx.x * (kFinThreads / 32) + warp;
  if (sk >= p.nsteps * p.g.nlev) return;
  LEC_FIN_PROLOGUE(sk)
  // sigma_k = g [T]/cp - (p g/Rd) d[T]/dp, floored at 0.03 (NaN -> 0.03)  (thermodynamics.py:26-73)
  if (lane == 0) {
    const double t0 = AA[6 * k];
    const double tm = AA[6 * (k > 0 ? k - 1 : k)], tp = AA[6 * (k < L - 1 ? k + 1 : k)];
    const double dTdp = p.g.pa[k] * (tm - t0) + p.g.pc[k] * (tp - t0);
    double sg = kG * t0 / kCp - (plev[k] * kG / kRd) * dTdp;
    if (!(sg > 0.03)) { sg = 0.03; if (p.out_flags) atomicOr(p.out_flags + s, 2); }
    sig[k] = sg;
  }
  // ---- phase 2: meridional sums per level ------------------------------------------------
  {
    const double T_AA = AA[6 * k], w_AA = AA[6 * k + 3], F_AA = AA[6 * k + 4], Q_AA = AA[6 * k + 5];
    const int km = (k > 0) ? k - 1 : k, kp = (k < L - 1) ? k + 1 : k;
    const double T_AAm = AA[6 * km], T_AAp = AA[6 * kp];
    const double pa = p.g.pa[k], pc = p.g.pc[k];
    double a[SQ_NSUM];
#pragma unroll
    for (int n = 0; n < SQ_NSUM; ++n) a[n] = 0.0;
    for (int jr = lane; jr < ny; jr += 32) {
      const int j = j0 + jr;
      const double* r = rec_s + ((long long)k * p.max_ny + jr) * LEC_NREC;
      RowQ q;
      derive_row(r, ix, sc, q);
      const double cj = coslat[j], yw = wphi(j), cw = yw * cj;
      const double T_AE = q.Tm - T_AA, w_AE = q.wm - w_AA, F_AE = q.Fm - F_AA, Qa_AE = q.Qm - Q_AA;
      // meridional neighbours (zonal means of rows j-1, j+1; one-sided at the box edges)
      const int jm = (jr > 0) ? jr - 1 : jr, jp = (jr < ny - 1) ? jr + 1 : jr;
      const double* rm = rec_s + ((long long)k * p.max_ny + jm) * LEC_NREC;
      const double* rp = rec_s + ((long long)k * p.max_ny + jp) * LEC_NREC;
      double ya, yc;
      if (jr == 0) { ya = 0.0; yc = 1.0 / (rlat[j + 1] - rlat[j]); }
      else if (jr == ny - 1) { ya = -1.0 / (rlat[j] - rlat[j - 1]); yc = 0.0; }
      else { ya = p.g.fya[j]; yc = p.g.fyc[j]; }
      const double cjm = coslat[j0 + jm], cjp = coslat[j0 + jp];
      double mm[3], mp[3];
      rec_means<3>(rm, ix, sc, mm);
      rec_means<3>(rp, ix, sc, mp);
      const double Tm_m = mm[0], Tm_p = mp[0], um_m = mm[1], um_p = mp[1], vm_m = mm[2], vm_p = mp[2];
      const double f0 = T_AE * cj;
      const double dphi_TAEc = ya * ((Tm_m - T_AA) * cjm - f0) + yc * ((Tm_p - T_AA) * cjp - f0);
      const double g0 = q.um / cj;
      const double dphi_uc = ya * (um_m / cjm - g0) + yc * (um_p / cjp - g0);
      const double dphi_v = ya * (vm_m - q.vm) + yc * (vm_p - q.vm);
      // vertical neighbours (same row, levels k-1, k+1; one-sided at the column ends via pa/pc)
      const double* rkm = rec_s + ((long long)km * p.max_ny + jr) * LEC_NREC;
      const double* rkp = rec_s + ((long long)kp * p.max_ny + jr) * LEC_NREC;
      double km2[2], kp2[2];
      rec_means<2>(rkm, ix, sc, km2);
      rec_means<2>(rkp, ix, sc, kp2);
      const double dp_TAE = pa * ((km2[0] - T_AAm) - T_AE) + pc * ((kp2[0] - T_AAp) - T_AE);
      // d[u]/dp as np.gradient takes it: on an exactly uniform level axis the centred difference never reads
      // [u] of level k, so Ck_5 (whose co-factor [w'v'] does not hold u) stays finite when u is missing at k
      const double dp_u = (p.g.p_2h != 0.0 && k > 0 && k < L - 1) ? (kp2[1] - km2[1]) / p.g.p_2h
                                                                 : pa * (km2[1] - q.um) + pc * (kp2[1] - q.um);

      const double uu_raw = q.uu + q.um * q.um, vv_raw = q.vv + q.vm * q.vm;   // ZA(u^2), ZA(v^2)
      const double uv_raw = q.uv + q.um * q.vm;
      // ZA(K* v), ZA(K* w): K* = u^2+v^2-u'^2-v'^2 = 2 u [u] - [u]^2 + 2 v [v] - [v]^2
      const double Ksv = 2.0 * q.um * uv_raw - q.um * q.um * q.vm + 2.0 * q.vm * vv_raw - q.vm * q.vm * q.vm;
      const double uw_raw = q.wu + q.um * q.wm, vw_raw = q.wv + q.vm * q.wm;
      const double Ksw = 2.0 * q.um * uw_raw - q.um * q.um * q.wm + 2.0 * q.vm * vw_raw - q.vm * q.vm * q.wm;
      const double Kp = q.uu + q.vv;                                            // ZA(K')
      const double Kpv = q.uuv + q.vvv + q.vm * Kp;
      const double Kpw = q.uuw + q.vvw + q.wm * Kp;
      const double vTT = q.vTTc + q.vm * q.TT, wTT = q.wTTc + q.wm * q.TT;
      (void)uu_raw;

      a[SQ_AZ] += cw * T_AE * T_AE;
      a[SQ_AE] += cw * q.TT;
      a[SQ_KZ] += cw * (q.um * q.um + q.vm * q.vm);
      a[SQ_KE] += cw * Kp;
      a[SQ_CZ2] += cw * w_AE * T_AE;
      a[SQ_CE2] += cw * q.wT;
      a[SQ_CA1] += cw * q.vT * dphi_TAEc;
      a[SQ_CA2] += cw * q.wT * dp_TAE;
      a[SQ_CK1] += cw * cj * q.uv * dphi_uc;
      a[SQ_CK2] += cw * q.vv * dphi_v;
      a[SQ_CK3] += cw * p.g.tanlat[j] * q.uu * q.vm;
      a[SQ_CK4] += cw * q.wu * dp_u;
      a[SQ_CK5] += cw * q.wv * dp_u;                 // sic: d[u]/dp (conversion_terms.py:225-229)
      a[SQ_GZ] += cw * Qa_AE * T_AE;
      a[SQ_GE] += cw * q.QT;
      a[SQ_BAZ3] += cw * (2.0 * q.wT * T_AE + q.wm * T_AE * T_AE);
      a[SQ_BAE3] += cw * wTT;
      a[SQ_BKZ3] += cw * Ksw;
      a[SQ_BKE3] += cw * Kpw;
      a[SQ_BOZ3] += cw * w_AE * F_AE;
      a[SQ_BOE3] += cw * q.wF;
      // east-minus-west fluxes, integrated over latitude WITHOUT cos (boundary_terms.py)
      const double TzE = q.TE - q.Tm, TzW = q.TW - q.Tm;            // T' at the edges
      const double uzE = q.uE - q.um, uzW = q.uW - q.um, vzE = q.vE - q.vm, vzW = q.vW - q.vm;
      a[Y_BAZ1] += yw * ((2.0 * T_AE * TzE * q.uE + T_AE * T_AE * q.uE) -
                         (2.0 * T_AE * TzW * q.uW + T_AE * T_AE * q.uW));
      a[Y_BAE1] += yw * (q.uE * TzE * TzE - q.uW * TzW * TzW);
      const double KpE = uzE * uzE + vzE * vzE, KpW = uzW * uzW + vzW * vzW;
      const double KsE = q.uE * q.uE + q.vE * q.vE - KpE, KsW = q.uW * q.uW + q.vW * q.vW - KpW;
      a[Y_BKZ1] += yw * (q.uE * KsE - q.uW * KsW);
      a[Y_BKE1] += yw * (q.uE * KpE - q.uW * KpW);
      a[Y_BOZ1] += yw * q.vm * F_AE;                                 // no E-W difference, sic
      a[Y_BOE1] += yw * (vzE - vzW) * F_AE;                          // v' [Phi]-area-eddy, sic
      if (jr == 0 || jr == ny - 1) {
        double* e = edges + (2 * k + (jr == 0 ? 1 : 0)) * N_NEDGE;   // [k][0]=north, [k][1]=south
        e[N_BAZ2] = (2.0 * q.vT * T_AE + T_AE * T_AE * q.vm) * cj;
        e[N_BAE2] = vTT * cj;
        e[N_BKZ2] = Ksv * cj;
        e[N_BKE2] = Kpv * cj;
        e[N_BOZ2] = q.vm * F_AE * cj;
      }
    }
    const double tot = butterfly_reduce<SQ_NSUM>(a, lane);
    const int idx = bitrev5(lane);
    if (idx < SQ_NSUM) sums[SQ_NSUM * k + idx] = tot;
  }
}

// F3: one CTA per step: per-level integrands, then the trapezoid over pressure -> 16 scalars
__global__ void __launch_bounds__(64)
lec_fin_integrate_kernel(const FinParams p) {
  constexpr int kThreads = 64;
  __shared__ int flag_sh;
  if (threadIdx.x == 0) flag_sh = 0;
  __syncthreads();
  LEC_FIN_PROLOGUE(blockIdx.x * p.g.nlev)
  // ---- phase 3: per-level integrands -------------------------------------------------------
  double* lv_out = p.out_levels ? p.out_levels + (long long)s * 19 * L : nullptr;
  for (int k = threadIdx.x; k < L; k += kThreads) {
    const double* q = sums + SQ_NSUM * k;
    const double* eN = edges + (2 * k) * N_NEDGE;
    const double* eS = eN + N_NEDGE;
    const double sg = sig[k], pk = plev[k];
    const double az = q[SQ_AZ] * iy / (2.0 * sg), ae = q[SQ_AE] * iy / (2.0 * sg);
    const double kz = q[SQ_KZ] * iy, ke = q[SQ_KE] * iy;
    const double cz1 = kRd / (pk * kG);
    const double cz2 = q[SQ_CZ2] * iy, ce2 = q[SQ_CE2] * iy;
    const double cz = -(cz1 * cz2), ce = -(cz1 * ce2);
    const double ca1 = q[SQ_CA1] * iy / (2.0 * kRe * sg), ca2 = q[SQ_CA2] * iy / sg;
    const double ca = -(ca1 + ca2);
    const double ck1 = q[SQ_CK1] * iy / kRe, ck2 = q[SQ_CK2] * iy / kRe, ck3 = q[SQ_CK3] * iy / kRe;
    const double ck4 = q[SQ_CK4] * iy, ck5 = q[SQ_CK5] * iy;
    const double ck = ck1 + ck2 + ck3 + ck4 + ck5;
    const double gz = q[SQ_GZ] * iy / (kCp * sg), ge = q[SQ_GE] * iy / (kCp * sg);
    double* b = bnd + kNB * k;
    b[0] = q[Y_BAZ1] / (2.0 * sg); b[1] = (eN[N_BAZ2] - eS[N_BAZ2]) / (2.0 * sg); b[2] = q[SQ_BAZ3] * iy / (2.0 * sg);
    b[3] = q[Y_BAE1] / (2.0 * sg); b[4] = (eN[N_BAE2] - eS[N_BAE2]) / (2.0 * sg); b[5] = q[SQ_BAE3] * iy / (2.0 * sg);
    b[6] = q[Y_BKZ1] / (2.0 * kG); b[7] = (eN[N_BKZ2] - eS[N_BKZ2]) / (2.0 * kG); b[8] = q[SQ_BKZ3] * iy / (2.0 * kG);
    b[9] = q[Y_BKE1] / (2.0 * kG); b[10] = (eN[N_BKE2] - eS[N_BKE2]) / (2.0 * kG); b[11] = q[SQ_BKE3] * iy / (2.0 * kG);
    b[12] = q[Y_BOZ1] / kG; b[13] = (eN[N_BOZ2] - eS[N_BOZ2]) / kG; b[14] = q[SQ_BOZ3] * iy / kG;
    b[15] = q[Y_BOE1] / kG; b[16] = b[13]; b[17] = q[SQ_BOE3] * iy / kG;
    // reuse the sums row for the level integrands (LEC_LV_* order of lec_b200.h)
    double lv[19] = {az, ae, kz, ke, ge, gz, cz, cz2, ca, ca1, ca2, ce, ce2, ck, ck1, ck2, ck3, ck4, ck5};
    bool bad = false;
#pragma unroll
    for (int n = 0; n < 19; ++n) {
      sums[SQ_NSUM * k + n] = lv[n];
      bad |= !isfinite(lv[n]);
      if (lv_out) lv_out[n * L + k] = lv[n];
    }
#pragma unroll
    for (int n = 0; n < kNB; ++n) {
      bad |= !isfinite(b[n]);
      if (p.out_bnd) p.out_bnd[((long long)s * kNB + n) * L + k] = b[n];
    }
    if (bad) atomicOr(&flag_sh, 1);
  }
  __syncthreads();

  // ---- phase 4: vertical trapezoids ----------------------------------------------------------
  if (threadIdx.x < 16) {
    const int t = threadIdx.x;
    auto vint = [&](const double* base, int stride) -> double {
      double acc = 0.0;
      for (int k = 0; k + 1 < L; ++k)
        acc += (plev[k + 1] - plev[k]) * 0.5 * (base[(k + 1) * stride] + base[k * stride]);
      return acc;
    };
    double v;
    // level-integrand slot (in `sums`) of the eight volume terms + Gz, Ge
    if (t < 8 || t >= 14) {
      const int slot[16] = {0, 1, 2, 3, 6, 8, 13, 11, -1, -1, -1, -1, -1, -1, 5, 4};
      v = vint(sums + slot[t], SQ_NSUM);
      if (t == 2 || t == 3) v /= (2.0 * kG);     // Kz, Ke
      if (t == 6) v /= kG;                        // Ck
    } else {
      const double* b = bnd + 3 * (t - 8);
      const double ew = vint(b, kNB), ns = vint(b + 1, kNB);
      const double bt = b[(L - 1) * kNB + 2] - b[2];
      v = ew * st.c1 + ns * st.c2 - bt;
    }
    p.out_terms[(long long)s * 16 + t] = v;
  }
  if (threadIdx.x == 0 && p.out_flags && flag_sh) atomicOr(p.out_flags + s, flag_sh);
}

}  // namespace lec
