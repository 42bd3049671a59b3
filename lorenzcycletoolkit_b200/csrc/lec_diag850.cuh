// 850-hPa track diagnostics of the moving framework (reference: src/frameworks/lec_moving_framework.py
// :650-663 wind speed + relative vorticity over the pre-sliced domain, :269-417 get_position, and
// src/utils/tools.py:95-128 find_extremum_coordinates): per time step, over the label-sliced box, the
// extrema of zeta, geopotential height and wind speed and WHERE they are, plus zeta at the grid point
// nearest to the track centre (the -z branch, :317-324).
//
// Vorticity is MetPy 1.6.2's `vorticity(u, v)` on a latitude / longitude grid (metpy/calc/kinematics.py):
//   zeta = [k dv/dx + u (h/k) dk/dy] - [h du/dy + v (k/h) dh/dx]
// with the "nominal" grid deltas dx = a dlambda, dy = meridian arc, the map factors k (parallel) and
// h (meridional) of the ellipsoid, and every derivative MetPy's 3-point `first_derivative` over the DOMAIN
// axes (second-order one-sided at the domain ends, not at the box edges).  The caller supplies dx, dy, k, h
// (utils/geodesy.py); the stencil coefficients are built from them on the host in MetPy's operation order.
// Everything is fp64 with explicitly rounded operations in numpy's evaluation order (no FMA contraction),
// so zeta has the bits of the numpy restatement and the arg-reductions select the same grid point.
// One CTA per time step; the box of one level is at most a few 10^4 points.
#pragma once
#include "lec_common.cuh"

namespace lec {

struct DiagAxis {          // first_derivative along one axis: out[i] = A[i] f[s] + B[i] f[s+1] + C[i] f[s+2],
  const double* A;         //   s = clamp(i - 1, 0, n - 3)
  const double* B;
  const double* C;
  int n;
};

struct DiagStepDev { int slot, i0, i1, j0, j1, ic, jc, ox, oy; };   // ox, oy: window origin of the slot's planes

struct DiagParams {
  const void* u; const void* v; const void* z;      // [slot][rows][ld] planes of the 850-hPa level: the domain, or a
                                                     // window of it (lec_diag850_host_windows; origin per step)
  DiagAxis ax, ay;
  const double* ps;        // [nlat] parallel scale k
  const double* ms;        // [nlat] meridional scale h
  const double* dxcorr;    // [nlat] (h / k) * dk/dy
  const double* pm;        // [nlat] k / h
  double su, sv, sz, zdiv;                            // unit factors; hgt = (z * sz) / zdiv
  const DiagStepDev* steps;
  double* out_val;                                     // [nsteps][5]: zeta min, zeta max, hgt min, wind max (NaNs skipped), zeta at the centre
  int* out_idx;                                        // [nsteps][4]: numpy argmin/argmax of the box, row-major flat index
  int nlon, nlat;           // the domain (the stencil clamps, the metric tables)
  int ld;                   // row length of the planes
  long long plane;          // elements per plane
};

__device__ __forceinline__ double diag_d3(const DiagAxis& A, int i, double f0, double f1, double f2) {
  return __dadd_rn(__dadd_rn(__dmul_rn(A.A[i], f0), __dmul_rn(A.B[i], f1)), __dmul_rn(A.C[i], f2));
}

// MetPy vorticity at domain point (j, i) of one slot
template <typename FT>
__device__ __forceinline__ double diag_zeta(const DiagParams& p, const FT* __restrict__ U, const FT* __restrict__ V,
                                            int j, int i, double& u0, double& v0) {
  const long long o = (long long)j * p.ld + i;
  u0 = __dmul_rn(double(U[o]), p.su); v0 = __dmul_rn(double(V[o]), p.sv);
  const int si = min(max(i - 1, 0), p.nlon - 3), sj = min(max(j - 1, 0), p.nlat - 3);
  const long long orow = (long long)j * p.ld + si, ocol = (long long)sj * p.ld + i;
  const double va = __dmul_rn(double(V[orow]), p.sv), vb = __dmul_rn(double(V[orow + 1]), p.sv),
               vc = __dmul_rn(double(V[orow + 2]), p.sv);
  const double ua = __dmul_rn(double(U[ocol]), p.su), ub = __dmul_rn(double(U[ocol + p.ld]), p.su),
               uc = __dmul_rn(double(U[ocol + 2LL * p.ld]), p.su);
  const double dvdx_n = diag_d3(p.ax, i, va, vb, vc);
  const double dudy_n = diag_d3(p.ay, j, ua, ub, uc);
  const double mj = p.ms[j], pj = p.ps[j];
  const double dmdx = diag_d3(p.ax, i, mj, mj, mj);                   // ~0: h does not vary along a parallel
  const double dudy = __dadd_rn(__dmul_rn(mj, dudy_n), __dmul_rn(v0, __dmul_rn(p.pm[j], dmdx)));
  const double dvdx = __dadd_rn(__dmul_rn(pj, dvdx_n), __dmul_rn(u0, p.dxcorr[j]));
  return __dsub_rn(dvdx, dudy);
}

// running extremum with numpy semantics: first occurrence wins ties, the first NaN wins argmin/argmax,
// the VALUE skips NaNs (nanmin / xarray's skipna)
struct DiagExt {
  double val; int idx; int nan_idx;
  __device__ __forceinline__ void init() { val = 0.0; idx = 0x7fffffff; nan_idx = 0x7fffffff; }
  template <bool MIN>
  __device__ __forceinline__ void take(double x, int i) {
    if (x != x) { nan_idx = min(nan_idx, i); return; }
    const bool better = (idx == 0x7fffffff) || (MIN ? x < val : x > val) || (x == val && i < idx);
    if (better) { val = x; idx = i; }
  }
  template <bool MIN>
  __device__ __forceinline__ void merge(double x, int i, int ni) {
    nan_idx = min(nan_idx, ni);
    if (i == 0x7fffffff) return;
    const bool better = (idx == 0x7fffffff) || (MIN ? x < val : x > val) || (x == val && i < idx);
    if (better) { val = x; idx = i; }
  }
};

template <bool MIN>
__device__ __forceinline__ void diag_warp_reduce(DiagExt& e) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const double x = __shfl_xor_sync(0xffffffffu, e.val, o);
    const int i = __shfl_xor_sync(0xffffffffu, e.idx, o);
    const int ni = __shfl_xor_sync(0xffffffffu, e.nan_idx, o);
    e.merge<MIN>(x, i, ni);
  }
}

constexpr int kDiagThreads = 256;

template <typename FT>
__global__ void __launch_bounds__(kDiagThreads) lec_diag850_kernel(const DiagParams p) {
  const DiagStepDev st = p.steps[blockIdx.x];
  const int nx = st.i1 - st.i0 + 1, ny = st.j1 - st.j0 + 1;
  // shifted by the window origin: domain indices (j, i) address the planes
  const long long base = st.slot * p.plane - ((long long)st.oy * p.ld + st.ox);
  const FT* __restrict__ U = static_cast<const FT*>(p.u) + base;
  const FT* __restrict__ V = static_cast<const FT*>(p.v) + base;
  const FT* __restrict__ Z = static_cast<const FT*>(p.z) + base;

  DiagExt zmin, zmax, hmin, wmax;
  zmin.init(); zmax.init(); hmin.init(); wmax.init();
  for (int q = threadIdx.x; q < nx * ny; q += kDiagThreads) {
    const int jr = q / nx, ir = q - jr * nx;
    const int j = st.j0 + jr, i = st.i0 + ir;
    double u0, v0;
    const double zeta = diag_zeta<FT>(p, U, V, j, i, u0, v0);
    const double wspd = __dsqrt_rn(__dadd_rn(__dmul_rn(u0, u0), __dmul_rn(v0, v0)));
    const double hgt = __ddiv_rn(__dmul_rn(double(Z[(long long)j * p.ld + i]), p.sz), p.zdiv);
    zmin.take<true>(zeta, q); zmax.take<false>(zeta, q); hmin.take<true>(hgt, q); wmax.take<false>(wspd, q);
  }
  if (threadIdx.x == kDiagThreads - 1) {       // zeta at the track centre (domain indices; -1 = not requested)
    double u0, v0;
    p.out_val[blockIdx.x * 5 + 4] = (st.ic >= 0 && st.jc >= 0) ? diag_zeta<FT>(p, U, V, st.jc, st.ic, u0, v0)
                                                              : __longlong_as_double(0x7ff8000000000000LL);
  }
  diag_warp_reduce<true>(zmin); diag_warp_reduce<false>(zmax); diag_warp_reduce<true>(hmin); diag_warp_reduce<false>(wmax);

  __shared__ double s_val[kDiagThreads / 32][4];
  __shared__ int s_idx[kDiagThreads / 32][4], s_nan[kDiagThreads / 32][4];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    s_val[warp][0] = zmin.val; s_idx[warp][0] = zmin.idx; s_nan[warp][0] = zmin.nan_idx;
    s_val[warp][1] = zmax.val; s_idx[warp][1] = zmax.idx; s_nan[warp][1] = zmax.nan_idx;
    s_val[warp][2] = hmin.val; s_idx[warp][2] = hmin.idx; s_nan[warp][2] = hmin.nan_idx;
    s_val[warp][3] = wmax.val; s_idx[warp][3] = wmax.idx; s_nan[warp][3] = wmax.nan_idx;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    const int m = threadIdx.x;
    DiagExt e; e.init();
    for (int w = 0; w < kDiagThreads / 32; ++w) {
      if (m == 0 || m == 2) e.merge<true>(s_val[w][m], s_idx[w][m], s_nan[w][m]);
      else e.merge<false>(s_val[w][m], s_idx[w][m], s_nan[w][m]);
    }
    p.out_val[blockIdx.x * 5 + m] = (e.idx == 0x7fffffff) ? __longlong_as_double(0x7ff8000000000000LL) : e.val;
    p.out_idx[blockIdx.x * 4 + m] = (e.nan_idx != 0x7fffffff) ? e.nan_idx : e.idx;
  }
}

}  // namespace lec
