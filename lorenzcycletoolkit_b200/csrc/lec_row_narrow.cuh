// Kernel A for NARROW boxes (Semi-Lagrangian track boxes: 7 ... 151 columns).
//
// lec_row_moments_kernel gives a whole warp to one row: a 61-column box (16 chunks of 128 bits) would
// use half of the lanes, a 7-column NCEP box two of them.  Here a row is swept by a GROUP of G = 16, 8
// or 4 lanes, so a warp carries 32/G rows of the same (step, level); shuffles are confined to the group
// (width G), the 22 sums are reduced with the first log2(G) steps of the halving butterfly, and each
// lane of a group ends up with ceil(22/G) of the row's totals.  Loads, arithmetic (lec_row_body.inc) and
// the row records are those of the wide kernel.
#pragma once
#include "lec_common.cuh"
#include "lec_pair.cuh"
#include "lec_row_moments.cuh"

namespace lec {

constexpr int kNarrowWarps = 1;                   // warps per CTA (1 / 2 / 4 measured on the C5 track: 1.80 / 1.83 / 1.86 ms)
constexpr int kNarrowThreads = kNarrowWarps * 32;

// Halving butterfly inside groups of G lanes: every lane ends with the group totals of the values
// idx = bitrev_{log2 G}(gl) + m * G, m = 0 .. ceil(N/G)-1, in out[m].
template <int N, int G>
__device__ __forceinline__ void butterfly_reduce_seg(const double (&v)[N], int gl, double (&out)[(N + G - 1) / G]) {
  constexpr int NP = ((N + G - 1) / G) * G;       // padded to a multiple of G
  double a[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) a[i] = (i < N) ? v[i] : 0.0;
  int n = NP;
#pragma unroll
  for (int bit = G / 2; bit >= 1; bit >>= 1) {
    n >>= 1;
    const bool hi = (gl & bit) != 0;
#pragma unroll
    for (int i = 0; i < n; ++i) {
      const double keep = hi ? a[2 * i + 1] : a[2 * i];
      const double send = hi ? a[2 * i] : a[2 * i + 1];
      a[i] = keep + __shfl_xor_sync(0xffffffffu, send, bit);
    }
  }
#pragma unroll
  for (int m = 0; m < (N + G - 1) / G; ++m) out[m] = a[m];
}

template <int G>
__device__ __forceinline__ int bitrev_group(int gl) {
  int r = 0;
#pragma unroll
  for (int b = 1, o = G / 2; b < G; b <<= 1, o >>= 1) r |= (gl & b) ? o : 0;
  return r;
}

// ST: stored element type -- FT, or int16 decoded on load (lec_run_device_packed; RowParams::pk)
template <typename FT, typename CT, int VEC, int LONW, int G, bool COMP, typename ST = FT>
// fp64 arithmetic: 12 warps/SM, 168 registers; fp32 values decoded from int16 in fp64 arithmetic: 8 warps/SM, 255 registers
__global__ void __launch_bounds__(kNarrowThreads, (sizeof(CT) == 8 ? (sizeof(ST) == 2 && sizeof(FT) == 4 ? 256 : 384) : 512) / kNarrowThreads)
lec_row_moments_narrow_kernel(const RowParams p) {
  constexpr int RPW = 32 / G;                     // rows per warp
  const int warp = threadIdx.x >> 5, lane31 = threadIdx.x & 31;
  const int lane = lane31 & (G - 1);              // lane within the row's group ("lane" for the shared body)
  const int wr = lane31 / G;                      // row within the warp
  const unsigned bid = blockIdx.x;
  unsigned ujt, uk, us;
  const unsigned q1 = p.dv_tiles.divmod(bid, ujt);
  const unsigned q2 = p.dv_lev.divmod(q1, uk);
  const int band = int(p.dv_steps.divmod(q2, us));
  const int jt = int(ujt), k = int(uk), s = int(us);

  const StepDev* __restrict__ st = p.steps + s;
  const int i0 = st->i0, i1 = st->i1, j0 = st->j0, j1 = st->j1;
  const int jrel_first = ((band * p.tiles_per_band + jt) * kNarrowWarps + warp) * RPW;
  if (jrel_first > j1 - j0) return;               // the whole warp is outside the box
  const bool row_on = jrel_first + wr <= j1 - j0; // groups past the last row compute on a clamped row, write nothing
  const int jrel = min(jrel_first + wr, j1 - j0);
  const int j = j0 + jrel;
  const int nlon = p.g.nlon, nlat = p.g.nlat, nlev = p.g.nlev;

  const long long plane = (long long)nlat * nlon;
  const long long row_c = ((long long)st->slot * nlev + k) * plane + (long long)j * nlon;
  const ST* __restrict__ Tc_row = static_cast<const ST*>(p.field[0]) + row_c;
  const ST* __restrict__ U_row = static_cast<const ST*>(p.field[1]) + row_c;
  const ST* __restrict__ V_row = static_cast<const ST*>(p.field[2]) + row_c;
  const ST* __restrict__ W_row = static_cast<const ST*>(p.field[3]) + row_c;
  const ST* __restrict__ F_row = static_cast<const ST*>(p.field[4]) + row_c;
  const int d_m = int((long long)(st->slot_m - st->slot) * p.slot_stride);
  const int d_p = int((long long)(st->slot_p - st->slot) * p.slot_stride);
  const int d_km = (k > 0) ? -int(plane) : 0, d_kp = (k < nlev - 1) ? int(plane) : 0;
  const int d_jm = (j > j0) ? -nlon : 0, d_jp = (j < j1) ? nlon : 0;

  // L2 prefetch of the row's later sweep iterations: the streams that come from DRAM (u, v, omega, Phi of this step,
  // T of the next time slot) -- lane gl of a group touches the line that iteration gl will read, one plain
  // prefetch.global.L2 per stream (the bulk form is serialised through the uniform datapath and was slower)
  // Straight-line on purpose (lines 1 .. G-1, clamped to the row end): the same prefetches inside a per-lane loop
  // over all lines of a longer row measured SLOWER than no prefetch (2.05 vs 1.99 ms), straight-line 1.83 ms on the
  // C5 track; 61-column boxes 0.49 -> 0.46 ms, 301-column boxes 7.66 -> 7.50 ms.  The stride is the bytes of one
  // fp sweep iteration whatever the stored type (int16 rows: lines 1 .. G-1 of the row, two iterations each).
  if (lane >= 1) {
    const int pc = min(i0 + lane * (G * VEC * (int)sizeof(FT) / (int)sizeof(ST)), i1);
    asm volatile("prefetch.global.L2 [%0];" ::"l"(U_row + pc));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(V_row + pc));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(W_row + pc));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(F_row + pc));
    asm volatile("prefetch.global.L2 [%0];" ::"l"(Tc_row + (pc + d_p)));
  }

  RowSetup<CT, LONW> rs;
  rs.init(p, st, j, k, j0, j1);
  const RowCoefS<CT>& rc = rs.rc;
  const CT cxa_u = rs.cxa_u, cxc_u = rs.cxc_u, cxW = rs.cxW, cxE = rs.cxE, wW = rs.wW, wE = rs.wE;
  [[maybe_unused]] const double fxd = rs.fxd;
  const bool box_aligned = (i0 % VEC == 0) && ((i1 + 1) % VEC == 0);

  using LD = RowLoad<ST, FT, VEC>;
  const FT shT = LD::template one<0>(Tc_row + i0, p.pk), shU = LD::template one<1>(U_row + i0, p.pk),
           shV = LD::template one<2>(V_row + i0, p.pk), shW = LD::template one<3>(W_row + i0, p.pk),
           shF = LD::template one<4>(F_row + i0, p.pk);
  const CT cshT = CT(shT), cshU = CT(shU), cshV = CT(shV), cshW = CT(shW), cshF = CT(shF);

  CT S[R_NSUM], Cc[R_NLIN];
#pragma unroll
  for (int n = 0; n < R_NSUM; ++n) S[n] = CT(0);
#pragma unroll
  for (int n = 0; n < R_NLIN; ++n) Cc[n] = CT(0);
  double* __restrict__ rec = p.rec + (((long long)s * nlev + k) * p.max_ny + jrel) * LEC_NREC;

  const int c0 = i0 / VEC, c1 = i1 / VEC;
  const int niter = (c1 - c0 + G) / G;
  // first and last sweep iteration peeled (box edges, lanes past the row end, rows past the box); the
  // iterations in between run the body without masks and selects
  {
    const int it = 0;
#define LEC_BODY_EDGE 1
#include "lec_row_iter_narrow.inc"
#undef LEC_BODY_EDGE
  }
  for (int it = 1; it < niter - 1; ++it) {
#define LEC_BODY_EDGE 0
#include "lec_row_iter_narrow.inc"
#undef LEC_BODY_EDGE
  }
  if (niter > 1) {
    const int it = niter - 1;
#define LEC_BODY_EDGE 1
#include "lec_row_iter_narrow.inc"
#undef LEC_BODY_EDGE
  }

  double Sd[R_NSUM];
#pragma unroll
  for (int n = 0; n < R_NSUM; ++n) Sd[n] = double(S[n]);
  if constexpr (sizeof(CT) == 4 && COMP) {
#pragma unroll
    for (int n = 0; n < R_NLIN; ++n) Sd[n] += double(Cc[n]);
  }
  constexpr int NOUT = (R_NSUM + G - 1) / G;
  double tot[NOUT];
  butterfly_reduce_seg<R_NSUM, G>(Sd, lane, tot);
  if (row_on) {
    const int r = bitrev_group<G>(lane);
#pragma unroll
    for (int m = 0; m < NOUT; ++m) {
      const int idx = r + m * G;
      if (idx < R_NSUM) rec[idx] = (LONW == 0) ? tot[m] * p.g.wl_u : tot[m];
    }
    if (lane == 1) {
      rec[R_SH_T] = double(shT); rec[R_SH_U] = double(shU); rec[R_SH_V] = double(shV);
      rec[R_SH_W] = double(shW); rec[R_SH_F] = double(shF);
    }
  }
}

}  // namespace lec
