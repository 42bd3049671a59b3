// Kernel A, TMA-tiled variant: the same sweep as lec_row_moments_kernel (same lane <-> column mapping,
// same per-lane accumulation order, same butterfly -- so the row records have the SAME BITS), fed from
// shared memory by the Tensor Memory Accelerator instead of per-lane global loads.
//
//  * One persistent CTA per SM walks the tile list (band, step, level, row-tile) -- the band-major order
//    of the direct kernel, so T(t+1) is still reused out of L2.  A tile is R consecutive box rows of one
//    (step, level); it is swept in chunks of 32 x 128 bit per row.
//  * ONE producer thread (its own warp, no arithmetic) issues, per chunk, 9 TMA tensor loads
//        T centre tile with the j-1 / j+1 rows and one vector of lon halo  ((R+2) x (C+2 VEC))
//        T(t-1), T(t+1), T(k-1), T(k+1), u, v, omega, Phi                     (R x C each)
//    into an S-stage shared-memory ring (full / empty mbarriers, expect_tx byte counting).  The j+-1 rows
//    are fetched once per tile instead of once per row (L2 -> SM traffic 9 + 2/R row streams instead of
//    11 + 2 scalar neighbours), and the bytes in flight ((S-1) stages, 110-170 KB per SM) no longer
//    depend on registers or occupancy.
//  * R consumer warps, one box row each: wait(full) -> 11 LDS.128, the lon neighbours of the chunk ends by
//    shuffle (lanes 0 / 31: one LDS.32 of the halo column) -> the shared iteration body (lec_row_body.inc)
//    -> arrive(empty).  No global addressing, no long-scoreboard stalls in the arithmetic warps; rows
//    outside the box or the grid are zero-filled by TMA and masked as before.
#pragma once
#include <cuda.h>

#include "lec_common.cuh"
#include "lec_pair.cuh"
#include "lec_row_moments.cuh"

namespace lec {

struct alignas(64) TmaMaps {
  CUtensorMap t_halo;    // T, box (C + 2 VEC) x (R + 2)
  CUtensorMap t_plain;   // T, box C x R
  CUtensorMap u, v, w, f;
};

// R = consumer warps = rows of a tile (the box height of the tensor maps); a chunk is 32 x 128 bit of a row.
// ST = stored element type: FT, or int16 (lec_run_device_packed), which keeps the lane <-> column map of FT (VEC) and
// shrinks the ring's bytes.  Every TMA box starts on a 16-byte boundary of the row: the fp chunks do by construction
// (VEC columns = 16 bytes), an int16 chunk starts at column c0 * VEC, a multiple of 4 (fp32) or 2 (fp64) only, so the
// int16 boxes start at that column rounded down to a multiple of 8 and are 8 columns wider (PW); the consumers add the
// row's shift (c0 * VEC) & 7.  The int16 lon halo is 8 columns (16 bytes) a side.
template <typename FT, int R, int NSTG, typename ST = FT>
struct TileGeom {
  static constexpr bool I16 = sizeof(ST) != sizeof(FT);
  static constexpr int VEC = 16 / sizeof(FT);
  static constexpr int HV = I16 ? 8 : VEC;                   // lon halo columns each side (16 bytes)
  static constexpr int C = 32 * VEC;                         // columns per chunk
  static constexpr int PW = I16 ? C + 8 : C;                 // plain tile pitch (elements)
  static constexpr int HP = PW + 2 * HV;                     // halo tile pitch (elements)
  static_assert(HP * sizeof(ST) % 16 == 0 && PW * sizeof(ST) % 16 == 0, "TMA boxes are whole 16-byte units wide");
  static constexpr int halo_bytes = (R + 2) * HP * sizeof(ST);
  static constexpr int halo_bytes_pad = (halo_bytes + 127) / 128 * 128;
  // (int16: every plain tile starts on a 128-byte boundary, the alignment of a TMA destination)
  static constexpr int tile_bytes = I16 ? (R * PW * (int)sizeof(ST) + 127) / 128 * 128 : R * C * sizeof(ST);
  static constexpr int stage_bytes = halo_bytes_pad + 8 * tile_bytes;
  static constexpr int smem_bytes = NSTG * stage_bytes + 128;               // + barriers
  static constexpr int threads = (R + 1) * 32;                           // R consumer warps + the producer warp
  static constexpr int tx_bytes = ((R + 2) * HP + 8 * R * PW) * (int)sizeof(ST);   // what the 9 loads of a chunk deliver
};

__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
// arrive on the barrier OFF bytes behind `bar` (the offset is an immediate of the instruction, not an addition)
template <int OFF>
__device__ __forceinline__ void mbar_arrive_off(unsigned bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0+%1];" ::"r"(bar), "n"(OFF) : "memory");
}
// the same load with an L2 eviction-priority hint (u, v, omega, Phi are read once: evict-first keeps them from
// displacing the T rows that the next two time steps and the neighbouring levels read again)
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void tma_load_4d_hint(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2, int c3,
                                                 unsigned long long pol) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5, %6}], [%2], %7;"
      ::"r"(dst), "l"(reinterpret_cast<unsigned long long>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "l"(pol)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(unsigned dst, const CUtensorMap* map, unsigned bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<unsigned long long>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// Shared-memory loads by 32-bit shared address (no generic -> shared conversion, immediate offsets).
// volatile: they must stay behind the mbarrier wait of their stage.
template <typename FT, int VEC>
__device__ __forceinline__ void lds_vec(unsigned a, FT (&v)[VEC]) {
  if constexpr (sizeof(FT) == 4) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(a));
  } else {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(a));
  }
}
__device__ __forceinline__ float lds_one(unsigned a, float) {
  float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v;
}
__device__ __forceinline__ double lds_one(unsigned a, double) {
  double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a)); return v;
}
// the same by stored type: int16 vectors (8 or 4 bytes) and elements are decoded (F = field)
template <typename ST, typename FT, int VEC, int F>
__device__ __forceinline__ void lds_row(unsigned a, FT (&v)[VEC], const PackedDev& pk) {
  if constexpr (sizeof(ST) == sizeof(FT)) {
    lds_vec<FT, VEC>(a, v);
  } else if constexpr (VEC == 4) {
    unsigned lo, hi;
    asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(a));
    unpack_i16_vec<FT, VEC, F, true>(lo, hi, v, pk);
  } else {
    unsigned lo;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(lo) : "r"(a));
    unpack_i16_vec<FT, VEC, F, true>(lo, 0u, v, pk);
  }
}
template <typename ST, typename FT, int F>
__device__ __forceinline__ FT lds_elem(unsigned a, const PackedDev& pk) {
  if constexpr (sizeof(ST) == sizeof(FT)) {
    return lds_one(a, FT());
  } else {
    unsigned short r;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r) : "r"(a));
    return unpack_i16<FT, F, true>(short(r), pk);
  }
}

// the tiled kernel's weight load: by 32-bit shared address when the table was copied behind the ring
template <bool SHARED, int VEC>
__device__ __forceinline__ void tab_load_tile(const float* ptr, unsigned saddr, float (&v)[VEC]) {
  if constexpr (SHARED && VEC == 4) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(saddr));
  } else {
    VecLoad<float, VEC>::ld(ptr, v);
  }
}

struct TileId { int band, s, k, jt; };
__device__ __forceinline__ TileId decode_tile(unsigned id, const RowParams& p) {
  TileId t;                                        // the host guarantees grid < 2^31 (FastDiv's range)
  unsigned jt, k, s;
  const unsigned a = p.dv_tiles.divmod(id, jt);
  const unsigned b = p.dv_lev.divmod(a, k);
  t.band = int(p.dv_steps.divmod(b, s));
  t.jt = int(jt); t.k = int(k); t.s = int(s);
  return t;
}

template <typename FT, typename CT, int LONW, int R, int NSTG, bool COMP, bool TABS, typename ST = FT>
__global__ void __launch_bounds__((R + 1) * 32, 1)
lec_row_moments_tile_kernel(const __grid_constant__ TmaMaps maps, const RowParams p) {
  using G = TileGeom<FT, R, NSTG, ST>;
  constexpr int VEC = G::VEC, C = G::C, PW = G::PW, HP = G::HP, HV = G::HV;
  extern __shared__ __align__(1024) unsigned char smem[];   // plain shared pointer: keeps LDS (not generic LD)
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + NSTG * G::stage_bytes);
  const unsigned full0 = smem_u32(bars), empty0 = smem_u32(bars + NSTG);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < NSTG; ++i) { mbar_init(full0 + 8 * i, 1); mbar_init(empty0 + 8 * i, R); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // TABS: the per-column trapezoid weights (LONW == 1, fp32) live in shared memory behind the ring -- one LDS.128
  // per iteration instead of a global load and its addressing (the host checks that the table fits)
  const float* wl_tab = p.g.wl32;
  if constexpr (TABS) {
    float* wl_s = reinterpret_cast<float*>(smem + G::smem_bytes);
    int ntab = p.g.nlon;                         // = the row length of fp fields (whole 128-bit chunks here)
    if constexpr (sizeof(ST) != sizeof(FT)) ntab = p.pk.ntab;
    for (int i = threadIdx.x; i < ntab; i += blockDim.x) wl_s[i] = __ldg(p.g.wl32 + i);
    wl_tab = wl_s;
  }
  __syncthreads();

  const int nlev = p.g.nlev;

  if (warp == R) {
    // ===================================== producer ==========================================
    // One thread walks the same (tile, chunk) sequence as the consumers and keeps the ring full; a chunk
    // costs one wait on its stage's empty barrier, one expect_tx and 9 tensor loads.
    if (lane == 0) {
      int stg = 0;
      unsigned phase = 0;
      [[maybe_unused]] unsigned long long pol_stream = 0;
      if constexpr (sizeof(FT) == 8) pol_stream = l2_policy_evict_first();
      for (unsigned id = blockIdx.x; id < (unsigned)p.grid; id += gridDim.x) {
        const TileId t = decode_tile(id, p);
        const StepDev* __restrict__ st = p.steps + t.s;
        const int jr = (t.band * p.tiles_per_band + t.jt) * R;
        if (jr > st->j1 - st->j0) continue;
        const int c0 = st->i0 / VEC, c1 = st->i1 / VEC;
        const int nch = (c1 - c0 + 32) / 32;
        const int jt0 = st->j0 + jr;
        const int k = t.k, km = k > 0 ? k - 1 : k, kp = k < nlev - 1 ? k + 1 : k;
        const int slot = st->slot, slot_m = st->slot_m, slot_p = st->slot_p;
        int col = c0 * VEC;
        if constexpr (G::I16) col &= ~7;             // 16-byte aligned box start
        for (int ch = 0; ch < nch; ++ch, col += C) {
          mbar_wait(empty0 + 8 * stg, phase ^ 1);
          const unsigned fb = full0 + 8 * stg;
          mbar_expect_tx(fb, (unsigned)G::tx_bytes);
          const unsigned base = smem_u32(smem) + (unsigned)stg * G::stage_bytes;
          tma_load_4d(base, &maps.t_halo, fb, col - HV, jt0 - 1, k, slot);
          unsigned d = base + G::halo_bytes_pad;
          // u, v, omega, Phi with the L2 evict-first hint over fp64 fields (decoded type for int16 fields): 46.7 -> 39.0
          // GB of DRAM reads per 24-step launch, +3.4 %.  With fp32 fields the working set of a band fits in L2 without
          // it and the hint costs 2 %.
          if constexpr (sizeof(FT) == 8) {
            tma_load_4d_hint(d, &maps.u, fb, col, jt0, k, slot, pol_stream); d += G::tile_bytes;
            tma_load_4d_hint(d, &maps.v, fb, col, jt0, k, slot, pol_stream); d += G::tile_bytes;
            tma_load_4d_hint(d, &maps.w, fb, col, jt0, k, slot, pol_stream); d += G::tile_bytes;
            tma_load_4d_hint(d, &maps.f, fb, col, jt0, k, slot, pol_stream); d += G::tile_bytes;
          } else {
            tma_load_4d(d, &maps.u, fb, col, jt0, k, slot); d += G::tile_bytes;
            tma_load_4d(d, &maps.v, fb, col, jt0, k, slot); d += G::tile_bytes;
            tma_load_4d(d, &maps.w, fb, col, jt0, k, slot); d += G::tile_bytes;
            tma_load_4d(d, &maps.f, fb, col, jt0, k, slot); d += G::tile_bytes;
          }
          tma_load_4d(d, &maps.t_plain, fb, col, jt0, k, slot_p); d += G::tile_bytes;
          tma_load_4d(d, &maps.t_plain, fb, col, jt0, k, slot_m); d += G::tile_bytes;
          tma_load_4d(d, &maps.t_plain, fb, col, jt0, km, slot); d += G::tile_bytes;
          tma_load_4d(d, &maps.t_plain, fb, col, jt0, kp, slot);
          if (++stg == NSTG) { stg = 0; phase ^= 1; }
        }
      }
    }
    return;
  }

  // ======================================= consumers ===========================================
  // per-lane tile offsets (bytes): own row of the halo tile (warp + 1) and of the eight plain tiles
  const unsigned sbase0 = smem_u32(smem);
  const unsigned off_hc = (unsigned)(((warp + 1) * HP + HV + lane * VEC) * sizeof(ST));
  const unsigned off_t = (unsigned)(G::halo_bytes_pad + (warp * PW + lane * VEC) * sizeof(ST));
  constexpr unsigned kTile = G::tile_bytes;
  // current stage: base address, its full barrier (the empty one sits 8 NSTG bytes behind it), index, phase; the
  // advance wraps by subtraction, so the ring needs no second copy of the base addresses in registers
  unsigned sb = sbase0, fb = full0;
  int stg = 0;
  unsigned phase = 0;
  // shared-memory copy of the trapezoid weights, as a 32-bit shared address (no generic -> shared conversion per load)
  [[maybe_unused]] unsigned wl_s32 = 0;
  if constexpr (TABS) wl_s32 = smem_u32(smem + G::smem_bytes);
  for (unsigned id = blockIdx.x; id < (unsigned)p.grid; id += gridDim.x) {
    const TileId t = decode_tile(id, p);
    const StepDev* __restrict__ st = p.steps + t.s;
    const int i0 = st->i0, i1 = st->i1, j0 = st->j0, j1 = st->j1;
    const int jrel0 = (t.band * p.tiles_per_band + t.jt) * R;
    if (jrel0 > j1 - j0) continue;                 // same test as the producer: no chunk was issued
    // warp_on: the warp's row lies in the tile and the box (warp-uniform: shuffles below); warps past the box sweep
    // the clamped last row and write nothing
    const bool warp_on = (warp < R) && (jrel0 + warp <= j1 - j0);
    const int jrel = warp_on ? jrel0 + warp : j1 - j0;
    const int j = j0 + jrel;
    const int k = t.k;
    const int c0 = i0 / VEC, c1 = i1 / VEC;
    const int niter = (c1 - c0 + 32) / 32;
    // int16: the row's first chunk sits this many bytes into the (16-byte aligned) boxes; 0 for fp fields
    const unsigned adj = G::I16 ? (unsigned)(((c0 * VEC) & 7) * (int)sizeof(ST)) : 0u;

    // (No L2 prefetch here: bulk prefetches of the next tile's rows -- issued by the producer thread or by the
    //  consumer warps -- were measured at 3.1-3.7 TB/s against 5.3-5.5 without; the ring alone covers DRAM latency.)
    RowSetup<CT, LONW> rs;
    rs.init(p, st, j, k, j0, j1);
    const RowCoefS<CT>& rc = rs.rc;
    const CT cxa_u = rs.cxa_u, cxc_u = rs.cxc_u, cxW = rs.cxW, cxE = rs.cxE, wW = rs.wW, wE = rs.wE;
    [[maybe_unused]] const double fxd = rs.fxd;
    const bool box_aligned = (i0 % VEC == 0) && ((i1 + 1) % VEC == 0);
    // at the box edges the j-1 / j+1 row falls back to the own row (its stencil coefficient is zero;
    // values outside the box are never touched)
    const unsigned off_hm = (j > j0) ? off_hc - (unsigned)(HP * sizeof(ST)) : off_hc;
    const unsigned off_hp = (j < j1) ? off_hc + (unsigned)(HP * sizeof(ST)) : off_hc;

    FT shT = FT(0), shU = FT(0), shV = FT(0), shW = FT(0), shF = FT(0);
    CT cshT = CT(0), cshU = CT(0), cshV = CT(0), cshW = CT(0), cshF = CT(0);
    CT S[R_NSUM], Cc[R_NLIN];
#pragma unroll
    for (int n = 0; n < R_NSUM; ++n) S[n] = CT(0);
#pragma unroll
    for (int n = 0; n < R_NLIN; ++n) Cc[n] = CT(0);
    double* __restrict__ rec = p.rec + (((long long)t.s * nlev + k) * p.max_ny + jrel) * LEC_NREC;


    // first and last sweep iteration peeled (box edges, lanes past the row end); interior iterations
    // run the short body
    {
      const int it = 0;
#define LEC_BODY_EDGE 1
#define LEC_ITER_FIRST 1
#include "lec_row_iter_tile.inc"
#undef LEC_ITER_FIRST
#undef LEC_BODY_EDGE
    }
    for (int it = 1; it < niter - 1; ++it) {
#define LEC_BODY_EDGE 0
#define LEC_ITER_FIRST 0
#include "lec_row_iter_tile.inc"
#undef LEC_ITER_FIRST
#undef LEC_BODY_EDGE
    }
    if (niter > 1) {
      const int it = niter - 1;
#define LEC_BODY_EDGE 1
#define LEC_ITER_FIRST 0
#include "lec_row_iter_tile.inc"
#undef LEC_ITER_FIRST
#undef LEC_BODY_EDGE
    }

    if (warp_on) {
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
  }
}

}  // namespace lec
