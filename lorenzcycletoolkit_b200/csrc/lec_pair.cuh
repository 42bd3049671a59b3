// Two-wide arithmetic for the row kernels.
//
// Blackwell (sm_100) issues packed fp32 FFMA2 / FADD2 / FMUL2 (PTX add/sub/mul/fma .f32x2): one
// warp instruction works on two fp32 values per lane, with a scalar operand broadcast for free.
// The row kernels are bound by instruction issue, not by the FMA pipe or DRAM, so the per-point
// operations are done on PAIRS of adjacent longitudes.  Pair<double> is the same
// interface with two scalar fp64 operations (fp64 fields / LEC_MATH_F64).
#pragma once
#include "lec_common.cuh"

namespace lec {

template <typename CT> struct Pair;

template <> struct Pair<float> {
  unsigned long long v;
  __device__ __forceinline__ static Pair make(float lo, float hi) {
    Pair p; asm("mov.b64 %0, {%1, %2};" : "=l"(p.v) : "f"(lo), "f"(hi)); return p;
  }
  __device__ __forceinline__ static Pair bcast(float s) { return make(s, s); }
  __device__ __forceinline__ float lo() const { return __uint_as_float((unsigned)(v & 0xffffffffull)); }
  __device__ __forceinline__ float hi() const { return __uint_as_float((unsigned)(v >> 32)); }
};
__device__ __forceinline__ Pair<float> operator+(Pair<float> a, Pair<float> b) {
  Pair<float> d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d.v) : "l"(a.v), "l"(b.v)); return d;
}
__device__ __forceinline__ Pair<float> operator-(Pair<float> a, Pair<float> b) {
  Pair<float> d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d.v) : "l"(a.v), "l"(b.v)); return d;
}
__device__ __forceinline__ Pair<float> operator*(Pair<float> a, Pair<float> b) {
  Pair<float> d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d.v) : "l"(a.v), "l"(b.v)); return d;
}
__device__ __forceinline__ Pair<float> pfma(Pair<float> a, Pair<float> b, Pair<float> c) {
  Pair<float> d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d.v) : "l"(a.v), "l"(b.v), "l"(c.v)); return d;
}

template <> struct Pair<double> {
  double l, h;
  __device__ __forceinline__ static Pair make(double lo, double hi) { Pair p; p.l = lo; p.h = hi; return p; }
  __device__ __forceinline__ static Pair bcast(double s) { return make(s, s); }
  __device__ __forceinline__ double lo() const { return l; }
  __device__ __forceinline__ double hi() const { return h; }
};
__device__ __forceinline__ Pair<double> operator+(Pair<double> a, Pair<double> b) { return Pair<double>::make(a.l + b.l, a.h + b.h); }
__device__ __forceinline__ Pair<double> operator-(Pair<double> a, Pair<double> b) { return Pair<double>::make(a.l - b.l, a.h - b.h); }
__device__ __forceinline__ Pair<double> operator*(Pair<double> a, Pair<double> b) { return Pair<double>::make(a.l * b.l, a.h * b.h); }
__device__ __forceinline__ Pair<double> pfma(Pair<double> a, Pair<double> b, Pair<double> c) {
  return Pair<double>::make(fma(a.l, b.l, c.l), fma(a.h, b.h, c.h));
}

}  // namespace lec
