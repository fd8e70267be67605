// tfg_num.cuh -- scalar types for the three arithmetic modes of the melt kernels.
//
// The physics (tfg_physics.cuh) is written once against Num<P>.  The policy P decides how an
// expression is evaluated:
//   StrictF64  every + - * / sqrt is a single IEEE round-to-nearest operation issued through the
//              __d*_rn intrinsics, which nvcc never contracts into FMAs.  Together with
//              host-precomputed constants this makes the non-transcendental part of a step
//              bit-identical to the NumPy reference; only exp/log/pow/atan/acos/sin/cos ulps differ.
//   FastF64    plain double arithmetic (FMA contraction allowed), cheaper formulations of pow.
//   FastF32    float with MUFU-backed intrinsics.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "tfg_math.cuh"

namespace tfg {

// `lean`: use the guard-free cores of tfg_math.cuh (valid only for physically sane arguments; the kernel
// checks the forcings and state of a warp each step and otherwise runs the same step under StrictF64).
struct StrictF64 { using raw = double; static constexpr bool strict = true,  f32 = false, lean = false; };
struct FastF64   { using raw = double; static constexpr bool strict = false, f32 = false, lean = true;  };
struct FastF32   { using raw = float;  static constexpr bool strict = false, f32 = true,  lean = false; };

template <class P>
struct Num {
  using raw = typename P::raw;
  raw v;
  __host__ __device__ Num() {}
  __host__ __device__ constexpr Num(double x) : v(static_cast<raw>(x)) {}
  __host__ __device__ constexpr Num(float x) : v(static_cast<raw>(x)) {}
  __host__ __device__ constexpr Num(int x) : v(static_cast<raw>(x)) {}
};

// ---- arithmetic ----------------------------------------------------------------------------------
template <class P> __device__ __forceinline__ Num<P> operator+(Num<P> a, Num<P> b) {
  if constexpr (P::strict) return Num<P>(__dadd_rn(a.v, b.v)); else return Num<P>(a.v + b.v);
}
template <class P> __device__ __forceinline__ Num<P> operator-(Num<P> a, Num<P> b) {
  if constexpr (P::strict) return Num<P>(__dsub_rn(a.v, b.v)); else return Num<P>(a.v - b.v);
}
template <class P> __device__ __forceinline__ Num<P> operator*(Num<P> a, Num<P> b) {
  if constexpr (P::strict) return Num<P>(__dmul_rn(a.v, b.v)); else return Num<P>(a.v * b.v);
}
template <class P> __device__ __forceinline__ Num<P> operator/(Num<P> a, Num<P> b) {
  if constexpr (P::strict) return Num<P>(__ddiv_rn(a.v, b.v));
  else if constexpr (P::f32) return Num<P>(__fdividef(a.v, b.v));
  else if constexpr (P::lean) return Num<P>(fm::div_fast(a.v, b.v));
  else return Num<P>(a.v / b.v);
}
template <class P> __device__ __forceinline__ Num<P> zdiv(Num<P> a, Num<P> b);
// division by a compile-time constant: a true division in strict mode, a multiplication by the
// (compile-time) reciprocal otherwise
template <class P> __device__ __forceinline__ Num<P> divk(Num<P> a, double c) {
  if constexpr (P::strict) return zdiv(a, Num<P>(c));
  else return Num<P>(a.v * static_cast<typename P::raw>(1.0 / c));
}
template <class P> __device__ __forceinline__ Num<P> operator-(Num<P> a) { return Num<P>(-a.v); }

#define TFG_MIXED(op)                                                                                         \
  template <class P> __device__ __forceinline__ Num<P> operator op(Num<P> a, double b) { return a op Num<P>(b); } \
  template <class P> __device__ __forceinline__ Num<P> operator op(double a, Num<P> b) { return Num<P>(a) op b; }
TFG_MIXED(+) TFG_MIXED(-) TFG_MIXED(*) TFG_MIXED(/)
#undef TFG_MIXED

#define TFG_CMP(op)                                                                                      \
  template <class P> __device__ __forceinline__ bool operator op(Num<P> a, Num<P> b) { return a.v op b.v; } \
  template <class P> __device__ __forceinline__ bool operator op(Num<P> a, double b) {                  \
    return a.v op static_cast<typename P::raw>(b);                                                       \
  }
TFG_CMP(<) TFG_CMP(<=) TFG_CMP(>) TFG_CMP(>=) TFG_CMP(==) TFG_CMP(!=)
#undef TFG_CMP

template <class P> __device__ __forceinline__ Num<P> sel(bool c, Num<P> a, Num<P> b) { return c ? a : b; }

// a*b + c and c - a*b.  Strict: the two roundings of the reference, in its order.  Fast modes: ONE fused operation,
// written out because the fast float64 translation unit is compiled with -fmad=false: which multiply-adds are fused
// is then decided here and not per template instantiation by the compiler, so recording kernels, aggregate kernels
// and TMA kernels of the fast mode return bit-identical state.
template <class P> __device__ __forceinline__ Num<P> fmadd(Num<P> a, Num<P> b, Num<P> c) {
  if constexpr (P::strict) return Num<P>(__dadd_rn(__dmul_rn(a.v, b.v), c.v));
  else if constexpr (P::f32) return Num<P>(fmaf(a.v, b.v, c.v));
  else return Num<P>(fma(a.v, b.v, c.v));
}
template <class P> __device__ __forceinline__ Num<P> fnmadd(Num<P> a, Num<P> b, Num<P> c) {
  if constexpr (P::strict) return Num<P>(__dsub_rn(c.v, __dmul_rn(a.v, b.v)));
  else if constexpr (P::f32) return Num<P>(fmaf(-a.v, b.v, c.v));
  else return Num<P>(fma(-a.v, b.v, c.v));
}

// np.minimum / np.maximum propagate NaN; fmin/fmax do not.  Strict mode keeps NumPy's behaviour.  float32: PTX
// max/min.NaN (FMNMX.NAN), one instruction that returns NaN if either operand is NaN and fmaxf/fminf's result otherwise
// -- the float32 kernel has no strict fallback, so a missing forcing must poison the cell through these as in the
// reference.  The fast float64 mode needs no NaN rule here: its non-finite inputs take the strict step.
template <class P> __device__ __forceinline__ Num<P> nmax(Num<P> a, Num<P> b) {
  if constexpr (P::strict) return Num<P>((a.v >= b.v) ? a.v : ((b.v > a.v) ? b.v : a.v + b.v));
  else if constexpr (P::f32) {
    float r;
    asm("max.ftz.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a.v), "f"(b.v));
    return Num<P>(r);
  } else {
    // setp + selp (3 instructions).  Written in PTX because nvcc turns `a > b ? a : b` back into fmax(), whose
    // NaN canonicalisation costs 6 instructions, two of them on the FP64 pipe.
    double r;
    asm("{ .reg .pred p; setp.gt.f64 p, %1, %2; selp.f64 %0, %1, %2, p; }" : "=d"(r) : "d"(a.v), "d"(b.v));
    return Num<P>(r);
  }
}
template <class P> __device__ __forceinline__ Num<P> nmin(Num<P> a, Num<P> b) {
  if constexpr (P::strict) return Num<P>((a.v <= b.v) ? a.v : ((b.v < a.v) ? b.v : a.v + b.v));
  else if constexpr (P::f32) {
    float r;
    asm("min.ftz.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a.v), "f"(b.v));
    return Num<P>(r);
  } else {
    double r;
    asm("{ .reg .pred p; setp.lt.f64 p, %1, %2; selp.f64 %0, %1, %2, p; }" : "=d"(r) : "d"(a.v), "d"(b.v));
    return Num<P>(r);
  }
}
// max(x, 0).  Fast float64: clears the value when the sign bit is set, with integer ops only (no FP64-pipe slot).
template <class P> __device__ __forceinline__ Num<P> relu(Num<P> a) {
  if constexpr (P::strict || P::f32) return nmax(a, Num<P>(0.0));
  else {
    const int hi = __double2hiint(a.v), keep = ~(hi >> 31);
    return Num<P>(__hiloint2double(hi & keep, __double2loint(a.v) & keep));
  }
}
template <class P> __device__ __forceinline__ Num<P> nabs(Num<P> a) {
  if constexpr (P::f32) return Num<P>(fabsf(a.v)); else return Num<P>(fabs(a.v));
}

// ---- single-rounding operations that no mode may contract or reassociate ----------------------------
// Used where the reference's exact rounding decides a discrete outcome (SWE/IWE reaching exactly 0,
// the 0.03 m snowfall threshold): an FMA there changes which cells are snow-free.
template <class P> __device__ __forceinline__ Num<P> xadd(Num<P> a, Num<P> b) {
  if constexpr (P::f32) return Num<P>(__fadd_rn(a.v, b.v)); else return Num<P>(__dadd_rn(a.v, b.v));
}
template <class P> __device__ __forceinline__ Num<P> xsub(Num<P> a, Num<P> b) {
  if constexpr (P::f32) return Num<P>(__fsub_rn(a.v, b.v)); else return Num<P>(__dsub_rn(a.v, b.v));
}
template <class P> __device__ __forceinline__ Num<P> xmul(Num<P> a, Num<P> b) {
  if constexpr (P::f32) return Num<P>(__fmul_rn(a.v, b.v)); else return Num<P>(__dmul_rn(a.v, b.v));
}
template <class P> __device__ __forceinline__ Num<P> xdiv(Num<P> a, Num<P> b) {
  if constexpr (P::f32) return Num<P>(__fdiv_rn(a.v, b.v)); else return Num<P>(__ddiv_rn(a.v, b.v));
}

// a/b with a single rounding and full IEEE semantics, arranged so that a ZERO NUMERATOR never enters CUDA's
// IEEE division: that routine sends a zero numerator down its ~100-instruction slow path, and if one lane of a
// warp does, the whole warp waits -- melt rates and rain are zero most of the time.  For a == 0 the quotient is
// a * (1/b): +-0 with the right sign, NaN for b = 0 or NaN.
template <class P> __device__ __forceinline__ Num<P> zdiv(Num<P> a, Num<P> b) {
  const bool z = (a.v == 0);
  const Num<P> q = xdiv(Num<P>(z ? static_cast<typename P::raw>(1.0) : a.v), b);
  return z ? xmul(a, q) : q;
}

// a / 3600 with a single rounding (the SWE/IWE mass balance, reference :1601-1606, :1612-1617).  Fast float64:
// Markstein's sequence q = a*y, r = fma(-3600, q, a), q' = fma(r, y, q) with y = RN(1/3600) is correctly rounded
// whenever r is exact, i.e. for a = 0 or |a| >= 2^-958 (tests/test_host_math.py); smaller values take the IEEE
// division.  3 FP64 instructions instead of ~13 and no slow path for the zero numerators that dominate.
template <class P> __device__ __forceinline__ Num<P> div3600(Num<P> a) {
  if constexpr (P::lean) {
    const unsigned hi = (unsigned)__double2hiint(a.v) & 0x7fffffffu;
    if (hi >= 0x04100000u || (hi | (unsigned)__double2loint(a.v)) == 0u) {
      const double y = 1.0 / 3600.0;
      const double q = __dmul_rn(a.v, y);
      return Num<P>(__fma_rn(__fma_rn(-3600.0, q, a.v), y, q));
    }
    return xdiv(a, Num<P>(3600.0));
  } else if constexpr (P::f32) {  // the same sequence in float32 (exact residual for |a| >= 2^-60, also under FTZ)
    if (fabsf(a.v) >= 8.6736174e-19f || a.v == 0.0f) {
      const float y = 1.0f / 3600.0f;
      const float q = __fmul_rn(a.v, y);
      return Num<P>(__fmaf_rn(__fmaf_rn(-3600.0f, q, a.v), y, q));
    }
    return zdiv(a, Num<P>(3600.0));
  } else {
    return zdiv(a, Num<P>(3600.0));
  }
}

// ---- transcendental functions ----------------------------------------------------------------------
template <class P> __device__ __forceinline__ Num<P> nsqrt(Num<P> a) {
  if constexpr (P::strict) return Num<P>(__dsqrt_rn(a.v));
  else if constexpr (P::f32) return Num<P>(__fsqrt_rn(a.v));
  else if constexpr (P::lean) return Num<P>(fm::sqrt_pos(a.v));
  else return Num<P>(sqrt(a.v));
}
template <class P> __device__ __forceinline__ Num<P> nexp(Num<P> a) {
  if constexpr (P::f32) return Num<P>(__expf(a.v));
  else if constexpr (P::lean) return Num<P>(fm::exp_tab(a.v));
  else return Num<P>(exp(a.v));
}
template <class P> __device__ __forceinline__ Num<P> nlog(Num<P> a) {
  if constexpr (P::f32) return Num<P>(__logf(a.v));
  else if constexpr (P::lean) return Num<P>(fm::log_tab(a.v));
  else return Num<P>(log(a.v));
}
template <class P> __device__ __forceinline__ Num<P> nsin(Num<P> a) {
  if constexpr (P::f32) return Num<P>(__sinf(a.v)); else return Num<P>(sin(a.v));
}
template <class P> __device__ __forceinline__ Num<P> ncos(Num<P> a) {
  if constexpr (P::f32) return Num<P>(__cosf(a.v)); else return Num<P>(cos(a.v));
}
template <class P> __device__ __forceinline__ Num<P> natan(Num<P> a) {
  if constexpr (P::f32) return Num<P>(fm::atan32(a.v));
  else if constexpr (P::lean) return Num<P>(fm::atan_core(a.v));
  else return Num<P>(atan(a.v));
}
template <class P> __device__ __forceinline__ Num<P> nacos(Num<P> a) {
  if constexpr (P::f32) return Num<P>(acosf(a.v)); else return Num<P>(acos(a.v));
}
// asin(x)*(180/pi) for x in [0,1] (fast modes only): the solar elevation angle in degrees
template <class P> __device__ __forceinline__ Num<P> nasin01(Num<P> a) {
  if constexpr (P::f32) return Num<P>(fm::asin01_32(a.v));
  else if constexpr (P::lean) return Num<P>(fm::asin01(a.v));
  else return Num<P>(asin(fmin(a.v, 1.0)));
}
// x**y for x > 0.  Strict: libdevice pow (NumPy calls its own / libm's pow).  Fast: exp(y*log(x)),
// whose relative error is ~|y*log(x)| ulp -- far inside the 1e-12 budget for the exponents used here.
template <class P> __device__ __forceinline__ Num<P> npow(Num<P> x, Num<P> y) {
  if constexpr (P::strict) return Num<P>(pow(x.v, y.v));
  else if constexpr (P::f32) return Num<P>(__expf(y.v * __logf(x.v)));
  else if constexpr (P::lean) return Num<P>(fm::exp_tab(y.v * fm::log_tab(x.v)));
  else return Num<P>(exp(y.v * log(x.v)));
}
template <class P> __device__ __forceinline__ Num<P> npow4(Num<P> x) {  // x**4.0
  if constexpr (P::strict) return Num<P>(pow(x.v, 4.0));
  else { auto s = x.v * x.v; return Num<P>(s * s); }
}
template <class P> __device__ __forceinline__ Num<P> npow15(Num<P> x) {  // x**1.5
  if constexpr (P::strict) return Num<P>(pow(x.v, 1.5));
  else return x * nsqrt(x);
}

}  // namespace tfg
