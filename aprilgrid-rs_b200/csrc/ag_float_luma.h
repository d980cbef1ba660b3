// Gray conversion of the float pixel formats (AG_RGB32F, AG_RGBA32F), as `image` 0.25 does it:
// to_luma32f for the stencils (src/detector.rs:409), to_luma8 for bit sampling (:507).  Written once
// for K1, the board kernel's bit sampling and the host test build of the board core
// (tests/host_board_test.cpp, tests/host_float_luma.cpp), so all three compute the same bits.
//
// rgb_to_luma on Rgb<f32> runs in f32::Larger = f64 (the reading is written down next to the
// format enum in include/aprilgrid_b200.h):
//   S = RN64(RN64(2126 r + 7152 g) + 722 b)   r, g, b widened to f64; the products are exact
//   L = (f32) clamp(RN64(S / 10000), -kLumaF32Bound, kLumaF32Bound)
//   to_luma32f = L,   to_luma8 = (u8) round_half_away(RN32(clamp(L, 0, 1) * 255))
// Alpha never enters.  Finite inputs only: NaN and infinities give unspecified (but memory-safe) values.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define AG_LUMA_HD __host__ __device__ __forceinline__
#else
#define AG_LUMA_HD inline
#endif

namespace ag {

// Enlargeable::clamp_from's bounds for f32 (Bounded::min_value / max_value = -+f32::MAX, as f64).
// No finite pixel reaches them: |S| / 10000 <= f32::MAX.
constexpr double kLumaF32Bound = 3.4028234663852886e+38;

// RN64(1 / 10000), the reciprocal Markstein's division below starts from.
constexpr double kInv10000 = 1.0e-4;

// to_luma32f of one R G B f32 pixel.  S / 10000 is divided as Markstein's correctly rounded division
// by a constant: with y = RN(1/10000) and q = RN(S y) (within an ulp of S / 10000), the residual
// S - 10000 q is exact (one FMA) and RN(q + residual y) is RN(S / 10000) -- no underflow or overflow
// is possible for |S| in [2^-149 * 722, 10000 * f32::MAX].  An exact quotient (residual 0) keeps q,
// so that -0.0 stays -0.0.  (__ddiv_rn computes the same bits but calls an out-of-line slow path
// that makes K1 spill.)
AG_LUMA_HD float rgb32f_luma(float r, float g, float b) {
#if defined(__CUDA_ARCH__)
  const double s = __dadd_rn(__dadd_rn(__dmul_rn(2126.0, (double)r), __dmul_rn(7152.0, (double)g)),
                             __dmul_rn(722.0, (double)b));
  const double q0 = __dmul_rn(s, kInv10000);
  const double rem = __fma_rn(-q0, 10000.0, s);
  double q = rem == 0.0 ? q0 : __fma_rn(rem, kInv10000, q0);
#else  // host (IEEE double arithmetic without contraction: the products are exact, one rounding per op)
  volatile double s = 2126.0 * (double)r + 7152.0 * (double)g;
  s = s + 722.0 * (double)b;
  volatile double q0 = s * kInv10000;
  const double rem = fma(-q0, 10000.0, s);
  volatile double q = rem == 0.0 ? q0 : fma(rem, kInv10000, q0);
#endif
  q = q < -kLumaF32Bound ? -kLumaF32Bound : (q > kLumaF32Bound ? kLumaF32Bound : q);
#if defined(__CUDA_ARCH__)
  return __double2float_rn(q);
#else
  return (float)q;
#endif
}

// to_luma8 of a to_luma32f value (image's FromPrimitive<f32> for u8): clamp to [0, 1], scale, round
// half away from zero.
AG_LUMA_HD uint32_t luma32f_to_u8(float l) {
  const float c = fminf(fmaxf(l, 0.0f), 1.0f);
#if defined(__CUDA_ARCH__)
  return (uint32_t)roundf(__fmul_rn(c, 255.0f));
#else
  volatile float y = c * 255.0f;
  return (uint32_t)roundf(y);
#endif
}

}  // namespace ag
