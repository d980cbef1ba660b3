// TEST-ONLY host build of the float formats' gray conversion (aprilgrid-rs_b200/csrc/ag_float_luma.h),
// linked into the host build of the board core, so that the CPU test-suite can compare the code K1 and
// the board kernel share with a restatement of `image`'s conversion.  Never part of the shipped library.
#include <stdint.h>

#include "ag_float_luma.h"

extern "C" {

// rgb: n pixels of `channels` (3 or 4) f32 -> to_luma32f and to_luma8 of each.
int hb_float_luma(const float* rgb, long long n, int channels, float* out_luma32f, uint8_t* out_luma8) {
  if (channels != 3 && channels != 4) return -1;
  for (long long i = 0; i < n; ++i) {
    const float* p = rgb + channels * i;
    out_luma32f[i] = ag::rgb32f_luma(p[0], p[1], p[2]);
    out_luma8[i] = (uint8_t)ag::luma32f_to_u8(out_luma32f[i]);
  }
  return 0;
}

}  // extern "C"
