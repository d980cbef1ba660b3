// Shared definitions of the aprilgrid B200 kernels.
//
// Arithmetic contract (SURVEY.md section 0.3): the Rust reference never contracts a*b+c,
// so every f32 expression on the parity path is "round the product, then round the sum".
// The library is compiled with -fmad=false AND the parity-critical expressions use the
// __fmul_rn/__fadd_rn/__fsub_rn/__fdiv_rn intrinsics, which the compiler never fuses.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/aprilgrid_b200.h"
#include "ag_float_luma.h"

#if defined(__CUDACC__)
#define AG_HD __host__ __device__ __forceinline__
#define AG_D __device__ __forceinline__
#else
#define AG_HD inline
#define AG_D inline
#endif

namespace ag {

// Internal pixel format of ag_detect_planes: the frame's Luma<f32> plane (the caller ran
// to_luma32f itself); not a value of the public format enum.
constexpr int kFmtF32 = 3;

// Bytes of one pixel of format `fmt` (a public AG_* format or kFmtF32); 0 for any other value.
AG_HD constexpr int bytes_per_px(int fmt) {
  return fmt == AG_L8 ? 1 : fmt == AG_L16 ? 2 : fmt == AG_RGB8 ? 3 : fmt == kFmtF32 ? 4 : fmt == AG_LA8 ? 2
       : fmt == AG_RGBA8 ? 4 : fmt == AG_LA16 ? 4 : fmt == AG_RGB16 ? 6 : fmt == AG_RGBA16 ? 8
       : fmt == AG_RGB32F ? 12 : fmt == AG_RGBA32F ? 16 : 0;
}
// Alignment in bytes of a pixel's channel words (1, 2 or 4): row strides, frame strides and the
// address of device frames must be multiples of it (K1 and K6 read the words with loads of that size).
AG_HD constexpr int channel_align(int fmt) {
  return fmt == AG_L16 || fmt == AG_LA16 || fmt == AG_RGB16 || fmt == AG_RGBA16 ? 2
       : fmt == AG_RGB32F || fmt == AG_RGBA32F ? 4 : 1;
}

constexpr int kBlurRadius = 3;  // ceil(2 * 1.5), src/image_util.rs:111
constexpr int kBlurTaps = 7;

// Per-frame capacities / geometry shared by kernels and host.
struct FrameGeom {
  int w, h;             // image size in pixels
  int wpr;              // mask words (32 px) per row
  int n_words;          // wpr * h
  int n_px;             // w * h
  size_t frame_stride;  // bytes between input frames
  size_t row_stride;    // bytes between input rows
  int format;           // a public AG_* pixel format, or kFmtF32
  // frame lists (ag_detect_frames_device): device table of the chunk's frame addresses, used in place
  // of frames + f * frame_stride when set; ptr_bits = the OR of those addresses, for the launchers'
  // alignment checks (the table itself is not readable on the host)
  const uint8_t* const* frame_ptrs = nullptr;
  uintptr_t ptr_bits = 0;
};

// First byte of frame f of a chunk.
AG_HD const uint8_t* frame_base(const uint8_t* frames, const FrameGeom& g, int f) {
  return g.frame_ptrs ? g.frame_ptrs[f] : frames + (size_t)f * g.frame_stride;
}

// Monotone float <-> uint key so that atomicMin on the key is a float min.
AG_HD uint32_t float_to_ordered(float f) {
#if defined(__CUDA_ARCH__)
  uint32_t b = __float_as_uint(f);
#else
  union { float f; uint32_t u; } c; c.f = f; uint32_t b = c.u;
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
AG_HD float ordered_to_float(uint32_t k) {
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#if defined(__CUDA_ARCH__)
  return __uint_as_float(b);
#else
  union { float f; uint32_t u; } c; c.u = b; return c.f;
#endif
}
constexpr uint32_t kOrderedFltMax = 0xff7fffffu;  // float_to_ordered(FLT_MAX)

}  // namespace ag
