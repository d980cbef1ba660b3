// Dense per-pixel stages of the aprilgrid front end, sm_100a.
//
//   K1  k_blur_hessian_*   gray conversion -> 7-tap separable Gaussian (sigma 1.5) ->
//                          3x3 determinant-of-Hessian -> per-frame min
//                          reference: src/detector.rs:409-418, src/image_util.rs:72-206
//   K2  k_threshold_mask   mask = resp < 0.05 * min, packed 32 px / word
//                          reference: src/detector.rs:418, :176-177 (the `v < threshold` test)
//
// All arithmetic is bit-exact with the reference: products and sums are rounded separately
// (no FMA), taps are accumulated in tap order 0..6 starting from 0, and the taps themselves
// are the glibc-expf values the reference computes at run time.
#include "ag_common.cuh"
#include "ag_kernels.h"

namespace ag {

// Normalised Gaussian taps for sigma = 1.5 (src/image_util.rs:111-124, f32::exp = expf).
// tests/test_oracle_pins.py checks these bit patterns against the oracle's run-time taps.
__constant__ float c_taps[kBlurTaps] = {
    0x1.2c18a6p-5f /*0x3d160c53*/, 0x1.c7ce56p-4f /*0x3de3e72b*/, 0x1.bbe4fap-3f /*0x3e5df27d*/,
    0x1.152db4p-2f /*0x3e8a96da*/, 0x1.bbe4fap-3f, 0x1.c7ce56p-4f, 0x1.2c18a6p-5f};

// ---- gray conversion (image 0.25: to_luma32f) ------------------------------------------
// v / 255 and v / 65535 correctly rounded, as two FP ops: with r_hi + r_lo = 1/max split in
// two floats, fma(v, r_hi, v * r_lo) equals RN(v / max) for every u8 / u16 v (checked
// exhaustively by tests/test_gpu_parity.py::test_unorm_conversion_exhaustive).
AG_D float unorm8_to_f32(float v) {
  const float rh = __uint_as_float(0x3b808081u), rl = __uint_as_float(0xaf7efeffu);
  return __fmaf_rn(v, rh, __fmul_rn(v, rl));
}
AG_D float unorm16_to_f32(float v) {
  const float rh = __uint_as_float(0x37800080u), rl = __uint_as_float(0x27800080u);
  return __fmaf_rn(v, rh, __fmul_rn(v, rl));
}
// image::color::rgb_to_luma on u8: integer sRGB weights, truncating division by 10000.
AG_D uint32_t rgb_luma_u8(uint32_t r, uint32_t g, uint32_t b) {
  return (2126u * r + 7152u * g + 722u * b) / 10000u;
}
// The same on u16 (Y16); the largest sum, 655 350 000, fits 32 bits.
AG_D uint32_t rgb_luma_u16(uint32_t r, uint32_t g, uint32_t b) {
  return (2126u * r + 7152u * g + 722u * b) / 10000u;
}

template <int FMT>
AG_D float load_luma(const uint8_t* __restrict__ frame, size_t row_stride, int x, int y) {
  const uint8_t* row = frame + (size_t)y * row_stride;
  const uint16_t* row16 = reinterpret_cast<const uint16_t*>(row);
  if (FMT == AG_L8) {
    return unorm8_to_f32((float)row[x]);
  } else if (FMT == AG_L16) {
    return unorm16_to_f32((float)row16[x]);
  } else if (FMT == kFmtF32) {
    return reinterpret_cast<const float*>(row)[x];
  } else if (FMT == AG_LA8) {  // alpha never contributes
    return unorm8_to_f32((float)row[2 * x]);
  } else if (FMT == AG_RGBA8) {
    const uint8_t* p = row + 4 * x;
    return unorm8_to_f32((float)rgb_luma_u8(p[0], p[1], p[2]));
  } else if (FMT == AG_LA16) {
    return unorm16_to_f32((float)row16[2 * x]);
  } else if (FMT == AG_RGB16 || FMT == AG_RGBA16) {
    const uint16_t* p = row16 + (FMT == AG_RGB16 ? 3 : 4) * x;
    return unorm16_to_f32((float)rgb_luma_u16(p[0], p[1], p[2]));
  } else if (FMT == AG_RGB32F || FMT == AG_RGBA32F) {
    const float* p = reinterpret_cast<const float*>(row) + (FMT == AG_RGB32F ? 3 : 4) * x;
    return rgb32f_luma(p[0], p[1], p[2]);
  } else {
    const uint8_t* p = row + 3 * x;
    return unorm8_to_f32((float)rgb_luma_u8(p[0], p[1], p[2]));
  }
}

AG_D float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// -----------------------------------------------------------------------------------------
// K1, generic tile version (any format, any size, any stride).  One CTA = 64 x 32 outputs.
// Used for L16 / RGB8 inputs and as the cross-check of the streaming L8 kernel.
// -----------------------------------------------------------------------------------------
constexpr int T_W = 64, T_H = 32;
constexpr int IN_W = T_W + 8, IN_H = T_H + 8;    // input halo: 3 (blur) + 1 (Hessian)
constexpr int TMP_W = T_W + 2, TMP_H = T_H + 8;  // H-pass output
constexpr int BL_W = T_W + 2, BL_H = T_H + 2;    // blurred tile incl. Hessian halo
constexpr int TMP_LD = TMP_W + 1, BL_LD = BL_W + 1;

template <int FMT, bool WRITE_BLUR>
__global__ void __launch_bounds__(256)
k_blur_hessian_tile(const uint8_t* __restrict__ frames, FrameGeom g, float* __restrict__ blur,
                    float* __restrict__ resp, uint32_t* __restrict__ frame_min) {
  __shared__ float s_in[IN_H][IN_W];
  __shared__ float s_tmp[TMP_H][TMP_LD];
  __shared__ float s_bl[BL_H][BL_LD];
  __shared__ float s_red[8];

  const int tid = threadIdx.x;
  const int x0 = blockIdx.x * T_W, y0 = blockIdx.y * T_H;
  const int f = blockIdx.z;
  const uint8_t* frame = frame_base(frames, g, f);

  // 1. gray conversion of the clamped (edge-replicated) input window
  for (int i = tid; i < IN_H * IN_W; i += 256) {
    int iy = i / IN_W, ix = i - iy * IN_W;
    int gx = min(max(x0 - 4 + ix, 0), g.w - 1);
    int gy = min(max(y0 - 4 + iy, 0), g.h - 1);
    s_in[iy][ix] = load_luma<FMT>(frame, g.row_stride, gx, gy);
  }
  __syncthreads();
  // 2. horizontal pass: val = 0; val += px * k[i], i = 0..6   (image_util.rs:138-185)
  for (int i = tid; i < TMP_H * TMP_W; i += 256) {
    int iy = i / TMP_W, jx = i - iy * TMP_W;
    float val = 0.0f;
#pragma unroll
    for (int t = 0; t < kBlurTaps; ++t) val = __fadd_rn(val, __fmul_rn(s_in[iy][jx + t], c_taps[t]));
    s_tmp[iy][jx] = val;
  }
  __syncthreads();
  // 3. vertical pass: out = 0; out += temp[ky] * k[i]           (image_util.rs:188-203)
  for (int i = tid; i < BL_H * BL_W; i += 256) {
    int jy = i / BL_W, jx = i - jy * BL_W;
    float val = 0.0f;
#pragma unroll
    for (int t = 0; t < kBlurTaps; ++t) val = __fadd_rn(val, __fmul_rn(s_tmp[jy + t][jx], c_taps[t]));
    s_bl[jy][jx] = val;
  }
  __syncthreads();
  // 4. Hessian response on the interior, 0 on the image border  (image_util.rs:83-106)
  float mn = 3.40282347e+38f;
  for (int i = tid; i < T_H * T_W; i += 256) {
    int ty = i / T_W, tx = i - ty * T_W;
    int gx = x0 + tx, gy = y0 + ty;
    if (gx >= g.w || gy >= g.h) continue;
    float r = 0.0f;
    if (gx >= 1 && gx < g.w - 1 && gy >= 1 && gy < g.h - 1) {
      float v11 = s_bl[ty][tx], v12 = s_bl[ty][tx + 1], v13 = s_bl[ty][tx + 2];
      float v21 = s_bl[ty + 1][tx], v22 = s_bl[ty + 1][tx + 1], v23 = s_bl[ty + 1][tx + 2];
      float v31 = s_bl[ty + 2][tx], v32 = s_bl[ty + 2][tx + 1], v33 = s_bl[ty + 2][tx + 2];
      float t2 = __fmul_rn(v22, 2.0f);
      float lxx = __fadd_rn(__fsub_rn(v21, t2), v23);
      float lyy = __fadd_rn(__fsub_rn(v12, t2), v32);
      float lxy = __fmul_rn(__fsub_rn(__fadd_rn(__fsub_rn(v13, v11), v31), v33), 0.25f);
      r = __fsub_rn(__fmul_rn(lxx, lyy), __fmul_rn(lxy, lxy));
    }
    size_t o = (size_t)f * g.n_px + (size_t)gy * g.w + gx;
    resp[o] = r;
    if (WRITE_BLUR) blur[o] = s_bl[ty + 1][tx + 1];
    mn = fminf(mn, r);
  }
  // 5. per-frame min (detector.rs:414-417)
  mn = warp_min(mn);
  if ((tid & 31) == 0) s_red[tid >> 5] = mn;
  __syncthreads();
  if (tid < 32) {
    float v = tid < 8 ? s_red[tid] : 3.40282347e+38f;
    v = warp_min(v);
    if (tid == 0) atomicMin(&frame_min[f], float_to_ordered(v));
  }
}

// -----------------------------------------------------------------------------------------
// K1, streaming version (8-bit gray is the benchmark path; 16-bit gray and RGB8 share it).
//
// One WARP owns a strip of 120 output columns (it computes 128: lanes 0 and 31 only provide the
// blurred halo column their neighbours need) and marches down a chunk of rows.  Each lane owns
// 4 adjacent columns, so the input is one coalesced 128-byte load per warp-row and the outputs
// are 480-byte float4 stores.  Everything between load and store lives in registers:
//   * horizontal pass: a 10-pixel window per lane, the 3 + 3 halo pixels come from the
//     neighbouring lanes by warp shuffle;
//   * vertical pass: 7 running partial sums per column.  A new horizontal-pass value t of row r
//     is the tap-i term of output row r + 3 - i; rows arrive in increasing r, so each output
//     row receives its terms in tap order 0..6 -- the reference's accumulation order -- and
//     the symmetric taps need only 4 products;
//   * Hessian: the last three blurred rows of the 4 columns plus one halo column per side.
// No shared memory, no block barrier.  Clamp-to-edge is obtained by clamping the loaded row /
// replicating the edge pixel.  Requires width % 4 == 0 and rows aligned to the lane's load
// (4 bytes for L8 and RGB8 -- a lane's 4 RGB pixels are three words --, 8 bytes for L16, LA8 and
// RGB16, 16 bytes for the other formats; see launch_blur_hessian).
// -----------------------------------------------------------------------------------------
constexpr int S_COLS = 120;  // output columns per warp
// Output rows per warp (chunk): the launcher picks one of these.  chunk + 8 row steps (7 rows of
// blur halo + 1 of Hessian halo) is a whole number of six-step loop trips for each of them.
// Taller chunks recompute less halo but leave a longer tail of half-empty SMs: measured on 1024
// frames of 1280x1024, 124 rows 0.663 of the HBM peak, 250 rows 0.653, 508 rows 0.637, 58 rows 0.647.
constexpr int kChunkRows[] = {124, 58};
constexpr int S_WARPS = 4;   // warps per CTA (adjacent strips of one row chunk)

AG_D float u8_lane(uint32_t word, int k) {  // byte k of a packed pixel word -> luma f32
  return unorm8_to_f32((float)((word >> (8 * k)) & 0xffu));
}

// A lane's 4 raw pixels of one row: as many 32-bit words as a pixel has bytes (1 for L8 ... 16 for RGBA32F).
template <int FMT>
struct RawPx {
  static constexpr int NW = bytes_per_px(FMT);
  uint32_t w[NW];
};
// What a lane keeps of a row of format FMT until its use.  The formats with alpha, 16-bit colour or
// float colour are reduced to gray one row step after the load, to one L8 word (LA8, RGBA8: the luma
// bytes), two L16 words (LA16, RGB16, RGBA16: the luma words) or four f32 words (RGB32F, RGBA32F:
// to_luma32f), so that only the newest row in flight costs its raw registers and the rest of the row
// step is the L8 / L16 / f32 code.
template <int FMT>
constexpr int kLaneFmt = (FMT == AG_LA8 || FMT == AG_RGBA8) ? AG_L8
                       : (FMT == AG_LA16 || FMT == AG_RGB16 || FMT == AG_RGBA16) ? AG_L16
                       : (FMT == AG_RGB32F || FMT == AG_RGBA32F) ? kFmtF32 : FMT;
AG_D uint32_t lo16(uint32_t v) { return v & 0xffffu; }
AG_D uint32_t hi16(uint32_t v) { return v >> 16; }
AG_D uint32_t rgba8_luma(uint32_t px) {  // one R G B A pixel word -> Y8
  return rgb_luma_u8(px & 0xffu, (px >> 8) & 0xffu, (px >> 16) & 0xffu);
}
// A lane's raw words of one row (vector loads as wide as the lane's alignment allows).
template <int FMT>
AG_D RawPx<FMT> load_raw(const uint8_t* p) {
  RawPx<FMT> r;
  constexpr int NW = RawPx<FMT>::NW;
  if (NW == 2) {  // L16, LA8: one 8-byte load
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    r.w[0] = v.x;
    r.w[NW - 1] = v.y;
  } else if (NW % 4 == 0) {  // f32, RGBA8, LA16: one 16-byte load; RGBA16: two; RGB32F: three; RGBA32F: four
#pragma unroll
    for (int i = 0; i < NW; i += 4) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(p) + i / 4);
      r.w[i] = v.x;
      r.w[(i + 1) % NW] = v.y;
      r.w[(i + 2) % NW] = v.z;
      r.w[(i + 3) % NW] = v.w;
    }
  } else if (NW == 6) {  // RGB16: three 8-byte loads
#pragma unroll
    for (int i = 0; i < NW; i += 2) {
      const uint2 v = __ldg(reinterpret_cast<const uint2*>(p) + i / 2);
      r.w[i] = v.x;
      r.w[(i + 1) % NW] = v.y;
    }
  } else {  // L8, RGB8: 32-bit words
#pragma unroll
    for (int i = 0; i < NW; ++i) r.w[i] = __ldg(reinterpret_cast<const uint32_t*>(p) + i);
  }
  return r;
}
// A lane's raw words -> what it keeps of the row (kLaneFmt); the identity for L8, L16, RGB8 and f32.
template <int FMT>
AG_D RawPx<kLaneFmt<FMT>> pack_raw(const RawPx<FMT>& v) {
  if constexpr (kLaneFmt<FMT> == FMT) {
    return v;
  } else {
    RawPx<kLaneFmt<FMT>> r;
    constexpr int NW = RawPx<kLaneFmt<FMT>>::NW, NI = RawPx<FMT>::NW;
    const uint32_t* x = v.w;
    if (FMT == AG_LA8) {  // L A L A | L A L A -> L L L L
      r.w[0] = __byte_perm(x[0], x[1 % NI], 0x6420);
    } else if (FMT == AG_RGBA8) {  // a pixel per word
      r.w[0] = rgba8_luma(x[0]) | (rgba8_luma(x[1 % NI]) << 8) | (rgba8_luma(x[2 % NI]) << 16) |
               (rgba8_luma(x[3 % NI]) << 24);
    } else if (FMT == AG_LA16) {  // L A per word
      r.w[0] = __byte_perm(x[0], x[1 % NI], 0x5410);
      r.w[1 % NW] = __byte_perm(x[2 % NI], x[3 % NI], 0x5410);
    } else if (FMT == AG_RGB32F || FMT == AG_RGBA32F) {  // R G B (A) per pixel, one f32 per word
      constexpr int C = FMT == AG_RGB32F ? 3 : 4;
#pragma unroll
      for (int k = 0; k < 4; ++k)
        r.w[k % NW] = __float_as_uint(rgb32f_luma(__uint_as_float(x[(C * k) % NI]), __uint_as_float(x[(C * k + 1) % NI]),
                                                  __uint_as_float(x[(C * k + 2) % NI])));
    } else if (FMT == AG_RGB16) {  // R0 G0 | B0 R1 | G1 B1 | R2 G2 | B2 R3 | G3 B3
      r.w[0] = rgb_luma_u16(lo16(x[0]), hi16(x[0]), lo16(x[1 % NI])) |
               (rgb_luma_u16(hi16(x[1 % NI]), lo16(x[2 % NI]), hi16(x[2 % NI])) << 16);
      r.w[1 % NW] = rgb_luma_u16(lo16(x[3 % NI]), hi16(x[3 % NI]), lo16(x[4 % NI])) |
                    (rgb_luma_u16(hi16(x[4 % NI]), lo16(x[5 % NI]), hi16(x[5 % NI])) << 16);
    } else {  // RGBA16: R G | B A per pixel
      r.w[0] = rgb_luma_u16(lo16(x[0]), hi16(x[0]), lo16(x[1 % NI])) |
               (rgb_luma_u16(lo16(x[2 % NI]), hi16(x[2 % NI]), lo16(x[3 % NI])) << 16);
      r.w[1 % NW] = rgb_luma_u16(lo16(x[4 % NI]), hi16(x[4 % NI]), lo16(x[5 % NI])) |
                    (rgb_luma_u16(lo16(x[6 % NI]), hi16(x[6 % NI]), lo16(x[7 % NI])) << 16);
    }
    return r;
  }
}
// luma f32 of pixel k (0..3) of the lane's raw pixels (image 0.25 to_luma32f, see load_luma)
template <int FMT>
AG_D float raw_luma(const RawPx<FMT>& r, int k) {
  if (FMT == AG_L8) {
    return u8_lane(r.w[0], k);
  } else if (FMT == kFmtF32) {  // a to_luma32f plane handed in as is (ag_detect_planes)
    return __uint_as_float(r.w[k % RawPx<FMT>::NW]);
  } else if (FMT == AG_L16) {
    return unorm16_to_f32((float)((r.w[(k >> 1) % RawPx<FMT>::NW] >> (16 * (k & 1))) & 0xffffu));
  } else {
    auto byte = [&](int j) { return (r.w[(j >> 2) % RawPx<FMT>::NW] >> (8 * (j & 3))) & 0xffu; };
    return unorm8_to_f32((float)rgb_luma_u8(byte(3 * k), byte(3 * k + 1), byte(3 * k + 2)));
  }
}

struct BlurRow {  // one blurred row: v[1..4] = the lane's 4 columns, v[0] / v[5] = halo columns
  float v[6];
};

template <int FMT, bool WRITE_BLUR>
#ifndef AG_K1_MIN_BLOCKS
#define AG_K1_MIN_BLOCKS 7
#endif
// The float formats keep a row of 12 or 16 raw words in flight and convert it in f64: they need 114-120
// registers, four blocks per SM (at 80 or 96 registers they spill).
__global__ void __launch_bounds__(S_WARPS * 32, FMT == AG_L8 ? AG_K1_MIN_BLOCKS
                                                : (FMT == AG_RGB32F || FMT == AG_RGBA32F) ? 4 : 6)
k_blur_hessian_stream(const uint8_t* __restrict__ frames, FrameGeom g, int chunk_rows, float* __restrict__ blur,
                      float* __restrict__ resp, uint32_t* __restrict__ frame_min) {
  const int lane = threadIdx.x & 31;
  const int strip = blockIdx.x * S_WARPS + (threadIdx.x >> 5);
  const int X0 = strip * S_COLS;
  if (X0 >= g.w) return;
  const int f = blockIdx.z;
  const int Y0 = blockIdx.y * chunk_rows, Y1 = min(Y0 + chunk_rows, g.h);
  const int c0 = X0 - 4 + 4 * lane;  // first of this lane's 4 columns (may lie outside the image)
  const int cw = min(max(c0, 0), g.w - 4);  // column of the word actually loaded
  constexpr int kBpp = bytes_per_px(FMT);
  constexpr int LF = kLaneFmt<FMT>;  // the format of what load_raw returns
  // frame bases are block-uniform; what varies per lane and row are 32-bit offsets (the launcher
  // checks that a frame's bytes fit them)
  // The lane's pointers into the frame are held in registers (opaque, or the compiler re-derives
  // them from blockIdx in every row step); a row then costs one 32x32->64 multiply-add per access.
  const uint8_t* src = frame_base(frames, g, f) + (size_t)cw * kBpp;
  asm volatile("" : "+l"(src));
  const uint32_t rs = (uint32_t)g.row_stride;
  const bool left_out = c0 < 0, right_out = c0 >= g.w;
  // strips at the left / right image border: replicated pixels, zeroed border columns
  const bool edge_strip = X0 == 0 || X0 + S_COLS + 4 >= g.w;  // warp-uniform
  const bool zero_first = c0 == 0, zero_last = c0 + 3 == g.w - 1;  // image border columns
  const float k0 = c_taps[0], k1 = c_taps[1], k2 = c_taps[2], k3 = c_taps[3];
  const int h1 = g.h - 1;
  // one register each for what every row step tests (kept opaque so that they are not recomputed
  // from the thread index in every step)
  int writer = (lane >= 1 && lane <= 30 && !right_out) ? 1 : 0;
  asm volatile("" : "+r"(writer));
  const int row_lo = max(Y0, 1);                         // first row with a non-zero response
  const uint32_t emit_span = (uint32_t)(Y1 - Y0);        // rows this chunk writes
  const uint32_t calc_span = (uint32_t)max(min(Y1, h1) - row_lo, 0);  // ... and computes

  auto load_row = [&](int r) -> RawPx<FMT> {
    const uint32_t rr = (uint32_t)min(max(r, 0), h1);
    return load_raw<FMT>(src + (uint64_t)rr * rs);
  };

  // vertical partial sums: aj[c] = what output row (r + 3 - j) has accumulated so far
  float a1[4], a2[4], a3[4], a4[4], a5[4], a6[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) a1[c] = a2[c] = a3[c] = a4[c] = a5[c] = a6[c] = 0.0f;
  BlurRow R0, R1, R2;
#pragma unroll
  for (int c = 0; c < 6; ++c) R0.v[c] = R1.v[c] = R2.v[c] = 0.0f;
  float mn = 3.40282347e+38f;
  char* resp_l = reinterpret_cast<char*>(resp + ((size_t)f * g.n_px + c0));  // row 0, the lane's columns
  char* blur_l = reinterpret_cast<char*>(blur + ((size_t)f * g.n_px + c0));
  asm volatile("" : "+l"(resp_l));
  if (WRITE_BLUR) asm volatile("" : "+l"(blur_l));
  const uint32_t out_row_bytes = (uint32_t)g.w * 4u;

  const int r_begin = Y0 - 4, r_end = Y1 + 3;  // temp rows r_begin..r_end inclusive
  // rows r + 1 and r + 2 as kept (kLaneFmt), row r + 3 as loaded: a row is reduced one step after its
  // load, when the load has had a row step to arrive
  RawPx<LF> w_cur = pack_raw<FMT>(load_row(r_begin)), w_n1 = pack_raw<FMT>(load_row(r_begin + 1));
  RawPx<FMT> w_n2 = load_row(r_begin + 2);

  // One row step: consumes raw row r, completes blurred row r-3 into N, emits Hessian row r-4
  // from M (row r-5), C (row r-4), N (row r-3).
  auto step = [&](int r, const BlurRow& M, const BlurRow& C, BlurRow& N) {
    RawPx<LF> wd = w_cur;
    w_cur = w_n1;
    w_n1 = pack_raw<FMT>(w_n2);
    w_n2 = load_row(r + 3);  // three rows ahead
    if (LF == AG_L8 && edge_strip) {
      if (left_out) wd.w[0] = (wd.w[0] & 0xffu) * 0x01010101u;  // replicate pixel 0
      if (right_out) wd.w[0] = (wd.w[0] >> 24) * 0x01010101u;   // replicate pixel w-1
    }
    // ---- gray conversion + halo exchange: p[0..9] = pixels c0-3 .. c0+6
    float p[10];
    p[3] = raw_luma<LF>(wd, 0); p[4] = raw_luma<LF>(wd, 1); p[5] = raw_luma<LF>(wd, 2);
    p[6] = raw_luma<LF>(wd, 3);
    if (LF != AG_L8 && edge_strip) {  // strips hanging over the image edge replicate the edge pixel
      if (left_out) p[4] = p[5] = p[6] = p[3];
      if (right_out) p[3] = p[4] = p[5] = p[6];
    }
    p[0] = __shfl_up_sync(0xffffffffu, p[4], 1);
    p[1] = __shfl_up_sync(0xffffffffu, p[5], 1);
    p[2] = __shfl_up_sync(0xffffffffu, p[6], 1);
    p[7] = __shfl_down_sync(0xffffffffu, p[3], 1);
    p[8] = __shfl_down_sync(0xffffffffu, p[4], 1);
    p[9] = __shfl_down_sync(0xffffffffu, p[5], 1);
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      // ---- horizontal pass (image_util.rs:138-185): val = 0; val += px * k[i], i = 0..6
      //      (0.0 + x*k0 == x*k0 for x >= 0; an f32 plane or float pixels may give negative values or
      //      -0.0, where 0.0 + (-0.0) = +0.0, so those instantiations keep the addition)
      float t = __fmul_rn(p[c], k0);
      if (LF == kFmtF32) t = __fadd_rn(0.0f, t);
      t = __fadd_rn(t, __fmul_rn(p[c + 1], k1));
      t = __fadd_rn(t, __fmul_rn(p[c + 2], k2));
      t = __fadd_rn(t, __fmul_rn(p[c + 3], k3));
      t = __fadd_rn(t, __fmul_rn(p[c + 4], k2));
      t = __fadd_rn(t, __fmul_rn(p[c + 5], k1));
      t = __fadd_rn(t, __fmul_rn(p[c + 6], k0));
      // ---- vertical pass (image_util.rs:188-203): temp row r is tap i of output row r + 3 - i
      const float q0 = __fmul_rn(t, k0), q1 = __fmul_rn(t, k1), q2 = __fmul_rn(t, k2),
                  q3 = __fmul_rn(t, k3);
      N.v[c + 1] = __fadd_rn(a6[c], q0);  // tap 6 completes row r - 3
      a6[c] = __fadd_rn(a5[c], q1);       // tap 5 of row r - 2
      a5[c] = __fadd_rn(a4[c], q2);       // tap 4 of row r - 1
      a4[c] = __fadd_rn(a3[c], q3);       // tap 3 of row r
      a3[c] = __fadd_rn(a2[c], q2);       // tap 2 of row r + 1
      a2[c] = __fadd_rn(a1[c], q1);       // tap 1 of row r + 2
      a1[c] = LF == kFmtF32 ? __fadd_rn(0.0f, q0) : q0;  // tap 0 of row r + 3 (0.0 + q0)
    }
    N.v[0] = __shfl_up_sync(0xffffffffu, N.v[4], 1);
    N.v[5] = __shfl_down_sync(0xffffffffu, N.v[1], 1);
    // ---- Hessian of row yh = r - 4 (image_util.rs:83-106)
    const int yh = r - 4;
    if ((uint32_t)(yh - Y0) < emit_span) {  // warp-uniform: Y0 <= yh < Y1
      float o[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      if ((uint32_t)(yh - row_lo) < calc_span) {  // warp-uniform; border rows stay 0
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float t2 = __fmul_rn(C.v[c + 1], 2.0f);
          const float lxx = __fadd_rn(__fsub_rn(C.v[c], t2), C.v[c + 2]);
          const float lyy = __fadd_rn(__fsub_rn(M.v[c + 1], t2), N.v[c + 1]);
          const float lxy =
              __fmul_rn(__fsub_rn(__fadd_rn(__fsub_rn(M.v[c + 2], M.v[c]), N.v[c]), N.v[c + 2]), 0.25f);
          o[c] = __fsub_rn(__fmul_rn(lxx, lyy), __fmul_rn(lxy, lxy));
        }
        if (edge_strip) {
          if (zero_first) o[0] = 0.0f;
          if (zero_last) o[3] = 0.0f;
        }
      }
      if (writer) {
        const uint64_t off = (uint64_t)(uint32_t)yh * out_row_bytes;
        __stcs(reinterpret_cast<float4*>(resp_l + off), make_float4(o[0], o[1], o[2], o[3]));
        if (WRITE_BLUR)
          __stcs(reinterpret_cast<float4*>(blur_l + off), make_float4(C.v[1], C.v[2], C.v[3], C.v[4]));
        mn = fminf(fminf(mn, fminf(o[0], o[1])), fminf(o[2], o[3]));
      }
    }
  };

  // The three blurred rows rotate roles with period 3 and the six partial sums of a column move up
  // one position per row (period 6), so six unconditional steps per trip leave EVERY value in the
  // register it started in: no register copies, no per-step loop tests.  Against a three-step loop
  // with a conditional tail that is 11 % fewer instructions (K1 alone: 0.56 -> 0.66 of the measured
  // HBM peak).  The chunk heights make chunk + 8 a multiple of six; in the last chunk of a frame the
  // steps past r_end load clamped rows and emit nothing (yh >= Y1).
  for (int r = r_begin; r <= r_end; r += 6) {
    step(r, R0, R1, R2);
    step(r + 1, R1, R2, R0);
    step(r + 2, R2, R0, R1);
    step(r + 3, R0, R1, R2);
    step(r + 4, R1, R2, R0);
    step(r + 5, R2, R0, R1);
  }
  mn = warp_min(mn);
  if (lane == 0) atomicMin(&frame_min[f], float_to_ordered(mn));
}

__global__ void k_fill_u32(uint32_t* p, int n, uint32_t v) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

// -----------------------------------------------------------------------------------------
// K2: threshold.  mask bit = resp < 0.05 * min (detector.rs:418, :176-177).
//
// Vector version (width % 32 == 0): a thread loads 4 consecutive responses with one 16-byte
// streaming load, eight lanes cover one 32-pixel mask word, and the 4-bit nibbles are ORed
// together with three shuffles, so a warp produces four mask words per load instruction.
// Generic version: one pixel per lane, one ballot per word.
// -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
k_threshold_mask_v4(const float* __restrict__ resp, FrameGeom g, const uint32_t* __restrict__ frame_min,
                    uint32_t* __restrict__ mask) {
  const int f = blockIdx.y;
  const float thr = __fmul_rn(ordered_to_float(frame_min[f]), 0.05f);  // detector.rs:418
  const float4* R = reinterpret_cast<const float4*>(resp + (size_t)f * g.n_px);
  uint32_t* M = mask + (size_t)f * g.n_words;
  const int lane = threadIdx.x & 31;
  const int n_vec = g.n_px >> 2;  // rows are whole words, so the frame is a flat run of words
  const int stride = gridDim.x * blockDim.x;
  constexpr int U = 4;
  for (int v0 = blockIdx.x * blockDim.x + threadIdx.x; v0 < n_vec; v0 += stride * U) {
    float4 q[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int v = v0 + u * stride;
      q[u] = v < n_vec ? __ldcs(R + v) : make_float4(3.0e38f, 3.0e38f, 3.0e38f, 3.0e38f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int v = v0 + u * stride;
      uint32_t b = (q[u].x < thr ? 1u : 0u) | (q[u].y < thr ? 2u : 0u) | (q[u].z < thr ? 4u : 0u) |
                   (q[u].w < thr ? 8u : 0u);
      b <<= 4 * (lane & 7);
      b |= __shfl_xor_sync(0xffffffffu, b, 1);
      b |= __shfl_xor_sync(0xffffffffu, b, 2);
      b |= __shfl_xor_sync(0xffffffffu, b, 4);
      if ((lane & 7) == 0 && v < n_vec) M[v >> 3] = b;
    }
  }
}

__global__ void __launch_bounds__(256)
k_threshold_mask(const float* __restrict__ resp, FrameGeom g, const uint32_t* __restrict__ frame_min,
                 uint32_t* __restrict__ mask) {
  const int f = blockIdx.y;
  const float thr = __fmul_rn(ordered_to_float(frame_min[f]), 0.05f);  // detector.rs:418
  const float* R = resp + (size_t)f * g.n_px;
  uint32_t* M = mask + (size_t)f * g.n_words;
  const int lane = threadIdx.x & 31;
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  constexpr int U = 4;
  for (int wi0 = warp * U; wi0 < g.n_words; wi0 += n_warps * U) {
    float v[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      int wi = wi0 + u;
      v[u] = 3.40282347e+38f;
      if (wi < g.n_words) {
        int row = wi / g.wpr, wc = wi - row * g.wpr;
        int x = wc * 32 + lane;
        if (x < g.w) v[u] = __ldcs(R + (size_t)row * g.w + x);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      uint32_t b = __ballot_sync(0xffffffffu, v[u] < thr);
      if (lane == 0 && wi0 + u < g.n_words) M[wi0 + u] = b;
    }
  }
}

// ---------------------------------------------------------------------------------------
// Standalone operators mirroring the reference's public image_util functions (f32 -> f32).
// ---------------------------------------------------------------------------------------
// image_util::gaussian_blur_f32(img, sigma): general radius, taps passed from the host.
__global__ void __launch_bounds__(256)
k_blur_f32_h(const float* __restrict__ in, float* __restrict__ tmp, int w, int h,
             const float* __restrict__ taps, int radius) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= w || y >= h) return;
  const float* r = in + (size_t)y * w;
  float val = 0.0f;
  for (int i = 0; i <= 2 * radius; ++i) {
    int kx = min(max(x + i - radius, 0), w - 1);
    val = __fadd_rn(val, __fmul_rn(r[kx], taps[i]));
  }
  tmp[(size_t)y * w + x] = val;
}
__global__ void __launch_bounds__(256)
k_blur_f32_v(const float* __restrict__ tmp, float* __restrict__ out, int w, int h,
             const float* __restrict__ taps, int radius) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= w || y >= h) return;
  float val = 0.0f;
  for (int i = 0; i <= 2 * radius; ++i) {
    int ky = min(max(y + i - radius, 0), h - 1);
    val = __fadd_rn(val, __fmul_rn(tmp[(size_t)ky * w + x], taps[i]));
  }
  out[(size_t)y * w + x] = val;
}
// gaussian_blur_f32 for radius 3 (1 < sigma <= 1.5: the detector's own sigma and bench_blur.rs's),
// width % 4 == 0: the streaming structure of K1 without the gray conversion and the Hessian -- one
// warp per 120-column strip, 4 columns per lane (one 16-byte load per lane-row, prefetched three
// rows ahead), halo pixels by shuffle, six running partial sums per column, a loop of six
// unconditional row steps.  8 B/px of traffic (4 in + 4 out), no intermediate image.
// The accumulations start from 0.0 explicitly: 0.0 + (-0.0) is +0.0 (image_util.rs:138-203
// accumulates into a zero-initialised value), which matters for inputs that are not >= 0.
__global__ void __launch_bounds__(S_WARPS * 32, 6)
k_blur_f32_stream(const float* __restrict__ in, float* __restrict__ out, int w, int h, int chunk_rows,
                  float k0, float k1, float k2, float k3) {
  const int lane = threadIdx.x & 31;
  const int strip = blockIdx.x * S_WARPS + (threadIdx.x >> 5);
  const int X0 = strip * S_COLS;
  if (X0 >= w) return;
  const int f = blockIdx.z;
  const int Y0 = blockIdx.y * chunk_rows, Y1 = min(Y0 + chunk_rows, h);
  const int c0 = X0 - 4 + 4 * lane;
  const int cw = min(max(c0, 0), w - 4);
  const size_t n_px = (size_t)w * h;
  const char* src = reinterpret_cast<const char*>(in + (f * n_px + cw));
  char* dst = reinterpret_cast<char*>(out + f * n_px) + (ptrdiff_t)c0 * 4;
  asm volatile("" : "+l"(src));
  asm volatile("" : "+l"(dst));
  const uint32_t row_bytes = (uint32_t)w * 4u;
  const bool left_out = c0 < 0, right_out = c0 >= w;
  const bool edge_strip = X0 == 0 || X0 + S_COLS + 4 >= w;  // warp-uniform
  int writer = (lane >= 1 && lane <= 30 && !right_out) ? 1 : 0;
  asm volatile("" : "+r"(writer));
  const int h1 = h - 1;
  const uint32_t emit_span = (uint32_t)(Y1 - Y0);
  auto load_row = [&](int r) -> float4 {
    const uint32_t rr = (uint32_t)min(max(r, 0), h1);
    return __ldg(reinterpret_cast<const float4*>(src + (uint64_t)rr * row_bytes));
  };
  float a1[4], a2[4], a3[4], a4[4], a5[4], a6[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) a1[c] = a2[c] = a3[c] = a4[c] = a5[c] = a6[c] = 0.0f;
  const int r_begin = Y0 - 3, r_end = Y1 + 2;  // input rows of this chunk's output rows
  float4 w_cur = load_row(r_begin), w_n1 = load_row(r_begin + 1), w_n2 = load_row(r_begin + 2);
  // consumes input row r, completes output row r - 3
  auto step = [&](int r) {
    const float4 wd = w_cur;
    w_cur = w_n1;
    w_n1 = w_n2;
    w_n2 = load_row(r + 3);
    float p[10];
    p[3] = wd.x; p[4] = wd.y; p[5] = wd.z; p[6] = wd.w;
    if (edge_strip) {  // lanes hanging over the image edge replicate the edge pixel
      if (left_out) p[4] = p[5] = p[6] = p[3];
      if (right_out) p[3] = p[4] = p[5] = p[6];
    }
    p[0] = __shfl_up_sync(0xffffffffu, p[4], 1);
    p[1] = __shfl_up_sync(0xffffffffu, p[5], 1);
    p[2] = __shfl_up_sync(0xffffffffu, p[6], 1);
    p[7] = __shfl_down_sync(0xffffffffu, p[3], 1);
    p[8] = __shfl_down_sync(0xffffffffu, p[4], 1);
    p[9] = __shfl_down_sync(0xffffffffu, p[5], 1);
    float o[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      float t = __fadd_rn(0.0f, __fmul_rn(p[c], k0));
      t = __fadd_rn(t, __fmul_rn(p[c + 1], k1));
      t = __fadd_rn(t, __fmul_rn(p[c + 2], k2));
      t = __fadd_rn(t, __fmul_rn(p[c + 3], k3));
      t = __fadd_rn(t, __fmul_rn(p[c + 4], k2));
      t = __fadd_rn(t, __fmul_rn(p[c + 5], k1));
      t = __fadd_rn(t, __fmul_rn(p[c + 6], k0));
      const float q0 = __fmul_rn(t, k0), q1 = __fmul_rn(t, k1), q2 = __fmul_rn(t, k2),
                  q3 = __fmul_rn(t, k3);
      o[c] = __fadd_rn(a6[c], q0);
      a6[c] = __fadd_rn(a5[c], q1);
      a5[c] = __fadd_rn(a4[c], q2);
      a4[c] = __fadd_rn(a3[c], q3);
      a3[c] = __fadd_rn(a2[c], q2);
      a2[c] = __fadd_rn(a1[c], q1);
      a1[c] = __fadd_rn(0.0f, q0);
    }
    const int yo = r - 3;
    if ((uint32_t)(yo - Y0) < emit_span && writer)
      __stcs(reinterpret_cast<float4*>(dst + (uint64_t)(uint32_t)yo * row_bytes), make_float4(o[0], o[1], o[2], o[3]));
  };
  for (int r = r_begin; r <= r_end; r += 6) {  // chunk heights are multiples of six; steps past r_end emit nothing
    step(r);
    step(r + 1);
    step(r + 2);
    step(r + 3);
    step(r + 4);
    step(r + 5);
  }
}

// image_util::hessian_response(img)
__global__ void __launch_bounds__(256)
k_hessian_f32(const float* __restrict__ img, float* __restrict__ out, int w, int h) {
  int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
  if (x >= w || y >= h) return;
  float r = 0.0f;
  if (x >= 1 && x < w - 1 && y >= 1 && y < h - 1) {
    const float* p = img + (size_t)(y - 1) * w + x;
    const float* c = p + w;
    const float* n = c + w;
    float t2 = __fmul_rn(c[0], 2.0f);
    float lxx = __fadd_rn(__fsub_rn(c[-1], t2), c[1]);
    float lyy = __fadd_rn(__fsub_rn(p[0], t2), n[0]);
    float lxy = __fmul_rn(__fsub_rn(__fadd_rn(__fsub_rn(p[1], p[-1]), n[-1]), n[1]), 0.25f);
    r = __fsub_rn(__fmul_rn(lxx, lyy), __fmul_rn(lxy, lxy));
  }
  out[(size_t)y * w + x] = r;
}

// Exhaustive check helper for the unorm conversions (test only): out[v] for v in [0, n).
__global__ void k_unorm_table(float* out8, float* out16, float* ref8, float* ref16) {
  int v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < 256) {
    out8[v] = unorm8_to_f32((float)v);
    ref8[v] = __fdiv_rn((float)v, 255.0f);
  }
  if (v < 65536) {
    out16[v] = unorm16_to_f32((float)v);
    ref16[v] = __fdiv_rn((float)v, 65535.0f);
  }
}

// The float formats' gray conversion of n pixels (test only): what K1 and the board kernel compute.
__global__ void k_float_luma(const float* __restrict__ rgb, long long n, int channels, float* __restrict__ luma32f,
                             uint8_t* __restrict__ luma8) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = rgb + (size_t)channels * i;
  const float l = rgb32f_luma(p[0], p[1], p[2]);
  luma32f[i] = l;
  luma8[i] = (uint8_t)luma32f_to_u8(l);
}

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
template <int FMT>
static void launch_tile(const uint8_t* frames, const FrameGeom& g, int n_frames, float* blur,
                        float* resp, uint32_t* frame_min, bool write_blur, cudaStream_t s) {
  dim3 grid((g.w + T_W - 1) / T_W, (g.h + T_H - 1) / T_H, n_frames);
  if (write_blur)
    k_blur_hessian_tile<FMT, true><<<grid, 256, 0, s>>>(frames, g, blur, resp, frame_min);
  else
    k_blur_hessian_tile<FMT, false><<<grid, 256, 0, s>>>(frames, g, blur, resp, frame_min);
}

int launch_blur_hessian(const uint8_t* frames, const FrameGeom& g, int n_frames, float* blur,
                        float* resp, uint32_t* frame_min, bool write_blur, int variant,
                        int chunk_rows_opt, cudaStream_t s) {
  int launches = 0;
  k_fill_u32<<<(n_frames + 255) / 256, 256, 0, s>>>(frame_min, n_frames, kOrderedFltMax);
  ++launches;
  // alignment of a lane's loads: L8 and RGB8 load 32-bit words, L16, LA8 and RGB16 8-byte words,
  // the others 16-byte words
  const int bpp = bytes_per_px(g.format);
  const size_t al = bpp == 1 || bpp == 3 ? 4 : (bpp == 2 || bpp == 6 ? 8 : 16);
  const bool can_stream = (g.w % 4) == 0 && g.w >= 8 && (g.row_stride % al) == 0 && (g.frame_stride % al) == 0 &&
                          (((uintptr_t)frames | g.ptr_bits) % al) == 0 && variant != 1 &&
                          (uint64_t)g.row_stride * (uint64_t)g.h < (1ull << 32);  // 32-bit offsets within a frame
  if (can_stream) {
    const int strips = (g.w + S_COLS - 1) / S_COLS;
    const int bx = (strips + S_WARPS - 1) / S_WARPS;
    // the taller chunk when it still gives every SM a few waves of blocks
    int chunk_rows = kChunkRows[1];
    if (chunk_rows_opt > 0 && (chunk_rows_opt + 8) % 6 == 0) {
      chunk_rows = chunk_rows_opt;  // option "k1_chunk_rows" (tests, experiments)
    } else {
      for (int c : kChunkRows) {
        const long blocks = (long)bx * ((g.h + c - 1) / c) * n_frames;
        if (blocks >= 148L * 7 * 4) { chunk_rows = c; break; }
      }
    }
    dim3 grid(bx, (g.h + chunk_rows - 1) / chunk_rows, n_frames);
    const dim3 block(S_WARPS * 32);
#define AG_STREAM(FMT)                                                                                          \
    if (write_blur) k_blur_hessian_stream<FMT, true><<<grid, block, 0, s>>>(frames, g, chunk_rows, blur, resp, frame_min); \
    else k_blur_hessian_stream<FMT, false><<<grid, block, 0, s>>>(frames, g, chunk_rows, blur, resp, frame_min)
    switch (g.format) {
      case AG_L8: AG_STREAM(AG_L8); break;
      case AG_L16: AG_STREAM(AG_L16); break;
      case kFmtF32: AG_STREAM(kFmtF32); break;
      case AG_LA8: AG_STREAM(AG_LA8); break;
      case AG_RGBA8: AG_STREAM(AG_RGBA8); break;
      case AG_LA16: AG_STREAM(AG_LA16); break;
      case AG_RGB16: AG_STREAM(AG_RGB16); break;
      case AG_RGBA16: AG_STREAM(AG_RGBA16); break;
      case AG_RGB32F: AG_STREAM(AG_RGB32F); break;
      case AG_RGBA32F: AG_STREAM(AG_RGBA32F); break;
      default: AG_STREAM(AG_RGB8); break;
    }
#undef AG_STREAM
    return launches + 1;
  }
  switch (g.format) {
    case AG_L8: launch_tile<AG_L8>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_L16: launch_tile<AG_L16>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case kFmtF32: launch_tile<kFmtF32>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_LA8: launch_tile<AG_LA8>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_RGBA8: launch_tile<AG_RGBA8>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_LA16: launch_tile<AG_LA16>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_RGB16: launch_tile<AG_RGB16>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_RGBA16: launch_tile<AG_RGBA16>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_RGB32F: launch_tile<AG_RGB32F>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    case AG_RGBA32F: launch_tile<AG_RGBA32F>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
    default: launch_tile<AG_RGB8>(frames, g, n_frames, blur, resp, frame_min, write_blur, s); break;
  }
  return launches + 1;
}

int launch_threshold(const float* resp, const FrameGeom& g, int n_frames, const uint32_t* frame_min,
                     uint32_t* mask, cudaStream_t s) {
  if ((g.w & 31) == 0 && (((uintptr_t)resp) & 15) == 0) {
    // whole-word rows: flat float4 version; 296 blocks per frame-row of the grid keep all SMs busy
    const int n_vec = g.n_px >> 2;
    int bx = (n_vec + 256 * 4 - 1) / (256 * 4);
    if (bx > 64) bx = 64;
    dim3 grid(bx, n_frames);
    k_threshold_mask_v4<<<grid, 256, 0, s>>>(resp, g, frame_min, mask);
    return 1;
  }
  int blocks_x = (g.n_words + 8 * 4 - 1) / (8 * 4);  // 8 warps x 4 words per block iteration
  if (blocks_x > 4096) blocks_x = 4096;
  if (blocks_x < 1) blocks_x = 1;
  dim3 grid(blocks_x, n_frames);
  k_threshold_mask<<<grid, 256, 0, s>>>(resp, g, frame_min, mask);
  return 1;
}

// n_frames contiguous f32 images; `taps` are the 2 * radius + 1 host-side taps, `d_taps` their device
// copy, `tmp` one image of scratch (only the general path uses the last two).
int launch_blur_f32(const float* in, float* tmp, float* out, int w, int h, int n_frames, const float* taps,
                    const float* d_taps, int radius, cudaStream_t s) {
  const bool can_stream = radius == 3 && (w % 4) == 0 && w >= 8 && ((uintptr_t)in % 16) == 0 &&
                          ((uintptr_t)out % 16) == 0 && (uint64_t)w * 4u * (uint64_t)h < (1ull << 32);
  if (can_stream) {
    const int strips = (w + S_COLS - 1) / S_COLS;
    const int bx = (strips + S_WARPS - 1) / S_WARPS;
    int chunk_rows = 60;
    if ((long)bx * ((h + 125) / 126) * n_frames >= 148L * 6 * 4) chunk_rows = 126;
    dim3 grid(bx, (h + chunk_rows - 1) / chunk_rows, n_frames);
    k_blur_f32_stream<<<grid, S_WARPS * 32, 0, s>>>(in, out, w, h, chunk_rows, taps[0], taps[1], taps[2], taps[3]);
    return 1;
  }
  dim3 grid((w + 255) / 256, h);
  for (int f = 0; f < n_frames; ++f) {
    const size_t o = (size_t)f * w * h;
    k_blur_f32_h<<<grid, 256, 0, s>>>(in + o, tmp, w, h, d_taps, radius);
    k_blur_f32_v<<<grid, 256, 0, s>>>(tmp, out + o, w, h, d_taps, radius);
  }
  return 2 * n_frames;
}
int launch_hessian_f32(const float* in, float* out, int w, int h, cudaStream_t s) {
  dim3 grid((w + 255) / 256, h);
  k_hessian_f32<<<grid, 256, 0, s>>>(in, out, w, h);
  return 1;
}
int launch_unorm_table(float* out8, float* out16, float* ref8, float* ref16, cudaStream_t s) {
  k_unorm_table<<<256, 256, 0, s>>>(out8, out16, ref8, ref16);
  return 1;
}
int launch_float_luma(const float* rgb, long long n, int channels, float* luma32f, uint8_t* luma8, cudaStream_t s) {
  k_float_luma<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(rgb, n, channels, luma32f, luma8);
  return 1;
}

}  // namespace ag
