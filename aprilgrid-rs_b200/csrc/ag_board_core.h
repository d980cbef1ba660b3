// Board assembly and tag decoding for ONE frame, written once for two compilation modes:
//
//   * device (nvcc, __CUDA_ARCH__): one thread block of a few warps per frame.  Inside a warp
//     all 32 lanes run the same control flow on the same data ("warp-uniform"); the lanes
//     split the data-parallel inner loops (neighbour searches, candidate-quad tests, bit
//     sampling, Hamming search) and lane 0 performs the stores.  The warps of a block work on
//     different seed saddles of try_find_best_board at the same time (speculatively: seeds are
//     independent until their results are merged in the reference's order).
//   * host (tests/host_board_test.cpp): the same source with a warp of one lane, so the
//     control logic can be unit-tested against the oracle in a container without a GPU.
//     That build is test-only; the shipped library has no CPU path.
//
// Reference: src/detector.rs:42-169 (decode), :448-476, :505-639; src/board.rs:26-235;
// src/saddle.rs:17-67; src/math_util.rs:15-33.
//
// Where the reference iterates a std HashMap (random order per process) this code uses a
// fixed order, the same one as the oracle:
//   * most populated round(theta) bin: ties -> the largest angle      (detector.rs:610-616)
//   * quads of a board are visited in ascending (x, y) lattice order  (board.rs:49-51)
#pragma once
#include <math.h>
#include <stdint.h>

#include "ag_float_luma.h"
#include "ag_libm.h"

#if defined(__CUDA_ARCH__)
#define AGB_DEVICE 1
#else
#define AGB_DEVICE 0
#endif

#if !defined(__CUDACC__)
struct float2 { float x, y; };  // host test build: the CUDA vector type is not available
#endif

#if defined(__CUDA_ARCH__)
#define AGB_UNROLL _Pragma("unroll")
#else
#define AGB_UNROLL
#endif

#if defined(__CUDACC__)
#define AGB_FN __host__ __device__ inline
#define AGB_NOINLINE __host__ __device__ __noinline__
#else
#define AGB_FN inline
#define AGB_NOINLINE __attribute__((noinline))
#endif

// Optional work counters for the host build (tools/board_work_counts.py); no-ops otherwise.
#if defined(AGB_WORK_COUNTERS) && !defined(__CUDA_ARCH__)
extern "C" long long agb_work_counters[32];
extern "C" void agb_note_query(int a, int b, int self_is_b, float qx, float qy, float r2);
extern "C" void agb_note_query(int a, int b, int self_is_b, float qx, float qy, float r2);
#define AGB_COUNT(slot, n) (agb_work_counters[(slot) + 12 * agb_work_counters[31]] += (n))
#else
#define AGB_COUNT(slot, n) ((void)0)
#endif

namespace agb {

constexpr int kMaxLattice = 64;  // lattice of tag positions: at most 64 x 64 (-32..31 per axis)
constexpr int kCells = kMaxLattice * kMaxLattice;
constexpr int kHistBins = 192;  // round(theta) + 90 in [0, 180]
constexpr int kMaxCodes = 640;  // >= 587
constexpr float kPi = 3.14159274101257324f;
constexpr int kNone = 0x7fffffff;

struct TagRec {  // == ag_tag
  uint32_t id;
  float xy[8];
};

// The board under construction (board.rs:18-25).  The lattice and the active mask are the
// randomly accessed structures (shared memory on the device); the counters are warp-uniform
// registers.
struct BoardState {
  int16_t* cell;     // [kCells] 0 = never visited, -1 = None, q+1 = Some(quad q)
  uint32_t* active;  // [max_saddles / 32] bit i = active_idxs[i]
  int16_t* quads;    // [max_quads][4] saddle indices
  int16_t* touched;  // [kCells] indices of non-zero cells (cheap reset)
  int n_quads, n_touched, score;
};
// Copy of the best board so far (what `best_board_option` holds in detector.rs:599-626).
struct BoardRecord {
  int16_t* quads;    // [max_quads][4]
  int16_t* touched;  // [kCells] cell indices
  int16_t* vals;     // [kCells] cell values
  int n_quads, n_touched, score;
};

struct Frame {
  int n;                 // saddles in the current round
  float *sx, *sy, *st;   // saddles (SoA): position, theta
  BoardState bs;        // this warp's live board
  BoardRecord seedbest; // this warp's best board of the seed it is processing
  BoardRecord best;     // the frame's best board so far (arrays shared by the block)
  int lat, lat_off;     // lattice side (power of two <= kMaxLattice) and its centre offset
  int warp, n_warps;    // warp index inside the frame's block (0 / 1 on the host)
  int* w_score;         // [n_warps] shared: per-warp result of the current wave of seeds
  int* ctl;             // [8] shared: 0 n_seeds, 1 n after compaction, 2..4 best n_quads/n_touched/score
  // uniform bucket grid over the saddles of the current round (null = brute-force search)
  uint16_t* g_start;  // [g_nx * g_ny + 1] first entry of each bucket in g_item
  uint16_t* g_item;   // [n] saddle indices sorted by bucket
  int g_nx, g_ny, g_cap_cells, g_cap_items;
  int g_on;           // 1 = the grid holds the current round's saddles (block-uniform)
  float g_inv;        // 1 / bucket size in pixels
  int16_t* stack;   // [2 * (max_quads + 1)] DFS stack: cell index, next direction
  int16_t* seeds;   // [max_saddles]
  int16_t* nn_idx;  // [64] 50-NN result
  int16_t* same;    // [64]
  int16_t* diff;    // [64]
  int16_t* samp;    // [64] sampled brightness (-1 = outside the image)
  int* hist;        // [kHistBins]
  uint8_t* remove;  // [max_saddles]
  int max_quads;
  // image for bit sampling (original pixels; converted to luma8 on the fly)
  const uint8_t* img;
  int w, h, format;
  size_t row_stride;
  // family
  const uint64_t* codes;
  int n_codes, edge, border, hamming;
  // results
  uint8_t* tag_valid;  // [kMaxCodes]
  TagRec* tag_by_id;   // [kMaxCodes]
  // optional tap: quads of the first board found, in visiting order
  int32_t* tap_quads;
  int* tap_n_quads;
  int tap_cap;
  uint32_t status;
  int lane;  // 0 on host
  // throughput path (device only, ag_board_fast.cuh); unused when fast_on == 0
  int fast_on;
  int round;             // board round being searched (0 = first board)
  uint16_t* g_base;      // unshifted bucket-grid array ([cells + 2])
  float2* g_pos;         // [n] saddle positions in g_item order (one load per scanned candidate)
  int active_words;      // words of bs.active
  int16_t* fx_qlist;     // [kQListCap][4] candidate quads of the current seed
  uint16_t* fx_qscore;   // [kQListCap]
  float *fx_dvx, *fx_dvy;  // [52] per `diff` entry: vector from the seed
  unsigned long long* fx_tmask;  // [52] per `diff` entry i: partners j > i passing the theta gate
  uint32_t* fx_squeue;   // [64] ring of pairs that passed the cheap gates
  uint8_t* fx_gstate;    // this warp's group states (aliases bs.cell)
  uint16_t* fx_wscore;   // [32] per wave slot: best score of the seed so far
  int16_t* fx_wquad;     // [32][4] ... and its quad
  uint8_t* fx_save0;     // global: warp 0's saved best board (header + group state); warp w's at
  size_t fx_save_stride; //   fx_save0 + w * fx_save_stride
  unsigned long long* fx_qcache;  // global: the frame's neighbour-search cache (kQCacheEntries entries)
  uint32_t* tm;          // optional per-frame timing / work counters ([16], may be null)
  int16_t* dec_qlist;    // decoding: the found board's quads in visiting order (warp 0's seed-best quads)
  unsigned long long* dec_qbits;  // ... and their bit patterns / decoded (id, rotation)
};

// ---- warp plumbing ---------------------------------------------------------------------
#if AGB_DEVICE
#define AGB_SYNC() __syncwarp()
#define AGB_BLOCK_SYNC() __syncthreads()
#define AGB_LANES 32
AGB_FN unsigned agb_ballot(bool p) { return __ballot_sync(0xffffffffu, p); }
#else
#define AGB_SYNC() ((void)0)
#define AGB_BLOCK_SYNC() ((void)0)
#define AGB_LANES 1
AGB_FN unsigned agb_ballot(bool p) { return p ? 1u : 0u; }
#endif
AGB_FN int agb_ffs(unsigned m) {  // index of lowest set bit, m != 0
#if AGB_DEVICE
  return __ffs((int)m) - 1;
#else
  return __builtin_ctz(m);
#endif
}
AGB_FN int agb_popcll(uint64_t v) {
#if AGB_DEVICE
  return __popcll(v);
#else
  return __builtin_popcountll(v);
#endif
}

// ---- exact f32 arithmetic (no contraction in either build) --------------------------------
#if AGB_DEVICE
AGB_FN float fmul(float a, float b) { return __fmul_rn(a, b); }
AGB_FN float fadd(float a, float b) { return __fadd_rn(a, b); }
AGB_FN float fsub(float a, float b) { return __fsub_rn(a, b); }
AGB_FN float fdiv(float a, float b) { return __fdiv_rn(a, b); }
#else
AGB_FN float fmul(float a, float b) { volatile float r = a * b; return r; }
AGB_FN float fadd(float a, float b) { volatile float r = a + b; return r; }
AGB_FN float fsub(float a, float b) { volatile float r = a - b; return r; }
AGB_FN float fdiv(float a, float b) { volatile float r = a / b; return r; }
#endif
// atan2f: glibc's routine restated operation for operation (ag_libm.h: the oracle's bits).
// cosf / sinf: evaluated in f64 and rounded once (glibc's are within an ulp of that; see DESIGN.md).
AGB_FN float atan2_cr(float y, float x) { return lm_atan2f(y, x); }
AGB_FN float cos_cr(float x) { return (float)cos((double)x); }
AGB_FN float sin_cr(float x) { return (float)sin((double)x); }

AGB_FN uint32_t sat_u32(float v) {  // Rust `as u32`
  if (!(v > 0.0f)) return 0u;
  if (v >= 4294967296.0f) return 0xffffffffu;
  return (uint32_t)v;
}
AGB_FN int sat_i32(float v) {  // Rust `as i32`
  if (v != v) return 0;
  if (v >= 2147483648.0f) return 2147483647;
  if (v <= -2147483648.0f) return (int)0x80000000;
  return (int)v;
}

// ---- math_util.rs:15-33 ------------------------------------------------------------------
AGB_FN float theta_distance_degree(float t0, float t1) {
  float d = fadd(fsub(t0, t1), 90.0f);
  if (d < 0.0f) d = fadd(d, 180.0f);
  else if (d > 180.0f) d = fsub(d, 180.0f);
  return d > 90.0f ? fsub(d, 90.0f) : fsub(90.0f, d);
}
AGB_FN float cross2(float ax, float ay, float bx, float by) { return fsub(fmul(ax, by), fmul(ay, bx)); }
AGB_FN float dot2(float ax, float ay, float bx, float by) { return fadd(fmul(ax, bx), fmul(ay, by)); }
AGB_FN float angle_degree(float ax, float ay, float bx, float by) {
  float y = fsub(fmul(by, ax), fmul(bx, ay));
  float x = fadd(fmul(ax, bx), fmul(ay, by));
  return fdiv(fmul(atan2_cr(y, x), 180.0f), kPi);
}

// Cheap f32 evaluation of the same angle (same exact y, x operands; atan2f instead of the f64
// route).  Its error is below 1e-4 degree, so a comparison against a threshold is decided by it
// with certainty unless the value lies within kGuardDeg of the threshold; only then is the
// exact expression evaluated.  The verdicts are therefore identical to the exact path.
constexpr float kGuardDeg = 4.0e-3f;
AGB_FN float angle_degree_fast(float ax, float ay, float bx, float by) {
  float y = fsub(fmul(by, ax), fmul(bx, ay));
  float x = fadd(fmul(ax, bx), fmul(ay, by));
  return atan2f(y, x) * 57.2957795f;
}
// Margin, in the units of a quantity m = A - B (both ~ a product of two vector lengths), that
// covers kGuardDeg of angle plus f32 rounding of the products: |dm / d angle| <= 1.02 * scale
// per radian for the tests below, kGuardDeg = 7e-5 rad.
constexpr float kGuardRel = 1.2e-4f;
// |angle(a) - angle(b)| > limit ?  with a = angle(p, q), b = angle(r, s): the atan2f path with
// its guard band, then the exact expression (rarely reached: see angle_gap_exceeds).
AGB_NOINLINE bool angle_gap_exceeds_slow(float px, float py, float qx, float qy, float rx, float ry,
                                         float sx, float sy, float limit) {
  const float fa = angle_degree_fast(px, py, qx, qy), fb = angle_degree_fast(rx, ry, sx, sy);
  const float g = fabsf(fa - fb);
  if (g > limit + kGuardDeg) return true;
  if (g < limit - kGuardDeg) return false;
  return fabsf(fsub(angle_degree(px, py, qx, qy), angle_degree(rx, ry, sx, sy))) > limit;
}
// |angle(a) - angle(b)| > limit ?  limit = 10 degrees.  Inline part: the trigonometry-free
// decision.  a = atan2(y1, x1), b = atan2(y2, x2).  When y1 and y2 have the same strict sign both
// angles lie in the same open half turn, so a - b = atan2(Y, X) with Y = y1 x2 - x1 y2,
// X = x1 x2 + y1 y2, and |a - b| <= limit  <=>  |Y| <= tan(limit) X.  Away from the threshold
// (margin: guard band + rounding) the verdict is certain; otherwise the slow path decides.
AGB_FN bool angle_gap_exceeds(float px, float py, float qx, float qy, float rx, float ry, float sx,
                              float sy, float limit) {
  const float y1 = py * qx - px * qy, x1 = px * qx + py * qy;  // atan2 arguments of angle_degree(p, q)
  const float y2 = ry * sx - rx * sy, x2 = rx * sx + ry * sy;
  if ((y1 > 0.0f && y2 > 0.0f) || (y1 < 0.0f && y2 < 0.0f)) {
    const float a1 = y1 * x2, a2 = x1 * y2, b1 = x1 * x2, b2 = y1 * y2;
    const float Y = a1 - a2, X = b1 + b2;
    const float kTan10 = 0.17632698f;
    const float m = fabsf(Y) - kTan10 * X;
    const float scale = fabsf(a1) + fabsf(a2) + fabsf(b1) + fabsf(b2);
    const float margin = (kGuardRel + 4.0e-7f) * scale;
    if (limit == 10.0f && scale < 1.0e30f && scale > 1.0e-30f) {
      if (m > margin) return true;
      if (m < -margin) return false;
    }
  }
  return angle_gap_exceeds_slow(px, py, qx, qy, rx, ry, sx, sy, limit);
}

// ---- saddle.rs:17-67, split in two so the (s0, s1)-only test can be hoisted ---------------
// Coordinate forms (inline; the throughput path loads the points once and passes them in
// registers) and index forms (noinline wrappers for the general path).
AGB_NOINLINE bool quad_diag_ok_slow(float v02x, float v02y, float th) {
  {
    const float fa = fabsf(angle_degree_fast(v02x, v02y, cosf(th), sinf(th)));
    if (fa > 60.0f + kGuardDeg && fa < 120.0f - kGuardDeg) return true;
    if (fa < 60.0f - kGuardDeg || fa > 120.0f + kGuardDeg) return false;
  }
  float vx = cos_cr(th), vy = sin_cr(th);
  float a = fabsf(angle_degree(v02x, v02y, vx, vy));
  return a >= 60.0f && a <= 120.0f;
}
AGB_FN bool quad_diag_ok_v(float x0, float y0, float t0, float x1, float y1) {  // "filter white block", :26-38
  float v02x = fsub(x1, x0), v02y = fsub(y1, y0);
  float th = fmul(fdiv(t0, 180.0f), kPi);
  {
    // |angle(v02, u)| in [60, 120] degrees  <=>  sqrt(3) |dot| <= |cross|  (u = unit vector of
    // theta); decided without atan2 away from the two thresholds.
#if AGB_DEVICE
    const float ux = __cosf(th), uy = __sinf(th);  // |th| <= pi: absolute error ~ 1e-6
#else
    const float ux = cosf(th), uy = sinf(th);
#endif
    const float a1 = uy * v02x, a2 = ux * v02y, b1 = v02x * ux, b2 = v02y * uy;
    const float cr = a1 - a2, dt = b1 + b2;
    const float m = 1.7320508f * fabsf(dt) - fabsf(cr);
    const float scale = fabsf(a1) + fabsf(a2) + fabsf(b1) + fabsf(b2);
    const float margin = (2.0f * kGuardRel + 4.0e-6f) * scale;
    if (scale < 1.0e30f && scale > 1.0e-30f && fabsf(th) <= 3.2f) {
      if (m < -margin) return true;
      if (m > margin) return false;
    }
  }
  return quad_diag_ok_slow(v02x, v02y, th);
}
// The remaining gates of is_valid_quad.  They only ever reject, so they are evaluated
// cheapest-first; the verdict equals the reference's (saddle.rs:18-66).
// Points: s0 = (x0, y0), d0 = (xa, ya, theta ta), s1 = (x1, y1), d1 = (xb, yb, theta tb).
AGB_FN bool quad_rest_ok_v(float x0, float y0, float xa, float ya, float ta, float x1, float y1, float xb,
                           float yb, float tb) {
  if (theta_distance_degree(ta, tb) > 5.0f) return false;
  float v01x = fsub(xa, x0), v01y = fsub(ya, y0);
  float v03x = fsub(xb, x0), v03y = fsub(yb, y0);
  float v02x = fsub(x1, x0), v02y = fsub(y1, y0);
  float c0 = cross2(v01x, v01y, v02x, v02y);
  float c1 = cross2(v02x, v02y, v03x, v03y);
  if (fmul(c0, c1) < 0.0f) return false;
  float v12x = fsub(x1, xa), v12y = fsub(y1, ya);
  float v23x = fsub(xb, x1), v23y = fsub(yb, y1);
  float c01 = cross2(v01x, v01y, v12x, v12y);
  float c12 = cross2(v12x, v12y, v23x, v23y);
  if (fmul(c01, c12) < 0.0f) return false;
  if (dot2(v01x, v01y, v02x, v02y) < 0.0f || dot2(v03x, v03y, v02x, v02y) < 0.0f) return false;
  float v30x = fsub(x0, xb), v30y = fsub(y0, yb);
  if (angle_gap_exceeds(v01x, v01y, v12x, v12y, v23x, v23y, v30x, v30y, 10.0f)) return false;  // a0, a2
  if (angle_gap_exceeds(v12x, v12y, v23x, v23y, v30x, v30y, v01x, v01y, 10.0f)) return false;  // a1, a3
  return true;
}
AGB_NOINLINE bool quad_diag_ok(const Frame& F, int s0, int s1) {
  return quad_diag_ok_v(F.sx[s0], F.sy[s0], F.st[s0], F.sx[s1], F.sy[s1]);
}
AGB_NOINLINE bool quad_rest_ok(const Frame& F, int s0, int d0, int s1, int d1) {
  return quad_rest_ok_v(F.sx[s0], F.sy[s0], F.sx[d0], F.sy[d0], F.st[d0], F.sx[s1], F.sy[s1], F.sx[d1],
                        F.sy[d1], F.st[d1]);
}
AGB_FN bool is_valid_quad(const Frame& F, int s0, int d0, int s1, int d1) {
  // Both halves only ever return false early, so evaluating the diagonal test first gives
  // the same verdict as the reference's order (saddle.rs:18-38).
  return quad_diag_ok(F, s0, s1) && quad_rest_ok(F, s0, d0, s1, d1);
}
// ---- nearest neighbours (kdtree 0.8 `nearest`, restated as exact search) -------------------
// squared_euclidean: (0 + dx*dx) + dy*dy
AGB_FN float dist2(const Frame& F, float qx, float qy, int i) {
  float dx = fsub(qx, F.sx[i]), dy = fsub(qy, F.sy[i]);
  return fadd(fmul(dx, dx), fmul(dy, dy));
}
// strict (d2, idx) lexicographic order; ties in distance resolve to the lower index
AGB_FN bool nn_less(float da, int ia, float db, int ib) { return da < db || (da == db && ia < ib); }

#if AGB_DEVICE
AGB_FN void warp_argmin(float& d, int& i) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    float od = __shfl_xor_sync(0xffffffffu, d, o);
    int oi = __shfl_xor_sync(0xffffffffu, i, o);
    if (nn_less(od, oi, d, i)) { d = od; i = oi; }
  }
}
#else
AGB_FN void warp_argmin(float&, int&) {}
#endif

// Bucket grid: saddles counting-sorted by (floor(y * inv), floor(x * inv)).  A radius query
// then only visits the buckets overlapping the query square, which still contains every point
// within the radius, so results are identical to the exhaustive search.
AGB_FN int grid_bucket(const Frame& F, float x, float y) {
  int bx = (int)(x * F.g_inv), by = (int)(y * F.g_inv);
  bx = bx < 0 ? 0 : (bx >= F.g_nx ? F.g_nx - 1 : bx);
  by = by < 0 ? 0 : (by >= F.g_ny ? F.g_ny - 1 : by);
  return by * F.g_nx + bx;
}
#if AGB_DEVICE
// The grid built by the whole warp.  Layout: G[0] = 0, G[b + 1] = first entry of bucket b,
// G[nc + 1] = n, with G = F.g_base; F.g_start = G + 1 afterwards (every warp of the block sets it
// when it learns that the grid is on).  Order inside a bucket is arbitrary: every query selects by
// the total order (d2, index).  with_pos: also the grid-ordered positions of the throughput path.
__device__ __forceinline__ void grid_build_parallel(Frame& F, bool with_pos) {
  F.g_on = 0;
  if (!F.g_base) return;
  const int nc = F.g_nx * F.g_ny;
  if (F.n > F.g_cap_items || nc > F.g_cap_cells || F.n > 65535) return;
  F.g_on = 1;
  uint16_t* G = F.g_base;
  for (int c = F.lane; c <= nc + 1; c += 32) G[c] = 0;
  __syncwarp();
  // counts into G[b + 1]
  for (int base = 0; base < F.n; base += 32) {
    const int i = base + F.lane;
    const int b = i < F.n ? grid_bucket(F, F.sx[i], F.sy[i]) : (0x10000 + F.lane);
    const unsigned peers = __match_any_sync(0xffffffffu, b);
    if (i < F.n && (__ffs((int)peers) - 1) == F.lane) G[b + 1] = (uint16_t)(G[b + 1] + __popc(peers));
    __syncwarp();
  }
  // inclusive scan of G[1 .. nc]: afterwards G[b + 1] = end of bucket b
  {
    const int per = (nc + 31) / 32;
    const int c0 = 1 + F.lane * per, c1 = min(c0 + per, nc + 1);
    unsigned sum = 0;
    for (int c = c0; c < c1; ++c) sum += G[c];
    unsigned incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
      if (F.lane >= o) incl += v;
    }
    unsigned run = incl - sum;
    for (int c = c0; c < c1; ++c) {
      run += G[c];
      G[c] = (uint16_t)run;
    }
  }
  __syncwarp();
  // fill from the back of every bucket: G[b + 1] walks down from end(b) to start(b)
  for (int base = 0; base < F.n; base += 32) {
    const int i = base + F.lane;
    const int b = i < F.n ? grid_bucket(F, F.sx[i], F.sy[i]) : (0x10000 + F.lane);
    const unsigned peers = __match_any_sync(0xffffffffu, b);
    if (i < F.n) {
      const int rank = __popc(peers & ((1u << F.lane) - 1u));
      const int e = G[b + 1];
      F.g_item[e - 1 - rank] = (uint16_t)i;
      if (with_pos) F.g_pos[e - 1 - rank] = make_float2(F.sx[i], F.sy[i]);
    }
    __syncwarp();
    if (i < F.n && (__ffs((int)peers) - 1) == F.lane) G[b + 1] = (uint16_t)(G[b + 1] - __popc(peers));
    __syncwarp();
  }
  if (F.lane == 0) G[nc + 1] = (uint16_t)F.n;
  F.g_start = G + 1;
  __syncwarp();
}
#endif
AGB_NOINLINE void grid_build(Frame& F) {
#if AGB_DEVICE
  grid_build_parallel(F, false);  // the general path does not use the grid-ordered positions
  return;
#endif
  F.g_on = 0;
  if (!F.g_start) return;
  const int nc = F.g_nx * F.g_ny;
  // too large for the on-chip grid: queries fall back to the exhaustive scan
  if (F.n > F.g_cap_items || nc > F.g_cap_cells || F.n > 65535) return;
  F.g_on = 1;
  for (int c = F.lane; c <= nc; c += AGB_LANES) F.g_start[c] = 0;
  AGB_SYNC();
  // histogram into g_start[bucket + 1]
  if (F.lane == 0)
    for (int i = 0; i < F.n; ++i) F.g_start[grid_bucket(F, F.sx[i], F.sy[i]) + 1] += 1;
  AGB_SYNC();
  // inclusive scan (lane 0; a few thousand adds at most, once per round)
  if (F.lane == 0) {
    unsigned run = 0;
    for (int c = 1; c <= nc; ++c) {
      run += F.g_start[c];
      F.g_start[c] = (uint16_t)run;
    }
    // fill from the back so that every bucket ends up in ascending saddle order
    for (int i = F.n - 1; i >= 0; --i) {
      const int b = grid_bucket(F, F.sx[i], F.sy[i]);
      // entries of bucket b occupy [start[b], start[b+1]); use start[b+1] as a moving cursor
      F.g_item[--F.g_start[b + 1]] = (uint16_t)i;
    }
    // the cursors now equal the bucket starts shifted by one slot: g_start[b + 1] == start of b
    // restore the canonical layout g_start[b] = start of b
    for (int c = 0; c < nc; ++c) F.g_start[c] = F.g_start[c + 1];
    F.g_start[nc] = (uint16_t)F.n;
  }
  AGB_SYNC();
}

// The (up to) 3 nearest saddles with d2 <= r2, ascending.  Equals "3 nearest overall, then
// drop those outside the radius" (board.rs:192-200): points inside the radius always precede
// points outside it in the distance order.
AGB_NOINLINE int nearest3_within(const Frame& F, float qx, float qy, float r2, int out[3]) {
  float bd[3] = {3.0e38f, 3.0e38f, 3.0e38f};
  int bi[3] = {kNone, kNone, kNone};
  auto consider = [&](int i) {
    float d = dist2(F, qx, qy, i);
    if (d <= r2 && nn_less(d, i, bd[2], bi[2])) {
      bd[2] = d; bi[2] = i;
      if (nn_less(bd[2], bi[2], bd[1], bi[1])) {
        float t = bd[1]; bd[1] = bd[2]; bd[2] = t;
        int u = bi[1]; bi[1] = bi[2]; bi[2] = u;
      }
      if (nn_less(bd[1], bi[1], bd[0], bi[0])) {
        float t = bd[0]; bd[0] = bd[1]; bd[1] = t;
        int u = bi[0]; bi[0] = bi[1]; bi[1] = u;
      }
    }
  };
  if (F.g_on && r2 >= 0.0f && r2 < 1.0e12f) {
    // conservative square around the query: r slightly enlarged, bucket range clamped
    const float r = sqrtf(r2) * 1.0001f + 0.01f;
    int x0 = (int)floorf((qx - r) * F.g_inv), x1 = (int)floorf((qx + r) * F.g_inv);
    int y0 = (int)floorf((qy - r) * F.g_inv), y1 = (int)floorf((qy + r) * F.g_inv);
    // both ends clamped INTO the grid: saddles outside the image sit in the border buckets
    // (grid_bucket clamps too), so a window hanging over the edge must still reach those
    x0 = x0 < 0 ? 0 : (x0 >= F.g_nx ? F.g_nx - 1 : x0); y0 = y0 < 0 ? 0 : (y0 >= F.g_ny ? F.g_ny - 1 : y0);
    x1 = x1 >= F.g_nx ? F.g_nx - 1 : (x1 < 0 ? 0 : x1); y1 = y1 >= F.g_ny ? F.g_ny - 1 : (y1 < 0 ? 0 : y1);
    const int bw = x1 - x0 + 1, bh = y1 - y0 + 1;
    if (bw > 0 && bh > 0) {
      // rows of buckets are contiguous in g_item: one (start, end) range per bucket row
      for (int row = F.lane; row < bh; row += AGB_LANES) {
        const int b0 = (y0 + row) * F.g_nx + x0;
        const int e0 = F.g_start[b0], e1 = F.g_start[b0 + bw];
        for (int e = e0; e < e1; ++e) consider(F.g_item[e]);
      }
    }
  } else {
    for (int i = F.lane; i < F.n; i += AGB_LANES) consider(i);
  }
  int cnt = 0;
  // merge the per-lane sorted triples: three rounds of warp arg-min over the lanes' heads
  for (int r = 0; r < 3; ++r) {
    float d = bd[0];
    int i = bi[0];
#if AGB_DEVICE
    if (__ballot_sync(0xffffffffu, i != kNone) == 0u) break;
#endif
    warp_argmin(d, i);
    if (i == kNone) break;  // warp-uniform
    out[cnt++] = i;
    if (bi[0] == i) {
      bd[0] = bd[1]; bi[0] = bi[1];
      bd[1] = bd[2]; bi[1] = bi[2];
      bd[2] = 3.0e38f; bi[2] = kNone;
    }
  }
  return cnt;
}

// Same query evaluated by ONE lane without warp collectives (four of them run side by side in
// try_expand_one).  Returns the count; out[] ascending by (d2, idx).
AGB_FN int nearest3_within_single(const Frame& F, float qx, float qy, float r2, int out[3]) {
  float bd[3] = {3.0e38f, 3.0e38f, 3.0e38f};
  int bi[3] = {kNone, kNone, kNone};
  auto consider = [&](int i) {
    float d = dist2(F, qx, qy, i);
    if (d <= r2 && nn_less(d, i, bd[2], bi[2])) {
      bd[2] = d; bi[2] = i;
      if (nn_less(bd[2], bi[2], bd[1], bi[1])) {
        float t = bd[1]; bd[1] = bd[2]; bd[2] = t;
        int u = bi[1]; bi[1] = bi[2]; bi[2] = u;
      }
      if (nn_less(bd[1], bi[1], bd[0], bi[0])) {
        float t = bd[0]; bd[0] = bd[1]; bd[1] = t;
        int u = bi[0]; bi[0] = bi[1]; bi[1] = u;
      }
    }
  };
  if (F.g_on && r2 >= 0.0f && r2 < 1.0e12f) {
    const float r = sqrtf(r2) * 1.0001f + 0.01f;
    int x0 = (int)floorf((qx - r) * F.g_inv), x1 = (int)floorf((qx + r) * F.g_inv);
    int y0 = (int)floorf((qy - r) * F.g_inv), y1 = (int)floorf((qy + r) * F.g_inv);
    // both ends clamped INTO the grid: saddles outside the image sit in the border buckets
    // (grid_bucket clamps too), so a window hanging over the edge must still reach those
    x0 = x0 < 0 ? 0 : (x0 >= F.g_nx ? F.g_nx - 1 : x0); y0 = y0 < 0 ? 0 : (y0 >= F.g_ny ? F.g_ny - 1 : y0);
    x1 = x1 >= F.g_nx ? F.g_nx - 1 : (x1 < 0 ? 0 : x1); y1 = y1 >= F.g_ny ? F.g_ny - 1 : (y1 < 0 ? 0 : y1);
    const int bw = x1 - x0 + 1;
    if (bw > 0)
      for (int by = y0; by <= y1; ++by) {
        const int b0 = by * F.g_nx + x0;
        const int e1 = F.g_start[b0 + bw];
        for (int e = F.g_start[b0]; e < e1; ++e) consider(F.g_item[e]);
      }
  } else {
    for (int i = 0; i < F.n; ++i) consider(i);
  }
  int cnt = 0;
  for (int r = 0; r < 3; ++r)
    if (bi[r] != kNone) out[cnt++] = bi[r];
  return cnt;
}

// Nearest single saddle (board.rs:88).
AGB_NOINLINE int nearest1(const Frame& F, float qx, float qy) {
  float bd = 3.0e38f;
  int bi = kNone;
  for (int i = F.lane; i < F.n; i += AGB_LANES) {
    float d = dist2(F, qx, qy, i);
    if (nn_less(d, i, bd, bi)) { bd = d; bi = i; }
  }
  warp_argmin(bd, bi);
  return bi;
}

// The k (<= 64) nearest saddles of a point, ascending, written to F.nn_idx; returns the count.
// Selection by repeated extraction: each round takes the smallest (d2, idx) strictly greater
// than the previous pick.
#if AGB_DEVICE
// ... restricted to a window of grid buckets around the query, when the grid is on: the selection
// below over the window's saddles only, accepted when the k-th distance found is strictly smaller
// than the distance from the query to every side of the window that has buckets beyond it (a
// saddle in a bucket beyond a side is at least that far away, also after rounding: dx, dx*dx and
// the sum are monotone), otherwise repeated with a larger window.  Same picks as the full scan.
__device__ __forceinline__ int nearest_k_window(Frame& F, float qx, float qy, int kk) {
  const int nx = F.g_nx, ny = F.g_ny;
  const float bsz = 1.0f / F.g_inv;  // a power of two: bucket edges are exact
  int cx = (int)floorf(qx * F.g_inv), cy = (int)floorf(qy * F.g_inv);
  cx = cx < 0 ? 0 : (cx >= nx ? nx - 1 : cx);
  cy = cy < 0 ? 0 : (cy >= ny ? ny - 1 : cy);
  // first half-width: the window holds ~2.5 k saddles at the frame's average density
  int w = 1;
  while ((long long)(2 * w + 1) * (2 * w + 1) * F.n * 2 < 5ll * kk * nx * ny && w < 64) ++w;
  for (;;) {
    const int x0 = cx - w < 0 ? 0 : cx - w, x1 = cx + w >= nx ? nx - 1 : cx + w;
    const int y0 = cy - w < 0 ? 0 : cy - w, y1 = cy + w >= ny ? ny - 1 : cy + w;
    const int bw = x1 - x0 + 1;
    int cnt = 0;
    float last_d = -1.0f;
    int last_i = -1;
    for (int r = 0; r < kk; ++r) {
      float bd = 3.0e38f;
      int bi = kNone;
      // eight bucket rows per pass, four lanes per row
      for (int rb = y0; rb <= y1; rb += 8) {
        const int row = rb + (F.lane >> 2);
        if (row <= y1) {
          const int b0 = row * nx + x0;
          const int e1 = F.g_start[b0 + bw];
          for (int e = F.g_start[b0] + (F.lane & 3); e < e1; e += 4) {
            const int i = F.g_item[e];
            const float d = dist2(F, qx, qy, i);
            if (nn_less(last_d, last_i, d, i) && nn_less(d, i, bd, bi)) { bd = d; bi = i; }
          }
        }
      }
      warp_argmin(bd, bi);
      if (bi == kNone) break;
      if (F.lane == 0) F.nn_idx[cnt] = (int16_t)bi;
      ++cnt;
      last_d = bd;
      last_i = bi;
    }
    const bool whole = x0 == 0 && y0 == 0 && x1 == nx - 1 && y1 == ny - 1;
    if (whole) return cnt;
    float r_in = 3.0e38f;
    if (x0 > 0) r_in = fminf(r_in, fsub(qx, (float)x0 * bsz));
    if (x1 < nx - 1) r_in = fminf(r_in, fsub((float)(x1 + 1) * bsz, qx));
    if (y0 > 0) r_in = fminf(r_in, fsub(qy, (float)y0 * bsz));
    if (y1 < ny - 1) r_in = fminf(r_in, fsub((float)(y1 + 1) * bsz, qy));
    if (cnt == kk && r_in > 0.0f && last_d < fmul(r_in, r_in)) return cnt;
    w *= 2;
  }
}
#endif
AGB_NOINLINE int nearest_k(Frame& F, float qx, float qy, int k) {
  int cnt = 0;
  float last_d = -1.0f;
  int last_i = -1;
  const int kk = k < F.n ? k : F.n;
#if AGB_DEVICE
  if (F.g_on && kk > 0 && fabsf(qx) < 1.0e9f && fabsf(qy) < 1.0e9f) {  // (false for NaN)
    cnt = nearest_k_window(F, qx, qy, kk);
    __syncwarp();
    return cnt;
  }
#endif
  for (int r = 0; r < kk; ++r) {
    float bd = 3.0e38f;
    int bi = kNone;
    for (int i = F.lane; i < F.n; i += AGB_LANES) {
      float d = dist2(F, qx, qy, i);
      if (nn_less(last_d, last_i, d, i) && nn_less(d, i, bd, bi)) { bd = d; bi = i; }
    }
    warp_argmin(bd, bi);
    if (bi == kNone) break;
    if (F.lane == 0) F.nn_idx[cnt] = (int16_t)bi;
    ++cnt;
    last_d = bd;
    last_i = bi;
  }
  AGB_SYNC();
  return cnt;
}

// ---- Board (board.rs) -----------------------------------------------------------------------
// x is the major axis so that ascending cell index == ascending (x, y).
AGB_FN int cell_index(const Frame& F, int x, int y) { return (x + F.lat_off) * F.lat + (y + F.lat_off); }
AGB_FN int cell_x(const Frame& F, int ci) { return ci / F.lat - F.lat_off; }
AGB_FN int cell_y(const Frame& F, int ci) { return ci % F.lat - F.lat_off; }
AGB_FN bool cell_in_range(const Frame& F, int x, int y) {
  return x >= -F.lat_off && x < F.lat_off && y >= -F.lat_off && y < F.lat_off;
}

AGB_FN bool is_active(const BoardState& B, int i) { return (B.active[i >> 5] >> (i & 31)) & 1u; }
// single-writer (lane 0) updates
AGB_FN void clear_active(BoardState& B, int i) { B.active[i >> 5] &= ~(1u << (i & 31)); }

// Undo everything the previous build on this state did (cells back to 0, saddles active).
AGB_FN void board_reset(Frame& F, BoardState& B) {
  for (int t = F.lane; t < B.n_touched; t += AGB_LANES) B.cell[B.touched[t]] = 0;
  AGB_SYNC();
  if (F.lane == 0)
    for (int t = 0; t < B.n_quads * 4; ++t) {
      const int i = B.quads[t];
      B.active[i >> 5] |= 1u << (i & 31);
    }
  AGB_SYNC();
  B.n_touched = 0;
  B.n_quads = 0;
  B.score = 0;
}

// best_board_option = Some(board): keep a copy of the live board.
AGB_FN void board_save(Frame& F, const BoardState& B, BoardRecord& R) {
  for (int t = F.lane; t < B.n_quads * 4; t += AGB_LANES) R.quads[t] = B.quads[t];
  for (int t = F.lane; t < B.n_touched; t += AGB_LANES) {
    const int ci = B.touched[t];
    R.touched[t] = (int16_t)ci;
    R.vals[t] = B.cell[ci];
  }
  R.n_quads = B.n_quads;
  R.n_touched = B.n_touched;
  R.score = B.score;
  AGB_SYNC();
}
// Make the saved board the live one again (its active mask is not needed any more).
AGB_FN void board_load(Frame& F, BoardState& B, const BoardRecord& R) {
  board_reset(F, B);
  for (int t = F.lane; t < R.n_quads * 4; t += AGB_LANES) B.quads[t] = R.quads[t];
  for (int t = F.lane; t < R.n_touched; t += AGB_LANES) {
    B.touched[t] = R.touched[t];
    B.cell[R.touched[t]] = R.vals[t];
  }
  B.n_quads = R.n_quads;
  B.n_touched = R.n_touched;
  B.score = R.score;
  AGB_SYNC();
}

// One of the four neighbour searches of try_expand_one: find_closest_potential_saddle_idxs
// (board.rs:177-234) for the edge a -> b, candidates for the successor of `self_is_b ? b : a`.
// Runs on a single lane.
AGB_FN int closest_candidates_single(const Frame& F, const BoardState& B, int a, int b, bool self_is_b,
                                     int out[3]) {
  const float ratio0 = fadd(1.0f, 0.3f);  // 1.0 + spacing_ratio; detector.rs:621 passes 0.3
  float dx = fsub(F.sx[a], F.sx[b]), dy = fsub(F.sy[a], F.sy[b]);
  float radius_sq = fmul(0.5f, fadd(fmul(dx, dx), fmul(dy, dy)));
  float v10x = fsub(F.sx[b], F.sx[a]), v10y = fsub(F.sy[b], F.sy[a]);
  const int self = self_is_b ? b : a;
  float px = fadd(F.sx[self], fmul(v10x, ratio0)), py = fadd(F.sy[self], fmul(v10y, ratio0));
  int nn[3];
#if defined(AGB_WORK_COUNTERS) && !defined(__CUDA_ARCH__)
  agb_note_query(a, b, self_is_b ? 1 : 0, px, py, radius_sq);
#endif
  const int c = nearest3_within_single(F, px, py, radius_sq, nn);
  int k = 0;
  for (int j = 0; j < c; ++j)
    if (is_active(B, nn[j]) && theta_distance_degree(F.st[self], F.st[nn[j]]) < 5.0f) out[k++] = nn[j];
  return k;
}

#if AGB_DEVICE
// The four neighbour searches of try_expand_one on one warp: 8 lanes per search, each lane
// scanning one row of grid buckets, then a 3-round minimum extraction inside the 8-lane group.
// A candidate is the 64-bit key (d2 bits << 32 | index): d2 >= 0, so unsigned key order is the
// (d2, index) order of nn_less.  Same candidates, same order as closest_candidates_single.
__device__ __forceinline__ void expand_queries_warp(const Frame& F, const BoardState& B, const int q[4],
                                                    int cand[4][3], int cnt[4]) {
  const int grp = F.lane >> 3, sub = F.lane & 7;
  // group 0: new_s0s (edge s0->s1, from s0)   group 1: new_s1s (edge s0->s1, from s1)
  // group 2: new_s2s (edge s3->s2, from s2)   group 3: new_s3s (edge s3->s2, from s3)
  const int a = grp < 2 ? q[0] : q[3], b = grp < 2 ? q[1] : q[2];
  const int self = (grp == 1 || grp == 2) ? b : a;
  const float ratio0 = fadd(1.0f, 0.3f);
  const float ax = F.sx[a], ay = F.sy[a], bx = F.sx[b], by = F.sy[b];
  const float dx = fsub(ax, bx), dy = fsub(ay, by);
  const float r2 = fmul(0.5f, fadd(fmul(dx, dx), fmul(dy, dy)));
  const float v10x = fsub(bx, ax), v10y = fsub(by, ay);
  const float qx = fadd(F.sx[self], fmul(v10x, ratio0)), qy = fadd(F.sy[self], fmul(v10y, ratio0));
  const unsigned long long kInf = ~0ull;
  unsigned long long k0 = kInf, k1 = kInf, k2 = kInf;
  auto consider = [&](int i) {
    const float d = dist2(F, qx, qy, i);
    if (d <= r2) {
      unsigned long long k = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)i;
      if (k < k2) {
        k2 = k;
        if (k2 < k1) { unsigned long long t = k1; k1 = k2; k2 = t; }
        if (k1 < k0) { unsigned long long t = k0; k0 = k1; k1 = t; }
      }
    }
  };
  if (F.g_on && r2 >= 0.0f && r2 < 1.0e12f) {
    const float r = sqrtf(r2) * 1.0001f + 0.01f;
    int x0 = (int)floorf((qx - r) * F.g_inv), x1 = (int)floorf((qx + r) * F.g_inv);
    int y0 = (int)floorf((qy - r) * F.g_inv), y1 = (int)floorf((qy + r) * F.g_inv);
    // both ends clamped INTO the grid: saddles outside the image sit in the border buckets
    // (grid_bucket clamps too), so a window hanging over the edge must still reach those
    x0 = x0 < 0 ? 0 : (x0 >= F.g_nx ? F.g_nx - 1 : x0); y0 = y0 < 0 ? 0 : (y0 >= F.g_ny ? F.g_ny - 1 : y0);
    x1 = x1 >= F.g_nx ? F.g_nx - 1 : (x1 < 0 ? 0 : x1); y1 = y1 >= F.g_ny ? F.g_ny - 1 : (y1 < 0 ? 0 : y1);
    const int bw = x1 - x0 + 1;
    if (bw > 0)
      for (int yy = y0 + sub; yy <= y1; yy += 8) {
        const int b0 = yy * F.g_nx + x0;
        const int e1 = F.g_start[b0 + bw];
        for (int e = F.g_start[b0]; e < e1; ++e) consider(F.g_item[e]);
      }
  } else {
    for (int i = sub; i < F.n; i += 8) consider(i);
  }
  // three rounds of group-minimum extraction (xor 1, 2, 4 stay inside the aligned 8-lane group)
  unsigned long long res[3];
#pragma unroll
  for (int rnd = 0; rnd < 3; ++rnd) {
    unsigned long long m = k0;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, m, o);
      m = other < m ? other : m;
    }
    res[rnd] = m;
    if (k0 == m && m != kInf) { k0 = k1; k1 = k2; k2 = kInf; }
  }
  // lanes 0..2 of each group filter one candidate each (active mask, theta), board.rs:199-210
  bool ok = false;
  if (sub < 3) {
    const unsigned long long k = sub == 0 ? res[0] : (sub == 1 ? res[1] : res[2]);
    if (k != kInf) {
      const int i = (int)(unsigned)k;
      ok = is_active(B, i) && theta_distance_degree(F.st[self], F.st[i]) < 5.0f;
    }
  }
  const unsigned bal = __ballot_sync(0xffffffffu, ok);
  const int i0 = (int)(unsigned)res[0], i1 = (int)(unsigned)res[1], i2 = (int)(unsigned)res[2];
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const int c0 = __shfl_sync(0xffffffffu, i0, g * 8);
    const int c1 = __shfl_sync(0xffffffffu, i1, g * 8);
    const int c2 = __shfl_sync(0xffffffffu, i2, g * 8);
    const unsigned m = (bal >> (g * 8)) & 7u;
    int n = 0;
    if (m & 1u) cand[g][n++] = c0;
    if (m & 2u) cand[g][n++] = c1;
    if (m & 4u) cand[g][n++] = c2;
    cnt[g] = n;
  }
}
#endif

// try_expand_one (board.rs:153-176).  The four neighbour searches are independent and run side
// by side; the candidate 4-tuples are then tested in the reference's nested-loop order (i0
// outermost, i3 innermost), 32 at a time, and the first valid one wins.
#if defined(AGB_WORK_COUNTERS) && !defined(__CUDA_ARCH__)
extern "C" void agb_note_key(int kind, unsigned long long key);
#define AGB_NOTE(kind, key) agb_note_key(kind, key)
#else
#define AGB_NOTE(kind, key) ((void)0)
#endif
AGB_NOINLINE bool try_expand_one(const Frame& F, const BoardState& B, const int q[4], int out[4]) {
  int cand[4][3], cnt[4];
  AGB_NOTE(0, ((unsigned long long)q[0] << 16) | q[1]);
  AGB_NOTE(0, ((unsigned long long)q[3] << 16) | q[2]);
  AGB_NOTE(1, ((unsigned long long)q[0] << 48) | ((unsigned long long)q[1] << 32) | ((unsigned long long)q[2] << 16) | q[3]);
#if AGB_DEVICE
  expand_queries_warp(F, B, q, cand, cnt);
#else
  cnt[0] = closest_candidates_single(F, B, q[0], q[1], false, cand[0]);
  cnt[1] = closest_candidates_single(F, B, q[0], q[1], true, cand[1]);
  cnt[2] = closest_candidates_single(F, B, q[3], q[2], true, cand[2]);
  cnt[3] = closest_candidates_single(F, B, q[3], q[2], false, cand[3]);
#endif
  const int total = cnt[0] * cnt[1] * cnt[2] * cnt[3];
  AGB_COUNT(4, 1);
  AGB_COUNT(6, total);
  for (int base = 0; base < total; base += AGB_LANES) {
    const int c = base + F.lane;
    bool valid = false;
    int i0 = 0, i1 = 0, i2 = 0, i3 = 0;
    if (c < total) {
      int r = c;
      i3 = r % cnt[3]; r /= cnt[3];
      i2 = r % cnt[2]; r /= cnt[2];
      i1 = r % cnt[1]; r /= cnt[1];
      i0 = r;
      valid = is_valid_quad(F, cand[0][i0], cand[1][i1], cand[2][i2], cand[3][i3]);
      AGB_NOTE(2, ((unsigned long long)cand[0][i0] << 48) | ((unsigned long long)cand[1][i1] << 32) | ((unsigned long long)cand[2][i2] << 16) | cand[3][i3]);
    }
    const unsigned m = agb_ballot(valid);
    if (m) {
      const int first = base + agb_ffs(m);
      int r = first;
      i3 = r % cnt[3]; r /= cnt[3];
      i2 = r % cnt[2]; r /= cnt[2];
      i1 = r % cnt[1]; r /= cnt[1];
      i0 = r;
      out[0] = cand[0][i0]; out[1] = cand[1][i1]; out[2] = cand[2][i2]; out[3] = cand[3][i3];
      return true;
    }
  }
  return false;
}

// Board::new + try_expand (board.rs:27-48, :114-152); the recursion runs on an explicit stack.
AGB_NOINLINE void board_build(Frame& F, BoardState& B, const int quad[4]) {
  board_reset(F, B);
  const int c0 = cell_index(F, 0, 0);
  if (F.lane == 0) {
    for (int j = 1; j < 4; ++j) clear_active(B, quad[j]);  // quad[0] stays active, as in :35-37
    for (int j = 0; j < 4; ++j) B.quads[j] = (int16_t)quad[j];
    B.cell[c0] = 1;
    B.touched[0] = (int16_t)c0;
    F.stack[0] = (int16_t)c0;
    F.stack[1] = 0;
  }
  B.n_quads = 1;
  B.n_touched = 1;
  B.score = 1;
  int depth = 1;
  AGB_SYNC();
  while (depth > 0) {
    const int ci = F.stack[2 * (depth - 1)];
    const int i = F.stack[2 * (depth - 1) + 1];
    AGB_SYNC();
    if (i == 4) {
      --depth;
      continue;
    }
    if (F.lane == 0) F.stack[2 * (depth - 1) + 1] = (int16_t)(i + 1);
    const int bx = cell_x(F, ci), by = cell_y(F, ci);
    const int qi = B.cell[ci] - 1;
    int qs[4];
    for (int j = 0; j < 4; ++j) qs[j] = B.quads[qi * 4 + ((j + i) & 3)];  // rotate_left(i)
    int nx = bx, ny = by;
    if (i == 0) nx = bx + 1;
    else if (i == 1) ny = by - 1;
    else if (i == 2) nx = bx - 1;
    else ny = by + 1;
    AGB_SYNC();
    if (!cell_in_range(F, nx, ny)) {
      F.status |= 4u;  // AG_FRAME_BOARD_OVERFLOW
      continue;
    }
    const int nci = cell_index(F, nx, ny);
    const int cur = B.cell[nci];
    if (cur > 0) continue;  // already Some (board.rs:131-135)
    int nq[4];
    const bool ok = (B.n_quads < F.max_quads) && try_expand_one(F, B, qs, nq);
    AGB_SYNC();
    if (cur == 0) {
      if (F.lane == 0) B.touched[B.n_touched] = (int16_t)nci;
      ++B.n_touched;
    }
    if (ok) {
      int v[4];
      for (int j = 0; j < 4; ++j) v[(j + i) & 3] = nq[j];  // rotate_right(i)
      if (F.lane == 0) {
        for (int j = 0; j < 4; ++j) {
          clear_active(B, v[j]);
          B.quads[B.n_quads * 4 + j] = (int16_t)v[j];
        }
        B.cell[nci] = (int16_t)(B.n_quads + 1);
        F.stack[2 * depth] = (int16_t)nci;
        F.stack[2 * depth + 1] = 0;
      }
      ++B.n_quads;
      ++B.score;
      ++depth;
    } else {
      if (F.lane == 0) B.cell[nci] = -1;
    }
    AGB_SYNC();
  }
}

// try_fix_missing (board.rs:52-112).  The reference first lists the fixable holes, then
// fills them; a hole filled in this pass must therefore not serve as a neighbour of another
// hole ("was Some when the list was built" == quad index below fix_base).
AGB_NOINLINE void board_fix_missing(Frame& F, BoardState& B) {
  const int n_t = B.n_touched;
  const int fix_base = B.n_quads;
  for (int t = 0; t < n_t; ++t) {
    const int ci = B.touched[t];
    const int cv = B.cell[ci];
    if (cv != -1) continue;
    const int x = cell_x(F, ci), y = cell_y(F, ci);
    const int e0 = cell_in_range(F, x + 1, y) ? B.cell[cell_index(F, x + 1, y)] : 0;
    const int e1 = cell_in_range(F, x - 1, y) ? B.cell[cell_index(F, x - 1, y)] : 0;
    int qa = -1, qb = -1;
    if (e0 != 0 && e1 != 0) {  // contains_key(b0) && contains_key(b1)
      if (e0 > 0 && e0 - 1 < fix_base && e1 > 0 && e1 - 1 < fix_base) { qa = e0 - 1; qb = e1 - 1; }
    } else {
      const int e2 = cell_in_range(F, x, y + 1) ? B.cell[cell_index(F, x, y + 1)] : 0;
      const int e3 = cell_in_range(F, x, y - 1) ? B.cell[cell_index(F, x, y - 1)] : 0;
      if (e2 > 0 && e2 - 1 < fix_base && e3 > 0 && e3 - 1 < fix_base) { qa = e2 - 1; qb = e3 - 1; }
    }
    if (qa < 0) continue;
    int sidx[4];
    for (int j = 0; j < 4; ++j) {
      const int ia = B.quads[qa * 4 + j], ib = B.quads[qb * 4 + j];
      float mx = fdiv(fadd(F.sx[ia], F.sx[ib]), 2.0f);
      float my = fdiv(fadd(F.sy[ia], F.sy[ib]), 2.0f);
      sidx[j] = nearest1(F, mx, my);
      AGB_COUNT(7, F.n);
    }
    if (B.n_quads < F.max_quads && is_valid_quad(F, sidx[0], sidx[1], sidx[2], sidx[3])) {
      AGB_SYNC();
      if (F.lane == 0) {
        for (int j = 0; j < 4; ++j) B.quads[B.n_quads * 4 + j] = (int16_t)sidx[j];
        B.cell[ci] = (int16_t)(B.n_quads + 1);
      }
      ++B.n_quads;
      AGB_SYNC();
    }
  }
}

// (i, j), i < j, of the c-th 2-combination of n items in lexicographic order (itertools).
AGB_FN void unrank_pair(int c, int n, int* i, int* j) {
  int a = 0;
  while (c >= n - 1 - a) {
    c -= n - 1 - a;
    ++a;
  }
  *i = a;
  *j = a + 1 + c;
}

// One seed of try_find_best_board: init_quads (detector.rs:543-586) and Board::new for every
// quad (:620-626).  Leaves the seed's best board in F.seedbest and returns its score (0 = the
// seed produced no quad).  Within a seed the first board reaching the maximum wins, which is
// what the reference's strict `board.score > best_score` keeps.
AGB_NOINLINE int process_seed(Frame& F, int s0) {
  F.seedbest.n_quads = F.seedbest.n_touched = F.seedbest.score = 0;
  AGB_COUNT(0, 1);
  const int n_nn = nearest_k(F, F.sx[s0], F.sy[s0], 50);
  AGB_COUNT(1, (long long)n_nn * F.n);
  int n_same = 0, n_diff = 0;
  for (int j = 1; j < n_nn; ++j) {  // nearest[1..]: the first hit is the seed itself
    const int si = F.nn_idx[j];
    const float td = theta_distance_degree(F.st[s0], F.st[si]);
    if (td < 5.0f) {
      if (F.lane == 0) F.same[n_same] = (int16_t)si;
      ++n_same;
    } else if (td > 80.0f) {
      if (F.lane == 0) F.diff[n_diff] = (int16_t)si;
      ++n_diff;
    }
  }
  AGB_SYNC();
  const int n_pairs = n_diff * (n_diff - 1) / 2;
  // the (s0, s1)-only gate of is_valid_quad, for all candidates s1 at once (n_same <= 49)
  unsigned diag_ok[2] = {0u, 0u};
  for (int blk = 0; blk * AGB_LANES < n_same && blk < 64; ++blk) {
    const int a = blk * AGB_LANES + F.lane;
    const bool ok = a < n_same && quad_diag_ok(F, s0, F.same[a]);
    const unsigned m = agb_ballot(ok);
#if AGB_DEVICE
    diag_ok[blk & 1] = m;
#else
    if (m) diag_ok[a >> 5] |= 1u << (a & 31);
#endif
  }
  for (int a = 0; a < n_same; ++a) {
    const int s1 = F.same[a];
    if (!((diag_ok[a >> 5] >> (a & 31)) & 1u)) continue;  // every quad with this (s0, s1) fails :31
    AGB_COUNT(2, n_pairs);
    for (int base = 0; base < n_pairs; base += AGB_LANES) {
      const int c = base + F.lane;
      bool valid = false;
      if (c < n_pairs) {
        int i, j;
        unrank_pair(c, n_diff, &i, &j);
        valid = quad_rest_ok(F, s0, F.diff[i], s1, F.diff[j]);
      }
      unsigned m = agb_ballot(valid);
      while (m) {
        const int b = agb_ffs(m);
        m &= m - 1;
        int i, j;
        unrank_pair(base + b, n_diff, &i, &j);
        const int d0 = F.diff[i], d1 = F.diff[j];
        const float c0 = cross2(fsub(F.sx[d0], F.sx[s0]), fsub(F.sy[d0], F.sy[s0]),
                                fsub(F.sx[s1], F.sx[s0]), fsub(F.sy[s1], F.sy[s0]));
        int quad[4];
        quad[0] = s0; quad[2] = s1;
        if (c0 > 0.0f) { quad[1] = d0; quad[3] = d1; }
        else { quad[1] = d1; quad[3] = d0; }
        AGB_COUNT(3, 1);
        board_build(F, F.bs, quad);  // Board::new(refined, active_mask, &q, 0.3, tree)
        if (F.bs.score > F.seedbest.score) board_save(F, F.bs, F.seedbest);
      }
    }
  }
  return F.seedbest.score;
}

// Most populated round(theta) bin -> seed list (detector.rs:601-616); one warp.  Leaves the
// number of seeds in F.ctl[0] and the grid flag in F.ctl[5].
AGB_NOINLINE void select_seeds(Frame& F) {
  // histogram of round(theta)
  for (int b = F.lane; b < kHistBins; b += AGB_LANES) F.hist[b] = 0;
  AGB_SYNC();
  for (int i = F.lane; i < F.n; i += AGB_LANES) {
    int key = sat_i32(roundf(F.st[i])) + 90;
    key = key < 0 ? 0 : (key >= kHistBins ? kHistBins - 1 : key);
#if AGB_DEVICE
    atomicAdd(&F.hist[key], 1);
#else
    F.hist[key] += 1;
#endif
  }
  AGB_SYNC();
  int best_cnt = -1, best_key = -1;
  for (int b = F.lane; b < kHistBins; b += AGB_LANES) {
    int c = F.hist[b];
    if (c > best_cnt || (c == best_cnt && b > best_key)) { best_cnt = c; best_key = b; }
  }
#if AGB_DEVICE
  for (int o = 16; o > 0; o >>= 1) {
    int oc = __shfl_xor_sync(0xffffffffu, best_cnt, o);
    int ok = __shfl_xor_sync(0xffffffffu, best_key, o);
    if (oc > best_cnt || (oc == best_cnt && ok > best_key)) { best_cnt = oc; best_key = ok; }
  }
#endif
  // seeds: members of that bin in ascending index order
  int n_seeds = 0;
  for (int base = 0; base < F.n; base += AGB_LANES) {
    int i = base + F.lane;
    bool in = false;
    if (i < F.n) {
      int key = sat_i32(roundf(F.st[i])) + 90;
      key = key < 0 ? 0 : (key >= kHistBins ? kHistBins - 1 : key);
      in = key == best_key;
    }
    unsigned m = agb_ballot(in);
#if AGB_DEVICE
    if (in) F.seeds[n_seeds + __popc(m & ((1u << F.lane) - 1u))] = (int16_t)i;
    n_seeds += __popc(m);
#else
    if (in) F.seeds[n_seeds] = (int16_t)i;
    n_seeds += (int)m;
#endif
  }
  AGB_COUNT(9, n_seeds);
  AGB_COUNT(10, F.n);
  if (F.lane == 0) {
    F.ctl[0] = n_seeds;
    F.ctl[5] = F.g_on;
  }
}

// try_find_best_board (detector.rs:588-639).  Seeds are handed to the warps of the block in
// waves; after each wave the per-seed results are merged in the reference's seed order, with
// its `score > best_score` replacement, its `best_score >= 36` early exit and its limit of 30
// seeds.  Work done for seeds past the early exit is discarded, so the outcome equals the
// sequential loop.  Returns 1 with the best board (after try_fix_missing) live in warp 0's
// F.bs, or -1 for None.  Every warp of the block must call it (block-wide barriers inside).
AGB_NOINLINE int find_best_board(Frame& F) {
  if (F.n == 0) return -1;
  if (F.warp == 0) {
    grid_build(F);
    select_seeds(F);
  }
  AGB_BLOCK_SYNC();
  int seeds_left = F.ctl[0];
  F.g_on = F.ctl[5];  // the grid was (or was not) built by warp 0 for everybody
#if AGB_DEVICE
  if (F.g_on) F.g_start = F.g_base + 1;  // layout of grid_build_parallel
#endif
  int best_score = 0, count = 0;
  bool stop = false;
  while (seeds_left > 0 && count < 30 && !stop) {
    // s0_idxs.pop(): seeds are taken from the back; warp w of this wave gets the w-th pop
    const int pos = seeds_left - 1 - F.warp;
    const bool valid = pos >= 0 && count + F.warp < 30;
    int sc = -1;
    if (valid) sc = process_seed(F, F.seeds[pos]);
    if (F.lane == 0) F.w_score[F.warp] = sc;
    AGB_BLOCK_SYNC();
    int winner = -1, consumed = 0;
    for (int w = 0; w < F.n_warps; ++w) {
      const int s = F.w_score[w];
      if (s < 0) break;
      ++consumed;
      if (s > best_score) { best_score = s; winner = w; }
      if (best_score >= 36) { stop = true; break; }
      ++count;
    }
    if (winner == F.warp) {  // best_board_option = Some(board)
      const BoardRecord& R = F.seedbest;
      for (int t = F.lane; t < R.n_quads * 4; t += AGB_LANES) F.best.quads[t] = R.quads[t];
      for (int t = F.lane; t < R.n_touched; t += AGB_LANES) {
        F.best.touched[t] = R.touched[t];
        F.best.vals[t] = R.vals[t];
      }
      if (F.lane == 0) {
        F.ctl[2] = R.n_quads;
        F.ctl[3] = R.n_touched;
        F.ctl[4] = R.score;
      }
    }
    seeds_left -= consumed;
    AGB_BLOCK_SYNC();
  }
  if (best_score == 0) return -1;
  if (F.warp == 0) {
    F.best.n_quads = F.ctl[2];
    F.best.n_touched = F.ctl[3];
    F.best.score = F.ctl[4];
    board_load(F, F.bs, F.best);
    board_fix_missing(F, F.bs);
  }
  return 1;
}

// ---- decoding (detector.rs:42-169, :448-476) ---------------------------------------------------
// to_luma8 of pixel x of a row of LA8 (4), RGBA8 (5), LA16 (6), RGB16 (7), RGBA16 (8), RGB32F (9) or
// RGBA32F (10): alpha is dropped, colour is the integer sRGB luma in the source width (u16 luma is
// scaled to u8) or, for f32, the f64 luma of ag_float_luma.h.  Out of line, so that the frame formats
// of the benchmark keep the board kernel's code as it was.
AGB_NOINLINE int luma8_wide(const uint8_t* row, uint32_t x, int format) {
  const uint16_t* r16 = (const uint16_t*)row;
  if (format >= 9) {
    const float* p = (const float*)row + (format == 9 ? 3 : 4) * (size_t)x;
    return (int)ag::luma32f_to_u8(ag::rgb32f_luma(p[0], p[1], p[2]));
  }
  if (format == 4) return row[2 * (size_t)x];
  if (format == 5) {
    const uint8_t* p = row + 4 * (size_t)x;
    return (int)((2126u * p[0] + 7152u * p[1] + 722u * p[2]) / 10000u);
  }
  if (format == 6) return (int)((((uint32_t)r16[2 * (size_t)x]) + 128u) / 257u);
  const uint16_t* p = r16 + (format == 7 ? 3 : 4) * (size_t)x;
  return (int)(((2126u * p[0] + 7152u * p[1] + 722u * p[2]) / 10000u + 128u) / 257u);
}

// image 0.25 to_luma8 of pixel (x, y) in the public pixel format F.format (include/aprilgrid_b200.h)
AGB_FN int luma8_at(const Frame& F, uint32_t x, uint32_t y) {
  const uint8_t* row = F.img + (size_t)y * F.row_stride;
  if (F.format == 0) return row[x];
  if (F.format == 1) return (int)((((uint32_t)((const uint16_t*)row)[x]) + 128u) / 257u);
  if (F.format != 2) return luma8_wide(row, x, F.format);
  const uint8_t* p = row + 3 * (size_t)x;
  return (int)((2126u * p[0] + 7152u * p[1] + 722u * p[2]) / 10000u);
}

// rotate_bits (detector.rs:124-140)
AGB_FN uint64_t rotate_bits(uint64_t bits, int edge) {
  uint64_t b = 0;
  int count = 0;
  for (int r = edge - 1; r >= 0; --r)
    for (int c = 0; c < edge; ++c) {
      int idx = r + c * edge;
      b |= ((bits >> idx) & 1ull) << count;
      ++count;
    }
  return b;
}

// Decode, phase 1: ONE LANE per quad (on the device; the host test build runs the same code).  decode_positions + tag_affine + bit_code
// (detector.rs:42-122) up to the bit pattern; returns the pattern with bit 63 set, or 0 when the
// quad is rejected.  32 quads run side by side, which hides the f64 arithmetic of the affine fit
// and the memory latency of the 36 samples that a whole warp per quad would wait for serially.
AGB_NOINLINE uint64_t decode_bits_lane(const Frame& F, int q0, int q1, int q2, int q3) {
  const float qx[4] = {F.sx[q0], F.sx[q1], F.sx[q2], F.sx[q3]};
  const float qy[4] = {F.sy[q0], F.sy[q1], F.sy[q2], F.sy[q3]};
  for (int j = 0; j < 4; ++j) {  // decode_positions :50-56
    const uint32_t x = sat_u32(roundf(qx[j])), y = sat_u32(roundf(qy[j]));
    if (x >= (uint32_t)F.w || y >= (uint32_t)F.h) return 0ull;
  }
  // tag_affine (image_util.rs:39-70), same arithmetic as decode_quad
  const int side = F.border * 2 + F.edge;
  const float lo = -0.5f, hi = (float)side - 1.0f + 0.5f;
  const double sxs[4] = {lo, lo, hi, hi};
  const double sys[4] = {lo, hi, hi, lo};
  double mx = 0, my = 0, mcx = 0, mcy = 0;
  for (int p = 0; p < 4; ++p) { mx += sxs[p]; my += sys[p]; mcx += qx[p]; mcy += qy[p]; }
  mx /= 4; my /= 4; mcx /= 4; mcy /= 4;
  double sxx = 0, syy = 0, axx = 0, axy = 0, ayx = 0, ayy = 0;
  for (int p = 0; p < 4; ++p) {
    double dx = sxs[p] - mx, dy = sys[p] - my;
    sxx += dx * dx; syy += dy * dy;
    axx += dx * qx[p]; axy += dy * qx[p];
    ayx += dx * qy[p]; ayy += dy * qy[p];
  }
  const double h0d = axx / sxx, h1d = axy / syy, h3d = ayx / sxx, h4d = ayy / syy;
  const float h0 = (float)h0d, h1 = (float)h1d, h2 = (float)(mcx - h0d * mx - h1d * my);
  const float h3 = (float)h3d, h4 = (float)h4d, h5 = (float)(mcy - h3d * mx - h4d * my);
  // bit_code :80-122; sample s = (x - border) * edge + (y - border), x outer.  Two passes over the
  // sample grid, one grid row (<= 6 samples, loaded together so their latencies overlap) per trip of
  // a ROLLED loop: first the brightness range, then the bits -- the second pass reads the same few
  // bytes again (cache hits).  Rolled on purpose: fully unrolled, this function was a third of the
  // board kernel's code and its instruction-cache footprint hurt the search loops of the other
  // frames on the SM.
  const int edge = F.edge, ns = edge * edge;
  auto sample_row = [&](int ix, int v[6]) -> bool {  // false: a sample outside the image
    bool inside = true;
    const float fx = (float)(F.border + ix);
AGB_UNROLL
    for (int iy = 0; iy < 6; ++iy) {
      v[iy] = 0;
      if (iy < edge) {
        const float fy = (float)(F.border + iy);
        const float px = fadd(fadd(fmul(h0, fx), fmul(h1, fy)), h2);
        const float py = fadd(fadd(fmul(h3, fx), fmul(h4, fy)), h5);
        const uint32_t x = sat_u32(roundf(px)), y = sat_u32(roundf(py));
        if (x < (uint32_t)F.w && y < (uint32_t)F.h) v[iy] = luma8_at(F, x, y);
        else inside = false;
      }
    }
    return inside;
  };
  int min_b = 255, max_b = 0;
  bool oob = false;
#if AGB_DEVICE
#pragma unroll 1
#endif
  for (int ix = 0; ix < edge; ++ix) {
    int v[6];
    if (!sample_row(ix, v)) oob = true;
AGB_UNROLL
    for (int iy = 0; iy < 6; ++iy)
      if (iy < edge) {
        min_b = v[iy] < min_b ? v[iy] : min_b;
        max_b = v[iy] > max_b ? v[iy] : max_b;
      }
  }
  if (oob) return 0ull;  // a sample outside the image
  if (max_b - min_b < 50) return 0ull;  // :97
  const int mid_b = (int)sat_u32(roundf(fdiv(fadd((float)min_b, (float)max_b), 2.0f)));
  uint64_t bits = 0;
  int invalid = 0;
#if AGB_DEVICE
#pragma unroll 1
#endif
  for (int ix = 0; ix < edge; ++ix) {
    int v[6];
    sample_row(ix, v);
AGB_UNROLL
    for (int iy = 0; iy < 6; ++iy)
      if (iy < edge) {
        const int dlt = mid_b - v[iy];
        if ((dlt < 0 ? -dlt : dlt) < 10) ++invalid;
        if (v[iy] > mid_b) bits |= 1ull << (ns - 1 - (ix * edge + iy));  // the first sample is the most significant bit
      }
  }
  if (invalid > 3) return 0ull;
  return bits | (1ull << 63);
}

// try_decode_quad for the host test build: the bit pattern by decode_bits_lane (the very function
// the device runs, one lane per quad), then best_tag as a plain loop (the device searches the code
// table with best_tag_warp below: all four rotations in one pass, same first-minimum rule).
// On success fills *out (id + rotated, reversed corners).
AGB_NOINLINE bool decode_quad(Frame& F, const int q[4], TagRec* out) {
  const uint64_t packed = decode_bits_lane(F, q[0], q[1], q[2], q[3]);
  if (!(packed >> 63)) return false;
  uint64_t bits = packed & ~(1ull << 63);
  // best_tag :142-169
  int id = -1, rot = 0;
  for (int rotated = 0; rotated < 4; ++rotated) {
    int bs = 1000, bi = kNone;
    for (int c = 0; c < F.n_codes; ++c) {
      const int sc = agb_popcll(F.codes[c] ^ bits);
      if (sc < bs) { bs = sc; bi = c; }  // first minimum
    }
    if (bs < F.hamming) {
      id = bi;
      rot = rotated;
      break;
    }
    if (rotated == 3) break;
    bits = rotate_bits(bits, F.edge);
  }
  if (id < 0) return false;
  out->id = (uint32_t)id;
  for (int j = 0; j < 4; ++j) {  // rotate_left(rot) then reverse() (:467-469)
    const int src = ((3 - j) + rot) & 3;
    out->xy[2 * j] = F.sx[q[src]];
    out->xy[2 * j + 1] = F.sy[q[src]];
  }
  return true;
}

#if AGB_DEVICE
__device__ int find_best_board_fast(Frame& F);  // ag_board_fast.cuh

// Device decode, phase 2: best_tag (detector.rs:142-169) for one pattern on the whole warp.
// Returns the id (and the rotation) or -1.
__device__ __noinline__ int best_tag_warp(const Frame& F, uint64_t bits, int* rot_out) {
  const uint64_t* __restrict__ codes = F.codes;  // the frame's fields, once (F lives in local memory)
  const int n_codes = F.n_codes, hamming = F.hamming, edge = F.edge, lane = F.lane;
  const int ns = edge * edge;
  uint64_t br[4];
  br[0] = bits;
  int src[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {  // rotate_bits: output bit `count` <- input bit r + c * edge
    const int count = lane + 32 * h;
    src[h] = count < ns ? (edge - 1 - count / edge) + (count % edge) * edge : -1;
  }
#pragma unroll
  for (int r = 1; r < 4; ++r) {
    const unsigned lo = __ballot_sync(0xffffffffu, src[0] >= 0 && ((br[r - 1] >> src[0]) & 1ull));
    const unsigned hi = __ballot_sync(0xffffffffu, src[1] >= 0 && ((br[r - 1] >> src[1]) & 1ull));
    br[r] = (uint64_t)lo | ((uint64_t)hi << 32);
  }
  unsigned key[4] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0xffffffffu};
#pragma unroll 4
  for (int c = lane; c < n_codes; c += 32) {
    const uint64_t code = __ldg(codes + c);
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const unsigned k = ((unsigned)__popcll(code ^ br[r]) << 16) | (unsigned)c;
      key[r] = k < key[r] ? k : key[r];
    }
  }
  int id = -1;
#pragma unroll
  for (int r = 3; r >= 0; --r) {
    const unsigned k = __reduce_min_sync(0xffffffffu, key[r]);
    if ((int)(k >> 16) < hamming) { id = (int)(k & 0xffffu); *rot_out = r; }
  }
  return id;
}

// Decoding of the found board (detector.rs:512-536) by the whole block.  Warp 0 lists the board's
// quads in visiting order; every thread of the block then takes quads for the bit patterns (one
// lane per quad: decode_positions, affine fit, 36 samples) and every warp takes quads for the
// code-table search (one warp per pattern); finally warp 0 enters the results into the map in
// visiting order, 32 at a time -- a repeated id overwrites, as HashMap::insert -- and marks the
// saddles of decoded quads for removal.  Returns the number of listed quads (tap).
__device__ __noinline__ int decode_board_block(Frame& F, int round) {
  int16_t* const qlist = F.dec_qlist;
  unsigned long long* const qbits = F.dec_qbits;
  if (F.warp == 0) {
    BoardState& B = F.bs;
    for (int i = F.lane; i < F.n; i += 32) F.remove[i] = 0;
    const int n_cells = F.lat * F.lat;
    int n_list = 0;
    for (int base = 0; base < n_cells; base += 32) {  // all_tag_indexes in ascending (x, y) order
      const int cv = B.cell[base + F.lane];
      const unsigned m = __ballot_sync(0xffffffffu, cv > 0);
      if (cv > 0) {
        const int dst = n_list + __popc(m & ((1u << F.lane) - 1u));
        for (int j = 0; j < 4; ++j) qlist[4 * dst + j] = B.quads[(cv - 1) * 4 + j];
      }
      n_list += __popc(m);
    }
    if (round == 0 && F.tap_quads)
      for (int i = F.lane; i < n_list && i < F.tap_cap; i += 32)
        for (int j = 0; j < 4; ++j) F.tap_quads[i * 4 + j] = qlist[4 * i + j];
    if (F.lane == 0) F.ctl[6] = n_list;
  }
  __syncthreads();
  const int n_list = F.ctl[6];
  // bit patterns: one lane per quad
  for (int i = (int)threadIdx.x; i < n_list; i += (int)blockDim.x)
    qbits[i] = decode_bits_lane(F, qlist[4 * i], qlist[4 * i + 1], qlist[4 * i + 2], qlist[4 * i + 3]);
  __syncthreads();
  // code-table search: one warp per pattern; the entry becomes valid << 63 | id << 8 | rotation
  for (int i = F.warp; i < n_list; i += F.n_warps) {
    const unsigned long long b = qbits[i];
    unsigned long long res = 0ull;
    if (b >> 63) {  // warp-uniform
      int rot = 0;
      const int id = best_tag_warp(F, b & ~(1ull << 63), &rot);
      if (id >= 0) res = (1ull << 63) | ((unsigned long long)id << 8) | (unsigned long long)rot;
    }
    __syncwarp();
    if (F.lane == 0) qbits[i] = res;
  }
  __syncthreads();
  if (F.warp == 0) {
    for (int base = 0; base < n_list; base += 32) {
      const int i = base + F.lane;
      const unsigned long long res = i < n_list ? qbits[i] : 0ull;
      const bool ok = (res >> 63) != 0ull;
      const int id = ok ? (int)((res >> 8) & 0xffffffull) : -1 - F.lane;
      const int rot = (int)(res & 3ull);
      // of the quads of this batch that decoded to the same id the last one wins (insert overwrites)
      const unsigned peers = __match_any_sync(0xffffffffu, id);
      if (ok) {
        if ((31 - __clz((int)peers)) == F.lane) {
          TagRec t;
          t.id = (uint32_t)id;
          for (int j = 0; j < 4; ++j) {  // rotate_left(rot) then reverse() (:467-469)
            const int sq = qlist[4 * i + (((3 - j) + rot) & 3)];
            t.xy[2 * j] = F.sx[sq];
            t.xy[2 * j + 1] = F.sy[sq];
          }
          F.tag_by_id[t.id] = t;
          F.tag_valid[t.id] = 1;
        }
        for (int j = 0; j < 4; ++j) F.remove[qlist[4 * i + j]] = 1;
      }
      __syncwarp();
    }
  }
  return n_list;
}
#endif
AGB_FN void detect_boards(Frame& F, int max_boards) {
  for (int round = 0; round < max_boards; ++round) {
#if defined(AGB_WORK_COUNTERS) && !defined(__CUDA_ARCH__)
    agb_work_counters[31] = round;
#endif
#if AGB_DEVICE
    F.round = round;
    const int found = F.fast_on ? find_best_board_fast(F) : find_best_board(F);
#else
    const int found = find_best_board(F);
#endif
    if (found < 0) continue;  // block-uniform
#if AGB_DEVICE
    const long long t_dec = clock64();
#endif
#if AGB_DEVICE
    const int n_tap_dev = decode_board_block(F, round);  // every warp of the block
#endif
    if (F.warp == 0) {
      BoardState& B = F.bs;
      int n_tap = 0;
      // all_tag_indexes in ascending (x, y) order
      const int n_cells = F.lat * F.lat;
#if AGB_DEVICE
      (void)B;
      (void)n_cells;
      n_tap = (round == 0 && F.tap_quads) ? n_tap_dev : 0;
#else
      // host test build (one lane): quad after quad through decode_quad
      for (int i = F.lane; i < F.n; i += AGB_LANES) F.remove[i] = 0;
      for (int base = 0; base < n_cells; base += AGB_LANES) {
        const int ci = base + F.lane;
        unsigned m = agb_ballot(B.cell[ci] > 0);
        while (m) {
          const int b = agb_ffs(m);
          m &= m - 1;
          const int qi = B.cell[base + b] - 1;
          int q[4];
          for (int j = 0; j < 4; ++j) q[j] = B.quads[qi * 4 + j];
          if (round == 0 && F.tap_quads) {
            if (F.lane == 0 && n_tap < F.tap_cap)
              for (int j = 0; j < 4; ++j) F.tap_quads[n_tap * 4 + j] = q[j];
            ++n_tap;
          }
          TagRec t;
          AGB_COUNT(8, 1);
          if (decode_quad(F, q, &t)) {
            if (F.lane == 0) {
              F.tag_by_id[t.id] = t;  // HashMap::insert: a repeated id overwrites
              F.tag_valid[t.id] = 1;
              for (int j = 0; j < 4; ++j) F.remove[q[j]] = 1;
            }
            AGB_SYNC();
          }
        }
      }
#endif
      if (round == 0 && F.tap_n_quads && F.lane == 0) *F.tap_n_quads = n_tap;
      AGB_SYNC();
      // refined.retain(not removed), order kept (:526-536).  In-place, order-preserving
      // compaction: block after block, every lane reads its element before any lane of the
      // block writes, and writes only go to indices at or below the block.
      int n_new = 0;
      for (int base = 0; base < F.n; base += AGB_LANES) {
        const int i = base + F.lane;
        const bool keep = i < F.n && !F.remove[i];
        float kx = 0.0f, ky = 0.0f, kt = 0.0f;
        if (keep) {
          kx = F.sx[i];
          ky = F.sy[i];
          kt = F.st[i];
        }
        unsigned m = agb_ballot(keep);
#if AGB_DEVICE
        const int dst = n_new + __popc(m & ((1u << F.lane) - 1u));
        const int cnt = __popc(m);
#else
        const int dst = n_new;
        const int cnt = (int)m;
#endif
        AGB_SYNC();
        if (keep) {
          F.sx[dst] = kx;
          F.sy[dst] = ky;
          F.st[dst] = kt;
        }
        AGB_SYNC();
        n_new += cnt;
      }
      if (F.lane == 0) F.ctl[1] = n_new;
#if AGB_DEVICE
      if (F.tm && F.lane == 0) F.tm[12] += (uint32_t)(clock64() - t_dec) & 0x7fffffffu;
#endif
    }
    // saddle indices changed: every warp forgets its board
    if (!F.fast_on) board_reset(F, F.bs);
    AGB_BLOCK_SYNC();
    F.n = F.ctl[1];
    AGB_BLOCK_SYNC();
  }
}

}  // namespace agb
