// =====================================================================================
// aprilgrid oracle -- TEST INFRASTRUCTURE ONLY.
//
// A single-threaded CPU restatement, in C++, of the per-frame detection front end of
// powei-lin/aprilgrid-rs 0.8.0 (the Rust crate cannot be built in this environment: no
// cargo/rustc, no vendored crates).  Every function cites the reference file:line it
// follows.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
// --impl reference legs may load this library; the product (aprilgrid-rs_b200/) never
// does and has no CPU path of its own.
//
// Parity status ("what pins this oracle"):
//   * pinned by the reference's own tests: the unit known-answers of
//     src/math_util.rs:35-90, src/saddle.rs:75-174, src/image_util.rs:238-317 and the
//     seven tag counts of tests/test_detector.rs:26-32 (66/36/36/36/36/36/72), see
//     tests/test_oracle_pins.py.
//   * PARITY UNPINNED at the bit level for arithmetic that lives in un-vendored crates:
//       image 0.25.9   (L8/L16/RGB8 -> luma f32 / luma u8 conversion formulas),
//       faer 0.23.2    (f32 Householder QR for the 25x6 pseudo-inverse and the 8x6 affine
//                       fit, 2x2 partial-pivot LU) -- restated here as exact rational /
//                       closed-form solutions evaluated in f64 and rounded once to f32,
//       kdtree 0.8.0   (k-NN; restated as exact brute force, ties -> lower index).
//   * Two places where the reference itself is nondeterministic (std HashMap iteration
//     order) are resolved by a fixed rule, see try_find_best_board() and Board.
//
// Build: g++ -O2 -ffp-contract=off (Rust never contracts a*b+c; neither may we).
// =====================================================================================
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <array>
#include <map>
#include <thread>
#include <utility>
#include <vector>

#include "codebook.inc"


namespace {

constexpr float kPi = 3.14159265358979323846264338327950288f;  // std::f32::consts::PI

struct Saddle {  // src/saddle.rs:3-9
  float x, y, k, theta, phi;
};

struct Params {  // src/detector.rs:25-41
  float tag_spacing_ratio = 0.3f;
  float min_saddle_angle = 30.0f;
  float max_saddle_angle = 60.0f;
  int max_num_of_boards = 2;
};

struct Family {  // src/detector.rs:369-405
  int edge, border, hamming;
  const uint64_t* codes;
  int n_codes;
};

bool family_by_id(int id, Family* f) {
  switch (id) {
    case 0: *f = {4, 2, 1, orc_t16h5_codes, orc_t16h5_count}; return true;
    case 1: *f = {5, 2, 2, orc_t25h7_codes, orc_t25h7_count}; return true;
    case 2: *f = {5, 2, 2, orc_t25h9_codes, orc_t25h9_count}; return true;
    case 3: *f = {6, 2, 3, orc_t36h11_codes, orc_t36h11_count}; return true;
    case 4: *f = {6, 1, 3, orc_t36h11_codes, orc_t36h11_count}; return true;  // T36H11B1
  }
  return false;
}

// Rust `f32 as u32` / `as i32` / `as u8`: saturating, NaN -> 0.
inline uint32_t sat_u32(float v) {
  if (!(v > 0.0f)) return 0u;
  if (v >= 4294967296.0f) return 0xffffffffu;
  return (uint32_t)v;
}
inline int32_t sat_i32(float v) {
  if (v != v) return 0;
  if (v >= 2147483648.0f) return INT32_MAX;
  if (v <= -2147483648.0f) return INT32_MIN;
  return (int32_t)v;
}

// ---------------------------------------------------------------------------------
// a-1  gray conversion -- `image` 0.25 DynamicImage::to_luma32f / to_luma8, called at
//      src/detector.rs:409 and :507.  fmt: 0 = L8, 1 = L16 (native endian), 2 = RGB8.
// ---------------------------------------------------------------------------------
inline uint8_t rgb_luma_u8(const uint8_t* p) {
  // image::color::rgb_to_luma: integer sRGB weights, truncating division.
  uint32_t l = 2126u * p[0] + 7152u * p[1] + 722u * p[2];
  return (uint8_t)(l / 10000u);
}

void to_luma_f32(const void* pixels, int w, int h, size_t stride, int fmt, float* out) {
  for (int y = 0; y < h; ++y) {
    const uint8_t* row = (const uint8_t*)pixels + (size_t)y * stride;
    float* o = out + (size_t)y * w;
    if (fmt == 0) {
      for (int x = 0; x < w; ++x) o[x] = (float)row[x] / 255.0f;
    } else if (fmt == 1) {
      const uint16_t* r16 = (const uint16_t*)row;
      for (int x = 0; x < w; ++x) o[x] = (float)r16[x] / 65535.0f;
    } else if (fmt == 3) {  // already a Luma<f32> plane (the caller ran to_luma32f itself): detect_planes
      memcpy(o, row, sizeof(float) * (size_t)w);
    } else {
      for (int x = 0; x < w; ++x) o[x] = (float)rgb_luma_u8(row + 3 * x) / 255.0f;
    }
  }
}

void to_luma_u8(const void* pixels, int w, int h, size_t stride, int fmt, uint8_t* out) {
  for (int y = 0; y < h; ++y) {
    const uint8_t* row = (const uint8_t*)pixels + (size_t)y * stride;
    uint8_t* o = out + (size_t)y * w;
    if (fmt == 0) {
      memcpy(o, row, (size_t)w);
    } else if (fmt == 1) {
      const uint16_t* r16 = (const uint16_t*)row;
      for (int x = 0; x < w; ++x) o[x] = (uint8_t)(((uint32_t)r16[x] + 128u) / 257u);
    } else {
      for (int x = 0; x < w; ++x) o[x] = rgb_luma_u8(row + 3 * x);
    }
  }
}

// ---------------------------------------------------------------------------------
// a-2  gaussian_blur_f32 -- src/image_util.rs:110-206
// ---------------------------------------------------------------------------------
void blur_taps(float sigma, std::vector<float>* taps, int* radius_out) {
  int radius = (int)ceilf(sigma * 2.0f);  // :111
  int size = radius * 2 + 1;
  taps->assign(size, 0.0f);
  float two_sigma_sq = 2.0f * sigma * sigma;
  float sum = 0.0f;
  for (int i = 0; i < size; ++i) {  // :116-121
    float x = (float)(i - radius);
    float v = expf(-(x * x) / two_sigma_sq);
    (*taps)[i] = v;
    sum += v;
  }
  for (float& v : *taps) v /= sum;  // :122-124
  *radius_out = radius;
}

void gaussian_blur(const float* img, int w, int h, float sigma, float* out) {
  std::vector<float> k;
  int radius;
  blur_taps(sigma, &k, &radius);
  const int size = 2 * radius + 1;
  std::vector<float> temp((size_t)w * h);
  // Horizontal pass (:138-185).  The reference splits the row into left border / centre /
  // right border; all three evaluate the same clamped sum in the same order, so one loop
  // restates them.  The centre is written without clamps so the compiler may vectorise it,
  // as LLVM does for the reference.
  for (int y = 0; y < h; ++y) {
    const float* r = img + (size_t)y * w;
    float* t = temp.data() + (size_t)y * w;
    int x = 0;
    auto clamped = [&](int xx) {
      float val = 0.0f;
      for (int i = 0; i < size; ++i) {
        int kx = std::min(std::max(xx + i - radius, 0), w - 1);
        val += r[kx] * k[i];
      }
      return val;
    };
    for (; x < std::min(radius, w); ++x) t[x] = clamped(x);
    for (; x < w - radius; ++x) {
      float val = 0.0f;
      const float* p = r + (x - radius);
      for (int i = 0; i < size; ++i) val += p[i] * k[i];
      t[x] = val;
    }
    for (; x < w; ++x) t[x] = clamped(x);
  }
  // Vertical pass (:188-203): out zero-initialised, then out[x] += temp[ky][x] * k[i] for
  // i = 0..size in order.
  for (int y = 0; y < h; ++y) {
    float* o = out + (size_t)y * w;
    for (int x = 0; x < w; ++x) o[x] = 0.0f;
    for (int i = 0; i < size; ++i) {
      int ky = std::min(std::max(y + i - radius, 0), h - 1);
      const float* t = temp.data() + (size_t)ky * w;
      const float kw = k[i];
      for (int x = 0; x < w; ++x) o[x] += t[x] * kw;
    }
  }
}

// ---------------------------------------------------------------------------------
// a-3  hessian_response -- src/image_util.rs:72-109
// ---------------------------------------------------------------------------------
void hessian_response(const float* img, int w, int h, float* out) {
  memset(out, 0, sizeof(float) * (size_t)w * h);
  for (int r = 1; r < h - 1; ++r) {
    const float* p = img + (size_t)(r - 1) * w;
    const float* c = img + (size_t)r * w;
    const float* n = img + (size_t)(r + 1) * w;
    float* o = out + (size_t)r * w;
    for (int x = 1; x < w - 1; ++x) {
      float v11 = p[x - 1], v12 = p[x], v13 = p[x + 1];
      float v21 = c[x - 1], v22 = c[x], v23 = c[x + 1];
      float v31 = n[x - 1], v32 = n[x], v33 = n[x + 1];
      float lxx = v21 - (v22 * 2.0f) + v23;           // :100
      float lyy = v12 - (v22 * 2.0f) + v32;           // :101
      float lxy = (v13 - v11 + v31 - v33) * 0.25f;    // :102
      o[x] = lxx * lyy - lxy * lxy;                   // :104
    }
  }
}

// a-4  global min and threshold -- src/detector.rs:414-418
float min_response(const float* resp, size_t n) {
  float acc = 3.40282347e+38f;  // f32::MAX
  for (size_t i = 0; i < n; ++i) acc = fminf(acc, resp[i]);  // f32::min
  return acc;
}

// ---------------------------------------------------------------------------------
// a-5  init_saddle_clusters + pixel_bfs -- src/detector.rs:171-187, src/image_util.rs:208-236
//      `mat` is consumed (visited pixels are overwritten with f32::MAX, as the reference
//      does).  Cluster order = raster order of the first pixel reached; pixel order inside
//      a cluster = the stack order of the reference.
// ---------------------------------------------------------------------------------
typedef std::vector<std::pair<uint32_t, uint32_t>> Cluster;

void pixel_bfs(float* mat, uint32_t w, uint32_t h, Cluster* cluster, uint32_t x, uint32_t y,
               float threshold, std::vector<std::pair<uint32_t, uint32_t>>* stack) {
  stack->clear();
  stack->push_back({x, y});
  while (!stack->empty()) {
    auto [cx, cy] = stack->back();
    stack->pop_back();
    if (cx >= w || cy >= h) continue;
    float v = mat[(size_t)cy * w + cx];
    if (v < threshold) {
      cluster->push_back({cx, cy});
      mat[(size_t)cy * w + cx] = 3.40282347e+38f;
      if (cx > 0) stack->push_back({cx - 1, cy});
      stack->push_back({cx + 1, cy});
      if (cy > 0) stack->push_back({cx, cy - 1});
      stack->push_back({cx, cy + 1});
    }
  }
}

void init_saddle_clusters(float* h_mat, int w, int h, float threshold,
                          std::vector<Cluster>* clusters) {
  Cluster cluster;
  std::vector<std::pair<uint32_t, uint32_t>> stack;
  for (int r = 1; r < h - 1; ++r) {
    for (int c = 1; c < w - 1; ++c) {
      float v = h_mat[(size_t)r * w + c];
      if (v < threshold) {
        cluster.clear();
        pixel_bfs(h_mat, (uint32_t)w, (uint32_t)h, &cluster, (uint32_t)c, (uint32_t)r, threshold,
                  &stack);
        if (!cluster.empty()) clusters->push_back(cluster);
      }
    }
  }
}

// a-6  centroid -- src/detector.rs:421-429 (f32 running sums in cluster order)
void cluster_centers(const std::vector<Cluster>& clusters, std::vector<std::pair<float, float>>* out) {
  out->clear();
  for (const Cluster& c : clusters) {
    float ax = 0.0f, ay = 0.0f;
    for (auto& e : c) {
      ax = ax + (float)e.first;
      ay = ay + (float)e.second;
    }
    float n = (float)c.size();
    out->push_back({ax / n, ay / n});
  }
}

// ---------------------------------------------------------------------------------
// L1 math helpers -- src/math_util.rs:5-33
// ---------------------------------------------------------------------------------
// find_xy: faer 2x2 partial-pivot LU (third-party, unpinned).  Restated as textbook LU with
// row pivoting on the larger |a|, f32 throughout.
void find_xy(float a0, float b0, float c0, float a1, float b1, float c1, float* x, float* y) {
  float r0 = -c0, r1 = -c1;
  if (fabsf(a1) > fabsf(a0)) {
    std::swap(a0, a1);
    std::swap(b0, b1);
    std::swap(r0, r1);
  }
  float l = a1 / a0;
  float u11 = b1 - l * b0;
  float z1 = r1 - l * r0;
  float yy = z1 / u11;
  float xx = (r0 - b0 * yy) / a0;
  *x = xx;
  *y = yy;
}

inline float theta_distance_degree(float t0, float t1) {  // :15-23
  float d = t0 - t1 + 90.0f;
  if (d < 0.0f) {
    d += 180.0f;
  } else if (d > 180.0f) {
    d -= 180.0f;
  }
  return d > 90.0f ? d - 90.0f : 90.0f - d;
}
inline float cross2(float ax, float ay, float bx, float by) { return ax * by - ay * bx; }  // :24
inline float dot2(float ax, float ay, float bx, float by) { return ax * bx + ay * by; }    // :27
inline float angle_degree(float ax, float ay, float bx, float by) {                         // :31
  return atan2f(by * ax - bx * ay, ax * bx + ay * by) * 180.0f / kPi;
}

// ---------------------------------------------------------------------------------
// a-7  rochade_refine -- src/detector.rs:194-361 (half_size_patch = 2 at the only call site)
// ---------------------------------------------------------------------------------
struct RochadeTables {
  int half, ksize, npix;
  std::vector<float> p_mat;   // [6][npix]
  std::vector<float> flat_k;  // [npix]
};

// The reference builds p_mat = pinv([x^2, xy, y^2, x, y, 1]) with faer's f32 QR (:208-237).
// For the symmetric (2h+1)^2 grid the normal equations decouple and the pseudo-inverse is a
// set of exact rationals; we evaluate them in f64 and round once.
void build_rochade_tables(int half, RochadeTables* t) {
  t->half = half;
  t->ksize = 2 * half + 1;
  t->npix = t->ksize * t->ksize;
  const int n = t->ksize;
  double s2 = 0, s4 = 0;  // sum of x^2 and x^4 over one axis
  for (int i = -half; i <= half; ++i) {
    s2 += (double)i * i;
    s4 += (double)i * i * i * i;
  }
  const double N = n;
  // [x^2, y^2, 1] block:  | N*s4   s2*s2  N*s2 |
  //                       | s2*s2  N*s4   N*s2 |
  //                       | N*s2   N*s2   N*N  |
  // Eliminating the constant gives a1 = (sum x^2 f - (s2/N) sum f) / (N*s4 - s2*s2).
  const double den_q = N * s4 - s2 * s2;
  t->p_mat.assign(6 * (size_t)t->npix, 0.0f);
  int idx = 0;
  for (int r = 0; r < n; ++r) {
    for (int c = 0; c < n; ++c, ++idx) {
      double x = c - half, y = r - half;
      double p1 = (x * x - s2 / N) / den_q;
      double p3 = (y * y - s2 / N) / den_q;
      double p2 = (x * y) / (s2 * s2);
      double p4 = x / (N * s2);
      double p5 = y / (N * s2);
      double p6 = (1.0 - N * s2 * (p1 + p3)) / (N * N);
      t->p_mat[0 * t->npix + idx] = (float)p1;
      t->p_mat[1 * t->npix + idx] = (float)p2;
      t->p_mat[2 * t->npix + idx] = (float)p3;
      t->p_mat[3 * t->npix + idx] = (float)p4;
      t->p_mat[4 * t->npix + idx] = (float)p5;
      t->p_mat[5 * t->npix + idx] = (float)p6;
    }
  }
  // cone kernel (:240-254)
  float gamma = (float)half;
  t->flat_k.assign(t->npix, 0.0f);
  for (int i = 0; i < n; ++i)
    for (int j = 0; j < n; ++j) {
      float v = gamma + 1.0f -
                sqrtf((gamma - (float)i) * (gamma - (float)i) + (gamma - (float)j) * (gamma - (float)j));
      t->flat_k[i * n + j] = fmaxf(0.0f, v);
    }
  float s = 0.0f;
  for (float v : t->flat_k) s += v;
  for (float& v : t->flat_k) v = v / s;
}

void rochade_refine(const float* img, int width, int height,
                    const std::vector<std::pair<float, float>>& initial, int half,
                    std::vector<Saddle>* out) {
  RochadeTables T;
  build_rochade_tables(half, &T);
  const int ks = T.ksize, np = T.npix, half2 = half * 2;
  std::vector<float> smooth(np);
  for (auto& ic : initial) {
    const float ix = ic.first, iy = ic.second;
    int round_x = sat_i32(roundf(ix));
    int round_y = sat_i32(roundf(iy));
    if (round_y - half2 < 0 || round_y + half2 >= height || round_x - half2 < 0 ||
        round_x + half2 >= width)
      continue;  // :268-274
    size_t start_x = (size_t)(round_x - half2), start_y = (size_t)(round_y - half2);
    for (int r = 0; r < ks; ++r)
      for (int c = 0; c < ks; ++c) {  // :280-317, same accumulation order in both branches
        float conv_p = 0.0f;
        int k_idx = 0;
        for (int pr = 0; pr < ks; ++pr) {
          const float* rp = img + (start_y + r + pr) * (size_t)width + start_x + c;
          for (int pc = 0; pc < ks; ++pc) {
            conv_p += rp[pc] * T.flat_k[k_idx];
            ++k_idx;
          }
        }
        smooth[r * ks + c] = conv_p;
      }
    float params[6];
    for (int j = 0; j < 6; ++j) {  // :321-328
      float sum = 0.0f;
      const float* col = &T.p_mat[(size_t)j * np];
      for (int i = 0; i < np; ++i) sum += col[i] * smooth[i];
      params[j] = sum;
    }
    float a1 = params[0], a2 = params[1], a3 = params[2], a4 = params[3], a5 = params[4];
    float fxx = 2.0f * a1, fyy = 2.0f * a3, fxy = a2;
    float d = fxx * fyy - fxy * fxy;
    if (d < 0.0f) {
      float x0, y0;
      find_xy(2.0f * a1, a2, a4, a2, 2.0f * a3, a5, &x0, &y0);
      if (fabsf(x0) <= 1.0f && fabsf(y0) <= 1.0f) {
        float c5 = (a1 + a3) / 2.0f;
        float c4 = (a1 - a3) / 2.0f;
        float c3 = a2 / 2.0f;
        float k = sqrtf(c4 * c4 + c3 * c3);
        if (fabsf(c5) < k) {
          float phi = acosf(-c5 / k) / 2.0f / kPi * 180.0f;
          float theta = atan2f(c3, c4) / 2.0f / kPi * 180.0f;
          out->push_back({roundf(ix) + x0, roundf(iy) + y0, k, theta, phi});
        }
      }
    }
  }
}

// a-8  filter -- src/detector.rs:432-445
void filter_saddles(const std::vector<Saddle>& in, const Params& prm, std::vector<Saddle>* out) {
  out->clear();
  if (in.empty()) return;
  float mk = -3.40282347e+38f;  // f32::MIN
  for (auto& s : in) mk = fmaxf(mk, s.k);
  mk = mk / 10.0f;
  for (auto& s : in)
    if (s.k >= mk && s.phi >= prm.min_saddle_angle && s.phi <= prm.max_saddle_angle)
      out->push_back(s);
}

// Dense front end with every intermediate kept (stage taps for the parity tests).
struct FrontEnd {
  std::vector<float> luma, blur, resp;
  float min_resp = 0, thr = 0;
  std::vector<Cluster> clusters;
  std::vector<std::pair<float, float>> centers;
  std::vector<Saddle> raw, refined;
};

// Wall time per stage, summed over all calling threads (benchmark bookkeeping only; bench.py prints
// it so the CPU number can be checked against the reference's own bench, benches/bench_detection.rs).
// 0 gray + blur + Hessian + min, 1 clusters + refinement + filter, 2 board search, 3 decode + map
std::atomic<long long> g_stage_ns[4];
std::atomic<long long> g_stage_frames;
struct StageTimer {
  int stage;
  std::chrono::steady_clock::time_point t0;
  explicit StageTimer(int s) : stage(s), t0(std::chrono::steady_clock::now()) {}
  ~StageTimer() {
    g_stage_ns[stage] += std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t0).count();
  }
};

void refined_saddle_points(const void* pixels, int w, int h, size_t stride, int fmt,
                           const Params& prm, FrontEnd* fe, bool keep_resp) {  // detector.rs:408
  size_t n = (size_t)w * h;
  StageTimer* tm = new StageTimer(0);
  fe->luma.resize(n);
  fe->blur.resize(n);
  fe->resp.resize(n);
  to_luma_f32(pixels, w, h, stride, fmt, fe->luma.data());
  gaussian_blur(fe->luma.data(), w, h, 1.5f, fe->blur.data());
  hessian_response(fe->blur.data(), w, h, fe->resp.data());
  fe->min_resp = min_response(fe->resp.data(), n);
  fe->thr = fe->min_resp * 0.05f;
  delete tm;
  StageTimer tm1(1);
  fe->clusters.clear();
  if (keep_resp) {
    std::vector<float> work(fe->resp);
    init_saddle_clusters(work.data(), w, h, fe->thr, &fe->clusters);
  } else {
    init_saddle_clusters(fe->resp.data(), w, h, fe->thr, &fe->clusters);
  }
  cluster_centers(fe->clusters, &fe->centers);
  fe->raw.clear();
  rochade_refine(fe->blur.data(), w, h, fe->centers, 2, &fe->raw);
  filter_saddles(fe->raw, prm, &fe->refined);
}

// ---------------------------------------------------------------------------------
// a-9  is_valid_quad -- src/saddle.rs:17-67
// ---------------------------------------------------------------------------------
bool is_valid_quad(const Saddle& s0, const Saddle& d0, const Saddle& s1, const Saddle& d1) {
  if (theta_distance_degree(d0.theta, d1.theta) > 5.0f) return false;
  float v01x = d0.x - s0.x, v01y = d0.y - s0.y;
  float v03x = d1.x - s0.x, v03y = d1.y - s0.y;
  float v02x = s1.x - s0.x, v02y = s1.y - s0.y;
  float s0_theta = s0.theta / 180.0f * kPi;
  float vtx = cosf(s0_theta), vty = sinf(s0_theta);
  float angle = fabsf(angle_degree(v02x, v02y, vtx, vty));
  if (!(angle >= 60.0f && angle <= 120.0f)) return false;
  float c0 = cross2(v01x, v01y, v02x, v02y);
  float c1 = cross2(v02x, v02y, v03x, v03y);
  if (c0 * c1 < 0.0f) return false;
  float v12x = s1.x - d0.x, v12y = s1.y - d0.y;
  float v23x = d1.x - s1.x, v23y = d1.y - s1.y;
  float c01 = cross2(v01x, v01y, v12x, v12y);
  float c12 = cross2(v12x, v12y, v23x, v23y);
  if (c01 * c12 < 0.0f) return false;
  float v30x = s0.x - d1.x, v30y = s0.y - d1.y;
  float a0 = angle_degree(v01x, v01y, v12x, v12y);
  float a1 = angle_degree(v12x, v12y, v23x, v23y);
  float a2 = angle_degree(v23x, v23y, v30x, v30y);
  float a3 = angle_degree(v30x, v30y, v01x, v01y);
  if (fabsf(a0 - a2) > 10.0f || fabsf(a1 - a3) > 10.0f) return false;
  if (dot2(v01x, v01y, v02x, v02y) < 0.0f || dot2(v03x, v03y, v02x, v02y) < 0.0f) return false;
  return true;
}

// ---------------------------------------------------------------------------------
// kdtree 0.8.0 `nearest(point, k, squared_euclidean)` (third-party, unpinned): the k closest
// points in ascending squared distance.  Restated as exact brute force; equal distances are
// ordered by ascending index.  squared_euclidean folds (a-b)^2 over the two axes from 0.
// ---------------------------------------------------------------------------------
struct Neighbour {
  float d2;
  int idx;
};
// The reference answers these queries with a k-d tree in O(log n); a linear scan per query would
// make the CPU baseline slower than the crate it stands for.  PointIndex therefore keeps the
// points in a uniform bucket grid and visits buckets in rings around the query until the k-th
// best distance is covered -- the SAME result as the linear scan (`nearest_scan`, kept as the
// definition; tests/test_oracle_pins.py compares the two on random and degenerate point sets).
struct PointIndex {
  const std::vector<Saddle>* pts;
  float x_min = 0, y_min = 0, inv = 0, side = 32.0f;
  int nx = 0, ny = 0;
  std::vector<int> start, item;

  explicit PointIndex(const std::vector<Saddle>* p) : pts(p) { build(); }

  static bool less(float da, int ia, float db, int ib) { return da < db || (da == db && ia < ib); }
  static void insert(float d2, int i, int k, std::vector<Neighbour>* out) {
    if ((int)out->size() == k && !less(d2, i, out->back().d2, out->back().idx)) return;
    int pos = (int)out->size();
    if ((int)out->size() < k) out->push_back({d2, i});
    else pos = k - 1;
    while (pos > 0 && less(d2, i, (*out)[pos - 1].d2, (*out)[pos - 1].idx)) {
      (*out)[pos] = (*out)[pos - 1];
      --pos;
    }
    (*out)[pos] = {d2, i};
  }
  // the definition: every point, ascending (d2, idx)
  void nearest_scan(float qx, float qy, int k, std::vector<Neighbour>* out) const {
    const auto& P = *pts;
    out->clear();
    for (int i = 0; i < (int)P.size(); ++i) {
      float dx = qx - P[i].x, dy = qy - P[i].y;
      insert(dx * dx + dy * dy, i, k, out);
    }
  }
  void build() {
    const auto& P = *pts;
    const int n = (int)P.size();
    bool finite = n > 0;
    float x0 = 0, x1 = 0, y0 = 0, y1 = 0;
    for (int i = 0; i < n && finite; ++i) {
      if (!(fabsf(P[i].x) < 1.0e7f) || !(fabsf(P[i].y) < 1.0e7f)) finite = false;
      if (i == 0) { x0 = x1 = P[i].x; y0 = y1 = P[i].y; }
      x0 = std::min(x0, P[i].x); x1 = std::max(x1, P[i].x);
      y0 = std::min(y0, P[i].y); y1 = std::max(y1, P[i].y);
    }
    nx = ny = 0;
    if (!finite || n < 16 || getenv("ORACLE_LINEAR_SCAN")) return;  // tiny or odd sets (or asked to): the scan
    // about two points per bucket, at most 256 x 256 buckets
    side = std::max(8.0f, sqrtf(2.0f * std::max(1.0f, (x1 - x0) * (y1 - y0)) / (float)n));
    side = std::max(side, std::max(x1 - x0, y1 - y0) / 256.0f + 1.0e-3f);
    inv = 1.0f / side;
    x_min = x0;
    y_min = y0;
    nx = (int)((x1 - x0) * inv) + 1;
    ny = (int)((y1 - y0) * inv) + 1;
    start.assign((size_t)nx * ny + 1, 0);
    item.resize(n);
    std::vector<int> cell(n);
    for (int i = 0; i < n; ++i) {
      int bx = std::min(nx - 1, std::max(0, (int)((P[i].x - x_min) * inv)));
      int by = std::min(ny - 1, std::max(0, (int)((P[i].y - y_min) * inv)));
      cell[i] = by * nx + bx;
      ++start[cell[i] + 1];
    }
    for (size_t c = 1; c < start.size(); ++c) start[c] += start[c - 1];
    std::vector<int> cur(start.begin(), start.end() - 1);
    for (int i = 0; i < n; ++i) item[cur[cell[i]]++] = i;
  }
  void nearest(float qx, float qy, int k, std::vector<Neighbour>* out) const {
    if (nx == 0 || !(fabsf(qx) < 1.0e7f) || !(fabsf(qy) < 1.0e7f)) return nearest_scan(qx, qy, k, out);
    const auto& P = *pts;
    out->clear();
    const int cx = std::min(nx - 1, std::max(0, (int)floorf((qx - x_min) * inv)));
    const int cy = std::min(ny - 1, std::max(0, (int)floorf((qy - y_min) * inv)));
    const int rings = std::max(std::max(cx, nx - 1 - cx), std::max(cy, ny - 1 - cy));
    auto bucket = [&](int bx, int by) {
      if (bx < 0 || by < 0 || bx >= nx || by >= ny) return;
      const int c = by * nx + bx;
      for (int e = start[c]; e < start[c + 1]; ++e) {
        const int i = item[e];
        float dx = qx - P[i].x, dy = qy - P[i].y;
        insert(dx * dx + dy * dy, i, k, out);
      }
    };
    for (int ring = 0; ring <= rings; ++ring) {
      if (ring == 0) {
        bucket(cx, cy);
      } else {
        for (int bx = cx - ring; bx <= cx + ring; ++bx) { bucket(bx, cy - ring); bucket(bx, cy + ring); }
        for (int by = cy - ring + 1; by <= cy + ring - 1; ++by) { bucket(cx - ring, by); bucket(cx + ring, by); }
      }
      // every point not visited yet is farther than ring * side from the query (the visited
      // buckets cover that distance around it, with a safety factor for the rounding of the bucket
      // coordinates): once the k-th best is closer, it stays
      const float covered = (float)ring * side * 0.999f;
      if ((int)out->size() == k && out->back().d2 < covered * covered) break;
    }
  }
};

typedef std::array<int, 4> Quad;

// ---------------------------------------------------------------------------------
// a-9  Board -- src/board.rs:18-235
//      found_board_idxs is a std HashMap in the reference; here an ordered map keyed (x, y).
//      That only fixes iteration order (all_tag_indexes / try_fix_missing), which the
//      reference leaves to the hasher's per-process random seed.
// ---------------------------------------------------------------------------------
struct Board {
  const std::vector<Saddle>& refined;
  std::vector<char> active;
  struct Cell {
    bool some;
    Quad q;
  };
  std::map<std::pair<int, int>, Cell> found;
  const PointIndex& tree;
  float spacing_ratio;
  uint32_t score;

  Board(const std::vector<Saddle>& r, const std::vector<char>& active_mask, const Quad& quad,
        float spacing, const PointIndex& t)
      : refined(r), active(active_mask), tree(t), spacing_ratio(spacing), score(1) {  // :27-48
    for (int i = 1; i < 4; ++i) active[quad[i]] = 0;
    found[{0, 0}] = {true, quad};
    try_expand(0, 0);
  }

  void all_tag_indexes(std::vector<Quad>* out) const {  // :49-51
    out->clear();
    for (auto& kv : found)
      if (kv.second.some) out->push_back(kv.second.q);
  }

  void find_closest(const Saddle& s0, const Saddle& s1, int out0[3], int* n0, int out1[3],
                    int* n1) const {  // :177-234
    float ratio0 = 1.0f + spacing_ratio;
    float dx = s0.x - s1.x, dy = s0.y - s1.y;
    float radius_sq = 0.5f * (dx * dx + dy * dy);  // glam length_squared = x*x + y*y
    const float angle_thres = 5.0f;
    float v10x = s1.x - s0.x, v10y = s1.y - s0.y;
    float nv0x = s0.x + v10x * ratio0, nv0y = s0.y + v10y * ratio0;
    float nv1x = s1.x + v10x * ratio0, nv1y = s1.y + v10y * ratio0;
    std::vector<Neighbour> nn;
    tree.nearest(nv0x, nv0y, 3, &nn);
    int c0 = 0;
    for (auto& n : nn) {
      if (n.d2 <= radius_sq && active[n.idx]) {
        if (theta_distance_degree(s0.theta, refined[n.idx].theta) < angle_thres) {
          out0[c0++] = n.idx;
          if (c0 == 3) break;
        }
      }
    }
    tree.nearest(nv1x, nv1y, 3, &nn);
    int c1 = 0;
    for (auto& n : nn) {
      if (n.d2 <= radius_sq && active[n.idx]) {
        if (theta_distance_degree(s1.theta, refined[n.idx].theta) < angle_thres) {
          out1[c1++] = n.idx;
          if (c1 == 3) break;
        }
      }
    }
    *n0 = c0;
    *n1 = c1;
  }

  bool try_expand_one(const Quad& q, Quad* out) const {  // :153-176
    const Saddle &s0 = refined[q[0]], &s1 = refined[q[1]], &s2 = refined[q[2]], &s3 = refined[q[3]];
    int a0[3], a1[3], a2[3], a3[3], n0, n1, n2, n3;
    find_closest(s0, s1, a0, &n0, a1, &n1);
    find_closest(s3, s2, a3, &n3, a2, &n2);
    for (int i0 = 0; i0 < n0; ++i0)
      for (int i1 = 0; i1 < n1; ++i1)
        for (int i2 = 0; i2 < n2; ++i2)
          for (int i3 = 0; i3 < n3; ++i3)
            if (is_valid_quad(refined[a0[i0]], refined[a1[i1]], refined[a2[i2]], refined[a3[i3]])) {
              *out = {a0[i0], a1[i1], a2[i2], a3[i3]};
              return true;
            }
    return false;
  }

  void try_expand(int bx, int by) {  // :114-152
    Cell start = found[{bx, by}];
    if (!start.some) return;
    for (int i = 0; i < 4; ++i) {
      Quad qs;
      for (int j = 0; j < 4; ++j) qs[j] = start.q[(j + i) % 4];  // rotate_left(i)
      int nx = bx, ny = by;
      switch (i) {
        case 0: nx = bx + 1; break;
        case 1: ny = by - 1; break;
        case 2: nx = bx - 1; break;
        case 3: ny = by + 1; break;
      }
      auto it = found.find({nx, ny});
      if (it != found.end() && it->second.some) continue;
      Quad nq;
      if (try_expand_one(qs, &nq)) {
        Quad v;
        for (int j = 0; j < 4; ++j) v[(j + i) % 4] = nq[j];  // rotate_right(i)
        for (int j = 0; j < 4; ++j) active[v[j]] = 0;
        score += 1;
        found[{nx, ny}] = {true, v};
        try_expand(nx, ny);
      } else {
        found[{nx, ny}] = {false, Quad{0, 0, 0, 0}};
      }
    }
  }

  void try_fix_missing() {  // :52-112
    std::vector<std::pair<std::pair<int, int>, std::pair<int, int>>> fix_list;
    auto has = [&](std::pair<int, int> b) { return found.find(b) != found.end(); };
    auto some = [&](std::pair<int, int> b) { return found.find(b)->second.some; };
    for (auto& kv : found) {
      if (kv.second.some) continue;
      int x = kv.first.first, y = kv.first.second;
      std::pair<int, int> b0{x + 1, y}, b1{x - 1, y}, b2{x, y + 1}, b3{x, y - 1};
      if (has(b0) && has(b1)) {
        if (some(b0) && some(b1)) fix_list.push_back({b0, b1});
      } else if (has(b2) && has(b3) && some(b2) && some(b3)) {
        fix_list.push_back({b2, b3});
      }
    }
    std::vector<Neighbour> nn;
    for (auto& f : fix_list) {
      Quad q0 = found[f.first].q, q1 = found[f.second].q;
      int sidx[4];
      for (int i = 0; i < 4; ++i) {
        float x = (refined[q0[i]].x + refined[q1[i]].x) / 2.0f;
        float y = (refined[q0[i]].y + refined[q1[i]].y) / 2.0f;
        tree.nearest(x, y, 1, &nn);
        sidx[i] = nn[0].idx;
      }
      if (is_valid_quad(refined[sidx[0]], refined[sidx[1]], refined[sidx[2]], refined[sidx[3]])) {
        std::pair<int, int> b{(f.first.first + f.second.first) / 2,
                              (f.first.second + f.second.second) / 2};
        found[b] = {true, Quad{sidx[0], sidx[1], sidx[2], sidx[3]}};
      }
    }
  }
};

// a-9  init_quads -- src/detector.rs:543-586
void init_quads(const std::vector<Saddle>& refined, int s0_idx, const PointIndex& tree,
                std::vector<Quad>* out) {
  out->clear();
  const Saddle& s0 = refined[s0_idx];
  std::vector<Neighbour> nn;
  tree.nearest(s0.x, s0.y, 50, &nn);
  std::vector<int> same, diff;
  for (size_t i = 1; i < nn.size(); ++i) {
    int si = nn[i].idx;
    float td = theta_distance_degree(s0.theta, refined[si].theta);
    if (td < 5.0f) same.push_back(si);
    else if (td > 80.0f) diff.push_back(si);
  }
  for (int s1_idx : same) {
    const Saddle& s1 = refined[s1_idx];
    for (size_t a = 0; a < diff.size(); ++a)
      for (size_t b = a + 1; b < diff.size(); ++b) {  // itertools combinations(2)
        const Saddle &d0 = refined[diff[a]], &d1 = refined[diff[b]];
        if (!is_valid_quad(s0, d0, s1, d1)) continue;
        float c0 = cross2(d0.x - s0.x, d0.y - s0.y, s1.x - s0.x, s1.y - s0.y);
        if (c0 > 0.0f) out->push_back(Quad{s0_idx, diff[a], s1_idx, diff[b]});
        else out->push_back(Quad{s0_idx, diff[b], s1_idx, diff[a]});
      }
  }
}

// a-9  try_find_best_board -- src/detector.rs:588-639
//      Seeds are the members of the most populated round(theta) bin.  The reference breaks
//      ties between equally populated bins by HashMap iteration order (random per process);
//      here: stable sort over ascending angle, last wins => the largest angle among ties.
bool try_find_best_board(const std::vector<Saddle>& refined, std::vector<Quad>* tags) {
  tags->clear();
  if (refined.empty()) return false;
  PointIndex tree(&refined);
  std::vector<char> active_mask(refined.size(), 1);
  std::map<int, std::vector<int>> hm;
  for (int i = 0; i < (int)refined.size(); ++i) hm[sat_i32(roundf(refined[i].theta))].push_back(i);
  const std::vector<int>* best_bin = nullptr;
  for (auto& kv : hm)
    if (!best_bin || kv.second.size() >= best_bin->size()) best_bin = &kv.second;
  std::vector<int> s0_idxs = *best_bin;
  uint32_t best_score = 0;
  Board* best = nullptr;
  int count = 0;
  std::vector<Quad> quads;
  while (!s0_idxs.empty() && count < 30) {
    int s0 = s0_idxs.back();
    s0_idxs.pop_back();
    init_quads(refined, s0, tree, &quads);
    for (auto& q : quads) {
      Board* b = new Board(refined, active_mask, q, 0.3f, tree);
      if (b->score > best_score) {
        best_score = b->score;
        delete best;
        best = b;
      } else {
        delete b;
      }
    }
    if (best_score >= 36) break;
    ++count;
  }
  if (!best) return false;
  best->try_fix_missing();
  best->all_tag_indexes(tags);
  delete best;
  return true;
}

// ---------------------------------------------------------------------------------
// a-10  tag_affine + decode_positions -- src/image_util.rs:39-70, src/detector.rs:42-72
//       faer's f32 QR least squares (unpinned) restated as the closed-form solution: the
//       source corners are a square, so the normal equations are diagonal after centring.
// ---------------------------------------------------------------------------------
void tag_affine(const float qx[4], const float qy[4], int side_bits, float margin, float H[6]) {
  float lo = -margin, hi = (float)side_bits - 1.0f + margin;
  const double sx[4] = {lo, lo, hi, hi};
  const double sy[4] = {lo, hi, hi, lo};
  double mx = 0, my = 0, mcx = 0, mcy = 0;
  for (int p = 0; p < 4; ++p) {
    mx += sx[p]; my += sy[p]; mcx += qx[p]; mcy += qy[p];
  }
  mx /= 4; my /= 4; mcx /= 4; mcy /= 4;
  double sxx = 0, syy = 0, axx = 0, axy = 0, ayx = 0, ayy = 0;
  for (int p = 0; p < 4; ++p) {
    double dx = sx[p] - mx, dy = sy[p] - my;
    sxx += dx * dx; syy += dy * dy;
    axx += dx * qx[p]; axy += dy * qx[p];
    ayx += dx * qy[p]; ayy += dy * qy[p];
  }
  double h0 = axx / sxx, h1 = axy / syy, h3 = ayx / sxx, h4 = ayy / syy;
  double h2 = mcx - h0 * mx - h1 * my, h5 = mcy - h3 * mx - h4 * my;
  H[0] = (float)h0; H[1] = (float)h1; H[2] = (float)h2;
  H[3] = (float)h3; H[4] = (float)h4; H[5] = (float)h5;
}

bool decode_positions(uint32_t img_w, uint32_t img_h, const float qx[4], const float qy[4],
                      int border, int edge, float margin, float* px, float* py) {
  for (int p = 0; p < 4; ++p) {
    uint32_t x = sat_u32(roundf(qx[p])), y = sat_u32(roundf(qy[p]));
    if (x >= img_w || y >= img_h) return false;
  }
  float H[6];
  tag_affine(qx, qy, border * 2 + edge, margin, H);
  int n = 0;
  for (int x = border; x < border + edge; ++x)
    for (int y = border; y < border + edge; ++y, ++n) {
      float fx = (float)x, fy = (float)y;
      px[n] = H[0] * fx + H[1] * fy + H[2];
      py[n] = H[3] * fx + H[4] * fy + H[5];
    }
  return true;
}

// a-11  bit_code -- src/detector.rs:74-122
bool bit_code(const uint8_t* img, uint32_t w, uint32_t h, const float* px, const float* py, int n,
              uint8_t valid_brightness_threshold, uint32_t max_invalid_bit, uint64_t* bits_out) {
  uint8_t b[64];
  for (int i = 0; i < n; ++i) {
    uint32_t x = sat_u32(roundf(px[i])), y = sat_u32(roundf(py[i]));
    if (x >= w || y >= h) return false;
    b[i] = img[(size_t)y * w + x];
  }
  int min_b = 255, max_b = 0;
  for (int i = 0; i < n; ++i) {
    min_b = std::min(min_b, (int)b[i]);
    max_b = std::max(max_b, (int)b[i]);
  }
  if (max_b - min_b < 50) return false;
  int mid_b = (int)sat_u32(roundf(((float)min_b + (float)max_b) / 2.0f));
  uint64_t bits = 0;
  uint32_t invalid = 0;
  for (int i = 0; i < n; ++i) {  // iter().rev().enumerate(): last sample is bit 0
    int v = b[n - 1 - i];
    if (abs(mid_b - v) < (int)valid_brightness_threshold) ++invalid;
    if (v > mid_b) bits |= (1ull << i);
  }
  if (invalid > max_invalid_bit) return false;
  *bits_out = bits;
  return true;
}

// a-12  rotate_bits / best_tag -- src/detector.rs:124-169
uint64_t rotate_bits(uint64_t bits, int edge) {
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

bool best_tag(uint64_t bits, int thres, const uint64_t* fam, int nfam, int edge, int* id, int* rot) {
  for (int rotated = 0; rotated < 4; ++rotated) {
    int best_idx = 0;
    uint32_t best_score = (uint32_t)__builtin_popcountll(fam[0] ^ bits);
    for (int i = 1; i < nfam; ++i) {
      uint32_t s = (uint32_t)__builtin_popcountll(fam[i] ^ bits);
      if (s < best_score) {
        best_score = s;
        best_idx = i;
      }
    }
    if (best_score < (uint32_t)thres) {
      *id = best_idx;
      *rot = rotated;
      return true;
    } else if (rotated == 3) {
      break;
    }
    bits = rotate_bits(bits, edge);
  }
  return false;
}

struct TagOut {  // mirrors ag_tag of include/aprilgrid_b200.h
  uint32_t id;
  float xy[8];
};

// a-13  try_decode_quad -- src/detector.rs:448-476
bool try_decode_quad(const Family& fam, const uint8_t* grey, uint32_t w, uint32_t h,
                     const float qx[4], const float qy[4], TagOut* out) {
  float px[64], py[64];
  if (!decode_positions(w, h, qx, qy, fam.border, fam.edge, 0.5f, px, py)) return false;
  uint64_t bits;
  if (!bit_code(grey, w, h, px, py, fam.edge * fam.edge, 10, 3, &bits)) return false;
  int id, rot;
  if (!best_tag(bits, fam.hamming, fam.codes, fam.n_codes, fam.edge, &id, &rot)) return false;
  out->id = (uint32_t)id;
  // rotate_left(rot) then reverse()
  for (int j = 0; j < 4; ++j) {
    int src = ((3 - j) + rot) % 4;
    out->xy[2 * j] = qx[src];
    out->xy[2 * j + 1] = qy[src];
  }
  return true;
}

// a-14  board rounds of detect -- src/detector.rs:511-536: `max_num_of_boards` rounds of board
//       search + decoding on the refined saddle list and the Luma<u8> plane `grey` (w x h, packed).
//       The result map is returned in ascending id order.  Quads of one board are visited in
//       Board::all_tag_indexes order (see Board); a repeated id overwrites, as HashMap::insert does.
int detect_from_saddles(const Family& fam, int max_boards, std::vector<Saddle> refined, const uint8_t* grey,
                        int w, int h, TagOut* out, int cap) {
  std::map<uint32_t, TagOut> detected;
  std::vector<Quad> quads;
  for (int b = 0; b < max_boards; ++b) {
    {
      StageTimer tm(2);
      if (!try_find_best_board(refined, &quads)) continue;
    }
    StageTimer tm(3);
    std::vector<char> remove(refined.size(), 0);
    for (auto& q : quads) {
      float qx[4], qy[4];
      for (int j = 0; j < 4; ++j) {
        qx[j] = refined[q[j]].x;
        qy[j] = refined[q[j]].y;
      }
      TagOut t;
      if (try_decode_quad(fam, grey, (uint32_t)w, (uint32_t)h, qx, qy, &t)) {
        detected[t.id] = t;
        for (int j = 0; j < 4; ++j) remove[q[j]] = 1;
      }
    }
    std::vector<Saddle> kept;
    for (size_t i = 0; i < refined.size(); ++i)
      if (!remove[i]) kept.push_back(refined[i]);
    refined.swap(kept);
  }
  int n = 0;
  for (auto& kv : detected) {
    if (n < cap) out[n] = kv.second;
    ++n;
  }
  return n;
}

// a-14  detect -- src/detector.rs:505-540: the gray planes, refined_saddle_points, then the rounds.
// grey_plane: null = to_luma8 of `pixels` (detector.rs:507); else the Luma<u8> plane itself, `pixels`
// then being the Luma<f32> plane (fmt 3): the frame as its two derived gray images (detect_planes).
int detect(const Family& fam, const Params& prm, const void* pixels, int w, int h, size_t stride,
           int fmt, TagOut* out, int cap, const uint8_t* grey_plane = nullptr, size_t grey_stride = 0) {
  std::vector<uint8_t> grey((size_t)w * h);
  {
    StageTimer tm(0);
    if (grey_plane) to_luma_u8(grey_plane, w, h, grey_stride ? grey_stride : (size_t)w, 0, grey.data());
    else to_luma_u8(pixels, w, h, stride, fmt, grey.data());
  }
  ++g_stage_frames;
  FrontEnd fe;
  refined_saddle_points(pixels, w, h, stride, fmt, prm, &fe, false);
  return detect_from_saddles(fam, prm.max_num_of_boards, fe.refined, grey.data(), w, h, out, cap);
}

}  // namespace

// =====================================================================================
// C entry points for the Python test harness (ctypes).  Names are orc_*.
// =====================================================================================
extern "C" {

// Test hook: the bucket-grid index against the linear scan for n points / queries drawn from a
// seeded generator (mode 0 uniform, 1 clustered with exact duplicates, 2 collinear).  Returns the
// number of queries whose (d2, idx) lists differ.
int orc_selftest_point_index(int n, int n_queries, int k, int mode, unsigned seed) {
  std::vector<Saddle> pts(n);
  unsigned s = seed * 2654435761u + 12345u;
  auto rnd = [&]() { s = s * 1664525u + 1013904223u; return (float)(s >> 8) / 16777216.0f; };
  for (int i = 0; i < n; ++i) {
    Saddle p{};
    if (mode == 1) { int c = (int)(rnd() * 7.0f); p.x = 100.0f + 150.0f * c + floorf(rnd() * 12.0f); p.y = 300.0f + floorf(rnd() * 12.0f) * 3.0f; }
    else if (mode == 2) { p.x = floorf(rnd() * 900.0f); p.y = 77.0f; }
    else { p.x = rnd() * 1280.0f; p.y = rnd() * 1024.0f; }
    pts[i] = p;
  }
  PointIndex idx(&pts);
  std::vector<Neighbour> a, b;
  int bad = 0;
  for (int q = 0; q < n_queries; ++q) {
    float qx = rnd() * 1600.0f - 160.0f, qy = rnd() * 1300.0f - 130.0f;
    if (q % 5 == 0 && n > 0) { qx = pts[q % n].x; qy = pts[q % n].y; }  // on a point: exact ties
    idx.nearest(qx, qy, k, &a);
    idx.nearest_scan(qx, qy, k, &b);
    bool same = a.size() == b.size();
    for (size_t i = 0; same && i < a.size(); ++i) same = a[i].idx == b[i].idx && a[i].d2 == b[i].d2;
    if (!same) ++bad;
  }
  return bad;
}


void orc_to_luma_f32(const void* px, int w, int h, size_t stride, int fmt, float* out) {
  to_luma_f32(px, w, h, stride, fmt, out);
}
void orc_to_luma_u8(const void* px, int w, int h, size_t stride, int fmt, uint8_t* out) {
  to_luma_u8(px, w, h, stride, fmt, out);
}
int orc_blur_taps(float sigma, float* taps, int cap) {
  std::vector<float> k;
  int radius;
  blur_taps(sigma, &k, &radius);
  for (int i = 0; i < (int)k.size() && i < cap; ++i) taps[i] = k[i];
  return (int)k.size();
}
void orc_gaussian_blur(const float* img, int w, int h, float sigma, float* out) {
  gaussian_blur(img, w, h, sigma, out);
}
void orc_hessian_response(const float* img, int w, int h, float* out) {
  hessian_response(img, w, h, out);
}
float orc_min_response(const float* resp, size_t n) { return min_response(resp, n); }

// pixel_bfs on a caller-owned matrix (mutated as the reference does); returns pixel count.
int orc_pixel_bfs(float* mat, int w, int h, int x, int y, float thr, uint32_t* xy_out, int cap) {
  Cluster c;
  std::vector<std::pair<uint32_t, uint32_t>> st;
  pixel_bfs(mat, (uint32_t)w, (uint32_t)h, &c, (uint32_t)x, (uint32_t)y, thr, &st);
  for (int i = 0; i < (int)c.size() && i < cap; ++i) {
    xy_out[2 * i] = c[i].first;
    xy_out[2 * i + 1] = c[i].second;
  }
  return (int)c.size();
}

// labels[i] = cluster id (reference order) or -1; centers = (cx, cy) per cluster.
int orc_clusters(const float* resp, int w, int h, float thr, int32_t* labels, float* centers,
                 int32_t* sizes, int cap) {
  std::vector<float> work(resp, resp + (size_t)w * h);
  std::vector<Cluster> cl;
  init_saddle_clusters(work.data(), w, h, thr, &cl);
  std::vector<std::pair<float, float>> ctr;
  cluster_centers(cl, &ctr);
  if (labels) {
    for (size_t i = 0; i < (size_t)w * h; ++i) labels[i] = -1;
    for (size_t c = 0; c < cl.size(); ++c)
      for (auto& p : cl[c]) labels[(size_t)p.second * w + p.first] = (int32_t)c;
  }
  for (size_t c = 0; c < cl.size() && (int)c < cap; ++c) {
    if (centers) {
      centers[2 * c] = ctr[c].first;
      centers[2 * c + 1] = ctr[c].second;
    }
    if (sizes) sizes[c] = (int32_t)cl[c].size();
  }
  return (int)cl.size();
}

void orc_find_xy(float a0, float b0, float c0, float a1, float b1, float c1, float* xy) {
  find_xy(a0, b0, c0, a1, b1, c1, &xy[0], &xy[1]);
}
float orc_theta_distance_degree(float a, float b) { return theta_distance_degree(a, b); }
float orc_cross(float ax, float ay, float bx, float by) { return cross2(ax, ay, bx, by); }
float orc_dot(float ax, float ay, float bx, float by) { return dot2(ax, ay, bx, by); }
float orc_angle_degree(float ax, float ay, float bx, float by) { return angle_degree(ax, ay, bx, by); }
int orc_is_valid_quad(const float* s) {  // 4 saddles x {x, y, k, theta, phi}
  const Saddle* p = (const Saddle*)s;
  return is_valid_quad(p[0], p[1], p[2], p[3]) ? 1 : 0;
}

void orc_rochade_tables(int half, float* p_mat, float* flat_k) {
  RochadeTables T;
  build_rochade_tables(half, &T);
  memcpy(p_mat, T.p_mat.data(), sizeof(float) * T.p_mat.size());
  memcpy(flat_k, T.flat_k.data(), sizeof(float) * T.flat_k.size());
}

int orc_rochade_refine(const float* img, int w, int h, const float* centers, int n, int half,
                       float* saddles_out, int cap) {
  std::vector<std::pair<float, float>> c(n);
  for (int i = 0; i < n; ++i) c[i] = {centers[2 * i], centers[2 * i + 1]};
  std::vector<Saddle> out;
  rochade_refine(img, w, h, c, half, &out);
  for (int i = 0; i < (int)out.size() && i < cap; ++i) memcpy(saddles_out + 5 * i, &out[i], 20);
  return (int)out.size();
}

// Full front end with taps.  Any output pointer may be NULL.  Returns refined count.
int orc_front_end(const void* px, int w, int h, size_t stride, int fmt, float min_angle,
                  float max_angle, float* blur, float* resp, float* min_thr /*[2]*/,
                  int32_t* labels, float* centers, int* n_clusters, int centers_cap,
                  float* raw_saddles, int* n_raw, float* refined, int saddle_cap) {
  Params prm;
  prm.min_saddle_angle = min_angle;
  prm.max_saddle_angle = max_angle;
  FrontEnd fe;
  refined_saddle_points(px, w, h, stride, fmt, prm, &fe, true);
  size_t n = (size_t)w * h;
  if (blur) memcpy(blur, fe.blur.data(), n * 4);
  if (resp) memcpy(resp, fe.resp.data(), n * 4);
  if (min_thr) {
    min_thr[0] = fe.min_resp;
    min_thr[1] = fe.thr;
  }
  if (labels) {
    for (size_t i = 0; i < n; ++i) labels[i] = -1;
    for (size_t c = 0; c < fe.clusters.size(); ++c)
      for (auto& p : fe.clusters[c]) labels[(size_t)p.second * w + p.first] = (int32_t)c;
  }
  if (n_clusters) *n_clusters = (int)fe.clusters.size();
  if (centers)
    for (int i = 0; i < (int)fe.centers.size() && i < centers_cap; ++i) {
      centers[2 * i] = fe.centers[i].first;
      centers[2 * i + 1] = fe.centers[i].second;
    }
  if (n_raw) *n_raw = (int)fe.raw.size();
  if (raw_saddles)
    for (int i = 0; i < (int)fe.raw.size() && i < saddle_cap; ++i)
      memcpy(raw_saddles + 5 * i, &fe.raw[i], 20);
  if (refined)
    for (int i = 0; i < (int)fe.refined.size() && i < saddle_cap; ++i)
      memcpy(refined + 5 * i, &fe.refined[i], 20);
  return (int)fe.refined.size();
}

// try_find_best_board on a caller-supplied saddle list; returns number of quads or -1 (None).
int orc_try_find_best_board(const float* saddles, int n, int32_t* quads_out, int cap) {
  std::vector<Saddle> s(n);
  if (n) memcpy(s.data(), saddles, (size_t)n * 20);
  std::vector<Quad> q;
  if (!try_find_best_board(s, &q)) return -1;
  for (int i = 0; i < (int)q.size() && i < cap; ++i)
    for (int j = 0; j < 4; ++j) quads_out[4 * i + j] = q[i][j];
  return (int)q.size();
}

int orc_init_quads(const float* saddles, int n, int s0_idx, int32_t* quads_out, int cap) {
  std::vector<Saddle> s(n);
  if (n) memcpy(s.data(), saddles, (size_t)n * 20);
  PointIndex tree(&s);
  std::vector<Quad> q;
  init_quads(s, s0_idx, tree, &q);
  for (int i = 0; i < (int)q.size() && i < cap; ++i)
    for (int j = 0; j < 4; ++j) quads_out[4 * i + j] = q[i][j];
  return (int)q.size();
}

void orc_tag_affine(const float* quad_xy, int side_bits, float margin, float* H9) {
  float qx[4], qy[4], H[6];
  for (int i = 0; i < 4; ++i) {
    qx[i] = quad_xy[2 * i];
    qy[i] = quad_xy[2 * i + 1];
  }
  tag_affine(qx, qy, side_bits, margin, H);
  for (int i = 0; i < 6; ++i) H9[i] = H[i];
  H9[6] = 0.0f;
  H9[7] = 0.0f;
  H9[8] = 1.0f;
}

int orc_decode_positions(uint32_t w, uint32_t h, const float* quad_xy, int border, int edge,
                         float margin, float* pts_out) {
  float qx[4], qy[4], px[64], py[64];
  for (int i = 0; i < 4; ++i) {
    qx[i] = quad_xy[2 * i];
    qy[i] = quad_xy[2 * i + 1];
  }
  if (!decode_positions(w, h, qx, qy, border, edge, margin, px, py)) return 0;
  for (int i = 0; i < edge * edge; ++i) {
    pts_out[2 * i] = px[i];
    pts_out[2 * i + 1] = py[i];
  }
  return 1;
}

int orc_bit_code(const uint8_t* img, uint32_t w, uint32_t h, const float* pts, int n, int vbt,
                 int max_invalid, uint64_t* bits) {
  float px[64], py[64];
  for (int i = 0; i < n; ++i) {
    px[i] = pts[2 * i];
    py[i] = pts[2 * i + 1];
  }
  return bit_code(img, w, h, px, py, n, (uint8_t)vbt, (uint32_t)max_invalid, bits) ? 1 : 0;
}

uint64_t orc_rotate_bits(uint64_t bits, int edge) { return rotate_bits(bits, edge); }

int orc_best_tag(uint64_t bits, int thres, int family, int* id, int* rot) {
  Family f;
  if (!family_by_id(family, &f)) return 0;
  return best_tag(bits, thres, f.codes, f.n_codes, f.edge, id, rot) ? 1 : 0;
}

int orc_family_info(int family, int* edge, int* border, int* hamming, int* n_codes,
                    const uint64_t** codes) {
  Family f;
  if (!family_by_id(family, &f)) return 0;
  *edge = f.edge; *border = f.border; *hamming = f.hamming; *n_codes = f.n_codes;
  if (codes) *codes = f.codes;
  return 1;
}

// Per-stage wall time (ms, summed over threads) and frames since the last reset.
void orc_stage_times(double* ms_out, long long* frames_out, int reset) {
  for (int i = 0; i < 4; ++i) {
    ms_out[i] = (double)g_stage_ns[i].load() * 1.0e-6;
    if (reset) g_stage_ns[i] = 0;
  }
  *frames_out = g_stage_frames.load();
  if (reset) g_stage_frames = 0;
}

// TagDetector::detect.  Returns the number of tags (may exceed cap; only cap are written).
int orc_detect(int family, float min_angle, float max_angle, int max_boards, const void* px, int w,
               int h, size_t stride, int fmt, void* tags_out, int cap) {
  Family f;
  if (!family_by_id(family, &f)) return -1;
  Params prm;
  prm.min_saddle_angle = min_angle;
  prm.max_saddle_angle = max_angle;
  prm.max_num_of_boards = max_boards;
  return detect(f, prm, px, w, h, stride, fmt, (TagOut*)tags_out, cap);
}

// The board rounds of detect on a caller-supplied refined saddle list (n x {x, y, k, theta, phi})
// over the frame `pixels` (L8 / L16 / RGB8, converted with to_luma8).  Returns the number of tags.
int orc_detect_from_saddles(int family, int max_boards, const float* saddles, int n, const void* px, int w,
                            int h, size_t stride, int fmt, void* tags_out, int cap) {
  Family f;
  if (!family_by_id(family, &f) || n < 0 || fmt < 0 || fmt > 2) return -1;
  std::vector<Saddle> s(n);
  if (n) memcpy(s.data(), saddles, (size_t)n * 20);
  std::vector<uint8_t> grey((size_t)w * h);
  to_luma_u8(px, w, h, stride, fmt, grey.data());
  return detect_from_saddles(f, max_boards, s, grey.data(), w, h, (TagOut*)tags_out, cap);
}

// detect on a frame given as its two gray planes: luma32f = to_luma32f(img), luma8 = to_luma8(img).
int orc_detect_planes(int family, float min_angle, float max_angle, int max_boards, const float* luma32f,
                      size_t f32_stride, const uint8_t* luma8, size_t u8_stride, int w, int h, void* tags_out, int cap) {
  Family f;
  if (!family_by_id(family, &f)) return -1;
  Params prm;
  prm.min_saddle_angle = min_angle;
  prm.max_saddle_angle = max_angle;
  prm.max_num_of_boards = max_boards;
  return detect(f, prm, luma32f, w, h, f32_stride ? f32_stride : sizeof(float) * (size_t)w, 3, (TagOut*)tags_out, cap, luma8,
                u8_stride);
}

// Frame-parallel batch for the CPU baseline: each frame runs the single-threaded detect()
// above on one of `threads` host threads (the reference has no threads of its own).
void orc_detect_batch(int family, float min_angle, float max_angle, int max_boards,
                      const void* frames, size_t frame_stride, int n_frames, int w, int h,
                      size_t stride, int fmt, void* tags_out, int cap_per_frame, int* n_per_frame,
                      int threads) {
  Family f;
  if (!family_by_id(family, &f)) return;
  Params prm;
  prm.min_saddle_angle = min_angle;
  prm.max_saddle_angle = max_angle;
  prm.max_num_of_boards = max_boards;
  if (threads < 1) threads = 1;
  auto work = [&](int t) {
    for (int i = t; i < n_frames; i += threads) {
      const uint8_t* p = (const uint8_t*)frames + (size_t)i * frame_stride;
      n_per_frame[i] = detect(f, prm, p, w, h, stride, fmt,
                              (TagOut*)tags_out + (size_t)i * cap_per_frame, cap_per_frame);
    }
  };
  if (threads == 1) {
    work(0);
  } else {
    std::vector<std::thread> th;
    for (int t = 0; t < threads; ++t) th.emplace_back(work, t);
    for (auto& t : th) t.join();
  }
}

}  // extern "C"
