// C++ host-side mirror of the aprilgrid-rs detector API over the C ABI (header only).
//
// The reference is a compiled Rust crate and no Rust toolchain exists in the build image, so
// this is the host side "in the reference's own shape": same type and method names, argument
// meaning and failure behaviour as aprilgrid 0.8.0 (src/detector.rs:17-41, :363-541):
//   TagDetector(TagFamily, optional<DetectorParams>)   -- infallible in Rust; throws here
//   detect(image)            -> std::unordered_map<uint32_t, std::array<std::pair<float,float>,4>>
//   detect_batch(frames...)  -> vector of such maps (new entry point)
//   refined_saddle_points(image) -> std::vector<Saddle>
#pragma once
#include <array>
#include <optional>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../include/aprilgrid_b200.h"

namespace aprilgrid {

enum class TagFamily { T16H5 = AG_T16H5, T25H7 = AG_T25H7, T25H9 = AG_T25H9, T36H11 = AG_T36H11, T36H11B1 = AG_T36H11B1 };

inline TagFamily tag_family_from_str(const std::string& s) {  // TagFamily::from_str
  int f = 0;
  if (ag_family_from_str(s.c_str(), &f) != AG_OK) throw std::invalid_argument("unknown tag family: " + s);
  return static_cast<TagFamily>(f);
}

struct DetectorParams {  // src/detector.rs:25-41
  float tag_spacing_ratio = 0.3f, min_saddle_angle = 30.0f, max_saddle_angle = 60.0f;
  uint8_t max_num_of_boards = 2;
  static DetectorParams default_params() { return {}; }
};

struct Saddle {  // src/saddle.rs:3-9
  std::pair<float, float> p;
  float k, theta, phi;
};

// A borrowed image in one of the DynamicImage variants (the AG_* pixel formats).
struct ImageView {
  const void* pixels;
  int width, height;
  size_t row_stride;  // bytes; 0 = tightly packed
  int format;         // AG_L8 .. AG_RGBA32F (include/aprilgrid_b200.h)
};

using TagMap = std::unordered_map<uint32_t, std::array<std::pair<float, float>, 4>>;

class TagDetector {
 public:
  TagDetector(TagFamily family, std::optional<DetectorParams> params = std::nullopt, int device = 0) {
    DetectorParams p = params.value_or(DetectorParams::default_params());
    ag_params cp{p.tag_spacing_ratio, p.min_saddle_angle, p.max_saddle_angle, p.max_num_of_boards};
    if (ag_create(static_cast<int>(family), &cp, device, &h_) != AG_OK)
      throw std::runtime_error(std::string("aprilgrid_b200: ") + ag_last_error(nullptr));
  }
  ~TagDetector() { ag_destroy(h_); }
  TagDetector(const TagDetector&) = delete;
  TagDetector& operator=(const TagDetector&) = delete;

  TagMap detect(const ImageView& img) const {
    std::vector<ag_tag> out(1024);
    int n = 0;
    check(ag_detect(h_, img.pixels, img.width, img.height, img.row_stride, img.format, out.data(), (int)out.size(), &n));
    return to_map(out.data(), n);
  }

  // frames: n_frames images of one shape, frame i at base + i * frame_stride
  std::vector<TagMap> detect_batch(const void* base, size_t frame_stride, int n_frames, int width, int height,
                                   size_t row_stride, int format, int cap_per_frame = 128) const {
    std::vector<ag_tag> out((size_t)n_frames * cap_per_frame);
    std::vector<int> cnt(n_frames);
    check(ag_detect_batch(h_, base, frame_stride, n_frames, width, height, row_stride, format, out.data(),
                          cap_per_frame, cnt.data(), nullptr));
    std::vector<TagMap> res(n_frames);
    for (int i = 0; i < n_frames; ++i) res[i] = to_map(out.data() + (size_t)i * cap_per_frame, cnt[i]);
    return res;
  }

  // Streaming form of detect_batch over host frames (option "host_async"): submit() returns once the
  // batch is enqueued, wait(keep_in_flight) once all but the newest keep_in_flight batches have
  // delivered; frames and the Batch object must stay alive and untouched until then.
  struct Batch {
    std::vector<ag_tag> tags;
    std::vector<int> counts;
    int cap_per_frame = 0;
    TagMap frame(int i) const { return to_map(tags.data() + (size_t)i * cap_per_frame, counts[i]); }
  };
  void set_streaming(bool on) const { check(ag_set_option(h_, "host_async", on ? 1 : 0)); }
  void submit(Batch& b, const void* base, size_t frame_stride, int n_frames, int width, int height,
              size_t row_stride, int format, int cap_per_frame = 128) const {
    b.tags.assign((size_t)n_frames * cap_per_frame, ag_tag{});
    b.counts.assign(n_frames, 0);
    b.cap_per_frame = cap_per_frame;
    check(ag_detect_batch(h_, base, frame_stride, n_frames, width, height, row_stride, format, b.tags.data(),
                          cap_per_frame, b.counts.data(), nullptr));
  }
  void wait(int keep_in_flight = 0) const { check(ag_detect_batch_wait(h_, keep_in_flight)); }

  std::vector<Saddle> refined_saddle_points(const ImageView& img) const {
    std::vector<ag_saddle> out(16384);
    int n = 0;
    check(ag_refined_saddle_points(h_, img.pixels, img.width, img.height, img.row_stride, img.format, out.data(),
                                   (int)out.size(), &n));
    std::vector<Saddle> r(n);
    for (int i = 0; i < n; ++i) r[i] = Saddle{{out[i].x, out[i].y}, out[i].k, out[i].theta, out[i].phi};
    return r;
  }

  ag_detector* handle() const { return h_; }

 private:
  void check(int rc) const {
    if (rc != AG_OK) throw std::runtime_error(std::string("aprilgrid_b200: ") + ag_last_error(h_));
  }
  static TagMap to_map(const ag_tag* t, int n) {
    TagMap m;
    for (int i = 0; i < n; ++i)
      m[t[i].id] = {{{t[i].xy[0], t[i].xy[1]}, {t[i].xy[2], t[i].xy[3]}, {t[i].xy[4], t[i].xy[5]}, {t[i].xy[6], t[i].xy[7]}}};
    return m;
  }
  ag_detector* h_ = nullptr;
};

// detect_batch over every GPU of the box (ag_multi_*): frames sharded image-wise, results in frame order.
class MultiTagDetector {
 public:
  explicit MultiTagDetector(TagFamily family, std::optional<DetectorParams> params = std::nullopt,
                            const std::vector<int>& devices = {}) {
    DetectorParams p = params.value_or(DetectorParams::default_params());
    ag_params cp{p.tag_spacing_ratio, p.min_saddle_angle, p.max_saddle_angle, p.max_num_of_boards};
    if (ag_multi_create(static_cast<int>(family), &cp, devices.empty() ? nullptr : devices.data(), (int)devices.size(),
                        &m_) != AG_OK)
      throw std::runtime_error(std::string("aprilgrid_b200: ") + ag_multi_last_error(nullptr));
  }
  ~MultiTagDetector() { ag_multi_destroy(m_); }
  MultiTagDetector(const MultiTagDetector&) = delete;
  MultiTagDetector& operator=(const MultiTagDetector&) = delete;
  int device_count() const { return ag_multi_device_count(m_); }

  std::vector<TagMap> detect_batch(const void* base, size_t frame_stride, int n_frames, int width, int height,
                                   size_t row_stride, int format, int cap_per_frame = 128) const {
    std::vector<ag_tag> out((size_t)n_frames * cap_per_frame);
    std::vector<int> cnt(n_frames);
    if (ag_multi_detect_batch(m_, base, frame_stride, n_frames, width, height, row_stride, format, out.data(),
                              cap_per_frame, cnt.data(), nullptr) != AG_OK)
      throw std::runtime_error(std::string("aprilgrid_b200: ") + ag_multi_last_error(m_));
    std::vector<TagMap> res(n_frames);
    for (int i = 0; i < n_frames; ++i) {
      TagMap m;
      const ag_tag* t = out.data() + (size_t)i * cap_per_frame;
      for (int k = 0; k < cnt[i] && k < cap_per_frame; ++k)
        m[t[k].id] = {{{t[k].xy[0], t[k].xy[1]}, {t[k].xy[2], t[k].xy[3]}, {t[k].xy[4], t[k].xy[5]}, {t[k].xy[6], t[k].xy[7]}}};
      res[i] = std::move(m);
    }
    return res;
  }

 private:
  ag_multi* m_ = nullptr;
};

}  // namespace aprilgrid
