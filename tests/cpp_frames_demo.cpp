// TEST-ONLY: exercises the frame-list methods of the C++ mirror (aprilgrid-rs_b200/cpp/aprilgrid_b200.hpp)
// end to end on a GPU: reads raw frames given as "path width height format" quadruples, runs
// TagDetector::detect_frames on the list and MultiTagDetector::detect_frames, and prints for every list
// position "frame i" followed by "id x0 y0 ... x3 y3" lines (sorted by id), then "frames same" when
// both equal TagDetector::detect of each frame alone.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "aprilgrid_b200.hpp"

int main(int argc, char** argv) {
  if (argc < 5 || (argc - 1) % 4) return 2;
  const int n = (argc - 1) / 4;
  std::vector<std::vector<unsigned char>> bufs(n);
  std::vector<aprilgrid::ImageView> views;
  static const int bpp[] = {1, 2, 3, 0, 2, 4, 4, 6, 8, 12, 16};
  for (int i = 0; i < n; ++i) {
    const int w = atoi(argv[4 * i + 2]), h = atoi(argv[4 * i + 3]), fmt = atoi(argv[4 * i + 4]);
    if (fmt < 0 || fmt > 10 || !bpp[fmt]) return 2;
    bufs[i].resize((size_t)w * h * bpp[fmt]);
    FILE* f = fopen(argv[4 * i + 1], "rb");
    if (!f || fread(bufs[i].data(), 1, bufs[i].size(), f) != bufs[i].size()) return 3;
    fclose(f);
    views.push_back({bufs[i].data(), w, h, 0, fmt});
  }
  try {
    aprilgrid::TagDetector det(aprilgrid::TagFamily::T36H11);
    const auto got = det.detect_frames(views, 256);
    aprilgrid::MultiTagDetector multi(aprilgrid::TagFamily::T36H11);
    const auto mgot = multi.detect_frames(views, 256);
    bool same = (int)got.size() == n && (int)mgot.size() == n;
    for (int i = 0; i < n; ++i) {
      const aprilgrid::TagMap one = det.detect(views[i]);
      same = same && got[i] == one && mgot[i] == one;
      printf("frame %d\n", i);
      std::vector<uint32_t> ids;
      for (auto& kv : got[i]) ids.push_back(kv.first);
      std::sort(ids.begin(), ids.end());
      for (uint32_t id : ids) {
        printf("%u", id);
        for (auto& c : got[i].at(id)) printf(" %.9g %.9g", c.first, c.second);
        printf("\n");
      }
    }
    printf("frames %s\n", same ? "same" : "DIFFERENT");
  } catch (const std::exception& e) {
    fprintf(stderr, "%s\n", e.what());
    return 1;
  }
  return 0;
}
