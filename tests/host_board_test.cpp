// TEST-ONLY host build of the product's board/decode control logic
// (aprilgrid-rs_b200/csrc/ag_board_core.h compiled with a warp of one lane).
// It lets the CPU test-suite compare that logic with the oracle without a GPU.  It is never
// linked into the shipped library and is not a CPU path of the product.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "ag_board_core.h"
#if defined(AGB_WORK_COUNTERS)
#include <set>
extern "C" { long long agb_work_counters[32] = {0}; }
static std::set<unsigned long long> g_keys[2][3];
extern "C" void agb_note_key(int kind, unsigned long long key) {
  int r = (int)agb_work_counters[31];
  agb_work_counters[24 + kind] += 1;  // total (both rounds)
  if (g_keys[r][kind].insert(key).second) agb_work_counters[27 + kind] += 1;  // distinct
}
static std::vector<float> g_queries;  // per query: round, a, b, self_is_b, qx, qy, r2
extern "C" void agb_note_query(int a, int b, int self_is_b, float qx, float qy, float r2) {
  const float rec[7] = {(float)agb_work_counters[31], (float)a, (float)b, (float)self_is_b, qx, qy, r2};
  g_queries.insert(g_queries.end(), rec, rec + 7);
}
extern "C" int agb_get_queries(float* out, int cap) {
  const int n = (int)(g_queries.size() / 7);
  for (int i = 0; i < n && i < cap; ++i) memcpy(out + 7 * i, &g_queries[7 * (size_t)i], 28);
  return n;
}
extern "C" void agb_reset_keys() { for (auto& a : g_keys) for (auto& b : a) b.clear(); g_queries.clear(); }
#endif

extern "C" {

// saddles: n x {x, y, k, theta, phi}.  Returns number of tags written (ascending id).
// smem_saddles: the on-chip saddle tier of the device launch being mirrored (320, 512, 1024 or 4096).
int hb_detect_from_saddles(const float* saddles, int n, const uint8_t* img, int w, int h,
                           size_t row_stride, int format, const uint64_t* codes, int n_codes,
                           int edge, int border, int hamming, int max_boards, int max_saddles,
                           agb::TagRec* out, int cap, int32_t* tap_quads, int* tap_n, int tap_cap,
                           uint32_t* status, int use_grid, int lattice, int smem_saddles) {
  using namespace agb;
  if (n > max_saddles) return -1;
  const int N = max_saddles, Q = N / 4 + 2;
  std::vector<float> pos(3 * (size_t)N, 0.0f);
  std::vector<int16_t> cell(kCells, 0), quads(4 * Q), touched(kCells);
  std::vector<int16_t> bquads(4 * Q), btouched(kCells), bvals(kCells);
  std::vector<uint32_t> active((N + 31) / 32, 0xffffffffu);
  std::vector<int16_t> stack(2 * (Q + 1)), seeds(N), nn(64), same(64), diff(64), samp(64);
  std::vector<int> hist(kHistBins);
  std::vector<uint8_t> remove(N), tag_valid(kMaxCodes, 0);
  std::vector<TagRec> tag_by_id(kMaxCodes);
  Frame F;
  memset(&F, 0, sizeof F);
  F.lane = 0;
  F.n = n;
  F.sx = &pos[0]; F.sy = &pos[N]; F.st = &pos[2 * (size_t)N];
  for (int i = 0; i < n; ++i) {
    F.sx[i] = saddles[5 * i]; F.sy[i] = saddles[5 * i + 1]; F.st[i] = saddles[5 * i + 3];
  }
  F.bs.cell = cell.data(); F.bs.quads = quads.data(); F.bs.touched = touched.data();
  F.bs.active = active.data();
  F.bs.n_quads = F.bs.n_touched = F.bs.score = 0;
  F.best.quads = bquads.data(); F.best.touched = btouched.data(); F.best.vals = bvals.data();
  F.best.n_quads = F.best.n_touched = F.best.score = 0;
  std::vector<int16_t> squads(4 * Q), stouched(kCells), svals(kCells);
  F.seedbest.quads = squads.data(); F.seedbest.touched = stouched.data(); F.seedbest.vals = svals.data();
  F.seedbest.n_quads = F.seedbest.n_touched = F.seedbest.score = 0;
  int ctl[16] = {0};
  F.ctl = ctl; F.w_score = ctl + 8;
  F.warp = 0; F.n_warps = 1;
  F.lat = lattice; F.lat_off = lattice / 2;
  // bucket grid, sized as the device kernel's general path sizes it: 1408 buckets (8192 in the 4096
  // tier), items for the tier's saddles -- or for max_saddles when the list is larger than the tier
  // and lives in global memory; use_grid = 0 tests the exhaustive scan
  int bucket = 32;
  const int grid_cap = smem_saddles == 4096 ? 8192 : 1408;
  while (((w + bucket - 1) / bucket) * ((h + bucket - 1) / bucket) > grid_cap) bucket *= 2;
  std::vector<uint16_t> gstart(grid_cap + 1), gitem(N);
  if (use_grid) {
    F.g_start = gstart.data(); F.g_item = gitem.data();
    F.g_nx = (w + bucket - 1) / bucket; F.g_ny = (h + bucket - 1) / bucket;
    F.g_cap_cells = grid_cap; F.g_cap_items = n <= smem_saddles ? smem_saddles : max_saddles;
    F.g_inv = 1.0f / (float)bucket;
  }
  F.stack = stack.data(); F.seeds = seeds.data(); F.nn_idx = nn.data(); F.same = same.data();
  F.diff = diff.data(); F.samp = samp.data(); F.hist = hist.data(); F.remove = remove.data();
  F.max_quads = Q;
  F.img = img; F.w = w; F.h = h; F.format = format; F.row_stride = row_stride;
  F.codes = codes; F.n_codes = n_codes; F.edge = edge; F.border = border; F.hamming = hamming;
  F.tag_valid = tag_valid.data(); F.tag_by_id = tag_by_id.data();
  F.tap_quads = tap_quads; F.tap_n_quads = tap_n; F.tap_cap = tap_cap;
  if (tap_n) *tap_n = 0;
  detect_boards(F, max_boards);
  int cnt = 0;
  for (int id = 0; id < n_codes; ++id)
    if (tag_valid[id]) {
      if (cnt < cap) out[cnt] = tag_by_id[id];
      ++cnt;
    }
  if (status) *status = F.status;
  return cnt;
}

}  // extern "C"
