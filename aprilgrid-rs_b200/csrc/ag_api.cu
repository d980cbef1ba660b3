// C ABI of the aprilgrid B200 library: handle, workspaces, chunked multi-stream pipeline.
// See include/aprilgrid_b200.h for the contract of every entry point.
#include <math.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "ag_codebook.h"
#include "ag_common.cuh"
#include "ag_kernels.h"

using namespace ag;

namespace {

struct FamilyInfo {
  int edge, border, hamming, n_codes;
  const uint64_t* codes;
};

bool family_info(int family, FamilyInfo* f) {  // src/detector.rs:369-405
  switch (family) {
    case AG_T16H5: *f = {4, 2, 1, ag_t16h5_count, ag_t16h5_codes}; return true;
    case AG_T25H7: *f = {5, 2, 2, ag_t25h7_count, ag_t25h7_codes}; return true;
    case AG_T25H9: *f = {5, 2, 2, ag_t25h9_count, ag_t25h9_codes}; return true;
    case AG_T36H11: *f = {6, 2, 3, ag_t36h11_count, ag_t36h11_codes}; return true;
    case AG_T36H11B1: *f = {6, 1, 3, ag_t36h11_count, ag_t36h11_codes}; return true;
  }
  return false;
}

// creation errors have no handle to live in: one message per calling thread
thread_local std::string g_create_error;

// Pipeline.  The dense front end (K1-K2) of a chunk runs on the dense stream, its sparse stages
// (K3-K4) on the detector's sparse stream, and the latency-bound board searches of earlier chunks
// on their board slots' own streams, side by side.  The dense buffers come in a ring of
// kDenseSets sets used by chunks in turn, so K1 of chunk i+1 runs while K3-K4 of chunk i still
// read chunk i's set; the light board-search side is multi-buffered further, so the board
// searches of up to kBoardSlots chunks overlap each other and the front end of later chunks,
// which hides the long tail of the slowest frames of a chunk.
constexpr int kDenseSets = 2;
constexpr int kBoardSlots = 8;
#ifndef AG_BIG_TIER_WARPS
#define AG_BIG_TIER_WARPS 2
#endif
constexpr int kBigTierBatchWarps = AG_BIG_TIER_WARPS;
#ifndef AG_SINGLE_WARPS
#define AG_SINGLE_WARPS 16
#endif
constexpr int kSingleFrameWarps = AG_SINGLE_WARPS;  // warps per frame when a launch holds only a few frames
constexpr size_t kMaxBlockSmem = 227 * 1024;       // dynamic shared memory a block may ask for on sm_100  // warps per frame of the 4096-tier batch launch

// Board-search side of a chunk: what K4 hands to K6, K6's workspace, its stream and events.
// A few hundred KB per frame, so many of these can be in flight (see kBoardSlots).
struct BoardSlot {
  cudaStream_t bstream = nullptr;
  cudaEvent_t ev_front = nullptr, ev_boards = nullptr;  // front end done / board search done
  bool pending = false;                                 // a board kernel may still be running
  int cap_frames = 0, cap_saddles = 0;
  long cfg_warps = -1, cfg_lattice = -1;
  ag_saddle* d_refined = nullptr;
  int* d_nref = nullptr;
  uint8_t* d_board_ws = nullptr;
  uint32_t* d_status = nullptr;
  uint32_t* d_board_tm = nullptr;  // optional per-frame timing of the board kernel ([frames][32])
  int32_t* d_tap_quads = nullptr;
  int* d_tap_nquads = nullptr;
  // [tier]: 0 = 320, 1 = 512, 2 = 1024 saddles on chip in the board kernel
  BoardWsLayout layout[4]{};        // sized for the largest warps-per-frame (allocation)
  BoardWsLayout layout_batch[4]{};  // layout used when many frames are in flight
  BoardWsLayout layout_split0{};    // ... by the first launch of a split batch: frames of at most 320 saddles only
  // host-frame path (ag_detect_batch) and the one-frame slot: staged input of the chunk (K6
  // samples the tag bits from it, so it lives as long as the slot's board search), device results
  // and pinned result staging
  uint8_t* d_in = nullptr;
  size_t cap_in_bytes = 0;
  uint8_t* h_in = nullptr;  // pinned staging for frames that arrive in pageable host memory
  size_t cap_h_in = 0;
  int hs_frames = 0, hs_tags = 0;
  ag_tag* d_tags = nullptr;
  int* d_ntags = nullptr;
  ag_tag* h_tags = nullptr;
  int* h_ntags = nullptr;
  uint32_t* h_status = nullptr;
  cudaEvent_t ev_up = nullptr, ev_done = nullptr;  // upload done / results on the host
};

// Dense and sparse buffers of one chunk (K1-K4).
struct Slot {
  cudaStream_t stream = nullptr;
  // the last work on the buffers is done: K3-K4 of the set's latest chunk (ring of the batch
  // pipelines), K2 (ag_dense_batch_device)
  cudaEvent_t done = nullptr;
  cudaEvent_t ev_dense = nullptr;  // ring: K1-K2 of the set's latest chunk done (the sparse stream waits on it)
  BoardSlot bb;  // the slot's own board-search side and host staging (one-frame slot only)
  // capacities in elements (frames x per-frame stride), except cap_frames
  int cap_frames = 0;
  size_t cap_px = 0, cap_words = 0, cap_list = 0, cap_cl = 0;
  int cap_clusters = 0;  // clusters per frame of the current call (stride of the cluster buffers)
  float *d_blur = nullptr, *d_resp = nullptr;
  uint32_t *d_min = nullptr, *d_mask = nullptr;
  int *d_parent = nullptr, *d_acc = nullptr, *d_ncl = nullptr;
  float2* d_centers = nullptr;
  ag_saddle* d_raw = nullptr;
  uint8_t* d_raw_valid = nullptr;
  // taps
  int* d_label_fallback = nullptr;  // K3: frames the run-based kernel handed to the pixel-list kernel
  uint32_t* d_pixlist = nullptr;   // K3: compact list of mask pixels / runs, [frames][pix_cap]
  int pix_cap = 0;  // list entries per frame of the current call
};

}  // namespace

struct ag_detector {
  int device = 0;
  int family = AG_T36H11;
  FamilyInfo fam{};
  ag_params params{};
  std::mutex mu;
  std::string err;
  // dense + sparse buffers of the batch pipelines, used by chunks in turn; dense[0]'s stream is the
  // detector's own dense stream (host-frame path, standalone operators, calls without a stream)
  Slot dense[kDenseSets];
  int dense_rr = 0;                      // next set of the ring (rotates across calls and both pipelines)
  cudaStream_t sparse_stream = nullptr;  // K3-K4 of the batch pipelines
  Slot big;  // one-frame slot with grown capacities: frames that overflowed max_clusters / max_saddles are re-run here
  BoardSlot bslot[kBoardSlots];
  int slot_rr = 0;            // next board slot of the device-batch pipeline (rotates across calls)
  cudaStream_t up_stream = nullptr;  // host-frame path: uploads, ahead of the kernels
  // host-buffer path: chunks whose results still sit in a board slot's pinned staging, with the
  // output arrays of the ag_detect_batch call they belong to (calls may overlap: "host_async")
  struct HostPend {
    bool live = false;
    int f0 = 0, n = 0, cap = 0;
    uint64_t seq = 0;
    ag_tag* out = nullptr;
    int* n_per_frame = nullptr;
    uint32_t* status = nullptr;
    const uint8_t* src = nullptr;  // host frames of the chunk (re-run of overflowed frames)
    FrameGeom g{};
  } hpend[kBoardSlots];
  uint64_t host_seq = 0;        // number of ag_detect_batch calls issued
  bool host_async = false;      // ag_detect_batch returns without collecting its results
  bool host_truncated = false;  // a collected frame had more tags than its call's cap_per_frame
  bool host_unresolved = false;  // a collected frame overflowed a capacity that could not be grown
  bool device_path_busy = false;  // device-batch work may still be in flight on the dense sets / the board slots
  bool device_async = false;  // ag_detect_batch_device returns without ordering the results on the
                              // caller's stream; ag_detect_batch_device_wait does that
  uint64_t launches = 0;
  long chunk_frames = 1024;  // measured on 1280x1024 frames, 1024 per call: 512 -> 102.8 k, 1024 -> 107.6 k frames/s (2048 with larger calls: 112 k)
  long host_chunk_frames = 128;  // chunk of the host-buffer path (ag_detect_batch)
  // per-frame capacities; 0 = automatic (from the image area, see set_caps).  A frame that still
  // overflows them is re-run on its own with grown capacities (host entry points), so they bound
  // memory, not results.
  long max_clusters = 0;
  long max_saddles = 0;
  int cur_clusters = 16384, cur_saddles = 2048;  // capacities in force for the current call
  uint64_t* d_codes = nullptr;  // family table in global memory (renderer)
  // stage-tap state
  FrameGeom tap_geom{};
  bool tap_valid = false;
  // 0 = auto: the streaming K1 where applicable; 1 = always the generic tile kernel
  long dense_variant = 0;
  long k1_chunk_rows = 0;  // 0 = automatic; else the rows per warp of the streaming K1 (6k + 4)
  long board_lattice = 64;  // side of the tag lattice a board may span (16 / 32 / 64)
  // warps per frame in the board kernel: 0 = automatic (1 when a launch has enough frames to
  // fill the GPU with one-warp blocks, 4 otherwise), or 1 / 2 / 4 / 8
  long board_warps = 0;
  long board_batch_frames = 148;  // automatic mode: launches with at least this many frames use 2 warps per frame
  long label_variant = 0;  // K3: 0 = run-based in shared memory, 1 = pixel list with per-pixel parents
  long board_saddle_tier = -1;  // -1 automatic, 0 = 512, 1 = 1024, 2 = 4096 saddles on chip in the board kernel
  bool board_timing = false;  // per-frame timing taps of the board kernel (ag_test_board_times)
  bool board_fast = true;  // four-lane group scoring of candidate boards (0 = general path only)
  long board_priority = 0;  // priority of the board-search streams: 0 = least (= default streams), 1 = greatest
  bool board_split = true;  // batches: small frames (<= 320 saddles) searched by their own launch with the small tier
  bool board_grid = true;  // bucket-grid radius queries in the board kernel (0 = exhaustive scan)
  bool profile = false;
  std::vector<cudaEvent_t> ev_pool;
  std::vector<int> ev_stage;  // stage id of the interval ENDING at event i, -1 = interval start
  size_t ev_used = 0;
  double stage_ms[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  uint64_t stage_n[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  // scratch for the standalone operators
  float *d_f32_a = nullptr, *d_f32_b = nullptr, *d_f32_c = nullptr, *d_taps = nullptr;
  size_t f32_cap = 0;
};

namespace {

#define AG_CUDA(det, call)                                                                   \
  do {                                                                                       \
    cudaError_t e__ = (call);                                                                \
    if (e__ != cudaSuccess) {                                                                \
      char b__[512];                                                                         \
      snprintf(b__, sizeof b__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),     \
               __FILE__, __LINE__);                                                          \
      (det)->err = b__;                                                                      \
      return AG_ERR_CUDA;                                                                    \
    }                                                                                        \
  } while (0)

// Host-buffer entry points and the standalone operators share the dense slot with the device-batch
// pipeline: wait until the latter has drained before touching the buffers.
int quiesce_device_path(ag_detector* det, bool host_too = true);

int fail(ag_detector* det, int code, const char* msg) {
  if (det) det->err = msg;
  return code;
}

int make_geom(ag_detector* det, int w, int h, size_t row_stride, size_t frame_stride, int format,
              FrameGeom* g) {
  if (w <= 0 || h <= 0) return fail(det, AG_ERR_INVALID, "width/height must be positive");
  if (format == kFmtF32 || bytes_per_px(format) == 0) return fail(det, AG_ERR_INVALID, "unknown pixel format");
  if ((long long)w * h > (1ll << 30)) return fail(det, AG_ERR_INVALID, "image too large");
  size_t min_row = (size_t)w * bytes_per_px(format);
  if (row_stride == 0) row_stride = min_row;
  if (row_stride < min_row) return fail(det, AG_ERR_INVALID, "row_stride smaller than a row");
  const size_t al = (size_t)channel_align(format);
  if (row_stride % al) return fail(det, AG_ERR_INVALID, "row_stride must be a multiple of the format's channel word");
  if (frame_stride == 0) frame_stride = row_stride * h;
  if (frame_stride < row_stride * (size_t)(h - 1) + min_row)
    return fail(det, AG_ERR_INVALID, "frame_stride smaller than a frame");
  // other frames of a misaligned stride would start misaligned: K1 and K6 read 16-bit and f32 channels
  // with loads of their size (the host path keeps the caller's frame stride in its device staging too)
  if (frame_stride % al)
    return fail(det, AG_ERR_INVALID, "frame_stride must be a multiple of the format's channel word");
  g->w = w;
  g->h = h;
  g->wpr = (w + 31) / 32;
  g->n_words = g->wpr * h;
  g->n_px = w * h;
  g->row_stride = row_stride;
  g->frame_stride = frame_stride;
  g->format = format;
  return AG_OK;
}

// Bytes from a frame's first pixel to its last: the padding after the last row is not the frame's.
size_t frame_bytes(const FrameGeom& g) {
  return g.row_stride * (size_t)(g.h - 1) + (size_t)g.w * bytes_per_px(g.format);
}

// Per-frame capacities in force for a call: the options when set, else sized from the image area
// (1280 x 1024 -> 16384 clusters, 2048 saddles; a 4K frame -> 103680 / 13056).  Real images stay
// far below them; a frame that does not is flagged and re-run alone with grown capacities.
void set_caps(ag_detector* det, const FrameGeom& g) {
  long ncl = det->max_clusters, nsd = det->max_saddles;
  if (ncl <= 0) ncl = std::min<long>(std::max<long>(g.n_px / 80, 16384), 1l << 22);
  if (nsd <= 0) nsd = std::min<long>(std::max<long>(((g.n_px / 640 + 255) / 256) * 256, 2048), 16384);
  det->cur_clusters = (int)ncl;
  det->cur_saddles = (int)nsd;
}
// Frames per chunk of the host-buffer path, before chunk_limit: the option host_chunk_frames, scaled
// down for formats above 8 bytes per pixel so that a board slot's staging (device, and pinned for
// pageable input) never holds more bytes per chunk than for RGBA16 frames of the same size.
long host_chunk_for(long host_chunk_frames, int format) {
  const int bpp = bytes_per_px(format);
  return bpp > 8 ? std::max<long>(1, host_chunk_frames * 8 / bpp) : host_chunk_frames;
}
// Frames per pipeline chunk: the option, bounded so that the dense buffers of a chunk (blur +
// response, 8 bytes per pixel) stay below 24 GB whatever the image size.  The bound is per set:
// the pipelines keep kDenseSets = 2 sets, about 8.6 bytes per pixel each with mask and pixel list,
// so chunks of 1024 frames of 1280 x 1024 take 2 x 11.6 GB = 23.2 GB of dense buffers.
int chunk_limit(const ag_detector* det, const FrameGeom& g, long want) {
  const long by_mem = std::max<long>(1, (long)((24ull << 30) / ((unsigned long long)g.n_px * 8ull)));
  return (int)std::max<long>(1, std::min<long>(want, by_mem));
}

template <typename T>
int regrow(ag_detector* det, T** p, size_t count) {
  if (*p) AG_CUDA(det, cudaFree(*p));
  *p = nullptr;
  if (count == 0) count = 1;
  AG_CUDA(det, cudaMalloc((void**)p, count * sizeof(T)));
  return AG_OK;
}

// Make sure a board slot can hold `frames` frames.  Waits for a board kernel that may still be
// using the slot only when its buffers have to be replaced (or when asked to: `drain`).
int ensure_board_slot(ag_detector* det, BoardSlot& B, int frames, bool drain) {
  int rc;
  if (!B.bstream) {
    // lowest priority: the long-lived board-search blocks must not keep the bandwidth-bound
    // front end of the following chunks (caller's stream, default priority) off the SMs
    int prio_least = 0, prio_greatest = 0;
    AG_CUDA(det, cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
    AG_CUDA(det, cudaStreamCreateWithPriority(&B.bstream, cudaStreamNonBlocking,
                                              det->board_priority ? prio_greatest : prio_least));
    AG_CUDA(det, cudaEventCreateWithFlags(&B.ev_front, cudaEventDisableTiming));
    AG_CUDA(det, cudaEventCreateWithFlags(&B.ev_boards, cudaEventDisableTiming));
  }
  const int nsd = det->cur_saddles;
  const bool realloc = frames > B.cap_frames || nsd != B.cap_saddles || det->board_warps != B.cfg_warps ||
                       det->board_lattice != B.cfg_lattice;
  if (B.pending && (realloc || drain)) {
    AG_CUDA(det, cudaEventSynchronize(B.ev_boards));
    B.pending = false;
  }
  if (!realloc) return AG_OK;
  const int F = std::max(frames, B.cap_frames);
  if ((rc = regrow(det, &B.d_nref, (size_t)F))) return rc;
  if ((rc = regrow(det, &B.d_status, (size_t)F))) return rc;
  if ((rc = regrow(det, &B.d_refined, (size_t)F * nsd))) return rc;
  // layouts for both tiers of on-chip saddle capacity (chosen per launch from the image size)
  for (int tier = 0; tier < 4; ++tier) {
    const int cap = tier == 0 ? 320 : (tier == 1 ? 512 : (tier == 2 ? 1024 : 4096));
    // warps per frame: halved until the tier's shared memory fits a block
    auto fitted = [&](int warps, bool with_gpos) {
      for (;;) {
        BoardWsLayout L = make_board_layout(nsd, (int)det->board_lattice, warps, cap, with_gpos);
        if (L.smem_per_block <= kMaxBlockSmem || warps == 1) return L;
        warps /= 2;
      }
    };
    // few frames per launch: as many warps per frame as there is room for
    B.layout[tier] = fitted(det->board_warps ? (int)det->board_warps : kSingleFrameWarps, true);
    // the batch launch of the 4096 tier only sees frames of more than 1024 saddles (general path):
    // no grid-ordered positions, two frames per SM instead of one
    B.layout_batch[tier] =
        fitted(det->board_warps ? (int)det->board_warps : (tier == 3 ? kBigTierBatchWarps : 2), tier != 3);
  }
  B.layout_split0 = make_board_layout(nsd, (int)det->board_lattice, B.layout_batch[0].warps, 320, true, 320);
  if ((rc = regrow(det, &B.d_board_ws, (size_t)F * B.layout[0].bytes_per_frame))) return rc;
  if ((rc = regrow(det, &B.d_tap_quads, (size_t)F * B.layout[0].max_quads * 4))) return rc;
  if ((rc = regrow(det, &B.d_tap_nquads, (size_t)F))) return rc;
  if ((rc = regrow(det, &B.d_board_tm, (size_t)F * 32))) return rc;
  B.cap_frames = F;
  B.cap_saddles = nsd;
  B.cfg_warps = det->board_warps;
  B.cfg_lattice = det->board_lattice;
  return AG_OK;
}

// Host-frame staging of a board slot: `frames` frames of `in_bytes_per_chunk` bytes in total,
// `cap_tags` result records per frame.
int ensure_host_stage(ag_detector* det, BoardSlot& B, size_t in_bytes, int frames, int cap_tags) {
  int rc;
  if (!B.ev_up) {
    AG_CUDA(det, cudaEventCreateWithFlags(&B.ev_up, cudaEventDisableTiming));
    AG_CUDA(det, cudaEventCreateWithFlags(&B.ev_done, cudaEventDisableTiming));
  }
  if (in_bytes > B.cap_in_bytes) {
    if ((rc = regrow(det, &B.d_in, in_bytes))) return rc;
    B.cap_in_bytes = in_bytes;
  }
  if (frames > B.hs_frames || cap_tags > B.hs_tags) {
    const int F = std::max(frames, B.hs_frames), ct = std::max(cap_tags, B.hs_tags);
    if ((rc = regrow(det, &B.d_tags, (size_t)F * ct))) return rc;
    if ((rc = regrow(det, &B.d_ntags, (size_t)F))) return rc;
    if (B.h_tags) cudaFreeHost(B.h_tags);
    if (B.h_ntags) cudaFreeHost(B.h_ntags);
    if (B.h_status) cudaFreeHost(B.h_status);
    AG_CUDA(det, cudaMallocHost((void**)&B.h_tags, sizeof(ag_tag) * (size_t)F * ct));
    AG_CUDA(det, cudaMallocHost((void**)&B.h_ntags, sizeof(int) * F));
    AG_CUDA(det, cudaMallocHost((void**)&B.h_status, sizeof(uint32_t) * F));
    B.hs_frames = F;
    B.hs_tags = ct;
  }
  return AG_OK;
}

void free_board_slot(BoardSlot& B) {
  cudaFree(B.d_in); cudaFree(B.d_tags); cudaFree(B.d_ntags);
  if (B.h_in) cudaFreeHost(B.h_in);
  if (B.h_tags) cudaFreeHost(B.h_tags);
  if (B.h_ntags) cudaFreeHost(B.h_ntags);
  if (B.h_status) cudaFreeHost(B.h_status);
  if (B.ev_up) cudaEventDestroy(B.ev_up);
  if (B.ev_done) cudaEventDestroy(B.ev_done);
  cudaFree(B.d_nref); cudaFree(B.d_status); cudaFree(B.d_refined); cudaFree(B.d_board_ws);
  cudaFree(B.d_tap_quads); cudaFree(B.d_tap_nquads); cudaFree(B.d_board_tm);
  if (B.ev_front) cudaEventDestroy(B.ev_front);
  if (B.ev_boards) cudaEventDestroy(B.ev_boards);
  if (B.bstream) cudaStreamDestroy(B.bstream);
  B = BoardSlot();
}

// Make sure a slot can hold `frames` frames of geometry g.  `own_board` = the slot's own
// board-search side is needed too, with host staging for `frames` frames of g.frame_stride bytes
// and every tag of the family per frame (the one-frame slot).
int ensure_slot(ag_detector* det, Slot& S, const FrameGeom& g, int frames, bool own_board = true,
                bool need_parent = false) {
  int rc;
  if (!S.stream) {
    AG_CUDA(det, cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
    AG_CUDA(det, cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
  }
  // (the standalone operators create the first set's stream and event without this one)
  if (!S.ev_dense) AG_CUDA(det, cudaEventCreateWithFlags(&S.ev_dense, cudaEventDisableTiming));
  if (own_board && ((rc = ensure_board_slot(det, S.bb, frames, true)) ||
                    (rc = ensure_host_stage(det, S.bb, (size_t)frames * g.frame_stride, frames, det->fam.n_codes))))
    return rc;
  // Per-frame strides follow this call's geometry; each buffer grows to the most elements (frames x
  // stride) a call has needed, not to the most frames times the largest image: a set that served
  // chunks of 1024 small frames and then 256 4K frames holds 256 x 4K pixels, not 1024 x 4K.
  // The saddle mask is 1-4 % full; a list of 1/8 of the pixels covers every real image, fuller
  // masks (noise) take the word-oriented labelling path.
  const int pix_cap = (int)std::min<size_t>(std::max<size_t>((size_t)g.n_px / 8, 32768), (size_t)1 << 20);
  const size_t px = (size_t)frames * g.n_px, words = (size_t)frames * g.n_words, list = (size_t)frames * pix_cap;
  if (px > S.cap_px || words > S.cap_words || list > S.cap_list) {
    // make sure nothing is in flight on the buffers we are about to free (the pipelines' chunks
    // run on the caller's and the sparse stream: their last work on the set is S.done)
    AG_CUDA(det, cudaStreamSynchronize(S.stream));
    AG_CUDA(det, cudaEventSynchronize(S.done));
    S.cap_px = std::max(px, S.cap_px);
    S.cap_words = std::max(words, S.cap_words);
    S.cap_list = std::max(list, S.cap_list);
    if ((rc = regrow(det, &S.d_blur, S.cap_px))) return rc;
    if ((rc = regrow(det, &S.d_resp, S.cap_px))) return rc;
    // per-pixel union-find parents: only the labels tap needs them kept; the labelling kernels
    // that want per-pixel scratch otherwise use the response buffer, which is dead after K2
    if (S.d_parent) { AG_CUDA(det, cudaFree(S.d_parent)); S.d_parent = nullptr; }
    if ((rc = regrow(det, &S.d_mask, S.cap_words))) return rc;
    if ((rc = regrow(det, &S.d_pixlist, S.cap_list))) return rc;
  }
  S.pix_cap = pix_cap;
  const int ncl = det->cur_clusters;
  const size_t cl = (size_t)frames * ncl;
  if (frames > S.cap_frames || cl > S.cap_cl) {
    AG_CUDA(det, cudaStreamSynchronize(S.stream));
    AG_CUDA(det, cudaEventSynchronize(S.done));
    S.cap_frames = std::max(frames, S.cap_frames);
    S.cap_cl = std::max(cl, S.cap_cl);
    if ((rc = regrow(det, &S.d_min, (size_t)S.cap_frames))) return rc;
    if ((rc = regrow(det, &S.d_ncl, (size_t)S.cap_frames))) return rc;
    if ((rc = regrow(det, &S.d_label_fallback, (size_t)S.cap_frames))) return rc;
    if ((rc = regrow(det, &S.d_acc, S.cap_cl * 3))) return rc;
    if ((rc = regrow(det, &S.d_centers, S.cap_cl))) return rc;
    if ((rc = regrow(det, &S.d_raw, S.cap_cl))) return rc;
    if ((rc = regrow(det, &S.d_raw_valid, S.cap_cl))) return rc;
  }
  S.cap_clusters = ncl;
  if (need_parent && !S.d_parent) {
    AG_CUDA(det, cudaStreamSynchronize(S.stream));
    AG_CUDA(det, cudaEventSynchronize(S.done));
    if ((rc = regrow(det, &S.d_parent, S.cap_px))) return rc;
  }
  return AG_OK;
}

void free_slot(Slot& S) {
  cudaFree(S.d_blur); cudaFree(S.d_resp); cudaFree(S.d_min); cudaFree(S.d_mask);
  cudaFree(S.d_parent); cudaFree(S.d_acc); cudaFree(S.d_ncl); cudaFree(S.d_centers); cudaFree(S.d_raw);
  cudaFree(S.d_raw_valid); cudaFree(S.d_pixlist); cudaFree(S.d_label_fallback);
  free_board_slot(S.bb);
  if (S.done) cudaEventDestroy(S.done);
  if (S.ev_dense) cudaEventDestroy(S.ev_dense);
  if (S.stream) cudaStreamDestroy(S.stream);
  S = Slot();
}

// Frames in ordinary (pageable) host memory -- a Vec<u8> packed from DynamicImages, a numpy array --
// cannot be read by the copy engine directly: cudaMemcpyAsync would stage them through the
// driver's small bounce buffer, synchronously and at a fraction of the link rate.  They are copied
// into the slot's own pinned staging buffer by several host threads instead (memcpy at memory
// bandwidth), from where the usual asynchronous upload takes them.
bool is_pageable(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return true;
  }
  return a.type == cudaMemoryTypeUnregistered;
}
// One thread's share: streaming (non-temporal) stores, so the destination lines are not read
// first -- the staging buffer is written once and then read by the copy engine, never by the CPU.
void stream_copy(uint8_t* dst, const uint8_t* src, size_t n) {
#if defined(__x86_64__) && defined(__SSE2__)
  if (n >= 4096 && ((uintptr_t)dst & 15) == 0) {
    size_t i = 0;
    for (; i + 64 <= n; i += 64) {
      const __m128i a = _mm_loadu_si128((const __m128i*)(src + i)), b = _mm_loadu_si128((const __m128i*)(src + i + 16));
      const __m128i c = _mm_loadu_si128((const __m128i*)(src + i + 32)), d = _mm_loadu_si128((const __m128i*)(src + i + 48));
      _mm_stream_si128((__m128i*)(dst + i), a);
      _mm_stream_si128((__m128i*)(dst + i + 16), b);
      _mm_stream_si128((__m128i*)(dst + i + 32), c);
      _mm_stream_si128((__m128i*)(dst + i + 48), d);
    }
    _mm_sfence();
    memcpy(dst + i, src + i, n - i);
    return;
  }
#endif
  memcpy(dst, src, n);
}
void parallel_copy(uint8_t* dst, const uint8_t* src, size_t bytes) {
  const unsigned hw = std::thread::hardware_concurrency();
  size_t nt = std::min<size_t>(std::max<unsigned>(hw, 1), 24);
  nt = std::min(nt, std::max<size_t>(bytes >> 22, 1));  // at least 4 MB per thread
  if (nt <= 1) {
    stream_copy(dst, src, bytes);
    return;
  }
  const size_t per = ((bytes + nt - 1) / nt + 4095) & ~(size_t)4095;
  std::vector<std::thread> th;
  for (size_t t = 1; t < nt; ++t) {
    const size_t lo = t * per;
    if (lo >= bytes) break;
    th.emplace_back([=] { stream_copy(dst + lo, src + lo, std::min(per, bytes - lo)); });
  }
  stream_copy(dst, src, std::min(per, bytes));
  for (auto& t : th) t.join();
}

// Stage ids for the optional timing: 0 K1 blur+hessian+min, 1 K2 threshold, 2 K3 label+centroid,
// 3 K4 refine+filter, 4 K6 boards+decode.
void prof_mark(ag_detector* det, int stage, cudaStream_t s) {
  if (!det->profile) return;
  if (det->ev_used == det->ev_pool.size()) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    det->ev_pool.push_back(e);
    det->ev_stage.push_back(-1);
  }
  det->ev_stage[det->ev_used] = stage;
  cudaEventRecord(det->ev_pool[det->ev_used], s);
  ++det->ev_used;
}

// Dense front end of one chunk on stream s: K1 + K2.
int run_dense(ag_detector* det, Slot& S, const uint8_t* d_frames, const FrameGeom& g, int n,
              bool write_blur, cudaStream_t s) {
  prof_mark(det, -1, s);
  const int variant = det->dense_variant == 1 ? 1 : 0;
  det->launches += launch_blur_hessian(d_frames, g, n, S.d_blur, S.d_resp, S.d_min, write_blur, variant,
                                       (int)det->k1_chunk_rows, s);
  prof_mark(det, 0, s);
  det->launches += launch_threshold(S.d_resp, g, n, S.d_min, S.d_mask, s);
  prof_mark(det, 1, s);
  AG_CUDA(det, cudaGetLastError());
  return AG_OK;
}

// Sparse stages up to the refined saddle list.
int run_sparse(ag_detector* det, Slot& S, BoardSlot& B, const FrameGeom& g, int n, uint32_t* d_status,
               cudaStream_t s, bool want_pixel_parents = false) {
  AG_CUDA(det, cudaMemsetAsync(d_status, 0, sizeof(uint32_t) * n, s));
  prof_mark(det, -1, s);
  // label_variant 0: run-based (no per-pixel parent array) unless the labels tap needs one
  const int variant = (det->label_variant == 0 && !want_pixel_parents) ? 0 : 1;
  // per-pixel parents: the kept array when the labels tap asked for one (taps), else the response
  // buffer as scratch (K2 has consumed it; nothing downstream reads it)
  int* parent = S.d_parent ? S.d_parent : reinterpret_cast<int*>(S.d_resp);
  det->launches += launch_label_clusters(S.d_mask, g, n, parent, S.cap_clusters, S.d_acc,
                                         S.d_centers, S.d_ncl, d_status, S.d_pixlist, S.pix_cap, variant,
                                         S.d_label_fallback, s);
  prof_mark(det, 2, s);
  det->launches += launch_refine_filter(S.d_blur, g, n, S.d_centers, S.d_ncl, S.cap_clusters, S.d_raw,
                                        S.d_raw_valid, det->params.min_saddle_angle,
                                        det->params.max_saddle_angle, B.cap_saddles, B.d_refined,
                                        B.d_nref, d_status, s);
  prof_mark(det, 3, s);
  AG_CUDA(det, cudaGetLastError());
  return AG_OK;
}

// Both sets of the pipelines' dense ring, for chunks of `frames` frames, and the sparse stream.
int ensure_ring(ag_detector* det, const FrameGeom& g, int frames) {
  int rc;
  for (auto& D : det->dense)
    if ((rc = ensure_slot(det, D, g, frames, false))) return rc;
  if (!det->sparse_stream) AG_CUDA(det, cudaStreamCreateWithFlags(&det->sparse_stream, cudaStreamNonBlocking));
  return AG_OK;
}

// Front end of one pipeline chunk into the next set of the dense ring: K1-K2 on the dense stream
// s, then K3-K4 on the sparse stream into board slot B; B.ev_front marks the refined saddles
// ready.  The set is reused only after the sparse stages of its previous chunk (which read its
// blur and use its response buffer as scratch), and B only after its previous board search (K4
// writes B's saddle list).  Ordering through the set's events also holds when consecutive calls
// come on different streams.
int run_front(ag_detector* det, BoardSlot& B, const uint8_t* d_frames, const FrameGeom& g, int n,
              uint32_t* d_status, cudaStream_t s) {
  int rc;
  Slot& D = det->dense[det->dense_rr];
  det->dense_rr = (det->dense_rr + 1) % kDenseSets;
  const cudaStream_t sp = det->sparse_stream;
  AG_CUDA(det, cudaStreamWaitEvent(s, D.done, 0));
  if ((rc = run_dense(det, D, d_frames, g, n, true, s))) return rc;
  AG_CUDA(det, cudaEventRecord(D.ev_dense, s));
  AG_CUDA(det, cudaStreamWaitEvent(sp, D.ev_dense, 0));
  if (B.pending) AG_CUDA(det, cudaStreamWaitEvent(sp, B.ev_boards, 0));
  if ((rc = run_sparse(det, D, B, g, n, d_status, sp))) return rc;
  AG_CUDA(det, cudaEventRecord(D.done, sp));
  AG_CUDA(det, cudaEventRecord(B.ev_front, sp));
  return AG_OK;
}

int run_boards(ag_detector* det, BoardSlot& S, const uint8_t* d_frames, const FrameGeom& g, int n,
               ag_tag* d_tags, int cap, int* d_ntags, uint32_t* d_status, bool taps,
               cudaStream_t s) {
  prof_mark(det, -1, s);
  // automatic warps per frame: throughput (2 warps: most frames resident per SM) once a launch can
  // fill the GPU, latency (8 warps share one frame's seeds) for a handful of frames.
  // On-chip saddle capacity (tier): 512 up to 1.5 Mpx, 1024 up to 6 Mpx, 4096 above (larger images
  // carry more saddles); frames beyond the tier keep their saddles in global memory and take the
  // general path inside the kernel.  A batch is searched by up to THREE launches: frames of at most
  // 320 saddles (one board) with the small tier -- 32 KB of shared memory per frame, seven frames
  // per SM --, frames of up to 512 / 1024 saddles with that tier, and (large images only) the rest
  // with the 4096 tier; a block whose frame belongs to another launch exits at once.
  const int big = det->board_saddle_tier >= 0 ? (int)det->board_saddle_tier + 1
                                              : ((long long)g.w * g.h > 6291456ll ? 3 : ((long long)g.w * g.h > 1572864ll ? 2 : 1));
  const bool many = n >= det->board_batch_frames;
  const bool batch = det->board_warps == 0 && many;
  const bool split = many && det->board_split;
  int tiers[3], n_launch = 0;
  if (split) {
    tiers[n_launch++] = 0;
    tiers[n_launch++] = big == 3 ? 2 : big;
    if (big == 3) tiers[n_launch++] = 3;
  } else {
    tiers[n_launch++] = (batch && big == 3) ? 2 : big;  // layout_batch[3] is for frames beyond the throughput path only
  }
  for (int pass = 0; pass < n_launch; ++pass) {
    const int tier = tiers[pass];
    const int n_above = pass == 0 ? -1 : S.layout[tiers[pass - 1]].smem_saddles;
    const int n_upto = pass == n_launch - 1 ? 0x7fffffff : S.layout[tier].smem_saddles;
    const BoardWsLayout& BL = batch ? ((split && pass == 0) ? S.layout_split0 : S.layout_batch[tier]) : S.layout[tier];
    det->launches += launch_boards_decode(
        d_frames, g, n, S.d_refined, S.d_nref, S.d_board_ws, BL, det->d_codes, det->fam.n_codes, det->fam.edge,
        det->fam.border, det->fam.hamming, det->params.max_num_of_boards, d_tags, cap, d_ntags,
        d_status, taps ? S.d_tap_quads : nullptr, taps ? S.d_tap_nquads : nullptr, S.layout[0].max_quads,
        det->board_grid ? 1 : 0, det->board_fast ? 1 : 0, det->board_timing ? S.d_board_tm : nullptr, n_above,
        n_upto, s);
  }
  prof_mark(det, 4, s);
  AG_CUDA(det, cudaGetLastError());
  return AG_OK;
}

constexpr uint32_t kGrowable = AG_FRAME_CLUSTER_OVERFLOW | AG_FRAME_SADDLE_OVERFLOW;

// What run_one_frame runs after K1-K4: K6, nothing (the refined saddles are the result), or K6
// keeping every intermediate for the stage taps.
enum class FrameRun { kTags, kSaddles, kTaps };

// One frame through the pipeline on the detector's one-frame slot (det->big), synchronously.  The
// slot has its own stream and buffers, so chunks of streaming calls may be in flight meanwhile.
// upload(d_in, stream) enqueues the copy of the frame into the slot's staged input; K1-K4 read it
// as geometry g, K6 samples the tag bits from geometry gb at d_in + bits_offset.
// A frame that overflows max_clusters / max_saddles is run again with what it overflowed grown
// (clusters x16 up to 2^22, saddles to 16384; the reference has no limits) until it fits or the
// capacities are at those limits.  first_status != 0 (the frame overflowed in a batch chunk) grows
// them before the first run; if none can grow, that status and 0 results come back without a run.
// The stage taps run once, at the call's capacities.
// Out: *count = tags found (refined saddles for kSaddles) and *status = the frame's status bits;
// the tags are in big.bb.h_tags, the refined saddles in big.bb.d_refined.
template <typename Upload>
int run_one_frame(ag_detector* det, const FrameGeom& g, const FrameGeom& gb, size_t bits_offset, Upload upload,
                  FrameRun what, uint32_t first_status, int* count, uint32_t* status) {
  struct RestoreCaps {  // the call's capacities come back on every exit
    ag_detector* det;
    int clusters, saddles;
    ~RestoreCaps() {
      det->cur_clusters = clusters;
      det->cur_saddles = saddles;
    }
  } restore{det, det->cur_clusters, det->cur_saddles};
  det->tap_valid = false;  // the taps read the buffers about to be overwritten
  Slot& S = det->big;
  BoardSlot& B = S.bb;
  const bool taps = what == FrameRun::kTaps;
  uint32_t st = first_status;
  int cnt = 0, rc;
  for (bool ran = false;; ran = true) {
    if (ran || st) {
      bool grew = false;
      if ((st & AG_FRAME_CLUSTER_OVERFLOW) && det->cur_clusters < (1 << 22)) {
        det->cur_clusters = (int)std::min<long>((long)det->cur_clusters * 16, 1l << 22);
        grew = true;
      }
      if ((st & AG_FRAME_SADDLE_OVERFLOW) && det->cur_saddles < 16384) {
        det->cur_saddles = 16384;
        grew = true;
      }
      if (taps || !grew) break;
    }
    if ((rc = ensure_slot(det, S, g, 1, true, taps))) return rc;
    const cudaStream_t s = S.stream;
    AG_CUDA(det, upload(B.d_in, s));
    if ((rc = run_dense(det, S, B.d_in, g, 1, true, s))) return rc;
    // taps: the labels tap reads the per-pixel parent array, which only the pixel-list kernel writes;
    // run it first, then the regular (run-based) labelling, whose centres the pipeline continues with
    if (taps && det->label_variant == 0 && (rc = run_sparse(det, S, B, g, 1, B.d_status, s, true))) return rc;
    if ((rc = run_sparse(det, S, B, g, 1, B.d_status, s))) return rc;
    if (what == FrameRun::kSaddles) {
      AG_CUDA(det, cudaMemcpyAsync(B.h_ntags, B.d_nref, sizeof(int), cudaMemcpyDeviceToHost, s));
    } else {  // (K6 reports 0 tags for a frame whose saddle list K3 / K4 flagged as truncated)
      if ((rc = run_boards(det, B, B.d_in + bits_offset, gb, 1, B.d_tags, B.hs_tags, B.d_ntags, B.d_status, taps, s)))
        return rc;
      AG_CUDA(det, cudaMemcpyAsync(B.h_ntags, B.d_ntags, sizeof(int), cudaMemcpyDeviceToHost, s));
      AG_CUDA(det, cudaMemcpyAsync(B.h_tags, B.d_tags, sizeof(ag_tag) * B.hs_tags, cudaMemcpyDeviceToHost, s));
    }
    AG_CUDA(det, cudaMemcpyAsync(B.h_status, B.d_status, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    AG_CUDA(det, cudaStreamSynchronize(s));
    cnt = B.h_ntags[0];
    st = B.h_status[0];
  }
  *count = cnt;
  *status = st;
  return AG_OK;
}

void copy_out_b(const BoardSlot& B, int n, int cap, ag_tag* out, int* n_per_frame, uint32_t* frame_status,
                int frame0, bool* truncated);

// Host-buffer path: wait for the chunk staged in board slot bi and hand its results to the output
// arrays of the call that submitted it.  A frame that overflowed max_clusters / max_saddles was
// truncated by the pipeline: it is run again, alone, with grown capacities, so the caller gets
// the untruncated result (the reference has no such limits, src/detector.rs:505-540) or an error.
int collect_host_slot(ag_detector* det, int bi) {
  auto& P = det->hpend[bi];
  if (!P.live) return AG_OK;
  BoardSlot& B = det->bslot[bi];
  AG_CUDA(det, cudaEventSynchronize(B.ev_done));
  copy_out_b(B, P.n, P.cap, P.out, P.n_per_frame, P.status, P.f0, &det->host_truncated);
  P.live = false;
  B.pending = false;
  for (int i = 0; i < P.n; ++i) {
    const uint32_t st = B.h_status[i];
    if (st & kGrowable) {
      FrameGeom g = P.g;
      g.frame_stride = g.row_stride * (size_t)g.h;
      const uint8_t* src = P.src + (size_t)i * P.g.frame_stride;
      auto upload = [&](uint8_t* d_in, cudaStream_t s) {
        return cudaMemcpyAsync(d_in, src, frame_bytes(g), cudaMemcpyHostToDevice, s);
      };
      int cnt = 0;
      uint32_t st2 = 0;
      int rc = run_one_frame(det, g, g, 0, upload, FrameRun::kTags, st, &cnt, &st2);
      if (rc) return rc;
      const BoardSlot& R = det->big.bb;
      memcpy(P.out + (size_t)(P.f0 + i) * P.cap, R.h_tags,
             sizeof(ag_tag) * (size_t)std::min(std::min(cnt, P.cap), R.hs_tags));
      if (cnt > P.cap) {
        st2 |= AG_FRAME_TAG_OVERFLOW;
        det->host_truncated = true;
      }
      P.n_per_frame[P.f0 + i] = cnt;
      if (P.status) P.status[P.f0 + i] = st2;
      if (st2 & (kGrowable | AG_FRAME_BOARD_OVERFLOW)) det->host_unresolved = true;
    } else if (st & AG_FRAME_BOARD_OVERFLOW) {
      det->host_unresolved = true;
    }
  }
  return AG_OK;
}
// ... for every chunk of the calls up to sequence number `upto`, oldest first (board slots are
// handed out round-robin, so the oldest chunk sits in the slot that is reused next)
int collect_host(ag_detector* det, uint64_t upto) {
  for (int k = 0; k < kBoardSlots; ++k) {
    const int bi = (det->slot_rr + k) % kBoardSlots;
    if (!det->hpend[bi].live || det->hpend[bi].seq > upto) continue;
    int rc = collect_host_slot(det, bi);
    if (rc) return rc;
  }
  return AG_OK;
}

int quiesce_device_path(ag_detector* det, bool host_too) {
  if (host_too) {
    int rc = collect_host(det, det->host_seq);
    if (rc) return rc;
  }
  if (!det->device_path_busy) return AG_OK;
  for (auto& D : det->dense)
    if (D.done) AG_CUDA(det, cudaEventSynchronize(D.done));
  for (auto& B : det->bslot)
    if (B.pending) {
      AG_CUDA(det, cudaEventSynchronize(B.ev_boards));
      B.pending = false;
    }
  det->device_path_busy = false;
  return AG_OK;
}

void rochade_tables_host(float cone[25], float pinv[150]) {
  // cone kernel, src/detector.rs:240-254 (half_size_patch = 2)
  const float gamma = 2.0f;
  for (int i = 0; i < 5; ++i)
    for (int j = 0; j < 5; ++j) {
      volatile float a = (gamma - (float)i) * (gamma - (float)i);
      volatile float b = (gamma - (float)j) * (gamma - (float)j);
      volatile float s = a + b;
      float v = gamma + 1.0f - sqrtf(s);
      cone[i * 5 + j] = v > 0.0f ? v : 0.0f;
    }
  volatile float sum = 0.0f;
  for (int i = 0; i < 25; ++i) sum = sum + cone[i];
  for (int i = 0; i < 25; ++i) cone[i] = cone[i] / sum;
  // Pseudo-inverse of the 25x6 design matrix [x^2, xy, y^2, x, y, 1], x, y in -2..2
  // (src/detector.rs:208-237 obtains it with an f32 QR).  On the symmetric grid the normal
  // equations decouple: with S2 = sum x^2 = 10, S4 = sum x^4 = 34 per axis and N = 5,
  //   a_xx = (x^2 - S2/N) / (N S4 - S2^2)            = (x^2 - 2) / 70
  //   a_xy = x y / S2^2                              = x y / 100
  //   a_x  = x / (N S2)                              = x / 50
  //   a_1  = (1 - N S2 (a_xx + a_yy)) / N^2          = (27 - 5 (x^2 + y^2)) / 175
  int idx = 0;
  for (int r = 0; r < 5; ++r)
    for (int c = 0; c < 5; ++c, ++idx) {
      const double x = c - 2, y = r - 2;
      const double p1 = (x * x - 2.0) / 70.0, p3 = (y * y - 2.0) / 70.0;
      pinv[0 * 25 + idx] = (float)p1;
      pinv[1 * 25 + idx] = (float)(x * y / 100.0);
      pinv[2 * 25 + idx] = (float)p3;
      pinv[3 * 25 + idx] = (float)(x / 50.0);
      pinv[4 * 25 + idx] = (float)(y / 50.0);
      pinv[5 * 25 + idx] = (float)((1.0 - 50.0 * (p1 + p3)) / 25.0);
    }
}

// Host copy-out of one chunk's results from a board slot's pinned staging.
void copy_out_b(const BoardSlot& B, int n, int cap, ag_tag* out, int* n_per_frame, uint32_t* frame_status,
                int frame0, bool* truncated) {
  for (int i = 0; i < n; ++i) {
    const int cnt = B.h_ntags[i];
    n_per_frame[frame0 + i] = cnt;
    if (cnt > cap) *truncated = true;
    const int m = std::min(cnt, cap);
    memcpy(out + (size_t)(frame0 + i) * cap, B.h_tags + (size_t)i * B.hs_tags, sizeof(ag_tag) * m);
    if (frame_status) frame_status[frame0 + i] = B.h_status[i];
  }
}

// What a synchronous host call / a wait reports after its chunks were collected.
int host_call_verdict(ag_detector* det) {
  const bool trunc = det->host_truncated, unres = det->host_unresolved;
  det->host_truncated = det->host_unresolved = false;
  if (unres)
    return fail(det, AG_ERR_CAPACITY,
                "a frame exceeds the detector's limits (clusters > 2^22, saddles > 16384 or a board wider than "
                "the +-31 tag lattice): its result is truncated, see frame_status");
  if (trunc) return fail(det, AG_ERR_CAPACITY, "cap_per_frame too small for at least one frame");
  return AG_OK;
}

}  // namespace

// =========================================================================================
extern "C" {

const char* ag_version(void) { return "aprilgrid-b200 0.1.0 (sm_100a)"; }

void ag_default_params(ag_params* out) {
  if (!out) return;
  out->tag_spacing_ratio = 0.3f;
  out->min_saddle_angle = 30.0f;
  out->max_saddle_angle = 60.0f;
  out->max_num_of_boards = 2;
}

int ag_family_from_str(const char* name, int* family_out) {
  if (!name || !family_out) return AG_ERR_INVALID;
  static const struct { const char* n; int f; } tab[] = {
      {"t16h5", AG_T16H5},   {"T16H5", AG_T16H5},   {"t25h7", AG_T25H7},      {"T25H7", AG_T25H7},
      {"t25h9", AG_T25H9},   {"T25H9", AG_T25H9},   {"t36h11", AG_T36H11},    {"T36H11", AG_T36H11},
      {"t36h11b1", AG_T36H11B1}, {"T36H11B1", AG_T36H11B1}};
  for (auto& e : tab)
    if (strcmp(name, e.n) == 0) {
      *family_out = e.f;
      return AG_OK;
    }
  return AG_ERR_INVALID;
}

int ag_family_info(int family, int* edge, int* border, int* hamming, int* n_codes,
                   const uint64_t** codes) {
  FamilyInfo f;
  if (!family_info(family, &f)) return AG_ERR_INVALID;
  if (edge) *edge = f.edge;
  if (border) *border = f.border;
  if (hamming) *hamming = f.hamming;
  if (n_codes) *n_codes = f.n_codes;
  if (codes) *codes = f.codes;
  return AG_OK;
}

const char* ag_last_error(const ag_detector* det) {
  return det ? det->err.c_str() : g_create_error.c_str();
}

int ag_create(int family, const ag_params* params, int device, ag_detector** out) {
  if (!out) return AG_ERR_INVALID;
  *out = nullptr;
  FamilyInfo fam;
  if (!family_info(family, &fam)) {
    g_create_error = "unknown tag family";
    return AG_ERR_INVALID;
  }
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev <= 0) {
    g_create_error = std::string("no CUDA device: ") + cudaGetErrorString(e) +
                     " (this library has no CPU path)";
    return AG_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n_dev) {
    g_create_error = "device ordinal out of range";
    return AG_ERR_INVALID;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess || prop.major != 10) {
    g_create_error = "device is not an sm_100 (Blackwell B200) part; kernels are built for sm_100a only";
    return AG_ERR_NO_DEVICE;
  }
  ag_detector* det = new ag_detector();
  det->device = device;
  det->family = family;
  det->fam = fam;
  if (params) det->params = *params;
  else ag_default_params(&det->params);
  if (cudaSetDevice(device) != cudaSuccess) {
    g_create_error = "cudaSetDevice failed";
    delete det;
    return AG_ERR_CUDA;
  }
  float cone[25], pinv[150];
  rochade_tables_host(cone, pinv);
  if (upload_rochade_tables(cone, pinv) != 0 ||
      cudaMalloc((void**)&det->d_codes, sizeof(uint64_t) * fam.n_codes) != cudaSuccess ||
      cudaMemcpy(det->d_codes, fam.codes, sizeof(uint64_t) * fam.n_codes, cudaMemcpyHostToDevice) !=
          cudaSuccess) {
    g_create_error = std::string("table upload failed: ") + cudaGetErrorString(cudaGetLastError());
    delete det;
    return AG_ERR_CUDA;
  }
  *out = det;
  return AG_OK;
}

void ag_destroy(ag_detector* det) {
  if (!det) return;
  cudaSetDevice(det->device);
  cudaDeviceSynchronize();
  for (auto& D : det->dense) free_slot(D);
  if (det->sparse_stream) cudaStreamDestroy(det->sparse_stream);
  free_slot(det->big);
  for (auto& B : det->bslot) free_board_slot(B);
  if (det->up_stream) cudaStreamDestroy(det->up_stream);
  for (auto e : det->ev_pool) cudaEventDestroy(e);
  cudaFree(det->d_codes);
  cudaFree(det->d_f32_a); cudaFree(det->d_f32_b); cudaFree(det->d_f32_c); cudaFree(det->d_taps);
  delete det;
}

int ag_set_option(ag_detector* det, const char* key, long value) {
  if (!det || !key) return AG_ERR_INVALID;
  std::lock_guard<std::mutex> lk(det->mu);
  if (!strcmp(key, "chunk_frames")) {
    if (value < 1 || value > 65535) return fail(det, AG_ERR_INVALID, "chunk_frames out of range");
    det->chunk_frames = value;
  } else if (!strcmp(key, "host_chunk_frames")) {
    if (value < 1 || value > 65535) return fail(det, AG_ERR_INVALID, "host_chunk_frames out of range");
    det->host_chunk_frames = value;
  } else if (!strcmp(key, "max_clusters")) {
    if (value != 0 && (value < 16 || value > (1 << 22))) return fail(det, AG_ERR_INVALID, "max_clusters out of range (0 = automatic)");
    det->max_clusters = value;
  } else if (!strcmp(key, "max_saddles")) {
    if (value != 0 && (value < 16 || value > 16384)) return fail(det, AG_ERR_INVALID, "max_saddles out of range (0 = automatic)");
    det->max_saddles = value;
  } else if (!strcmp(key, "dense_variant")) {
    det->dense_variant = value;
  } else if (!strcmp(key, "k1_chunk_rows")) {
    if (value != 0 && (value < 4 || value > 65536 || (value + 8) % 6 != 0))
      return fail(det, AG_ERR_INVALID, "k1_chunk_rows must be 0 or 6k + 4");
    det->k1_chunk_rows = value;
  } else if (!strcmp(key, "board_lattice")) {
    if (value != 16 && value != 32 && value != 64) return fail(det, AG_ERR_INVALID, "board_lattice must be 16, 32 or 64");
    det->board_lattice = value;

  } else if (!strcmp(key, "board_warps")) {
    if (value != 0 && value != 1 && value != 2 && value != 4 && value != 8 && value != 16)
      return fail(det, AG_ERR_INVALID, "board_warps must be 0 (auto), 1, 2, 4, 8 or 16");
    det->board_warps = value;
  } else if (!strcmp(key, "device_async")) {
    det->device_async = value != 0;
  } else if (!strcmp(key, "host_async")) {
    det->host_async = value != 0;
  } else if (!strcmp(key, "board_batch_frames")) {
    if (value < 1) return fail(det, AG_ERR_INVALID, "board_batch_frames must be positive");
    det->board_batch_frames = value;
#ifdef AG_EXPERIMENTS  // occupancy experiments only (tools/build_variant.sh); not in the shipped library
  } else if (!strcmp(key, "board_smem_pad")) {
    ag::g_board_smem_pad = (int)value;
#endif
  } else if (!strcmp(key, "label_variant")) {
    if (value < 0 || value > 1) return fail(det, AG_ERR_INVALID, "label_variant must be 0 or 1");
    det->label_variant = value;
  } else if (!strcmp(key, "board_saddle_tier")) {
    if (value < -1 || value > 2) return fail(det, AG_ERR_INVALID, "board_saddle_tier must be -1, 0 (512), 1 (1024) or 2 (4096)");
    det->board_saddle_tier = value;
  } else if (!strcmp(key, "board_timing")) {
    det->board_timing = value != 0;
  } else if (!strcmp(key, "board_fast")) {
    det->board_fast = value != 0;
  } else if (!strcmp(key, "board_priority")) {  // takes effect for board streams created afterwards
    det->board_priority = value != 0;
  } else if (!strcmp(key, "board_split")) {
    det->board_split = value != 0;
  } else if (!strcmp(key, "board_grid")) {
    det->board_grid = value != 0;
  } else if (!strcmp(key, "profile")) {
    det->profile = value != 0;
  } else {
    return fail(det, AG_ERR_INVALID, "unknown option");
  }
  return AG_OK;
}

uint64_t ag_launch_count(const ag_detector* det) { return det ? det->launches : 0; }

int ag_stage_times(ag_detector* det, double* ms_out, uint64_t* n_out, int reset) {
  if (!det) return AG_ERR_INVALID;
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  AG_CUDA(det, cudaDeviceSynchronize());
  for (size_t i = 1; i < det->ev_used; ++i) {
    int st = det->ev_stage[i];
    if (st < 0 || st >= 8) continue;
    float ms = 0.0f;
    if (cudaEventElapsedTime(&ms, det->ev_pool[i - 1], det->ev_pool[i]) == cudaSuccess) {
      det->stage_ms[st] += ms;
      det->stage_n[st] += 1;
    }
  }
  det->ev_used = 0;
  for (int i = 0; i < 8; ++i) {
    if (ms_out) ms_out[i] = det->stage_ms[i];
    if (n_out) n_out[i] = det->stage_n[i];
    if (reset) {
      det->stage_ms[i] = 0;
      det->stage_n[i] = 0;
    }
  }
  return AG_OK;
}

int ag_detect_batch_device(ag_detector* det, const void* d_frames, size_t frame_stride, int n_frames,
                           int width, int height, size_t row_stride, int format, ag_tag* d_out,
                           int cap_per_frame, int* d_n_per_frame, uint32_t* d_frame_status,
                           void* stream) {
  if (!det) return AG_ERR_INVALID;
  if (!d_frames || !d_out || !d_n_per_frame || n_frames < 0 || cap_per_frame < 1)
    return fail(det, AG_ERR_INVALID, "null pointer or bad count");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  FrameGeom g;
  int rc = make_geom(det, width, height, row_stride, frame_stride, format, &g);
  if (rc) return rc;
  if ((uintptr_t)d_frames % channel_align(format))
    return fail(det, AG_ERR_INVALID, "device frames must start at a multiple of the format's channel word");
  // chunks of host-buffer calls still in flight share the dense buffers and the board slots:
  // hand their results out first (streaming host calls and device calls do not overlap)
  if ((rc = collect_host(det, det->host_seq))) return rc;
  set_caps(det, g);
  const int chunk = chunk_limit(det, g, std::min<long>(det->chunk_frames, std::max(n_frames, 1)));
  // The ring of dense sets (K1-K2 on stream s, K3-K4 on the sparse stream, see run_front),
  // kBoardSlots board-search sides: chunk i's K6 runs on its board slot's own stream, so the
  // searches of up to kBoardSlots chunks (of this call and of earlier calls) overlap each other
  // and the front end of the following chunks.
  if ((rc = ensure_ring(det, g, chunk))) return rc;
  cudaStream_t s = stream ? (cudaStream_t)stream : det->dense[0].stream;
  // all board slots are sized up front: an allocation (which synchronises the device) must not
  // happen in the middle of a streaming sequence of calls
  for (auto& B : det->bslot)
    if ((rc = ensure_board_slot(det, B, chunk, false))) return rc;
  for (int f0 = 0; f0 < n_frames; f0 += chunk) {
    BoardSlot& B = det->bslot[det->slot_rr];
    det->slot_rr = (det->slot_rr + 1) % kBoardSlots;
    if ((rc = ensure_board_slot(det, B, chunk, false))) return rc;
    const int n = std::min(chunk, n_frames - f0);
    const uint8_t* in = (const uint8_t*)d_frames + (size_t)f0 * g.frame_stride;
    uint32_t* st = d_frame_status ? d_frame_status + f0 : B.d_status;
    if ((rc = run_front(det, B, in, g, n, st, s))) return rc;
    AG_CUDA(det, cudaStreamWaitEvent(B.bstream, B.ev_front, 0));
    if ((rc = run_boards(det, B, in, g, n, d_out + (size_t)f0 * cap_per_frame, cap_per_frame,
                         d_n_per_frame + f0, st, false, B.bstream)))
      return rc;
    AG_CUDA(det, cudaEventRecord(B.ev_boards, B.bstream));
    B.pending = true;
  }
  det->device_path_busy = true;
  // results become visible in the caller's stream order (unless the caller asked to do that
  // itself with ag_detect_batch_device_wait, which lets consecutive calls overlap)
  if (!det->device_async)
    for (auto& B : det->bslot)
      if (B.pending) AG_CUDA(det, cudaStreamWaitEvent(s, B.ev_boards, 0));
  return AG_OK;
}

int ag_detect_batch_device_wait(ag_detector* det, void* stream) {
  if (!det) return AG_ERR_INVALID;
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  for (auto& B : det->bslot) {
    if (!B.pending) continue;
    if (stream) AG_CUDA(det, cudaStreamWaitEvent((cudaStream_t)stream, B.ev_boards, 0));
    else AG_CUDA(det, cudaEventSynchronize(B.ev_boards));
  }
  return AG_OK;
}

int ag_dense_batch_device(ag_detector* det, const void* d_frames, size_t frame_stride, int n_frames,
                          int width, int height, size_t row_stride, int format, void* stream) {
  if (!det) return AG_ERR_INVALID;
  if (!d_frames || n_frames < 0) return fail(det, AG_ERR_INVALID, "null pointer or bad count");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  { int qrc = quiesce_device_path(det); if (qrc) return qrc; }
  FrameGeom g;
  int rc = make_geom(det, width, height, row_stride, frame_stride, format, &g);
  if (rc) return rc;
  if ((uintptr_t)d_frames % channel_align(format))
    return fail(det, AG_ERR_INVALID, "device frames must start at a multiple of the format's channel word");
  Slot& S = det->dense[0];
  set_caps(det, g);
  const int chunk = chunk_limit(det, g, std::min<long>(det->chunk_frames, std::max(n_frames, 1)));
  if ((rc = ensure_slot(det, S, g, chunk, false))) return rc;
  cudaStream_t s = stream ? (cudaStream_t)stream : S.stream;
  for (int f0 = 0; f0 < n_frames; f0 += chunk) {
    const int n = std::min(chunk, n_frames - f0);
    const uint8_t* in = (const uint8_t*)d_frames + (size_t)f0 * g.frame_stride;
    if ((rc = run_dense(det, S, in, g, n, true, s))) return rc;
  }
  // later calls on this handle (any stream) order themselves after this one through the dense slot's event
  AG_CUDA(det, cudaEventRecord(S.done, s));
  det->device_path_busy = true;
  return AG_OK;
}

// ag_detect_batch proper.  async_call: return once the chunks are enqueued (streaming use, option
// host_async); otherwise the results are in the output arrays when the call returns.
static int detect_batch_host(ag_detector* det, const void* frames, size_t frame_stride, int n_frames, int width,
                             int height, size_t row_stride, int format, ag_tag* out, int cap_per_frame,
                             int* n_per_frame, uint32_t* frame_status, bool async_call) {
  if (!det) return AG_ERR_INVALID;
  if (!frames || !out || !n_per_frame || n_frames < 0 || cap_per_frame < 1)
    return fail(det, AG_ERR_INVALID, "null pointer or bad count");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  // streaming calls leave the chunks of earlier calls in flight; a synchronous call first hands
  // out everything that is still pending (to the output arrays of the calls that submitted it)
  { int qrc = quiesce_device_path(det, !async_call); if (qrc) return qrc; }
  FrameGeom g;
  int rc = make_geom(det, width, height, row_stride, frame_stride, format, &g);
  if (rc) return rc;
  const uint64_t seq = ++det->host_seq;
  if (n_frames == 0) return async_call ? AG_OK : host_call_verdict(det);
  set_caps(det, g);
  // Host frames go through the same pipeline as device-resident ones: the ring of dense sets,
  // eight board slots.  A chunk is uploaded on the upload stream (ahead of the kernels), K1-K2
  // run on the dense stream, K3-K4 on the sparse stream, K6 and the download of the results on
  // the board slot's stream, so uploads, front end, board searches and downloads of up to eight
  // chunks overlap.  The staged input of a chunk stays in its board slot until K6 (which samples
  // the tag bits) is done.
  const int chunk = chunk_limit(
      det, g, std::min<long>(std::min<long>(det->chunk_frames, host_chunk_for(det->host_chunk_frames, format)), n_frames));
  if ((rc = ensure_ring(det, g, chunk))) return rc;
  if (!det->up_stream) AG_CUDA(det, cudaStreamCreateWithFlags(&det->up_stream, cudaStreamNonBlocking));
  cudaStream_t s = det->dense[0].stream, up = det->up_stream;
  const size_t chunk_bytes = (size_t)chunk * g.frame_stride;
  const bool pageable = is_pageable(frames);
  // Chunk schedule: the pipeline fills while the first chunk uploads and drains while the last one
  // is searched, so a large batch starts and ends with quarter and half chunks.
  auto next_chunk = [&](int f0) {
    const int left = n_frames - f0;
    if (n_frames < 4 * chunk || async_call) return std::min(chunk, left);  // streaming: no fill / drain
    if (f0 == 0) return chunk / 4 > 0 ? chunk / 4 : 1;
    if (f0 < chunk) return std::min(chunk / 2 > 0 ? chunk / 2 : 1, left);
    if (left <= chunk / 4) return left;
    if (left <= chunk / 4 + chunk / 2) return std::min(left - chunk / 4 > 0 ? left - chunk / 4 : left, left);
    if (left < chunk + chunk / 4 + chunk / 2) return left - (chunk / 4 + chunk / 2);
    return chunk;
  };
  for (int f0 = 0, n_this = 0; f0 < n_frames; f0 += n_this) {
    n_this = next_chunk(f0);
    const int bi = det->slot_rr;
    BoardSlot& B = det->bslot[bi];
    det->slot_rr = (det->slot_rr + 1) % kBoardSlots;
    // the slot's previous chunk (of this call or an earlier one): wait for its results, hand them out
    if ((rc = collect_host_slot(det, bi))) return rc;
    if ((rc = ensure_board_slot(det, B, chunk, true))) return rc;
    if ((rc = ensure_host_stage(det, B, chunk_bytes, chunk, cap_per_frame))) return rc;
    const int n = n_this;
    const uint8_t* src = (const uint8_t*)frames + (size_t)f0 * g.frame_stride;
    const size_t bytes = (size_t)(n - 1) * g.frame_stride + frame_bytes(g);
    const uint8_t* up_src = src;
    if (pageable) {  // (the slot's previous upload is long done: its chunk has been collected)
      if (chunk_bytes > B.cap_h_in) {
        if (B.h_in) cudaFreeHost(B.h_in);
        B.h_in = nullptr;
        B.cap_h_in = 0;
        AG_CUDA(det, cudaMallocHost((void**)&B.h_in, chunk_bytes));
        B.cap_h_in = chunk_bytes;
      }
      parallel_copy(B.h_in, src, bytes);
      up_src = B.h_in;
    }
    AG_CUDA(det, cudaMemcpyAsync(B.d_in, up_src, bytes, cudaMemcpyHostToDevice, up));
    AG_CUDA(det, cudaEventRecord(B.ev_up, up));
    AG_CUDA(det, cudaStreamWaitEvent(s, B.ev_up, 0));
    if ((rc = run_front(det, B, B.d_in, g, n, B.d_status, s))) return rc;
    AG_CUDA(det, cudaStreamWaitEvent(B.bstream, B.ev_front, 0));
    if ((rc = run_boards(det, B, B.d_in, g, n, B.d_tags, B.hs_tags, B.d_ntags, B.d_status, false, B.bstream)))
      return rc;
    // the same events the device-batch path orders itself by: a later device call (or a quiesce)
    // sees this chunk's board kernel and front end like one of its own
    AG_CUDA(det, cudaEventRecord(B.ev_boards, B.bstream));
    AG_CUDA(det, cudaMemcpyAsync(B.h_ntags, B.d_ntags, sizeof(int) * n, cudaMemcpyDeviceToHost, B.bstream));
    AG_CUDA(det, cudaMemcpyAsync(B.h_status, B.d_status, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost,
                                 B.bstream));
    AG_CUDA(det, cudaMemcpyAsync(B.h_tags, B.d_tags, sizeof(ag_tag) * (size_t)n * B.hs_tags,
                                 cudaMemcpyDeviceToHost, B.bstream));
    AG_CUDA(det, cudaEventRecord(B.ev_done, B.bstream));
    B.pending = true;
    auto& P = det->hpend[bi];
    P.live = true;
    P.f0 = f0;
    P.n = n;
    P.cap = cap_per_frame;
    P.seq = seq;
    P.out = out;
    P.n_per_frame = n_per_frame;
    P.status = frame_status;
    P.src = src;
    P.g = g;
  }
  // (a later device-batch call first collects these chunks -- it blocks until they are done -- so
  // the host path needs no busy flag of its own; streaming host calls must not drain each other)
  if (async_call) return AG_OK;  // results are collected by later calls / ag_detect_batch_wait
  if ((rc = collect_host(det, seq))) return rc;
  return host_call_verdict(det);
}

int ag_detect_batch(ag_detector* det, const void* frames, size_t frame_stride, int n_frames, int width,
                    int height, size_t row_stride, int format, ag_tag* out, int cap_per_frame,
                    int* n_per_frame, uint32_t* frame_status) {
  return detect_batch_host(det, frames, frame_stride, n_frames, width, height, row_stride, format, out,
                           cap_per_frame, n_per_frame, frame_status, det ? det->host_async : false);
}

int ag_detect_batch_wait(ag_detector* det, int keep_in_flight) {
  if (!det) return AG_ERR_INVALID;
  if (keep_in_flight < 0) return fail(det, AG_ERR_INVALID, "keep_in_flight must be >= 0");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  if ((uint64_t)keep_in_flight >= det->host_seq) return AG_OK;
  int rc = collect_host(det, det->host_seq - (uint64_t)keep_in_flight);
  if (rc) return rc;
  return host_call_verdict(det);
}

// TagDetector::detect: ALWAYS synchronous (its output arrays usually live on the caller's stack),
// whatever the streaming option of the handle says; chunks of streaming calls that are still in
// flight are handed to their own output arrays first.
int ag_detect(ag_detector* det, const void* pixels, int width, int height, size_t row_stride,
              int format, ag_tag* out, int cap, int* n) {
  if (!n) return det ? fail(det, AG_ERR_INVALID, "n is null") : AG_ERR_INVALID;
  int cnt = 0;
  int rc = detect_batch_host(det, pixels, 0, 1, width, height, row_stride, format, out, cap, &cnt, nullptr,
                             false);
  *n = cnt;
  return rc;
}

// detect on a frame given as the two gray planes the reference derives from its DynamicImage:
// luma32f = img.to_luma32f() (the stencil chain, detector.rs:409) and luma8 = img.to_luma8() (bit
// sampling, :507).  One frame, synchronous, on the one-frame slot; capacities grow as in ag_detect.
int ag_detect_planes(ag_detector* det, const float* luma32f, size_t f32_row_stride, const uint8_t* luma8,
                     size_t u8_row_stride, int width, int height, ag_tag* out, int cap, int* n) {
  if (!det) return AG_ERR_INVALID;
  if (!luma32f || !luma8 || !out || !n || cap < 1 || width <= 0 || height <= 0)
    return fail(det, AG_ERR_INVALID, "null pointer or bad size");
  if ((long long)width * height > (1ll << 30)) return fail(det, AG_ERR_INVALID, "image too large");
  if (f32_row_stride == 0) f32_row_stride = sizeof(float) * (size_t)width;
  if (u8_row_stride == 0) u8_row_stride = (size_t)width;
  if (f32_row_stride < sizeof(float) * (size_t)width || (f32_row_stride & 3) || u8_row_stride < (size_t)width)
    return fail(det, AG_ERR_INVALID, "bad row stride");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  const size_t px = (size_t)width * height;
  FrameGeom gf;  // the f32 plane, packed
  gf.w = width; gf.h = height; gf.wpr = (width + 31) / 32; gf.n_words = gf.wpr * height; gf.n_px = width * height;
  gf.row_stride = sizeof(float) * (size_t)width;
  gf.frame_stride = 5 * px;  // the u8 plane follows the f32 plane in the slot's input buffer
  gf.format = kFmtF32;
  FrameGeom g8 = gf;  // the u8 plane
  g8.row_stride = (size_t)width;
  g8.format = AG_L8;
  set_caps(det, gf);
  auto upload = [&](uint8_t* d_in, cudaStream_t s) {
    const cudaError_t e = cudaMemcpy2DAsync(d_in, gf.row_stride, luma32f, f32_row_stride, gf.row_stride, height,
                                            cudaMemcpyHostToDevice, s);
    return e != cudaSuccess ? e
                            : cudaMemcpy2DAsync(d_in + 4 * px, g8.row_stride, luma8, u8_row_stride, g8.row_stride,
                                                height, cudaMemcpyHostToDevice, s);
  };
  int cnt = 0;
  uint32_t st = 0;
  const int rc = run_one_frame(det, gf, g8, 4 * px, upload, FrameRun::kTags, 0, &cnt, &st);
  if (rc) return rc;
  const BoardSlot& B = det->big.bb;
  *n = cnt;
  memcpy(out, B.h_tags, sizeof(ag_tag) * (size_t)std::min(std::min(cnt, cap), B.hs_tags));
  if (st & (kGrowable | AG_FRAME_BOARD_OVERFLOW))
    return fail(det, AG_ERR_CAPACITY, "frame exceeds the detector's limits (clusters > 2^22, saddles > 16384 or a board wider than the lattice)");
  return cnt > cap ? fail(det, AG_ERR_CAPACITY, "cap too small") : AG_OK;
}

// ---- stage taps -----------------------------------------------------------------------------
int ag_stage_run(ag_detector* det, const void* pixels, int width, int height, size_t row_stride,
                 int format) {
  if (!det) return AG_ERR_INVALID;
  if (!pixels) return fail(det, AG_ERR_INVALID, "pixels is null");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  det->tap_valid = false;
  FrameGeom g;
  int rc = make_geom(det, width, height, row_stride, 0, format, &g);
  if (rc) return rc;
  set_caps(det, g);
  auto upload = [&](uint8_t* d_in, cudaStream_t s) {
    return cudaMemcpyAsync(d_in, pixels, frame_bytes(g), cudaMemcpyHostToDevice, s);
  };
  int cnt = 0;
  uint32_t st = 0;
  if ((rc = run_one_frame(det, g, g, 0, upload, FrameRun::kTaps, 0, &cnt, &st))) return rc;
  det->tap_geom = g;
  det->tap_valid = true;
  return AG_OK;
}

#define AG_TAP_PROLOGUE()                                                         \
  if (!det) return AG_ERR_INVALID;                                                \
  std::lock_guard<std::mutex> lk(det->mu);                                        \
  if (!det->tap_valid) return fail(det, AG_ERR_INVALID, "call ag_stage_run first"); \
  AG_CUDA(det, cudaSetDevice(det->device));                                       \
  Slot& S = det->big;                                                             \
  const FrameGeom& g = det->tap_geom;                                             \
  (void)g;

int ag_stage_blur(ag_detector* det, float* out) {
  AG_TAP_PROLOGUE();
  AG_CUDA(det, cudaMemcpy(out, S.d_blur, sizeof(float) * g.n_px, cudaMemcpyDeviceToHost));
  return AG_OK;
}
int ag_stage_response(ag_detector* det, float* out) {
  AG_TAP_PROLOGUE();
  AG_CUDA(det, cudaMemcpy(out, S.d_resp, sizeof(float) * g.n_px, cudaMemcpyDeviceToHost));
  return AG_OK;
}
int ag_stage_threshold(ag_detector* det, float* min_and_thr) {
  AG_TAP_PROLOGUE();
  uint32_t k;
  AG_CUDA(det, cudaMemcpy(&k, S.d_min, sizeof(k), cudaMemcpyDeviceToHost));
  float m = ordered_to_float(k);
  volatile float t = m * 0.05f;
  min_and_thr[0] = m;
  min_and_thr[1] = t;
  return AG_OK;
}
static int tap_labels(ag_detector* det, Slot& S, const FrameGeom& g, int32_t* labels, uint8_t* mask) {
  int32_t* d_lab = nullptr;
  uint8_t* d_m = nullptr;
  if (labels) AG_CUDA(det, cudaMalloc((void**)&d_lab, sizeof(int32_t) * g.n_px));
  if (mask) AG_CUDA(det, cudaMalloc((void**)&d_m, g.n_px));
  det->launches += launch_labels_tap(S.d_mask, g, S.d_parent, d_lab, d_m, S.stream);
  AG_CUDA(det, cudaStreamSynchronize(S.stream));
  if (labels) AG_CUDA(det, cudaMemcpy(labels, d_lab, sizeof(int32_t) * g.n_px, cudaMemcpyDeviceToHost));
  if (mask) AG_CUDA(det, cudaMemcpy(mask, d_m, g.n_px, cudaMemcpyDeviceToHost));
  cudaFree(d_lab);
  cudaFree(d_m);
  return AG_OK;
}
int ag_stage_mask(ag_detector* det, uint8_t* out) {
  AG_TAP_PROLOGUE();
  return tap_labels(det, S, g, nullptr, out);
}
int ag_stage_labels(ag_detector* det, int32_t* out) {
  AG_TAP_PROLOGUE();
  return tap_labels(det, S, g, out, nullptr);
}
int ag_stage_centers(ag_detector* det, float* xy_out, int cap, int* n) {
  AG_TAP_PROLOGUE();
  int cnt = 0;
  AG_CUDA(det, cudaMemcpy(&cnt, S.d_ncl, sizeof(int), cudaMemcpyDeviceToHost));
  *n = cnt;
  int m = std::min(cnt, cap);
  if (m > 0) AG_CUDA(det, cudaMemcpy(xy_out, S.d_centers, sizeof(float2) * m, cudaMemcpyDeviceToHost));
  return AG_OK;
}
int ag_stage_saddles(ag_detector* det, int which, ag_saddle* out, int cap, int* n) {
  AG_TAP_PROLOGUE();
  if (which == 1) {
    int cnt = 0;
    AG_CUDA(det, cudaMemcpy(&cnt, S.bb.d_nref, sizeof(int), cudaMemcpyDeviceToHost));
    *n = cnt;
    int m = std::min(cnt, cap);
    if (m > 0) AG_CUDA(det, cudaMemcpy(out, S.bb.d_refined, sizeof(ag_saddle) * m, cudaMemcpyDeviceToHost));
    return AG_OK;
  }
  int ncl = 0;
  AG_CUDA(det, cudaMemcpy(&ncl, S.d_ncl, sizeof(int), cudaMemcpyDeviceToHost));
  std::vector<ag_saddle> raw(std::max(ncl, 1));
  std::vector<uint8_t> valid(std::max(ncl, 1));
  if (ncl > 0) {
    AG_CUDA(det, cudaMemcpy(raw.data(), S.d_raw, sizeof(ag_saddle) * ncl, cudaMemcpyDeviceToHost));
    AG_CUDA(det, cudaMemcpy(valid.data(), S.d_raw_valid, ncl, cudaMemcpyDeviceToHost));
  }
  int cnt = 0;
  for (int i = 0; i < ncl; ++i)
    if (valid[i]) {
      if (cnt < cap) out[cnt] = raw[i];
      ++cnt;
    }
  *n = cnt;
  return AG_OK;
}
int ag_stage_board_quads(ag_detector* det, int32_t* quads_out, int cap, int* n) {
  AG_TAP_PROLOGUE();
  int cnt = 0;
  AG_CUDA(det, cudaMemcpy(&cnt, S.bb.d_tap_nquads, sizeof(int), cudaMemcpyDeviceToHost));
  *n = cnt;
  int m = std::min(std::min(cnt, cap), S.bb.layout[0].max_quads);
  if (m > 0) AG_CUDA(det, cudaMemcpy(quads_out, S.bb.d_tap_quads, sizeof(int32_t) * 4 * m, cudaMemcpyDeviceToHost));
  return AG_OK;
}
int ag_stage_tags(ag_detector* det, ag_tag* out, int cap, int* n) {
  AG_TAP_PROLOGUE();
  int cnt = 0;
  AG_CUDA(det, cudaMemcpy(&cnt, S.bb.d_ntags, sizeof(int), cudaMemcpyDeviceToHost));
  *n = cnt;
  int m = std::min(std::min(cnt, cap), S.bb.hs_tags);
  if (m > 0) AG_CUDA(det, cudaMemcpy(out, S.bb.d_tags, sizeof(ag_tag) * m, cudaMemcpyDeviceToHost));
  return AG_OK;
}

int ag_refined_saddle_points(ag_detector* det, const void* pixels, int width, int height,
                             size_t row_stride, int format, ag_saddle* out, int cap, int* n) {
  if (!det) return AG_ERR_INVALID;
  if (!pixels || !out || !n) return fail(det, AG_ERR_INVALID, "null pointer");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  FrameGeom g;
  int rc = make_geom(det, width, height, row_stride, 0, format, &g);
  if (rc) return rc;
  set_caps(det, g);
  auto upload = [&](uint8_t* d_in, cudaStream_t s) {
    return cudaMemcpyAsync(d_in, pixels, frame_bytes(g), cudaMemcpyHostToDevice, s);
  };
  int cnt = 0;
  uint32_t st = 0;
  if ((rc = run_one_frame(det, g, g, 0, upload, FrameRun::kSaddles, 0, &cnt, &st))) return rc;
  *n = cnt;
  int m = std::min(cnt, cap);
  if (m > 0) AG_CUDA(det, cudaMemcpy(out, det->big.bb.d_refined, sizeof(ag_saddle) * m, cudaMemcpyDeviceToHost));
  if (st & kGrowable) return fail(det, AG_ERR_CAPACITY, "frame exceeds the detector's limits (clusters > 2^22 or saddles > 16384)");
  return cnt > cap ? fail(det, AG_ERR_CAPACITY, "saddle capacity too small") : AG_OK;
}

// ---- standalone operators ---------------------------------------------------------------------
static int ensure_f32(ag_detector* det, size_t n) {
  if (n <= det->f32_cap) return AG_OK;
  int rc;
  if ((rc = regrow(det, &det->d_f32_a, n))) return rc;
  if ((rc = regrow(det, &det->d_f32_b, n))) return rc;
  if ((rc = regrow(det, &det->d_f32_c, n))) return rc;
  if (!det->d_taps && (rc = regrow(det, &det->d_taps, 256))) return rc;
  det->f32_cap = n;
  return AG_OK;
}

// taps exactly as src/image_util.rs:111-124 computes them at run time (platform expf)
static bool blur_taps_host(float sigma, std::vector<float>& taps, int& radius) {
  radius = (int)ceilf(sigma * 2.0f);
  if (!(sigma > 0.0f) || radius < 0 || radius > 100) return false;
  taps.assign(2 * radius + 1, 0.0f);
  volatile float two_sigma_sq = 2.0f * sigma * sigma;
  volatile float sum = 0.0f;
  for (int i = 0; i <= 2 * radius; ++i) {
    float x = (float)(i - radius);
    volatile float xx = x * x;
    float v = expf(-xx / two_sigma_sq);
    taps[i] = v;
    sum = sum + v;
  }
  for (auto& v : taps) v = v / sum;
  return true;
}

int ag_gaussian_blur_f32(ag_detector* det, const float* img, int width, int height, float sigma,
                         float* out) {
  if (!det) return AG_ERR_INVALID;
  if (!img || !out || width <= 0 || height <= 0) return fail(det, AG_ERR_INVALID, "bad argument");
  int radius = 0;
  std::vector<float> taps;
  if (!blur_taps_host(sigma, taps, radius)) return fail(det, AG_ERR_INVALID, "sigma out of range");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  { int qrc = quiesce_device_path(det); if (qrc) return qrc; }
  const size_t n = (size_t)width * height;
  int rc = ensure_f32(det, n);
  if (rc) return rc;
  Slot& S = det->dense[0];
  if (!S.stream) {
    AG_CUDA(det, cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
    AG_CUDA(det, cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
  }
  AG_CUDA(det, cudaMemcpyAsync(det->d_taps, taps.data(), sizeof(float) * taps.size(),
                               cudaMemcpyHostToDevice, S.stream));
  AG_CUDA(det, cudaMemcpyAsync(det->d_f32_a, img, sizeof(float) * n, cudaMemcpyHostToDevice, S.stream));
  det->launches += launch_blur_f32(det->d_f32_a, det->d_f32_b, det->d_f32_c, width, height, 1, taps.data(),
                                   det->d_taps, radius, S.stream);
  AG_CUDA(det, cudaGetLastError());
  AG_CUDA(det, cudaMemcpyAsync(out, det->d_f32_c, sizeof(float) * n, cudaMemcpyDeviceToHost, S.stream));
  AG_CUDA(det, cudaStreamSynchronize(S.stream));
  return AG_OK;
}

int ag_gaussian_blur_f32_device(ag_detector* det, const float* d_in, int n_frames, int width, int height,
                                float sigma, float* d_out, void* stream) {
  if (!det) return AG_ERR_INVALID;
  if (n_frames < 0 || width <= 0 || height <= 0 || (n_frames > 0 && (!d_in || !d_out || d_in == d_out)))
    return fail(det, AG_ERR_INVALID, "bad argument");
  int radius = 0;
  std::vector<float> taps;
  if (!blur_taps_host(sigma, taps, radius)) return fail(det, AG_ERR_INVALID, "sigma out of range");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  if (n_frames == 0) return AG_OK;
  const size_t n = (size_t)width * height;
  int rc = ensure_f32(det, n);  // scratch image + tap buffer of the general path
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  // the tap upload is synchronous with respect to the host (pageable source), ordered on s
  AG_CUDA(det, cudaMemcpyAsync(det->d_taps, taps.data(), sizeof(float) * taps.size(), cudaMemcpyHostToDevice, s));
  det->launches += launch_blur_f32(d_in, det->d_f32_b, d_out, width, height, n_frames, taps.data(), det->d_taps,
                                   radius, s);
  AG_CUDA(det, cudaGetLastError());
  return AG_OK;
}

int ag_hessian_response(ag_detector* det, const float* img, int width, int height, float* out) {
  if (!det) return AG_ERR_INVALID;
  if (!img || !out || width <= 0 || height <= 0) return fail(det, AG_ERR_INVALID, "bad argument");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  { int qrc = quiesce_device_path(det); if (qrc) return qrc; }
  const size_t n = (size_t)width * height;
  int rc = ensure_f32(det, n);
  if (rc) return rc;
  Slot& S = det->dense[0];
  if (!S.stream) {
    AG_CUDA(det, cudaStreamCreateWithFlags(&S.stream, cudaStreamNonBlocking));
    AG_CUDA(det, cudaEventCreateWithFlags(&S.done, cudaEventDisableTiming));
  }
  AG_CUDA(det, cudaMemcpyAsync(det->d_f32_a, img, sizeof(float) * n, cudaMemcpyHostToDevice, S.stream));
  det->launches += launch_hessian_f32(det->d_f32_a, det->d_f32_c, width, height, S.stream);
  AG_CUDA(det, cudaGetLastError());
  AG_CUDA(det, cudaMemcpyAsync(out, det->d_f32_c, sizeof(float) * n, cudaMemcpyDeviceToHost, S.stream));
  AG_CUDA(det, cudaStreamSynchronize(S.stream));
  return AG_OK;
}

int ag_render_boards_device(ag_detector* det, void* d_frames, int n_frames, int width, int height,
                            int cols, int rows, uint64_t seed, void* stream) {
  if (!det) return AG_ERR_INVALID;
  if (!d_frames || n_frames < 0 || width <= 0 || height <= 0 || cols < 1 || rows < 1)
    return fail(det, AG_ERR_INVALID, "bad argument");
  if (cols * rows > det->fam.n_codes) return fail(det, AG_ERR_INVALID, "board has more tags than the family has codes");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  if (n_frames == 0) return AG_OK;
  for (int f0 = 0; f0 < n_frames; f0 += 32768) {
    int n = std::min(32768, n_frames - f0);
    det->launches += launch_render_boards((uint8_t*)d_frames + (size_t)f0 * width * height, n, width,
                                          height, cols, rows, det->d_codes, det->fam.edge,
                                          det->fam.border, seed + (uint64_t)f0 * 0x51ed27ull, nullptr, 1,
                                          (cudaStream_t)stream);
  }
  AG_CUDA(det, cudaGetLastError());
  return AG_OK;
}

// Test hook (not in the public header; needs no GPU): the board kernel's shared-memory / workspace
// budget for a configuration, so that CPU tests can pin the residency the design counts on
// (seven 2-warp frames per SM in the 320-saddle tier, every tier within a block's 227 KB).
// out = {smem_per_block, bytes_per_frame, warps, smem_saddles}.
AG_API int ag_test_board_layout(int max_saddles, int lattice, int warps, int smem_saddles, int with_gpos,
                                int active_cap, long long out[4]) {
  if (!out || max_saddles < 1) return AG_ERR_INVALID;
  const BoardWsLayout L = make_board_layout(max_saddles, lattice, warps, smem_saddles, with_gpos != 0, active_cap);
  out[0] = (long long)L.smem_per_block;
  out[1] = (long long)L.bytes_per_frame;
  out[2] = L.warps;
  out[3] = L.smem_saddles;
  return AG_OK;
}

// Test hook (not in the public header; needs no GPU): the decode scratch of the board kernel for a
// configuration.  The bit patterns of the listed quads (8 bytes each) go to warp 0's seed-best values;
// out = {bytes of that region up to the next array of the warp, most quads a board can list}.
AG_API int ag_test_board_decode_room(int max_saddles, int lattice, int warps, long long out[2]) {
  if (!out || max_saddles < 1 || lattice < 1) return AG_ERR_INVALID;
  const BoardWsLayout L = make_board_layout(max_saddles, lattice, warps, max_saddles);
  out[0] = (long long)(L.woff_stack - L.woff_sb_vals);
  out[1] = std::min(L.max_quads, lattice * lattice);
  return AG_OK;
}

// Test hook (not in the public header; needs no GPU): the frames per chunk of the host-buffer path
// for a host_chunk_frames option and a pixel format, before the dense-buffer bound of chunk_limit.
AG_API int ag_test_host_chunk(long long host_chunk_frames, int format, long long* out) {
  if (!out || host_chunk_frames < 1 || format == kFmtF32 || bytes_per_px(format) == 0) return AG_ERR_INVALID;
  *out = host_chunk_for((long)host_chunk_frames, format);
  return AG_OK;
}

// Test hook (not in the public header): ONE frame of the renderer under a GIVEN pose -- hinv maps
// image (x, y, 1) to page coordinates in tag sides (row-major 3x3, host pointer) -- with or without
// the noise, so that tests can pin the renderer's geometry (id <-> lattice position, corner
// positions) against tests/synth.py and scripts/generate_aprilgrid.py:1114-1167.
AG_API int ag_test_render_pose(ag_detector* det, void* d_frame, int width, int height, int cols, int rows,
                               const float* hinv, int noise, uint64_t seed) {
  if (!det || !d_frame || !hinv || width <= 0 || height <= 0 || cols < 1 || rows < 1) return AG_ERR_INVALID;
  if (cols * rows > det->fam.n_codes) return fail(det, AG_ERR_INVALID, "board has more tags than the family has codes");
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  float* d_h = nullptr;
  AG_CUDA(det, cudaMalloc((void**)&d_h, sizeof(float) * 9));
  AG_CUDA(det, cudaMemcpy(d_h, hinv, sizeof(float) * 9, cudaMemcpyHostToDevice));
  det->launches += launch_render_boards((uint8_t*)d_frame, 1, width, height, cols, rows, det->d_codes, det->fam.edge,
                                        det->fam.border, seed, d_h, noise, 0);
  AG_CUDA(det, cudaDeviceSynchronize());
  cudaFree(d_h);
  return AG_OK;
}

// Test hook (not in the public header): the board search + decoding (K6) on GIVEN saddle lists over
// host frames -- so that tests can put saddles exactly on the gates of init_quads / is_valid_quad /
// the theta histogram, and frames exactly on the saddle counts where the launches of a batch and the
// on-chip tiers part.  Frame f has n_saddles[f] saddles at saddles + f * saddle_stride (records of
// {x, y, k, theta, phi}) and its pixels at pixels + f * frame_stride (0 = packed).  All n_frames go
// through ONE run_boards, so the handle's board options pick the launches as in the pipeline.
// Out, per frame: the quads of the first best board (quads_out + f * quad_cap * 4, n_quads[f] of
// them), tag_cap tag records (tags_out + f * tag_cap, n_tags[f] of them valid) and the status bits.
// Counts start at -1 and records at all-ones bytes: a frame that no launch took comes back so.
AG_API int ag_test_boards_from_saddles(ag_detector* det, const ag_saddle* saddles, size_t saddle_stride,
                                       const int* n_saddles, int n_frames, const void* pixels, size_t frame_stride,
                                       int width, int height, size_t row_stride, int format, int32_t* quads_out,
                                       int quad_cap, int* n_quads, ag_tag* tags_out, int tag_cap, int* n_tags,
                                       uint32_t* status) {
  if (!det || !saddles || !n_saddles || n_frames < 1 || !pixels || !quads_out || quad_cap < 0 || !n_quads ||
      !tags_out || tag_cap < 0 || !n_tags || !status)
    return AG_ERR_INVALID;
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  det->tap_valid = false;  // the taps read the one-frame slot's board side
  FrameGeom g;
  int rc = make_geom(det, width, height, row_stride, frame_stride, format, &g);
  if (rc) return rc;
  set_caps(det, g);
  int max_n = 0;
  for (int f = 0; f < n_frames; ++f) {
    if (n_saddles[f] < 0) return fail(det, AG_ERR_INVALID, "negative saddle count");
    max_n = std::max(max_n, n_saddles[f]);
  }
  if (max_n > det->cur_saddles) return fail(det, AG_ERR_INVALID, "more saddles than max_saddles");
  if ((size_t)max_n > saddle_stride) return fail(det, AG_ERR_INVALID, "saddle_stride smaller than a list");
  // the board side of the one-frame slot only: its dense buffers are not needed
  BoardSlot& B = det->big.bb;
  if ((rc = ensure_board_slot(det, B, n_frames, true)) ||
      (rc = ensure_host_stage(det, B, (size_t)n_frames * g.frame_stride, n_frames, det->fam.n_codes)))
    return rc;
  const cudaStream_t s = B.bstream;
  const int cap = B.hs_tags, mq = B.layout[0].max_quads;
  AG_CUDA(det, cudaMemcpyAsync(B.d_in, pixels, g.frame_stride * (size_t)(n_frames - 1) + frame_bytes(g),
                               cudaMemcpyHostToDevice, s));
  if (max_n > 0)
    AG_CUDA(det, cudaMemcpy2DAsync(B.d_refined, sizeof(ag_saddle) * (size_t)B.cap_saddles, saddles,
                                   sizeof(ag_saddle) * saddle_stride,
                                   sizeof(ag_saddle) * (size_t)max_n, n_frames, cudaMemcpyHostToDevice, s));
  AG_CUDA(det, cudaMemcpyAsync(B.d_nref, n_saddles, sizeof(int) * n_frames, cudaMemcpyHostToDevice, s));
  AG_CUDA(det, cudaMemsetAsync(B.d_status, 0, sizeof(uint32_t) * n_frames, s));
  AG_CUDA(det, cudaMemsetAsync(B.d_ntags, 0xff, sizeof(int) * n_frames, s));
  AG_CUDA(det, cudaMemsetAsync(B.d_tags, 0xff, sizeof(ag_tag) * (size_t)cap * n_frames, s));
  AG_CUDA(det, cudaMemsetAsync(B.d_tap_nquads, 0xff, sizeof(int) * n_frames, s));
  AG_CUDA(det, cudaMemsetAsync(B.d_tap_quads, 0xff, sizeof(int32_t) * 4 * (size_t)mq * n_frames, s));
  if ((rc = run_boards(det, B, B.d_in, g, n_frames, B.d_tags, cap, B.d_ntags, B.d_status, true, s))) return rc;
  AG_CUDA(det, cudaMemcpyAsync(n_quads, B.d_tap_nquads, sizeof(int) * n_frames, cudaMemcpyDeviceToHost, s));
  AG_CUDA(det, cudaMemcpyAsync(n_tags, B.d_ntags, sizeof(int) * n_frames, cudaMemcpyDeviceToHost, s));
  AG_CUDA(det, cudaMemcpyAsync(status, B.d_status, sizeof(uint32_t) * n_frames, cudaMemcpyDeviceToHost, s));
  const int kq = std::min(quad_cap, mq), kt = std::min(tag_cap, cap);
  if (kq > 0)
    AG_CUDA(det, cudaMemcpy2DAsync(quads_out, sizeof(int32_t) * 4 * (size_t)quad_cap, B.d_tap_quads,
                                   sizeof(int32_t) * 4 * (size_t)mq, sizeof(int32_t) * 4 * (size_t)kq, n_frames,
                                   cudaMemcpyDeviceToHost, s));
  if (kt > 0)
    AG_CUDA(det, cudaMemcpy2DAsync(tags_out, sizeof(ag_tag) * (size_t)tag_cap, B.d_tags, sizeof(ag_tag) * (size_t)cap,
                                   sizeof(ag_tag) * (size_t)kt, n_frames, cudaMemcpyDeviceToHost, s));
  AG_CUDA(det, cudaStreamSynchronize(s));
  return AG_OK;
}

// Profiling hook (not in the public header): per-frame timing taps of the last board-kernel launch
// on pipeline slot `slot` (needs ag_set_option("board_timing", 1)); out = n_frames x 16 u32.
AG_API int ag_test_board_times(ag_detector* det, int slot, uint32_t* out, int n_frames) {
  if (!det || slot < 0 || slot >= kBoardSlots || !out) return AG_ERR_INVALID;
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  BoardSlot& S = det->bslot[slot];
  if (!S.d_board_tm || n_frames > S.cap_frames) return fail(det, AG_ERR_INVALID, "no timing data");
  AG_CUDA(det, cudaDeviceSynchronize());
  AG_CUDA(det, cudaMemcpy(out, S.d_board_tm, sizeof(uint32_t) * 32 * (size_t)n_frames, cudaMemcpyDeviceToHost));
  return AG_OK;
}

// Test hook (not in the public header): exhaustive unorm conversion tables.
AG_API int ag_test_unorm_tables(ag_detector* det, float* out8, float* out16, float* ref8, float* ref16) {
  if (!det) return AG_ERR_INVALID;
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  float* d = nullptr;
  AG_CUDA(det, cudaMalloc((void**)&d, sizeof(float) * (256 + 65536) * 2));
  float *d8 = d, *d16 = d + 256, *r8 = d16 + 65536, *r16 = r8 + 256;
  det->launches += launch_unorm_table(d8, d16, r8, r16, 0);
  AG_CUDA(det, cudaDeviceSynchronize());
  AG_CUDA(det, cudaMemcpy(out8, d8, 256 * 4, cudaMemcpyDeviceToHost));
  AG_CUDA(det, cudaMemcpy(out16, d16, 65536 * 4, cudaMemcpyDeviceToHost));
  AG_CUDA(det, cudaMemcpy(ref8, r8, 256 * 4, cudaMemcpyDeviceToHost));
  AG_CUDA(det, cudaMemcpy(ref16, r16, 65536 * 4, cudaMemcpyDeviceToHost));
  cudaFree(d);
  return AG_OK;
}

// Test hook (not in the public header): the device's gray conversion of n float pixels (channels 3:
// R G B, 4: R G B A, host array) -> to_luma32f and to_luma8 of each (host arrays of n).
AG_API int ag_test_float_luma(ag_detector* det, const float* rgb, long long n, int channels, float* out_luma32f,
                              uint8_t* out_luma8) {
  if (!det || !rgb || !out_luma32f || !out_luma8 || n < 0 || (channels != 3 && channels != 4)) return AG_ERR_INVALID;
  if (n == 0) return AG_OK;
  std::lock_guard<std::mutex> lk(det->mu);
  AG_CUDA(det, cudaSetDevice(det->device));
  const size_t in_bytes = sizeof(float) * channels * (size_t)n, out_bytes = 5 * (size_t)n;
  uint8_t* d = nullptr;
  AG_CUDA(det, cudaMalloc((void**)&d, in_bytes + out_bytes));
  float* d_in = (float*)d;
  float* d_l32 = (float*)(d + in_bytes);
  uint8_t* d_l8 = d + in_bytes + 4 * (size_t)n;
  cudaError_t e = cudaMemcpy(d_in, rgb, in_bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    det->launches += launch_float_luma(d_in, n, channels, d_l32, d_l8, 0);
    e = cudaDeviceSynchronize();
  }
  if (e == cudaSuccess) e = cudaMemcpy(out_luma32f, d_l32, 4 * (size_t)n, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(out_luma8, d_l8, (size_t)n, cudaMemcpyDeviceToHost);
  cudaFree(d);
  AG_CUDA(det, e);
  return AG_OK;
}

// Page-locked host memory for callers that assemble batches themselves (a shim packing
// DynamicImages, a capture loop): frames written here are uploaded by the copy engine directly, at
// the link rate, without the staging copy ordinary (pageable) memory needs.
void* ag_host_alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0 || cudaMallocHost(&p, bytes) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  return p;
}
void ag_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

// ---- one detector over several GPUs ------------------------------------------------------------
// Frames are independent (TagDetector::detect is stateless, src/detector.rs:505-540): a batch is
// cut into contiguous frame ranges [g * B / G, (g + 1) * B / G), one per device, each range goes
// through that device's own pipeline on its own host thread, and every device writes its results
// straight into the caller's arrays at its frames' positions -- the "gather" is the placement.
struct ag_multi {
  std::vector<ag_detector*> dets;
  std::vector<double> h2d_gbs;  // host-to-device rate of each device, all devices copying at once
  std::string err;
};

// Pinned host -> device rate of every device of the set, measured with all of them copying at the
// same time (64 MB x 4 each).  The GPUs of a box do not all get the same share of the host's
// bandwidth, and a host-fed batch is as slow as its slowest shard.
static void measure_h2d_rates(ag_multi* m) {
  const int G = (int)m->dets.size();
  m->h2d_gbs.assign(G, 0.0);
  if (G < 2) return;
  const size_t bytes = 64u << 20;
  std::atomic<int> ready(0);
  std::vector<std::thread> th;
  for (int g = 0; g < G; ++g)
    th.emplace_back([&, g] {
      void *h = nullptr, *d = nullptr;
      cudaStream_t s = nullptr;
      cudaEvent_t e0 = nullptr, e1 = nullptr;
      bool ok = cudaSetDevice(m->dets[g]->device) == cudaSuccess && cudaMallocHost(&h, bytes) == cudaSuccess &&
                cudaMalloc(&d, bytes) == cudaSuccess && cudaStreamCreate(&s) == cudaSuccess &&
                cudaEventCreate(&e0) == cudaSuccess && cudaEventCreate(&e1) == cudaSuccess;
      if (ok) {
        memset(h, 1, bytes);
        ok = cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s) == cudaSuccess && cudaStreamSynchronize(s) == cudaSuccess;
      }
      ++ready;
      while (ready.load() < G) std::this_thread::yield();  // start together
      if (ok) {
        cudaEventRecord(e0, s);
        for (int i = 0; i < 4; ++i) cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s);
        cudaEventRecord(e1, s);
        float ms = 0.0f;
        if (cudaStreamSynchronize(s) == cudaSuccess && cudaEventElapsedTime(&ms, e0, e1) == cudaSuccess && ms > 0.0f)
          m->h2d_gbs[g] = 4.0 * (double)bytes / (ms * 1e-3) / 1e9;
      }
      if (e0) cudaEventDestroy(e0);
      if (e1) cudaEventDestroy(e1);
      if (s) cudaStreamDestroy(s);
      if (d) cudaFree(d);
      if (h) cudaFreeHost(h);
    });
  for (auto& t : th) t.join();
  cudaGetLastError();
}

int ag_multi_create(int family, const ag_params* params, const int* devices, int n_devices, ag_multi** out) {
  if (!out) return AG_ERR_INVALID;
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev <= 0) {
    g_create_error = "no CUDA device (this library has no CPU path)";
    return AG_ERR_NO_DEVICE;
  }
  std::vector<int> devs;
  if (devices && n_devices > 0) devs.assign(devices, devices + n_devices);
  else for (int d = 0; d < n_dev; ++d) devs.push_back(d);  // NULL / 0: every visible device
  ag_multi* m = new ag_multi();
  for (int d : devs) {
    ag_detector* det = nullptr;
    const int rc = ag_create(family, params, d, &det);
    if (rc != AG_OK) {
      for (auto* p : m->dets) ag_destroy(p);
      delete m;
      return rc;  // g_create_error holds the reason
    }
    m->dets.push_back(det);
  }
  // distinct devices only: two handles on one GPU (tests) share a link, equal shards are right there
  bool distinct = true;
  for (size_t i = 0; i < devs.size(); ++i)
    for (size_t j = 0; j < i; ++j) distinct = distinct && devs[i] != devs[j];
  if (distinct) measure_h2d_rates(m);
  else m->h2d_gbs.assign(devs.size(), 0.0);
  *out = m;
  return AG_OK;
}

void ag_multi_destroy(ag_multi* m) {
  if (!m) return;
  for (auto* d : m->dets) ag_destroy(d);
  delete m;
}

int ag_multi_device_count(const ag_multi* m) { return m ? (int)m->dets.size() : 0; }

const char* ag_multi_last_error(const ag_multi* m) { return m ? m->err.c_str() : g_create_error.c_str(); }

int ag_multi_set_option(ag_multi* m, const char* key, long value) {
  if (!m) return AG_ERR_INVALID;
  for (auto* d : m->dets) {
    const int rc = ag_set_option(d, key, value);
    if (rc != AG_OK) {
      m->err = ag_last_error(d);
      return rc;
    }
  }
  return AG_OK;
}

int ag_multi_detect_batch(ag_multi* m, const void* frames, size_t frame_stride, int n_frames, int width,
                          int height, size_t row_stride, int format, ag_tag* out, int cap_per_frame,
                          int* n_per_frame, uint32_t* frame_status) {
  if (!m || m->dets.empty()) return AG_ERR_INVALID;
  if (!frames || !out || !n_per_frame || n_frames < 0 || cap_per_frame < 1) {
    m->err = "null pointer or bad count";
    return AG_ERR_INVALID;
  }
  // the strides every shard's offsets are computed with (0 = tightly packed, as in ag_detect_batch)
  const size_t rs = row_stride ? row_stride : (size_t)(width > 0 ? width : 0) * bytes_per_px(format);
  const size_t fs = frame_stride ? frame_stride : rs * (size_t)(height > 0 ? height : 0);
  const int G = (int)m->dets.size();
  std::vector<int> rcs(G, AG_OK);
  // shard boundaries: equal ranges, or -- when the devices' measured host-to-device rates differ by
  // more than 5 % -- ranges in proportion to those rates
  std::vector<long long> bound(G + 1, 0);
  {
    double lo_r = 1e300, hi_r = 0.0, sum = 0.0;
    for (double r : m->h2d_gbs) { lo_r = std::min(lo_r, r); hi_r = std::max(hi_r, r); sum += r; }
    const bool weighted = (int)m->h2d_gbs.size() == G && lo_r > 0.0 && hi_r > 1.05 * lo_r;
    double acc = 0.0;
    for (int g = 0; g < G; ++g) {
      acc += weighted ? m->h2d_gbs[g] / sum : 1.0 / G;
      bound[g + 1] = g + 1 == G ? n_frames : std::min<long long>(n_frames, (long long)llround(acc * n_frames));
      if (bound[g + 1] < bound[g]) bound[g + 1] = bound[g];
    }
  }
  auto work = [&](int g) {
    const long long lo = bound[g], hi = bound[g + 1];
    if (hi <= lo) return;
    // synchronous whatever a device's "host_async" says (ag_multi has no wait entry point), as ag_detect
    rcs[g] = detect_batch_host(m->dets[g], (const uint8_t*)frames + (size_t)lo * fs, fs, (int)(hi - lo), width,
                               height, rs, format, out + (size_t)lo * cap_per_frame, cap_per_frame, n_per_frame + lo,
                               frame_status ? frame_status + lo : nullptr, /*async_call=*/false);
  };
  std::vector<std::thread> th;
  for (int g = 1; g < G; ++g) th.emplace_back(work, g);
  work(0);
  for (auto& t : th) t.join();
  int worst = AG_OK;
  for (int g = 0; g < G; ++g)
    if (rcs[g] != AG_OK && (worst == AG_OK || rcs[g] != AG_ERR_CAPACITY)) {  // a hard error outranks a capacity notice
      worst = rcs[g];
      m->err = std::string("device ") + std::to_string(m->dets[g]->device) + ": " + ag_last_error(m->dets[g]);
    }
  return worst;
}

}  // extern "C"
