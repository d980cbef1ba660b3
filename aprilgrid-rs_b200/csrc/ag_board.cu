// K6/K7: board assembly + tag decoding, one warp per frame (see ag_board_core.h).
// reference: src/detector.rs:505-639, src/board.rs, src/saddle.rs.
#include "ag_board_core.h"
#include "ag_board_fast.cuh"
#include "ag_common.cuh"
#include "ag_kernels.h"

#include <algorithm>

namespace ag {

// The family's code table is read from global memory (the detector's own copy): lanes read
// consecutive codes (coalesced, L1-resident), whereas constant memory would serialise the 32
// different addresses of a warp; it also keeps detectors of different families independent.

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

#ifndef AG_MAX_BOARD_WARPS
#define AG_MAX_BOARD_WARPS 16
#endif
constexpr int kMaxBoardWarps = AG_MAX_BOARD_WARPS;  // warps per frame (one block per frame): 1, 2, 4, 8 or 16

int g_board_smem_pad = 0;  // experiment: extra dynamic shared memory per block (limits blocks per SM)

BoardWsLayout make_board_layout(int max_saddles, int lattice, int warps, int smem_saddles, bool with_gpos,
                                int active_cap) {
  const int kBoardWarps = warps < 1 ? 1 : (warps > kMaxBoardWarps ? kMaxBoardWarps : warps);
  BoardWsLayout L;
  const int N = max_saddles;
  const int Q = N / 4 + 2;
  L.max_saddles = N;
  L.max_quads = Q;
  L.lattice = lattice;
  L.warps = kBoardWarps;
  const int cells = lattice * lattice;
  size_t o = 0;
  auto take = [&](size_t bytes) {
    size_t r = o;
    o = align_up(o + bytes, 16);
    return r;
  };
  // global workspace, per frame
  for (int i = 0; i < 3; ++i) L.off_pos[i] = take(sizeof(float) * N);
  L.off_best_quads = take(sizeof(int16_t) * 4 * Q);
  L.off_best_touched = take(sizeof(int16_t) * cells);
  L.off_best_vals = take(sizeof(int16_t) * cells);
  L.off_seeds = take(sizeof(int16_t) * N);
  L.off_remove = take(N);
  L.off_tag_valid = take(agb::kMaxCodes);
  L.off_tag_by_id = take(sizeof(agb::TagRec) * agb::kMaxCodes);
  L.off_qcache = take(sizeof(unsigned long long) * agb::kQCacheEntries);
  L.off_gitem = take(sizeof(uint16_t) * N);  // bucket-grid items of frames with more saddles than the on-chip tier
  // ... and per warp of the frame's block
  L.off_warp0 = o;
  size_t w = 0;
  auto wtake = [&](size_t bytes) {
    size_t r = w;
    w = align_up(w + bytes, 16);
    return r;
  };
  L.woff_quads = wtake(sizeof(int16_t) * 4 * Q);
  L.woff_touched = wtake(sizeof(int16_t) * cells);
  L.woff_sb_quads = wtake(sizeof(int16_t) * 4 * Q);
  L.woff_sb_touched = wtake(sizeof(int16_t) * cells);
  // warp 0's seed-best values double as the decode's bit patterns: 8 bytes for each quad the board
  // lists, and a board lists at most min(Q, lattice^2) quads
  L.woff_sb_vals = wtake(std::max(sizeof(int16_t) * cells, sizeof(unsigned long long) * std::min(Q, cells)));
  L.woff_stack = wtake(sizeof(int16_t) * 2 * (Q + 1));
  L.bytes_per_warp = align_up(w, 64);
  L.bytes_per_frame = align_up(L.off_warp0 + L.bytes_per_warp * kBoardWarps, 256);
  // shared memory of the block: frame-wide part, then one part per warp
  // tier: 320 (the usual frame: one board, ~270 saddles; seven frames per SM), 512 or 1024 saddles
  // on chip (the throughput path handles up to 1024), 4096 for large images (general path, saddle
  // list and bucket grid still on chip)
  L.smem_saddles = smem_saddles <= 320 ? 320 : (smem_saddles <= 512 ? 512 : (smem_saddles <= 1024 ? 1024 : 4096));
  L.grid_cap_cells = agb::kGridCapCells;  // 1280x1024 at 32 px buckets = 1280 buckets
  size_t sm = 0;
  auto stake = [&](size_t bytes) {
    size_t r = sm;
    sm = align_up(sm + bytes, 16);
    return r;
  };
  L.sm_pos = stake(sizeof(float) * 3 * L.smem_saddles);
  // bucket starts (a fixed size), grid-ordered positions, grid-ordered item indices: the throughput
  // path derives the addresses of the last two from the first (agb::kGridStartBytes, 8 bytes per
  // saddle of the tier), so the order and the sizes here are part of its contract
  L.sm_gstart = stake(sizeof(uint16_t) * (L.grid_cap_cells + 2));
  // (a layout without them -- the launch that only ever sees frames beyond the throughput path's
  // 1024 saddles -- saves 8 bytes per saddle; the kernel then finds the contract broken and
  // takes the general path, which does not use the grid-ordered positions)
  L.sm_gpos = stake(with_gpos ? sizeof(float2) * L.smem_saddles : 0);
  L.sm_gitem = stake(sizeof(uint16_t) * L.smem_saddles);
  // Large images, general path: the 1408 buckets above would be 128 px wide on a 4K frame (a radius
  // query then scans two or three rows of a dozen saddles each with two or three of its eight
  // lanes); 8192 buckets keep them at 32 px -- one or two saddles per row and lane.
  L.grid_cap_cells_big = L.smem_saddles == 4096 ? 8192 : 0;
  L.sm_gstart_big = L.grid_cap_cells_big ? stake(sizeof(uint16_t) * (L.grid_cap_cells_big + 2)) : 0;
  L.sm_ctl = stake(sizeof(int) * (16 + kMaxBoardWarps));  // 16 control words, then one score per warp
  // throughput path (ag_board_fast.cuh): per wave slot best score + quad
  L.sm_wave = stake(32 * (sizeof(uint16_t) + 4 * sizeof(int16_t)));
  L.sm_warp0 = sm;
  size_t sw = 0;
  auto swtake = [&](size_t bytes) {
    size_t r = sw;
    sw = align_up(sw + bytes, 16);
    return r;
  };
  // the lattice region doubles as the eight 1 KB group states of the throughput path
  L.smw_cell = swtake(std::max(sizeof(int16_t) * cells, (size_t)agb::kGroupsPerWarp * agb::kGroupBytes));
  // a launch that only ever sees frames of at most active_cap saddles needs no larger masks
  L.active_saddles = active_cap > 0 && active_cap < N ? active_cap : N;
  L.smw_active = swtake(sizeof(uint32_t) * ((L.active_saddles + 31) / 32));
  L.smw_small = swtake(sizeof(int16_t) * 64 * 4);  // nn_idx, same, diff, samp
  // throughput path: the warp's quad list and enumeration scratch
  L.smw_qlist = swtake(sizeof(int16_t) * 4 * agb::kQListCap);
  L.smw_qscore = swtake(sizeof(uint16_t) * agb::kQListCap);
  L.smw_fvec = swtake(sizeof(float) * 64 * 4);
  L.smw_squeue = swtake(sizeof(uint32_t) * 64);
  // the theta histogram of select_seeds (warp 0, before any seed is enumerated) borrows warp 0's
  // enumeration scratch
  static_assert(sizeof(int) * agb::kHistBins <= sizeof(float) * 64 * 4, "histogram must fit the enumeration scratch");
  L.sm_hist = L.sm_warp0 + L.smw_fvec;
  L.smem_per_warp = sw;
  L.smem_per_block = L.sm_warp0 + sw * kBoardWarps;
  return L;
}

// Register cap: the 320-saddle tier runs seven 2-warp blocks per SM, so registers are not what
// limits K6's residency -- what they decide is how many K1 blocks (72 registers x 128 threads) fit
// beside them.  Measured in the detect pipeline: 80 registers 101.1 k frames/s, 88 103.6 k,
// 96 104.0 k, 104 102.0 k, 112 102.3 k, 128 99.8 k (alone K6 keeps getting faster: fewer spills).
#ifndef AG_K6_MAXNREG
#define AG_K6_MAXNREG 96
#endif
__global__ void __maxnreg__(AG_K6_MAXNREG)
k_boards_decode(const uint8_t* __restrict__ frames, FrameGeom g, int n_frames,
                const ag_saddle* __restrict__ refined, const int* __restrict__ n_refined,
                uint8_t* __restrict__ ws, BoardWsLayout L, const uint64_t* __restrict__ codes,
                int n_codes, int edge, int border,
                int hamming, int max_boards, ag_tag* __restrict__ out, int cap,
                int* __restrict__ n_out, uint32_t* __restrict__ frame_status,
                int32_t* __restrict__ tap_quads, int* __restrict__ tap_n_quads, int tap_cap,
                int use_grid, int fast, uint32_t* __restrict__ timing, int n_above, int n_upto) {
  extern __shared__ __align__(16) uint8_t smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int f = blockIdx.x;  // one block per frame
  // A chunk is searched by two launches with different shared-memory tiers (small frames: more
  // blocks per SM); a block whose frame belongs to the other launch leaves at once.
  {
    const int nf = n_refined[f];
    if (nf <= n_above || nf > n_upto) return;  // block-uniform
  }
  // A frame whose cluster / saddle list was truncated (flagged by K3 / K4) has no meaningful board:
  // it reports no tags and keeps its flags; the host entry points re-run it with grown capacities.
  if (frame_status[f] & (uint32_t)(AG_FRAME_CLUSTER_OVERFLOW | AG_FRAME_SADDLE_OVERFLOW)) {  // block-uniform
    if (threadIdx.x == 0) {
      n_out[f] = 0;
      if (tap_n_quads) tap_n_quads[f] = 0;
    }
    return;
  }
  uint8_t* W = ws + (size_t)f * L.bytes_per_frame;
  uint8_t* WW = W + L.off_warp0 + (size_t)warp * L.bytes_per_warp;
  uint8_t* SW = smem + L.sm_warp0 + (size_t)warp * L.smem_per_warp;

  agb::Frame F;
  F.lane = lane;
  F.warp = warp;
  F.n_warps = L.warps;
  F.lat = L.lattice;
  F.lat_off = L.lattice / 2;
  F.n = n_refined[f];
  if (F.n <= L.smem_saddles) {  // the usual case: the saddle list lives in shared memory
    F.sx = (float*)(smem + L.sm_pos);
    F.sy = F.sx + L.smem_saddles;
    F.st = F.sy + L.smem_saddles;
  } else {
    F.sx = (float*)(W + L.off_pos[0]);
    F.sy = (float*)(W + L.off_pos[1]);
    F.st = (float*)(W + L.off_pos[2]);
  }
  F.bs.cell = (int16_t*)(SW + L.smw_cell);
  F.bs.active = (uint32_t*)(SW + L.smw_active);
  F.bs.quads = (int16_t*)(WW + L.woff_quads);
  F.bs.touched = (int16_t*)(WW + L.woff_touched);
  F.bs.n_quads = F.bs.n_touched = F.bs.score = 0;
  F.seedbest.quads = (int16_t*)(WW + L.woff_sb_quads);
  F.seedbest.touched = (int16_t*)(WW + L.woff_sb_touched);
  F.seedbest.vals = (int16_t*)(WW + L.woff_sb_vals);
  F.seedbest.n_quads = F.seedbest.n_touched = F.seedbest.score = 0;
  F.best.quads = (int16_t*)(W + L.off_best_quads);
  F.best.touched = (int16_t*)(W + L.off_best_touched);
  F.best.vals = (int16_t*)(W + L.off_best_vals);
  F.best.n_quads = F.best.n_touched = F.best.score = 0;
  F.stack = (int16_t*)(WW + L.woff_stack);
  F.dec_qlist = (int16_t*)(W + L.off_warp0 + L.woff_sb_quads);  // warp 0's seed-best arrays: free while decoding
  F.dec_qbits = (unsigned long long*)(W + L.off_warp0 + L.woff_sb_vals);
  F.seeds = (int16_t*)(W + L.off_seeds);
  // block-uniform: the whole frame takes the throughput path or the general one
  F.fast_on = (fast && use_grid && F.n <= agb::kFastMaxSaddles && F.n <= L.smem_saddles &&
               L.sm_gpos - L.sm_gstart == (size_t)agb::kGridStartBytes &&
               L.sm_gitem - L.sm_gpos == sizeof(float2) * (size_t)L.smem_saddles) ? 1 : 0;
  // bucket grid: 32 px buckets, doubled until the grid fits its shared-memory budget (the general
  // path of the 4096 tier has a larger budget of its own)
  {
    const bool big_grid = !F.fast_on && L.grid_cap_cells_big > 0;
    const int cap_cells = big_grid ? L.grid_cap_cells_big : L.grid_cap_cells;
    int bucket = 32;
    while (((g.w + bucket - 1) / bucket) * ((g.h + bucket - 1) / bucket) > cap_cells) bucket *= 2;
    F.g_base = use_grid ? (uint16_t*)(smem + (big_grid ? L.sm_gstart_big : L.sm_gstart)) : nullptr;
    F.g_start = F.g_base;
    F.g_item = (uint16_t*)(smem + L.sm_gitem);
    F.g_pos = (float2*)(smem + L.sm_gpos);
    F.g_nx = (g.w + bucket - 1) / bucket;
    F.g_ny = (g.h + bucket - 1) / bucket;
    F.g_cap_cells = cap_cells;
    F.g_cap_items = L.smem_saddles;
    if (F.n > L.smem_saddles) {
      // a frame too large for the on-chip tier (the general path): the bucket starts stay in shared
      // memory, the sorted item list goes to the frame's global workspace -- a radius query still
      // visits a few buckets instead of every saddle of the frame
      F.g_item = (uint16_t*)(W + L.off_gitem);
      F.g_cap_items = L.max_saddles;
    }
    F.g_inv = 1.0f / (float)bucket;
    F.g_on = 0;
  }
  F.hist = (int*)(smem + L.sm_hist);
  F.ctl = (int*)(smem + L.sm_ctl);
  F.w_score = F.ctl + 16;
  F.nn_idx = (int16_t*)(SW + L.smw_small);
  F.same = F.nn_idx + 64;
  F.diff = F.same + 64;
  F.samp = F.diff + 64;
  F.remove = W + L.off_remove;
  F.max_quads = L.max_quads;
  F.img = frame_base(frames, g, f);
  F.w = g.w;
  F.h = g.h;
  F.format = g.format;
  F.row_stride = g.row_stride;
  F.codes = codes;
  F.n_codes = n_codes;
  F.edge = edge;
  F.border = border;
  F.hamming = hamming;
  F.tag_valid = W + L.off_tag_valid;
  F.tag_by_id = (agb::TagRec*)(W + L.off_tag_by_id);
  F.tap_quads = tap_quads ? tap_quads + (size_t)f * tap_cap * 4 : nullptr;
  F.tap_n_quads = tap_n_quads ? tap_n_quads + f : nullptr;
  F.tap_cap = tap_cap;
  F.status = 0;
  F.active_words = (L.active_saddles + 31) / 32;
  F.tm = timing ? timing + (size_t)f * 32 : nullptr;
  unsigned long long t_start = 0;
  if (F.tm) {
    if (threadIdx.x < 32) F.tm[threadIdx.x] = 0u;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_start));
  }
  F.fx_qlist = (int16_t*)(SW + L.smw_qlist);
  F.fx_qscore = (uint16_t*)(SW + L.smw_qscore);
  F.fx_dvx = (float*)(SW + L.smw_fvec);
  F.fx_dvy = F.fx_dvx + agb::kDiffCap;
  F.fx_tmask = (unsigned long long*)(F.fx_dvy + agb::kDiffCap);  // 416 bytes in: 8-byte aligned
  F.fx_squeue = (uint32_t*)(SW + L.smw_squeue);
  F.fx_gstate = SW + L.smw_cell;
  // the seed-best arrays of the general path are free on the throughput path: they hold each
  // warp's saved best board there
  F.fx_save0 = W + L.off_warp0 + L.woff_sb_touched;
  F.fx_save_stride = L.bytes_per_warp;
  F.fx_qcache = (unsigned long long*)(W + L.off_qcache);
  F.fx_wscore = (uint16_t*)(smem + L.sm_wave);
  F.fx_wquad = (int16_t*)(F.fx_wscore + 32);
  // init: every warp clears its lattice and activates every saddle; warp 0 clears the tag map
  {
    const int cells = L.lattice * L.lattice;
    uint32_t* c = (uint32_t*)F.bs.cell;
    for (int i = lane; i < cells / 2; i += 32) c[i] = 0u;
    for (int i = lane; i < (L.active_saddles + 31) / 32; i += 32) F.bs.active[i] = 0xffffffffu;
    if (warp == 0) {
      uint32_t* tv = (uint32_t*)F.tag_valid;
      for (int i = lane; i < agb::kMaxCodes / 4; i += 32) tv[i] = 0;
      if (F.tap_n_quads && lane == 0) *F.tap_n_quads = 0;
      if (lane < 16) F.ctl[lane] = 0;
    }
  }
  if (F.fast_on) {  // empty neighbour-search cache (tag 0 = no entry)
    uint4* q = (uint4*)F.fx_qcache;
    for (int i = threadIdx.x; i < agb::kQCacheEntries / 2; i += blockDim.x) __stcg(q + i, make_uint4(0u, 0u, 0u, 0u));
  }
  // saddles AoS -> SoA (block-wide)
  const ag_saddle* S = refined + (size_t)f * L.max_saddles;
  for (int i = threadIdx.x; i < F.n; i += blockDim.x) {
    ag_saddle s = S[i];
    F.sx[i] = s.x;
    F.sy[i] = s.y;
    F.st[i] = s.theta;
  }
  __syncthreads();

  agb::detect_boards(F, max_boards);

  if (warp != 0) return;
  // emit the map in ascending id order
  ag_tag* O = out + (size_t)f * cap;
  int n = 0;
  for (int base = 0; base < n_codes; base += 32) {
    const int id = base + lane;
    const bool v = id < n_codes && F.tag_valid[id];
    const unsigned m = __ballot_sync(0xffffffffu, v);
    const int dst = n + __popc(m & ((1u << lane) - 1u));
    if (v && dst < cap) {
      const agb::TagRec t = F.tag_by_id[id];
      ag_tag o;
      o.id = t.id;
#pragma unroll
      for (int j = 0; j < 8; ++j) o.xy[j] = t.xy[j];
      O[dst] = o;
    }
    n += __popc(m);
  }
  if (lane == 0) {
    if (F.tm) {
      unsigned long long t_end;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
      F.tm[0] = (uint32_t)(t_end - t_start);
      F.tm[11] = (uint32_t)n_refined[f];
      F.tm[12] |= (uint32_t)F.fast_on << 31;
    }
    n_out[f] = n;
    uint32_t st = F.status;
    if (n > cap) st |= (uint32_t)AG_FRAME_TAG_OVERFLOW;
    if (st) atomicOr(frame_status + f, st);
  }
}

int launch_boards_decode(const uint8_t* frames, const FrameGeom& g, int n_frames,
                         const ag_saddle* refined, const int* n_refined, uint8_t* ws,
                         const BoardWsLayout& L, const uint64_t* d_codes, int n_codes, int edge, int border,
                         int hamming,
                         int max_boards, ag_tag* out, int cap, int* n_out, uint32_t* frame_status,
                         int32_t* tap_quads, int* tap_n_quads, int tap_cap, int use_grid, int fast,
                         uint32_t* timing, int n_above, int n_upto, cudaStream_t s) {
  const int blocks = n_frames;
  if (blocks == 0) return 0;
  const size_t smem = L.smem_per_block + (size_t)g_board_smem_pad;
  // per-device function attributes (cheap host calls; a process may drive several devices)
  if (cudaFuncSetAttribute(k_boards_decode, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
          cudaSuccess ||
      cudaFuncSetAttribute(k_boards_decode, cudaFuncAttributePreferredSharedMemoryCarveout,
                           cudaSharedmemCarveoutMaxShared) != cudaSuccess)
    return 0;
  k_boards_decode<<<blocks, L.warps * 32, smem, s>>>(
      frames, g, n_frames, refined, n_refined, ws, L, d_codes, n_codes, edge, border, hamming, max_boards,
      out, cap, n_out, frame_status, tap_quads, tap_n_quads, tap_cap, use_grid, fast, timing, n_above, n_upto);
  return 1;
}

}  // namespace ag
