// Host-callable launchers of the aprilgrid kernels (internal to the library).
// Every launcher returns the number of kernel launches it enqueued.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ag_common.cuh"

namespace ag {

struct BoardWsLayout {
  int max_saddles, max_quads, lattice, warps;
  // global workspace per frame: frame-wide part, then `warps` per-warp parts
  size_t off_pos[3];
  size_t off_best_quads, off_best_touched, off_best_vals;
  size_t off_seeds, off_remove, off_tag_valid, off_tag_by_id, off_qcache, off_gitem;
  size_t off_warp0, bytes_per_warp;
  size_t woff_quads, woff_touched, woff_sb_quads, woff_sb_touched, woff_sb_vals, woff_stack;
  size_t bytes_per_frame;
  // shared memory per block (= per frame in flight): frame-wide part, then per-warp parts
  int smem_saddles, grid_cap_cells;
  int active_saddles;  // saddles the per-warp `active` bit masks cover (max_saddles unless the launch bounds its frames)
  // 4096 tier only: a second, finer bucket-start array for the general path (0 = none)
  size_t sm_gstart_big;
  int grid_cap_cells_big;
  size_t sm_pos, sm_gstart, sm_gitem, sm_hist, sm_ctl, sm_warp0;
  size_t sm_wave, sm_gpos;
  size_t smw_cell, smw_active, smw_small, smw_qlist, smw_qscore, smw_fvec, smw_squeue;
  size_t smem_per_warp, smem_per_block;
};
BoardWsLayout make_board_layout(int max_saddles, int lattice, int warps, int smem_saddles, bool with_gpos = true,
                                int active_cap = 0);

// ag_dense.cu
int launch_blur_hessian(const uint8_t* frames, const FrameGeom& g, int n_frames, float* blur,
                        float* resp, uint32_t* frame_min, bool write_blur, int variant,
                        int chunk_rows_opt, cudaStream_t s);
int launch_threshold(const float* resp, const FrameGeom& g, int n_frames, const uint32_t* frame_min,
                     uint32_t* mask, cudaStream_t s);
int launch_blur_f32(const float* in, float* tmp, float* out, int w, int h, int n_frames, const float* taps,
                    const float* d_taps, int radius, cudaStream_t s);
int launch_hessian_f32(const float* in, float* out, int w, int h, cudaStream_t s);
int launch_unorm_table(float* out8, float* out16, float* ref8, float* ref16, cudaStream_t s);
int launch_float_luma(const float* rgb, long long n, int channels, float* luma32f, uint8_t* luma8, cudaStream_t s);

// ag_sparse.cu
int upload_rochade_tables(const float* cone25, const float* pinv150);
int launch_label_clusters(const uint32_t* mask, const FrameGeom& g, int n_frames, int* parent,
                          int max_clusters, int* acc, float2* centers, int* n_clusters,
                          uint32_t* frame_status, uint32_t* pixlist, int list_cap, int variant,
                          int* fallback, cudaStream_t s);
int launch_labels_tap(const uint32_t* mask, const FrameGeom& g, const int* parent, int32_t* labels,
                      uint8_t* mask_u8, cudaStream_t s);
int launch_refine_filter(const float* blur, const FrameGeom& g, int n_frames, const float2* centers,
                         const int* n_clusters, int max_clusters, ag_saddle* raw, uint8_t* raw_valid,
                         float min_angle, float max_angle, int max_saddles, ag_saddle* refined,
                         int* n_refined, uint32_t* frame_status, cudaStream_t s);
// the saddle entry points' result: K4's lists (in_stride per frame) -> out (out_stride per frame),
// n_out = exact count (0 if the frame's list was truncated), AG_FRAME_TAG_OVERFLOW when n > cap
// idx (frame lists, may be null): frame f's results go to the caller's frame idx[f], and its final status
// bits to status_out[idx[f]] when status_out is set
int launch_saddles_out(const ag_saddle* refined, int in_stride, const int* n_refined, uint32_t* frame_status,
                       int n_frames, ag_saddle* out, int out_stride, int cap, int* n_out, cudaStream_t s,
                       const int* idx = nullptr, uint32_t* status_out = nullptr);
// frame lists: the chunk-local tags, counts and status bits of the board search (in_stride records per
// frame) -> the caller's frame idx[f] (cap records per frame; status_out may be null)
int launch_tags_out(const ag_tag* tags, int in_stride, const int* n_tags, const uint32_t* frame_status, int n_frames,
                    const int* idx, ag_tag* out, int cap, int* n_out, uint32_t* status_out, cudaStream_t s);

// ag_board.cu
extern int g_board_smem_pad;
int launch_boards_decode(const uint8_t* frames, const FrameGeom& g, int n_frames,
                         const ag_saddle* refined, const int* n_refined, uint8_t* ws,
                         const BoardWsLayout& L, const uint64_t* d_codes, int n_codes, int edge, int border,
                         int hamming,
                         int max_boards, ag_tag* out, int cap, int* n_out, uint32_t* frame_status,
                         int32_t* tap_quads, int* tap_n_quads, int tap_cap, int use_grid, int fast,
                         uint32_t* timing, int n_above, int n_upto, cudaStream_t s);

// ag_render.cu
int launch_render_boards(uint8_t* frames, int n_frames, int w, int h, int cols, int rows,
                         const uint64_t* d_codes, int edge, int border, uint64_t seed,
                         const float* d_fixed_hinv, int noise, cudaStream_t s);

}  // namespace ag
