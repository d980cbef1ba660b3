/*
 * aprilgrid_b200.h -- C ABI of the B200-native aprilgrid detection front end.
 *
 * Drop-in boundary for powei-lin/aprilgrid-rs 0.8.0.  The reference has no FFI of its own;
 * these entry points are what a Rust shim (aprilgrid-rs_b200/rust/) binds so that
 *
 *     TagDetector::new(&TagFamily, Option<DetectorParams>)        src/detector.rs:364-406
 *     TagDetector::detect(&DynamicImage)                          src/detector.rs:505-540
 *     TagDetector::detect_kornia(&kornia::image::Image<u8, N>)    src/detector.rs:478-503
 *     TagDetector::refined_saddle_points(&DynamicImage)           src/detector.rs:408-446
 *     image_util::gaussian_blur_f32 / hessian_response            src/image_util.rs:72-206
 *
 * keep their signatures while the work runs as hand-written sm_100a kernels, plus the added
 * batched entry point detect_batch.  Plain pointers and sizes only; no C++ or torch types.
 *
 * There is NO CPU fallback: every compute entry point returns AG_ERR_NO_DEVICE /
 * AG_ERR_CUDA when no usable sm_100 GPU is present.
 *
 * Threading: one ag_detector may be used from many host threads (the Rust TagDetector is
 * Send + Sync and detect takes &self); calls on one handle are serialised by an internal
 * lock.  Create one handle per GPU (and per thread, if concurrency on one GPU is wanted).
 */
#ifndef APRILGRID_B200_H_
#define APRILGRID_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AG_API __attribute__((visibility("default")))

/* ---- status codes --------------------------------------------------------------- */
enum {
  AG_OK = 0,
  AG_ERR_INVALID = 1,    /* bad argument (null pointer, unknown family/format, w/h <= 0 ...) */
  AG_ERR_NO_DEVICE = 2,  /* no CUDA device / not an sm_100 part / extension not usable    */
  AG_ERR_CUDA = 3,       /* a CUDA call failed; see ag_last_error()                       */
  AG_ERR_CAPACITY = 4,   /* output capacity too small for a frame (results truncated)     */
  AG_ERR_UNSUPPORTED = 5
};

/* ---- TagFamily (src/tag_families.rs:5-13) ---------------------------------------- */
enum {
  AG_T16H5 = 0,
  AG_T25H7 = 1,
  AG_T25H9 = 2,
  AG_T36H11 = 3,
  AG_T36H11B1 = 4 /* 1-bit border */
};

/* ---- pixel formats: the DynamicImage variants, channels interleaved -------------------
 * Gray conversion as `image` 0.25 does it (to_luma32f for the stencils, to_luma8 for bit
 * sampling); alpha is dropped.
 * Integer formats: colour is the integer sRGB luma (2126 R + 7152 G + 722 B) / 10000, computed
 * and truncated in the source type's width (u8 -> Y8, u16 -> Y16, 32-bit arithmetic); then
 * to_luma32f = Y8 / 255 or Y16 / 65535 (correctly rounded) and to_luma8 = Y8 or (Y16 + 128) / 257.
 * Float formats: rgb_to_luma runs in f32::Larger = f64.  With r, g, b widened to f64 (the
 * products are exact) and RN the round-to-nearest-even of each operation, left to right:
 *   S = RN64(RN64(2126 r + 7152 g) + 722 b),  L = (f32) clamp(RN64(S / 10000), -f32::MAX, f32::MAX)
 *   to_luma32f = L,  to_luma8 = round_half_away(RN32(clamp(L, 0, 1) * 255))
 * The clamp is Enlargeable::clamp_from with Bounded::min_value / max_value as its bounds; it
 * never acts on finite pixels.  Channel values outside [0, 1] are converted like any other;
 * NaN and infinities are outside this contract (their result is unspecified).
 * 16-bit words and f32 values are native endian.  Value 3 is reserved (an internal f32 plane).
 * Row and frame strides must be multiples of a channel word (2 bytes for the 16-bit formats,
 * 4 for the float ones) everywhere, and so must the address of device frames on the device
 * entry points (else AG_ERR_INVALID; nothing runs).  Host frames may start at any address.  */
enum {
  AG_L8 = 0,       /* ImageLuma8   : 1 byte / px                                   */
  AG_L16 = 1,      /* ImageLuma16  : 2 bytes / px                                  */
  AG_RGB8 = 2,     /* ImageRgb8    : 3 bytes / px, R G B (detect_kornia N=3)       */
  AG_LA8 = 4,      /* ImageLumaA8  : 2 bytes / px, L A                             */
  AG_RGBA8 = 5,    /* ImageRgba8   : 4 bytes / px, R G B A                         */
  AG_LA16 = 6,     /* ImageLumaA16 : 4 bytes / px, L A (u16 each)                  */
  AG_RGB16 = 7,    /* ImageRgb16   : 6 bytes / px, R G B (u16 each)                */
  AG_RGBA16 = 8,   /* ImageRgba16  : 8 bytes / px, R G B A (u16 each)              */
  AG_RGB32F = 9,   /* ImageRgb32F  : 12 bytes / px, R G B (f32 each)               */
  AG_RGBA32F = 10  /* ImageRgba32F : 16 bytes / px, R G B A (f32 each)             */
};

/* ---- DetectorParams (src/detector.rs:25-41) -------------------------------------- */
typedef struct ag_params {
  float tag_spacing_ratio;   /* 0.3  (unused by the reference as well, detector.rs:621)  */
  float min_saddle_angle;    /* 30.0 */
  float max_saddle_angle;    /* 60.0 */
  uint8_t max_num_of_boards; /* 2    */
} ag_params;

/* One detection: the value type of the reference's HashMap<u32, [(f32, f32); 4]>.      */
typedef struct ag_tag {
  uint32_t id;
  float xy[8]; /* x0,y0 .. x3,y3 in the reference's corner order, integer = pixel centre */
} ag_tag;

/* Saddle (src/saddle.rs:3-9), 20 bytes. */
typedef struct ag_saddle {
  float x, y, k, theta, phi;
} ag_saddle;

/* per-frame status bits written to `frame_status` of the batch calls (0 = clean).
 * The reference has no per-frame limits (src/detector.rs:505-540).  The HOST entry points
 * (ag_detect, ag_detect_batch, ag_refined_saddle_points) therefore re-run a frame that overflowed
 * max_clusters / max_saddles with grown capacities (up to 2^22 clusters, 16384 saddles) and report
 * the untruncated result; only a frame beyond those hard limits, or a board wider than the
 * lattice, keeps its bits, and the call then returns AG_ERR_CAPACITY -- never AG_OK with a
 * truncated map.  The DEVICE entry point cannot re-run (its results stay on the device): a frame
 * with CLUSTER / SADDLE overflow reports zero tags and its bits; the caller checks them. */
enum {
  AG_FRAME_CLUSTER_OVERFLOW = 1, /* more saddle clusters than max_clusters            */
  AG_FRAME_SADDLE_OVERFLOW = 2,  /* more refined saddles than max_saddles             */
  AG_FRAME_BOARD_OVERFLOW = 4,   /* board grew outside the internal +-31 tag lattice  */
  AG_FRAME_TAG_OVERFLOW = 8      /* more results (tags; saddles on the saddle entry points) than cap_per_frame */
};

typedef struct ag_detector ag_detector;

/* DetectorParams::default_params() */
AG_API void ag_default_params(ag_params* out);

/* TagFamily::from_str (src/tag_families.rs:15-28).  Returns AG_OK or AG_ERR_INVALID.   */
AG_API int ag_family_from_str(const char* name, int* family_out);

/* (edge bits, border bits, hamming threshold, number of codes, code table) of a family,
 * as TagDetector::new selects them (src/detector.rs:369-405). */
AG_API int ag_family_info(int family, int* edge, int* border, int* hamming, int* n_codes,
                          const uint64_t** codes);

/* TagDetector::new.  params may be NULL (defaults).  device = CUDA ordinal.            */
AG_API int ag_create(int family, const ag_params* params, int device, ag_detector** out);
AG_API void ag_destroy(ag_detector* det);

/* Human-readable text of the last error on this handle (or of creation if det == NULL). */
AG_API const char* ag_last_error(const ag_detector* det);

/* Tunables.  key: "chunk_frames" (frames per pipeline chunk), "max_clusters",
 * "max_saddles" (per-frame capacities of the batch pipeline; 0 = automatic, sized from the image
 * area -- they bound memory, not results: see the frame status bits), "profile" (0/1, see ag_stage_times), "device_async"
 * (see ag_detect_batch_device_wait), "host_async" (see ag_detect_batch_wait), "dense_variant" (K1: 0 auto, 1 generic tile kernel),
 * "k1_chunk_rows" (rows per warp of the streaming K1: 0 automatic, else 6k + 4), "board_warps" (warps per frame in the board search:
 * 0 = automatic, 1/2/4/8/16; fewer where a tier's shared memory would not fit), "board_fast" (0 = general board path only), "board_lattice", "board_saddle_tier" (saddles kept on chip by the
 * board kernel: -1 automatic from the image size, 0 / 1 / 2 = 512 / 1024 / 4096), "board_batch_frames" (launches with at
 * least this many frames use the batch configuration), "board_split", "board_priority" (1 = board streams at the
 * greatest stream priority; set before the first detect call).
 * Capacities must be set before the first detect call that needs them larger. */
AG_API int ag_set_option(ag_detector* det, const char* key, long value);

/* TagDetector::detect on one host image.  `out` receives up to `cap` tags in ascending id
 * order; *n = number found (may exceed cap => AG_ERR_CAPACITY, first cap written).
 * Always synchronous, also on a handle whose streaming option "host_async" is on.        */
AG_API int ag_detect(ag_detector* det, const void* pixels, int width, int height,
                     size_t row_stride, int format, ag_tag* out, int cap, int* n);

/* TagDetector::detect on a frame given as the TWO gray planes the reference derives from its
 * DynamicImage itself: luma32f = img.to_luma32f() (the stencil chain, src/detector.rs:409) and
 * luma8 = img.to_luma8() (bit sampling, :507).  A shim that computes both planes with the `image`
 * crate and calls this gets the reference's own conversion, whatever the DynamicImage variant.
 * Row strides in bytes (0 = packed).  Synchronous; same result and error conventions as ag_detect. */
AG_API int ag_detect_planes(ag_detector* det, const float* luma32f, size_t f32_row_stride,
                            const uint8_t* luma8, size_t u8_row_stride, int width, int height,
                            ag_tag* out, int cap, int* n);

/* detect_batch: n_frames host images of one shape at frames + i*frame_stride.
 * out[i*cap_per_frame ..], n_per_frame[i]; frame_status may be NULL.
 * Strides in bytes (0 = packed), multiples of the format's channel word (else AG_ERR_INVALID). */
AG_API int ag_detect_batch(ag_detector* det, const void* frames, size_t frame_stride,
                           int n_frames, int width, int height, size_t row_stride, int format,
                           ag_tag* out, int cap_per_frame, int* n_per_frame,
                           uint32_t* frame_status);

/* Same, frames already resident in device memory; outputs are DEVICE pointers
 * (d_out: n_frames*cap_per_frame ag_tag, d_n_per_frame: n_frames int32,
 *  d_frame_status: n_frames uint32 or NULL).  Work is enqueued on `stream`
 * (a cudaStream_t, NULL = the detector's own stream) and is asynchronous.
 * Frames must start at a multiple of the channel word (else AG_ERR_INVALID; nothing runs). */
AG_API int ag_detect_batch_device(ag_detector* det, const void* d_frames, size_t frame_stride,
                                  int n_frames, int width, int height, size_t row_stride,
                                  int format, ag_tag* d_out, int cap_per_frame,
                                  int* d_n_per_frame, uint32_t* d_frame_status, void* stream);

/* Streaming use of ag_detect_batch_device.  By default every call orders its results on
 * `stream` before returning control to the stream, so back-to-back calls drain the internal
 * pipeline at each call boundary.  After ag_set_option(det, "device_async", 1) a call only
 * enqueues its work; ag_detect_batch_device_wait(det, stream) then makes `stream` (NULL = the
 * host thread) wait for every call issued so far.  Output buffers of calls that are still in
 * flight must not be reused.  (detect_batch over an unbounded frame sequence.)            */
AG_API int ag_detect_batch_device_wait(ag_detector* det, void* stream);

/* Streaming use of ag_detect_batch (host buffers).  By default a call returns with its results in
 * the output arrays, so the pipeline fills and drains once per call.  After
 * ag_set_option(det, "host_async", 1) a call returns as soon as its chunks are enqueued (it
 * blocks only to recycle staging buffers, handing out the results of older chunks while it does);
 * ag_detect_batch_wait(det, keep_in_flight) then returns once all but the newest
 * `keep_in_flight` calls are complete (0 = every call), so that the uploads of one call overlap
 * the board searches of the one before.  The frames and the output arrays of a call must stay
 * valid and untouched until a wait has covered it.  AG_ERR_CAPACITY is reported by the wait.
 * (detect over an unbounded sequence of host images: src/detector.rs:505-540 `detect`, batched.)  */
AG_API int ag_detect_batch_wait(ag_detector* det, int keep_in_flight);

/* TagDetector::refined_saddle_points: refined saddles of one host image, reference order. */
AG_API int ag_refined_saddle_points(ag_detector* det, const void* pixels, int width, int height,
                                    size_t row_stride, int format, ag_saddle* out, int cap,
                                    int* n);

/* refined_saddle_points on n_frames host images of one shape (layout and strides as ag_detect_batch).
 * out[i*cap_per_frame ..]: frame i's refined saddles in the reference's order, n_per_frame[i] = their
 * exact number; frame_status may be NULL.  Always synchronous (also on a "host_async" handle).
 * Contract of the three saddle batch entry points (this one, _device and ag_multi_):
 *  - Frame i's list is byte-identical to what ag_refined_saddle_points returns for that frame alone.
 *  - Host calls: a frame that overflowed max_clusters / max_saddles in its chunk is re-run alone with
 *    grown capacities and comes back untruncated; a frame beyond the hard limits (2^22 clusters,
 *    16384 saddles) keeps its bits (and the list ag_refined_saddle_points gives it), and the call
 *    returns AG_ERR_CAPACITY.  The device call cannot re-run: such a frame reports n = 0 and its bits.
 *  - n_per_frame[i] > cap_per_frame: the count stays exact, the first cap_per_frame saddles are
 *    written, the frame's status gets AG_FRAME_TAG_OVERFLOW, and the host calls return
 *    AG_ERR_CAPACITY (the device call reports it through the bit only).  Nothing past
 *    min(n, cap_per_frame) records of a frame's slot is written.
 *  - n_frames == 0: AG_OK, nothing runs.  Null pointers, cap_per_frame < 1, n_frames < 0, bad
 *    strides or a misaligned device address: AG_ERR_INVALID, nothing runs.
 *  - Saddle and detect calls may be interleaved freely on one handle, on any streams; neither
 *    changes the other's results.  A host saddle call first collects the detect chunks of
 *    "host_async" calls still in flight, as ag_detect does. */
AG_API int ag_refined_saddle_points_batch(ag_detector* det, const void* frames, size_t frame_stride,
                                          int n_frames, int width, int height, size_t row_stride,
                                          int format, ag_saddle* out, int cap_per_frame,
                                          int* n_per_frame, uint32_t* frame_status);

/* Same, frames and outputs in device memory (d_out: n_frames*cap_per_frame ag_saddle,
 * d_n_per_frame: n_frames int32, d_frame_status: n_frames uint32 or NULL), enqueued on `stream`;
 * option "device_async" and ag_detect_batch_device_wait apply to it exactly as to
 * ag_detect_batch_device. */
AG_API int ag_refined_saddle_points_batch_device(ag_detector* det, const void* d_frames,
                                                 size_t frame_stride, int n_frames, int width,
                                                 int height, size_t row_stride, int format,
                                                 ag_saddle* d_out, int cap_per_frame,
                                                 int* d_n_per_frame, uint32_t* d_frame_status,
                                                 void* stream);

/* ---- lists of frames of mixed sizes and pixel formats ---------------------------------------
 * One frame of a list: the fields and their order are those of the C++ mirror's ImageView. */
typedef struct ag_frame {
  const void* pixels; /* host or device address, as the entry point says */
  int width, height;
  size_t row_stride; /* bytes, 0 = packed */
  int format;        /* AG_L8 .. AG_RGBA32F */
} ag_frame;

/* detect / refined_saddle_points on a list of n_frames frames, each with its own address, size,
 * row stride and pixel format.  Outputs are laid out as on the _batch siblings and indexed by list
 * position: out[i*cap_per_frame ..], n_per_frame[i], frame_status[i] (may be NULL).
 * Contract of the six list entry points (these two, the _device pair and the ag_multi_ pair):
 *  - Frame i's result is byte-identical to what ag_detect / ag_refined_saddle_points returns for
 *    that frame alone; the grouping and order of the list never change a result.
 *  - Every descriptor is checked before anything runs: null pixels, width or height <= 0, an
 *    unknown format, a row stride shorter than a row or not a multiple of the channel word, and (on
 *    the device calls) a device address that is not a multiple of the channel word.  One bad
 *    descriptor, a null list, n_frames < 0 or cap_per_frame < 1: AG_ERR_INVALID, nothing runs and no
 *    output is touched.  n_frames == 0: AG_OK.  Frames may alias each other.
 *  - Capacities as on the _batch siblings: the host calls re-run a frame that overflowed
 *    max_clusters / max_saddles alone with grown capacities; a frame beyond the hard limits keeps
 *    its bits and the call returns AG_ERR_CAPACITY; the device calls report n = 0 and the bits.
 *    n_per_frame[i] > cap_per_frame: the count stays exact, the first cap_per_frame records are
 *    written, AG_FRAME_TAG_OVERFLOW is set (and the host calls return AG_ERR_CAPACITY).  The
 *    per-frame capacities of a list call are those the largest frame of the list would get alone, so
 *    the device call flags no frame that ag_detect_batch_device on that frame's shape would not.
 *  - Frames are grouped by (width, height, format, row_stride) in order of first appearance; each
 *    group runs in chunks of one geometry through the same pipeline as a batch, so the groups
 *    overlap in it.  A group of one frame still costs one chunk's launches.
 *  - List calls and the other calls may be interleaved on one handle, on any streams, without
 *    changing each other's results.  A host list call first collects the chunks of "host_async"
 *    calls still in flight; it is always synchronous. */
AG_API int ag_detect_frames(ag_detector* det, const ag_frame* frames, int n_frames, ag_tag* out,
                            int cap_per_frame, int* n_per_frame, uint32_t* frame_status);
AG_API int ag_refined_saddle_points_frames(ag_detector* det, const ag_frame* frames, int n_frames,
                                           ag_saddle* out, int cap_per_frame, int* n_per_frame,
                                           uint32_t* frame_status);
/* Same, with `pixels` of every descriptor a DEVICE address (the descriptor array itself is on the
 * host) and DEVICE outputs (d_out: n_frames*cap_per_frame records, d_n_per_frame: n_frames int32,
 * d_frame_status: n_frames uint32 or NULL).  Enqueued on `stream` as ag_detect_batch_device; option
 * "device_async" and ag_detect_batch_device_wait apply to them exactly as to that call.  The frames
 * must stay valid until the results are ordered on the stream. */
AG_API int ag_detect_frames_device(ag_detector* det, const ag_frame* frames, int n_frames, ag_tag* d_out,
                                   int cap_per_frame, int* d_n_per_frame, uint32_t* d_frame_status,
                                   void* stream);
AG_API int ag_refined_saddle_points_frames_device(ag_detector* det, const ag_frame* frames, int n_frames,
                                                  ag_saddle* d_out, int cap_per_frame, int* d_n_per_frame,
                                                  uint32_t* d_frame_status, void* stream);

/* image_util::gaussian_blur_f32(img, sigma) and image_util::hessian_response(img):
 * f32 -> f32, host buffers, width*height floats each.                                   */
AG_API int ag_gaussian_blur_f32(ag_detector* det, const float* img, int width, int height,
                                float sigma, float* out);
AG_API int ag_hessian_response(ag_detector* det, const float* img, int width, int height,
                               float* out);
/* gaussian_blur_f32 on n_frames contiguous device-resident f32 images (d_out != d_in), enqueued on
 * `stream` (0 = the default stream); returns when enqueued.  This is the operator
 * benches/bench_blur.rs:34-46 times (src/image_util.rs:110-206), batched: 8 B/px of traffic.
 * The scratch image of the general path (radius != 3 or width % 4 != 0) belongs to the handle:
 * one such call at a time per handle.                                                          */
AG_API int ag_gaussian_blur_f32_device(ag_detector* det, const float* d_in, int n_frames, int width,
                                       int height, float sigma, float* d_out, void* stream);

/* Dense front end only (gray -> blur -> Hessian -> min -> threshold mask), device-resident
 * frames, results stay in the detector's workspace.  This is the unit bench.py times for
 * the "blur / threshold kernels alone" configuration.  Address and strides aligned as above. */
AG_API int ag_dense_batch_device(ag_detector* det, const void* d_frames, size_t frame_stride,
                                 int n_frames, int width, int height, size_t row_stride,
                                 int format, void* stream);

/* ---- stage taps (test only) -------------------------------------------------------
 * ag_stage_run processes ONE host image through the whole pipeline keeping every
 * intermediate; the getters then copy one stage to host so it can be diffed against the
 * oracle.  Sizes: blur/response width*height f32; mask width*height u8 (0/1);
 * labels width*height i32 (cluster id in reference order, -1 = background).            */
AG_API int ag_stage_run(ag_detector* det, const void* pixels, int width, int height,
                        size_t row_stride, int format);
AG_API int ag_stage_blur(ag_detector* det, float* out);
AG_API int ag_stage_response(ag_detector* det, float* out);
AG_API int ag_stage_threshold(ag_detector* det, float* min_and_thr /* [2] */);
AG_API int ag_stage_mask(ag_detector* det, uint8_t* out);
AG_API int ag_stage_labels(ag_detector* det, int32_t* out);
AG_API int ag_stage_centers(ag_detector* det, float* xy_out, int cap, int* n);
/* which: 0 = every refined candidate before the k/phi filter, 1 = after it */
AG_API int ag_stage_saddles(ag_detector* det, int which, ag_saddle* out, int cap, int* n);
/* quads (4 saddle indices each, into the `which = 1` list) of the first best board */
AG_API int ag_stage_board_quads(ag_detector* det, int32_t* quads_out, int cap, int* n);
AG_API int ag_stage_tags(ag_detector* det, ag_tag* out, int cap, int* n);

/* Number of kernel launches issued by this handle since creation (bench bookkeeping). */
AG_API uint64_t ag_launch_count(const ag_detector* det);

/* Per-stage device time, accumulated with CUDA events on the launching stream while the
 * option "profile" is 1.  ms_out[8] / n_out[8]: total milliseconds and number of launches of
 * stage 0 = blur+Hessian+min, 1 = threshold, 2 = label+centroid, 3 = refine+filter,
 * 4 = boards+decode.  Synchronises the device.  reset != 0 clears the accumulators.       */
AG_API int ag_stage_times(ag_detector* det, double* ms_out, uint64_t* n_out, int reset);

/* Synthetic AprilGrid renderer (benchmark / test data generator, runs on the GPU):
 * renders n_frames u8 gray frames of a cols x rows board of `family` tags (ids from 0,
 * row-major from the bottom row, spacing ratio 0.3; geometry of
 * scripts/generate_aprilgrid.py:1114-1167) under a seeded random pose.  d_frames is a
 * device pointer to n_frames*width*height bytes.                                         */
AG_API int ag_render_boards_device(ag_detector* det, void* d_frames, int n_frames, int width,
                                   int height, int cols, int rows, uint64_t seed, void* stream);

/* Page-locked host memory for batches the caller assembles itself (the Rust shim packs its
 * DynamicImages into it): uploaded at the link rate without a staging copy.  Frames in ordinary
 * (pageable) memory are accepted everywhere too -- the library then stages them through its own
 * pinned buffers with several host threads, at memory-copy speed.  NULL on failure.            */
AG_API void* ag_host_alloc(size_t bytes);
AG_API void ag_host_free(void* p);

/* ---- one detector over several GPUs of one box ---------------------------------------------
 * detect_batch for a multi-GPU host: frames are independent (src/detector.rs:505-540), so the
 * batch is cut into contiguous frame ranges [g*B/G, (g+1)*B/G), one per device, each handled by
 * that device's own pipeline on its own host thread; every device writes its results into the
 * caller's arrays at its frames' positions (no collective on the data path).  The ranges are equal
 * unless the devices' host-to-device rates (measured at creation, all devices copying at once)
 * differ by more than 5 %: then they are proportional to those rates.  devices = NULL or
 * n_devices = 0: every visible device.  Same arguments, results and error behaviour as
 * ag_detect_batch, but always synchronous, whatever the devices' "host_async" option says;
 * byte-identical to one device processing the batch.                                          */
typedef struct ag_multi ag_multi;
AG_API int ag_multi_create(int family, const ag_params* params, const int* devices, int n_devices,
                           ag_multi** out);
AG_API void ag_multi_destroy(ag_multi* m);
AG_API int ag_multi_device_count(const ag_multi* m);
AG_API const char* ag_multi_last_error(const ag_multi* m);
AG_API int ag_multi_set_option(ag_multi* m, const char* key, long value); /* applied to every device */
AG_API int ag_multi_detect_batch(ag_multi* m, const void* frames, size_t frame_stride, int n_frames,
                                 int width, int height, size_t row_stride, int format, ag_tag* out,
                                 int cap_per_frame, int* n_per_frame, uint32_t* frame_status);
/* ag_refined_saddle_points_batch over every device of m (same sharding as ag_multi_detect_batch). */
AG_API int ag_multi_refined_saddle_points_batch(ag_multi* m, const void* frames, size_t frame_stride,
                                                int n_frames, int width, int height,
                                                size_t row_stride, int format, ag_saddle* out,
                                                int cap_per_frame, int* n_per_frame,
                                                uint32_t* frame_status);
/* ag_detect_frames / ag_refined_saddle_points_frames over every device of m: the list is cut into
 * contiguous index ranges of about equal frame bytes (weighted by the devices' host-to-device rates
 * as above); byte-identical to one device processing the list. */
AG_API int ag_multi_detect_frames(ag_multi* m, const ag_frame* frames, int n_frames, ag_tag* out,
                                  int cap_per_frame, int* n_per_frame, uint32_t* frame_status);
AG_API int ag_multi_refined_saddle_points_frames(ag_multi* m, const ag_frame* frames, int n_frames,
                                                 ag_saddle* out, int cap_per_frame, int* n_per_frame,
                                                 uint32_t* frame_status);

AG_API const char* ag_version(void);

#ifdef __cplusplus
}
#endif
#endif /* APRILGRID_B200_H_ */
