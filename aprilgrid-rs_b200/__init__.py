"""aprilgrid_rs_b200 -- Python mirror of the aprilgrid-rs detector API over the B200 C ABI.

The names follow the reference crate (``aprilgrid::TagFamily``, ``aprilgrid::detector::
TagDetector``, ``DetectorParams``; src/detector.rs:17-41, :363-541) so that tests read like
the reference's own: ``TagDetector(TagFamily.T36H11).detect(img)`` returns
``{id: 4x2 float32 corners}``.  All work happens in ``lib/libaprilgrid_b200.so``
(hand-written sm_100a kernels, include/aprilgrid_b200.h); there is no CPU path: constructing
a detector without a B200 raises ``RuntimeError``.

The directory name contains a hyphen, so import it through ``__graft_entry__.load_package()``
(or importlib) under the module name ``aprilgrid_rs_b200``.
"""
import ctypes as C
import enum
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libaprilgrid_b200.so")
if os.environ.get("AG_LIB"):  # profiling tools only: another build of the same library (tools/build_variant.sh)
    LIB_PATH = os.path.abspath(os.environ["AG_LIB"])

AG_OK, AG_ERR_INVALID, AG_ERR_NO_DEVICE, AG_ERR_CUDA, AG_ERR_CAPACITY, AG_ERR_UNSUPPORTED = range(6)
FMT_L8, FMT_L16, FMT_RGB8 = 0, 1, 2
FMT_LA8, FMT_RGBA8, FMT_LA16, FMT_RGB16, FMT_RGBA16 = 4, 5, 6, 7, 8  # 3 is reserved
FMT_RGB32F, FMT_RGBA32F = 9, 10
# (channels, dtype) -> pixel format of an H x W x channels image (DynamicImage LumaA / Rgb / Rgba)
_CHANNEL_FORMATS = {(2, np.uint8): FMT_LA8, (3, np.uint8): FMT_RGB8, (4, np.uint8): FMT_RGBA8,
                    (2, np.uint16): FMT_LA16, (3, np.uint16): FMT_RGB16, (4, np.uint16): FMT_RGBA16,
                    (3, np.float32): FMT_RGB32F, (4, np.float32): FMT_RGBA32F}

TAG_DTYPE = np.dtype([("id", np.uint32), ("xy", np.float32, (8,))])
SADDLE_DTYPE = np.dtype([("x", np.float32), ("y", np.float32), ("k", np.float32),
                         ("theta", np.float32), ("phi", np.float32)])


class TagFamily(enum.IntEnum):
    """src/tag_families.rs:5-13"""
    T16H5 = 0
    T25H7 = 1
    T25H9 = 2
    T36H11 = 3
    T36H11B1 = 4

    @staticmethod
    def from_str(name):
        """TagFamily::from_str (src/tag_families.rs:15-28): raises ValueError on unknown names."""
        fam = C.c_int(0)
        if lib().ag_family_from_str(name.encode(), C.byref(fam)) != AG_OK:
            raise ValueError("unknown tag family %r" % (name,))
        return TagFamily(fam.value)


class _Params(C.Structure):
    _fields_ = [("tag_spacing_ratio", C.c_float), ("min_saddle_angle", C.c_float),
                ("max_saddle_angle", C.c_float), ("max_num_of_boards", C.c_uint8)]


class DetectorParams:
    """src/detector.rs:25-41"""

    def __init__(self, tag_spacing_ratio=0.3, min_saddle_angle=30.0, max_saddle_angle=60.0,
                 max_num_of_boards=2):
        self.tag_spacing_ratio = tag_spacing_ratio
        self.min_saddle_angle = min_saddle_angle
        self.max_saddle_angle = max_saddle_angle
        self.max_num_of_boards = max_num_of_boards

    @staticmethod
    def default_params():
        return DetectorParams()

    def _c(self):
        return _Params(self.tag_spacing_ratio, self.min_saddle_angle, self.max_saddle_angle,
                       self.max_num_of_boards)


_lib = None


def lib():
    """Load the C-ABI library.  Fails loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`"
                               " (there is no CPU fallback)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        vp, ci, sz = C.c_void_p, C.c_int, C.c_size_t
        L.ag_version.restype = C.c_char_p
        L.ag_last_error.restype = C.c_char_p
        L.ag_last_error.argtypes = [vp]
        L.ag_default_params.argtypes = [vp]
        L.ag_family_from_str.argtypes = [C.c_char_p, vp]
        L.ag_family_info.argtypes = [ci, vp, vp, vp, vp, vp]
        L.ag_create.argtypes = [ci, vp, ci, vp]
        L.ag_destroy.argtypes = [vp]
        L.ag_set_option.argtypes = [vp, C.c_char_p, C.c_long]
        L.ag_detect.argtypes = [vp, vp, ci, ci, sz, ci, vp, ci, vp]
        L.ag_detect_planes.argtypes = [vp, vp, sz, vp, sz, ci, ci, vp, ci, vp]
        L.ag_detect_batch.argtypes = [vp, vp, sz, ci, ci, ci, sz, ci, vp, ci, vp, vp]
        L.ag_detect_batch_device.argtypes = [vp, vp, sz, ci, ci, ci, sz, ci, vp, ci, vp, vp, vp]
        L.ag_detect_batch_device_wait.argtypes = [vp, vp]
        L.ag_detect_batch_wait.argtypes = [vp, ci]
        L.ag_dense_batch_device.argtypes = [vp, vp, sz, ci, ci, ci, sz, ci, vp]
        L.ag_refined_saddle_points.argtypes = [vp, vp, ci, ci, sz, ci, vp, ci, vp]
        L.ag_gaussian_blur_f32.argtypes = [vp, vp, ci, ci, C.c_float, vp]
        L.ag_hessian_response.argtypes = [vp, vp, ci, ci, vp]
        L.ag_gaussian_blur_f32_device.argtypes = [vp, vp, ci, ci, ci, C.c_float, vp, vp]
        L.ag_stage_run.argtypes = [vp, vp, ci, ci, sz, ci]
        for n in ("ag_stage_blur", "ag_stage_response", "ag_stage_threshold", "ag_stage_mask",
                  "ag_stage_labels"):
            getattr(L, n).argtypes = [vp, vp]
        L.ag_stage_centers.argtypes = [vp, vp, ci, vp]
        L.ag_stage_saddles.argtypes = [vp, ci, vp, ci, vp]
        L.ag_stage_board_quads.argtypes = [vp, vp, ci, vp]
        L.ag_stage_tags.argtypes = [vp, vp, ci, vp]
        L.ag_launch_count.restype = C.c_uint64
        L.ag_launch_count.argtypes = [vp]
        L.ag_stage_times.argtypes = [vp, vp, vp, ci]
        L.ag_render_boards_device.argtypes = [vp, vp, ci, ci, ci, ci, ci, C.c_uint64, vp]
        L.ag_host_alloc.restype = vp
        L.ag_host_alloc.argtypes = [sz]
        L.ag_host_free.argtypes = [vp]
        L.ag_multi_create.argtypes = [ci, vp, vp, ci, vp]
        L.ag_multi_destroy.argtypes = [vp]
        L.ag_multi_device_count.argtypes = [vp]
        L.ag_multi_last_error.restype = C.c_char_p
        L.ag_multi_last_error.argtypes = [vp]
        L.ag_multi_set_option.argtypes = [vp, C.c_char_p, C.c_long]
        L.ag_multi_detect_batch.argtypes = [vp, vp, sz, ci, ci, ci, sz, ci, vp, ci, vp, vp]
        L.ag_test_unorm_tables.argtypes = [vp, vp, vp, vp, vp]
        L.ag_test_board_times.argtypes = [vp, ci, vp, ci]
        L.ag_test_board_layout.argtypes = [ci, ci, ci, ci, ci, ci, vp]
        L.ag_test_board_decode_room.argtypes = [ci, ci, ci, vp]
        L.ag_test_render_pose.argtypes = [vp, vp, ci, ci, ci, ci, vp, ci, C.c_uint64]
        L.ag_test_boards_from_saddles.argtypes = [vp, vp, sz, vp, ci, vp, sz, ci, ci, sz, ci, vp, ci, vp, vp, ci,
                                                  vp, vp]
        L.ag_test_float_luma.argtypes = [vp, vp, C.c_longlong, ci, vp, vp]
        L.ag_test_host_chunk.argtypes = [C.c_longlong, ci, vp]
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def image_format(img):
    """(fmt, width, height, row_stride_bytes) for HxW u8 (Luma8) / u16 (Luma16), HxWxN u8 / u16
    with N = 2 (LumaA8 / LumaA16), 3 (Rgb8 / Rgb16) or 4 (Rgba8 / Rgba16), and HxWxN float32 with
    N = 3 (Rgb32F) or 4 (Rgba32F); channels interleaved.  HxW float32 is no DynamicImage variant:
    see TagDetector.detect_planes."""
    if img.ndim == 2 and img.dtype == np.uint8:
        return FMT_L8, img.shape[1], img.shape[0], img.strides[0]
    if img.ndim == 2 and img.dtype == np.uint16:
        return FMT_L16, img.shape[1], img.shape[0], img.strides[0]
    if img.ndim == 3 and (img.shape[2], img.dtype.type) in _CHANNEL_FORMATS:
        return _CHANNEL_FORMATS[(img.shape[2], img.dtype.type)], img.shape[1], img.shape[0], img.strides[0]
    raise ValueError("unsupported image: shape %s dtype %s (want HxW or HxWxN u8/u16 with N in 2..4, "
                     "or HxWxN float32 with N in 3..4)"
                     % (img.shape, img.dtype))


def family_info(family):
    e, b, h, n = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int(0)
    codes = C.POINTER(C.c_uint64)()
    rc = lib().ag_family_info(int(family), C.byref(e), C.byref(b), C.byref(h), C.byref(n), C.byref(codes))
    if rc != AG_OK:
        raise ValueError("unknown family")
    return dict(edge=e.value, border=b.value, hamming=h.value,
                codes=np.array([codes[i] for i in range(n.value)], np.uint64))


def _tags_to_dict(rec):
    return {int(t["id"]): t["xy"].reshape(4, 2).copy() for t in rec}


class TagDetector:
    """aprilgrid::detector::TagDetector (src/detector.rs:17-23, :363-541) on one B200."""

    def __init__(self, tag_family=TagFamily.T36H11, optional_detector_params=None, device=0):
        self._h = C.c_void_p(None)
        params = optional_detector_params or DetectorParams.default_params()
        cp = params._c()
        rc = lib().ag_create(int(tag_family), C.byref(cp), int(device), C.byref(self._h))
        if rc != AG_OK:
            msg = lib().ag_last_error(None).decode()
            self._h = C.c_void_p(None)
            raise RuntimeError("ag_create failed (%d): %s" % (rc, msg))
        self.family = TagFamily(int(tag_family))
        self.params = params
        self.device = device

    # -- plumbing ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().ag_destroy(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, allow=()):
        if rc != AG_OK and rc not in allow:
            raise RuntimeError("aprilgrid_b200 error %d: %s" % (rc, lib().ag_last_error(self._h).decode()))
        return rc

    def set_option(self, key, value):
        self._check(lib().ag_set_option(self._h, key.encode(), int(value)))

    @property
    def launch_count(self):
        return int(lib().ag_launch_count(self._h))

    STAGE_NAMES = ("blur_hessian_min", "threshold", "label_centroid", "refine_filter", "boards_decode")

    def stage_times(self, reset=True):
        """{stage: (total_ms, launches)} accumulated while option "profile" is 1."""
        ms = np.zeros(8, np.float64)
        cnt = np.zeros(8, np.uint64)
        self._check(lib().ag_stage_times(self._h, _p(ms), _p(cnt), 1 if reset else 0))
        return {n: (float(ms[i]), int(cnt[i])) for i, n in enumerate(self.STAGE_NAMES)}

    # -- reference API -----------------------------------------------------------------
    def detect(self, img, cap=1024):
        """TagDetector::detect(&DynamicImage) -> HashMap<u32, [(f32, f32); 4]> (detector.rs:505)."""
        img = np.asarray(img)
        fmt, w, h, st = image_format(img)
        if img.strides[-1] != img.itemsize or (img.ndim == 3 and img.strides[1] != img.shape[2] * img.itemsize):
            img = np.ascontiguousarray(img)
            fmt, w, h, st = image_format(img)
        out = np.zeros(cap, TAG_DTYPE)
        n = C.c_int(0)
        self._check(lib().ag_detect(self._h, _p(img), w, h, st, fmt, _p(out), cap, C.byref(n)))
        return _tags_to_dict(out[:n.value])

    def detect_planes(self, luma32f, luma8, cap=1024):
        """detect on a frame given as its two gray planes: to_luma32f(img) (H x W float32) and to_luma8(img)
        (H x W uint8) -- for DynamicImage variants whose conversion the caller does with `image` itself."""
        f = np.ascontiguousarray(luma32f, np.float32)
        g = np.ascontiguousarray(luma8, np.uint8)
        if f.ndim != 2 or f.shape != g.shape:
            raise ValueError("luma32f and luma8 must be H x W arrays of one shape")
        out = np.zeros(cap, TAG_DTYPE)
        n = C.c_int(0)
        self._check(lib().ag_detect_planes(self._h, _p(f), 0, _p(g), 0, f.shape[1], f.shape[0], _p(out), cap, C.byref(n)))
        return _tags_to_dict(out[:n.value])

    def detect_kornia(self, img):
        """detect_kornia(&Image<u8, N>) (detector.rs:478-503): HxWxN u8 with N in {1, 3}."""
        img = np.asarray(img)
        if img.dtype != np.uint8 or img.ndim != 3 or img.shape[2] not in (1, 3):
            raise ValueError("Only support u8c1 and u8c3")  # the reference panics (detector.rs:500)
        if img.shape[2] == 1:
            img = img[:, :, 0]
        return self.detect(np.ascontiguousarray(img))

    def detect_batch(self, frames, cap_per_frame=128, return_status=False):
        """New batched entry point: frames is N x H x W or N x H x W x C (C in 2..4), u8 or u16, or
        N x H x W x C (C in 3..4) float32."""
        frames = np.asarray(frames)
        if not frames.flags.c_contiguous:
            frames = np.ascontiguousarray(frames)
        n = frames.shape[0]
        if n == 0:
            return ([], np.zeros(0, np.uint32)) if return_status else []
        fmt, w, h, st = image_format(frames[0])
        out = np.zeros((n, cap_per_frame), TAG_DTYPE)
        cnt = np.zeros(n, np.int32)
        status = np.zeros(n, np.uint32)
        self._check(lib().ag_detect_batch(self._h, _p(frames), frames.strides[0], n, w, h, st, fmt,
                                          _p(out), cap_per_frame, _p(cnt), _p(status)))
        res = [_tags_to_dict(out[i, :cnt[i]]) for i in range(n)]
        return (res, status) if return_status else res

    def detect_batch_into(self, frames, out, cnt, status=None):
        """detect_batch writing into caller-provided (ideally pinned) numpy arrays; no allocation."""
        n = frames.shape[0]
        fmt, w, h, st = image_format(frames[0])
        return self._check(lib().ag_detect_batch(self._h, _p(frames), frames.strides[0], n, w, h, st,
                                                 fmt, _p(out), out.shape[1], _p(cnt), _p(status)))

    def detect_batch_wait(self, keep_in_flight=0):
        """With option host_async = 1: block until all but the newest `keep_in_flight` detect_batch_into
        calls have delivered their results."""
        return self._check(lib().ag_detect_batch_wait(self._h, keep_in_flight))

    def detect_batch_device(self, d_frames_ptr, n_frames, width, height, fmt, d_out_ptr, cap_per_frame,
                            d_counts_ptr, d_status_ptr=None, stream=None, frame_stride=0, row_stride=0):
        """Device-resident frames, device-resident results, asynchronous on `stream` (raw pointers)."""
        return self._check(lib().ag_detect_batch_device(
            self._h, C.c_void_p(d_frames_ptr), frame_stride, n_frames, width, height, row_stride, fmt,
            C.c_void_p(d_out_ptr), cap_per_frame, C.c_void_p(d_counts_ptr),
            C.c_void_p(d_status_ptr) if d_status_ptr else None, C.c_void_p(stream) if stream else None))

    def detect_batch_device_wait(self, stream=None):
        """With option device_async = 1: order every detect_batch_device call issued so far on `stream`
        (None = block the host thread)."""
        return self._check(lib().ag_detect_batch_device_wait(self._h, C.c_void_p(stream) if stream else None))

    def dense_batch_device(self, d_frames_ptr, n_frames, width, height, fmt, stream=None):
        return self._check(lib().ag_dense_batch_device(
            self._h, C.c_void_p(d_frames_ptr), 0, n_frames, width, height, 0, fmt,
            C.c_void_p(stream) if stream else None))

    def refined_saddle_points(self, img, cap=16384):
        """TagDetector::refined_saddle_points (detector.rs:408-446) -> structured array of Saddle."""
        img = np.ascontiguousarray(img)
        fmt, w, h, st = image_format(img)
        out = np.zeros(cap, SADDLE_DTYPE)
        n = C.c_int(0)
        self._check(lib().ag_refined_saddle_points(self._h, _p(img), w, h, st, fmt, _p(out), cap, C.byref(n)))
        return out[:n.value].copy()

    def gaussian_blur_f32(self, img, sigma=1.5):
        """image_util::gaussian_blur_f32 (image_util.rs:110-206)."""
        a = np.ascontiguousarray(img, np.float32)
        out = np.empty_like(a)
        self._check(lib().ag_gaussian_blur_f32(self._h, _p(a), a.shape[1], a.shape[0], sigma, _p(out)))
        return out

    def gaussian_blur_f32_device(self, d_in_ptr, n_frames, width, height, sigma, d_out_ptr, stream=None):
        """gaussian_blur_f32 on n_frames contiguous device-resident f32 images (enqueued on `stream`)."""
        return self._check(lib().ag_gaussian_blur_f32_device(
            self._h, C.c_void_p(d_in_ptr), n_frames, width, height, sigma, C.c_void_p(d_out_ptr),
            C.c_void_p(stream) if stream else None))

    def hessian_response(self, img):
        """image_util::hessian_response (image_util.rs:72-109)."""
        a = np.ascontiguousarray(img, np.float32)
        out = np.empty_like(a)
        self._check(lib().ag_hessian_response(self._h, _p(a), a.shape[1], a.shape[0], _p(out)))
        return out

    def render_boards_device(self, d_frames_ptr, n_frames, width, height, cols=6, rows=6, seed=0,
                             stream=None):
        return self._check(lib().ag_render_boards_device(
            self._h, C.c_void_p(d_frames_ptr), n_frames, width, height, cols, rows, seed,
            C.c_void_p(stream) if stream else None))

    # -- stage taps (tests) ----------------------------------------------------------------
    def stages(self, img, want_labels=True):
        """Run one image keeping every intermediate; returns a dict shaped like oracle.front_end()."""
        img = np.ascontiguousarray(img)
        fmt, w, h, st = image_format(img)
        L = lib()
        self._check(L.ag_stage_run(self._h, _p(img), w, h, st, fmt))
        blur = np.empty((h, w), np.float32)
        resp = np.empty((h, w), np.float32)
        mt = np.zeros(2, np.float32)
        mask = np.empty((h, w), np.uint8)
        self._check(L.ag_stage_blur(self._h, _p(blur)))
        self._check(L.ag_stage_response(self._h, _p(resp)))
        self._check(L.ag_stage_threshold(self._h, _p(mt)))
        self._check(L.ag_stage_mask(self._h, _p(mask)))
        labels = None
        if want_labels:
            labels = np.empty((h, w), np.int32)
            self._check(L.ag_stage_labels(self._h, _p(labels)))
        n = C.c_int(0)
        cap = max(1 << 16, w * h // 4)
        centers = np.zeros((cap, 2), np.float32)
        self._check(L.ag_stage_centers(self._h, _p(centers), cap, C.byref(n)))
        centers = centers[:n.value].copy()
        raw = np.zeros(cap, SADDLE_DTYPE)
        self._check(L.ag_stage_saddles(self._h, 0, _p(raw), cap, C.byref(n)))
        raw = raw[:n.value].copy()
        ref = np.zeros(cap, SADDLE_DTYPE)
        self._check(L.ag_stage_saddles(self._h, 1, _p(ref), cap, C.byref(n)))
        ref = ref[:n.value].copy()
        quads = np.zeros((4096, 4), np.int32)
        self._check(L.ag_stage_board_quads(self._h, _p(quads), 4096, C.byref(n)))
        quads = quads[:n.value].copy()
        tags = np.zeros(1024, TAG_DTYPE)
        self._check(L.ag_stage_tags(self._h, _p(tags), 1024, C.byref(n)))
        return dict(blur=blur, resp=resp, min=float(mt[0]), thr=float(mt[1]), mask=mask, labels=labels,
                    centers=centers, raw=raw, refined=ref, quads=quads, tags=_tags_to_dict(tags[:n.value]))

    def _boards_from_saddles(self, saddles, img):
        """Test hook: board search + decode on a given saddle list (N x 5 float32: x, y, k, theta, phi).
        Returns (quads of the first best board [M x 4 int32], {id: corners})."""
        quads, rec, n_tags, _ = self._boards_from_saddle_batch([saddles], np.asarray(img)[None])
        return quads[0], _tags_to_dict(rec[0, :n_tags[0]])

    def _boards_from_saddle_batch(self, saddle_lists, frames, tag_cap=1024):
        """Test hook: board search + decode of frames[f] (N x H x W[...] with the saddle list
        saddle_lists[f] (N_f x 5 float32) each, all in ONE run of the board kernel's launches, which the
        handle's board options pick as in the pipeline.  Returns (quads of the first best board per
        frame [list of M_f x 4 int32], tag records [frames x tag_cap TAG_DTYPE], tag counts [frames],
        status bits [frames]).  A count of -1 means that no launch took the frame; records past the
        count are all-ones bytes unless the kernel wrote them."""
        lists = [np.ascontiguousarray(s, np.float32).reshape(-1, 5) for s in saddle_lists]
        frames = np.ascontiguousarray(frames)
        n = len(lists)
        if n != frames.shape[0] or n == 0:
            raise ValueError("one saddle list per frame, at least one frame")
        fmt, w, h, st = image_format(frames[0])
        counts = np.array([len(s) for s in lists], np.int32)
        stride = max(1, int(counts.max()))
        packed = np.zeros((n, stride, 5), np.float32)
        for f, s in enumerate(lists):
            packed[f, :len(s)] = s
        rec = np.zeros((n, tag_cap), TAG_DTYPE)
        n_quads, n_tags, status = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint32)
        quad_cap = stride // 4 + 2  # the board kernel's own bound on the quads of a list
        while True:
            quads = np.zeros((n, quad_cap, 4), np.int32)
            self._check(lib().ag_test_boards_from_saddles(
                self._h, _p(packed), stride, _p(counts), n, _p(frames), frames.strides[0], w, h, st, fmt, _p(quads),
                quad_cap, _p(n_quads), _p(rec), tag_cap, _p(n_tags), _p(status)))
            if n_quads.max() <= quad_cap:
                break
            quad_cap = int(n_quads.max())
        return [quads[f, :max(0, n_quads[f])].copy() for f in range(n)], rec, n_tags, status

    def _render_pose(self, d_frame_ptr, width, height, cols, rows, hinv, noise=False, seed=0):
        """Test hook: one frame of the device renderer under a given image -> page homography."""
        h = np.ascontiguousarray(hinv, np.float32).reshape(9)
        self._check(lib().ag_test_render_pose(self._h, C.c_void_p(d_frame_ptr), width, height, cols, rows, _p(h),
                                              1 if noise else 0, seed))

    def _board_times(self, slot, n_frames):
        """Profiling hook: n_frames x 32 u32 timing taps of the last board-kernel launch of a slot."""
        out = np.zeros((n_frames, 32), np.uint32)
        self._check(lib().ag_test_board_times(self._h, slot, _p(out), n_frames))
        return out

    def _float_luma(self, pixels):
        """Test hook: the device's to_luma32f / to_luma8 of float pixels (M x 3 or M x 4 float32)."""
        px = np.ascontiguousarray(pixels, np.float32)
        if px.ndim != 2 or px.shape[1] not in (3, 4):
            raise ValueError("want M x 3 or M x 4 float32 pixels")
        l32, l8 = np.zeros(len(px), np.float32), np.zeros(len(px), np.uint8)
        self._check(lib().ag_test_float_luma(self._h, _p(px), len(px), px.shape[1], _p(l32), _p(l8)))
        return l32, l8

    def _unorm_tables(self):
        o8, o16 = np.zeros(256, np.float32), np.zeros(65536, np.float32)
        r8, r16 = np.zeros(256, np.float32), np.zeros(65536, np.float32)
        self._check(lib().ag_test_unorm_tables(self._h, _p(o8), _p(o16), _p(r8), _p(r16)))
        return o8, o16, r8, r16


def host_chunk_frames(host_chunk, fmt):
    """Test hook (no GPU): frames per chunk of the host-buffer path for option host_chunk_frames and a
    pixel format, before the bound on the dense buffers."""
    out = C.c_longlong(0)
    if lib().ag_test_host_chunk(int(host_chunk), int(fmt), C.byref(out)) != AG_OK:
        raise ValueError("bad host_chunk_frames or format")
    return out.value


def pinned_empty(shape, dtype=np.uint8):
    """numpy array in page-locked host memory (ag_host_alloc); keep the returned array alive while in use
    and release it with pinned_free(arr)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    ptr = lib().ag_host_alloc(max(n, 1))
    if not ptr:
        raise MemoryError("ag_host_alloc(%d) failed" % n)
    buf = (C.c_uint8 * max(n, 1)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[arr.__array_interface__["data"][0]] = ptr
    return arr


_PINNED = {}


def pinned_free(arr):
    ptr = _PINNED.pop(arr.__array_interface__["data"][0], None)
    if ptr:
        lib().ag_host_free(ptr)


class MultiTagDetector:
    """detect_batch over several GPUs of one box (ag_multi_*): the batch is cut into contiguous
    frame ranges, one per device; results come back in frame order, byte-identical to one device."""

    def __init__(self, tag_family=TagFamily.T36H11, optional_detector_params=None, devices=None):
        self._h = C.c_void_p(None)
        params = optional_detector_params or DetectorParams.default_params()
        cp = params._c()
        devs = np.asarray(devices if devices is not None else [], np.int32)
        rc = lib().ag_multi_create(int(tag_family), C.byref(cp), _p(devs) if len(devs) else None, len(devs),
                                   C.byref(self._h))
        if rc != AG_OK:
            self._h = C.c_void_p(None)
            raise RuntimeError("ag_multi_create failed (%d): %s" % (rc, lib().ag_multi_last_error(None).decode()))
        self.n_devices = int(lib().ag_multi_device_count(self._h))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().ag_multi_destroy(self._h)
            self._h = C.c_void_p(None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, key, value):
        if lib().ag_multi_set_option(self._h, key.encode(), int(value)) != AG_OK:
            raise RuntimeError("aprilgrid_b200: %s" % lib().ag_multi_last_error(self._h).decode())

    def detect_batch_into(self, frames, out, cnt, status=None):
        n = frames.shape[0]
        fmt, w, h, st = image_format(frames[0])
        rc = lib().ag_multi_detect_batch(self._h, _p(frames), frames.strides[0], n, w, h, st, fmt, _p(out),
                                         out.shape[1], _p(cnt), _p(status))
        if rc != AG_OK:
            raise RuntimeError("aprilgrid_b200 error %d: %s" % (rc, lib().ag_multi_last_error(self._h).decode()))
        return rc

    def detect_batch(self, frames, cap_per_frame=128):
        frames = np.ascontiguousarray(frames)
        n = frames.shape[0]
        out = np.zeros((n, cap_per_frame), TAG_DTYPE)
        cnt = np.zeros(n, np.int32)
        status = np.zeros(n, np.uint32)
        if n:
            self.detect_batch_into(frames, out, cnt, status)
        return [_tags_to_dict(out[i, :cnt[i]]) for i in range(n)]


def saddles_as_array(s):
    """structured Saddle array -> N x 5 float32 (x, y, k, theta, phi), the oracle's layout."""
    return np.stack([s["x"], s["y"], s["k"], s["theta"], s["phi"]], axis=1).astype(np.float32) \
        if len(s) else np.zeros((0, 5), np.float32)
