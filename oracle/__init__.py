"""ctypes binding of the CPU oracle (oracle/aprilgrid_oracle.cpp) -- TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module.  The product package never does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")

FMT_L8, FMT_L16, FMT_RGB8 = 0, 1, 2
FAMILY = {"t16h5": 0, "t25h7": 1, "t25h9": 2, "t36h11": 3, "t36h11b1": 4}


def build(force=False):
    src = os.path.join(_HERE, "aprilgrid_oracle.cpp")
    if force or not os.path.exists(_LIB_PATH) or (
            os.path.exists(src) and os.path.getmtime(src) > os.path.getmtime(_LIB_PATH)):
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        f32p, i32p, u8p, vp = (C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint8),
                               C.c_void_p)
        L.orc_min_response.restype = C.c_float
        L.orc_min_response.argtypes = [vp, C.c_size_t]
        L.orc_theta_distance_degree.restype = C.c_float
        L.orc_theta_distance_degree.argtypes = [C.c_float, C.c_float]
        for n in ("orc_cross", "orc_dot", "orc_angle_degree"):
            getattr(L, n).restype = C.c_float
            getattr(L, n).argtypes = [C.c_float] * 4
        L.orc_find_xy.argtypes = [C.c_float] * 6 + [vp]
        L.orc_rotate_bits.restype = C.c_uint64
        L.orc_rotate_bits.argtypes = [C.c_uint64, C.c_int]
        L.orc_to_luma_f32.argtypes = [vp, C.c_int, C.c_int, C.c_size_t, C.c_int, vp]
        L.orc_to_luma_u8.argtypes = [vp, C.c_int, C.c_int, C.c_size_t, C.c_int, vp]
        L.orc_gaussian_blur.argtypes = [vp, C.c_int, C.c_int, C.c_float, vp]
        L.orc_hessian_response.argtypes = [vp, C.c_int, C.c_int, vp]
        L.orc_blur_taps.argtypes = [C.c_float, vp, C.c_int]
        L.orc_pixel_bfs.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, C.c_int]
        L.orc_clusters.argtypes = [vp, C.c_int, C.c_int, C.c_float, vp, vp, vp, C.c_int]
        L.orc_is_valid_quad.argtypes = [vp]
        L.orc_rochade_tables.argtypes = [C.c_int, vp, vp]
        L.orc_rochade_refine.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, C.c_int]
        L.orc_front_end.argtypes = [vp, C.c_int, C.c_int, C.c_size_t, C.c_int, C.c_float, C.c_float,
                                    vp, vp, vp, vp, vp, vp, C.c_int, vp, vp, vp, C.c_int]
        L.orc_try_find_best_board.argtypes = [vp, C.c_int, vp, C.c_int]
        L.orc_init_quads.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int]
        L.orc_tag_affine.argtypes = [vp, C.c_int, C.c_float, vp]
        L.orc_decode_positions.argtypes = [C.c_uint32, C.c_uint32, vp, C.c_int, C.c_int, C.c_float, vp]
        L.orc_bit_code.argtypes = [vp, C.c_uint32, C.c_uint32, vp, C.c_int, C.c_int, C.c_int, vp]
        L.orc_best_tag.argtypes = [C.c_uint64, C.c_int, C.c_int, vp, vp]
        L.orc_family_info.argtypes = [C.c_int, vp, vp, vp, vp, vp]
        L.orc_detect.argtypes = [C.c_int, C.c_float, C.c_float, C.c_int, vp, C.c_int, C.c_int,
                                 C.c_size_t, C.c_int, vp, C.c_int]
        L.orc_detect_batch.argtypes = [C.c_int, C.c_float, C.c_float, C.c_int, vp, C.c_size_t,
                                       C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_int, vp, C.c_int,
                                       vp, C.c_int]
        _lib = L
    return _lib


def stage_times(reset=True):
    """{stage: ms per frame} of detect() since the last reset (wall time summed over threads)."""
    ms = np.zeros(4, np.float64)
    n = C.c_longlong(0)
    L = lib()
    L.orc_stage_times.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.orc_stage_times(ms.ctypes.data_as(C.c_void_p), C.byref(n), 1 if reset else 0)
    k = max(1, n.value)
    return {"frames": int(n.value), "dense_ms": ms[0] / k, "clusters_refine_ms": ms[1] / k,
            "board_search_ms": ms[2] / k, "decode_ms": ms[3] / k}


def selftest_point_index(n, n_queries, k, mode, seed):
    L = lib()
    L.orc_selftest_point_index.argtypes = [C.c_int] * 4 + [C.c_uint]
    return int(L.orc_selftest_point_index(n, n_queries, k, mode, seed))


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


TAG_DTYPE = np.dtype([("id", np.uint32), ("xy", np.float32, (8,))])
SADDLE_FIELDS = ("x", "y", "k", "theta", "phi")


def image_format(img):
    """(fmt, width, height, row_stride_bytes) of a numpy image: HxW u8, HxW u16 or HxWx3 u8."""
    img = np.ascontiguousarray(img)
    if img.ndim == 2 and img.dtype == np.uint8:
        return FMT_L8, img.shape[1], img.shape[0], img.shape[1]
    if img.ndim == 2 and img.dtype == np.uint16:
        return FMT_L16, img.shape[1], img.shape[0], img.shape[1] * 2
    if img.ndim == 3 and img.shape[2] == 3 and img.dtype == np.uint8:
        return FMT_RGB8, img.shape[1], img.shape[0], img.shape[1] * 3
    raise ValueError("unsupported image: shape %s dtype %s" % (img.shape, img.dtype))


def to_luma_f32(img):
    img = np.ascontiguousarray(img)
    fmt, w, h, st = image_format(img)
    out = np.empty((h, w), np.float32)
    lib().orc_to_luma_f32(_p(img), w, h, st, fmt, _p(out))
    return out


def to_luma_u8(img):
    img = np.ascontiguousarray(img)
    fmt, w, h, st = image_format(img)
    out = np.empty((h, w), np.uint8)
    lib().orc_to_luma_u8(_p(img), w, h, st, fmt, _p(out))
    return out


def blur_taps(sigma=1.5):
    t = np.zeros(64, np.float32)
    n = lib().orc_blur_taps(sigma, _p(t), 64)
    return t[:n].copy()


def gaussian_blur(f32img, sigma=1.5):
    a = np.ascontiguousarray(f32img, np.float32)
    out = np.empty_like(a)
    lib().orc_gaussian_blur(_p(a), a.shape[1], a.shape[0], sigma, _p(out))
    return out


def hessian_response(f32img):
    a = np.ascontiguousarray(f32img, np.float32)
    out = np.empty_like(a)
    lib().orc_hessian_response(_p(a), a.shape[1], a.shape[0], _p(out))
    return out


def min_response(resp):
    a = np.ascontiguousarray(resp, np.float32)
    return float(lib().orc_min_response(_p(a), a.size))


def pixel_bfs(mat, x, y, thr):
    """Mutates `mat` (float32, C-contiguous) like the reference; returns [(x, y), ...]."""
    assert mat.dtype == np.float32 and mat.flags.c_contiguous
    out = np.zeros((mat.size, 2), np.uint32)
    n = lib().orc_pixel_bfs(_p(mat), mat.shape[1], mat.shape[0], x, y, thr, _p(out), mat.size)
    return [tuple(int(v) for v in r) for r in out[:n]]


def clusters(resp, thr):
    a = np.ascontiguousarray(resp, np.float32)
    h, w = a.shape
    labels = np.empty((h, w), np.int32)
    cap = max(1, a.size // 2)
    centers = np.zeros((cap, 2), np.float32)
    sizes = np.zeros(cap, np.int32)
    n = lib().orc_clusters(_p(a), w, h, np.float32(thr), _p(labels), _p(centers), _p(sizes), cap)
    return labels, centers[:n].copy(), sizes[:n].copy()


def rochade_tables(half=2):
    n = (2 * half + 1) ** 2
    p = np.zeros((6, n), np.float32)
    k = np.zeros(n, np.float32)
    lib().orc_rochade_tables(half, _p(p), _p(k))
    return p, k


def rochade_refine(blur, centers, half=2):
    a = np.ascontiguousarray(blur, np.float32)
    c = np.ascontiguousarray(centers, np.float32).reshape(-1, 2)
    out = np.zeros((max(1, len(c)), 5), np.float32)
    n = lib().orc_rochade_refine(_p(a), a.shape[1], a.shape[0], _p(c), len(c), half, _p(out), len(out))
    return out[:n].copy()


def front_end(img, min_angle=30.0, max_angle=60.0, want_labels=True):
    """All stage outputs of refined_saddle_points for one image (dict of numpy arrays)."""
    img = np.ascontiguousarray(img)
    fmt, w, h, st = image_format(img)
    blur = np.empty((h, w), np.float32)
    resp = np.empty((h, w), np.float32)
    mt = np.zeros(2, np.float32)
    labels = np.empty((h, w), np.int32) if want_labels else None
    cap = w * h // 2 + 1
    centers = np.zeros((cap, 2), np.float32)
    ncl = C.c_int(0)
    nraw = C.c_int(0)
    raw = np.zeros((cap, 5), np.float32)
    ref = np.zeros((cap, 5), np.float32)
    n = lib().orc_front_end(_p(img), w, h, st, fmt, min_angle, max_angle, _p(blur), _p(resp), _p(mt),
                            _p(labels), _p(centers), C.byref(ncl), cap, _p(raw), C.byref(nraw),
                            _p(ref), cap)
    return dict(blur=blur, resp=resp, min=float(mt[0]), thr=float(mt[1]), labels=labels,
                centers=centers[:ncl.value].copy(), raw=raw[:nraw.value].copy(),
                refined=ref[:n].copy())


def is_valid_quad(s0, d0, s1, d1):
    a = np.ascontiguousarray([s0, d0, s1, d1], np.float32)
    assert a.shape == (4, 5)
    return bool(lib().orc_is_valid_quad(_p(a)))


def try_find_best_board(saddles):
    s = np.ascontiguousarray(saddles, np.float32).reshape(-1, 5)
    out = np.zeros((max(1, len(s)), 4), np.int32)
    n = lib().orc_try_find_best_board(_p(s), len(s), _p(out), len(out))
    return None if n < 0 else out[:n].copy()


def init_quads(saddles, s0_idx):
    s = np.ascontiguousarray(saddles, np.float32).reshape(-1, 5)
    out = np.zeros((200000, 4), np.int32)
    n = lib().orc_init_quads(_p(s), len(s), s0_idx, _p(out), len(out))
    return out[:n].copy()


def tag_affine(quad_xy, side_bits, margin):
    q = np.ascontiguousarray(quad_xy, np.float32).reshape(4, 2)
    H = np.zeros(9, np.float32)
    lib().orc_tag_affine(_p(q), side_bits, margin, _p(H))
    return H.reshape(3, 3)


def decode_positions(w, h, quad_xy, border, edge, margin=0.5):
    q = np.ascontiguousarray(quad_xy, np.float32).reshape(4, 2)
    out = np.zeros((edge * edge, 2), np.float32)
    ok = lib().orc_decode_positions(w, h, _p(q), border, edge, margin, _p(out))
    return out if ok else None


def bit_code(grey, pts, valid_brightness_threshold=10, max_invalid_bit=3):
    g = np.ascontiguousarray(grey, np.uint8)
    p = np.ascontiguousarray(pts, np.float32).reshape(-1, 2)
    bits = C.c_uint64(0)
    ok = lib().orc_bit_code(_p(g), g.shape[1], g.shape[0], _p(p), len(p), valid_brightness_threshold,
                            max_invalid_bit, C.byref(bits))
    return int(bits.value) if ok else None


def rotate_bits(bits, edge):
    return int(lib().orc_rotate_bits(bits, edge))


def best_tag(bits, thres, family="t36h11"):
    i, r = C.c_int(0), C.c_int(0)
    ok = lib().orc_best_tag(bits, thres, FAMILY[family], C.byref(i), C.byref(r))
    return (i.value, r.value) if ok else None


def family_info(family="t36h11"):
    e, b, hd, n = C.c_int(0), C.c_int(0), C.c_int(0), C.c_int(0)
    codes = C.POINTER(C.c_uint64)()
    ok = lib().orc_family_info(FAMILY[family], C.byref(e), C.byref(b), C.byref(hd), C.byref(n),
                               C.byref(codes))
    assert ok
    return dict(edge=e.value, border=b.value, hamming=hd.value,
                codes=[int(codes[i]) for i in range(n.value)])


def detect(img, family="t36h11", min_angle=30.0, max_angle=60.0, max_boards=2, cap=1024):
    """TagDetector::detect -> {id: 4x2 float32 corners}."""
    img = np.ascontiguousarray(img)
    fmt, w, h, st = image_format(img)
    out = np.zeros(cap, TAG_DTYPE)
    n = lib().orc_detect(FAMILY[family], min_angle, max_angle, max_boards, _p(img), w, h, st, fmt,
                         _p(out), cap)
    assert 0 <= n <= cap, n
    return {int(t["id"]): t["xy"].reshape(4, 2).copy() for t in out[:n]}


def detect_from_saddles(img, saddles, family="t36h11", max_boards=2, cap=1024):
    """The board rounds of detect (board search + decoding, detector.rs:511-536) on a given refined
    saddle list (N x 5 float32: x, y, k, theta, phi) over img -> {id: 4x2 float32 corners}."""
    img = np.ascontiguousarray(img)
    fmt, w, h, st = image_format(img)
    s = np.ascontiguousarray(saddles, np.float32).reshape(-1, 5)
    out = np.zeros(cap, TAG_DTYPE)
    L = lib()
    L.orc_detect_from_saddles.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                          C.c_size_t, C.c_int, C.c_void_p, C.c_int]
    n = L.orc_detect_from_saddles(FAMILY[family], max_boards, _p(s), len(s), _p(img), w, h, st, fmt, _p(out), cap)
    assert 0 <= n <= cap, n
    return {int(t["id"]): t["xy"].reshape(4, 2).copy() for t in out[:n]}


def detect_planes(luma32f, luma8, family="t36h11", min_angle=30.0, max_angle=60.0, max_boards=2, cap=1024):
    """detect on a frame given as its two gray planes (to_luma32f / to_luma8 of the DynamicImage)."""
    f = np.ascontiguousarray(luma32f, np.float32)
    g = np.ascontiguousarray(luma8, np.uint8)
    assert f.shape == g.shape and f.ndim == 2
    h, w = f.shape
    out = np.zeros(cap, TAG_DTYPE)
    L = lib()
    L.orc_detect_planes.argtypes = [C.c_int, C.c_float, C.c_float, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                    C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_int]
    n = L.orc_detect_planes(FAMILY[family], min_angle, max_angle, max_boards, _p(f), 0, _p(g), 0, w, h, _p(out), cap)
    return {int(t["id"]): t["xy"].reshape(4, 2).copy() for t in out[:min(n, cap)]}


def detect_batch(frames, family="t36h11", threads=1, cap=128, max_boards=2):
    """frames: N x H x W (u8/u16) or N x H x W x 3 (u8), C-contiguous.  Returns list of dicts."""
    frames = np.ascontiguousarray(frames)
    fmt, w, h, st = image_format(frames[0])
    n = frames.shape[0]
    out = np.zeros((n, cap), TAG_DTYPE)
    cnt = np.zeros(n, np.int32)
    lib().orc_detect_batch(FAMILY[family], 30.0, 60.0, max_boards, _p(frames), frames[0].nbytes, n, w,
                           h, st, fmt, _p(out), cap, _p(cnt), threads)
    return [{int(t["id"]): t["xy"].reshape(4, 2).copy() for t in out[i, :min(cnt[i], cap)]}
            for i in range(n)]
