"""The pixel formats RGB32F and RGBA32F on the CPU: the gray conversion the kernels share
(csrc/ag_float_luma.h, through its host build in tests/host_float_luma.cpp) against the numpy restatement
of float_formats_ref, the facts the GPU tests rely on, tag decoding at its gates through the host build of
the board core sampling float frames, and the frames per host-path chunk of every format."""
import ctypes as C

import numpy as np
import pytest

import float_formats_ref as ffr
import synth
from test_board_core_host import hb, host_detect  # noqa: F401  (hb is a fixture)
from test_decode_gates_host import same_tags

FORMATS = list(ffr.FLOAT_FORMATS)


def host_luma(hb, px):
    px = np.ascontiguousarray(px, np.float32)
    l32, l8 = np.zeros(len(px), np.float32), np.zeros(len(px), np.uint8)
    vp = C.c_void_p
    assert hb.hb_float_luma(px.ctypes.data_as(vp), C.c_longlong(len(px)), px.shape[1], l32.ctypes.data_as(vp),
                            l8.ctypes.data_as(vp)) == 0
    return l32, l8


def assert_same_planes(got, want, what):
    bad = np.flatnonzero(got[0].view(np.uint32) != want[0].view(np.uint32))
    assert len(bad) == 0, (what, "to_luma32f", len(bad), bad[:4])
    bad = np.flatnonzero(got[1] != want[1])
    assert len(bad) == 0, (what, "to_luma8", len(bad), bad[:4])


def pixel_sets():
    """The pixel sets of the conversion tests, 10^7 pixels and more in all (each in both layouts)."""
    steps = ffr.luma8_steps().ravel()
    return {"uniform": ffr.uniform_pixels(3_000_000, seed=1),
            "wide_range": ffr.wide_range_pixels(1_800_000, seed=2),
            "ties": ffr.tie_triples(200_000, seed=3),
            "steps": np.repeat(steps[:, None], 3, axis=1)}


def test_conversion_equals_restatement(hb):  # noqa: F811
    n = 0
    for name, px in pixel_sets().items():
        for c in (3, 4):
            p = np.ascontiguousarray(px[:, :c]) if px.shape[1] >= c else np.concatenate(
                [px, np.full((len(px), 1), 0.5, np.float32)], axis=1)
            assert_same_planes(host_luma(hb, p), ffr.planes(p), (name, c))
            n += len(p)
        # alpha never enters: the same colours with other alpha values
        if px.shape[1] == 4:
            p = px.copy()
            p[:, 3] = -p[:, 3]
            assert_same_planes(host_luma(hb, p), ffr.planes(px[:, :3]), (name, "alpha"))
            n += len(p)
    assert n >= 10_000_000, n


def test_gray_pixels_keep_their_value():
    px = ffr.wide_range_pixels(500_000, seed=4)[:, 0]
    l32, _ = ffr.planes(np.repeat(px[:, None], 3, axis=1))
    assert np.array_equal(l32.view(np.uint32), px.view(np.uint32))


def test_l8_round_trip(oracle):
    """f32(k / 255) as R = G = B gives to_luma8 = k and the L8 frame's to_luma32f; a widened L8 frame with
    random alpha has the L8 frame's planes."""
    k = np.arange(256, dtype=np.uint8)
    l32, l8 = ffr.planes(np.repeat(ffr.unorm8(k)[:, None], 3, axis=1))
    assert np.array_equal(l8, k)
    assert np.array_equal(l32.view(np.uint32), oracle.to_luma_f32(k[None, :])[0].view(np.uint32))
    img = synth.render_board_numpy(320, 240, seed=2, tag_px=40.0)
    for fmt in FORMATS:
        l32, l8 = ffr.planes(ffr.widen(img, fmt, seed=5))
        assert np.array_equal(l8, img)
        assert np.array_equal(l32.view(np.uint32), oracle.to_luma_f32(img).view(np.uint32))


def test_tie_triples_are_exact_ties():
    """S = 10000 (v + ulp / 2) exactly, and L is v + ulp / 2 rounded to even -- where a conversion in f32
    arithmetic errs on about half of them."""
    px = ffr.tie_triples(100_000, seed=6)
    w = np.array([2126.0, 7152.0, 722.0])
    # v = G + 8 ulp (all three channels share v's binade, so they share its ulp)
    v = (px[:, 1] + np.float32(8) * ffr.ulp(np.abs(px[:, 1])) * np.sign(px[:, 1]).astype(np.float32)).astype(np.float32)
    u =ffr.ulp(np.abs(v)).astype(np.float64) * np.sign(v)
    s = (w[0] * px[:, 0].astype(np.float64) + w[1] * px[:, 1].astype(np.float64)) + w[2] * px[:, 2].astype(np.float64)
    assert np.array_equal(s, 10000.0 * (v.astype(np.float64) + u / 2))
    l32, _ = ffr.planes(px)
    even = (v.view(np.uint32) & 1) == 0
    want = np.where(even, v, (v.astype(np.float64) + u).astype(np.float32))
    assert np.array_equal(l32.view(np.uint32), want.view(np.uint32))
    f32_way = ((np.float32(0.2126) * px[:, 0] + np.float32(0.7152) * px[:, 1]) + np.float32(0.0722) * px[:, 2])
    assert (f32_way.view(np.uint32) != l32.view(np.uint32)).mean() > 0.25


def test_luma8_steps():
    s = ffr.luma8_steps()
    k = np.arange(1, 256)
    for side, want in ((0, k - 1), (1, k)):
        _, l8 = ffr.planes(np.repeat(s[:, side, None], 3, axis=1))
        assert np.array_equal(l8, want), side
    assert np.array_equal(np.nextafter(s[:, 1], np.float32(0)).view(np.uint32), s[:, 0].view(np.uint32))


# ---- tag decoding at its gates ---------------------------------------------------------------------
_FRAMES = {}


def frames_of(oracle, family):
    if family not in _FRAMES:
        _FRAMES[family] = ffr.gate_frames(oracle, family)
    return _FRAMES[family]


@pytest.mark.parametrize("family", list(synth.GATE_FAMILIES))
def test_painted_frames_identical_to_reference(hb, pkg, oracle, family):  # noqa: F811
    """The decode-gate scenarios in both float formats, painted on the to_luma8 steps: the reference on the
    u8 plane decodes what each painting was built for, and the host build of the board core, sampling the
    float frame itself, equals it."""
    ref = ffr.FloatOracle(oracle)
    tf = pkg.TagFamily[family.upper()]
    n_tags = dict.fromkeys(FORMATS, 0)
    for name, scene, tags, fmt, frame, mbs in frames_of(oracle, family):
        saddles = ref.front_end(frame, want_labels=False)["refined"]
        grey = ref.to_luma_u8(frame)
        for mb in mbs:
            want = ref.detect(frame, family=family, max_boards=mb)
            assert want == {} or sorted(want) == sorted(ref.detect_from_saddles(frame, saddles, family=family,
                                                                                max_boards=mb))
            n_tags[fmt] += synth.check_expectations(scene, tags, want, grey)
            got, quads, status, _ = host_detect(hb, pkg, ref, frame, saddles=saddles, family=tf, max_boards=mb)
            assert status == 0, (name, fmt, mb)
            assert np.array_equal(quads, oracle.try_find_best_board(saddles)), (name, fmt)
            same_tags(got, want)
    assert all(n == 20 + 20 + 3 * 20 + 48 for n in n_tags.values()), n_tags


# ---- bindings and chunking -------------------------------------------------------------------------
def test_image_format_maps_float_frames(pkg):
    for c, code in ((3, pkg.FMT_RGB32F), (4, pkg.FMT_RGBA32F)):
        img = np.zeros((6, 10, c), np.float32)
        assert pkg.image_format(img) == (code, 10, 6, 10 * c * 4)
    for bad in (np.zeros((6, 10), np.float32), np.zeros((6, 10, 2), np.float32), np.zeros((6, 10, 3), np.float64)):
        with pytest.raises(ValueError):
            pkg.image_format(bad)


def test_host_chunk_per_format(pkg):
    """The eight integer formats keep the option's chunk; the float formats get at most the bytes of an
    RGBA16 chunk: max(1, chunk * 8 / bytes_per_pixel)."""
    codes = {0: 1, 1: 2, 2: 3, 4: 2, 5: 4, 6: 4, 7: 6, 8: 8, 9: 12, 10: 16}
    for chunk in (1, 2, 3, 7, 8, 64, 128, 1000, 65535):
        for code, bpp in codes.items():
            want = chunk if bpp <= 8 else max(1, chunk * 8 // bpp)
            assert pkg.host_chunk_frames(chunk, code) == want, (chunk, code)
    assert pkg.host_chunk_frames(128, pkg.FMT_RGB32F) == 85 and pkg.host_chunk_frames(128, pkg.FMT_RGBA32F) == 64
    for bad_fmt in (3, 11, -1):
        with pytest.raises(ValueError):
            pkg.host_chunk_frames(128, bad_fmt)
