"""The pixel formats LA8, RGBA8, LA16, RGB16 and RGBA16 on the CPU: the integer restatement of their
gray conversion (formats_ref) against the oracle's conversions of L8 / L16 / RGB8, and tag decoding at
its gates through the host build of the board core (csrc/ag_board_core.h `luma8_at`) in each of them."""
import numpy as np
import pytest

import formats_ref as fr
import synth
from test_board_core_host import hb, host_detect  # noqa: F401  (hb is a fixture)
from test_decode_gates_host import same_tags

FORMATS = list(fr.NEW_FORMATS)
CHANNELS = {"la8": (2, np.uint8), "rgba8": (4, np.uint8), "la16": (2, np.uint16), "rgb16": (3, np.uint16),
            "rgba16": (4, np.uint16)}


def want_planes(img):
    """to_luma32f / to_luma8 of a frame, restated: Y / 255 or Y / 65535 (f32, correctly rounded) and Y8 or
    (Y16 + 128) / 257."""
    y = fr.luma_int(img)
    if img.dtype == np.uint16:
        return np.float32(y) / np.float32(65535), ((y + 128) // 257).astype(np.uint8)
    return np.float32(y) / np.float32(255), y.astype(np.uint8)


def frames(fmt, seed):
    c, dt = CHANNELS[fmt]
    top = np.iinfo(dt).max
    rng = np.random.default_rng(seed)
    out = [rng.integers(0, top + 1, (37, 41, c)).astype(dt),  # random, alpha included
           np.zeros((3, 5, c), dt), np.full((3, 5, c), top, dt)]
    for ch in range(c - (1 if c in (2, 4) else 0)):  # one colour channel at its maximum
        one = np.zeros((3, 5, c), dt)
        one[:, :, ch] = top
        out.append(one)
    return out


@pytest.mark.parametrize("fmt", FORMATS)
def test_reference_conversions(oracle, fmt):
    """The restatement equals the oracle's conversion of the reference frame (for RGBA8, the oracle's own
    RGB8 luma), alpha never enters it, and white is Y16 = 65535 / to_luma8 = 255 / to_luma32f = 1.0."""
    for k, img in enumerate(frames(fmt, seed=len(fmt))):
        f32, u8 = want_planes(img)
        ref = fr.reference_frame(img)
        got32, got8 = oracle.to_luma_f32(ref), oracle.to_luma_u8(ref)
        assert np.array_equal(got32.view(np.uint32), f32.view(np.uint32)), (fmt, k)
        assert np.array_equal(got8, u8), (fmt, k)
        if img.shape[2] in (2, 4):
            for a in (0, np.iinfo(img.dtype).max):
                other = img.copy()
                other[:, :, -1] = a
                assert np.array_equal(fr.reference_frame(other), ref), (fmt, k, a)
    c, dt = CHANNELS[fmt]
    full = np.full((2, 2, c), np.iinfo(dt).max, dt)
    assert fr.luma_int(full).min() == np.iinfo(dt).max
    assert oracle.to_luma_u8(fr.reference_frame(full)).min() == 255
    assert oracle.to_luma_f32(fr.reference_frame(full)).min() == np.float32(1.0)


def test_rgb16_boundary_words():
    """The painted RGB16 words reach exactly the first and last Y16 of each to_luma8 value."""
    for t in (0, 1, 40, 110, 129, 190, 254, 255):
        for upper in (True, False):
            r, g, b = fr.rgb16_word(t, upper)
            s = 2126 * r + 7152 * g + 722 * b
            y = s // 10000
            assert (y + 128) // 257 == t, (t, upper)
            if upper:
                assert y == max(0, 257 * t - 128)
            else:
                assert y == min(65535, 257 * t + 128)
                assert s == min(fr.Y16_MAX_SUM, 10000 * (257 * t + 129) - 2)


_FRAMES = {}


def frames_of(family):
    if family not in _FRAMES:
        _FRAMES[family] = fr.gate_frames(family)
    return _FRAMES[family]


@pytest.mark.parametrize("family", list(synth.GATE_FAMILIES))
def test_painted_frames_identical_to_reference(hb, pkg, oracle, family):  # noqa: F811
    """The decode-gate scenarios of test_decode_gates_host in every new format: the reference decodes
    what each painting was built for, and the host build of the board core, sampling the frame in its
    own format, equals it."""
    ref = fr.RefOracle(oracle)
    tf = pkg.TagFamily[family.upper()]
    n_tags = dict.fromkeys(FORMATS, 0)
    for name, scene, tags, fmt, frame, mbs in frames_of(family):
        saddles = ref.front_end(frame, want_labels=False)["refined"]
        grey = ref.to_luma_u8(frame)
        for mb in mbs:
            want = ref.detect(frame, family=family, max_boards=mb)
            n_tags[fmt] += synth.check_expectations(scene, tags, want, grey)
            got, quads, status, _ = host_detect(hb, pkg, ref, frame, saddles=saddles, family=tf, max_boards=mb)
            assert status == 0, (name, fmt, mb)
            assert np.array_equal(quads, oracle.try_find_best_board(saddles)), (name, fmt)
            same_tags(got, want)
    assert all(n == 20 + 20 + 3 * 20 + 48 for n in n_tags.values()), n_tags


@pytest.mark.parametrize("family", list(synth.GATE_FAMILIES))
def test_translated_saddle_lists_identical_to_reference(hb, pkg, oracle, family):  # noqa: F811
    ref = fr.RefOracle(oracle)
    tf = pkg.TagFamily[family.upper()]
    scene = synth.gate_scene(family)
    s, img, tid, _ = synth.half_sample_case(scene)
    for name, s, img, tid, decodes in [("half_sample", s, img, tid, True)] + synth.edge_corner_cases(scene):
        for fmt in FORMATS:
            frame = fr.encode(img, {}, fmt, {})
            want = ref.detect_from_saddles(frame, s, family=family)
            assert (tid in want) == decodes, (name, fmt)
            got, _, status, _ = host_detect(hb, pkg, ref, frame, saddles=s, family=tf)
            assert status == 0
            same_tags(got, want)
