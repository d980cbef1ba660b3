"""Frames in the pixel formats LA8, RGBA8, LA16, RGB16 and RGBA16, and their reference results.

The CPU oracle reads L8, L16 and RGB8 frames.  The gray conversion of the other integer formats is,
in `image` 0.25, the one of those formats applied to a plane derived with integer arithmetic: alpha
is dropped, and colour is the luma (2126 R + 7152 G + 722 B) / 10000 computed in the source width,
then scaled like L8 (u8) or L16 (u16).  `reference_frame` restates that derivation in numpy (int64),
and `RefOracle` runs the oracle on the derived frame, so that a frame in any integer format has a
reference result:

    LA8 -> its L8 plane             RGBA8 -> its RGB8 channels
    LA16 -> its L16 plane           RGB16, RGBA16 -> the L16 plane of Y16

The painted decode-gate frames of synth (synth.gate_frames) are built here in these formats too."""
import numpy as np

import synth

NEW_FORMATS = ("la8", "rgba8", "la16", "rgb16", "rgba16")
ALPHA_FORMATS = ("la8", "rgba8", "la16", "rgba16")
CODE = {"l8": 0, "l16": 1, "rgb8": 2, "la8": 4, "rgba8": 5, "la16": 6, "rgb16": 7, "rgba16": 8}
BPP = {"l8": 1, "l16": 2, "rgb8": 3, "la8": 2, "rgba8": 4, "la16": 4, "rgb16": 6, "rgba16": 8}
# (channels, dtype) -> format name of an H x W x channels frame
_CHANNELS = {(2, np.uint8): "la8", (3, np.uint8): "rgb8", (4, np.uint8): "rgba8",
             (2, np.uint16): "la16", (3, np.uint16): "rgb16", (4, np.uint16): "rgba16"}


def format_of(img):
    if img.ndim == 2:
        return "l16" if img.dtype == np.uint16 else "l8"
    return _CHANNELS[(img.shape[2], img.dtype.type)]


def luma_int(img):
    """Y8 / Y16 of an H x W x C frame as int64: the luma channel, or (2126 R + 7152 G + 722 B) / 10000."""
    a = img.astype(np.int64)
    if img.shape[2] == 2:
        return a[:, :, 0]
    return (2126 * a[:, :, 0] + 7152 * a[:, :, 1] + 722 * a[:, :, 2]) // 10000


def reference_frame(img):
    """The L8 / L16 / RGB8 frame whose gray conversion is that of `img` (returned as is if it is one)."""
    fmt = format_of(img)
    if fmt in ("l8", "l16", "rgb8"):
        return img
    if fmt == "rgba8":
        return np.ascontiguousarray(img[:, :, :3])
    return np.ascontiguousarray(luma_int(img).astype(img.dtype))


class RefOracle:
    """The oracle, with every image argument replaced by its reference_frame.  image_format reports the
    library's format codes (for helpers that pass frames to the host build of the board core)."""
    _IMAGE_FIRST = ("to_luma_f32", "to_luma_u8", "front_end", "detect", "detect_from_saddles")

    def __init__(self, oracle):
        self._o = oracle

    def __getattr__(self, name):
        f = getattr(self._o, name)
        if name in self._IMAGE_FIRST:
            return lambda img, *a, **k: f(reference_frame(np.ascontiguousarray(img)), *a, **k)
        if name == "detect_batch":
            return lambda frames, *a, **k: f(np.stack([reference_frame(x) for x in frames]), *a, **k)
        return f

    @staticmethod
    def image_format(img):
        img = np.ascontiguousarray(img)
        return CODE[format_of(img)], img.shape[1], img.shape[0], img.strides[0]


# ---- painted decode-gate frames -----------------------------------------------------------------------
_RGB16_CACHE = {}
Y16_MAX_SUM = 10000 * 65535  # 2126 + 7152 + 722 = 10000: every channel at 65535


def rgb16_for_sum(s):
    """(r, g, b) u16 with 2126 r + 7152 g + 722 b == s exactly (s even), close to gray."""
    if s not in _RGB16_CACHE:
        m = s // 10000
        r, g = np.meshgrid(np.arange(max(0, m - 400), min(65535, m + 400) + 1, dtype=np.int64),
                           np.arange(max(0, m - 8), min(65535, m + 8) + 1, dtype=np.int64), indexing="ij")
        rem = s - 2126 * r - 7152 * g
        ok = (rem >= 0) & (rem % 722 == 0) & (rem // 722 <= 65535)
        k = np.flatnonzero(ok.ravel())
        assert len(k), s
        b = rem.ravel()[k] // 722
        best = np.argmin(np.abs(r.ravel()[k] - b) + np.abs(g.ravel()[k] - b))
        _RGB16_CACHE[s] = (int(r.ravel()[k][best]), int(g.ravel()[k][best]), int(b[best]))
    return _RGB16_CACHE[s]


def rgb16_word(t, upper):
    """Y16 = (2126 r + 7152 g + 722 b) / 10000 truncated, to_luma8 = (Y16 + 128) / 257: 10000 (257 t - 128)
    is the smallest sum giving t; the weights are even, so 10000 (257 t + 129) - 2 is the largest."""
    s = 10000 * max(0, 257 * t - 128) if upper else min(Y16_MAX_SUM, 10000 * (257 * t + 129) - 2)
    return rgb16_for_sum(s)


def alpha_plane(shape, wide, seed=0):
    """Random alpha of an H x W frame (u8, or u16 when `wide`)."""
    return np.random.default_rng(seed).integers(0, 65536 if wide else 256, shape).astype(
        np.uint16 if wide else np.uint8)


def encode(l8, painted, fmt, mids):
    """synth.encode for the formats of NEW_FORMATS, with random alpha: unpainted pixels convert exactly
    (v * 257, gray RGB); painted ones sit on a to_luma8 boundary, above / below `mids[(y, x)]` -- LA8 and
    LA16 with the L8 / L16 words of synth, RGBA8 with its RGB8 words, RGB16 / RGBA16 with rgb16_word."""
    if fmt in ("l8", "l16", "rgb8"):
        return synth.encode(l8, painted, fmt, mids)
    if fmt in ALPHA_FORMATS:
        base = encode(l8, painted, {"la8": "l8", "rgba8": "rgb8", "la16": "l16", "rgba16": "rgb16"}[fmt], mids)
        if base.ndim == 2:
            base = base[:, :, None]
        return np.concatenate([base, alpha_plane(l8.shape, fmt.endswith("16"))[:, :, None]], axis=2)
    out = np.repeat((l8.astype(np.uint16) * np.uint16(257))[:, :, None], 3, axis=2)  # rgb16
    for key, v in painted.items():
        out[key] = rgb16_word(v, v > mids[key])
    return out


def scenario_frame(scene, tags, fmt):
    """synth.scenario_frame in any format: paint `tags`, encode in fmt; raises if the painted frame no
    longer has the board the painting used."""
    l8, painted = synth.paint(scene, [t[1] for t in tags])
    mids = {}
    for pts, t in zip(scene["pts"], tags):
        if t[1] is not None:
            m = (min(t[1]) + max(t[1]) + 1) // 2
            for x, y in pts:
                mids[(synth.ref_round_u32(y), synth.ref_round_u32(x))] = m
    frame = encode(l8, painted, fmt, mids)
    if not synth.gate_guard(scene, reference_frame(frame)):
        raise AssertionError("painted %s frame of %s lost its board" % (fmt, scene["family"]))
    return frame


def gate_frames(family, fmts=NEW_FORMATS):
    """The scenarios of synth.gate_frames in formats `fmts`: [(name, scene, tags, fmt, frame, max_boards)]."""
    small = synth.gate_scene(family)
    big = synth.gate_scene(family, w=960, h=720, cols=8, rows=6)
    sets = [("gates", small, synth.gate_tags(small["fam"], 20), (2,)),
            ("repeat_3_9", small, synth.repeat_tags(small["fam"], 20, 3, 9), (2,)),
            ("rejected", small, synth.rejected_board_tags(small["fam"], 20), (1, 2, 3)),
            ("repeat_3_40", big, synth.repeat_tags(big["fam"], 48, 3, 40), (2,))]
    return [(name, scene, tags, fmt, scenario_frame(scene, tags, fmt), mbs)
            for name, scene, tags, mbs in sets for fmt in fmts]
