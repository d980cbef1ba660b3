"""Frames in the pixel formats RGB32F and RGBA32F, and their reference results.

`image` 0.25 converts Rgb<f32> to gray in f64 (include/aprilgrid_b200.h states the reading):

    S = RN64(RN64(2126 r + 7152 g) + 722 b)            r, g, b widened to f64; products exact
    L = (f32) clamp(RN64(S / 10000), -f32::MAX, f32::MAX)
    to_luma32f = L,  to_luma8 = round_half_away(RN32(clamp(L, 0, 1) * 255))

`planes` restates it in numpy, in f64 or exactly (numpy's f64 operations round each result once and never
fuse; np.round rounds half to even and is not used).  The oracle reads L8 / L16 / RGB8 frames and a Luma<f32>
plane (its format 3, the input of detect_planes); `FloatOracle` runs it on the restated planes: the f32
plane for the stencils, the u8 plane as an L8 frame for bit sampling.

Three facts the tests build on (checked by tests/test_float_formats_host.py):
- gray pixels: R = G = B = v gives L = v for every finite f32 v (10000 v is exact in f64);
- the L8 round trip: v = f32(k / 255) gives to_luma8 = k and to_luma32f = the L8 path's RN(k / 255), so a
  float frame widened from an L8 frame has exactly the L8 frame's two planes;
- exact ties: channels v + (33, -8, -11) ulp(v) in the binade of v give S = 10000 (v + ulp / 2) exactly, an
  f32 tie that the f64 division leaves to round-to-even."""
import ctypes as C

import numpy as np

import synth

FLOAT_FORMATS = ("rgb32f", "rgba32f")
CODE = {"rgb32f": 9, "rgba32f": 10}
BPP = {"rgb32f": 12, "rgba32f": 16}
CHANNELS = {"rgb32f": 3, "rgba32f": 4}
F32_MAX = float(np.finfo(np.float32).max)  # Enlargeable::clamp_from's bound (Bounded::max_value)
TIE_OFFSETS = (33, -8, -11)  # 2126 * 33 - 7152 * 8 - 722 * 11 = 5000


def format_of(frame):
    return {3: "rgb32f", 4: "rgba32f"}[frame.shape[-1]]


def round_half_away(y):
    """round() of non-negative f32 values, exactly: y + 0.5 is exact in f64."""
    return np.floor(np.asarray(y, np.float32).astype(np.float64) + 0.5)


def planes(px):
    """(to_luma32f f32, to_luma8 u8) of float pixels (... x C, C >= 3; alpha ignored)."""
    px = np.asarray(px, np.float32)
    r, g, b = (px[..., i].astype(np.float64) for i in range(3))
    s = 2126.0 * r + 7152.0 * g
    s = s + 722.0 * b
    q = np.minimum(np.maximum(s / 10000.0, -F32_MAX), F32_MAX)
    l32 = q.astype(np.float32)
    y = np.minimum(np.maximum(l32, np.float32(0)), np.float32(1)) * np.float32(255)
    return l32, round_half_away(y).astype(np.uint8)


def unorm8(l8):
    """f32(k / 255), correctly rounded (what to_luma32f gives an L8 frame)."""
    return np.asarray(l8).astype(np.float32) / np.float32(255)


def widen(l8, fmt, seed=0, noise=0.0, lo=None, hi=None):
    """An L8 frame as a float frame: every channel starts from f32(v / 255); `noise` > 0 adds a different
    uniform noise to R, G and B (so that a swapped channel order or a wrong weight changes the luma);
    lo / hi rescale the frame to that range first.  Alpha is random in [0, 1]."""
    rng = np.random.default_rng(seed)
    base = unorm8(l8)
    if lo is not None:
        base = (np.float32(lo) + base * np.float32(hi - lo)).astype(np.float32)
    chans = [(base + (rng.uniform(-noise, noise, l8.shape).astype(np.float32) if noise else np.float32(0)))
             .astype(np.float32) for _ in range(3)]
    if fmt == "rgba32f":
        chans.append(rng.uniform(0, 1, l8.shape).astype(np.float32))
    return np.ascontiguousarray(np.stack(chans, axis=2))


# ---- pixel sets of the conversion -----------------------------------------------------------------------
def ulp(v):
    v = np.asarray(v, np.float32)
    return (np.nextafter(v, np.float32(np.inf)) - v).astype(np.float32)


def tie_triples(n=200000, seed=0):
    """n x 3 f32 pixels v + (33, -8, -11) ulp(v), all in the binade of v (positive and negative v, from the
    smallest normals to 2^127): S = 10000 (v + ulp / 2) exactly."""
    rng = np.random.default_rng(seed)
    e = rng.integers(-125, 127, n)
    m = rng.integers(16, (1 << 23) - 40, n)  # mantissa away from both ends of the binade
    mag = np.ldexp(1.0 + m / float(1 << 23), e).astype(np.float32)
    v = np.where(rng.integers(0, 2, n) == 1, -mag, mag).astype(np.float32)
    u = ulp(np.abs(v)) * np.sign(v).astype(np.float32)
    px = np.stack([v + np.float32(k) * u for k in TIE_OFFSETS], axis=1).astype(np.float32)
    return px


def luma8_steps():
    """For each k in 1..255: (the largest f32 L with to_luma8 = k - 1, the smallest with to_luma8 = k),
    found by bisection on the bit patterns of [0, 1] (to_luma8 is monotone there).  Returns 255 x 2 f32."""
    lo = np.zeros(255, np.uint32)                       # to_luma8(lo) < k
    hi = np.full(255, np.float32(1).view(np.uint32))    # to_luma8(hi) >= k
    k = np.arange(1, 256)
    while (hi - lo > 1).any():
        mid = lo + (hi - lo) // 2
        below = planes(np.repeat(mid.view(np.float32)[:, None], 3, axis=1))[1] < k
        lo = np.where(below, mid, lo)
        hi = np.where(below, hi, mid)
    return np.stack([lo.view(np.float32), hi.view(np.float32)], axis=1)


def uniform_pixels(n, seed=0):
    return np.random.default_rng(seed).uniform(0, 1, (n, 4)).astype(np.float32)


def wide_range_pixels(n, seed=0):
    """n x 4 pixels over the whole finite f32 range: random bit patterns (normals and subnormals of both
    signs), values in [-0.5, 3], and +-0, subnormals and +-f32::MAX mixed into every channel."""
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 1 << 32, (n, 4), dtype=np.uint64).astype(np.uint32)
    bits[(bits & 0x7f800000) == 0x7f800000] &= 0xbfffffff  # no infinities / NaN
    px = bits.view(np.float32).copy()
    third = n // 3
    px[:third] = rng.uniform(-0.5, 3.0, (third, 4)).astype(np.float32)
    special = np.array([0.0, -0.0, 1e-45, -1e-45, 1e-40, -3e-39, F32_MAX, -F32_MAX, 1.0, -1.0], np.float32)
    mix = rng.integers(0, len(special), (n // 3, 4))
    pick = rng.integers(0, 2, (n // 3, 4)) == 1
    seg = px[third:2 * third]
    seg[pick] = special[mix][pick]
    return px


# ---- the oracle on the restated planes ----------------------------------------------------------------
class FloatOracle:
    """The oracle on a float frame: front_end on its f32 plane (the oracle's format 3), detect through
    detect_planes, detect_from_saddles on its u8 plane; every other function passes through.
    image_format reports the library's format codes (for the host build of the board core)."""

    def __init__(self, oracle):
        self._o = oracle

    def __getattr__(self, name):
        return getattr(self._o, name)

    @staticmethod
    def image_format(img):
        img = np.ascontiguousarray(img)
        return CODE[format_of(img)], img.shape[1], img.shape[0], img.strides[0]

    def to_luma_f32(self, img):
        return planes(img)[0]

    def to_luma_u8(self, img):
        return planes(img)[1]

    def front_end(self, img, min_angle=30.0, max_angle=60.0, want_labels=True):
        l32 = np.ascontiguousarray(planes(img)[0])
        h, w = l32.shape
        blur, resp = np.empty((h, w), np.float32), np.empty((h, w), np.float32)
        mt = np.zeros(2, np.float32)
        labels = np.empty((h, w), np.int32) if want_labels else None
        cap = w * h // 2 + 1
        centers = np.zeros((cap, 2), np.float32)
        raw, ref = np.zeros((cap, 5), np.float32), np.zeros((cap, 5), np.float32)
        ncl, nraw = C.c_int(0), C.c_int(0)
        p = self._o._p
        n = self._o.lib().orc_front_end(p(l32), w, h, 4 * w, 3, min_angle, max_angle, p(blur), p(resp), p(mt),
                                        p(labels), p(centers), C.byref(ncl), cap, p(raw), C.byref(nraw), p(ref), cap)
        return dict(blur=blur, resp=resp, min=float(mt[0]), thr=float(mt[1]), labels=labels,
                    centers=centers[:ncl.value].copy(), raw=raw[:nraw.value].copy(), refined=ref[:n].copy())

    def detect(self, img, family="t36h11", min_angle=30.0, max_angle=60.0, max_boards=2):
        l32, l8 = planes(img)
        return self._o.detect_planes(l32, l8, family=family, min_angle=min_angle, max_angle=max_angle,
                                     max_boards=max_boards)

    def detect_from_saddles(self, img, saddles, family="t36h11", max_boards=2):
        return self._o.detect_from_saddles(planes(img)[1], saddles, family=family, max_boards=max_boards)


# ---- painted decode-gate frames -------------------------------------------------------------------------
_STEPS = []


def step_value(t, upper):
    """The f32 luma on a to_luma8 step: the smallest L giving t when `upper`, else the largest."""
    if not _STEPS:
        _STEPS.append(luma8_steps())
    s = _STEPS[0]
    if upper:
        return np.float32(0) if t == 0 else s[t - 1, 1]
    return np.float32(1) if t == 255 else s[t, 0]


def encode(l8, painted, fmt, mids):
    """synth.encode for the float formats: unpainted pixels are gray f32(v / 255) (their planes are the L8
    frame's); painted ones are gray at a to_luma8 step, above / below `mids[(y, x)]`.  Random alpha."""
    out = widen(l8, fmt)
    for key, v in painted.items():
        out[key][:3] = step_value(v, v > mids[key])
    return out


def gate_guard(oracle, scene, frame):
    """synth.gate_guard on the float frame's f32 plane."""
    s2 = FloatOracle(oracle).front_end(frame, want_labels=False)["refined"]
    q2 = oracle.try_find_best_board(s2)
    want = scene["saddles"][scene["quads"], :2]
    return q2 is not None and q2.shape == scene["quads"].shape and np.array_equal(s2[q2, :2], want)


def scenario_frame(oracle, scene, tags, fmt):
    l8, painted = synth.paint(scene, [t[1] for t in tags])
    mids = {}
    for pts, t in zip(scene["pts"], tags):
        if t[1] is not None:
            m = (min(t[1]) + max(t[1]) + 1) // 2
            for x, y in pts:
                mids[(synth.ref_round_u32(y), synth.ref_round_u32(x))] = m
    frame = encode(l8, painted, fmt, mids)
    if not gate_guard(oracle, scene, frame):
        raise AssertionError("painted %s frame of %s lost its board" % (fmt, scene["family"]))
    return frame


def gate_frames(oracle, family, fmts=FLOAT_FORMATS):
    """The scenarios of synth.gate_frames in the float formats: [(name, scene, tags, fmt, frame, max_boards)]."""
    small = synth.gate_scene(family)
    big = synth.gate_scene(family, w=960, h=720, cols=8, rows=6)
    sets = [("gates", small, synth.gate_tags(small["fam"], 20), (2,)),
            ("repeat_3_9", small, synth.repeat_tags(small["fam"], 20, 3, 9), (2,)),
            ("rejected", small, synth.rejected_board_tags(small["fam"], 20), (1, 2, 3)),
            ("repeat_3_40", big, synth.repeat_tags(big["fam"], 48, 3, 40), (2,))]
    return [(name, scene, tags, fmt, scenario_frame(oracle, scene, tags, fmt), mbs)
            for name, scene, tags, mbs in sets for fmt in fmts]
