"""Synthetic AprilGrid frames for the tests (numpy; no GPU, no reference files needed).

Board geometry as in the reference's chart generator (scripts/generate_aprilgrid.py:1086-1167):
cols x rows tags of side 1, gaps 0.3, black squares of side 0.3 at every lattice corner, ids
row-major from the BOTTOM row, each tag (edge + 2*border)^2 cells, bit "1" = white, MSB first,
rows from the top of the tag.  Paper 200, ink 30.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _codes(family="t36h11"):
    import oracle
    return oracle.family_info(family)


def board_is_white(X, Y, cols, rows, codes, edge, border):
    """Vectorised page lookup: X right, Y down, units = tag sides. Returns bool array."""
    sp, pitch = 0.3, 1.3
    wb, hb = cols * pitch + sp, rows * pitch + sp
    inside = (X >= 0) & (Y >= 0) & (X < wb) & (Y < hb)
    Yb = hb - Y
    i = np.floor(X / pitch).astype(np.int64)
    j = np.floor(Yb / pitch).astype(np.int64)
    fx = X - i * pitch
    fy = Yb - j * pitch
    corner = (fx < sp) & (fy < sp)
    in_tag = (fx >= sp) & (fy >= sp) & (i < cols) & (j < rows) & (i >= 0) & (j >= 0)
    cells = edge + 2 * border
    tx = fx - sp
    ty = 1.0 - (fy - sp)
    cc = np.clip((tx * cells).astype(np.int64), 0, cells - 1)
    cr = np.clip((ty * cells).astype(np.int64), 0, cells - 1)
    in_border = (cc < border) | (cr < border) | (cc >= border + edge) | (cr >= border + edge)
    idx = np.clip((cr - border) * edge + (cc - border), 0, edge * edge - 1)
    tag_id = np.clip(j * cols + i, 0, len(codes) - 1)
    code = np.asarray(codes, dtype=np.uint64)[tag_id]
    bit = ((code >> (edge * edge - 1 - idx).astype(np.uint64)) & np.uint64(1)).astype(bool)
    white = np.ones(X.shape, bool)
    white[inside & corner] = False
    tag_black = inside & in_tag & (in_border | ~bit)
    white[tag_black] = False
    return white


def homography(w, h, cols, rows, seed, tag_px=None, max_rot_deg=45.0, max_tilt_deg=30.0):
    rng = np.random.default_rng(seed)
    sp = 0.3
    wb, hb = cols * (1 + sp) + sp, rows * (1 + sp) + sp
    alpha = np.deg2rad(rng.uniform(-max_rot_deg, max_rot_deg))
    bx = np.deg2rad(rng.uniform(-max_tilt_deg, max_tilt_deg))
    by = np.deg2rad(rng.uniform(-max_tilt_deg, max_tilt_deg))
    t = float(tag_px) if tag_px else rng.uniform(60.0, 120.0)
    focal = 1.2 * w
    ca, sa, cx, sx, cy, sy = np.cos(alpha), np.sin(alpha), np.cos(bx), np.sin(bx), np.cos(by), np.sin(by)
    r = np.array([[cy, 0.0], [sx * sy, cx], [-cx * sy, sx]])
    q = np.array([[ca * r[0, 0] - sa * r[1, 0], ca * r[0, 1] - sa * r[1, 1]],
                  [sa * r[0, 0] + ca * r[1, 0], sa * r[0, 1] + ca * r[1, 1]],
                  [r[2, 0], r[2, 1]]])
    for _ in range(10):
        H = np.array([
            [focal * t * q[0, 0], focal * t * q[0, 1], -focal * t * (q[0, 0] * wb + q[0, 1] * hb) / 2],
            [focal * t * q[1, 0], focal * t * q[1, 1], -focal * t * (q[1, 0] * wb + q[1, 1] * hb) / 2],
            [t * q[2, 0], t * q[2, 1], focal - t * (q[2, 0] * wb + q[2, 1] * hb) / 2]])
        c = np.array([[0, 0, 1], [wb, 0, 1], [wb, hb, 1], [0, hb, 1]], float).T
        p = H @ c
        p = p[:2] / p[2]
        mn, mx = p.min(axis=1), p.max(axis=1)
        margin = 12.0
        bw, bh = mx - mn
        if bw > w - 2 * margin or bh > h - 2 * margin:
            t *= 0.9 * min((w - 2 * margin) / bw, (h - 2 * margin) / bh)
            continue
        tx = margin - mn[0] + rng.uniform() * (w - 2 * margin - bw)
        ty = margin - mn[1] + rng.uniform() * (h - 2 * margin - bh)
        T = np.array([[1, 0, tx], [0, 1, ty], [0, 0, 1.0]])
        return T @ H
    raise RuntimeError("board does not fit")


def render_board_numpy(w=640, h=480, cols=6, rows=6, seed=0, tag_px=None, family="t36h11", noise=2.0,
                       ss=4, H=None, dtype=np.uint8, rgb=False):
    fam = _codes(family)
    if H is None:
        H = homography(w, h, cols, rows, seed, tag_px)
    Hinv = np.linalg.inv(H)
    ys, xs = np.mgrid[0:h, 0:w].astype(np.float64)
    acc = np.zeros((h, w), np.float64)
    for sy in range(ss):
        for sx in range(ss):
            px = xs + (sx + 0.5) * (1.4 / ss) - 0.7
            py = ys + (sy + 0.5) * (1.4 / ss) - 0.7
            W = Hinv[2, 0] * px + Hinv[2, 1] * py + Hinv[2, 2]
            X = (Hinv[0, 0] * px + Hinv[0, 1] * py + Hinv[0, 2]) / W
            Y = (Hinv[1, 0] * px + Hinv[1, 1] * py + Hinv[1, 2]) / W
            acc += board_is_white(X, Y, cols, rows, fam["codes"], fam["edge"], fam["border"])
    v = 30.0 + 170.0 * acc / (ss * ss)
    rng = np.random.default_rng(seed + 7919)
    if noise > 0:
        v = v + rng.normal(0.0, noise, v.shape)
    v = np.clip(np.rint(v), 0, 255)
    if dtype == np.uint16:
        img = (v * 257.0).astype(np.uint16)
    else:
        img = v.astype(np.uint8)
    if rgb:
        img = np.repeat(img[:, :, None], 3, axis=2).copy()
    return img


def composite_boards(tiles, tile_w, tile_h, grid_cols, canvas=None):
    """Boards of different layouts, one per tile of a grid (row-major), in one L8 frame.
    tiles: (cols, rows, seed, tag_px) each.  Every board numbers its tags from 0, so the id ranges
    overlap and a board found in a later round of the board search overwrites earlier ids.
    canvas: (height, width) of a larger paper-white frame the grid is placed in at (0, 0)."""
    grid_rows = (len(tiles) + grid_cols - 1) // grid_cols
    h, w = canvas or (grid_rows * tile_h, grid_cols * tile_w)
    img = np.full((h, w), 200, np.uint8)
    for k, (cols, rows, seed, tag_px) in enumerate(tiles):
        r, c = divmod(k, grid_cols)
        img[r * tile_h:(r + 1) * tile_h, c * tile_w:(c + 1) * tile_w] = render_board_numpy(
            tile_w, tile_h, cols=cols, rows=rows, seed=seed, tag_px=tag_px)
    return img


# 1280 x 960: 456 refined saddles (512-saddle tier of the board kernel); the oracle finds the 3 x 3
# board with one round, the 6 x 6 board (overwriting all 9 ids) with two, and with three rounds 12 ids
# carry the 4 x 3 board's corners
FOUR_BOARDS = ([(6, 6, 3, 44.0), (4, 3, 5, 60.0), (5, 4, 8, 52.0), (3, 3, 11, 70.0)], 640, 480, 2)
# four small boards in the same 1280 x 960 frame, <= 320 refined saddles (the small tier); every
# round up to the fourth changes the result
SMALL_BOARDS = ([(3, 3, 11, 60.0), (4, 3, 5, 52.0), (3, 2, 7, 60.0), (2, 2, 2, 70.0)], 320, 320, 2)


def fixture_like_frames(n, w, h, seed=0, **kw):
    return np.stack([render_board_numpy(w, h, seed=seed + i, **kw) for i in range(n)])


def ulp_step(v, k):
    v = np.float32(v)
    for _ in range(abs(int(k))):
        v = np.nextafter(v, np.float32(np.inf if k > 0 else -np.inf), dtype=np.float32)
    return v


def adversarial_saddle_sets(base, rng):
    """Saddle lists sitting ON the discontinuous gates of the board search (detector.rs:556-560, :603;
    saddle.rs:18-66): theta differences of 5 / 80 degrees give or take a few ulps, theta at x.5
    (round() boundaries of the seed histogram), and projective distortions that put the
    opposite-angle difference of the tag quads at 10 degrees +- 1e-4."""
    n = len(base)
    d2 = ((base[:, None, :2] - base[None, :, :2]) ** 2).sum(-1)
    near = np.argsort(d2, axis=1)[:, 1:12]

    def wrap(t):  # keep theta in (-90, 90]: theta_distance_degree works modulo 180
        t = np.float32(t)
        while t > 90:
            t = np.float32(t - np.float32(180))
        while t <= -90:
            t = np.float32(t + np.float32(180))
        return t

    for trial in range(24):  # (a) theta gates, (b) histogram boundaries
        s = base.copy()
        for _ in range(40):
            i = int(rng.integers(n))
            j = int(near[i, rng.integers(near.shape[1])])
            gate = np.float32(rng.choice([5.0, -5.0, 80.0, -80.0, 100.0, -100.0, 175.0, -175.0]))
            s[j, 3] = wrap(ulp_step(np.float32(s[i, 3] + gate), int(rng.integers(-2, 3))))
        for _ in range(25):
            i = int(rng.integers(n))
            s[i, 3] = wrap(ulp_step(np.float32(np.floor(s[i, 3]) + 0.5), int(rng.integers(-2, 3))))
        yield "theta%d" % trial, s

    def angle_gap(q):  # |a0 - a2| of a quad given as 4 x 2 (saddle.rs:47-54), float64
        v = [q[(k + 1) % 4] - q[k] for k in range(4)]
        ang = lambda a, b: np.degrees(np.arctan2(b[1] * a[0] - b[0] * a[1], a[0] * b[0] + a[1] * b[1]))
        return abs(ang(v[0], v[1]) - ang(v[2], v[3]))

    c = base[:, :2].mean(axis=0)
    ref = base[np.argsort(((base[:, :2] - c) ** 2).sum(-1))[:1], :2][0]
    quad_ix = np.argsort(((base[:, :2] - ref) ** 2).sum(-1))[:4]
    order = quad_ix[np.argsort(np.arctan2(*(base[quad_ix, :2] - base[quad_ix, :2].mean(0)).T[::-1]))]
    for trial in range(16):  # (c) projective keystone: bisect its strength onto the 10-degree gate
        ax = rng.uniform(-1, 1, 2)
        ax /= np.linalg.norm(ax)

        def warp(strength, pts):
            wgt = 1.0 + strength * ((pts - c) @ ax)
            return c + (pts - c) / wgt[:, None]

        lo, hi = 0.0, 4e-3
        target = 10.0 + rng.choice([-1e-4, -1e-5, 0.0, 1e-5, 1e-4])
        for _ in range(60):
            mid = 0.5 * (lo + hi)
            if angle_gap(warp(mid, base[order, :2].astype(np.float64))) < target:
                lo = mid
            else:
                hi = mid
        s = base.copy()
        s[:, :2] = warp(0.5 * (lo + hi), base[:, :2].astype(np.float64)).astype(np.float32)
        yield "keystone%d" % trial, s



# ---- decode-gate scenarios -------------------------------------------------------------------------
# Frames whose tag samples are painted onto the thresholds of bit_code and best_tag (detector.rs:74-169).
# A board is rendered without noise; the oracle's refined saddles and best-board quads give, through
# decode_positions, the exact f32 sample points of every tag, and the painter writes chosen gray values
# at (round(x), round(y)) -- the first sample is the most significant bit.  Painting only those pixels
# leaves the board's corner saddles in place; every painted frame is checked for that (gate_guard).

def ref_round_u32(v):
    """Rust `f32::round() as u32`: halves away from zero, saturating at 0."""
    v = float(v)
    return int(np.floor(v + 0.5)) if v > 0 else 0


def ref_bit_code(grey, pts, vbt=10, max_invalid=3):
    """bit_code (detector.rs:74-122) restated on integers; None where the reference returns None."""
    h, w = grey.shape
    b = []
    for x, y in pts:
        xi, yi = ref_round_u32(x), ref_round_u32(y)
        if xi >= w or yi >= h:
            return None
        b.append(int(grey[yi, xi]))
    lo, hi = min(b), max(b)
    if hi - lo < 50:
        return None
    mid = (lo + hi + 1) // 2  # round((lo + hi) / 2): a half rounds up (away from zero)
    bits, invalid = 0, 0
    for i, v in enumerate(reversed(b)):  # the last sample is bit 0
        invalid += abs(mid - v) < vbt
        bits |= (v > mid) << i
    return None if invalid > max_invalid else bits


def ref_rotate_bits(bits, edge):
    """rotate_bits (detector.rs:124-140)."""
    out, count = 0, 0
    for r in range(edge - 1, -1, -1):
        for c in range(edge):
            out |= ((bits >> (r + c * edge)) & 1) << count
            count += 1
    return out


def ref_best_tag(bits, hamming, codes, edge):
    """best_tag (detector.rs:142-169): (id, rotation) of the first code within hamming - 1 bits."""
    for rot in range(4):
        scores = [bin(int(c) ^ bits).count("1") for c in codes]
        best = min(scores)
        if best < hamming:
            return scores.index(best), rot
        bits = ref_rotate_bits(bits, edge)
    return None


def ref_corners(saddles, quad, rot):
    """try_decode_quad's corners (detector.rs:467-469): rotate_left(rot), then reverse."""
    return np.stack([saddles[quad[(3 - j + rot) % 4], :2] for j in range(4)]).astype(np.float32)


# family -> render seed of the 640 x 480 5 x 4 board and of the 960 x 720 8 x 6 board: poses on which
# every painted frame keeps its board (gate_guard)
GATE_SEEDS = {"t16h5": (6, 2), "t25h7": (6, 1), "t25h9": (6, 3), "t36h11": (6, 2), "t36h11b1": (9, 4)}
GATE_FAMILIES = tuple(GATE_SEEDS)


def gate_scene(family, w=640, h=480, cols=5, rows=4, seed=None, tag_px=60.0):
    """A noise-free board and what the painter needs of it: the oracle's refined saddles, the quads of
    its best board in visiting order and every quad's sample points."""
    import oracle
    fam = oracle.family_info(family)
    if seed is None:
        seed = GATE_SEEDS[family][0 if cols * rows <= 20 else 1]
    img = render_board_numpy(w, h, cols=cols, rows=rows, seed=seed, tag_px=tag_px, family=family, noise=0.0)
    s = oracle.front_end(img, want_labels=False)["refined"]
    quads = oracle.try_find_best_board(s)
    assert quads is not None and len(quads) == cols * rows, (family, None if quads is None else len(quads))
    pts = [oracle.decode_positions(w, h, s[q, :2], fam["border"], fam["edge"]) for q in quads]
    assert all(p is not None for p in pts)
    return dict(family=family, img=img, saddles=s, quads=quads, pts=pts, fam=fam)


def code_values(code, ns, lo, hi):
    """Sample values painting `code` (MSB = first sample)."""
    return [hi if (int(code) >> (ns - 1 - i)) & 1 else lo for i in range(ns)]


def spread(k, ns, skip=()):
    """k sample indices spread over the tag."""
    out = []
    for j in range(k):
        i = (j * ns) // k + (ns // (2 * k))
        while i in out or i in skip:
            i = (i + 1) % ns
        out.append(i)
    return out


def gate_tags(fam, n_tags):
    """One scenario per tag of a 20-tag board: [(name, values or None, expectation)], expectation
    being ('id', id, rot), ('absent', id) or ('none',) (nothing may decode from the tag)."""
    edge, H, codes = fam["edge"], fam["hamming"], fam["codes"]
    ns, n_codes = edge * edge, len(fam["codes"])
    ids = iter([0, n_codes - 1] + [int(v) for v in np.linspace(1, n_codes - 2, n_tags).round()])
    used = set()

    def next_id():
        i = next(ids)
        while i in used:
            i = next(ids)
        used.add(i)
        return i

    tags = []
    for _ in range(3):  # exact codes, ids 0 and n_codes - 1 among them
        i = next_id()
        tags.append(("exact", code_values(codes[i], ns, 40, 190), ("id", i, 0)))
    for k in range(1, H + 1):  # k bit errors: k < hamming decodes, k = hamming does not
        i = next_id()
        v = code_values(codes[i], ns, 45, 185)
        for j in spread(k, ns):
            v[j] = 45 if v[j] == 185 else 185
        tags.append(("errors%d" % k, v, ("id", i, 0) if k < H else ("absent", i)))
    for r in (1, 2, 3):  # rotate_bits^r of the code: found at rotation 4 - r
        i = next_id()
        c = int(codes[i])
        for _ in range(r):
            c = ref_rotate_bits(c, edge)
        tags.append(("rotation%d" % r, code_values(c, ns, 35, 180), ("id", i, 4 - r)))
    for d in (49, 50):  # contrast gate max - min < 50
        i = next_id()
        tags.append(("contrast%d" % d, code_values(codes[i], ns, 100, 100 + d),
                     ("id", i, 0) if d >= 50 else ("absent", i)))
    # (lo + hi) / 2 = 120.5: round() gives 121, round-half-even would give 120; samples at exactly 121
    # are bit 0 (strict v > mid), samples at 122 bit 1
    i = next_id()
    v = code_values(codes[i], ns, 60, 181)
    zeros = [j for j in range(ns) if v[j] == 60][1:4]
    for j in zeros:
        v[j] = 121
    tags.append(("halfmid_at_mid", v, ("id", i, 0)))
    i = next_id()
    v = code_values(codes[i], ns, 60, 181)
    zeros = [j for j in range(ns) if v[j] == 60][1:2]
    ones = [j for j in range(ns) if v[j] == 181][1:3]
    for j in zeros:
        v[j] = 121
    for j in ones:
        v[j] = 122
    tags.append(("halfmid_above", v, ("id", i, 0)))
    # uncertain samples |mid - v| < 10 at most 3: mid = 120, 3 or 4 samples 9 away, 4 exactly 10 away
    for n9 in (3, 4):
        i = next_id()
        v = code_values(codes[i], ns, 70, 170)
        lo_j = [j for j in range(ns) if v[j] == 70][1:]
        hi_j = [j for j in range(ns) if v[j] == 170][1:]
        near = (lo_j[:2] + hi_j[:2])[:n9]
        far = lo_j[2:4] + hi_j[2:4]
        for j in near:
            v[j] = 111 if v[j] == 70 else 129
        for j in far:
            v[j] = 110 if v[j] == 70 else 130
        tags.append(("uncertain%d" % n9, v, ("id", i, 0) if n9 <= 3 else ("absent", i)))
    while len(tags) < n_tags:
        i = next_id()
        tags.append(("exact", code_values(codes[i], ns, 40, 190), ("id", i, 0)))
    return tags


def paint(scene, values_per_tag):
    """L8 frame with the tag samples painted, and the painted pixels' values (y, x) -> v."""
    img = scene["img"].copy()
    painted = {}
    for pts, vals in zip(scene["pts"], values_per_tag):
        if vals is None:
            continue
        for (x, y), v in zip(pts, vals):
            key = (ref_round_u32(y), ref_round_u32(x))
            assert painted.get(key, v) == v, "two samples on one pixel"
            painted[key] = v
            img[key] = v
    return img, painted


# Gray values through the other formats, placed on the boundaries of to_luma8 (image 0.25): a painted
# value t above the tag's mid level is written as the smallest word that converts to t, one at or below
# it as the largest -- so a conversion that is off by one on either side moves max - min and mid.
def l16_word(t, upper):
    """(v + 128) / 257 == t; 257 t - 128 (= 257 (t - 1) + 129) is the smallest such v, 257 t + 128 the largest."""
    return max(0, 257 * t - 128) if upper else min(65535, 257 * t + 128)


_RGB_CACHE = {}


def rgb_for_sum(s):
    """(r, g, b) with 2126 r + 7152 g + 722 b == s exactly (the sRGB luma weights of to_luma8)."""
    if s not in _RGB_CACHE:
        r, g = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
        rem = s - 2126 * r - 7152 * g
        ok = (rem >= 0) & (rem % 722 == 0) & (rem // 722 <= 255)
        k = np.flatnonzero(ok.ravel())
        assert len(k), s
        # the candidate closest to gray keeps the frame's look
        b = rem.ravel()[k] // 722
        best = np.argmin(np.abs(r.ravel()[k] - b) + np.abs(g.ravel()[k] - b))
        _RGB_CACHE[s] = (int(r.ravel()[k][best]), int(g.ravel()[k][best]), int(b[best]))
    return _RGB_CACHE[s]


def rgb_word(t, upper):
    """luma = (2126 r + 7152 g + 722 b) / 10000, truncated: 10000 t is the smallest sum giving t; the
    weights are even, so 10000 (t + 1) - 2 is the largest."""
    return rgb_for_sum(10000 * t if upper else 10000 * (t + 1) - 2)


def encode(l8, painted, fmt, mids):
    """The L8 frame in format fmt ('l8', 'l16', 'rgb8').  Unpainted pixels convert exactly (v * 257,
    gray RGB); painted ones sit on a conversion boundary, above / below `mids[(y, x)]`."""
    if fmt == "l8":
        return l8.copy()
    if fmt == "l16":
        out = l8.astype(np.uint16) * np.uint16(257)
        for key, v in painted.items():
            out[key] = l16_word(v, v > mids[key])
        return out
    out = np.repeat(l8[:, :, None], 3, axis=2).copy()
    for key, v in painted.items():
        out[key] = rgb_word(v, v > mids[key])
    return out


def gate_guard(scene, frame):
    """The board the painting used must be the oracle's best board of the painted frame: the same
    corner coordinates, quad for quad, in visiting order."""
    import oracle
    s2 = oracle.front_end(frame, want_labels=False)["refined"]
    q2 = oracle.try_find_best_board(s2)
    want = scene["saddles"][scene["quads"], :2]
    return q2 is not None and q2.shape == scene["quads"].shape and np.array_equal(s2[q2, :2], want)


def scenario_frame(scene, tags, fmt):
    """Paint `tags` ([(name, values, expectation)] in visiting order) and encode in fmt; raises if the
    painted frame no longer has the board the painting used."""
    l8, painted = paint(scene, [t[1] for t in tags])
    mids = {}
    for pts, t in zip(scene["pts"], tags):
        if t[1] is not None:
            m = (min(t[1]) + max(t[1]) + 1) // 2
            for x, y in pts:
                mids[(ref_round_u32(y), ref_round_u32(x))] = m
    frame = encode(l8, painted, fmt, mids)
    if not gate_guard(scene, frame):
        raise AssertionError("painted %s frame of %s lost its board" % (fmt, scene["family"]))
    return frame


def check_expectations(scene, tags, got, grey):
    """The oracle's (or any) result `got` on a painted frame is the one each tag was built for; the
    integer restatement of bit_code / best_tag agrees with the decoded outcome of every tag.  Returns
    the number of tags checked."""
    import oracle
    fam = scene["fam"]
    s = scene["saddles"]
    for k, (q, pts, (name, vals, exp)) in enumerate(zip(scene["quads"], scene["pts"], tags)):
        bits = ref_bit_code(grey, pts)
        assert oracle.bit_code(grey, pts) == bits, (k, name)
        res = None if bits is None else ref_best_tag(bits, fam["hamming"], fam["codes"], fam["edge"])
        if bits is not None:
            assert oracle.best_tag(bits, fam["hamming"], scene["family"]) == res, (k, name)
        if exp[0] == "id":
            assert res == (exp[1], exp[2]), (k, name, res, exp)
            assert exp[1] in got and np.array_equal(got[exp[1]], ref_corners(s, q, exp[2])), (k, name)
        elif exp[0] == "shadowed":  # decodes, but a later quad of the same id overwrites it
            assert res == (exp[1], 0), (k, name, res, exp)
            assert exp[1] in got and not np.array_equal(got[exp[1]], ref_corners(s, q, 0)), (k, name)
        elif exp[0] == "absent":
            assert res is None or res[0] != exp[1], (k, name, res)
            assert exp[1] not in got, (k, name)
        else:
            assert res is None, (k, name, res)
    return len(tags)


def repeat_tags(fam, n_tags, pos_a, pos_b):
    """Tags pos_a < pos_b (visiting order) carry one code; every other tag a code of its own, or none
    (one flat gray level: the contrast gate rejects it) once the family runs out of codes."""
    edge, codes = fam["edge"], fam["codes"]
    ns, n_codes = edge * edge, len(codes)
    rep = n_codes // 2
    others = iter([i for i in range(n_codes) if i != rep])
    tags = []
    for k in range(n_tags):
        if k in (pos_a, pos_b):
            exp = ("shadowed", rep) if k == pos_a else ("id", rep, 0)
            tags.append(("repeat", code_values(codes[rep], ns, 40, 190), exp))
            continue
        i = next(others, None)
        if i is None:
            tags.append(("flat", [120] * ns, ("none",)))
        else:
            tags.append(("exact", code_values(codes[i], ns, 40, 190), ("id", i, 0)))
    return tags


def rejected_board_tags(fam, n_tags, keep=(0, 7, 13)):
    """A board whose tags are flat gray (rejected by the contrast gate) but for a few exact codes: the
    saddles of the decoded few are removed and later rounds search the rest of the board again."""
    edge, codes = fam["edge"], fam["codes"]
    ns = edge * edge
    tags = []
    for k in range(n_tags):
        if k in keep:
            i = len(codes) - 1 - keep.index(k)
            tags.append(("exact", code_values(codes[i], ns, 40, 190), ("id", i, 0)))
        else:
            tags.append(("flat", [90 + k] * ns, ("none",)))
    return tags


def gate_frames(family):
    """Every painted full-pipeline frame of a family: [(name, scene, tags, fmt, frame, max_boards)]."""
    small = gate_scene(family)
    big = gate_scene(family, w=960, h=720, cols=8, rows=6)
    sets = [("gates", small, gate_tags(small["fam"], 20), (2,)),
            ("repeat_3_9", small, repeat_tags(small["fam"], 20, 3, 9), (2,)),
            ("rejected", small, rejected_board_tags(small["fam"], 20), (1, 2, 3)),
            ("repeat_3_40", big, repeat_tags(big["fam"], 48, 3, 40), (2,))]
    out = []
    for name, scene, tags, mbs in sets:
        for fmt in ("l8", "l16", "rgb8"):
            out.append((name, scene, tags, fmt, scenario_frame(scene, tags, fmt), mbs))
    return out


# ---- cases set up through a given saddle list ------------------------------------------------------
def paint_codes(img, sample_sets, codes, edge, lo=40, hi=190):
    """Paint code codes[k] on sample set k (None = leave it)."""
    ns = edge * edge
    for pts, c in zip(sample_sets, codes):
        if pts is None or c is None:
            continue
        for (x, y), v in zip(pts, code_values(c, ns, lo, hi)):
            img[ref_round_u32(y), ref_round_u32(x)] = v
    return img


def _board_samples(s, quads, w, h, fam):
    import oracle
    return [oracle.decode_positions(w, h, s[q, :2], fam["border"], fam["edge"]) for q in quads]


def half_sample_case(scene, trials=2000, seed=0):
    """Translate the saddle list by f32 steps until a sample point of a board tag lies exactly on
    k + 0.5 (k even) in x or y, where round() and round-half-even part: paint pixels k and k + 1 with
    opposite bits, the one round() reads carrying the code's bit, and hamming - 1 errors elsewhere in
    the tag -- it decodes with round() and would not with round-half-even.  Returns (saddles, image,
    intended id, tag index) or None when no translation was found."""
    import oracle
    fam, s0 = scene["fam"], scene["saddles"]
    h, w = scene["img"].shape[:2]
    edge, H, codes = fam["edge"], fam["hamming"], fam["codes"]
    ns = edge * edge
    rng = np.random.default_rng(seed)
    for _ in range(trials):
        d = rng.uniform(-3.0, 3.0, 2).astype(np.float32)
        s = s0.copy()
        s[:, 0] = s[:, 0] + d[0]
        s[:, 1] = s[:, 1] + d[1]
        pts = _board_samples(s, scene["quads"], w, h, fam)
        hit = None
        for t, p in enumerate(pts):
            if p is None:
                continue
            for j, (x, y) in enumerate(p):
                for axis, v in ((0, x), (1, y)):
                    f = float(v) - np.floor(float(v))
                    if f == 0.5 and int(np.floor(float(v))) % 2 == 0:
                        hit = (t, j, axis)
            if hit:
                break
        if not hit:
            continue
        q = oracle.try_find_best_board(s)
        if q is None or not np.array_equal(q, scene["quads"]):
            continue
        t, j, axis = hit
        img = np.full((h, w), 120, np.uint8)
        ids = [(7 * k + 3) % len(codes) for k in range(len(pts))]
        ids[t] = len(codes) - 1 if t != len(codes) - 1 else 0
        paint_codes(img, pts, [codes[i] for i in ids], edge)
        vals = code_values(codes[ids[t]], ns, 40, 190)
        for e in spread(H - 1, ns, skip=(j,)):  # hamming - 1 errors away from the half sample
            x, y = pts[t][e]
            img[ref_round_u32(y), ref_round_u32(x)] = 40 if vals[e] == 190 else 190
        x, y = pts[t][j]
        xi, yi = ref_round_u32(x), ref_round_u32(y)
        other = (yi, xi - 1) if axis == 0 else (yi - 1, xi)  # the pixel round-half-even would read
        img[yi, xi] = vals[j]
        img[other] = 40 if vals[j] == 190 else 190
        return s, img, ids[t], t
    return None


def edge_corner_cases(scene):
    """The board's corner saddles alone, translated so that the right-most (bottom-most) corner sits at
    exactly w - 0.5 (h - 0.5), which round() takes to w (h) -- decode_positions rejects the quad -- and
    one ulp below it, where the quad decodes.  Every saddle stays inside [0, w) x [0, h).  Returns
    [(name, saddles, image, id of the corner's tag, decodes?)]."""
    import oracle
    fam = scene["fam"]
    h, w = scene["img"].shape[:2]
    codes = fam["codes"]
    sub = scene["saddles"][np.unique(scene["quads"].ravel())]
    out = []
    for axis, size in ((0, w), (1, h)):
        edge_v = np.float32(size - 0.5)
        below = np.nextafter(edge_v, np.float32(0))
        i = int(np.argmax(sub[:, axis]))
        # paint from the "below" placement (the rejected placement has no sample points)
        placed = {}
        for name, target in (("at", edge_v), ("below", below)):
            dv = np.float32(target - sub[i, axis])
            s = sub.copy()
            s[:, axis] = s[:, axis] + dv
            assert s[i, axis] == target and s[:, axis].min() >= 0 and s[:, axis].max() < size
            placed[name] = s
        s = placed["below"]
        q = oracle.try_find_best_board(s)
        q_at = oracle.try_find_best_board(placed["at"])
        assert q is not None and q_at is not None and np.array_equal(q, q_at)
        t = [k for k, qq in enumerate(q) if i in qq]
        assert len(t) == 1
        pts = _board_samples(s, q, w, h, fam)
        assert all(p is not None for p in pts)
        ids = [(11 * k + 2) % len(codes) for k in range(len(q))]
        img = paint_codes(np.full((h, w), 120, np.uint8), pts, [codes[k] for k in ids], fam["edge"])
        for name in ("at", "below"):
            out.append(("%s_%s" % ("xy"[axis], name), placed[name], img, ids[t[0]], name == "below"))
    return out
