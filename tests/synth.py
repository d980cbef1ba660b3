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
