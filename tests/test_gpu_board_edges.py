"""The board kernel (K6) at the edges where its routing changes, against the oracle.  Needs a B200: -m gpu.

Which code searches a frame depends on its refined-saddle count n and on the image size: the
launch of a split batch (n <= 320, then up to the tier, then the rest on large images), whether
the saddles live on chip (n <= the tier: 320 / 512 / 1024 / 4096) or in the frame's global
workspace, whether the throughput path may take the frame (n <= 1024 and on chip), the tier itself
(from the image area: 1536 x 1024 and 3072 x 2048 are the last images of the 512 and 1024 tiers)
and the bucket size of the grid (32 px buckets while the image has at most 1408 of them, 8192 in the
general path of the 4096 tier: 1408 x 1024 and 4096 x 2048 are the last images with 32 px buckets).

Saddle lists of an exact size sit on both sides of every such cut, several to a batch, through the
board kernel's test hook in every board option that changes the routing.  Each frame must be taken by
a launch (count >= 0), carry no status bit, give the oracle's quads and tags bit for bit on the same
list, and give the same bytes as the list run alone.  Boards wider than the tag lattice must be
flagged, never truncated.  Real frames of every class go through the device pipeline in one batch."""
import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu

AG_FRAME_BOARD_OVERFLOW = 4
GROWABLE = 1 | 2  # AG_FRAME_CLUSTER_OVERFLOW | AG_FRAME_SADDLE_OVERFLOW

# Boards whose oracle saddle lists the exact-size lists are cut from: a 12 x 9 board of 582 refined
# saddles in 1280 x 768, and a 29 x 20 board of 2903 in 3072 x 1536; each is pasted at (0, 0) of the
# canvas, whose rows below it stay paper-white (the band that takes the decoy saddles).
TILES = {"12x9": dict(w=1280, h=768, cols=12, rows=9, seed=4, tag_px=44.0, ss=4),
         "29x20": dict(w=3072, h=1536, cols=29, rows=20, seed=9, tag_px=70.0, ss=2)}

# canvas: (width, height, tile, saddle counts, max_saddles option; 0 = automatic)
CANVASES = {
    # 512 tier; 320 / 512 / 1024 / 2048 (the automatic max_saddles) saddles
    "1280x1024": (1280, 1024, "12x9", (0, 1, 4, 5, 319, 320, 321, 511, 512, 513, 1023, 1024, 1025, 2048), 0),
    # the last image of the 512 tier and the first of the 1024 tier
    "1536x1024": (1536, 1024, "12x9", (320, 321, 512, 513, 1024, 1025), 0),
    "1537x1024": (1537, 1024, "12x9", (320, 321, 512, 513, 1024, 1025), 0),
    # the last image of the 1024 tier and the first of the 4096 tier (three launches)
    "3072x2048": (3072, 2048, "29x20", (320, 321, 1024, 1025, 4096, 4097), 0),
    "3073x2048": (3073, 2048, "29x20", (320, 321, 1024, 1025, 4096, 4097), 0),
    # 1408 buckets of 32 px, then 64 px buckets
    "1408x1024": (1408, 1024, "12x9", (320, 321, 1024), 0),
    "1409x1024": (1409, 1024, "12x9", (320, 321, 1024), 0),
    # 8192 buckets of 32 px in the 4096 tier's general path, then 64 px buckets
    "4096x2048": (4096, 2048, "29x20", (1025, 4096, 4097), 0),
    "4097x2048": (4097, 2048, "29x20", (1025, 4096, 4097), 0),
    # the hard limit of a saddle list: global workspace, general path
    "3840x2160": (3840, 2160, "29x20", (16384,), 16384),
}

# board options that change which launch, layout and path take a frame; all but "latency" make
# every batch (and every frame run alone) a split batch of batch layouts
OPTION_SETS = {
    "batch": dict(board_batch_frames=1),
    "latency": dict(),  # few frames: one launch, 16 warps per frame
    "unsplit": dict(board_batch_frames=1, board_split=0),
    "general": dict(board_batch_frames=1, board_fast=0),
    "tier0": dict(board_batch_frames=1, board_saddle_tier=0),
    "tier1": dict(board_batch_frames=1, board_saddle_tier=1),
    "tier2": dict(board_batch_frames=1, board_saddle_tier=2),
    "warps1": dict(board_batch_frames=1, board_warps=1),
    "warps4": dict(board_batch_frames=1, board_warps=4),
}

_TILE_CACHE, _CANVAS_CACHE, _LIST_CACHE = {}, {}, {}


def tile(name, oracle):
    if name not in _TILE_CACHE:
        kw = dict(TILES[name])
        img = synth.render_board_numpy(kw.pop("w"), kw.pop("h"), **kw)
        _TILE_CACHE[name] = img, oracle.front_end(img, want_labels=False)["refined"]
    return _TILE_CACHE[name]


def canvas(key, oracle):
    if key not in _CANVAS_CACHE:
        w, h, tname = CANVASES[key][:3]
        img = np.full((h, w), 200, np.uint8)
        t, _ = tile(tname, oracle)
        img[:t.shape[0], :t.shape[1]] = t
        _CANVAS_CACHE[key] = img
    return _CANVAS_CACHE[key]


def theta_bins(theta):
    """round(theta) as the board search bins it (f32::round: halves away from zero)."""
    t = np.asarray(theta, np.float64)
    return (np.sign(t) * np.floor(np.abs(t) + 0.5)).astype(np.int64)


def exact_list(real, n, w, h, band_top, seed):
    """A saddle list of exactly n saddles from a board's list `real`: the n nearest the board's median
    point in their original order, or all of them plus seeded decoys in the band of rows from band_top
    down, inserted at seeded positions.  Every round(theta) bin of the decoys stays below the board's
    most populated one, so the board search seeds on the board as with the real list."""
    if n <= len(real):
        c = np.median(real[:, :2], axis=0)
        d = ((real[:, :2] - c) ** 2).sum(axis=1)
        return real[np.sort(np.argsort(d, kind="stable")[:n])].copy()
    rng = np.random.default_rng(seed)
    k = n - len(real)
    hist = np.bincount(theta_bins(real[:, 3]) + 90, minlength=181)
    room = np.maximum(hist.max() - 1 - hist, 0)
    room[0] = room[180] = 0  # bins -90 and 90: half of them lies outside the saddles' angle range
    pool = np.repeat(np.arange(181) - 90, room)
    assert len(pool) >= k, (len(pool), k)
    theta = rng.choice(pool, k, replace=False) + rng.uniform(-0.45, 0.45, k)
    decoys = np.stack([rng.uniform(16.0, w - 16.0, k), rng.uniform(band_top + 16.0, h - 16.0, k),
                       np.full(k, np.median(real[:, 2])), theta, np.full(k, 45.0)], axis=1).astype(np.float32)
    at = np.sort(rng.integers(0, len(real) + 1, k))
    return np.insert(real, at, decoys, axis=0)


def exact_case(key, n, oracle):
    """(saddle list, oracle quads or None, oracle tags) of the list of n saddles on a canvas."""
    if (key, n) not in _LIST_CACHE:
        w, h, tname = CANVASES[key][:3]
        t, real = tile(tname, oracle)
        s = exact_list(real, n, w, h, t.shape[0], seed=n * 7919 + w)
        assert len(s) == n
        img = canvas(key, oracle)
        want_q = oracle.try_find_best_board(s)
        want_t = oracle.detect_from_saddles(img, s)
        if n >= 300:
            assert len(want_t) >= 10, (key, n, len(want_t))
        _LIST_CACHE[key, n] = s, want_q, want_t
    return _LIST_CACHE[key, n]


def batch_order(key):
    """Indices into the canvas's saddle counts, shuffled, with one list again at least two frames
    after its first place (a canvas of one list gets an empty list between the two)."""
    ns = CANVASES[key][3]
    rng = np.random.default_rng(len(key) * 131 + CANVASES[key][0])
    order = [int(i) for i in rng.permutation(len(ns))]
    if len(order) == 1:
        return order + [None] + order
    pos = int(rng.integers(2, len(order) + 1))  # order[0] again at index pos >= 2
    return order[:pos] + [order[0]] + order[pos:]


def tags_of(pkg, rec, n):
    return pkg._tags_to_dict(rec[:n])


def same_tags(got, want, what):
    assert sorted(got) == sorted(want), (what, sorted(got), sorted(want))
    for k in want:
        assert np.array_equal(got[k], want[k]), (what, k, got[k], want[k])


def check_frame(pkg, what, quads, rec, cnt, st, want_q, want_t):
    assert cnt >= 0, "no launch of the board kernel took %s (count %d)" % (what, cnt)
    assert st == 0, (what, st)
    if want_q is None:
        assert len(quads) == 0, what
    else:
        assert np.array_equal(quads, want_q), what
    same_tags(tags_of(pkg, rec, cnt), want_t, what)


@pytest.mark.parametrize("opts", list(OPTION_SETS), ids=str)
@pytest.mark.parametrize("key", list(CANVASES), ids=str)
def test_saddle_count_and_image_size_edges(pkg, oracle, key, opts):
    w, h, _, ns, max_saddles = CANVASES[key]
    img = canvas(key, oracle)
    order = batch_order(key)
    cases = [exact_case(key, ns[i], oracle) if i is not None else (np.zeros((0, 5), np.float32), None, {})
             for i in order]
    frames = np.broadcast_to(img, (len(order),) + img.shape)
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for k, v in OPTION_SETS[opts].items():
            det.set_option(k, v)
        if max_saddles:
            det.set_option("max_saddles", max_saddles)
        quads, rec, cnt, st = det._boards_from_saddle_batch([c[0] for c in cases], frames)
        alone = {}
        for f, (i, (s, want_q, want_t)) in enumerate(zip(order, cases)):
            what = "%s, frame %d of the batch: %d saddles" % (key, f, len(s))
            check_frame(pkg, what, quads[f], rec[f], cnt[f], st[f], want_q, want_t)
            if i not in alone:
                alone[i] = det._boards_from_saddle_batch([s], img[None])
            aq, arec, acnt, ast = alone[i]
            check_frame(pkg, what + " (alone)", aq[0], arec[0], acnt[0], ast[0], want_q, want_t)
            assert acnt[0] == cnt[f] and ast[0] == st[f] and np.array_equal(aq[0], quads[f]), what
            assert arec[0].tobytes() == rec[f].tobytes(), what
    finally:
        det.close()


# ---- boards wider than the tag lattice ----
STRIPS = [(6, 3), (8, 2), (10, 3), (12, 2), (14, 3), (16, 2), (18, 3), (20, 2)]  # (tags across, rows)
_STRIP_CACHE = {}


def strip_frames(oracle):
    """1280 x 1024 strips of 6 to 20 tags across, and a 3840 x 2160 board of 36 x 3 tags: (frame,
    saddle list, oracle quads, oracle tags) each."""
    if not _STRIP_CACHE:
        small = [synth.render_board_numpy(1280, 1024, cols=c, rows=r, seed=c, tag_px=60.0) for c, r in STRIPS]
        wide = [synth.render_board_numpy(3840, 2160, cols=36, rows=3, seed=1, tag_px=80.0, ss=2)]
        for name, imgs in (("small", small), ("wide", wide)):
            out = []
            for img in imgs:
                s = oracle.front_end(img, want_labels=False)["refined"]
                out.append((img, s, oracle.try_find_best_board(s), oracle.detect_from_saddles(img, s)))
            _STRIP_CACHE[name] = out
    return _STRIP_CACHE


@pytest.mark.parametrize("lattice,which", [(16, "small"), (32, "small"), (64, "wide")])
@pytest.mark.parametrize("opts", ["batch", "latency"])
def test_board_wider_than_the_lattice_is_flagged(pkg, oracle, lattice, which, opts):
    """A board that leaves the tag lattice is flagged AG_FRAME_BOARD_OVERFLOW (and the host entry
    points report AG_ERR_CAPACITY); every other frame equals the oracle."""
    items = strip_frames(oracle)[which]
    frames = np.stack([it[0] for it in items])
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("board_lattice", lattice)
        for k, v in OPTION_SETS[opts].items():
            det.set_option(k, v)
        quads, rec, cnt, st = det._boards_from_saddle_batch([it[1] for it in items], frames)
        flagged = exact = 0
        for f, (img, s, want_q, want_t) in enumerate(items):
            what = "%s frame %d, lattice %d" % (which, f, lattice)
            assert cnt[f] >= 0, what
            if st[f] == 0:
                check_frame(pkg, what, quads[f], rec[f], cnt[f], st[f], want_q, want_t)
                exact += 1
                continue
            assert st[f] == AG_FRAME_BOARD_OVERFLOW, (what, st[f])
            flagged += 1
            with pytest.raises(RuntimeError, match="error 4: .*limits"):
                det.detect(img)
            with pytest.raises(RuntimeError, match="error 4: .*limits"):
                det.detect_batch(img[None])
        if lattice == 16:
            assert flagged >= 1 and exact >= 1, (flagged, exact)
    finally:
        det.close()


# ---- real frames through the device pipeline ----
def test_frames_of_every_class_through_the_device_pipeline(pkg, oracle):
    """One detect_batch_device call on 1280 x 1024 frames in chunks of three, batch layouts and split
    launches: a 6 x 6 board (<= 320 saddles), a 12 x 9 board (512 < n <= 1024), a 14 x 2 strip, an
    empty frame and iid noise (more clusters than the automatic capacity).  The boards equal the
    oracle; the noise frame comes back flagged with no tags; every output slot is written.
    detect_batch re-runs the noise frame with grown capacities: all five equal the oracle."""
    import torch
    boards = [synth.render_board_numpy(1280, 1024, seed=3, tag_px=60.0),
              synth.render_board_numpy(1280, 1024, cols=12, rows=9, seed=4, tag_px=58.0),
              synth.render_board_numpy(1280, 1024, cols=14, rows=2, seed=4, tag_px=60.0)]
    n_ref = [len(oracle.front_end(b, want_labels=False)["refined"]) for b in boards]
    assert n_ref[0] <= 320 and 512 < n_ref[1] <= 1024, n_ref
    empty = np.full((1024, 1280), 128, np.uint8)
    noise = np.random.default_rng(77).integers(0, 256, (1024, 1280), dtype=np.uint8)
    kinds = ["6x6", "12x9", "14x2", "empty", "noise"]
    imgs = boards + [empty, noise]
    perm = [int(i) for i in np.random.default_rng(5).permutation(5)]
    frames = np.stack([imgs[i] for i in perm])
    want = [oracle.detect(imgs[i]) for i in perm]
    assert [len(want[perm.index(i)]) for i in range(5)][:3] == [36, 108, 28]
    n, cap = len(perm), 256
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("chunk_frames", 3)
        det.set_option("board_batch_frames", 1)
        d = torch.from_numpy(frames).cuda()
        out = torch.full((n, cap * 9), -1, dtype=torch.int32, device="cuda")
        cnt = torch.full((n,), -7, dtype=torch.int32, device="cuda")
        st = torch.full((n,), 0x5A5A5A5A, dtype=torch.int32, device="cuda")
        det.detect_batch_device(d.data_ptr(), n, 1280, 1024, pkg.FMT_L8, out.data_ptr(), cap, cnt.data_ptr(),
                                st.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        rec = out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, cap)
        c, s = cnt.cpu().numpy(), st.cpu().numpy().view(np.uint32)
        for f, i in enumerate(perm):
            what = "%s (frame %d)" % (kinds[i], f)
            if kinds[i] == "noise":
                assert s[f] & GROWABLE and c[f] == 0, (what, s[f], c[f])
                continue
            assert s[f] == 0 and c[f] >= 0, (what, s[f], c[f])
            same_tags(pkg._tags_to_dict(rec[f, :c[f]]), want[f], what)
        got, status = det.detect_batch(frames, cap_per_frame=cap, return_status=True)
        assert not status.any(), status
        for f, i in enumerate(perm):
            same_tags(got[f], want[f], kinds[i])
    finally:
        det.close()
