"""Refined saddle points of whole batches (ag_refined_saddle_points_batch, _device and
ag_multi_refined_saddle_points_batch) against the oracle.  Needs a B200: -m gpu.

Every list must equal the oracle's front_end(img)["refined"] (assert_saddles_match) and be
byte-identical to refined_saddle_points of the frame alone.  Covered: the fixture images and a
batch of rendered 1280 x 1024 boards with an empty frame; all ten pixel formats with padded rows and
gaps between frames; frames that overflow the cluster / saddle capacities (re-run on the host call,
flagged on the device call) and one beyond the hard limit; cap_per_frame below a frame's count
(exact count, the oracle's prefix, AG_FRAME_TAG_OVERFLOW, nothing written past the prefix); small
chunks that wrap the dense ring and all board slots with asynchronous saddle and detect calls
interleaved on two streams; empty and invalid calls; and several devices."""
import ctypes as C

import numpy as np
import pytest

import float_formats_ref as ffr
import formats_ref as fr
import synth
from conftest import FIXTURE_NAMES
from test_gpu_parity import assert_saddles_match

pytestmark = pytest.mark.gpu

CANARY = 0xDEADBEEF
GROWABLE = 1 | 2  # AG_FRAME_CLUSTER_OVERFLOW | AG_FRAME_SADDLE_OVERFLOW
TAG_OVERFLOW = 8
ALL_FORMATS = ("l8", "l16", "rgb8") + fr.NEW_FORMATS + ffr.FLOAT_FORMATS
CODE = dict(fr.CODE, **ffr.CODE)
BPP = dict(fr.BPP, **ffr.BPP)


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def geometry(pkg, frames):
    fmt, w, h, rs = pkg.image_format(frames[0])
    return fmt, w, h, rs, frames.strides[0]


def records(pkg, words, i, k):
    """The first k saddle records of frame i of an output array of N x (cap * 5) words."""
    return words[i, :5 * k].view(pkg.SADDLE_DTYPE)


def host_call(pkg, det, base, n, w, h, rs, fs, fmt, cap):
    """ag_refined_saddle_points_batch into canary-filled outputs: (rc, words, counts, status)."""
    m = max(n, 1)
    words = np.full((m, cap * 5), CANARY, np.uint32)
    cnt = np.full(m, -7, np.int32)
    st = np.full(m, CANARY, np.uint32)
    rc = pkg.lib().ag_refined_saddle_points_batch(det._h, base, fs, n, w, h, rs, fmt, vp(words), cap, vp(cnt), vp(st))
    return rc, words, cnt, st


def host_frames(pkg, det, frames, cap):
    fmt, w, h, rs, fs = geometry(pkg, frames)
    return host_call(pkg, det, vp(frames), len(frames), w, h, rs, fs, fmt, cap)


def device_call(pkg, det, torch, dptr, n, w, h, rs, fs, fmt, cap):
    """ag_refined_saddle_points_batch_device on the current stream, canary-filled outputs:
    (rc, words, counts, status) on the host."""
    m = max(n, 1)
    d_out = torch.full((m, cap * 5), CANARY - (1 << 32), dtype=torch.int32, device="cuda")
    d_cnt = torch.full((m,), -7, dtype=torch.int32, device="cuda")
    d_st = torch.full((m,), CANARY - (1 << 32), dtype=torch.int32, device="cuda")
    rc = pkg.lib().ag_refined_saddle_points_batch_device(
        det._h, C.c_void_p(dptr), fs, n, w, h, rs, fmt, C.c_void_p(d_out.data_ptr()), cap,
        C.c_void_p(d_cnt.data_ptr()), C.c_void_p(d_st.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return (rc, d_out.cpu().numpy().view(np.uint32), d_cnt.cpu().numpy(), d_st.cpu().numpy().view(np.uint32))


def device_frames(pkg, det, torch, frames, cap):
    fmt, w, h, rs, fs = geometry(pkg, frames)
    host = frames.view(np.int16) if frames.dtype == np.uint16 else frames  # torch has no uint16 copy
    d = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    return device_call(pkg, det, torch, d.data_ptr(), len(frames), w, h, rs, fs, fmt, cap)


def assert_untouched_past(words, cnt, cap):
    for i, c in enumerate(cnt):
        assert (words[i, 5 * min(max(int(c), 0), cap):] == CANARY).all(), ("written past the list", i)


def assert_exact(pkg, res, want, singles, cap):
    """res = (rc, words, cnt, st) of a batch call whose frames all fit: each list is the oracle's and the
    single-frame call's bytes, and nothing past it was written."""
    rc, words, cnt, st = res
    assert rc == pkg.AG_OK
    assert not st[:len(want)].any(), st
    for i, (o, one) in enumerate(zip(want, singles)):
        assert cnt[i] == len(o), (i, cnt[i], len(o))
        g = records(pkg, words, i, cnt[i])
        assert_saddles_match(g, o)
        assert g.tobytes() == one.tobytes(), i
    assert_untouched_past(words[:len(want)], cnt[:len(want)], cap)


def oracle_lists(oracle, frames):
    return [oracle.front_end(np.ascontiguousarray(f), want_labels=False)["refined"] for f in frames]


def single_lists(det, frames):
    return [det.refined_saddle_points(np.ascontiguousarray(f), cap=16384) for f in frames]


# ---- 1. fixtures and a batch of rendered boards --------------------------------------------------------------
def test_fixture_images(pkg, oracle, images, torch_mod):
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for name in FIXTURE_NAMES:
            img = images[name][None]
            want, one = oracle_lists(oracle, img), single_lists(det, img)
            h = host_frames(pkg, det, img, 16384)
            d = device_frames(pkg, det, torch_mod, img, 16384)
            assert_exact(pkg, h, want, one, 16384)
            assert_exact(pkg, d, want, one, 16384)
    finally:
        det.close()


@pytest.fixture(scope="module")
def boards_1280(oracle):
    # six seeds in four orientations each (rendering is slow on the host), cycled to 63 frames, and a
    # constant frame without saddles
    seeds = synth.fixture_like_frames(6, 1280, 1024, seed=700)
    distinct = [f[::a, ::b] for f in seeds for a in (1, -1) for b in (1, -1)]
    frames = np.stack([distinct[(5 * i) % len(distinct)] for i in range(63)])
    frames = np.concatenate([frames[:40], np.full((1, 1024, 1280), 117, np.uint8), frames[40:]])
    want = oracle_lists(oracle, frames)
    assert len(want[40]) == 0 and all(len(w) > 0 for i, w in enumerate(want) if i != 40)
    return frames, want


def test_rendered_batch_host_and_device(pkg, boards_1280, torch_mod):
    frames, want = boards_1280
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        one = single_lists(det, frames)
        h = host_frames(pkg, det, frames, 2048)
        d = device_frames(pkg, det, torch_mod, frames, 2048)
        assert_exact(pkg, h, want, one, 2048)
        assert_exact(pkg, d, want, one, 2048)
        assert np.array_equal(h[1], d[1]) and np.array_equal(h[2], d[2])
        # chunks of 9 frames through the host call's fill / drain schedule, from pinned memory
        det.set_option("host_chunk_frames", 9)
        pin = pkg.pinned_empty(frames.shape, np.uint8)
        try:
            pin[...] = frames
            assert_exact(pkg, host_frames(pkg, det, pin, 2048), want, one, 2048)
        finally:
            pkg.pinned_free(pin)
        # the Python wrapper
        got, status = det.refined_saddle_points_batch(frames, return_status=True)
        assert not status.any() and all(g.tobytes() == o.tobytes() for g, o in zip(got, one))
    finally:
        det.close()


# ---- 2. every pixel format, padded rows and gaps between frames ---------------------------------------------
def format_frame(board, fmt, seed, noise=True):
    """board in format fmt; noise=False gives R = G = B and 16-bit words of gray * 257 (a constant
    frame stays constant, without saddles)."""
    if fmt == "l8":
        return board
    if fmt == "l16":
        return np.ascontiguousarray(fr_to_format(board, "la16", seed, noise)[:, :, 0])
    if fmt in ffr.FLOAT_FORMATS:
        return ffr.widen(board, fmt, seed=seed, noise=0.03 if noise else 0.0)
    return fr_to_format(board, fmt, seed, noise)


def fr_to_format(l8, fmt, seed, noise):
    from test_gpu_formats import to_format
    return to_format(l8, fmt, seed=seed, noise=noise)


@pytest.fixture(scope="module")
def board_640():
    return synth.render_board_numpy(640, 480, seed=43, tag_px=44.0)


@pytest.mark.parametrize("fmt", ALL_FORMATS)
def test_every_format_padded(pkg, oracle, torch_mod, board_640, fmt):
    torch = torch_mod
    ref = ffr.FloatOracle(oracle) if fmt in ffr.FLOAT_FORMATS else fr.RefOracle(oracle)
    board = board_640
    frames = np.stack([format_frame(board, fmt, 1), format_frame(board[::-1, ::-1].copy(), fmt, 2),
                       format_frame(np.full_like(board, 117), fmt, 3, noise=False)])
    n, h, w = frames.shape[:3]
    want = [ref.front_end(f, want_labels=False)["refined"] for f in frames]
    assert len(want[0]) > 100 and len(want[2]) == 0
    rb = w * BPP[fmt]
    rs, fs = rb + 32, (rb + 32) * h + 64
    buf = np.zeros(fs * n + 64, np.uint8)
    view = np.ndarray(frames.shape, frames.dtype, buffer=buf, strides=(fs, rs) + frames.strides[2:])
    view[...] = frames
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("chunk_frames", 2)
        one = single_lists(det, frames)
        hres = host_call(pkg, det, vp(buf), n, w, h, rs, fs, CODE[fmt], 2048)
        assert_exact(pkg, hres, want, one, 2048)
        dbuf = torch.from_numpy(buf).cuda()
        dres = device_call(pkg, det, torch, dbuf.data_ptr(), n, w, h, rs, fs, CODE[fmt], 2048)
        assert_exact(pkg, dres, want, one, 2048)
    finally:
        det.close()


# ---- 3. capacity overflow ---------------------------------------------------------------------------------
def test_overflowing_frames(pkg, oracle, torch_mod):
    rng = np.random.default_rng(5)
    H, W = 1024, 1280
    noise = rng.integers(0, 256, (H, W), dtype=np.uint8)
    yy, xx = np.mgrid[0:H, 0:W]
    checker = np.where(((yy // 12) + (xx // 12)) % 2 == 0, 40, 200).astype(np.uint8)
    board = synth.render_board_numpy(W, H, seed=5)
    frames = np.stack([board, noise, board[::-1].copy(), checker, noise[::-1].copy()])
    want = oracle_lists(oracle, frames)
    assert len(want[1]) > 8000 and len(want[3]) > 4000
    cap = 16384
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        one = single_lists(det, frames)
        assert_exact(pkg, host_frames(pkg, det, frames, cap), want, one, cap)
        rc, words, cnt, st = device_frames(pkg, det, torch_mod, frames, cap)
        assert rc == pkg.AG_OK
        for i, o in enumerate(want):
            if i in (1, 3, 4):  # overflowed at the automatic capacities: flagged, no list
                assert cnt[i] == 0 and st[i] & GROWABLE and not int(st[i]) & ~GROWABLE, (i, st[i])
            else:
                assert st[i] == 0 and cnt[i] == len(o)
                assert records(pkg, words, i, cnt[i]).tobytes() == one[i].tobytes()
        assert_untouched_past(words, cnt, cap)
        # beyond the hard limit of 16384 saddles: the frame keeps its bits, the call fails, the rest is exact
        dense = np.where(((yy // 5) + (xx // 5)) % 2 == 0, 40, 200).astype(np.uint8)
        if len(oracle.front_end(dense, want_labels=False)["refined"]) > 16384:
            mixed = np.stack([board, dense, checker])
            rc, words, cnt, st = host_frames(pkg, det, mixed, cap)
            assert rc == pkg.AG_ERR_CAPACITY
            assert st[1] & GROWABLE and st[0] == 0 and st[2] == 0
            for i in (0, 2):
                assert cnt[i] == len(want[3 * (i // 2)])
                assert_saddles_match(records(pkg, words, i, cnt[i]), want[3 * (i // 2)])
            with pytest.raises(RuntimeError, match="limits"):
                det.refined_saddle_points_batch(mixed, cap_per_frame=cap)
    finally:
        det.close()


# ---- 4. cap_per_frame below a frame's count -------------------------------------------------------------------
def test_cap_below_count(pkg, oracle, torch_mod, board_640):
    board = board_640
    frames = np.stack([board, np.zeros_like(board), board[:, ::-1].copy()])
    want = oracle_lists(oracle, frames)
    cap = 50
    assert len(want[0]) > cap and len(want[2]) > cap and len(want[1]) == 0
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for call in (host_frames, lambda p, d, f, c: device_frames(p, d, torch_mod, f, c)):
            rc, words, cnt, st = call(pkg, det, frames, cap)
            assert rc == (pkg.AG_ERR_CAPACITY if call is host_frames else pkg.AG_OK)
            for i, o in enumerate(want):
                assert cnt[i] == len(o)
                assert st[i] == (TAG_OVERFLOW if len(o) > cap else 0)
                k = min(len(o), cap)
                assert_saddles_match(records(pkg, words, i, k), o[:k])
            assert_untouched_past(words, cnt, cap)
        with pytest.raises(RuntimeError, match="cap_per_frame"):
            det.refined_saddle_points_batch(frames, cap_per_frame=cap)
    finally:
        det.close()


# ---- 5. pipeline wrap: asynchronous calls on two streams, interleaved with detect calls ---------------------
def test_interleaved_async_calls_wrap_the_pipeline(pkg, torch_mod):
    torch = torch_mod
    W, H, CAP_S, CAP_T = 640, 480, 4096, 64  # (the noise frame has a few thousand saddles)
    rng = np.random.default_rng(3)
    distinct = [synth.render_board_numpy(W, H, seed=s, tag_px=44.0) for s in (51, 52, 53)]
    distinct.append(rng.integers(0, 256, (H, W), dtype=np.uint8))  # overflows max_clusters below
    distinct.append(np.full((H, W), 90, np.uint8))
    order = [(3 * i) % len(distinct) for i in range(61)]
    frames = np.stack([distinct[k] for k in order])
    n = len(frames)
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    det.set_option("chunk_frames", 7)
    det.set_option("max_clusters", 8192)
    try:
        # synchronous single-call results of both kinds
        ref_s = host_frames(pkg, det, frames, CAP_S)
        assert ref_s[0] == pkg.AG_OK
        ref_t_rec = np.zeros((n, CAP_T), pkg.TAG_DTYPE)
        ref_t_cnt = np.zeros(n, np.int32)
        det.detect_batch_into(frames, ref_t_rec, ref_t_cnt)
        d_frames = torch.from_numpy(frames).cuda()
        sync_dev = device_frames(pkg, det, torch, frames, CAP_S)
        flagged = [i for i in range(n) if sync_dev[3][i] & GROWABLE]
        assert flagged == [i for i in range(n) if order[i] == 3]  # the noise frames

        det.set_option("device_async", 1)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        # every call's outputs are allocated up front: buffers of calls in flight are never reused
        bufs = {"s": [(torch.full((n, CAP_S * 5), 1, dtype=torch.int32, device="cuda"),
                       torch.zeros(n, dtype=torch.int32, device="cuda"),
                       torch.zeros(n, dtype=torch.int32, device="cuda")) for _ in range(4)],
                "t": [(torch.zeros((n, CAP_T * 9), dtype=torch.int32, device="cuda"),
                       torch.zeros(n, dtype=torch.int32, device="cuda"),
                       torch.zeros(n, dtype=torch.int32, device="cuda")) for _ in range(2)]}
        torch.cuda.synchronize()
        outs = []

        def saddles_on(stream):
            o = bufs["s"].pop()
            det.refined_saddle_points_batch_device(d_frames.data_ptr(), n, W, H, pkg.FMT_L8, o[0].data_ptr(), CAP_S,
                                                   o[1].data_ptr(), o[2].data_ptr(), stream=stream.cuda_stream)
            outs.append(("s", o))

        def tags_on(stream):
            o = bufs["t"].pop()
            det.detect_batch_device(d_frames.data_ptr(), n, W, H, pkg.FMT_L8, o[0].data_ptr(), CAP_T,
                                    o[1].data_ptr(), o[2].data_ptr(), stream=stream.cuda_stream)
            outs.append(("t", o))

        pin = pkg.pinned_empty(frames.shape, np.uint8)
        host_out = [(np.zeros((n, CAP_T), pkg.TAG_DTYPE), np.zeros(n, np.int32)) for _ in range(2)]
        try:
            pin[...] = frames
            saddles_on(s1)
            tags_on(s2)
            saddles_on(s2)
            det.set_option("host_async", 1)
            det.detect_batch_into(pin, *host_out[0])
            saddles_on(s1)  # collects the streaming host chunks first
            det.detect_batch_into(pin, *host_out[1])
            tags_on(s1)
            saddles_on(s2)
            det.detect_batch_wait(0)
            det.set_option("host_async", 0)
            det.detect_batch_device_wait(None)
            torch.cuda.synchronize()
            for rec, cnt in host_out:
                assert np.array_equal(cnt, ref_t_cnt) and rec.tobytes() == ref_t_rec.tobytes()
        finally:
            pkg.pinned_free(pin)
        for kind, (o, c, st) in outs:
            c, st = c.cpu().numpy(), st.cpu().numpy().view(np.uint32)
            if kind == "s":
                words = o.cpu().numpy().view(np.uint32)
                assert np.array_equal(c, sync_dev[2]) and np.array_equal(st, sync_dev[3])
                for i in range(n):
                    assert np.array_equal(words[i, :5 * c[i]], sync_dev[1][i, :5 * c[i]]), i
                    if i not in flagged:
                        assert np.array_equal(words[i, :5 * c[i]], ref_s[1][i, :5 * c[i]]), i
            else:
                rec = o.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP_T)
                for i in range(n):
                    if i in flagged:
                        assert c[i] == 0 and st[i] & GROWABLE
                    else:
                        assert c[i] == ref_t_cnt[i] and rec[i, :c[i]].tobytes() == ref_t_rec[i, :c[i]].tobytes(), i
    finally:
        det.close()


# ---- 6. empty and invalid calls -------------------------------------------------------------------------
def test_empty_and_invalid_calls(pkg, torch_mod):
    torch = torch_mod
    L = pkg.lib()
    W, H = 64, 48
    frames = np.zeros((2, H, W), np.uint16)
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    d = torch.zeros(2 * H * W + 8, dtype=torch.int16, device="cuda")
    fs, rs = H * W * 2, W * 2
    try:
        out = np.full((2, 16 * 5), CANARY, np.uint32)
        cnt = np.full(2, -7, np.int32)
        st = np.full(2, CANARY, np.uint32)
        ok = (vp(frames), fs, 2, W, H, rs, pkg.FMT_L16, vp(out), 16, vp(cnt), vp(st))
        cases = {
            "empty": dict(n=0), "null frames": dict(frames=None), "null out": dict(out=None),
            "null counts": dict(cnt=None), "cap 0": dict(cap=0), "negative n": dict(n=-1),
            "short rows": dict(rs=2 * W - 2), "short frames": dict(fs=rs * (H - 1)), "odd rows": dict(rs=2 * W + 1),
            "odd frames": dict(fs=fs + 1), "bad format": dict(fmt=3),
        }
        names = ("frames", "fs", "n", "w", "h", "rs", "fmt", "out", "cap", "cnt", "st")
        for name, change in cases.items():
            args = list(ok)
            for k, v in change.items():
                args[names.index(k)] = v
            want = pkg.AG_OK if name == "empty" else pkg.AG_ERR_INVALID
            assert L.ag_refined_saddle_points_batch(det._h, *args) == want, name
            assert L.ag_multi_refined_saddle_points_batch(multi._h, *args) == want, name
            dargs = list(args)  # (host output arrays stand in for device ones: nothing may run)
            if dargs[0] is not None:
                dargs[0] = C.c_void_p(d.data_ptr())
            assert L.ag_refined_saddle_points_batch_device(det._h, *dargs, None) == want, name
            assert (out == CANARY).all() and (cnt == -7).all() and (st == CANARY).all(), name
        # a 16-bit frame at an odd device address
        args = list(ok)
        args[0] = C.c_void_p(d.data_ptr() + 1)
        assert L.ag_refined_saddle_points_batch_device(det._h, *args, None) == pkg.AG_ERR_INVALID
        assert (out == CANARY).all() and (cnt == -7).all()
        # no handle
        assert L.ag_refined_saddle_points_batch(None, *ok) == pkg.AG_ERR_INVALID
        assert L.ag_refined_saddle_points_batch_device(None, *ok, None) == pkg.AG_ERR_INVALID
        assert L.ag_multi_refined_saddle_points_batch(None, *ok) == pkg.AG_ERR_INVALID
        assert det.refined_saddle_points_batch(frames[:0]) == []
        torch.cuda.synchronize()
    finally:
        multi.close()
        det.close()


# ---- 7. several devices -----------------------------------------------------------------------------------
def test_multi_device_equals_one_device(pkg, torch_mod):
    board = [synth.render_board_numpy(640, 480, seed=s, tag_px=44.0) for s in (61, 62, 63)]
    frames = np.stack([board[i % 3] if i % 4 else board[i % 3][::-1] for i in range(11)])
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        one = det.refined_saddle_points_batch(frames)
    finally:
        det.close()
    setups = [[0, 0]]
    if torch_mod.cuda.device_count() >= 2:
        setups.append(None)
    for devices in setups:
        multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=devices)
        try:
            for batch in (frames, frames[:7]):  # 11 and 7 frames: shards of unequal size
                got = multi.refined_saddle_points_batch(batch)
                assert len(got) == len(batch)
                assert all(g.tobytes() == o.tobytes() for g, o in zip(got, one)), devices
        finally:
            multi.close()
    if torch_mod.cuda.device_count() < 2:
        pytest.skip("one GPU: sharding checked over two handles on device 0 only")
