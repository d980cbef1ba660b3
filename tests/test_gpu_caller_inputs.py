"""Inputs a caller chooses through the C ABI, against the CPU oracle.  Needs a B200: -m gpu.

- DetectorParams: max_num_of_boards (the number of board-search rounds) on frames holding four
  boards whose tag ids overlap, and the saddle-angle gate (min / max_saddle_angle), down to the
  f32 value a saddle's phi sits on.
- Frame layouts: padded rows, gaps between frames, the smallest legal frame stride and unaligned
  base addresses, in L8, L16 and RGB8, through every entry point that takes strides.  The records
  must be byte-identical to the same frames packed.
- L16 frames at odd addresses / strides are refused by the device entry points; multi-GPU calls
  are synchronous whatever "host_async" says; cap_per_frame overflow on the device path."""
import ctypes as C

import numpy as np
import pytest

import synth
from test_gpu_parity import BOARD_VARIANTS, assert_saddles_match, assert_tags_match

pytestmark = pytest.mark.gpu

MAX_BOARDS = [0, 1, 2, 3, 4, 255]  # 255: the largest uint8_t, rounds past 127 (search cache off)
CAP = 64


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def same_tags(a, b):
    return sorted(a) == sorted(b) and all(np.array_equal(a[k], b[k]) for k in a)


def records_to_dicts(pkg, out, cnt):
    return [pkg._tags_to_dict(out[i, :cnt[i]]) for i in range(len(cnt))]


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


# ---- 1. several boards per frame, max_num_of_boards ----------------------------------------------
@pytest.fixture(scope="module")
def boards():
    """Six 1280 x 960 frames: the four-board composite (456 saddles) and the small-board one (<= 320
    saddles), each also turned by 180 degrees, a blank frame, and the first frame again."""
    big = synth.composite_boards(*synth.FOUR_BOARDS)
    small = synth.composite_boards(*synth.SMALL_BOARDS, canvas=big.shape)
    frames = np.stack([big, small, big[::-1, ::-1], small[::-1, ::-1], np.full_like(big, 200), big])
    return frames


@pytest.fixture(scope="module")
def board_want(oracle, boards):
    cache = {}

    def want(i, k):
        key = (0 if i == 5 else i, k)  # frame 5 is frame 0
        if key not in cache:
            cache[key] = oracle.detect(boards[key[0]], max_boards=k)
        return cache[key]
    return want


def test_composites_separate_the_rounds(oracle, boards, board_want):
    """Guard on the input: one, two and three rounds give three different answers, on both tiers."""
    for i in range(4):
        n_ref = len(oracle.front_end(boards[i], want_labels=False)["refined"])
        assert (n_ref <= 320) == (i % 2 == 1) and n_ref <= 512, (i, n_ref)
        r1, r2, r3 = board_want(i, 1), board_want(i, 2), board_want(i, 3)
        assert len(r1) > 0 and not same_tags(r1, r2) and not same_tags(r2, r3) and not same_tags(r1, r3), i
    assert board_want(0, 0) == {} and board_want(4, 255) == {}
    assert not same_tags(board_want(1, 3), board_want(1, 4))


@pytest.mark.parametrize("k", MAX_BOARDS)
def test_max_boards_detect_and_stage_taps(pkg, oracle, boards, board_want, k):
    det = pkg.TagDetector(pkg.TagFamily.T36H11, pkg.DetectorParams(max_num_of_boards=k))
    try:
        for i in (0, 1):
            img = boards[i]
            assert_tags_match(det.detect(img), board_want(i, k))
            g = det.stages(img, want_labels=False)
            o = oracle.front_end(img, want_labels=False)
            assert_saddles_match(g["refined"], o["refined"])
            if k == 0:
                assert len(g["quads"]) == 0
            else:
                oq = oracle.try_find_best_board(o["refined"])
                assert oq is not None and np.array_equal(g["quads"], oq), i
            assert_tags_match(g["tags"], board_want(i, k))
    finally:
        det.close()


@pytest.mark.parametrize("k", MAX_BOARDS)
def test_max_boards_every_board_variant(pkg, boards, board_want, k):
    for variant in BOARD_VARIANTS:
        det = pkg.TagDetector(pkg.TagFamily.T36H11, pkg.DetectorParams(max_num_of_boards=k))
        try:
            for key, v in variant.items():
                det.set_option(key, v)
            for i in (0, 1):
                assert_tags_match(det.detect(boards[i]), board_want(i, k))
        finally:
            det.close()


@pytest.mark.parametrize("k", MAX_BOARDS)
def test_max_boards_batch_device_and_multi(pkg, boards, board_want, torch_mod, k):
    """Batch mode (both tiers in split launches), the device entry point and a MultiTagDetector."""
    torch = torch_mod
    n, h, w = boards.shape
    params = pkg.DetectorParams(max_num_of_boards=k)
    want = [board_want(i, k) for i in range(n)]
    det = pkg.TagDetector(pkg.TagFamily.T36H11, params)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, params, devices=[0, 0])
    try:
        det.set_option("board_batch_frames", 1)
        got, status = det.detect_batch(boards, cap_per_frame=CAP, return_status=True)
        assert not status.any(), status
        for g, wt in zip(got, want):
            assert_tags_match(g, wt)
        d_frames = torch.from_numpy(boards).cuda()
        out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
        cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
        st = torch.zeros(n, dtype=torch.int32, device="cuda")
        det.detect_batch_device(d_frames.data_ptr(), n, w, h, pkg.FMT_L8, out.data_ptr(), CAP, cnt.data_ptr(),
                                st.data_ptr(), stream=torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert not st.cpu().numpy().any()
        rec = out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
        for g, wt in zip(records_to_dicts(pkg, rec, cnt.cpu().numpy()), want):
            assert_tags_match(g, wt)
        for g, wt in zip(multi.detect_batch(boards, cap_per_frame=CAP), want):
            assert_tags_match(g, wt)
    finally:
        multi.close()
        det.close()


# ---- 2. the saddle-angle gate ----------------------------------------------------------------------
ANGLES = [(20.0, 70.0), (35.0, 55.0), (40.0, 50.0), (45.0, 45.0), (0.0, 90.0), (60.0, 30.0)]


def check_stages_with_params(det, oracle, img, min_angle, max_angle, max_boards=2):
    """check_stages of test_gpu_parity for a detector created with non-default DetectorParams."""
    g = det.stages(img, want_labels=False)
    o = oracle.front_end(img, min_angle, max_angle, want_labels=False)
    assert np.array_equal(g["blur"].view(np.uint32), o["blur"].view(np.uint32)), "blur not bit-exact"
    assert np.array_equal(g["resp"].view(np.uint32), o["resp"].view(np.uint32)), "response not bit-exact"
    assert_saddles_match(g["raw"], o["raw"])
    assert_saddles_match(g["refined"], o["refined"])
    oq = oracle.try_find_best_board(o["refined"])
    if oq is None or max_boards == 0:
        assert len(g["quads"]) == 0
    else:
        assert np.array_equal(g["quads"], oq)
    assert_tags_match(g["tags"], oracle.detect(img, min_angle=min_angle, max_angle=max_angle, max_boards=max_boards))
    return g, o


@pytest.fixture(scope="module")
def angle_images(images):
    return {"EuRoC": images["EuRoC"], "synthetic": synth.render_board_numpy(640, 480, seed=5, tag_px=44.0)}


@pytest.mark.parametrize("angles", ANGLES, ids=lambda a: "%g-%g" % a)
def test_saddle_angle_gate_matches_oracle(pkg, oracle, angle_images, angles):
    lo, hi = angles
    det = pkg.TagDetector(pkg.TagFamily.T36H11, pkg.DetectorParams(min_saddle_angle=lo, max_saddle_angle=hi))
    try:
        for name, img in angle_images.items():
            g, o = check_stages_with_params(det, oracle, img, lo, hi)
            if lo > hi:
                assert len(o["refined"]) == 0 and g["tags"] == {}, name
            assert_saddles_match(det.refined_saddle_points(img), o["refined"])
            assert_tags_match(det.detect(img), oracle.detect(img, min_angle=lo, max_angle=hi))
    finally:
        det.close()


def _refined_with(pkg, img, lo, hi):
    det = pkg.TagDetector(pkg.TagFamily.T36H11, pkg.DetectorParams(min_saddle_angle=float(lo),
                                                                    max_saddle_angle=float(hi)))
    try:
        return det.refined_saddle_points(img)
    finally:
        det.close()


def _has(saddles, s):
    return bool(((saddles["x"].view(np.uint32) == np.float32(s[0]).view(np.uint32)) &
                 (saddles["y"].view(np.uint32) == np.float32(s[1]).view(np.uint32))).any())


def test_saddle_angle_gate_is_inclusive_to_the_ulp(pkg, oracle, angle_images):
    """min_saddle_angle = a saddle's exact f32 phi keeps the saddle, one ulp above drops it; the same
    for max_saddle_angle from below (phi >= min and phi <= max, detector.rs)."""
    img = angle_images["synthetic"]
    base = oracle.front_end(img, want_labels=False)["refined"]
    assert len(base) > 100
    s_lo = base[np.argmin(base[:, 4])]
    s_hi = base[np.argmax(base[:, 4])]
    phi_lo, phi_hi = np.float32(s_lo[4]), np.float32(s_hi[4])
    above = np.nextafter(phi_lo, np.float32(np.inf), dtype=np.float32)
    below = np.nextafter(phi_hi, np.float32(-np.inf), dtype=np.float32)
    for lo, hi, s, kept in ((phi_lo, 60.0, s_lo, True), (above, 60.0, s_lo, False),
                            (30.0, phi_hi, s_hi, True), (30.0, below, s_hi, False)):
        got = _refined_with(pkg, img, lo, hi)
        assert _has(got, s) == kept, (lo, hi, s, kept)
        assert_saddles_match(got, oracle.front_end(img, float(lo), float(hi), want_labels=False)["refined"])


# ---- 3. frame layouts through every entry point ------------------------------------------------------
FORMATS = ["l8", "l16", "rgb8"]


@pytest.fixture(scope="module")
def layout_frames():
    """{width: two board frames} at 640 (streaming K1 possible) and 642 (tile K1 only), L8."""
    return {w: [synth.render_board_numpy(w, 480, seed=s, tag_px=44.0) for s in (31, 32)] for w in (640, 642)}


def in_format(img8, fmt):
    if fmt == "l16":
        return img8.astype(np.uint16) * np.uint16(257)  # what render_board_numpy(dtype=np.uint16) gives
    if fmt == "rgb8":  # channels that differ: a swapped channel order changes the luma
        return np.stack([img8, img8, 255 - img8], axis=2)
    return img8


def layouts(fmt, w, h):
    """(name, row_stride, frame_stride, host base offset, device base offset)."""
    bpp = {"l8": 1, "l16": 2, "rgb8": 3}[fmt]
    rb = w * bpp
    pad = 2 if fmt == "l16" else 1  # the smallest legal row pad: rows no longer a multiple of the lane load
    wide = rb + 32  # a multiple of every lane load
    odd = 2 if fmt == "l16" else 1
    return [("rows_stream", wide, wide * h, 0, 0),
            ("rows_tile", rb + pad, (rb + pad) * h, 0, 0),
            ("frame_gap", wide, wide * h + 136, 0, 0),
            ("odd_frame_gap", rb, rb * h + odd, 0, 0),
            ("minimal_frame_stride", rb + pad, (rb + pad) * (h - 1) + rb, 0, 0),
            ("offset4", wide, wide * h, 4, 4),
            ("offset_odd", rb + pad, (rb + pad) * h, 1, odd)]


def lay_out(frames, rs, fs, offset, seed):
    """A byte buffer holding `frames` at buf[offset + i*fs + y*rs ...]; padding bytes are random."""
    n, h, w = frames.shape[:3]
    rb = frames[0, 0].nbytes
    size = offset + (n - 1) * fs + rs * (h - 1) + rb
    buf = np.random.default_rng(seed).integers(0, 256, size + 64, dtype=np.uint8)
    view = np.ndarray(frames.shape, frames.dtype, buffer=buf, offset=offset,
                      strides=(fs, rs) + frames.strides[2:])
    view[...] = frames
    return buf


TAG_DTYPE = np.dtype([("id", np.uint32), ("xy", np.float32, (8,))])  # ag_tag


def new_out(n):
    """(records, counts, status) arrays of a batch call."""
    return np.zeros((n, CAP), TAG_DTYPE), np.zeros(n, np.int32), np.zeros(n, np.uint32)


FMT_CODE = {"l8": 0, "l16": 1, "rgb8": 2}


@pytest.mark.parametrize("w", [640, 642])
@pytest.mark.parametrize("fmt", FORMATS)
def test_frame_layouts_through_every_entry_point(pkg, oracle, layout_frames, torch_mod, fmt, w):
    torch = torch_mod
    L = pkg.lib()
    h = 480
    a, b = (in_format(f, fmt) for f in layout_frames[w])
    frames = np.stack([a, np.zeros_like(a), b])  # chunks of two: [board, blank], [board]
    n, code = len(frames), FMT_CODE[fmt]
    rb = frames[0, 0].nbytes
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    grown = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    try:
        for d in (det, grown, multi):
            d.set_option("chunk_frames", 2)
        grown.set_option("max_clusters", 16)  # every board frame overflows: re-run from the caller's frames
        ref = new_out(n)
        det._check(L.ag_detect_batch(det._h, vp(frames), frames.strides[0], n, w, h, rb, code, vp(ref[0]), CAP,
                                     vp(ref[1]), vp(ref[2])))
        assert not ref[2].any() and ref[1][1] == 0 and ref[1][0] >= 30 and ref[1][2] >= 30
        for g, wt in zip(records_to_dicts(pkg, *ref[:2]), [oracle.detect(f) for f in frames]):
            assert_tags_match(g, wt)
        o0 = oracle.front_end(frames[0], want_labels=False)

        for name, rs, fs, off, doff in layouts(fmt, w, h):
            buf = lay_out(frames, rs, fs, off, seed=rs + fs)
            base = buf.ctypes.data + off
            case = (name, rs, fs, off)
            # ag_detect, frame by frame
            got = new_out(n)
            for i in range(n):
                cnt = C.c_int(0)
                det._check(L.ag_detect(det._h, base + i * fs, w, h, rs, code, got[0][i].ctypes.data, CAP, C.byref(cnt)))
                got[1][i] = cnt.value
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), ("detect",) + case
            # ag_detect_batch from pageable memory, and with capacities so small that every board frame
            # is re-run with grown ones from the strided source
            for d in (det, grown):
                got = new_out(n)
                d._check(L.ag_detect_batch(d._h, base, fs, n, w, h, rs, code, vp(got[0]), CAP, vp(got[1]), vp(got[2])))
                assert all(np.array_equal(x, y) for x, y in zip(got, ref)), ("batch",) + case
            # ... from page-locked memory
            pin = pkg.pinned_empty(buf.shape)
            try:
                pin[...] = buf
                got = new_out(n)
                det._check(L.ag_detect_batch(det._h, pin.ctypes.data + off, fs, n, w, h, rs, code, vp(got[0]), CAP,
                                             vp(got[1]), vp(got[2])))
                assert all(np.array_equal(x, y) for x, y in zip(got, ref)), ("pinned",) + case
            finally:
                pkg.pinned_free(pin)
            # ag_multi_detect_batch
            got = new_out(n)
            rc = L.ag_multi_detect_batch(multi._h, base, fs, n, w, h, rs, code, vp(got[0]), CAP, vp(got[1]), vp(got[2]))
            assert rc == pkg.AG_OK and all(np.array_equal(x, y) for x, y in zip(got, ref)), ("multi",) + case
            # ag_detect_batch_device on a strided view of a device byte buffer
            # (at an offset of its own: L16 frames must be 2-byte aligned on the device)
            dbuf = torch.from_numpy(buf if doff == off else lay_out(frames, rs, fs, doff, seed=rs + fs)).cuda()
            view = torch.as_strided(dbuf, (n, h, rb), (fs, rs, 1), storage_offset=doff)
            assert view.contiguous().cpu().numpy().tobytes() == frames.tobytes()
            d_out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
            d_cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
            d_st = torch.zeros(n, dtype=torch.int32, device="cuda")
            det.detect_batch_device(view.data_ptr(), n, w, h, code, d_out.data_ptr(), CAP, d_cnt.data_ptr(),
                                    d_st.data_ptr(), frame_stride=fs, row_stride=rs)
            torch.cuda.synchronize()
            rec = d_out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
            assert np.array_equal(rec, ref[0]) and np.array_equal(d_cnt.cpu().numpy(), ref[1]), ("device",) + case
            assert not d_st.cpu().numpy().any()
            # refined_saddle_points and the stage taps with a row stride (first frame)
            out = np.zeros(16384, pkg.SADDLE_DTYPE)
            cnt = C.c_int(0)
            det._check(L.ag_refined_saddle_points(det._h, base, w, h, rs, code, vp(out), 16384, C.byref(cnt)))
            assert_saddles_match(out[:cnt.value], o0["refined"])
            det._check(L.ag_stage_run(det._h, base, w, h, rs, code))
            blur, resp = np.empty((h, w), np.float32), np.empty((h, w), np.float32)
            det._check(L.ag_stage_blur(det._h, vp(blur)))
            det._check(L.ag_stage_response(det._h, vp(resp)))
            assert np.array_equal(blur.view(np.uint32), o0["blur"].view(np.uint32)), ("blur",) + case
            assert np.array_equal(resp.view(np.uint32), o0["resp"].view(np.uint32)), ("resp",) + case
    finally:
        multi.close()
        grown.close()
        det.close()


# ---- 4. L16 alignment and synchronous multi-GPU calls -----------------------------------------------
def test_l16_odd_frame_strides_and_device_addresses_are_refused(pkg, oracle, torch_mod):
    """2-byte pixels at odd addresses would be misaligned loads in the kernels: an odd L16 frame stride
    is refused by every entry point, an odd device address by the device ones, before anything is
    launched; odd HOST addresses are fine (frames are copied into aligned buffers)."""
    torch = torch_mod
    L = pkg.lib()
    w, h = 640, 480
    img = synth.render_board_numpy(w, h, seed=33, tag_px=44.0, dtype=np.uint16)
    want = oracle.detect(img)
    assert len(want) == 36
    rb = 2 * w
    buf = np.zeros(2 * (rb * h + 1) + 16, np.uint8)
    dbuf = torch.zeros(buf.size, dtype=torch.uint8, device="cuda")
    odd_ptr = dbuf.data_ptr() + 1
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    try:
        out = torch.zeros((2, CAP * 9), dtype=torch.int32, device="cuda")
        cnt = torch.full((2,), -7, dtype=torch.int32, device="cuda")
        fmt = pkg.FMT_L16

        def device_call(ptr, n, fs):
            return L.ag_detect_batch_device(det._h, ptr, fs, n, w, h, rb, fmt, out.data_ptr(), CAP, cnt.data_ptr(),
                                            None, None)

        def dense_call(ptr, n, fs):
            return L.ag_dense_batch_device(det._h, ptr, fs, n, w, h, rb, fmt, None)

        # Empty batches first: they launch nothing whatever the checks, so a library without them
        # fails here before any odd-address case can run.
        for call in (device_call, dense_call):
            assert call(odd_ptr, 0, 0) == pkg.AG_ERR_INVALID, call.__name__
            assert call(dbuf.data_ptr(), 0, rb * h + 1) == pkg.AG_ERR_INVALID, call.__name__
        for call in (device_call, dense_call):
            assert call(odd_ptr, 2, 0) == pkg.AG_ERR_INVALID
            assert call(odd_ptr + 2, 1, 0) == pkg.AG_ERR_INVALID
            assert call(dbuf.data_ptr(), 2, rb * h + 1) == pkg.AG_ERR_INVALID
        torch.cuda.synchronize()
        assert (cnt.cpu().numpy() == -7).all()
        # host entry points: an odd frame stride is refused, nothing is written
        h_out, h_cnt, h_st = new_out(2)
        h_cnt[:] = -7
        assert L.ag_detect_batch(det._h, vp(buf), rb * h + 1, 2, w, h, rb, fmt, vp(h_out), CAP, vp(h_cnt),
                                 vp(h_st)) == pkg.AG_ERR_INVALID
        assert L.ag_multi_detect_batch(multi._h, vp(buf), rb * h + 1, 2, w, h, rb, fmt, vp(h_out), CAP, vp(h_cnt),
                                       vp(h_st)) == pkg.AG_ERR_INVALID
        assert (h_cnt == -7).all() and not h_out["id"].any()
        # ... odd host addresses with even strides work
        for off in (1, 3):
            raw = lay_out(np.stack([img, img]), rb, rb * h + 2, off, seed=off)
            n1 = C.c_int(0)
            det._check(L.ag_detect(det._h, raw.ctypes.data + off, w, h, rb, fmt, vp(h_out[0]), CAP, C.byref(n1)))
            assert_tags_match(pkg._tags_to_dict(h_out[0, :n1.value]), want)
            got = new_out(2)
            det._check(L.ag_detect_batch(det._h, raw.ctypes.data + off, rb * h + 2, 2, w, h, rb, fmt, vp(got[0]), CAP,
                                         vp(got[1]), vp(got[2])))
            for g in records_to_dicts(pkg, *got[:2]):
                assert_tags_match(g, want)
            got = new_out(2)
            assert L.ag_multi_detect_batch(multi._h, raw.ctypes.data + off, rb * h + 2, 2, w, h, rb, fmt, vp(got[0]),
                                           CAP, vp(got[1]), vp(got[2])) == pkg.AG_OK
            for g in records_to_dicts(pkg, *got[:2]):
                assert_tags_match(g, want)
    finally:
        multi.close()
        det.close()


def test_multi_detect_batch_is_synchronous_on_streaming_handles(pkg, torch_mod):
    """ag_multi has no wait entry point: with host_async (and device_async) set on every device, each
    call still returns with its results in the caller's arrays, byte-identical to one device."""
    torch = torch_mod
    n, w, h = 12, 640, 480
    single = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    try:
        d_frames = torch.empty((2 * n, h, w), dtype=torch.uint8, device="cuda")
        single.render_boards_device(d_frames.data_ptr(), 2 * n, w, h, 6, 6, 515)
        torch.cuda.synchronize()
        batches = [np.ascontiguousarray(f) for f in np.split(d_frames.cpu().numpy(), 2)]
        refs = []
        for frames in batches:
            ref = new_out(n)
            single.detect_batch_into(frames, *ref)
            assert ref[1].sum() > 25 * n
            refs.append(ref)
        multi.set_option("host_async", 1)
        multi.set_option("device_async", 1)
        multi.set_option("host_chunk_frames", 2)
        for frames, ref in zip(batches, refs):
            got = new_out(n)
            multi.detect_batch_into(frames, *got)
            assert all(np.array_equal(x, y) for x, y in zip(got, ref))
    finally:
        multi.close()
        single.close()


# ---- 5. cap_per_frame overflow on the device path ------------------------------------------------------
@pytest.mark.parametrize("cap", [1, 5])
def test_device_tag_capacity_overflow(detector, pkg, torch_mod, cap):
    """Frames with more tags than cap_per_frame: AG_FRAME_TAG_OVERFLOW, the full count, the first cap
    records of the uncapped result, and not a byte written outside the output array."""
    torch = torch_mod
    n, w, h = 7, 640, 480
    frames = torch.zeros((n, h, w), dtype=torch.uint8, device="cuda")
    detector.render_boards_device(frames.data_ptr(), n - 1, w, h, 6, 6, 808)
    torch.cuda.synchronize()  # the last frame stays blank

    def run(c, guard):
        canary = 0x5A5A5A5A
        buf = torch.full((guard + n * c * 9 + guard,), canary, dtype=torch.int32, device="cuda")
        cnt = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        st = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        detector.detect_batch_device(frames.data_ptr(), n, w, h, pkg.FMT_L8, buf[guard:].data_ptr(), c,
                                     cnt.data_ptr(), st.data_ptr())
        torch.cuda.synchronize()
        b = buf.cpu().numpy()
        assert (b[:guard] == canary).all() and (b[guard + n * c * 9:] == canary).all()
        rec = b[guard:guard + n * c * 9].view(pkg.TAG_DTYPE).reshape(n, c)
        return rec, cnt.cpu().numpy(), st.cpu().numpy().view(np.uint32)

    full, full_cnt, full_st = run(64, 0)
    assert not full_st.any() and full_cnt[-1] == 0 and (full_cnt[:-1] > 5).sum() >= n - 2, full_cnt
    rec, cnt, st = run(cap, 4096)
    assert np.array_equal(cnt, full_cnt)
    for i in range(n):
        if full_cnt[i] > cap:
            assert st[i] == 8, (i, st[i])  # AG_FRAME_TAG_OVERFLOW
            assert rec[i].tobytes() == full[i, :cap].tobytes(), i
        else:
            assert st[i] == 0, (i, st[i])
            assert rec[i, :cnt[i]].tobytes() == full[i, :cnt[i]].tobytes(), i
