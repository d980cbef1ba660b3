"""The pixel formats RGB32F and RGBA32F on the GPU.  Needs a B200: -m gpu.

- The device's gray conversion (ag_test_float_luma) equals the restatement of float_formats_ref bit for
  bit on the pixel sets of test_float_formats_host.
- Parity with the oracle on the restated planes (float_formats_ref.FloatOracle): rendered boards widened
  with colour noise and a frame with channels over [-0.5, 3], bit-exact through every stage and with
  equal tags through every entry point that takes a frame.
- Equivalence: a frame widened from L8 (R = G = B = f32(k / 255)) is the L8 frame in every tap and entry point.
- Both K1 kernels with padded rows, gaps between frames, a base offset of 4 and dense_variant 1.
- The painted decode-gate frames of float_formats_ref.gate_frames.
- Strides and device addresses that are not multiples of 4 are refused before anything runs."""
import ctypes as C

import numpy as np
import pytest

import float_formats_ref as ffr
import synth
from test_float_formats_host import assert_same_planes, pixel_sets
from test_gpu_formats import assert_same_results, lay_out, same_tags, vp
from test_gpu_parity import assert_saddles_match, check_stages

pytestmark = pytest.mark.gpu

FORMATS = list(ffr.FLOAT_FORMATS)
CODE, BPP = ffr.CODE, ffr.BPP
CAP = 128


@pytest.fixture(scope="module")
def ref(oracle):
    return ffr.FloatOracle(oracle)


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def device_batch(pkg, det, torch, frames, code, fs=0, rs=0, async_=False):
    n, h, w = frames.shape[:3]
    d = torch.from_numpy(np.ascontiguousarray(frames)).cuda()
    out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    det.set_option("device_async", 1 if async_ else 0)
    try:
        det.detect_batch_device(d.data_ptr(), n, w, h, code, out.data_ptr(), CAP, cnt.data_ptr(), st.data_ptr(),
                                stream=s, frame_stride=fs, row_stride=rs)
        if async_:
            det.detect_batch_device_wait(stream=s)
        torch.cuda.synchronize()
    finally:
        det.set_option("device_async", 0)
    rec = out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
    c = cnt.cpu().numpy()
    assert not st.cpu().numpy().any()
    return [pkg._tags_to_dict(rec[i, :c[i]]) for i in range(n)]


# ---- the conversion itself ---------------------------------------------------------------------------
def test_device_conversion_equals_restatement(detector):
    n = 0
    for name, px in pixel_sets().items():
        for c in (3, 4):
            p = np.ascontiguousarray(px[:, :c]) if px.shape[1] >= c else np.concatenate(
                [px, np.full((len(px), 1), 0.5, np.float32)], axis=1)
            assert_same_planes(detector._float_luma(p), ffr.planes(p), (name, c))
            n += len(p)
    assert n >= 10_000_000


# ---- parity with the oracle, every entry point -----------------------------------------------------
def frames_for(fmt):
    board = synth.render_board_numpy(640, 480, seed=41, tag_px=44.0)
    return [ffr.widen(board, fmt, seed=1, noise=0.03), ffr.widen(board, fmt, seed=2, noise=0.05, lo=-0.5, hi=3.0)]


@pytest.mark.parametrize("fmt", FORMATS)
def test_parity_every_entry_point(pkg, ref, torch_mod, fmt):
    torch = torch_mod
    board, spread = frames_for(fmt)
    want = ref.detect(board)
    assert len(want) == 36
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    try:
        for img in (board, spread):
            check_stages(det, ref, img)  # ag_stage_run: every stage bit-exact, equal tags
            same_tags(det.detect(img), ref.detect(img))
            same_tags(det.detect_planes(*ffr.planes(img)), ref.detect(img))
            assert_saddles_match(det.refined_saddle_points(img), ref.front_end(img, want_labels=False)["refined"])
        o = ref.front_end(board, want_labels=False)["refined"]
        quads, tags = det._boards_from_saddles(o, board)
        assert np.array_equal(quads, ref.try_find_best_board(o))
        same_tags(tags, want)
        batch = np.stack([board, np.zeros_like(board), spread, board[::-1, ::-1].copy()])
        wants = [ref.detect(f) for f in batch]
        for got in (det.detect_batch(batch, cap_per_frame=CAP), multi.detect_batch(batch, cap_per_frame=CAP),
                    device_batch(pkg, det, torch, batch, CODE[fmt]),
                    device_batch(pkg, det, torch, batch, CODE[fmt], async_=True)):
            for g, wt in zip(got, wants):
                same_tags(g, wt)
        pin = pkg.pinned_empty(batch.shape, batch.dtype)
        try:
            pin[...] = batch
            for async_ in (0, 1):
                det.set_option("host_async", async_)
                out = np.zeros((len(batch), CAP), pkg.TAG_DTYPE)
                cnt = np.zeros(len(batch), np.int32)
                det.detect_batch_into(pin, out, cnt)
                if async_:
                    det.detect_batch_wait()
                for i, wt in enumerate(wants):
                    same_tags(pkg._tags_to_dict(out[i, :cnt[i]]), wt)
            det.set_option("host_async", 0)
        finally:
            pkg.pinned_free(pin)
        d = torch.from_numpy(batch).cuda()
        n0 = det.launch_count
        det.dense_batch_device(d.data_ptr(), len(batch), batch.shape[2], batch.shape[1], CODE[fmt])
        torch.cuda.synchronize()
        assert det.launch_count > n0
    finally:
        multi.close()
        det.close()


# ---- equivalence with L8 ---------------------------------------------------------------------------
def results(pkg, det, torch, img, code):
    """Every tap of ag_stage_run, then ag_detect_batch and ag_detect_batch_device on [img, img flipped]."""
    g = det.stages(img)
    batch = np.stack([img, img[::-1, ::-1].copy()])
    out = np.zeros((2, CAP), pkg.TAG_DTYPE)
    cnt, st = np.zeros(2, np.int32), np.zeros(2, np.uint32)
    w, h = img.shape[1], img.shape[0]
    det._check(pkg.lib().ag_detect_batch(det._h, vp(batch), batch.strides[0], 2, w, h, batch.strides[1], code,
                                         vp(out), CAP, vp(cnt), vp(st)))
    return g, out.tobytes(), cnt.tobytes(), device_batch(pkg, det, torch, batch, code)


@pytest.mark.parametrize("fmt", FORMATS)
def test_widened_l8_frames_equal_l8(pkg, torch_mod, fmt):
    torch = torch_mod
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for l8 in (synth.render_board_numpy(640, 480, seed=43, tag_px=44.0),
                   np.random.default_rng(5).integers(0, 256, (96, 128)).astype(np.uint8)):
            want = results(pkg, det, torch, l8, pkg.FMT_L8)
            assert_same_results(results(pkg, det, torch, ffr.widen(l8, fmt, seed=7), CODE[fmt]), want, fmt)
            img = ffr.widen(l8, fmt, seed=8)
            same_tags(det.detect(img), det.detect(l8))
            assert det.refined_saddle_points(img).tobytes() == det.refined_saddle_points(l8).tobytes()
    finally:
        det.close()


# ---- both K1 kernels: strided frames ---------------------------------------------------------------
def layouts(fmt, w, h):
    """(name, row_stride, frame_stride, base offset, dense_variant): rows at 0 (mod 16) take the streaming
    K1, rows at 4 (mod 16) the tile K1; a gap between frames; a base offset of 4; the tile K1 forced."""
    rb = w * BPP[fmt]
    r16 = (rb + 15) // 16 * 16
    return [("rows_stream", r16 + 32, (r16 + 32) * h, 0, 0), ("rows_tile", r16 + 4, (r16 + 4) * h, 0, 0),
            ("frame_gap", r16 + 32, (r16 + 32) * h + 20, 0, 0), ("offset", r16 + 32, (r16 + 32) * h, 4, 0),
            ("variant_1", r16 + 32, (r16 + 32) * h, 0, 1)]


@pytest.mark.parametrize("w", [640, 642])
@pytest.mark.parametrize("fmt", FORMATS)
def test_frame_layouts(pkg, ref, torch_mod, fmt, w):
    torch, oracle_ref = torch_mod, ref
    L = pkg.lib()
    h = 480
    board = ffr.widen(synth.render_board_numpy(w, h, seed=31, tag_px=44.0), fmt, seed=3, noise=0.03)
    frames = np.stack([board, np.zeros_like(board), board[::-1, ::-1].copy()])
    n, code, rb = len(frames), CODE[fmt], frames[0, 0].nbytes
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("chunk_frames", 2)
        want = (np.zeros((n, CAP), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.zeros(n, np.uint32))
        det._check(L.ag_detect_batch(det._h, vp(frames), frames.strides[0], n, w, h, rb, code, vp(want[0]), CAP,
                                     vp(want[1]), vp(want[2])))
        assert not want[2].any() and want[1][0] >= 30 and want[1][1] == 0 and want[1][2] >= 30
        same_tags(pkg._tags_to_dict(want[0][0, :want[1][0]]), oracle_ref.detect(board))
        o0 = oracle_ref.front_end(board, want_labels=False)
        for name, rs, fs, off, variant in layouts(fmt, w, h):
            case = (fmt, w, name)
            det.set_option("dense_variant", variant)
            buf = lay_out(frames, rs, fs, off, seed=rs + fs)
            base = buf.ctypes.data + off
            got = (np.zeros((n, CAP), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.zeros(n, np.uint32))
            det._check(L.ag_detect_batch(det._h, base, fs, n, w, h, rs, code, vp(got[0]), CAP, vp(got[1]), vp(got[2])))
            assert all(np.array_equal(x, y) for x, y in zip(got, want)), ("batch",) + case
            cnt = C.c_int(0)
            one = np.zeros(CAP, pkg.TAG_DTYPE)
            det._check(L.ag_detect(det._h, base, w, h, rs, code, vp(one), CAP, C.byref(cnt)))
            assert cnt.value == want[1][0] and np.array_equal(one[:cnt.value], want[0][0, :cnt.value]), ("detect",) + case
            dbuf = torch.from_numpy(buf).cuda()
            view = torch.as_strided(dbuf, (n, h, rb), (fs, rs, 1), storage_offset=off)
            d_out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
            d_cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
            det.detect_batch_device(view.data_ptr(), n, w, h, code, d_out.data_ptr(), CAP, d_cnt.data_ptr(),
                                    None, frame_stride=fs, row_stride=rs)
            torch.cuda.synchronize()
            rec = d_out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
            assert rec.tobytes() == want[0].tobytes() and np.array_equal(d_cnt.cpu().numpy(), want[1]), ("device",) + case
            det._check(L.ag_stage_run(det._h, base, w, h, rs, code))
            blur, resp = np.empty((h, w), np.float32), np.empty((h, w), np.float32)
            det._check(L.ag_stage_blur(det._h, vp(blur)))
            det._check(L.ag_stage_response(det._h, vp(resp)))
            assert np.array_equal(blur.view(np.uint32), o0["blur"].view(np.uint32)), ("blur",) + case
            assert np.array_equal(resp.view(np.uint32), o0["resp"].view(np.uint32)), ("resp",) + case
        det.set_option("dense_variant", 0)
    finally:
        det.close()


# ---- decode gates ----------------------------------------------------------------------------------
@pytest.mark.parametrize("family", list(synth.GATE_FAMILIES))
def test_painted_frames(pkg, oracle, ref, torch_mod, family):
    torch = torch_mod
    tf = pkg.TagFamily[family.upper()]
    det = pkg.TagDetector(tf)
    try:
        det.set_option("chunk_frames", 3)
        batches = {}
        for name, scene, tags, fmt, frame, mbs in ffr.gate_frames(oracle, family):
            if 2 not in mbs:
                continue
            want = ref.detect(frame, family=family)
            same_tags(det.detect(frame), want)
            g = det.stages(frame, want_labels=False)
            o = ref.front_end(frame, want_labels=False)
            assert np.array_equal(g["blur"].view(np.uint32), o["blur"].view(np.uint32)), (name, fmt)
            assert_saddles_match(g["refined"], o["refined"])
            assert np.array_equal(g["quads"], ref.try_find_best_board(o["refined"])), (name, fmt)
            same_tags(g["tags"], want)
            batches.setdefault((fmt, frame.shape), []).append((frame, want))
        for (fmt, _), items in batches.items():
            frames = np.stack([f for f, _ in items] * 2)
            wants = [w for _, w in items] * 2
            for g, wt in zip(det.detect_batch(frames, cap_per_frame=CAP), wants):
                same_tags(g, wt)
            for g, wt in zip(device_batch(pkg, det, torch, frames, CODE[fmt]), wants):
                same_tags(g, wt)
    finally:
        det.close()


# ---- refusals --------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", FORMATS)
def test_misaligned_strides_and_addresses_are_refused(pkg, torch_mod, fmt):
    torch = torch_mod
    L = pkg.lib()
    w, h = 64, 48
    rb = w * BPP[fmt]
    code = CODE[fmt]
    buf = np.zeros(2 * (rb + 2) * h + 64, np.uint8)
    dbuf = torch.zeros(buf.size, dtype=torch.uint8, device="cuda")
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    try:
        out, cnt, st = np.zeros((2, CAP), pkg.TAG_DTYPE), np.zeros(2, np.int32), np.zeros(2, np.uint32)
        d_out = torch.zeros((2, CAP * 9), dtype=torch.int32, device="cuda")
        d_cnt = torch.full((2,), -7, dtype=torch.int32, device="cuda")
        n0 = det.launch_count
        calls = {
            "detect": lambda p, rs, fs: L.ag_detect(det._h, p, w, h, rs, code, vp(out), CAP, vp(cnt)),
            "batch": lambda p, rs, fs: L.ag_detect_batch(det._h, p, fs, 2, w, h, rs, code, vp(out), CAP, vp(cnt), vp(st)),
            "multi": lambda p, rs, fs: L.ag_multi_detect_batch(multi._h, p, fs, 2, w, h, rs, code, vp(out), CAP, vp(cnt),
                                                               vp(st)),
            "saddles": lambda p, rs, fs: L.ag_refined_saddle_points(det._h, p, w, h, rs, code, vp(out), CAP, vp(cnt)),
            "stage": lambda p, rs, fs: L.ag_stage_run(det._h, p, w, h, rs, code),
        }
        dev_calls = {
            "device": lambda p, rs, fs: L.ag_detect_batch_device(det._h, p, fs, 2, w, h, rs, code, d_out.data_ptr(), CAP,
                                                                 d_cnt.data_ptr(), None, None),
            "dense": lambda p, rs, fs: L.ag_dense_batch_device(det._h, p, fs, 2, w, h, rs, code, None),
        }
        for name, call in calls.items():
            assert call(buf.ctypes.data, rb + 2, 0) == pkg.AG_ERR_INVALID, (name, "row stride 2 (mod 4)")
            if name in ("batch", "multi"):
                assert call(buf.ctypes.data, rb, rb * h + 2) == pkg.AG_ERR_INVALID, (name, "frame stride 2 (mod 4)")
        for name, call in dev_calls.items():
            assert call(dbuf.data_ptr(), rb + 2, 0) == pkg.AG_ERR_INVALID, (name, "row stride 2 (mod 4)")
            assert call(dbuf.data_ptr(), rb, rb * h + 2) == pkg.AG_ERR_INVALID, (name, "frame stride 2 (mod 4)")
            assert call(dbuf.data_ptr() + 2, rb, 0) == pkg.AG_ERR_INVALID, (name, "address 2 (mod 4)")
        torch.cuda.synchronize()
        assert det.launch_count == n0
        assert (d_cnt.cpu().numpy() == -7).all()
    finally:
        multi.close()
        det.close()
