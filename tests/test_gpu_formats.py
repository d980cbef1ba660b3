"""The pixel formats LA8, RGBA8, LA16, RGB16 and RGBA16 on the GPU.  Needs a B200: -m gpu.

- Parity with the oracle on each frame's reference frame (formats_ref: L8 / L16 / RGB8 frames of the
  same gray conversion): a rendered board and a noisy synthetic frame in each format, with random
  alpha, bit-exact through every stage and through every entry point that takes a frame.
- Equivalence with the formats the library had before, independent of the oracle: LA8 = L8,
  RGBA8 = RGB8 without alpha, LA16 = L16, RGB16 / RGBA16 = L16 of their Y16 plane; alpha 0, max and
  random give identical results.
- Both K1 kernels (streaming and tile) with padded rows, gaps between frames and misaligned bases.
- The painted decode-gate frames of synth.gate_frames, built in each format by formats_ref.
- Odd strides and device addresses of the 16-bit formats are refused before anything runs."""
import ctypes as C

import numpy as np
import pytest

import formats_ref as fr
import synth
from test_gpu_parity import assert_saddles_match, assert_tags_match, check_stages

pytestmark = pytest.mark.gpu

FORMATS = list(fr.NEW_FORMATS)
CODE, BPP = fr.CODE, fr.BPP
CAP = 128


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def same_tags(got, want):
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for k in want:
        assert np.array_equal(got[k], want[k]), (k, got[k], want[k])


@pytest.fixture(scope="module")
def ref(oracle):
    return fr.RefOracle(oracle)


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def to_format(l8, fmt, seed=0, noise=True):
    """An L8 frame in format fmt: colour channels differ by a seeded noise (so a swapped channel order
    or a wrong weight changes the luma), 16-bit words use all their bits, alpha is random."""
    rng = np.random.default_rng(seed)
    wide = fmt.endswith("16")
    top = 65535 if wide else 255
    base = l8.astype(np.int64) * (257 if wide else 1)
    if wide:
        base = base + (rng.integers(-128, 129, l8.shape) if noise else 0)
    n_col = 1 if fmt.startswith("la") else 3
    chans = [base] if n_col == 1 else [base + (rng.integers(-9, 10, l8.shape) * (257 if wide else 1) if noise else 0)
                                         for _ in range(3)]
    if fmt in fr.ALPHA_FORMATS:
        chans.append(rng.integers(0, top + 1, l8.shape))
    return np.ascontiguousarray(np.clip(np.stack(chans, axis=2), 0, top).astype(np.uint16 if wide else np.uint8))


def frames_for(fmt):
    board = synth.render_board_numpy(640, 480, seed=41, tag_px=44.0)
    noise = np.random.default_rng(5).integers(0, 256, (96, 128)).astype(np.uint8)
    return [to_format(board, fmt, seed=1), to_format(noise, fmt, seed=2)]


def device_batch(pkg, det, torch, frames, fmt, fs=0, rs=0, ptr=None):
    n, h, w = frames.shape[:3]
    host = frames.view(np.int16) if frames.dtype == np.uint16 else frames  # torch has no uint16 copy
    d = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    det.detect_batch_device(d.data_ptr() if ptr is None else ptr, n, w, h, CODE[fmt], out.data_ptr(), CAP,
                            cnt.data_ptr(), st.data_ptr(), stream=torch.cuda.current_stream().cuda_stream,
                            frame_stride=fs, row_stride=rs)
    torch.cuda.synchronize()
    rec = out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
    c = cnt.cpu().numpy()
    assert not st.cpu().numpy().any()
    return [pkg._tags_to_dict(rec[i, :c[i]]) for i in range(n)]


# ---- parity with the oracle, every entry point ---------------------------------------------------
@pytest.mark.parametrize("fmt", FORMATS)
def test_parity_every_entry_point(pkg, ref, torch_mod, fmt):
    torch = torch_mod
    board, noise = frames_for(fmt)
    want = ref.detect(board)
    assert len(want) == 36
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    multi = pkg.MultiTagDetector(pkg.TagFamily.T36H11, None, devices=[0, 0])
    try:
        for img in (board, noise):
            check_stages(det, ref, img)  # ag_stage_run: every stage bit-exact
            assert_tags_match(det.detect(img), ref.detect(img))
            assert_saddles_match(det.refined_saddle_points(img), ref.front_end(img, want_labels=False)["refined"])
        o = ref.front_end(board, want_labels=False)["refined"]
        quads, tags = det._boards_from_saddles(o, board)
        assert np.array_equal(quads, ref.try_find_best_board(o))
        same_tags(tags, want)
        batch = np.stack([board, np.zeros_like(board), board[::-1, ::-1].copy()])
        wants = [ref.detect(f) for f in batch]
        for got in (det.detect_batch(batch, cap_per_frame=CAP), multi.detect_batch(batch, cap_per_frame=CAP),
                    device_batch(pkg, det, torch, batch, fmt)):
            for g, wt in zip(got, wants):
                same_tags(g, wt)
        # pinned host frames, synchronous and streaming
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
        # the dense front end alone runs on the format
        d = torch.from_numpy(batch.view(np.int16) if batch.dtype == np.uint16 else batch).cuda()
        n0 = det.launch_count
        det.dense_batch_device(d.data_ptr(), len(batch), batch.shape[2], batch.shape[1], CODE[fmt])
        torch.cuda.synchronize()
        assert det.launch_count > n0
    finally:
        multi.close()
        det.close()


# ---- equivalence with the existing formats -------------------------------------------------------
def results(pkg, det, torch, img, fmt):
    g = det.stages(img)
    batch = np.stack([img, img[::-1, ::-1].copy()])
    out = np.zeros((2, CAP), pkg.TAG_DTYPE)
    cnt, st = np.zeros(2, np.int32), np.zeros(2, np.uint32)
    w, h = img.shape[1], img.shape[0]
    det._check(pkg.lib().ag_detect_batch(det._h, vp(batch), batch.strides[0], 2, w, h, batch.strides[1], CODE[fmt],
                                         vp(out), CAP, vp(cnt), vp(st)))
    dev = device_batch(pkg, det, torch, batch, fmt)
    return g, out.tobytes(), cnt.tobytes(), dev


def assert_same_results(a, b, what):
    ga, gb = a[0], b[0]
    for k in ("blur", "resp", "mask", "labels", "centers", "raw", "refined", "quads"):
        assert np.asarray(ga[k]).tobytes() == np.asarray(gb[k]).tobytes(), (what, k)
    assert np.float32(ga["min"]) == np.float32(gb["min"]) and np.float32(ga["thr"]) == np.float32(gb["thr"])
    same_tags(ga["tags"], gb["tags"])
    assert a[1] == b[1] and a[2] == b[2], what
    for x, y in zip(a[3], b[3]):
        same_tags(x, y)


@pytest.mark.parametrize("fmt", FORMATS)
def test_equivalent_to_existing_formats(pkg, torch_mod, fmt):
    torch = torch_mod
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for img in frames_for(fmt):
            ref_img = fr.reference_frame(img)
            ref_fmt = fr.format_of(ref_img)
            want = results(pkg, det, torch, ref_img, ref_fmt)
            assert_same_results(results(pkg, det, torch, img, fmt), want, (fmt, ref_fmt))
            if fmt in fr.ALPHA_FORMATS:
                for a in (0, np.iinfo(img.dtype).max):
                    other = img.copy()
                    other[:, :, -1] = a
                    assert_same_results(results(pkg, det, torch, other, fmt), want, (fmt, "alpha", a))
    finally:
        det.close()


# ---- both K1 kernels: strided and misaligned frames ----------------------------------------------
def layouts(fmt, w, h):
    """(name, row_stride, frame_stride, base offset): rows and frames aligned for the streaming K1, rows
    padded so that it cannot run, a gap between frames, and a base offset that breaks its alignment
    (even for the 16-bit formats, whose pixels must stay 2-byte aligned)."""
    rb = w * BPP[fmt]
    wide = rb + 32
    pad = 2 if fmt.endswith("16") else 1
    return [("rows_stream", wide, wide * h, 0), ("rows_tile", rb + pad, (rb + pad) * h, 0),
            ("frame_gap", wide, wide * h + 16 * pad, 0), ("offset", wide, wide * h, 2 if pad == 2 else 4),
            ("offset_small", rb + pad, (rb + pad) * h, pad)]


def lay_out(frames, rs, fs, offset, seed):
    n, h = frames.shape[:2]
    rb = frames[0, 0].nbytes
    size = offset + (n - 1) * fs + rs * (h - 1) + rb
    buf = np.random.default_rng(seed).integers(0, 256, size + 64, dtype=np.uint8)
    view = np.ndarray(frames.shape, frames.dtype, buffer=buf, offset=offset, strides=(fs, rs) + frames.strides[2:])
    view[...] = frames
    return buf


@pytest.mark.parametrize("w", [640, 642])
@pytest.mark.parametrize("fmt", FORMATS)
def test_frame_layouts(pkg, ref, torch_mod, fmt, w):
    torch, oracle_ref = torch_mod, ref
    L = pkg.lib()
    h = 480
    board = to_format(synth.render_board_numpy(w, h, seed=31, tag_px=44.0), fmt, seed=3)
    frames = np.stack([board, np.zeros_like(board), board[::-1, ::-1].copy()])
    n, code, rb = len(frames), CODE[fmt], frames[0, 0].nbytes
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("chunk_frames", 2)
        ref = (np.zeros((n, CAP), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.zeros(n, np.uint32))
        det._check(L.ag_detect_batch(det._h, vp(frames), frames.strides[0], n, w, h, rb, code, vp(ref[0]), CAP,
                                     vp(ref[1]), vp(ref[2])))
        assert not ref[2].any() and ref[1][0] >= 30 and ref[1][1] == 0 and ref[1][2] >= 30
        same_tags(pkg._tags_to_dict(ref[0][0, :ref[1][0]]), oracle_ref.detect(board))
        o0 = oracle_ref.front_end(board, want_labels=False)
        for name, rs, fs, off in layouts(fmt, w, h):
            case = (fmt, w, name)
            buf = lay_out(frames, rs, fs, off, seed=rs + fs)
            base = buf.ctypes.data + off
            got = (np.zeros((n, CAP), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.zeros(n, np.uint32))
            det._check(L.ag_detect_batch(det._h, base, fs, n, w, h, rs, code, vp(got[0]), CAP, vp(got[1]), vp(got[2])))
            assert all(np.array_equal(x, y) for x, y in zip(got, ref)), ("batch",) + case
            cnt = C.c_int(0)
            one = np.zeros(CAP, pkg.TAG_DTYPE)
            det._check(L.ag_detect(det._h, base, w, h, rs, code, vp(one), CAP, C.byref(cnt)))
            assert cnt.value == ref[1][0] and np.array_equal(one[:cnt.value], ref[0][0, :cnt.value]), ("detect",) + case
            dbuf = torch.from_numpy(buf).cuda()
            view = torch.as_strided(dbuf, (n, h, rb), (fs, rs, 1), storage_offset=off)
            d_out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
            d_cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
            det.detect_batch_device(view.data_ptr(), n, w, h, code, d_out.data_ptr(), CAP, d_cnt.data_ptr(),
                                    None, frame_stride=fs, row_stride=rs)
            torch.cuda.synchronize()
            rec = d_out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
            assert np.array_equal(rec, ref[0]) and np.array_equal(d_cnt.cpu().numpy(), ref[1]), ("device",) + case
            det._check(L.ag_stage_run(det._h, base, w, h, rs, code))
            blur, resp = np.empty((h, w), np.float32), np.empty((h, w), np.float32)
            det._check(L.ag_stage_blur(det._h, vp(blur)))
            det._check(L.ag_stage_response(det._h, vp(resp)))
            assert np.array_equal(blur.view(np.uint32), o0["blur"].view(np.uint32)), ("blur",) + case
            assert np.array_equal(resp.view(np.uint32), o0["resp"].view(np.uint32)), ("resp",) + case
    finally:
        det.close()


# ---- decode gates ----------------------------------------------------------------------------------
@pytest.mark.parametrize("family", list(synth.GATE_FAMILIES))
def test_painted_frames(pkg, ref, torch_mod, family):
    torch = torch_mod
    tf = pkg.TagFamily[family.upper()]
    det = pkg.TagDetector(tf)
    try:
        det.set_option("chunk_frames", 3)
        batches = {}
        for name, scene, tags, fmt, frame, mbs in fr.gate_frames(family):
            if 2 not in mbs:
                continue
            want = ref.detect(frame, family=family)
            same_tags(det.detect(frame), want)
            batches.setdefault((fmt, frame.shape), []).append((frame, want))
        for (fmt, _), items in batches.items():
            frames = np.stack([f for f, _ in items] * 2)
            wants = [w for _, w in items] * 2
            for g, wt in zip(det.detect_batch(frames, cap_per_frame=CAP), wants):
                same_tags(g, wt)
            for g, wt in zip(device_batch(pkg, det, torch, frames, fmt), wants):
                same_tags(g, wt)
    finally:
        det.close()


# ---- refusals -------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["la16", "rgb16", "rgba16"])
def test_16bit_odd_strides_and_addresses_are_refused(pkg, torch_mod, fmt):
    torch = torch_mod
    L = pkg.lib()
    w, h = 64, 48
    rb = w * BPP[fmt]
    code = CODE[fmt]
    buf = np.zeros(2 * (rb + 1) * h + 64, np.uint8)
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
            assert call(buf.ctypes.data, rb + 1, 0) == pkg.AG_ERR_INVALID, (name, "odd row stride")
            if name in ("batch", "multi"):
                assert call(buf.ctypes.data, rb, rb * h + 1) == pkg.AG_ERR_INVALID, (name, "odd frame stride")
        for name, call in dev_calls.items():
            assert call(dbuf.data_ptr(), rb + 1, 0) == pkg.AG_ERR_INVALID, (name, "odd row stride")
            assert call(dbuf.data_ptr(), rb, rb * h + 1) == pkg.AG_ERR_INVALID, (name, "odd frame stride")
            assert call(dbuf.data_ptr() + 1, rb, 0) == pkg.AG_ERR_INVALID, (name, "odd address")
        torch.cuda.synchronize()
        assert det.launch_count == n0
        assert (d_cnt.cpu().numpy() == -7).all()
    finally:
        multi.close()
        det.close()
