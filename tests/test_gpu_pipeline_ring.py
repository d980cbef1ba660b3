"""The batch pipelines' dense ring and sparse stream, against the oracle.  Needs a B200: -m gpu.

Chunks use the two sets of dense buffers in turn: K1-K2 of a chunk run on the dense stream while
K3-K4 of the chunk before still read the other set on the sparse stream, and K6 runs on one of
eight board slots.  Small chunks over long batches wrap the ring and the board slots many times,
with different content in consecutive chunks: rendered boards, a board whose lower half is noise
(more runs than the run-based labeller holds, so K3 hands the frame to the pixel-list kernel,
which uses the set's response buffer as per-pixel scratch), full-frame noise and a fine
checkerboard (they overflow max_clusters / max_saddles) and a blank frame.  Every frame must give
the oracle's ids and corners and the same bytes as the frame detected alone; overflowed frames carry
their status bits on the device path and are re-run on the host path."""
import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu

W, H, CAP = 640, 480, 64
CORNER_TOL = 1e-3
GROWABLE = 1 | 2  # AG_FRAME_CLUSTER_OVERFLOW | AG_FRAME_SADDLE_OVERFLOW
RUN_CAP = 12288  # runs per frame the run-based labeller holds in shared memory (csrc/ag_sparse.cu)
# capacities between what the fitting frames need and what the overflowing ones need
OPTIONS = dict(max_clusters=8192, max_saddles=1536)


def _runs(labels):
    m = labels >= 0
    return int((m & ~np.pad(m, ((0, 0), (1, 0)))[:, :-1]).sum())


@pytest.fixture(scope="module")
def scenes(oracle):
    """Distinct frames, their oracle tags and whether they overflow OPTIONS."""
    rng = np.random.default_rng(11)
    boards = [synth.render_board_numpy(W, H, seed=s, tag_px=44.0) for s in (21, 22, 23)]
    band = boards[0].copy()
    band[H - 240:] = rng.integers(0, 256, (240, W), dtype=np.uint8)
    noise = rng.integers(0, 256, (H, W), dtype=np.uint8)
    yy, xx = np.mgrid[0:H, 0:W]
    checker = np.where(((yy // 12) + (xx // 12)) % 2 == 0, 40, 200).astype(np.uint8)
    blank = np.full((H, W), 128, np.uint8)
    frames = boards + [band, noise, checker, blank]
    kinds = ["board"] * 3 + ["band", "noise", "checker", "blank"]
    fe = {k: oracle.front_end(f) for k, f in zip(kinds[3:6], frames[3:6])}
    # premises: the band frame fits but takes the pixel-list labeller; noise and checker overflow
    assert _runs(fe["band"]["labels"]) > RUN_CAP
    assert len(fe["band"]["centers"]) <= OPTIONS["max_clusters"]
    assert len(fe["band"]["refined"]) <= OPTIONS["max_saddles"]
    assert len(fe["noise"]["centers"]) > OPTIONS["max_clusters"]
    assert len(fe["checker"]["refined"]) > OPTIONS["max_saddles"]
    want = [oracle.detect(f) for f in frames]
    assert all(len(w) == 36 for w in want[:3]) and len(want[3]) > 0
    overflow = [k in ("noise", "checker") for k in kinds]
    return frames, want, overflow


def _order(n, n_distinct, offset=0):
    # a stride coprime to the number of distinct frames: every chunk of 4 or 8 frames is mixed, and
    # consecutive chunks (other set of the ring) differ
    return [(3 * i + offset) % n_distinct for i in range(n)]


def _detector(pkg, **opts):
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    for k, v in dict(OPTIONS, **opts).items():
        det.set_option(k, v)
    return det


def _tags(rec, cnt):
    return [{int(t["id"]): t["xy"].reshape(4, 2).copy() for t in rec[i, :cnt[i]]} for i in range(len(cnt))]


def _assert_same(got, want, exact):
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for k in want:
        if exact:
            assert np.array_equal(got[k], want[k]), (k, got[k], want[k])
        else:
            assert np.abs(got[k] - want[k]).max() <= CORNER_TOL, (k, got[k], want[k])


def _singles(det, frames):
    return [det.detect(f) for f in frames]


def _device_out(torch, n):
    return (torch.full((n, CAP * 9), -1, dtype=torch.int32, device="cuda"),
            torch.full((n,), -1, dtype=torch.int32, device="cuda"),
            torch.full((n,), -1, dtype=torch.int32, device="cuda"))


def _read(pkg, out):
    tags, cnt, st = (t.cpu().numpy() for t in out)
    return _tags(tags.view(pkg.TAG_DTYPE).reshape(len(cnt), CAP), cnt), st.view(np.uint32)


def _check_device(got, status, order, scenes, singles):
    frames, want, overflow = scenes
    for i, k in enumerate(order):
        if overflow[k]:
            assert status[i] & GROWABLE, (i, k, status[i])
            continue
        assert status[i] == 0, (i, k, status[i])
        _assert_same(got[i], want[k], exact=False)
        _assert_same(got[i], singles[k], exact=True)


@pytest.mark.parametrize("chunk", [4, 8])
def test_device_batches_wrap_the_ring(pkg, scenes, chunk):
    """ag_detect_batch_device, synchronising calls: 96 frames in chunks of 4 / 8 (24 / 12 chunks:
    the two dense sets and the eight board slots wrap several times), twice on the same handle."""
    import torch
    frames, want, overflow = scenes
    det = _detector(pkg, chunk_frames=chunk)
    try:
        singles = _singles(det, frames)
        for k in range(len(frames)):
            if not overflow[k]:
                _assert_same(singles[k], want[k], exact=False)
        stream = torch.cuda.Stream()
        for offset in (0, 1):
            order = _order(96, len(frames), offset)
            d_frames = torch.from_numpy(np.stack([frames[k] for k in order])).cuda()
            out = _device_out(torch, 96)
            torch.cuda.synchronize()
            det.detect_batch_device(d_frames.data_ptr(), 96, W, H, pkg.FMT_L8, out[0].data_ptr(), CAP,
                                    out[1].data_ptr(), out[2].data_ptr(), stream=stream.cuda_stream)
            stream.synchronize()
            got, status = _read(pkg, out)
            _check_device(got, status, order, scenes, singles)
    finally:
        det.close()


def test_host_batches_wrap_the_ring_and_rerun_overflows(pkg, scenes):
    """ag_detect_batch in chunks of 4: frames that overflowed their chunk are re-run alone with grown
    capacities, so every frame gives the oracle's result and no status bit."""
    frames, want, _ = scenes
    det = _detector(pkg, host_chunk_frames=4)
    try:
        singles = _singles(det, frames)
        order = _order(64, len(frames))
        got, status = det.detect_batch(np.stack([frames[k] for k in order]), cap_per_frame=CAP, return_status=True)
        assert not status.any()
        for i, k in enumerate(order):
            _assert_same(got[i], want[k], exact=False)
            _assert_same(got[i], singles[k], exact=True)
    finally:
        det.close()


def test_async_device_calls_on_two_streams(pkg, scenes):
    """device_async calls back to back on two caller streams, different frames in each, then one
    ag_detect_batch_device_wait: the second call's K1 must not overwrite a set whose K3-K4 of the
    first call are still to run, whatever stream each call came on."""
    import torch
    frames, want, overflow = scenes
    det = _detector(pkg, chunk_frames=4)
    try:
        singles = _singles(det, frames)
        s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        orders = [_order(72, len(frames), off) for off in (0, 2, 5)]
        d_frames = [torch.from_numpy(np.stack([frames[k] for k in o])).cuda() for o in orders]
        outs = [_device_out(torch, 72) for _ in orders]
        torch.cuda.synchronize()
        det.set_option("device_async", 1)
        for s, d, out in zip((s1, s2, s1), d_frames, outs):
            det.detect_batch_device(d.data_ptr(), 72, W, H, pkg.FMT_L8, out[0].data_ptr(), CAP, out[1].data_ptr(),
                                    out[2].data_ptr(), stream=s.cuda_stream)
        det.detect_batch_device_wait(stream=s3.cuda_stream)
        det.set_option("device_async", 0)
        s3.synchronize()
        for o, out in zip(orders, outs):
            got, status = _read(pkg, out)
            _check_device(got, status, o, scenes, singles)
    finally:
        det.close()


def test_streaming_host_calls_interleaved_with_device_calls(pkg, scenes):
    """host_async calls in flight while device calls run on the same handle: both pipelines share the
    ring, the sparse stream and the board slots; every result is complete and correct."""
    import torch
    frames, want, overflow = scenes
    det = _detector(pkg, chunk_frames=4, host_chunk_frames=4)
    try:
        singles = _singles(det, frames)
        n = 40
        orders = [_order(n, len(frames), off) for off in range(4)]
        host_src = [np.stack([frames[k] for k in o]) for o in orders]
        d_frames = [torch.from_numpy(h).cuda() for h in host_src]
        host_outs = [(np.zeros((n, CAP), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.ones(n, np.uint32))
                     for _ in orders]
        dev_outs = [_device_out(torch, n) for _ in orders]
        stream = torch.cuda.Stream()
        torch.cuda.synchronize()
        det.set_option("host_async", 1)
        for j in range(len(orders)):
            det.detect_batch_into(host_src[j], *host_outs[j])
            out = dev_outs[(j + 1) % len(orders)]
            d = d_frames[(j + 1) % len(orders)]
            det.detect_batch_device(d.data_ptr(), n, W, H, pkg.FMT_L8, out[0].data_ptr(), CAP, out[1].data_ptr(),
                                    out[2].data_ptr(), stream=stream.cuda_stream)
        det.detect_batch_wait(0)
        det.set_option("host_async", 0)
        stream.synchronize()
        for j, o in enumerate(orders):
            tags, cnt, st = host_outs[j]
            assert not st.any()
            for t, k in zip(_tags(tags, cnt), o):
                _assert_same(t, want[k], exact=False)
                _assert_same(t, singles[k], exact=True)
            got, status = _read(pkg, dev_outs[j])
            _check_device(got, status, o, scenes, singles)
    finally:
        det.close()


def test_operator_before_the_first_batch(pkg, scenes):
    """A standalone operator as the handle's first call sets up the first dense set's stream; the
    batch pipelines called after it still find every event of the ring."""
    frames, want, _ = scenes
    det = _detector(pkg)
    try:
        det.gaussian_blur_f32(frames[0].astype(np.float32))
        got = det.detect_batch(np.stack(frames[:3]), cap_per_frame=CAP)
        for g, w in zip(got, want[:3]):
            _assert_same(g, w, exact=False)
    finally:
        det.close()
