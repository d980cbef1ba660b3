"""The detector's one-frame slot, which runs detect_planes, refined_saddle_points, the stage taps and
the re-run of batch frames that overflowed their capacities.  Needs a B200: -m gpu."""
import ctypes as C

import numpy as np
import pytest

import synth
from test_gpu_parity import assert_tags_match

pytestmark = pytest.mark.gpu

H, W = 1024, 1280


@pytest.fixture(scope="module")
def noise():
    """iid noise: 65 k clusters and 11 k refined saddles, beyond the default 16384 / 2048 of the size."""
    return np.random.default_rng(5).integers(0, 256, (H, W), dtype=np.uint8)


def test_detect_planes_grows_capacities(pkg, oracle, noise):
    """detect_planes re-runs a frame that overflows the capacities with grown ones, like detect; a frame
    beyond 16384 refined saddles is an error, never a truncated map."""
    assert len(oracle.front_end(noise, want_labels=False)["refined"]) > 8000
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        f, u = oracle.to_luma_f32(noise), oracle.to_luma_u8(noise)
        assert_tags_match(det.detect_planes(f, u), oracle.detect_planes(f, u))
        yy, xx = np.mgrid[0:H, 0:W]
        dense = np.where(((yy // 5) + (xx // 5)) % 2 == 0, 40, 200).astype(np.uint8)
        if len(oracle.front_end(dense, want_labels=False)["refined"]) > 16384:
            with pytest.raises(RuntimeError, match="limits"):
                det.detect_planes(oracle.to_luma_f32(dense), oracle.to_luma_u8(dense))
    finally:
        det.close()


def test_batch_rerun_invalidates_the_stage_taps(pkg, oracle):
    """A batch frame re-run on the one-frame slot overwrites the buffers the stage taps read: after it,
    the taps refuse until the next stages() call instead of returning another frame's data."""
    L = pkg.lib()
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.stages(synth.render_board_numpy(160, 120, seed=3), want_labels=False)
        det.set_option("max_clusters", 16)  # every board frame overflows and is re-run
        frames = np.stack([synth.render_board_numpy(640, 480, seed=s, tag_px=44.0) for s in (3, 4)])
        tags, status = det.detect_batch(frames, return_status=True)
        assert not status.any()
        for t, f in zip(tags, frames):
            assert_tags_match(t, oracle.detect(f))
        # only taps that copy a buffer: the labels tap would launch a kernel on the overwritten slot
        blur = np.zeros((120, 160), np.float32)
        min_thr = np.zeros(2, np.float32)
        out = np.zeros(1024, pkg.TAG_DTYPE)
        n = C.c_int(0)
        assert L.ag_stage_blur(det._h, pkg._p(blur)) == pkg.AG_ERR_INVALID
        assert L.ag_stage_threshold(det._h, pkg._p(min_thr)) == pkg.AG_ERR_INVALID
        assert L.ag_stage_tags(det._h, pkg._p(out), len(out), C.byref(n)) == pkg.AG_ERR_INVALID
    finally:
        det.close()


def test_stage_taps_of_an_overflowed_frame(pkg, oracle, noise):
    """The taps show an overflowed frame as the pipeline left it: the first 16384 centres, and no
    quads or tags from the board search, which skips a frame flagged as truncated (no tap shows the
    status itself), even right after a frame that had both."""
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        g = det.stages(synth.render_board_numpy(W, H, seed=5), want_labels=False)
        assert len(g["quads"]) > 0 and len(g["tags"]) == 36
        g = det.stages(noise, want_labels=False)
        o = oracle.front_end(noise, want_labels=False)
        assert len(o["centers"]) > 16384
        assert np.array_equal(g["centers"].view(np.uint32), o["centers"][:16384].view(np.uint32))
        assert len(g["quads"]) == 0 and len(g["tags"]) == 0
    finally:
        det.close()


@pytest.mark.parametrize("key", ["dense_streams", "label_list"])
def test_removed_options_are_refused(pkg, detector, key):
    assert pkg.lib().ag_set_option(detector._h, key.encode(), 1) == pkg.AG_ERR_INVALID
