"""Tag decoding at its gates on the GPU, against the oracle.  Needs a B200: -m gpu.

The painted frames of synth.gate_frames (contrast 49 / 50, mid levels on a half, uncertain samples
at 9 and 10 from mid, 1 .. hamming bit errors, rotations, repeated ids inside one lane batch and
across two, boards rejected but for a few tags, L16 and RGB8 values on the to_luma8 boundaries) go
through the whole pipeline -- detect, detect_batch, detect_batch_device and the stage taps -- and
their saddle lists through the board kernel's test hook in every board-search variant.  Tag ids must
be equal and corners array_equal: the corners are saddle positions, so they are exact."""
import numpy as np
import pytest

import synth
from test_gpu_parity import BOARD_VARIANTS

pytestmark = pytest.mark.gpu

FAMILIES = list(synth.GATE_FAMILIES)
FMT = {"l8": 0, "l16": 1, "rgb8": 2}
CAP = 128


def same_tags(got, want):
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for k in want:
        assert np.array_equal(got[k], want[k]), (k, got[k], want[k])


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


_FRAMES = {}


def frames_of(family):
    if family not in _FRAMES:
        _FRAMES[family] = synth.gate_frames(family)
    return _FRAMES[family]


def detect_device(pkg, det, torch, frames, fmt):
    n, h, w = frames.shape[:3]
    host = frames.view(np.int16) if frames.dtype == np.uint16 else frames  # torch has no uint16 copy
    d = torch.from_numpy(np.ascontiguousarray(host)).cuda()
    out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    det.detect_batch_device(d.data_ptr(), n, w, h, FMT[fmt], out.data_ptr(), CAP, cnt.data_ptr(), st.data_ptr(),
                            stream=torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    rec = out.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, CAP)
    c = cnt.cpu().numpy()
    return [pkg._tags_to_dict(rec[i, :c[i]]) for i in range(n)], st.cpu().numpy()


@pytest.mark.parametrize("family", FAMILIES)
def test_painted_frames_full_pipeline(pkg, oracle, torch_mod, family):
    tf = pkg.TagFamily[family.upper()]
    dets = {mb: pkg.TagDetector(tf, pkg.DetectorParams(max_num_of_boards=mb)) for mb in (1, 2, 3)}
    try:
        batches = {}
        for name, scene, tags, fmt, frame, mbs in frames_of(family):
            for mb in mbs:
                want = oracle.detect(frame, family=family, max_boards=mb)
                synth.check_expectations(scene, tags, want, oracle.to_luma_u8(frame))
                same_tags(dets[mb].detect(frame), want)
                g = dets[mb].stages(frame, want_labels=False)
                o = oracle.front_end(frame, want_labels=False)["refined"]
                assert np.array_equal(g["quads"], oracle.try_find_best_board(o)), (name, fmt)
                same_tags(g["tags"], want)
                batches.setdefault((mb, fmt, frame.shape), []).append((frame, want))
        # batches mixing the scenario frames of one format and size, in chunks of three
        det = dets[2]
        det.set_option("chunk_frames", 3)
        for (mb, fmt, _), items in batches.items():
            if mb != 2:
                continue
            frames = np.stack([f for f, _ in items] * 2)  # every frame twice: ragged chunks
            wants = [wt for _, wt in items] * 2
            got, status = det.detect_batch(frames, cap_per_frame=CAP, return_status=True)
            assert not status.any(), status
            for g_, wt in zip(got, wants):
                same_tags(g_, wt)
            got, status = detect_device(pkg, det, torch_mod, frames, fmt)
            assert not status.any(), status
            for g_, wt in zip(got, wants):
                same_tags(g_, wt)
    finally:
        for d in dets.values():
            d.close()


@pytest.mark.parametrize("family", FAMILIES)
def test_saddle_hook_every_board_variant(pkg, oracle, family):
    """The painted frames' saddle lists, a sample on k + 0.5 (k even) and a quad corner at w - 0.5 /
    h - 0.5 and one ulp below, through the board kernel's hook in every board-search variant."""
    tf = pkg.TagFamily[family.upper()]
    scene = synth.gate_scene(family)
    half = synth.half_sample_case(scene)
    assert half is not None
    s, img, tid, _ = half
    cases = [("half_sample", s, img, tid, True)] + synth.edge_corner_cases(scene)
    inputs = []
    for name, s, img, tid, decodes in cases:
        for fmt in FMT:
            frame = synth.encode(img, {}, fmt, {})
            want = oracle.detect_from_saddles(frame, s, family=family)
            assert (tid in want) == decodes, (name, fmt)
            inputs.append((name, s, frame, want))
    for name, scene_, tags, fmt, frame, mbs in frames_of(family):
        if 2 in mbs:
            sd = oracle.front_end(frame, want_labels=False)["refined"]
            inputs.append((name, sd, frame, oracle.detect_from_saddles(frame, sd, family=family)))
    for variant in BOARD_VARIANTS:
        det = pkg.TagDetector(tf)
        try:
            for key, v in variant.items():
                det.set_option(key, v)
            for name, sd, frame, want in inputs:
                quads, tags = det._boards_from_saddles(sd, frame)
                assert np.array_equal(quads, oracle.try_find_best_board(sd)), (name, variant)
                same_tags(tags, want)
        finally:
            det.close()


def test_large_board_decode_scratch_per_frame(pkg, oracle):
    """A board listing more quads than the decode scratch of the board kernel used to hold (lattice 32,
    max_saddles 4096: room for 772 bit patterns before the layout was fixed), one warp per frame: three
    identical frames in one batch give byte-identical tags and status to the frame run alone.  The
    board is wider than the 32-cell lattice, so the frame is flagged (AG_ERR_CAPACITY) either way."""
    import ctypes as C
    # T16H5: 3636 refined saddles, within max_saddles (a T36H11 board of this size has 4404)
    img = synth.render_board_numpy(2600, 2600, cols=30, rows=30, seed=1, family="t16h5", noise=0.0, ss=2)
    det = pkg.TagDetector(pkg.TagFamily.T16H5)
    L = pkg.lib()

    def batch(frames):
        n = len(frames)
        out = np.zeros((n, 1024), pkg.TAG_DTYPE)
        cnt = np.zeros(n, np.int32)
        st = np.zeros(n, np.uint32)
        rc = L.ag_detect_batch(det._h, pkg._p(frames), frames.strides[0], n, 2600, 2600, 2600, pkg.FMT_L8,
                               pkg._p(out), 1024, pkg._p(cnt), pkg._p(st))
        assert rc in (pkg.AG_OK, pkg.AG_ERR_CAPACITY), rc
        return out, cnt, st

    try:
        det.set_option("board_lattice", 32)
        det.set_option("max_saddles", 4096)
        det.set_option("board_warps", 1)
        out1, cnt1, st1 = batch(np.ascontiguousarray(img[None]))
        assert L.ag_stage_run(det._h, pkg._p(img), 2600, 2600, 2600, pkg.FMT_L8) in (pkg.AG_OK, pkg.AG_ERR_CAPACITY)
        quads, nq = np.zeros((4096, 4), np.int32), C.c_int(0)
        assert L.ag_stage_board_quads(det._h, pkg._p(quads), 4096, C.byref(nq)) == pkg.AG_OK
        print("large board: %d listed quads in the first round, %d tags, status %d"
              % (nq.value, cnt1[0], int(st1[0])))
        out3, cnt3, st3 = batch(np.stack([img] * 3))
        for k in range(3):
            assert st3[k] == st1[0] and cnt3[k] == cnt1[0]
            assert out3[k].tobytes() == out1[0].tobytes()
    finally:
        det.close()
