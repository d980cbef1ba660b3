"""Frame lists of mixed sizes and pixel formats (ag_detect_frames, ag_refined_saddle_points_frames, their
_device and ag_multi_ forms).  Needs a B200: -m gpu.

Every frame's result must be byte-identical to the one-frame call on that frame alone (ag_detect /
ag_refined_saddle_points: count, records, status), and nothing past min(n, cap) records of a frame's
slot may be written.  Covered: the reference fixtures in one shuffled list with repeats; all ten pixel
formats with odd and streaming widths, padded rows, odd host addresses and device addresses that rule
out the streaming K1 for some frames of a chunk; groups of 1 to 7 frames in chunks of three that wrap
the dense ring and every board slot; device calls on two streams and asynchronous calls interleaved with
detect_batch_device; capacity overflows; invalid lists; uniform lists against the batch calls; several
devices; and the C++ mirror."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import float_formats_ref as ffr
import formats_ref as fr
import synth
from conftest import FIXTURE_NAMES
from test_gpu_board_edges import STRIPS
from test_gpu_parity import assert_tags_match
from test_gpu_saddle_batch import format_frame

pytestmark = pytest.mark.gpu

CANARY = 0xDEADBEEF
GROWABLE = 1 | 2
BOARD_OVERFLOW = 4
TAG_OVERFLOW = 8
WORDS = {"tags": 9, "saddles": 5}
ALL_FORMATS = ("l8", "l16", "rgb8") + fr.NEW_FORMATS + ffr.FLOAT_FORMATS
CODE = dict(fr.CODE, **ffr.CODE)
BPP = dict(fr.BPP, **ffr.BPP)
ALIGN = {f: 4 if f in ffr.FLOAT_FORMATS else 2 if f in ("l16", "la16", "rgb16", "rgba16") else 1 for f in ALL_FORMATS}


@pytest.fixture(scope="module")
def torch_mod():
    import torch
    assert torch.cuda.is_available()
    return torch


def vp(a):
    return a.ctypes.data_as(C.c_void_p)


def one_call(pkg, det, img, kind):
    """(rc, record bytes, count, status-free) of the one-frame call on img."""
    img = np.asarray(img)
    fmt, w, h, st = pkg.image_format(img)
    n = C.c_int(0)
    if kind == "tags":
        out = np.zeros(1024, pkg.TAG_DTYPE)
        rc = pkg.lib().ag_detect(det._h, vp(img), w, h, st, fmt, vp(out), 1024, C.byref(n))
    else:
        out = np.zeros(16384, pkg.SADDLE_DTYPE)
        rc = pkg.lib().ag_refined_saddle_points(det._h, vp(img), w, h, st, fmt, vp(out), 16384, C.byref(n))
    return rc, out[:min(n.value, len(out))].tobytes(), n.value


def host_list(pkg, det, imgs, cap, kind, lib_fn=None):
    """The host list call into canary-filled outputs: (rc, words, counts, status)."""
    descs, _keep = pkg.frame_list(imgs)
    n, m = len(imgs), max(len(imgs), 1)
    words = np.full((m, cap * WORDS[kind]), CANARY, np.uint32)
    cnt = np.full(m, -7, np.int32)
    st = np.full(m, CANARY, np.uint32)
    fn = lib_fn or (pkg.lib().ag_detect_frames if kind == "tags" else pkg.lib().ag_refined_saddle_points_frames)
    rc = fn(det._h, descs, n, vp(words), cap, vp(cnt), vp(st))
    return rc, words, cnt, st


def to_device(torch, img):
    a = np.ascontiguousarray(img)
    return torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda()


def tensor_desc(pkg, t, img):
    fmt, w, h, _ = pkg.image_format(np.asarray(img))
    return (t.data_ptr(), w, h, fmt, t.stride(0) * t.element_size())


class DeviceOut:
    """Canary-filled device outputs of one device list call."""

    def __init__(self, torch, n, cap, kind):
        m = max(n, 1)
        self.torch, self.cap, self.kind = torch, cap, kind
        self.out = torch.full((m, cap * WORDS[kind]), CANARY - (1 << 32), dtype=torch.int32, device="cuda")
        self.cnt = torch.full((m,), -7, dtype=torch.int32, device="cuda")
        self.st = torch.full((m,), CANARY - (1 << 32), dtype=torch.int32, device="cuda")

    def call(self, pkg, det, descs, stream=None, status=True):
        fn = pkg.lib().ag_detect_frames_device if self.kind == "tags" else pkg.lib().ag_refined_saddle_points_frames_device
        s = stream if stream is not None else self.torch.cuda.current_stream()
        return fn(det._h, pkg.device_frame_list(descs), len(descs), C.c_void_p(self.out.data_ptr()), self.cap,
                  C.c_void_p(self.cnt.data_ptr()), C.c_void_p(self.st.data_ptr()) if status else None,
                  C.c_void_p(s.cuda_stream))

    def host(self):
        self.torch.cuda.synchronize()
        return (self.out.cpu().numpy().view(np.uint32), self.cnt.cpu().numpy(), self.st.cpu().numpy().view(np.uint32))


def device_list(pkg, det, torch, descs, cap, kind, stream=None):
    o = DeviceOut(torch, len(descs), cap, kind)
    rc = o.call(pkg, det, descs, stream)
    return (rc,) + o.host()


def assert_untouched_past(words, cnt, cap, kind):
    k = WORDS[kind]
    for i, c in enumerate(cnt):
        assert (words[i, k * min(max(int(c), 0), cap):] == CANARY).all(), ("written past the records", i)


def assert_list(pkg, res, singles, cap, kind, rc=None):
    """res of a list call whose frames are all clean at the call's capacities: frame i is singles[i]."""
    got_rc, words, cnt, st = res
    assert got_rc == (pkg.AG_OK if rc is None else rc), got_rc
    for i, (_, rec, n) in enumerate(singles):
        assert cnt[i] == n, (i, cnt[i], n)
        m = min(n, cap)
        assert words[i, :WORDS[kind] * m].tobytes() == rec[:WORDS[kind] * 4 * m], i
        assert st[i] == (TAG_OVERFLOW if n > cap else 0), (i, st[i])
    assert_untouched_past(words[:len(singles)], cnt[:len(singles)], cap, kind)


def tags_of(pkg, words, i, n):
    return {int(t["id"]): t["xy"].reshape(4, 2) for t in words[i, :9 * n].view(pkg.TAG_DTYPE)}


# ---- 1. the reference fixtures in one list ------------------------------------------------------------------
def test_reference_fixtures(pkg, images, expected, torch_mod):
    rng = np.random.default_rng(1)
    names = list(FIXTURE_NAMES) + ["EuRoC", "iphone", "top", "two_boards"]
    names = [names[i] for i in rng.permutation(len(names))]
    imgs = [images[n] for n in names]
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for kind in ("tags", "saddles"):
            cap = 1024 if kind == "tags" else 16384
            singles = [one_call(pkg, det, im, kind) for im in imgs]
            res = host_list(pkg, det, imgs, cap, kind)
            assert_list(pkg, res, singles, cap, kind)
            if kind == "tags":
                for i, name in enumerate(names):
                    want = expected[name]["oracle"]
                    got = tags_of(pkg, res[1], i, res[2][i])
                    assert sorted(got) == sorted(want["ids"]), name
                    assert_tags_match(got, {int(k): np.array(v, np.float32) for k, v in want["corners"].items()})
            ts = [to_device(torch_mod, im) for im in imgs]
            descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
            assert_list(pkg, device_list(pkg, det, torch_mod, descs, cap, kind), singles, cap, kind)
        # the Python wrappers
        got = det.detect_frames(imgs, cap_per_frame=1024)
        assert [sorted(g) for g in got] == [sorted(det.detect(im)) for im in imgs]
        sad = det.refined_saddle_points_frames(imgs, cap_per_frame=16384)
        assert all(s.tobytes() == det.refined_saddle_points(im).tobytes() for s, im in zip(sad, imgs))
    finally:
        det.close()


# ---- 2. all ten formats, strides and addresses ---------------------------------------------------------------
@pytest.fixture(scope="module")
def boards():
    return (synth.render_board_numpy(640, 480, seed=43, tag_px=44.0),
            synth.render_board_numpy(641, 481, seed=44, tag_px=40.0))


def padded(img, pad, offset=0):
    """img (H x W[ x C]) copied into rows of pad extra bytes, starting `offset` bytes into its buffer."""
    img = np.ascontiguousarray(img)
    h, row = img.shape[0], img.strides[0]
    buf = np.zeros(offset + h * (row + pad), np.uint8)
    rows = buf[offset:].reshape(h, row + pad)[:, :row]
    rows[...] = img.view(np.uint8).reshape(h, row)
    return rows.view(img.dtype).reshape(img.shape) if img.ndim == 2 else \
        rows.view(img.dtype).reshape(h, img.shape[1], img.shape[2])


def format_list(boards):
    b640, b641 = boards
    imgs = []
    for k, fmt in enumerate(ALL_FORMATS):
        a = format_frame(b640, fmt, 2 * k)
        b = format_frame(b641, fmt, 2 * k + 1)
        off = 1 if ALIGN[fmt] == 1 else 0  # host frames of the 8-bit formats at odd addresses
        imgs += [padded(a, 64, off), padded(b, 4 * (k + 1), off), a]
    rng = np.random.default_rng(2)
    return [imgs[i] for i in rng.permutation(len(imgs))]


def test_every_format_interleaved(pkg, torch_mod, boards):
    torch = torch_mod
    imgs = format_list(boards)
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for kind in ("tags", "saddles"):
            cap = 256 if kind == "tags" else 4096
            singles = [one_call(pkg, det, im, kind) for im in imgs]
            assert all(rc == pkg.AG_OK for rc, _, _ in singles)
            assert sum(n > 0 for _, _, n in singles) > len(imgs) // 2
            assert_list(pkg, host_list(pkg, det, imgs, cap, kind), singles, cap, kind)
            # device: every frame in one buffer, at offsets of its channel word; every other frame of a
            # format off the 16-byte grid, so that chunks mixing them must take the tile K1
            sizes = [im.strides[0] * im.shape[0] for im in imgs]
            buf = torch.zeros(sum(sizes) + 64 * len(imgs), dtype=torch.uint8, device="cuda")
            descs, pos = [], 0
            for i, im in enumerate(imgs):
                fmt, w, h, rs = pkg.image_format(im)
                al = CODE_ALIGN.get(fmt, 1)
                pos = (pos + 15) // 16 * 16 + (al * (1 + 2 * (i % 2)) if i % 3 else 0)
                row = w * BPP_OF[fmt]
                rows = np.zeros((h, rs), np.uint8)
                rows[:, :row] = np.ascontiguousarray(im).view(np.uint8).reshape(h, row)
                buf[pos:pos + h * rs].copy_(torch.from_numpy(rows.reshape(-1)))
                descs.append((buf.data_ptr() + pos, w, h, fmt, rs))
                pos += h * rs
            assert_list(pkg, device_list(pkg, det, torch, descs, cap, kind), singles, cap, kind)
    finally:
        det.close()


CODE_ALIGN = {CODE[f]: ALIGN[f] for f in ALL_FORMATS}
BPP_OF = {CODE[f]: BPP[f] for f in ALL_FORMATS}


# ---- 3. chunk and ring edges ---------------------------------------------------------------------------------
def grouped_list(boards, repeat):
    """Groups of 1, 2, 3, 4 and 7 frames of five geometries, interleaved round-robin, `repeat` times over."""
    b640 = boards[0]
    shapes = [lambda b: b, lambda b: np.ascontiguousarray(b[:470, :630]), lambda b: format_frame(b, "rgb8", 3),
              lambda b: format_frame(b, "l16", 4), lambda b: np.ascontiguousarray(b[8:, 16:])]
    variants = [lambda b: b, lambda b: b[::-1].copy(), lambda b: b[:, ::-1].copy(), lambda b: np.roll(b, 37, 1),
                lambda b: np.roll(b, 11, 0), lambda b: b[::-1, ::-1].copy(), lambda b: np.roll(b, -53, 1)]
    groups = [[shapes[g](variants[v](b640)) for v in range(size)] for g, size in enumerate((1, 2, 3, 4, 7))]
    out = []
    for _ in range(repeat):
        for k in range(7):
            out += [grp[k] for grp in groups if k < len(grp)]
    return out


def test_chunk_and_ring_edges(pkg, torch_mod, boards):
    imgs = grouped_list(boards, 3)  # 51 frames; chunks of three: 17 chunks, two turns of the board slots
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("chunk_frames", 3)
        det.set_option("host_chunk_frames", 3)
        for kind in ("tags", "saddles"):
            cap = 128 if kind == "tags" else 2048
            singles = [one_call(pkg, det, im, kind) for im in imgs]
            assert_list(pkg, host_list(pkg, det, imgs, cap, kind), singles, cap, kind)
            ts = [to_device(torch_mod, im) for im in imgs]
            descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
            for _ in range(2):  # the slots and the ring start where the last call left them
                assert_list(pkg, device_list(pkg, det, torch_mod, descs, cap, kind), singles, cap, kind)
    finally:
        det.close()


def test_device_chunks_mixing_aligned_and_misaligned_frames(pkg, torch_mod, boards):
    """Groups of one geometry and row stride in one device buffer: the first frame of a group on the
    16-byte grid, later ones off it by a multiple of the channel word (so off the alignment the streaming
    K1's vector loads need), and one group aligned throughout.  In chunks of the whole group and of two
    frames, every frame must equal the one-frame call: a chunk takes the streaming K1 only when all of its
    addresses allow it."""
    torch = torch_mod
    b = boards[0]
    variants = [b, b[::-1, ::-1].copy(), np.roll(b, 37, 1), np.roll(b, 11, 0)]
    # (format, offset of frame k from a 16-byte boundary)
    specs = [("l8", (0, 17, 32, 49)), ("rgba32f", (0, 4, 16, 36)), ("l16", (0, 2, 16, 18)), ("rgb8", (0, 1, 16, 35)),
             ("la8", (0, 16, 32, 48))]
    imgs, offs = [], []
    for k in range(4):
        for fmt, o in specs:
            imgs.append(format_frame(variants[k], fmt, k))
            offs.append(o[k])
    buf = torch.zeros(sum(im.nbytes for im in imgs) + 64 * len(imgs), dtype=torch.uint8, device="cuda")
    assert buf.data_ptr() % 16 == 0
    descs, pos = [], 0
    for im, o in zip(imgs, offs):
        pos = (pos + 15) // 16 * 16 + o
        raw = np.ascontiguousarray(im).view(np.uint8).reshape(-1)
        buf[pos:pos + raw.size].copy_(torch.from_numpy(raw))
        fmt, w, h, rs = pkg.image_format(im)
        descs.append((buf.data_ptr() + pos, w, h, fmt, rs))
        pos += raw.size
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for kind in ("tags", "saddles"):
            cap = 256 if kind == "tags" else 4096
            singles = [one_call(pkg, det, im, kind) for im in imgs]
            assert sum(n > 0 for _, _, n in singles) > len(imgs) // 2
            for chunk in (1024, 2):
                det.set_option("chunk_frames", chunk)
                assert_list(pkg, device_list(pkg, det, torch, descs, cap, kind), singles, cap, kind)
    finally:
        det.close()


def test_host_lists_from_pinned_and_pageable_frames(pkg, boards):
    """Host frames in pinned memory (uploaded directly) and in pageable memory (through the slot's pinned
    staging), mixed within one group's chunks, a group all pinned and one all pageable."""
    b640, b641 = boards
    pinned = []

    def pin(img):
        p = pkg.pinned_empty(img.shape, img.dtype)
        p[...] = img
        pinned.append(p)
        return p

    mixed = [pin(b640), np.roll(b640, 29, 1), pin(b640[::-1, ::-1].copy()), np.roll(b640, -31, 0), pin(np.roll(b640, 5, 1))]
    all_pinned = [pin(b641), pin(np.roll(b641, 40, 1))]
    pageable = [format_frame(b640, "rgb8", 1), format_frame(np.roll(b640, 13, 1), "rgb8", 2)]
    imgs = [mixed[0], all_pinned[0], pageable[0], mixed[1], mixed[2], all_pinned[1], mixed[3], pageable[1], mixed[4]]
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for kind in ("tags", "saddles"):
            cap = 128 if kind == "tags" else 2048
            singles = [one_call(pkg, det, im, kind) for im in imgs]
            for chunk in (128, 2):
                det.set_option("host_chunk_frames", chunk)
                assert_list(pkg, host_list(pkg, det, imgs, cap, kind), singles, cap, kind)
    finally:
        det.close()
        for p in pinned:
            pkg.pinned_free(p)


# ---- 4. streams, asynchronous calls, outputs -----------------------------------------------------------------
def test_device_streams_and_async_calls(pkg, torch_mod, boards):
    torch = torch_mod
    imgs = grouped_list(boards, 1)
    stack = np.stack([boards[0]] * 3 + [boards[0][::-1].copy()] * 3)
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        det.set_option("chunk_frames", 2)
        singles = [one_call(pkg, det, im, "tags") for im in imgs]
        ssingles = [one_call(pkg, det, im, "saddles") for im in imgs]
        bsingles = [one_call(pkg, det, im, "tags") for im in stack]
        ts = [to_device(torch, im) for im in imgs]
        descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            assert_list(pkg, device_list(pkg, det, torch, descs, 64, "tags", stream=side), singles, 64, "tags")
        assert_list(pkg, device_list(pkg, det, torch, descs, 64, "tags"), singles, 64, "tags")
        # device_async: list, batch, list (saddles), then one wait
        det.set_option("device_async", 1)
        d_stack = torch.from_numpy(stack).cuda()
        a = DeviceOut(torch, len(imgs), 64, "tags")
        c = DeviceOut(torch, len(imgs), 1024, "saddles")
        b_out = torch.full((len(stack), 64 * 9), CANARY - (1 << 32), dtype=torch.int32, device="cuda")
        b_cnt = torch.full((len(stack),), -7, dtype=torch.int32, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        torch.cuda.synchronize()
        assert a.call(pkg, det, descs) == pkg.AG_OK
        assert pkg.lib().ag_detect_batch_device(det._h, C.c_void_p(d_stack.data_ptr()), 0, len(stack), 640, 480, 0,
                                                pkg.FMT_L8, C.c_void_p(b_out.data_ptr()), 64,
                                                C.c_void_p(b_cnt.data_ptr()), None, C.c_void_p(s)) == pkg.AG_OK
        assert c.call(pkg, det, descs, status=False) == pkg.AG_OK
        det.detect_batch_device_wait(s)
        assert_list(pkg, (pkg.AG_OK,) + a.host(), singles, 64, "tags")
        words, cnt, st = c.host()
        assert_list(pkg, (pkg.AG_OK, words, cnt, np.zeros_like(st)), ssingles, 1024, "saddles")
        assert (st[:len(imgs)] == CANARY).all()  # no status array given: none written
        bw, bc = b_out.cpu().numpy().view(np.uint32), b_cnt.cpu().numpy()
        assert_list(pkg, (pkg.AG_OK, bw, bc, np.zeros(len(stack), np.uint32)), bsingles, 64, "tags")
        det.set_option("device_async", 0)
    finally:
        det.close()


# ---- 5. capacities -------------------------------------------------------------------------------------------
def test_capacity_overflows(pkg, torch_mod, boards):
    torch = torch_mod
    rng = np.random.default_rng(5)
    noise = rng.integers(0, 256, (1024, 1280), dtype=np.uint8)
    big = synth.render_board_numpy(1280, 1024, seed=5)
    imgs = [boards[0], noise, big, boards[1], format_frame(boards[0], "rgb8", 9)]
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for kind in ("tags", "saddles"):
            cap = 1024 if kind == "tags" else 16384
            singles = [one_call(pkg, det, im, kind) for im in imgs]
            assert all(rc == pkg.AG_OK for rc, _, _ in singles)
            # host: the noise frame overflows the call's capacities and is re-run alone
            assert_list(pkg, host_list(pkg, det, imgs, cap, kind), singles, cap, kind)
            # device: n = 0 and its bits, neighbours exact
            ts = [to_device(torch, im) for im in imgs]
            descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
            rc, words, cnt, st = device_list(pkg, det, torch, descs, cap, kind)
            assert rc == pkg.AG_OK
            assert cnt[1] == 0 and st[1] & GROWABLE and not int(st[1]) & ~(GROWABLE | BOARD_OVERFLOW), st[1]
            keep = [i for i in range(len(imgs)) if i != 1]
            assert_list(pkg, (rc, words[keep], cnt[keep], st[keep]), [singles[i] for i in keep], cap, kind)
            assert_untouched_past(words, cnt, cap, kind)
            # cap_per_frame below the counts: exact counts, TAG_OVERFLOW, AG_ERR_CAPACITY on the host call
            small = 5
            clean = [boards[0], big, boards[1]]
            sc = [one_call(pkg, det, im, kind) for im in clean]
            assert all(n > small for _, _, n in sc)
            assert_list(pkg, host_list(pkg, det, clean, small, kind), sc, small, kind, rc=pkg.AG_ERR_CAPACITY)
            ts = [to_device(torch, im) for im in clean]
            descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, clean)]
            assert_list(pkg, device_list(pkg, det, torch, descs, small, kind), sc, small, kind)
        # a board wider than a 16 x 16 lattice: BOARD_OVERFLOW and AG_ERR_CAPACITY
        det.set_option("board_lattice", 16)
        strips = [synth.render_board_numpy(1280, 1024, cols=c, rows=r, seed=c, tag_px=60.0) for c, r in STRIPS[-3:]]
        imgs = [boards[0]] + strips + [big]
        singles = [one_call(pkg, det, im, "tags") for im in imgs]
        flagged = [i for i, (rc, _, _) in enumerate(singles) if rc == pkg.AG_ERR_CAPACITY]
        assert flagged and singles[0][0] == pkg.AG_OK
        rc, words, cnt, st = host_list(pkg, det, imgs, 1024, "tags")
        assert rc == pkg.AG_ERR_CAPACITY
        ts = [to_device(torch, im) for im in imgs]
        descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
        drc, dwords, dcnt, dst = device_list(pkg, det, torch, descs, 1024, "tags")
        assert drc == pkg.AG_OK
        for i, (_, rec, n) in enumerate(singles):
            assert st[i] == dst[i] == (BOARD_OVERFLOW if i in flagged else 0), (i, st[i], dst[i])
            assert cnt[i] == dcnt[i] == n
            assert words[i, :9 * n].tobytes() == dwords[i, :9 * n].tobytes() == rec
    finally:
        det.close()


# ---- 6. invalid lists ----------------------------------------------------------------------------------------
def test_invalid_lists(pkg, torch_mod, boards):
    torch = torch_mod
    L = pkg.lib()
    imgs = [boards[0], boards[1]] * 10
    ts = [to_device(torch, im) for im in imgs]
    good = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
    d16 = torch.zeros(480 * 640 + 8, dtype=torch.int16, device="cuda")
    d32 = torch.zeros(480 * 640 * 3 + 8, dtype=torch.float32, device="cuda")
    host_bad = [(None, 640, 480, pkg.FMT_L8, 0), (1, 640, 480, 3, 0), (1, 0, 480, pkg.FMT_L8, 0),
                (1, 640, 480, pkg.FMT_L8, 639), (1, 640, 480, pkg.FMT_L16, 1281)]
    dev_bad = host_bad[:4] + [(d16.data_ptr() + 1, 640, 480, pkg.FMT_L16, 0),
                              (d32.data_ptr() + 2, 640, 480, pkg.FMT_RGB32F, 0)]
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    keep = [np.ascontiguousarray(im) for im in imgs]
    try:
        for kind in ("tags", "saddles"):
            hfn = L.ag_detect_frames if kind == "tags" else L.ag_refined_saddle_points_frames
            base = [(im.ctypes.data, im.shape[1], im.shape[0], pkg.FMT_L8, 0) for im in keep]

            def host_call(descs, n=None, cap=8, arr=True):
                a = pkg.device_frame_list(descs)  # (host addresses here: only the layout matters)
                m = max(len(descs), 1)
                words = np.full((m, 8 * WORDS[kind]), CANARY, np.uint32)
                cnt = np.full(m, -7, np.int32)
                st = np.full(m, CANARY, np.uint32)
                before = det.launch_count
                rc = hfn(det._h, a if arr else None, len(descs) if n is None else n, vp(words), cap, vp(cnt), vp(st))
                assert det.launch_count == before
                assert (words == CANARY).all() and (cnt == -7).all() and (st == CANARY).all()
                return rc

            for bad in host_bad:
                bad = tuple(keep[0].ctypes.data if v == 1 and k == 0 else v for k, v in enumerate(bad))
                assert host_call(base + [bad]) == pkg.AG_ERR_INVALID, bad
            assert host_call(base, cap=0) == pkg.AG_ERR_INVALID
            assert host_call(base, n=-1) == pkg.AG_ERR_INVALID
            assert host_call(base, arr=False) == pkg.AG_ERR_INVALID
            assert host_call(base, n=0) == pkg.AG_OK

            for bad in dev_bad:
                bad = tuple(ts[0].data_ptr() if v == 1 and k == 0 else v for k, v in enumerate(bad))
                o = DeviceOut(torch, len(good) + 1, 8, kind)
                before = det.launch_count
                assert o.call(pkg, det, good + [bad]) == pkg.AG_ERR_INVALID, bad
                assert det.launch_count == before
                words, cnt, st = o.host()
                assert (words == CANARY).all() and (cnt == -7).all() and (st == CANARY).all()
            o = DeviceOut(torch, len(good), 8, kind)
            dfn = L.ag_detect_frames_device if kind == "tags" else L.ag_refined_saddle_points_frames_device
            arr = pkg.device_frame_list(good)
            args = (C.c_void_p(o.out.data_ptr()),)
            for a, n, cap in ((arr, len(good), 0), (arr, -1, 8), (None, len(good), 8)):
                assert dfn(det._h, a, n, args[0], cap, C.c_void_p(o.cnt.data_ptr()), None, None) == pkg.AG_ERR_INVALID
            assert dfn(det._h, arr, 0, args[0], 8, C.c_void_p(o.cnt.data_ptr()), None, None) == pkg.AG_OK
            words, cnt, st = o.host()
            assert (words == CANARY).all() and (cnt == -7).all()
    finally:
        det.close()


# ---- 7. uniform lists and the other calls --------------------------------------------------------------------
def test_uniform_lists_equal_the_batch_calls(pkg, torch_mod):
    torch = torch_mod
    frames = synth.fixture_like_frames(4, 1280, 1024, seed=90)
    frames = np.concatenate([frames, frames[:, ::-1], frames[:, :, ::-1]])
    imgs = [np.ascontiguousarray(f) for f in frames]  # separately allocated
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        n = len(frames)
        ref = (np.zeros((n, 64), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.ones(n, np.uint32))
        det.detect_batch_into(frames, *ref)
        batch = [(pkg.AG_OK, ref[0][i, :ref[1][i]].tobytes(), int(ref[1][i])) for i in range(n)]
        assert not ref[2].any()
        assert_list(pkg, host_list(pkg, det, imgs, 64, "tags"), batch, 64, "tags")
        d = torch.from_numpy(frames).cuda()
        ts = [to_device(torch, im) for im in imgs]
        descs = [tensor_desc(pkg, t, im) for t, im in zip(ts, imgs)]
        dres = device_list(pkg, det, torch, descs, 64, "tags")
        b = DeviceOut(torch, n, 64, "tags")
        assert pkg.lib().ag_detect_batch_device(det._h, C.c_void_p(d.data_ptr()), 0, n, 1280, 1024, 0, pkg.FMT_L8,
                                                C.c_void_p(b.out.data_ptr()), 64, C.c_void_p(b.cnt.data_ptr()),
                                                C.c_void_p(b.st.data_ptr()), None) == pkg.AG_OK
        bw, bc, bs = b.host()
        assert dres[0] == pkg.AG_OK and np.array_equal(dres[1], bw) and np.array_equal(dres[2], bc)
        assert np.array_equal(dres[3], bs) and np.array_equal(bc, ref[1])
        # host_async batch calls in flight around a list call on the same handle
        det.set_option("host_async", 1)
        got = [(np.zeros((n, 64), pkg.TAG_DTYPE), np.zeros(n, np.int32), np.ones(n, np.uint32)) for _ in range(2)]
        det.detect_batch_into(frames, *got[0])
        res2 = host_list(pkg, det, imgs[::-1], 64, "tags")
        det.detect_batch_into(frames, *got[1])
        sres = host_list(pkg, det, imgs, 2048, "saddles")
        det.detect_batch_wait(0)
        det.set_option("host_async", 0)
        for g in got:
            assert g[0].tobytes() == ref[0].tobytes() and np.array_equal(g[1], ref[1])
        assert_list(pkg, res2, batch[::-1], 64, "tags")
        assert_list(pkg, sres, [one_call(pkg, det, im, "saddles") for im in imgs], 2048, "saddles")
    finally:
        det.close()


# ---- 8. several devices --------------------------------------------------------------------------------------
def test_multi_device_equals_one_device(pkg, torch_mod, boards):
    imgs = grouped_list(boards, 2) + format_list(boards)[:10]
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        want = {k: host_list(pkg, det, imgs, 128 if k == "tags" else 2048, k) for k in WORDS}
    finally:
        det.close()
    sets = [[0, 0]] + ([None] if torch_mod.cuda.device_count() >= 2 else [])
    for devs in sets:
        m = pkg.MultiTagDetector(pkg.TagFamily.T36H11, devices=devs)
        try:
            m.set_option("host_chunk_frames", 4)
            for kind, fn in (("tags", pkg.lib().ag_multi_detect_frames),
                             ("saddles", pkg.lib().ag_multi_refined_saddle_points_frames)):
                got = host_list(pkg, m, imgs, 128 if kind == "tags" else 2048, kind, lib_fn=fn)
                assert got[0] == want[kind][0] == pkg.AG_OK
                for a, b in zip(got[1:], want[kind][1:]):
                    assert np.array_equal(a, b)
            res = m.detect_frames(imgs[:5])
            assert len(res) == 5
        finally:
            m.close()


# ---- 9. the C++ mirror ---------------------------------------------------------------------------------------
def test_cpp_mirror_frames(pkg, oracle, tmp_path):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / "cpp_frames_demo")
    libdir = os.path.join(root, "aprilgrid-rs_b200", "lib")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "aprilgrid-rs_b200", "cpp"), "-o", exe,
                           os.path.join(root, "tests", "cpp_frames_demo.cpp"), "-L" + libdir, "-laprilgrid_b200",
                           "-Wl,-rpath," + libdir])
    a = synth.render_board_numpy(640, 480, seed=12, tag_px=44.0)
    b = synth.render_board_numpy(800, 600, seed=13, tag_px=50.0)
    args = []
    a180 = np.ascontiguousarray(a[::-1, ::-1])
    for k, (img, fmt) in enumerate(((a, 0), (np.repeat(b[:, :, None], 3, axis=2), 2), (a180, 0))):
        p = tmp_path / ("f%d.raw" % k)
        p.write_bytes(np.ascontiguousarray(img).tobytes())
        args += [str(p), str(img.shape[1]), str(img.shape[0]), str(fmt)]
    out = subprocess.check_output([exe] + args, text=True).strip().splitlines()
    assert out[-1] == "frames same"
    got, cur = {}, None
    for ln in out[:-1]:
        f = ln.split()
        if f[0] == "frame":
            cur = int(f[1])
            got[cur] = {}
        else:
            got[cur][int(f[0])] = np.array([float(v) for v in f[1:]], np.float32).reshape(4, 2)
    for k, img in enumerate((a, b, a180)):  # R = G = B: the luma of the RGB frame is b
        want = oracle.detect(img)
        assert len(want) > 0
        assert_tags_match(got[k], want)
