"""The product's board-assembly / decode control logic (csrc/ag_board_core.h), compiled for the
host with a one-lane warp (tests/host_board_test.cpp, test-only), against the oracle.
Input to both: the oracle's refined saddle list, so only the board/decode logic is compared."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import synth
from conftest import FIXTURE_NAMES, ROOT

HOSTLIB = os.path.join(ROOT, "aprilgrid-rs_b200", "lib", "libag_board_hosttest.so")


@pytest.fixture(scope="module")
def hb():
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "aprilgrid-rs_b200"),
                           "lib/libag_board_hosttest.so"])
    return C.CDLL(HOSTLIB)


def host_detect(hb, pkg, oracle, img, saddles=None, family=None, max_boards=2, max_saddles=2048,
                use_grid=1, lattice=64, smem_saddles=512):
    family = pkg.TagFamily.T36H11 if family is None else family  # T16H5 is 0
    fam = pkg.family_info(family)
    if saddles is None:
        saddles = oracle.front_end(img, want_labels=False)["refined"]
    s = np.ascontiguousarray(saddles, np.float32)
    fmt, w, h, st = oracle.image_format(img)
    out = np.zeros(1024, pkg.TAG_DTYPE)
    quads = np.zeros((1024, 4), np.int32)
    tapn, status = C.c_int(0), C.c_uint32(0)
    codes = fam["codes"]
    vp = C.c_void_p
    n = hb.hb_detect_from_saddles(
        s.ctypes.data_as(vp), len(s), img.ctypes.data_as(vp), w, h, C.c_size_t(st), fmt,
        codes.ctypes.data_as(vp), len(codes), fam["edge"], fam["border"], fam["hamming"], max_boards,
        max_saddles, out.ctypes.data_as(vp), 1024, quads.ctypes.data_as(vp), C.byref(tapn), 1024,
        C.byref(status), use_grid, lattice, smem_saddles)
    assert n >= 0
    return ({int(t["id"]): t["xy"].reshape(4, 2).copy() for t in out[:n]}, quads[:tapn.value],
            status.value, s)


@pytest.mark.parametrize("name", FIXTURE_NAMES)
def test_fixtures_identical_to_oracle(hb, pkg, oracle, images, name):
    img = images[name]
    got, quads, status, s = host_detect(hb, pkg, oracle, img)
    want = oracle.detect(img)
    assert status == 0
    assert sorted(got) == sorted(want)
    for k in want:
        assert np.array_equal(got[k], want[k])
    oq = oracle.try_find_best_board(s)
    assert oq is not None and np.array_equal(oq, quads)


@pytest.mark.parametrize("seed", range(6))
def test_synthetic_boards_identical_to_oracle(hb, pkg, oracle, seed):
    img = synth.render_board_numpy(640, 480, seed=seed, tag_px=40.0 + 2 * seed)
    got, quads, status, s = host_detect(hb, pkg, oracle, img)
    want = oracle.detect(img)
    assert sorted(got) == sorted(want) and len(want) == 36
    for k in want:
        assert np.array_equal(got[k], want[k])


def test_bucket_grid_and_exhaustive_search_agree(hb, pkg, oracle, images):
    """The radius queries go through a bucket grid on the device; same answers as the full scan."""
    for name in ("EuRoC", "two_boards"):
        img = images[name]
        a = host_detect(hb, pkg, oracle, img, use_grid=1)
        b = host_detect(hb, pkg, oracle, img, use_grid=0)
        assert sorted(a[0]) == sorted(b[0]) and np.array_equal(a[1], b[1])
        for k in a[0]:
            assert np.array_equal(a[0][k], b[0][k])


def test_more_saddles_than_the_on_chip_grid_holds(hb, pkg, oracle):
    """> 512 saddles with the 512 tier: the bucket grid's items live in the frame's workspace, as on
    the device; result unchanged."""
    img = synth.render_board_numpy(1600, 1200, cols=12, rows=9, seed=4, tag_px=70.0)
    fe = oracle.front_end(img, want_labels=False)
    assert len(fe["refined"]) > 512
    got, quads, status, s = host_detect(hb, pkg, oracle, img, saddles=fe["refined"])
    want = oracle.detect(img)
    assert sorted(got) == sorted(want) and len(want) >= 100
    for k in want:
        assert np.array_equal(got[k], want[k])


@pytest.mark.parametrize("key", ["1408x1024", "1409x1024"])
def test_bucket_grid_edge_lists_identical_to_oracle(hb, pkg, oracle, key):
    """The exact-size saddle lists of the GPU suite's bucket-grid edge (1408 x 1024: 32 px buckets,
    1409 x 1024: 64 px) through the general path as each launch of the 512 tier runs it (320 and 512
    saddles on chip; a list beyond them keeps its grid items in the frame's workspace), and with the
    exhaustive scan."""
    from test_gpu_board_edges import CANVASES, canvas, exact_case
    img = canvas(key, oracle)
    for n in CANVASES[key][3]:
        s, want_q, want_t = exact_case(key, n, oracle)
        for smem, use_grid in ((320, 1), (512, 1), (512, 0)):
            got, quads, status, _ = host_detect(hb, pkg, oracle, img, saddles=s, use_grid=use_grid,
                                                smem_saddles=smem)
            what = (key, n, smem, use_grid)
            assert status == 0 and want_q is not None and np.array_equal(quads, want_q), what
            assert sorted(got) == sorted(want_t) and len(want_t) >= 10, what
            for k in want_t:
                assert np.array_equal(got[k], want_t[k]), what


def test_small_lattice_same_result_and_overflow_flag(hb, pkg, oracle, images):
    """A 6x6 board fits a 32-wide lattice (same answer); a 16-wide one may overflow and says so."""
    img = images["EuRoC"]
    a = host_detect(hb, pkg, oracle, img, lattice=64)
    b = host_detect(hb, pkg, oracle, img, lattice=32)
    assert sorted(a[0]) == sorted(b[0]) and b[2] == 0
    c = host_detect(hb, pkg, oracle, img, lattice=16)
    assert c[2] in (0, 4)  # AG_FRAME_BOARD_OVERFLOW when the board leaves the -8..7 lattice
    if c[2] == 0:
        assert sorted(c[0]) == sorted(a[0])


def test_empty_and_degenerate_saddle_lists(hb, pkg, oracle):
    img = np.full((64, 64), 128, np.uint8)
    got, quads, status, _ = host_detect(hb, pkg, oracle, img, saddles=np.zeros((0, 5), np.float32))
    assert got == {} and len(quads) == 0
    # a handful of random saddles: no board, must terminate and agree with the oracle (None)
    rng = np.random.default_rng(0)
    s = np.stack([rng.uniform(5, 60, 12), rng.uniform(5, 60, 12), np.ones(12),
                  rng.uniform(-90, 90, 12), np.full(12, 45.0)], axis=1).astype(np.float32)
    got, quads, status, _ = host_detect(hb, pkg, oracle, img, saddles=s)
    oq = oracle.try_find_best_board(s)
    assert got == {}
    assert (oq is None and len(quads) == 0) or np.array_equal(oq, quads)


def test_one_board_limit(hb, pkg, oracle, images):
    """max_num_of_boards = 1 on the two-board image finds exactly one board's tags."""
    img = images["two_boards"]
    got, _, _, _ = host_detect(hb, pkg, oracle, img, max_boards=1)
    want = oracle.detect(img, max_boards=1)
    assert sorted(got) == sorted(want) and 0 < len(want) < 72


def test_gate_adversarial_saddle_sets(hb, pkg, oracle):
    """Saddle lists sitting on the discontinuous gates of the board search (theta differences of
    5 / 80 degrees +- ulps, theta at x.5, opposite-angle differences of 10 degrees +- 1e-4; some
    saddles outside the image): the product's board logic == the oracle, quads in the same order.
    (The GPU suite runs the same sets through the kernel.)"""
    img = synth.render_board_numpy(640, 480, seed=3, tag_px=44.0)
    base = oracle.front_end(img, want_labels=False)["refined"]
    rng = np.random.default_rng(2024)
    n_boards = 0
    for name, s in synth.adversarial_saddle_sets(base, rng):
        want = oracle.try_find_best_board(s)
        _, quads, _, _ = host_detect(hb, pkg, oracle, img, saddles=s)
        if want is None:
            assert len(quads) == 0, name
        else:
            assert np.array_equal(quads, want), name
            n_boards += 1
    assert n_boards >= 30
