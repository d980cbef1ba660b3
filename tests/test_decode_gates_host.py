"""Tag decoding at its gates: the host build of the board core (csrc/ag_board_core.h through
tests/host_board_test.cpp) against the oracle, on frames whose sample pixels were painted onto the
thresholds of bit_code / best_tag (detector.rs:74-169) -- see synth.decode_gate_frames.  Also the
size of the board kernel's decode scratch for every configuration the API can choose."""
import ctypes as C

import numpy as np
import pytest

import synth
from test_board_core_host import hb, host_detect  # noqa: F401  (hb is a fixture)

FAMILIES = list(synth.GATE_FAMILIES)
FORMATS = ["l8", "l16", "rgb8"]


# ---- decode scratch of the board kernel ------------------------------------------------------------
def test_decode_scratch_holds_every_listed_quad(pkg):
    """The bit patterns of a board's listed quads (8 bytes each, warp 0's seed-best values) must fit
    their region for every max_saddles the API can choose: the automatic 2048 / 4096 / 5120 / 13056,
    the 16384 of the regrowth path and every user value from 16 to 16384."""
    lib = pkg.lib()
    out = (C.c_longlong * 2)()
    values = sorted(set(range(16, 16385)) | {2048, 4096, 5120, 13056, 16384})
    short = []
    for lattice in (16, 32, 64):
        for warps in (1, 2, 4, 8, 16):
            for n in values:
                assert lib.ag_test_board_decode_room(n, lattice, warps, out) == 0
                room, listed = int(out[0]), int(out[1])
                assert listed == min(n // 4 + 2, lattice * lattice)
                if room < 8 * listed:
                    short.append((n, lattice, warps, room // 8, listed))
    assert not short, "%d configurations too small, e.g. (max_saddles, lattice, warps, room, listed) %s" % (
        len(short), short[:4])
    # the default 1280 x 1024 configuration keeps its workspace
    lay = (C.c_longlong * 4)()
    assert lib.ag_test_board_layout(2048, 64, 2, 320, 1, 320, lay) == 0
    assert lib.ag_test_board_decode_room(2048, 64, 2, out) == 0 and out[0] == 2 * 64 * 64


# ---- painted frames through the host build -----------------------------------------------------------
_FRAMES = {}


def frames_of(family):
    if family not in _FRAMES:
        _FRAMES[family] = synth.gate_frames(family)
    return _FRAMES[family]


def same_tags(got, want):
    assert sorted(got) == sorted(want), (sorted(got), sorted(want))
    for k in want:
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("family", FAMILIES)
def test_painted_frames_identical_to_oracle(hb, pkg, oracle, family, fmt):  # noqa: F811
    """Every scenario frame: the oracle decodes what the painting was built for (and the integer
    restatement of bit_code / best_tag agrees with it tag by tag); the oracle's detect equals its
    detect_from_saddles on the refined list; the host build of the board core equals both."""
    tf = pkg.TagFamily[family.upper()]
    n_tags = 0
    for name, scene, tags, f, frame, mbs in frames_of(family):
        if f != fmt:
            continue
        saddles = oracle.front_end(frame, want_labels=False)["refined"]
        grey = oracle.to_luma_u8(frame)
        for mb in mbs:
            want = oracle.detect(frame, family=family, max_boards=mb)
            n_tags += synth.check_expectations(scene, tags, want, grey)
            same_tags(oracle.detect_from_saddles(frame, saddles, family=family, max_boards=mb), want)
            got, quads, status, _ = host_detect(hb, pkg, oracle, frame, saddles=saddles, family=tf,
                                                max_boards=mb)
            assert status == 0, (name, mb)
            assert np.array_equal(quads, oracle.try_find_best_board(saddles)), name
            same_tags(got, want)
    assert n_tags == 20 + 20 + 3 * 20 + 48


@pytest.mark.parametrize("family", FAMILIES)
def test_translated_saddle_lists_identical_to_oracle(hb, pkg, oracle, family):  # noqa: F811
    """A sample point exactly on k + 0.5 (k even) and a quad corner at w - 0.5 / h - 0.5 and one ulp
    below, set up by translating the saddle list: the host build equals the oracle, and the oracle
    decodes what each case was built for."""
    tf = pkg.TagFamily[family.upper()]
    scene = synth.gate_scene(family)
    half = synth.half_sample_case(scene)
    assert half is not None, "no translation puts a sample on k + 0.5"
    s, img, tid, _ = half
    cases = [("half_sample", s, img, tid, True)] + synth.edge_corner_cases(scene)
    for name, s, img, tid, decodes in cases:
        for fmt in FORMATS:
            frame = synth.encode(img, {}, fmt, {})
            want = oracle.detect_from_saddles(frame, s, family=family)
            assert (tid in want) == decodes, (name, fmt)
            got, _, status, _ = host_detect(hb, pkg, oracle, frame, saddles=s, family=tf)
            assert status == 0
            same_tags(got, want)
