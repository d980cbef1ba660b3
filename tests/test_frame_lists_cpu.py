"""CPU-side checks of the frame-list entry points (ag_detect_frames, ag_refined_saddle_points_frames,
their _device and ag_multi_ forms): declared, exported, typed in the Python wrapper, used by the C++
mirror, ag_frame laid out as the ctypes structure says, refused without a handle, and the plan the
library runs a list by -- grouping, chunking and the multi-GPU split -- pinned through the test hook."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_cabi_cpu import declared_symbols

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FRAMES = ("ag_detect_frames", "ag_refined_saddle_points_frames", "ag_detect_frames_device",
          "ag_refined_saddle_points_frames_device", "ag_multi_detect_frames", "ag_multi_refined_saddle_points_frames")


def test_declared_and_exported(pkg):
    syms = declared_symbols()
    lib = C.CDLL(pkg.LIB_PATH)
    for s in FRAMES:
        assert s in syms
        assert hasattr(lib, s), "missing export: " + s


def test_wrapper_types_the_entry_points(pkg):
    L = pkg.lib()
    for s in FRAMES:
        assert len(getattr(L, s).argtypes) == (8 if s.endswith("_device") else 7), s
    for name in ("detect_frames", "refined_saddle_points_frames", "detect_frames_device",
                 "refined_saddle_points_frames_device"):
        assert callable(getattr(pkg.TagDetector, name))
    for name in ("detect_frames", "refined_saddle_points_frames"):
        assert callable(getattr(pkg.MultiTagDetector, name))


def test_cpp_mirror_uses_them(tmp_path):
    src = tmp_path / "use.cpp"
    src.write_text('#include "aprilgrid_b200.hpp"\n'
                   "using V = std::vector<aprilgrid::ImageView>;\n"
                   "std::vector<aprilgrid::TagMap> a(const aprilgrid::TagDetector& d, const V& v) {\n"
                   "  return d.detect_frames(v, 64);\n}\n"
                   "std::vector<std::vector<aprilgrid::Saddle>> b(const aprilgrid::TagDetector& d, const V& v) {\n"
                   "  return d.refined_saddle_points_frames(v);\n}\n"
                   "std::vector<aprilgrid::TagMap> c(const aprilgrid::MultiTagDetector& m, const V& v) {\n"
                   "  return m.detect_frames(v);\n}\n"
                   "std::vector<std::vector<aprilgrid::Saddle>> e(const aprilgrid::MultiTagDetector& m, const V& v) {\n"
                   "  return m.refined_saddle_points_frames(v, 512);\n}\n"
                   "int main() { return 0; }\n")
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(ROOT, "aprilgrid-rs_b200", "cpp"), str(src)])


def test_struct_layout_matches_ctypes(pkg, tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "aprilgrid_b200.h"\n'
                   "int main(void) { printf(\"%zu %zu %zu %zu %zu %zu\\n\", sizeof(ag_frame), offsetof(ag_frame, pixels),"
                   " offsetof(ag_frame, width), offsetof(ag_frame, height), offsetof(ag_frame, row_stride),"
                   " offsetof(ag_frame, format)); return 0; }\n")
    exe = str(tmp_path / "layout")
    subprocess.check_call(["gcc", "-std=c99", "-I", os.path.join(ROOT, "include"), "-o", exe, str(src)])
    got = [int(v) for v in subprocess.check_output([exe], text=True).split()]
    F = pkg.AgFrame
    want = [C.sizeof(F)] + [getattr(F, f).offset for f in ("pixels", "width", "height", "row_stride", "format")]
    assert got == want


def test_null_handle_is_invalid(pkg):
    L = pkg.lib()
    px = (C.c_uint8 * 64)()
    descs = (pkg.AgFrame * 1)(pkg.AgFrame(C.addressof(px), 8, 8, 0, pkg.FMT_L8))
    out = (C.c_float * 10)()
    n = (C.c_int * 1)(-5)
    st = (C.c_uint32 * 1)(77)
    assert L.ag_detect_frames(None, descs, 1, out, 1, n, st) == pkg.AG_ERR_INVALID
    assert L.ag_refined_saddle_points_frames(None, descs, 1, out, 1, n, st) == pkg.AG_ERR_INVALID
    assert L.ag_detect_frames_device(None, descs, 1, out, 1, n, st, None) == pkg.AG_ERR_INVALID
    assert L.ag_refined_saddle_points_frames_device(None, descs, 1, out, 1, n, st, None) == pkg.AG_ERR_INVALID
    assert L.ag_multi_detect_frames(None, descs, 1, out, 1, n, st) == pkg.AG_ERR_INVALID
    assert L.ag_multi_refined_saddle_points_frames(None, descs, 1, out, 1, n, st) == pkg.AG_ERR_INVALID
    assert n[0] == -5 and st[0] == 77 and all(v == 0.0 for v in out)


GEOMS = [(1280, 1024, 0, 0), (848, 480, 2, 0), (752, 480, 0, 768), (1024, 1024, 1, 0), (1920, 1080, 9, 0),
         (33, 17, 5, 0), (3840, 2160, 10, 0)]


def interleaved(n, seed):
    """n geometries drawn from GEOMS, interleaved; (752, 480, L8) also appears packed (row stride 0 and
    752 are the same group)."""
    rng = np.random.default_rng(seed)
    out = []
    for k in rng.integers(0, len(GEOMS) + 1, n):
        out.append(GEOMS[k] if k < len(GEOMS) else (752, 480, 0, 752))
    return out


def key(pkg, g):
    w, h, fmt, rs = g
    bpp = {0: 1, 1: 2, 2: 3, 5: 4, 9: 12, 10: 16}[fmt]
    return (w, h, fmt, rs or w * bpp)


@pytest.mark.parametrize("n", [0, 1, 7, 3000])
@pytest.mark.parametrize("host", [True, False])
def test_plan_groups_and_chunks(pkg, n, host):
    geoms = interleaved(n, n)
    cf, hcf = 5, 3
    order, chunk0, _ = pkg.frame_plan(geoms, chunk_frames=cf, host_chunk_frames=hcf, host=host)
    assert sorted(order.tolist()) == list(range(n))  # every index exactly once
    keys = [key(pkg, g) for g in geoms]
    # groups in order of first appearance, list order within a group
    first = {}
    for i, k in enumerate(keys):
        first.setdefault(k, i)
    want = sorted(range(n), key=lambda i: (first[keys[i]], i))
    assert order.tolist() == want
    assert chunk0[0] == 0 and chunk0[-1] == n and np.all(np.diff(chunk0) > 0)
    for a, b in zip(chunk0[:-1], chunk0[1:]):
        ks = {keys[i] for i in order[a:b]}
        assert len(ks) == 1  # one geometry per chunk
        w, h, fmt, _ = next(iter(ks))
        bpp = {0: 1, 1: 2, 2: 3, 5: 4, 9: 12, 10: 16}[fmt]
        lim = cf
        if host:
            lim = min(lim, max(1, hcf * 8 // bpp) if bpp > 8 else hcf)
        lim = max(1, min(lim, (24 << 30) // (w * h * 8)))
        assert b - a <= lim
    # a group is cut into full chunks but its last
    for a, b, c in zip(chunk0[:-2], chunk0[1:-1], chunk0[2:]):
        if keys[order[a]] == keys[order[b]]:
            assert b - a >= c - b


def test_plan_default_options_take_whole_groups(pkg):
    geoms = [(640, 480, 0, 0), (320, 240, 2, 0)] * 50
    order, chunk0, _ = pkg.frame_plan(geoms, host=False)
    assert chunk0.tolist() == [0, 50, 100]
    assert order[:50].tolist() == list(range(0, 100, 2))


def frame_bytes(g):
    w, h, fmt, rs = g
    bpp = {0: 1, 1: 2, 2: 3, 5: 4, 9: 12, 10: 16}[fmt]
    return (rs or w * bpp) * (h - 1) + w * bpp


@pytest.mark.parametrize("n", [0, 1, 7, 3000])
@pytest.mark.parametrize("G", [1, 2, 3, 8])
def test_multi_bounds_cover_the_list(pkg, n, G):
    geoms = interleaved(n, 7 * n + G)
    _, _, b = pkg.frame_plan(geoms, n_devices=G)
    assert b[0] == 0 and b[-1] == n and np.all(np.diff(b) >= 0)
    if n >= G * 20:  # byte shares within one frame of equal
        by = np.array([frame_bytes(g) for g in geoms], np.float64)
        total, biggest = by.sum(), by.max()
        for g in range(G):
            assert abs(by[b[g]:b[g + 1]].sum() - total / G) <= biggest


def test_multi_bounds_split_by_bytes(pkg):
    big, small = (3840, 2160, 0, 0), (384, 216, 0, 0)  # 100 x the pixels
    geoms = [big] + [small] * 100
    _, _, b = pkg.frame_plan(geoms, n_devices=2)
    assert b.tolist() == [0, 1, 101]  # not 50 / 51 frames
    geoms = [small] * 100 + [big] * 3
    _, _, b = pkg.frame_plan(geoms, n_devices=2)
    assert b.tolist() == [0, 101, 103]  # 200 : 200 small frames' bytes
    # measured rates that differ by more than 5 % weight the split
    geoms = [small] * 300
    _, _, b = pkg.frame_plan(geoms, n_devices=2, rates=[10.0, 20.0])
    assert b.tolist() == [0, 100, 300]
    _, _, b = pkg.frame_plan(geoms, n_devices=2, rates=[10.0, 10.2])
    assert b.tolist() == [0, 150, 300]


def test_plan_refuses_bad_descriptors(pkg):
    with pytest.raises(ValueError):
        pkg.frame_plan([(640, 480, 0, 0), (0, 480, 0, 0)])
    with pytest.raises(ValueError):
        pkg.frame_plan([(640, 480, 3, 0)])
    with pytest.raises(ValueError):
        pkg.frame_plan([(640, 480, 1, 641)])
