"""CPU-side checks of the saddle batch entry points (ag_refined_saddle_points_batch, _device and
ag_multi_refined_saddle_points_batch): declared, exported, typed in the Python wrapper, present in
the C++ mirror, and refused without a handle.  No compute calls are made here."""
import ctypes as C
import os
import subprocess

from test_cabi_cpu import declared_symbols

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SADDLE_BATCH = ("ag_refined_saddle_points_batch", "ag_refined_saddle_points_batch_device",
                "ag_multi_refined_saddle_points_batch")


def test_declared_and_exported(pkg):
    syms = declared_symbols()
    lib = C.CDLL(pkg.LIB_PATH)
    for s in SADDLE_BATCH:
        assert s in syms
        assert hasattr(lib, s), "missing export: " + s


def test_wrapper_types_the_entry_points(pkg):
    L = pkg.lib()
    assert len(L.ag_refined_saddle_points_batch.argtypes) == 12
    assert len(L.ag_refined_saddle_points_batch_device.argtypes) == 13
    assert len(L.ag_multi_refined_saddle_points_batch.argtypes) == 12
    for cls in (pkg.TagDetector, pkg.MultiTagDetector):
        assert callable(getattr(cls, "refined_saddle_points_batch"))
    assert callable(pkg.TagDetector.refined_saddle_points_batch_into)
    assert callable(pkg.TagDetector.refined_saddle_points_batch_device)


def test_cpp_mirror_uses_them(tmp_path):
    src = tmp_path / "use.cpp"
    src.write_text('#include "aprilgrid_b200.hpp"\n'
                   "std::vector<std::vector<aprilgrid::Saddle>> one(const aprilgrid::TagDetector& d, const void* f) {\n"
                   "  return d.refined_saddle_points_batch(f, 0, 2, 64, 48, 0, AG_L8);\n}\n"
                   "std::vector<std::vector<aprilgrid::Saddle>> many(const aprilgrid::MultiTagDetector& m, const void* f) {\n"
                   "  return m.refined_saddle_points_batch(f, 0, 2, 64, 48, 0, AG_L8, 512);\n}\n"
                   "int main() { return 0; }\n")
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(ROOT, "aprilgrid-rs_b200", "cpp"), str(src)])


def test_null_handle_is_invalid(pkg):
    L = pkg.lib()
    frames = (C.c_uint8 * 64)()
    out = (C.c_float * 5)()
    n = (C.c_int * 1)()
    st = (C.c_uint32 * 1)()
    assert L.ag_refined_saddle_points_batch(None, frames, 0, 1, 8, 8, 0, pkg.FMT_L8, out, 1, n, st) == pkg.AG_ERR_INVALID
    assert L.ag_refined_saddle_points_batch_device(None, frames, 0, 1, 8, 8, 0, pkg.FMT_L8, out, 1, n, st,
                                                   None) == pkg.AG_ERR_INVALID
    assert L.ag_multi_refined_saddle_points_batch(None, frames, 0, 1, 8, 8, 0, pkg.FMT_L8, out, 1, n,
                                                  st) == pkg.AG_ERR_INVALID
    assert n[0] == 0 and st[0] == 0
