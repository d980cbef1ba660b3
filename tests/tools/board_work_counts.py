#!/usr/bin/env python3
"""Work counters of the board-search logic (csrc/ag_board_core.h, host build with
-DAGB_WORK_COUNTERS) on synthetic 1280x1024 board frames: where K6's time can go.
usage: python tests/tools/board_work_counts.py [n_frames]"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle  # noqa: E402
import synth  # noqa: E402

so = "/tmp/libag_board_counts.so"
subprocess.check_call(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared",
                       "-DAGB_WORK_COUNTERS", "-I" + os.path.join(ROOT, "aprilgrid-rs_b200", "csrc"),
                       "-o", so, os.path.join(ROOT, "tests", "host_board_test.cpp")])
hb = C.CDLL(so)
cnt = (C.c_longlong * 32).in_dll(hb, "agb_work_counters")
names = ["seeds processed", "nearest_k dist evals", "init_quads rest_ok tests", "board_build calls",
         "try_expand_one calls", "-", "expand 4-tuples tested", "nearest1 dist evals", "decode calls",
         "seeds in bin", "saddles"]
fam = oracle.family_info("t36h11")
codes = np.asarray(fam["codes"], np.uint64)
TAG = np.dtype([("id", np.uint32), ("xy", np.float32, (8,))])
n = int(sys.argv[1]) if len(sys.argv) > 1 else 8
tot = np.zeros(32, np.int64)
import time
t_total = 0.0
for i in range(n):
    img = synth.render_board_numpy(1280, 1024, seed=100 + i)
    s = np.ascontiguousarray(oracle.front_end(img, want_labels=False)["refined"], np.float32)
    for k in range(32):
        cnt[k] = 0
    hb.agb_reset_keys()
    out = np.zeros(1024, TAG)
    st = C.c_uint32(0)
    vp = C.c_void_p
    t0 = time.perf_counter()
    r = hb.hb_detect_from_saddles(s.ctypes.data_as(vp), len(s), img.ctypes.data_as(vp), 1280, 1024,
                                  C.c_size_t(1280), 0, codes.ctypes.data_as(vp), len(codes), fam["edge"],
                                  fam["border"], fam["hamming"], 2, 2048, out.ctypes.data_as(vp), 1024,
                                  None, None, 0, C.byref(st), 1, 64, 512)
    t_total += time.perf_counter() - t0
    c = np.array([cnt[k] for k in range(32)], np.int64)
    tot += c
    print("frame %d: %d tags, %d saddles; round0 %s | round1 %s" % (i, r, len(s), list(c[:11]), list(c[12:23])))
print("edge queries total %.0f distinct %.0f | expand quads total %.0f distinct %.0f | 4-tuple tests total %.0f distinct %.0f"
      % (tot[24] / n, tot[27] / n, tot[25] / n, tot[28] / n, tot[26] / n, tot[29] / n))
print("\nmean per frame (host one-lane build %.2f ms/frame):" % (1e3 * t_total / n))
for r in range(2):
    print(" round %d:" % r)
    for k, nm in enumerate(names):
        if nm != "-":
            print("   %-28s %10.1f" % (nm, tot[12 * r + k] / n))
