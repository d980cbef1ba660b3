#!/usr/bin/env python3
"""Shape of the neighbour searches of the board growth (host build with -DAGB_WORK_COUNTERS): per
round, how large the query windows are and how many saddles they hold -- what a GPU mapping of
find_closest_potential_saddle_idxs (board.rs:177-234) has to cope with.
usage: python tests/tools/search_stats.py [n_frames]"""
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
fam = oracle.family_info("t36h11")
codes = np.asarray(fam["codes"], np.uint64)
TAG = np.dtype([("id", np.uint32), ("xy", np.float32, (8,))])
n = int(sys.argv[1]) if len(sys.argv) > 1 else 4
vp = C.c_void_p
allq = []
for i in range(n):
    img = synth.render_board_numpy(1280, 1024, seed=100 + i)
    s = np.ascontiguousarray(oracle.front_end(img, want_labels=False)["refined"], np.float32)
    for k in range(32):
        cnt[k] = 0
    hb.agb_reset_keys()
    out = np.zeros(1024, TAG)
    st = C.c_uint32(0)
    hb.hb_detect_from_saddles(s.ctypes.data_as(vp), len(s), img.ctypes.data_as(vp), 1280, 1024,
                              C.c_size_t(1280), 0, codes.ctypes.data_as(vp), len(codes), fam["edge"],
                              fam["border"], fam["hamming"], 2, 2048, out.ctypes.data_as(vp), 1024,
                              None, None, 0, C.byref(st), 1, 64, 512)
    q = np.zeros((400000, 7), np.float32)
    m = hb.agb_get_queries(q.ctypes.data_as(vp), len(q))
    q = q[:m]
    # saddle sets per round: round 0 = all refined; round 1 = unknown here -> use distances to the
    # round's own query answers is not needed: count saddles of the FULL list in the window (upper
    # bound for round 1, whose list is a subset)
    allq.append((q, s[:, :2].copy()))
for rnd in (0, 1):
    rows, cands, rad, uniq, tot = [], [], [], 0, 0
    for q, pts in allq:
        qq = q[q[:, 0] == rnd]
        tot += len(qq)
        key = qq[:, 1] * 4096 * 2 + qq[:, 2] * 2 + qq[:, 3]
        _, first = np.unique(key, return_index=True)
        qq = qq[first]
        uniq += len(qq)
        r = np.sqrt(qq[:, 6]) * 1.0001 + 0.01
        y0 = np.floor((qq[:, 5] - r) / 32).clip(0, 31)
        y1 = np.floor((qq[:, 5] + r) / 32).clip(0, 31)
        rows.append(y1 - y0 + 1)
        rad.append(r)
        d2 = (qq[:, 4][:, None] - pts[None, :, 0]) ** 2 + (qq[:, 5][:, None] - pts[None, :, 1]) ** 2
        cands.append((d2 <= qq[:, 6][:, None]).sum(axis=1))
    rows, cands, rad = np.concatenate(rows), np.concatenate(cands), np.concatenate(rad)
    print("round %d: %.0f queries / frame, %.0f distinct (a, b, self); radius px p10/50/90/99 = %s; bucket rows "
          "p50/90/99 = %s; saddles within the radius (full list) p50/90/99/max = %s; share with none %.2f, < 3 %.2f"
          % (rnd, tot / n, uniq / n, np.percentile(rad, [10, 50, 90, 99]).round(1).tolist(),
             np.percentile(rows, [50, 90, 99]).tolist(), np.percentile(cands, [50, 90, 99, 100]).tolist(),
             (cands == 0).mean(), (cands < 3).mean()))
