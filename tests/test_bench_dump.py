"""bench.py --dump-outputs: the arrays written for the results of the timed path's last step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from conftest import ROOT


def fake_results(pkg, n, cap):
    """Device-layout outputs of one detect_batch_device call (as CPU tensors), stale slots past
    each frame's count, and one status word with the top bit set."""
    rec = np.zeros((n, cap), pkg.TAG_DTYPE)
    cnt = (np.arange(n, dtype=np.int32) * 3) % (cap + 1)
    rec["id"] = 777
    rec["xy"] = 5.5
    for i in range(n):
        rec[i, :cnt[i]]["id"] = np.arange(cnt[i]) + i
        rec[i, :cnt[i]]["xy"] = np.arange(8 * cnt[i], dtype=np.float32).reshape(cnt[i], 8) + 0.25 * i
    status = np.zeros(n, np.uint32)
    status[1] = 0x80000004
    return (torch.from_numpy(rec.view(np.int32).reshape(n, cap * 9).copy()), torch.from_numpy(cnt),
            torch.from_numpy(status.view(np.int32)), rec, cnt, status)


def load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def check_rows(out, rec, cnt, status, cap):
    idx = out["frame_index"].astype(np.int64)
    assert np.array_equal(out["tag_counts"], cnt[idx]) and np.array_equal(out["frame_status"], status[idx])
    for row, i in enumerate(idx):
        k = cnt[i]
        assert np.array_equal(out["tag_ids"][row, :k], rec[i, :k]["id"]) and (out["tag_ids"][row, k:] == -1).all()
        assert np.array_equal(out["tag_corners"][row, :k], rec[i, :k]["xy"].reshape(k, 4, 2))
        assert (out["tag_corners"][row, k:] == 0).all()


def test_dump_detections_files(pkg, tmp_path):
    n, cap = 12, 8
    d_tags, d_cnt, d_status, rec, cnt, status = fake_results(pkg, n, cap)
    bench.dump_detections(str(tmp_path), pkg.TAG_DTYPE, d_tags, d_cnt, d_status, cap)
    out = load(tmp_path)
    assert sorted(out) == ["frame_index", "frame_status", "tag_corners", "tag_counts", "tag_ids"]
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert out["tag_corners"].shape == (n, cap, 4, 2) and out["tag_ids"].shape == (n, cap)
    assert np.array_equal(out["frame_index"], np.arange(n)) and out["frame_status"][1] == 0x80000004
    check_rows(out, rec, cnt, status, cap)


def test_dump_detections_samples_above_the_limit(pkg, tmp_path):
    n, cap = 50, 8
    d_tags, d_cnt, d_status, rec, cnt, status = fake_results(pkg, n, cap)
    per_frame = 3 * 8 + cap * 8 + cap * 32
    limit = 7 * per_frame + 5
    for d in ("a", "b"):
        bench.dump_detections(str(tmp_path / d), pkg.TAG_DTYPE, d_tags, d_cnt, d_status, cap, limit=limit)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sum(v.nbytes for v in a.values()) <= limit
    idx = a["frame_index"]
    assert len(idx) == 7 and np.array_equal(idx, np.unique(idx)) and idx.max() < n
    assert all(np.array_equal(a[k], b[k]) for k in a)  # a fixed sample
    check_rows(a, rec, cnt, status, cap)


@pytest.mark.gpu
def test_bench_dump_is_the_library_result_on_the_same_frames(detector, pkg, tmp_path):
    """bench.py's detect workload with --dump-outputs: the files hold exactly what a direct
    ag_detect_batch_device call returns for the benchmark's seeded frames."""
    n, cap = 64, 64
    out_dir = tmp_path / "dump"
    line = subprocess.check_output(
        [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
         "--batch", str(n), "--no-e2e", "--no-cpu", "--no-extras", "--dump-outputs", str(out_dir)],
        cwd=str(tmp_path), text=True).strip().splitlines()[-1]
    assert json.loads(line)["steps"] == 2
    got = load(out_dir)
    frames = torch.empty((n, bench.H, bench.W), dtype=torch.uint8, device="cuda")
    detector.render_boards_device(frames.data_ptr(), n, bench.W, bench.H, 6, 6, bench.SEED)
    tags = torch.zeros((n, cap * 9), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
    status = torch.zeros(n, dtype=torch.int32, device="cuda")
    detector.detect_batch_device(frames.data_ptr(), n, bench.W, bench.H, pkg.FMT_L8, tags.data_ptr(), cap,
                                 cnt.data_ptr(), status.data_ptr())
    torch.cuda.synchronize()
    rec = tags.cpu().numpy().view(pkg.TAG_DTYPE).reshape(n, cap)
    assert cnt.sum().item() > 30 * n
    check_rows(got, rec, cnt.cpu().numpy(), status.cpu().numpy().view(np.uint32), cap)
