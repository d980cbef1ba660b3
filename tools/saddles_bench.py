"""Refined saddle points of whole batches against detect and against today's one-frame loop.  Prints the
GPU's name and power limit first: the numbers belong to that card at that limit.

    python tools/saddles_bench.py [--frames 1024] [--host-frames 512] [--single-frames 200] [--reps 7]

Per image size (1280 x 1024 and 2048 x 1536, a 6 x 6 board rendered on the device, one pose per frame):
- frames/s of refined_saddle_points_batch_device and of detect_batch_device on the same frames, one call
  of --frames frames per repetition, timed with CUDA events on the stream the calls order their results
  on, after a warm-up call;
  median, min and max over --reps repetitions;
- frames/s of refined_saddle_points_batch on the same frames in pinned host memory (host clock, the call
  is synchronous);
- frames/s of a loop of one-frame refined_saddle_points calls over the pinned frames.
Before any timing, a sample of frames from both batch calls is checked byte for byte against the
one-frame call."""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as entry  # noqa: E402

pkg = entry.load_package()
CAP_S, CAP_T = 2048, 128


def event_rates(fn, n, reps, stream):
    """frames/s of fn() over reps repetitions, CUDA events on `stream` (the stream fn's calls order
    their results on), after one warm-up."""
    fn()
    torch.cuda.synchronize()
    rates = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        fn()
        e1.record(stream)
        torch.cuda.synchronize()
        rates.append(n / (e0.elapsed_time(e1) * 1e-3))
    return rates


def host_rates(fn, n, reps):
    fn()
    rates = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        rates.append(n / (time.perf_counter() - t0))
    return rates


def fmt_rates(r):
    return "%9.0f [%.0f .. %.0f]" % (np.median(r), min(r), max(r))


def bench_size(det, W, H, a):
    n = a.frames
    ts = torch.cuda.Stream()  # the calls order their results on it ("device_async" off)
    stream = ts.cuda_stream
    gray = torch.empty((n, H, W), dtype=torch.uint8, device="cuda")
    det.render_boards_device(gray.data_ptr(), n, W, H, 6, 6, 2024 + W)
    d_sad = torch.zeros((n, CAP_S * 5), dtype=torch.int32, device="cuda")
    d_tag = torch.zeros((n, CAP_T * 9), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    m = min(a.host_frames, n)
    pin = pkg.pinned_empty((m, H, W))
    torch.cuda.synchronize()
    pin[...] = gray[:m].cpu().numpy()
    h_out = np.zeros((m, CAP_S), pkg.SADDLE_DTYPE)
    h_cnt = np.zeros(m, np.int32)
    h_st = np.zeros(m, np.uint32)

    def saddles_dev():
        det.refined_saddle_points_batch_device(gray.data_ptr(), n, W, H, pkg.FMT_L8, d_sad.data_ptr(), CAP_S,
                                               cnt.data_ptr(), st.data_ptr(), stream=stream)

    def detect_dev():
        det.detect_batch_device(gray.data_ptr(), n, W, H, pkg.FMT_L8, d_tag.data_ptr(), CAP_T, cnt.data_ptr(),
                                st.data_ptr(), stream=stream)

    def saddles_host():
        det._check(pkg.lib().ag_refined_saddle_points_batch(det._h, pin.ctypes.data, W * H, m, W, H, W, pkg.FMT_L8,
                                                            h_out.ctypes.data, CAP_S, h_cnt.ctypes.data,
                                                            h_st.ctypes.data))

    # correctness first: a sample of frames from both batch calls against the one-frame call
    saddles_dev()
    torch.cuda.synchronize()
    d_words, d_cnt, d_st = d_sad.cpu().numpy(), cnt.cpu().numpy(), st.cpu().numpy()
    saddles_host()
    assert not d_st.any() and not h_st.any()
    for i in sorted(set(np.linspace(0, m - 1, 16).astype(int))):
        one = det.refined_saddle_points(pin[i], cap=16384)
        assert len(one) > 0 and d_cnt[i] == len(one) and h_cnt[i] == len(one), i
        assert d_words[i, :5 * len(one)].tobytes() == one.tobytes(), i
        assert h_out[i, :len(one)].tobytes() == one.tobytes(), i
    n_saddles = float(d_cnt.mean())

    r_sad = event_rates(saddles_dev, n, a.reps, ts)
    r_det = event_rates(detect_dev, n, a.reps, ts)
    torch.cuda.synchronize()
    r_host = host_rates(saddles_host, m, max(3, a.reps // 2))
    k = min(a.single_frames, m)

    def single_loop():
        for i in range(k):
            det.refined_saddle_points(pin[i], cap=CAP_S)
    r_one = host_rates(single_loop, k, 3)
    pkg.pinned_free(pin)
    print("%dx%d, 6x6 board, %.0f refined saddles per frame on average" % (W, H, n_saddles))
    print("  refined_saddle_points_batch_device %5d frames/call  %s frames/s" % (n, fmt_rates(r_sad)))
    print("  detect_batch_device                %5d frames/call  %s frames/s" % (n, fmt_rates(r_det)))
    print("  refined_saddle_points_batch pinned %5d frames/call  %s frames/s" % (m, fmt_rates(r_host)))
    print("  refined_saddle_points loop         %5d frames       %s frames/s" % (k, fmt_rates(r_one)))
    print("  device saddle batch / device detect: %.2f x; device saddle batch / one-frame loop: %.0f x"
          % (np.median(r_sad) / np.median(r_det), np.median(r_sad) / np.median(r_one)))
    del gray, d_sad, d_tag
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--host-frames", type=int, default=512)
    ap.add_argument("--single-frames", type=int, default=200)
    ap.add_argument("--reps", type=int, default=7)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("GPU: %s (name, power limit, max SM clock)" % (q[0] if q else "unknown"))
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    try:
        for W, H in ((1280, 1024), (2048, 1536)):
            bench_size(det, W, H, a)
    finally:
        det.close()


if __name__ == "__main__":
    main()
