"""Frame lists against the batch calls, on one GPU: what a mixed list costs in one call, and what the
per-frame address table costs on a uniform list.  Writes profiles/frames_bench_b200.txt (or --out).

  rig list   512 frames of 1280 x 1024 L8 interleaved with 512 frames of 848 x 480 RGB8 (a colour camera
             and its mono partner), every frame its own allocation:
             device: one detect_frames_device call, against (a) two detect_batch_device calls on
             per-camera tensors stacked beforehand and (b) torch.stack per camera plus those two calls;
             host:   one detect_frames call over separate pageable arrays, against np.stack per camera plus
             two detect_batch calls.
  uniform    1024 separately allocated 1280 x 1024 L8 frames through detect_frames_device, against
             detect_batch_device on one tensor holding the same frames.

Device times are CUDA events on the calling stream (a side stream: the library takes a null stream for
its own) around whole calls, whose results are ordered on that stream;
host times a wall clock around synchronous calls.  Each figure is the median of --reps timed calls after
one warm-up call of every variant.  Before timing, a sample of frames of each list is checked against
the one-frame calls (byte-identical tag records).

    python tools/frames_bench.py [--reps 7] [--out profiles/frames_bench_b200.txt]
"""
import argparse
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

CAP = 128


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    return subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip()


def render(torch, det, n, w, h, seed, rgb):
    """n frames of w x h, each its own allocation (RGB8: gray repeated in three channels)."""
    stack = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    det.render_boards_device(stack.data_ptr(), n, w, h, 6, 6, seed)
    torch.cuda.synchronize()
    return [(stack[i].unsqueeze(-1).repeat(1, 1, 3) if rgb else stack[i].clone()).contiguous() for i in range(n)]


def desc(pkg, t):
    h, w = t.shape[0], t.shape[1]
    fmt = pkg.FMT_RGB8 if t.dim() == 3 else pkg.FMT_L8
    return (t.data_ptr(), w, h, fmt, t.stride(0))


def time_device(torch, fn, reps):
    s = torch.cuda.current_stream()
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(s)
        fn()
        e1.record(s)
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def time_host(fn, reps):
    fn()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ms.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ms)), float(min(ms)), float(max(ms))


def check_sample(pkg, det, imgs, recs, cnts, idx):
    for i in idx:
        img = imgs[i]
        fmt, w, h, st = pkg.image_format(img)
        out = np.zeros(1024, pkg.TAG_DTYPE)
        n = C.c_int(0)
        assert pkg.lib().ag_detect(det._h, img.ctypes.data_as(C.c_void_p), w, h, st, fmt,
                                   out.ctypes.data_as(C.c_void_p), 1024, C.byref(n)) == pkg.AG_OK
        assert cnts[i] == n.value and recs[i, :n.value].tobytes() == out[:n.value].tobytes(), i


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "frames_bench_b200.txt"))
    args = ap.parse_args()
    import torch
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        run(args, torch)


def run(args, torch):
    pkg = entry.load_package()
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    lines = ["GPU: " + gpu_info() + " (name, power limit, SM clock, max SM clock)"]
    L = pkg.lib()
    s = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731

    # ---- rig list
    cam = render(torch, det, 512, 1280, 1024, 11, False)
    mono = render(torch, det, 512, 848, 480, 12, True)
    frames = [f for pair in zip(cam, mono) for f in pair]
    n = len(frames)
    descs = [desc(pkg, t) for t in frames]
    d_out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
    d_cnt = torch.empty(n, dtype=torch.int32, device="cuda")
    d_st = torch.empty(n, dtype=torch.int32, device="cuda")
    cam_t, mono_t = torch.stack(cam), torch.stack(mono)
    out_a = torch.zeros((512, CAP * 9), dtype=torch.int32, device="cuda")
    out_b = torch.zeros_like(out_a)
    cnt_a = torch.empty(512, dtype=torch.int32, device="cuda")
    cnt_b = torch.empty_like(cnt_a)

    def listcall():
        det.detect_frames_device(descs, d_out.data_ptr(), CAP, d_cnt.data_ptr(), d_st.data_ptr(),
                                 torch.cuda.current_stream().cuda_stream)

    def two_batches(a, b):
        for t, o, c, w, h, fmt in ((a, out_a, cnt_a, 1280, 1024, pkg.FMT_L8), (b, out_b, cnt_b, 848, 480, pkg.FMT_RGB8)):
            assert L.ag_detect_batch_device(det._h, C.c_void_p(t.data_ptr()), 0, 512, w, h, 0, fmt,
                                            C.c_void_p(o.data_ptr()), CAP, C.c_void_p(c.data_ptr()), None, s()) == 0

    listcall()
    torch.cuda.synchronize()
    host_imgs = [f.cpu().numpy() for f in frames]
    recs = d_out.cpu().numpy().view(pkg.TAG_DTYPE)
    cnts = d_cnt.cpu().numpy()
    sample = list(range(0, n, 97)) + [1, n - 1]
    check_sample(pkg, det, host_imgs, recs, cnts, sample)
    two_batches(cam_t, mono_t)
    torch.cuda.synchronize()
    assert out_a.cpu().numpy().tobytes() == d_out.cpu().numpy()[0::2].tobytes()
    assert out_b.cpu().numpy().tobytes() == d_out.cpu().numpy()[1::2].tobytes()
    lines.append("rig list: 512 x 1280x1024 L8 interleaved with 512 x 848x480 RGB8, every frame its own allocation; "
                 "%d tags in total; sample of %d frames byte-identical to ag_detect" % (int(cnts.sum()), len(sample)))
    t_list = time_device(torch, listcall, args.reps)
    t_a = time_device(torch, lambda: two_batches(cam_t, mono_t), args.reps)
    t_b = time_device(torch, lambda: two_batches(torch.stack(cam), torch.stack(mono)), args.reps)
    fmt_t = lambda t: "%8.2f ms (min %.2f, max %.2f)" % t  # noqa: E731
    lines.append("  device  detect_frames_device, one call            " + fmt_t(t_list) + "  %7.0f frames/s" % (n / t_list[0] * 1e3))
    lines.append("  device  (a) 2 x detect_batch_device, pre-stacked  " + fmt_t(t_a) + "  %7.0f frames/s" % (n / t_a[0] * 1e3))
    lines.append("  device  (b) torch.stack + 2 x detect_batch_device " + fmt_t(t_b) + "  %7.0f frames/s" % (n / t_b[0] * 1e3))
    # what enqueueing costs the calling thread: with device_async the call returns once its chunks are
    # enqueued, so this is host time only, measured while the GPU still works on the call before
    det.set_option("device_async", 1)
    enq = []
    for _ in range(args.reps):
        listcall()
        t0 = time.perf_counter()
        listcall()
        enq.append((time.perf_counter() - t0) * 1e3)
        det.detect_batch_device_wait(None)
    det.set_option("device_async", 0)
    lines.append("  device  detect_frames_device with device_async: the calling thread returns after %.2f ms "
                 "(median; min %.2f, max %.2f) while the GPU works on the call before" %
                 (float(np.median(enq)), min(enq), max(enq)))
    h_out = np.zeros((n, CAP), pkg.TAG_DTYPE)
    h_cnt = np.zeros(n, np.int32)
    descs_h, keep = pkg.frame_list(host_imgs)
    ha = np.zeros((512, CAP), pkg.TAG_DTYPE)
    hb = np.zeros((512, CAP), pkg.TAG_DTYPE)
    ca, cb = np.zeros(512, np.int32), np.zeros(512, np.int32)

    def host_list():
        assert L.ag_detect_frames(det._h, descs_h, n, h_out.ctypes.data_as(C.c_void_p), CAP,
                                  h_cnt.ctypes.data_as(C.c_void_p), None) == 0

    def host_pack():
        det.detect_batch_into(np.stack(host_imgs[0::2]), ha, ca)
        det.detect_batch_into(np.stack(host_imgs[1::2]), hb, cb)

    host_list()
    assert np.array_equal(h_cnt, cnts) and h_out.tobytes() == recs[:, :CAP].tobytes()
    t_hl = time_host(host_list, args.reps)
    t_hp = time_host(host_pack, args.reps)
    lines.append("  host    detect_frames, separate pageable arrays   " + fmt_t(t_hl) + "  %7.0f frames/s" % (n / t_hl[0] * 1e3))
    lines.append("  host    np.stack + 2 x detect_batch               " + fmt_t(t_hp) + "  %7.0f frames/s" % (n / t_hp[0] * 1e3))
    del keep, cam, mono, frames, cam_t, mono_t

    # ---- uniform list
    uni = render(torch, det, 1024, 1280, 1024, 21, False)
    udescs = [desc(pkg, t) for t in uni]
    ustack = torch.stack(uni)
    u_out = torch.zeros((1024, CAP * 9), dtype=torch.int32, device="cuda")
    u_cnt = torch.empty(1024, dtype=torch.int32, device="cuda")
    b_out, b_cnt = torch.zeros_like(u_out), torch.empty_like(u_cnt)

    def ulist():
        det.detect_frames_device(udescs, u_out.data_ptr(), CAP, u_cnt.data_ptr(), None,
                                 torch.cuda.current_stream().cuda_stream)

    def ubatch():
        assert L.ag_detect_batch_device(det._h, C.c_void_p(ustack.data_ptr()), 0, 1024, 1280, 1024, 0, pkg.FMT_L8,
                                        C.c_void_p(b_out.data_ptr()), CAP, C.c_void_p(b_cnt.data_ptr()), None, s()) == 0

    ulist()
    ubatch()
    torch.cuda.synchronize()
    assert torch.equal(u_out, b_out) and torch.equal(u_cnt, b_cnt)
    t_ul, t_ub = time_device(torch, ulist, args.reps), time_device(torch, ubatch, args.reps)
    lines.append("uniform list: 1024 x 1280x1024 L8, separately allocated; results identical to the batch call")
    lines.append("  device  detect_frames_device, one call            " + fmt_t(t_ul) + "  %7.0f frames/s" % (1024 / t_ul[0] * 1e3))
    lines.append("  device  detect_batch_device on one tensor         " + fmt_t(t_ub) + "  %7.0f frames/s" % (1024 / t_ub[0] * 1e3))
    lines.append("GPU after: " + gpu_info())
    text = "\n".join(lines) + "\n"
    print(text, end="")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)
    det.close()


if __name__ == "__main__":
    main()
