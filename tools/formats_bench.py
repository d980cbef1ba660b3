"""Per pixel format: K1 alone against the measured copy peak, device-resident and pinned-host detect
throughput at 1280 x 1024 (6 x 6 board), and 4K RGBA8 against 4K RGB8.  Prints the GPU's name and power
limit first: the numbers belong to that card at that limit.

    python tools/formats_bench.py [--frames 1024] [--host-frames 256] [--reps 5]

K1's algorithmic bytes are its input (B/px) plus its two f32 outputs, blur and response (8 B/px); its
time is the CUDA-event time of stage 0 (K1 and the per-frame min reset) with option "profile" on.
The copy peak is a device-to-device copy of 4 GB (read + write), larger than L2.  Board frames are
rendered on the device and widened there: R = G = B = gray, 16-bit words = gray * 257, f32 values =
gray / 255, random alpha.  Every format must find the L8 frames' tags."""
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
FORMATS = [("L8", pkg.FMT_L8, 1, 1), ("L16", pkg.FMT_L16, 1, 2), ("RGB8", pkg.FMT_RGB8, 3, 1),
           ("LA8", pkg.FMT_LA8, 2, 1), ("RGBA8", pkg.FMT_RGBA8, 4, 1), ("LA16", pkg.FMT_LA16, 2, 2),
           ("RGB16", pkg.FMT_RGB16, 3, 2), ("RGBA16", pkg.FMT_RGBA16, 4, 2),
           ("RGB32F", pkg.FMT_RGB32F, 3, 4), ("RGBA32F", pkg.FMT_RGBA32F, 4, 4)]  # name, code, channels, bytes/channel
CAP = 128


def widen(gray, channels, width):
    """N x H x W u8 gray -> N x H x (W * channels * width) bytes of the interleaved format."""
    if width == 4:  # f32: gray / 255, alpha random in [0, 1]
        g = gray.to(torch.float32) / 255.0
        chans = [g] * 3
        if channels == 4:
            chans.append(torch.rand(gray.shape, device=gray.device,
                                    generator=torch.Generator(device=gray.device).manual_seed(1)))
        px = torch.stack(chans, dim=-1).contiguous()
        return px.view(torch.uint8).reshape(gray.shape[0], gray.shape[1], -1).contiguous()
    g = gray.to(torch.int32) * (257 if width == 2 else 1)
    n_col = 1 if channels <= 2 else 3
    chans = [g] * n_col
    if channels in (2, 4):
        chans.append(torch.randint(0, 256 ** width, gray.shape, dtype=torch.int32, device=gray.device,
                                   generator=torch.Generator(device=gray.device).manual_seed(1)))
    px = torch.stack(chans, dim=-1)
    if width == 2:  # little-endian words as bytes
        px = torch.stack([(px & 255), (px >> 8)], dim=-1)
    return px.to(torch.uint8).reshape(gray.shape[0], gray.shape[1], -1).contiguous()


def copy_peak_gbs():
    n = 4 << 30
    a = torch.empty(n, dtype=torch.uint8, device="cuda")
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    gbs = 2 * n * 10 / (e0.elapsed_time(e1) * 1e-3) / 1e9
    del a, b
    torch.cuda.empty_cache()
    return gbs


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=1024)
    ap.add_argument("--host-frames", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print("GPU: %s (name, power limit)" % (q[0] if q else "unknown"))
    peak = copy_peak_gbs()
    print("measured copy peak: %.0f GB/s (device-to-device, 4 GB, read + write)" % peak)
    W, H, n = 1280, 1024, a.frames
    det = pkg.TagDetector(pkg.TagFamily.T36H11)
    gray = torch.empty((n, H, W), dtype=torch.uint8, device="cuda")
    det.render_boards_device(gray.data_ptr(), n, W, H, 6, 6, 1000)
    torch.cuda.synchronize()
    out = torch.zeros((n, CAP * 9), dtype=torch.int32, device="cuda")
    cnt = torch.zeros(n, dtype=torch.int32, device="cuda")
    st = torch.zeros(n, dtype=torch.int32, device="cuda")
    print("%-7s %5s %9s %9s %10s %12s %12s" % ("format", "B/px", "K1 ms", "K1 GB/s", "K1/peak", "device f/s",
                                                  "pinned f/s"))
    ref_tags = None
    for name, code, ch, wd in FORMATS:
        fr = widen(gray, ch, wd)
        bpp = ch * wd
        # K1 alone (stage 0 under "profile")
        det.set_option("profile", 1)
        det.dense_batch_device(fr.data_ptr(), n, W, H, code)
        torch.cuda.synchronize()
        det.stage_times(reset=True)
        for _ in range(a.reps):
            det.dense_batch_device(fr.data_ptr(), n, W, H, code)
        ms, _ = det.stage_times(reset=True)["blur_hessian_min"]
        det.set_option("profile", 0)
        k1_ms = ms / a.reps
        k1_gbs = (bpp + 8) * W * H * n / (k1_ms * 1e-3) / 1e9
        # device-resident detect
        def dev():
            det.detect_batch_device(fr.data_ptr(), n, W, H, code, out.data_ptr(), CAP, cnt.data_ptr(), st.data_ptr())
        t_dev = timed(dev, a.reps)
        tags = cnt.cpu().numpy().copy()
        if ref_tags is None:
            ref_tags = tags
        assert np.array_equal(tags, ref_tags) and not st.cpu().numpy().any(), name
        # pinned host detect
        m = a.host_frames
        pin = pkg.pinned_empty((m, H, W * bpp))
        pin[...] = fr[:m].cpu().numpy()
        h_out = np.zeros((m, CAP), pkg.TAG_DTYPE)
        h_cnt = np.zeros(m, np.int32)

        def host():
            det._check(pkg.lib().ag_detect_batch(det._h, pin.ctypes.data, W * H * bpp, m, W, H, W * bpp, code,
                                                 h_out.ctypes.data, CAP, h_cnt.ctypes.data, None))
        t_host = timed(host, max(2, a.reps // 2))
        assert np.array_equal(h_cnt, ref_tags[:m]), name
        pkg.pinned_free(pin)
        print("%-7s %5d %9.3f %9.0f %10.3f %12.0f %12.0f" % (name, bpp, k1_ms, k1_gbs, k1_gbs / peak, n / t_dev,
                                                              m / t_host))
        del fr
        torch.cuda.empty_cache()
    # 4K: RGBA8 against RGB8
    W4, H4, n4 = 3840, 2160, 128
    g4 = torch.empty((n4, H4, W4), dtype=torch.uint8, device="cuda")
    det.render_boards_device(g4.data_ptr(), n4, W4, H4, 24, 13, 7)
    out4 = torch.zeros((n4, 512 * 9), dtype=torch.int32, device="cuda")
    cnt4 = torch.zeros(n4, dtype=torch.int32, device="cuda")
    res = {}
    for name, code, ch in (("RGB8", pkg.FMT_RGB8, 3), ("RGBA8", pkg.FMT_RGBA8, 4)):
        fr = widen(g4, ch, 1)
        t = timed(lambda: det.detect_batch_device(fr.data_ptr(), n4, W4, H4, code, out4.data_ptr(), 512,
                                                  cnt4.data_ptr()), a.reps)
        res[name] = (n4 / t, cnt4.cpu().numpy().copy())
        del fr
        torch.cuda.empty_cache()
    assert np.array_equal(res["RGB8"][1], res["RGBA8"][1])
    print("4K 3840x2160 24x13 board, %d frames, device-resident: RGB8 %.0f frames/s, RGBA8 %.0f frames/s (%.3f x)"
          % (n4, res["RGB8"][0], res["RGBA8"][0], res["RGBA8"][0] / res["RGB8"][0]))
    det.close()


if __name__ == "__main__":
    main()
