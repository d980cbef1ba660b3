#!/usr/bin/env python3
"""bench.py -- frames/s of the aprilgrid detect path on B200 (BASELINE.json metric).

A "step" is one pass of the hot path (TagDetector::detect semantics, every stage) over one
batch of synthetic frames.  Per-GPU batch is fixed (weak scaling); frames shard image-wise
across ranks with no data-path collective.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload detect|dense|dense4k|rig] [--batch B] [--dump-outputs DIR]

Workloads (BASELINE.json configs):
  detect   configs[2]: rendered 6x6 T36H11 boards, 1280x1024 L8, 1024 frames per GPU per step (default)
  dense    configs[1]: blur + Hessian + threshold kernels alone, 256 frames per step
  dense4k  configs[3]: 3840x2160 RGB8 frames of a dense 24x13 board, 256 frames per GPU per step
  rig      configs[4]: one 2048x1536 camera stream per GPU, frames submitted ONE AT A TIME;
           sustained frames/s and the submit -> result latency distribution

One JSON line on stdout (rank 0).  `value` = device-resident throughput, `e2e` = through
ag_detect_batch with HOST buffers (H2D + D2H inside the timed region).  The default line also
carries short runs of dense4k, the f32 blur operator alone (benches/bench_blur.rs) and rig under "extras".
`--impl reference` times the reference's CPU algorithm (the oracle port, all host threads) on
the first frames of the same device-rendered batch.

`--dump-outputs DIR` (detect and dense4k workloads) writes, after the timed steps, the detections
of rank 0's last timed step as DIR/<name>.npy (see dump_detections).  The frames are rendered
from a fixed seed, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import glob
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402

W, H = 1280, 1024
METRIC = "frames/sec @1280x1024 gray"
UNIT = "frames/s"
BYTES_PER_PX_DETECT = 17  # SURVEY.md 8(d): K1 9 B/px + K2 8 B/px
BYTES_PER_PX_K1 = 9       # 1 in + 4 blur out + 4 response out
SEED = 1000


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def k1_traffic_from_profiles():
    """DRAM bytes per frame of a K1 launch from the newest committed ncu --set full summary
    (profiles/r*_ncu_full_summary.txt).  Returns (bytes_per_frame, file) or (None, None)."""
    best = (None, None)
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_summary.txt"))):
        try:
            txt = open(path).read()
        except OSError:
            continue
        for block in txt.split("---"):
            if "k_blur_hessian_stream" not in block:
                continue
            rd = re.search(r"dram__bytes_read\.sum\s+([\d.]+)\s+Gbyte", block)
            wr = re.search(r"dram__bytes_write\.sum\s+([\d.]+)\s+Gbyte", block)
            grid = re.search(r"launch__grid_size\s+(\d+)", block)
            per_launch = re.search(r"(\d+) frames per launch", txt[:400])
            if rd and wr and (grid or per_launch):
                # frames of that launch: stated in the summary's header, else from the grid
                # (3 strip groups x 9 row chunks of 124 rows per 1280x1024 frame)
                frames = float(per_launch.group(1)) if per_launch else int(grid.group(1)) / 27.0
                best = ((float(rd.group(1)) + float(wr.group(1))) * 1e9 / frames, os.path.relpath(path, ROOT))
            break
    return best


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], False, None
        self.t_begin = self.t_end = None  # host clock window of the timed region

    def run(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "200"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        inside = [r for t, r in self.rows
                  if self.t_begin is None or (self.t_begin <= t <= (self.t_end or t) + 0.2)]
        for r in (inside or [r for _, r in self.rows[-3:]]):
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def gpu_host_link(local):
    """PCIe generation / width of this rank's GPU and the NUMA node it hangs off (None if the guest hides it)."""
    info = {"pcie_gen": None, "pcie_width": None, "pcie_gen_max": None, "pcie_width_max": None, "numa_node": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pcie.link.gen.current,"
                              "pcie.link.width.current,pcie.link.gen.max,pcie.link.width.max,pci.bus_id",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=20).stdout
        f = [c.strip() for c in out.strip().split(",")]
        info.update(pcie_gen=int(f[0]), pcie_width=int(f[1]), pcie_gen_max=int(f[2]), pcie_width_max=int(f[3]))
        bdf = f[4].lower()
        if bdf.startswith("00000000:"):
            bdf = "0000:" + bdf[9:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        info["numa_node"] = node if node >= 0 else None
    except Exception:
        pass
    return info


def bind_to_numa_node(node):
    """Pin this rank's host threads (and so the first-touch placement of its pinned staging buffers)
    to the NUMA node its GPU hangs off, when the host exposes one."""
    try:
        if node is None:
            return False
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return True
    except Exception:
        pass
    return False


def render_frames(det, torch, n, w, h, cols, rows, seed, stream):
    frames = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    det.render_boards_device(frames.data_ptr(), n, w, h, cols, rows, seed, stream=stream)
    return frames


DUMP_LIMIT_BYTES = 64 << 20


def dump_detections(out_dir, tag_dtype, d_tags, d_cnt, d_status, cap, limit=DUMP_LIMIT_BYTES):
    """Write the results of one detect_batch_device call (its three output tensors) as .npy files:
    frame_index (frames,), tag_counts (frames,), frame_status (frames,) and tag_ids (frames, cap)
    in float64, tag_corners (frames, cap, 4, 2) in float32.  Slots past a frame's count hold id -1
    and corners 0.  Above `limit` bytes in all, a fixed seeded sample of the frames is written;
    frame_index says which frames of the batch the rows are."""
    n = d_cnt.shape[0]
    per_frame = 3 * 8 + cap * 8 + cap * 8 * 4
    keep = min(n, limit // per_frame)
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    rec = d_tags.cpu().numpy().view(tag_dtype).reshape(n, cap)[idx]
    cnt = d_cnt.cpu().numpy()[idx]
    valid = np.arange(cap)[None, :] < cnt[:, None]
    arrays = {"frame_index": idx.astype(np.float64),
              "tag_counts": cnt.astype(np.float64),
              "frame_status": d_status.cpu().numpy().view(np.uint32)[idx].astype(np.float64),
              "tag_ids": np.where(valid, rec["id"].astype(np.float64), -1.0),
              "tag_corners": np.where(valid[..., None], rec["xy"], np.float32(0)).reshape(keep, cap, 4, 2)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def gather_list(value, world, device):
    """This rank's python float from every rank, as a list (rank order)."""
    if world == 1:
        return [float(value)]
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    out = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [float(o.item()) for o in out]


# -------------------------------------------------------------------------------------------
# the reference arm: the reference's own CPU algorithm on this box's host cores
# -------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    oracle = entry.load_oracle()
    cores = os.cpu_count() or 1
    per_step = max(cores * 2, 16)
    same_frames = False
    frames = None
    try:  # the very frames the GPU arm runs on: the first `per_step` of rank 0's device-rendered batch
        import torch
        if torch.cuda.is_available():
            pkg = entry.load_package()
            det = pkg.TagDetector(pkg.TagFamily.T36H11, None, device=0)
            d = render_frames(det, torch, per_step, W, H, 6, 6, SEED, None)
            torch.cuda.synchronize()
            frames = np.ascontiguousarray(d.cpu().numpy())
            det.close()
            same_frames = True
    except Exception:
        frames = None
    if frames is None:  # no GPU here: frames from the numpy renderer (same board geometry)
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import synth
        base = synth.fixture_like_frames(8, W, H, seed=100)
        frames = np.ascontiguousarray(np.concatenate([base] * ((per_step + 7) // 8))[:per_step])
    for _ in range(max(args.warmup, 1)):
        oracle.detect_batch(frames[:cores], threads=cores)
    oracle.stage_times(reset=True)
    t0 = time.perf_counter()
    n_tags = 0
    for _ in range(args.steps):
        res = oracle.detect_batch(frames, threads=cores)
        n_tags += sum(len(r) for r in res)
    dt = time.perf_counter() - t0
    st = oracle.stage_times(reset=True)
    fps = args.steps * per_step / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "detect_1280x1024_t36h11_6x6", "frames_per_step": per_step,
                   "image": [W, H], "format": "L8",
                   "frames": ("the first %d frames of the GPU arm's device-rendered batch (seed %d)" % (per_step, SEED))
                   if same_frames else "numpy-rendered boards of the same geometry (no GPU to render on)",
                   "same_config": same_frames},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d frames per step, %d steps, one single-threaded detect per frame on %d "
                                   "host threads (the reference has no threads of its own); C++ restatement of "
                                   "the reference: same arithmetic and allocation pattern, kdtree 0.8 replaced "
                                   "by an exact bucket-grid index" % (per_step, args.steps, cores),
                         "ms_per_frame_per_thread": {k: float(v) for k, v in st.items() if k != "frames"}},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "tags_per_frame": n_tags / max(1, args.steps * per_step),
    }
    print(json.dumps(line), flush=True)
    return 0


# -------------------------------------------------------------------------------------------
# configs[4]: camera rig -- single-frame submits
# -------------------------------------------------------------------------------------------
def run_rig(pkg, det, torch, n_frames, warmup, stream, seed):
    """One 2048x1536 stream on this GPU: 32 distinct frames in pinned host memory, cycled, submitted one
    at a time.  (a) synchronous ag_detect per frame: latency = the call; (b) pipelined: single-frame
    ag_detect_batch calls with host_async, 4 frames in flight: sustained rate, latency = submit -> wait."""
    w, h = 2048, 1536
    d = render_frames(det, torch, 32, w, h, 6, 6, seed, stream)
    torch.cuda.synchronize()
    hf = torch.empty((32, h, w), dtype=torch.uint8).pin_memory()
    hf.copy_(d)
    torch.cuda.synchronize()
    del d
    frames = hf.numpy()
    lat = []
    n_tags = 0
    for i in range(warmup + n_frames):
        t0 = time.perf_counter()
        tags = det.detect(frames[i % 32])
        if i >= warmup:
            lat.append(time.perf_counter() - t0)
            n_tags += len(tags)
    lat = np.asarray(lat)
    sync = {"frames_per_s": float(len(lat) / lat.sum()), "latency_ms_p50": float(1e3 * np.percentile(lat, 50)),
            "latency_ms_p99": float(1e3 * np.percentile(lat, 99)), "latency_ms_max": float(1e3 * lat.max()),
            "tags_per_frame": n_tags / float(len(lat))}
    # pipelined single-frame submits
    depth, cap = 4, 64
    outs = [(np.zeros((1, cap), pkg.TAG_DTYPE), np.zeros(1, np.int32), np.zeros(1, np.uint32)) for _ in range(depth + 1)]
    det.set_option("host_async", 1)
    t_submit, lat2 = {}, []
    t_start = time.perf_counter()
    total = warmup + n_frames
    for i in range(total):
        if i == warmup:
            t_start = time.perf_counter()
        t_submit[i] = time.perf_counter()
        det.detect_batch_into(frames[i % 32][None], *outs[i % (depth + 1)])
        if i >= depth:
            det.detect_batch_wait(depth)  # frame i - depth is complete
            if i - depth >= warmup:
                lat2.append(time.perf_counter() - t_submit[i - depth])
    det.detect_batch_wait(0)
    t_end = time.perf_counter()
    det.set_option("host_async", 0)
    lat2 = np.asarray(lat2) if lat2 else np.zeros(1)
    piped = {"frames_per_s": float(n_frames / (t_end - t_start)), "in_flight": depth,
             "latency_ms_p50": float(1e3 * np.percentile(lat2, 50)), "latency_ms_p99": float(1e3 * np.percentile(lat2, 99))}
    return {"image": [w, h], "format": "L8", "frames": n_frames, "synchronous_detect": sync,
            "pipelined_single_frame_submits": piped}


# -------------------------------------------------------------------------------------------
# configs[3]: 4K RGB dense board
# -------------------------------------------------------------------------------------------
def run_dense4k(pkg, det, torch, n, steps, warmup, stream, seed, dump_dir=None):
    """Streaming calls like the detect workload: device_async, two sets of result buffers, one wait
    after the last step (the board searches of step k overlap the front end of step k + 1).
    With `dump_dir`, the last timed step's detections are written there (dump_detections)."""
    w, h, cap = 3840, 2160, 512
    gray = render_frames(det, torch, n, w, h, 24, 13, seed, stream.cuda_stream)
    rgb = gray[..., None].expand(n, h, w, 3).contiguous()
    del gray
    tags = [torch.zeros((n, cap * 9), dtype=torch.int32, device="cuda") for _ in range(2)]
    cnt = [torch.zeros(n, dtype=torch.int32, device="cuda") for _ in range(2)]
    st = [torch.zeros(n, dtype=torch.int32, device="cuda") for _ in range(2)]
    k = [0]

    def step():
        i = k[0] & 1
        k[0] += 1
        det.detect_batch_device(rgb.data_ptr(), n, w, h, pkg.FMT_RGB8, tags[i].data_ptr(), cap, cnt[i].data_ptr(),
                                st[i].data_ptr(), stream=stream.cuda_stream)

    det.set_option("device_async", 1)
    try:
        for _ in range(max(warmup, 1)):
            step()
        det.detect_batch_device_wait(stream=stream.cuda_stream)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            step()
        det.detect_batch_device_wait(stream=stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
    finally:
        det.set_option("device_async", 0)
    ms = e0.elapsed_time(e1)
    assert steps < 2 or bool((cnt[0] == cnt[1]).all()), "steps disagree on the same frames"
    if dump_dir:
        last = (k[0] - 1) & 1
        dump_detections(dump_dir, pkg.TAG_DTYPE, tags[last], cnt[last], st[last], cap)
    return {"image": [w, h], "format": "RGB8", "board": "24x13 T36H11", "frames_per_step": n, "steps": steps,
            "frames_per_s": float(n * steps / (ms * 1e-3)), "ms_per_step": ms / steps,
            "calls": "streaming (device_async, two result sets, one wait after the last step)",
            "tags_per_frame": float(cnt[0].float().mean()),
            "status_bits": sorted(set(int(x) for x in st[0].cpu().tolist()) | set(int(x) for x in st[1].cpu().tolist()))}


# -------------------------------------------------------------------------------------------
# benches/bench_blur.rs: gaussian_blur_f32(luma_f32, 1.5) alone, f32 -> f32, batched on the device
# -------------------------------------------------------------------------------------------
def run_blur_f32(pkg, det, torch, n, steps, stream):
    w, h = 1280, 1024
    src = torch.rand((n, h, w), dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    for _ in range(3):
        det.gaussian_blur_f32_device(src.data_ptr(), n, w, h, 1.5, dst.data_ptr(), stream=stream.cuda_stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        det.gaussian_blur_f32_device(src.data_ptr(), n, w, h, 1.5, dst.data_ptr(), stream=stream.cuda_stream)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    peak, peak_src = measured_peaks()
    gbs = 8.0 * n * w * h / (ms * 1e-3) / 1e9
    return {"operator": "image_util::gaussian_blur_f32(sigma 1.5), f32 -> f32 (benches/bench_blur.rs)",
            "image": [w, h], "frames_per_step": n, "steps": steps, "ms_per_step": ms,
            "frames_per_s": float(n / (ms * 1e-3)), "algorithmic_bytes_per_px": 8,
            "achieved_gbs": gbs, "peak_gbs": peak, "frac": gbs / peak, "peak_source": peak_src,
            "l2": "input + output (2.7 GB per step) larger than L2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="detect", choices=["detect", "dense", "dense4k", "rig"])
    ap.add_argument("--batch", type=int, default=0, help="frames per GPU per step (default 1024; dense 256; dense4k 256)")
    ap.add_argument("--chunk", type=int, default=0, help="override pipeline chunk_frames")
    ap.add_argument("--lattice", type=int, default=0, help="override board_lattice (16/32/64)")
    ap.add_argument("--board-warps", type=int, default=-1, help="override board_warps (0 auto, 1/2/4/8/16)")
    ap.add_argument("--sync-calls", action="store_true",
                    help="order every step's results on the stream before the next step starts "
                         "(default: steps stream through the pipeline, one wait at the end)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-sync", action="store_true",
                    help="e2e with synchronous ag_detect_batch calls (default: streaming, two calls in flight)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short dense4k / rig runs of the default line")
    ap.add_argument("--opt", action="append", default=[], metavar="KEY=VALUE",
                    help="extra ag_set_option settings (experiments), e.g. --opt k1_chunk_rows=124")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's detections of the last timed step as "
                         "DIR/<name>.npy (detect and dense4k workloads)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload not in ("detect", "dense4k")):
        ap.error("--dump-outputs: only the detect and dense4k workloads return detections to the caller")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    link = gpu_host_link(local)
    numa_bound = bind_to_numa_node(link["numa_node"]) if world > 1 else False
    if world > 1:
        # NCCL prints its version banner on stdout at the first collective; keep stdout for the
        # single JSON line by pointing fd 1 at stderr until the communicator exists.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    pkg = entry.load_package()
    from aprilgrid_rs_b200 import shard
    det = pkg.TagDetector(pkg.TagFamily.T36H11, None, device=local)
    if args.chunk:
        det.set_option("chunk_frames", args.chunk)
    if args.lattice:
        det.set_option("board_lattice", args.lattice)
    if args.board_warps >= 0:
        det.set_option("board_warps", args.board_warps)
    for kv in args.opt:
        key, _, val = kv.partition("=")
        det.set_option(key, int(val))
    stream = torch.cuda.Stream()  # a real (non-default) stream: the kernels and the events share it
    torch.cuda.set_stream(stream)
    sp = stream.cuda_stream
    assert sp != 0

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def finish(line):
        if rank == 0:
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        det.close()
        return 0

    base = {"n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic"}
    par = "frames sharded image-wise, %d rank(s), no collective on the data path" % world

    # ---- configs[4]: rig --------------------------------------------------------------------
    if args.workload == "rig":
        n_frames = args.batch or max(args.steps, 100)
        barrier()
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
            time.sleep(0.5)
            sampler.t_begin = time.perf_counter()
        r = run_rig(pkg, det, torch, n_frames, max(args.warmup, 3), sp, SEED + 7919 * rank)
        if sampler:
            sampler.t_end = time.perf_counter()
        clocks = sampler.finish() if sampler else None
        fps_all = gather_list(r["pipelined_single_frame_submits"]["frames_per_s"], world, "cuda")
        p99_all = gather_list(r["pipelined_single_frame_submits"]["latency_ms_p99"], world, "cuda")
        sync_all = gather_list(r["synchronous_detect"]["frames_per_s"], world, "cuda")
        line = dict(base, metric="frames/sec, 2048x1536 camera streams, one per GPU, single-frame submits",
                    value=float(sum(fps_all)), unit=UNIT, ms_per_step=1e3 / max(min(fps_all), 1e-9),
                    steps=n_frames,
                    config={"workload": "rig_2048x1536_one_stream_per_gpu", "image": [2048, 1536], "format": "L8",
                            "frames_per_gpu": n_frames, "parallelism": "camera c -> GPU c, %d rank(s)" % world,
                            "l2": "32 distinct frames (100 MB) cycled from pinned host memory"},
                    e2e={"value": float(sum(fps_all)), "unit": UNIT, "h2d_bytes_per_step": 2048 * 1536 * world,
                         "d2h_bytes_per_step": (64 * 36 + 8) * world,
                         "timing": "host wall clock, every frame uploaded from pinned host memory and its tags "
                                   "delivered to host memory"},
                    gpu_launches=int(det.launch_count), clocks=clocks, rig=r,
                    per_rank={"pipelined_frames_per_s": fps_all, "pipelined_latency_ms_p99": p99_all,
                              "synchronous_frames_per_s": sync_all})
        return finish(line)

    # ---- configs[3]: 4K RGB dense boards ------------------------------------------------------
    if args.workload == "dense4k":
        B = args.batch or 256
        barrier()
        launches0 = det.launch_count
        sampler = ClockSampler(local) if rank == 0 else None
        if sampler:
            sampler.start()
            time.sleep(0.5)
            sampler.t_begin = time.perf_counter()
        r = run_dense4k(pkg, det, torch, B, args.steps, max(args.warmup, 3), stream, SEED + 7919 * rank,
                        dump_dir=args.dump_outputs if rank == 0 else None)
        if sampler:
            sampler.t_end = time.perf_counter()
        clocks = sampler.finish() if sampler else None
        ms_max = shard.max_over_ranks(r["ms_per_step"] * args.steps, device="cuda")
        line = dict(base, metric="frames/sec @3840x2160 RGB8, dense 24x13 board", unit=UNIT,
                    value=world * B * args.steps / (ms_max * 1e-3), ms_per_step=ms_max / args.steps,
                    config={"workload": "detect_3840x2160_rgb8_t36h11_24x13_batch%d" % B, "frames_per_gpu_per_step": B,
                            "image": [3840, 2160], "format": "RGB8", "parallelism": par,
                            "l2": "inputs (%.2f GB per step) larger than L2" % (B * 3840 * 2160 * 3 / 1e9)},
                    e2e=None, gpu_launches=int(det.launch_count - launches0), clocks=clocks, dense4k=r)
        return finish(line)

    # ---- configs[2] (detect) and configs[1] (dense) -------------------------------------------
    B = args.batch or (1024 if args.workload == "detect" else 256)
    cap = 64
    frames = render_frames(det, torch, B, W, H, 6, 6, SEED + 7919 * rank, sp)
    # two sets of result buffers: with streaming calls, step k+1 starts while step k's board
    # search is still running, so consecutive steps must not share output buffers
    d_tags = [torch.zeros((B, cap * 9), dtype=torch.int32, device="cuda") for _ in range(2)]
    d_cnt = [torch.zeros(B, dtype=torch.int32, device="cuda") for _ in range(2)]
    d_status = [torch.zeros(B, dtype=torch.int32, device="cuda") for _ in range(2)]
    streaming = args.workload == "detect" and not args.sync_calls
    if streaming:
        det.set_option("device_async", 1)
    step_no = [0]

    def step_device():
        if args.workload == "detect":
            k = step_no[0] & 1
            step_no[0] += 1
            det.detect_batch_device(frames.data_ptr(), B, W, H, pkg.FMT_L8, d_tags[k].data_ptr(), cap,
                                    d_cnt[k].data_ptr(), d_status[k].data_ptr(), stream=sp)
        else:
            det.dense_batch_device(frames.data_ptr(), B, W, H, pkg.FMT_L8, stream=sp)

    def drain():
        if streaming:
            det.detect_batch_device_wait(stream=sp)

    # ---- device-resident throughput ("value") ---------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step_device()
    drain()
    barrier()
    det.stage_times(reset=True)
    det.set_option("profile", 1)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.5)  # nvidia-smi start-up; its samples are filtered to the timed window below
    launches0 = det.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if sampler:
        sampler.t_begin = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        step_device()
    drain()  # every step's results are complete before the closing event
    e1.record(stream)
    barrier()
    if sampler:
        sampler.t_end = time.perf_counter()
    ms = e0.elapsed_time(e1)
    launches = det.launch_count - launches0
    clocks = sampler.finish() if sampler else None
    det.set_option("profile", 0)
    stage = det.stage_times(reset=True)
    ms_max = shard.max_over_ranks(ms, device="cuda")
    value = world * B * args.steps / (ms_max * 1e-3)
    per_rank_value = [B * args.steps / (m * 1e-3) for m in gather_list(ms, world, "cuda")]
    # K1 (+K2) alone, same frames, nothing else on the GPU: the roofline figure without the board
    # kernels of earlier chunks sharing the SMs (reported next to the in-step figure)
    k1_alone_ms = None
    if args.workload == "detect":
        torch.cuda.synchronize()
        det.stage_times(reset=True)
        det.set_option("profile", 1)
        for _ in range(3):
            det.dense_batch_device(frames.data_ptr(), B, W, H, pkg.FMT_L8, stream=sp)
        torch.cuda.synchronize()
        det.set_option("profile", 0)
        st_alone = det.stage_times(reset=True)
        k1_alone_ms = st_alone["blur_hessian_min"][0] / max(st_alone["blur_hessian_min"][1], 1)
    cnt_host = d_cnt[0].cpu().numpy() if args.workload == "detect" else None
    if cnt_host is not None:
        assert np.array_equal(cnt_host, d_cnt[1].cpu().numpy()), "steps disagree on the same frames"
        assert not d_status[0].any().item(), "a frame of the benchmark batch was flagged"
    if args.dump_outputs and rank == 0:
        last = (step_no[0] - 1) & 1  # result buffers of the last timed step
        dump_detections(args.dump_outputs, pkg.TAG_DTYPE, d_tags[last], d_cnt[last], d_status[last], cap)
    if streaming:
        det.set_option("device_async", 0)

    # ---- host -> device ceiling of this box, all ranks at once --------------------------------
    h2d_gbs = None
    if args.workload == "detect" and not args.no_e2e:
        nbytes = 256 << 20
        hp = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        dp = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        # the best of several passes, with one and with two streams feeding the copy engine (the
        # e2e path keeps two uploads queued); a single pass on one stream under-reads the link
        dp2 = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        s2 = torch.cuda.Stream()
        for _ in range(2):
            dp.copy_(hp, non_blocking=True)
        rates = []
        for two in (False, True, False, True):
            torch.cuda.synchronize()
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record(stream)
            if two:
                s2.wait_stream(stream)
            for i in range(12):
                if two and (i & 1):
                    with torch.cuda.stream(s2):
                        dp2.copy_(hp, non_blocking=True)
                else:
                    dp.copy_(hp, non_blocking=True)
            if two:
                stream.wait_stream(s2)
            c1.record(stream)
            barrier()
            rates.append(12 * nbytes / (c0.elapsed_time(c1) * 1e-3) / 1e9)
        h2d_gbs = max(rates)
        del dp2
        del hp, dp

    # ---- end to end through the host-buffer C-ABI call ("e2e") -------------------------------
    e2e = None
    if args.workload == "detect" and not args.no_e2e:
        # Frames per rank.  The GPUs of a box do not all get the same share of the host's memory /
        # PCIe bandwidth (measured above, all ranks copying at once), and a host-fed job is as slow as
        # its slowest rank: the N x B frames of a step are therefore sharded in proportion to each
        # rank's measured host-to-device rate (equal shards when the rates agree within 5 %, and
        # always at N = 1).  The equal-shard figure is measured too and reported beside it.
        h2d_all = gather_list(h2d_gbs, world, "cuda")
        balanced = world > 1 and max(h2d_all) > 1.05 * min(h2d_all)
        Be = B
        if balanced:
            Be = int(round(world * B * h2d_all[rank] / sum(h2d_all) / 8.0)) * 8
            Be = max(8, min(Be, 2 * B))
        shard_frames = [int(round(v)) for v in gather_list(Be, world, "cuda")]
        h_frames = torch.empty((max(Be, B), H, W), dtype=torch.uint8).pin_memory()
        for lo in range(0, max(Be, B), B):
            n_cp = min(B, max(Be, B) - lo)
            h_frames[lo:lo + n_cp].copy_(frames[:n_cp])
        torch.cuda.synchronize()
        hf_all = h_frames.numpy()
        hf = hf_all[:B]
        Bo = max(Be, B)

        def pinned_out():
            return (torch.zeros((Bo, cap * 9), dtype=torch.int32).pin_memory().numpy().view(pkg.TAG_DTYPE).reshape(Bo, cap),
                    torch.zeros(Bo, dtype=torch.int32).pin_memory().numpy(),
                    torch.zeros(Bo, dtype=torch.int32).pin_memory().numpy().view(np.uint32))

        # streaming: a second set of output arrays, two calls in flight (the uploads of step i+1
        # overlap the board searches of step i); every step still uploads its frames and
        # delivers its tags to host memory inside the timed region
        outs = [pinned_out(), pinned_out()]
        e2e_streaming = not args.e2e_sync
        det.set_option("host_async", 1 if e2e_streaming else 0)

        def host_steps(k, src):
            n_src = src.shape[0]
            for i in range(k):
                o = outs[i & 1]
                det.detect_batch_into(src, o[0][:n_src], o[1][:n_src], o[2][:n_src])
                if e2e_streaming:
                    det.detect_batch_wait(1)
            if e2e_streaming:
                det.detect_batch_wait(0)

        host_steps(2, hf)
        barrier()
        t0 = time.perf_counter()
        host_steps(args.steps, hf)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        dt_all = gather_list(dt, world, "cuda")
        assert np.array_equal(outs[0][1][:B], cnt_host), "host-path and device-path results differ"
        assert args.steps < 2 or np.array_equal(outs[1][1][:B], cnt_host), "host-path and device-path results differ"
        assert args.steps < 2 or np.array_equal(outs[1][0][:B], outs[0][0][:B]), "streaming host calls disagree"
        dt_bal_all = None
        if balanced:  # the same steps with the shards sized by each rank's link rate
            src_b = hf_all[:Be]
            host_steps(2, src_b)
            barrier()
            t0 = time.perf_counter()
            host_steps(args.steps, src_b)
            torch.cuda.synchronize()
            dt_bal_all = gather_list(time.perf_counter() - t0, world, "cuda")
            nb = min(B, Be)
            assert np.array_equal(outs[0][1][:nb], cnt_host[:nb]), "balanced host path and device path differ"
        # the same calls on PAGEABLE frames (a plain numpy array: what detect_batch(&[DynamicImage])
        # hands over after packing)
        pg = np.empty((B, H, W), np.uint8)
        pg[...] = hf
        pg_steps = max(2, min(args.steps, 10))
        host_steps(1, pg)
        barrier()
        t0 = time.perf_counter()
        host_steps(pg_steps, pg)
        torch.cuda.synchronize()
        dt_pg = time.perf_counter() - t0
        dt_pg_all = gather_list(dt_pg, world, "cuda")
        assert np.array_equal(outs[0][1][:B], cnt_host), "pageable host path and device path differ"
        det.set_option("host_async", 0)
        ceil_rank = [g * 1e9 / (W * H) for g in h2d_all]
        equal = {"value": world * B * args.steps / max(dt_all), "frames_per_rank_per_step": B,
                 "per_rank": [B * args.steps / d for d in dt_all]}
        if balanced:
            total_frames = sum(shard_frames)
            e2e_value = total_frames * args.steps / max(dt_bal_all)
            per_rank = [n * args.steps / d for n, d in zip(shard_frames, dt_bal_all)]
            sharding = ("%d frames per step in all, sharded in proportion to each rank's measured host-to-device "
                        "rate: %s frames per rank" % (total_frames, shard_frames))
        else:
            total_frames = world * B
            e2e_value, per_rank = equal["value"], equal["per_rank"]
            sharding = "equal shards, %d frames per rank per step" % B
        e2e = {"value": e2e_value, "unit": UNIT,
               "h2d_bytes_per_step": int(total_frames * W * H),
               "d2h_bytes_per_step": int(total_frames * (cap * 36 + 8)),
               "timing": "host wall clock around ag_detect_batch, pinned host frames, max over ranks",
               "calls": "streaming (host_async): 2 calls in flight, ag_detect_batch_wait" if e2e_streaming
                        else "synchronous",
               "sharding": sharding, "equal_shards": equal,
               "per_rank": per_rank,
               "h2d_ceiling_gbs_per_rank": h2d_all,
               "h2d_ceiling_note": "best of 4 passes of 12 pinned 256 MB cudaMemcpyAsync (one and two streams), all "
                                   "ranks copying at the same time, in this run; frames/s ceiling = GB/s / 1.31 MB",
               "ceiling_frames_per_s": float(sum(ceil_rank)),
               "frac_of_ceiling": e2e_value / max(sum(ceil_rank), 1e-9),
               "pageable": {"value": world * B * pg_steps / max(dt_pg_all), "unit": UNIT, "steps": pg_steps,
                            "per_rank": [B * pg_steps / d for d in dt_pg_all],
                            "note": "same calls, frames in ordinary (pageable) host memory"},
               "host_link": link, "numa_bound": numa_bound}

    # final gather of detections to host over NCCL: every rank's records to rank 0, frame order
    total_tags = int(cnt_host.sum()) if cnt_host is not None else 0
    gathered = None
    if world > 1 and cnt_host is not None:
        tg = torch.tensor([total_tags], dtype=torch.int64, device="cuda")
        dist.all_reduce(tg)
        total_tags = int(tg.item())
        rec = d_tags[0].cpu().numpy().view(pkg.TAG_DTYPE).reshape(B, cap)
        t0 = time.perf_counter()
        tags_all, counts_all = shard.gather_detections(rec, cnt_host, world * B, device="cuda")
        if rank == 0:
            assert int(counts_all.sum()) == total_tags and tags_all.shape == (world * B, cap)
            assert np.array_equal(tags_all[:B], rec) and np.array_equal(counts_all[:B], cnt_host)
            gathered = {"frames": int(world * B), "tags": int(counts_all.sum()), "backend": dist.get_backend(),
                        "ms": 1e3 * (time.perf_counter() - t0)}

    # ---- short runs of the other BASELINE configs, so that the default line records them -------
    extras = None
    if args.workload == "detect" and not args.no_extras and rank == 0:
        extras = {}
        try:
            extras["dense4k"] = run_dense4k(pkg, det, torch, 256, 3, 1, stream, SEED)
        except Exception as ex:  # never lose the headline line over an extra
            extras["dense4k"] = {"error": repr(ex)}
        try:
            extras["blur_f32"] = run_blur_f32(pkg, det, torch, 256, 10, stream)
        except Exception as ex:
            extras["blur_f32"] = {"error": repr(ex)}
        try:
            extras["rig"] = run_rig(pkg, det, torch, 200, 10, sp, SEED)
        except Exception as ex:
            extras["rig"] = {"error": repr(ex)}
    if world > 1:
        dist.barrier()

    line = None
    if rank == 0:
        peak, peak_src = measured_peaks()
        k1_ms, k1_n = stage["blur_hessian_min"]
        frames_per_launch = (B * args.steps) / max(k1_n, 1)
        k1_avg_s = (k1_ms / max(k1_n, 1)) * 1e-3
        achieved = BYTES_PER_PX_K1 * W * H * frames_per_launch / max(k1_avg_s, 1e-12) / 1e9
        alg = BYTES_PER_PX_K1 * W * H * frames_per_launch
        in_step = achieved
        if k1_alone_ms:
            # primary figure: K1 timed alone (CUDA events, live in this run, same frames, right after
            # the timed region) against the burst copy bandwidth; inside the streaming step K1
            # shares every SM with the board-search kernels of earlier chunks, so its launch
            # duration there is not a statement about the kernel (kept as in_step_*)
            achieved = alg / (k1_alone_ms * 1e-3) / 1e9
        traffic_pf, traffic_src = k1_traffic_from_profiles()
        roofline = {"bound": "hbm", "kernel": "k_blur_hessian_stream (K1: gray->blur->Hessian->min)",
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src,
                    "traffic": traffic_pf * frames_per_launch if traffic_pf else None,
                    "traffic_source": ("%s (ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum of that "
                                       "launch, scaled to this run's %d frames per launch)" % (traffic_src, frames_per_launch))
                    if traffic_pf else None,
                    "algorithmic_bytes_per_launch": alg,
                    "avg_launch_ms": k1_alone_ms if k1_alone_ms else k1_avg_s * 1e3,
                    "timed": ("K1 alone: CUDA events around each launch, 3 passes over the same frames after "
                              "the timed region" if k1_alone_ms else "CUDA events around each K1 launch"),
                    "in_step_avg_launch_ms": k1_avg_s * 1e3, "in_step_launches_timed": k1_n,
                    "in_step_achieved": in_step, "in_step_frac": in_step / peak,
                    "in_step_note": "same kernel timed inside the streaming step, where it overlaps the "
                                    "board searches of up to 8 earlier chunks",
                    "pipeline_achieved_gbs": BYTES_PER_PX_DETECT * W * H * value / world / 1e9,
                    "pipeline_frac": BYTES_PER_PX_DETECT * W * H * value / world / 1e9 / peak}
        total_stage = sum(v[0] for v in stage.values()) or 1.0
        cpu = None
        if not args.no_cpu and cnt_host is not None:
            oracle = entry.load_oracle()
            cores = os.cpu_count() or 1
            n_cpu = min(B, max(4 * cores, 64))
            sample = frames[:n_cpu].cpu().numpy()
            oracle.detect_batch(sample[:cores], threads=cores)
            oracle.stage_times(reset=True)
            t0 = time.perf_counter()
            res = oracle.detect_batch(sample, threads=cores)
            dt = time.perf_counter() - t0
            st_cpu = oracle.stage_times(reset=True)
            # ids and corners of the sample, not only counts: the GPU batch against the oracle
            rec = d_tags[0][:n_cpu].cpu().numpy().view(pkg.TAG_DTYPE).reshape(n_cpu, cap)
            same = True
            for i, r in enumerate(res):
                got = {int(t["id"]): t["xy"].reshape(4, 2) for t in rec[i, :cnt_host[i]]}
                same = same and sorted(got) == sorted(r) and all(np.abs(got[k] - r[k]).max() <= 1e-3 for k in r)
            cpu = {"value": n_cpu / dt, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": "first %d frames of rank 0's batch, oracle detect (C++ port of the reference), "
                             "one frame per thread on %d threads" % (n_cpu, cores),
                   "ms_per_frame_per_thread": {k: float(v) for k, v in st_cpu.items() if k != "frames"},
                   "ids_and_corners_equal_gpu": bool(same)}
        full_boards = float((cnt_host == 36).mean()) if cnt_host is not None else None
        line = dict(base, metric=METRIC, value=value, unit=UNIT, ms_per_step=ms_max / args.steps,
                    config={"workload": ("detect_1280x1024_t36h11_6x6_batch%d" % B) if args.workload == "detect"
                            else ("dense_blur_hessian_threshold_1280x1024_batch%d" % B),
                            "frames_per_gpu_per_step": B, "image": [W, H], "format": "L8", "parallelism": par,
                            "l2": "inputs (%.2f GB per step) larger than L2" % (B * W * H / 1e9),
                            "frames": "rendered on the device: seeded pose, tag side 60-120 px, boards may leave the "
                                      "image (%.1f %% of the frames show all 36 tags)" % (100.0 * (full_boards or 0.0)),
                            "calls": "streaming (ag_detect_batch_device with device_async, one wait after the "
                                     "last step)" if streaming else "one synchronising call per step"},
                    e2e=e2e, gpu_launches=int(launches), clocks=clocks, roofline=roofline, cpu_baseline=cpu,
                    per_rank_value=per_rank_value, gathered_over_nccl=gathered,
                    stage_share={k: v[0] / total_stage for k, v in stage.items()},
                    stage_ms_per_step={k: v[0] / args.steps for k, v in stage.items()},
                    tags_per_frame=total_tags / float(world * B) if cnt_host is not None else None,
                    extras=extras)
    return finish(line)


if __name__ == "__main__":
    sys.exit(main())
