"""Time the device resize (csrc/image_prep.cu) against the host cv2.resize it replaces.

    python tools/image_prep_bench.py [--n 32] [--src 720x1280] [--size 368] [--iters 200] [--out FILE]

Device: n decoded uint8 images of one source size -> the stem's fp16 space-to-depth input at size x size (mode (a),
what unipose.forward_images launches), CUDA-event timed over `iters` launches after warm-up, 5 windows, median.  The
launches rotate over 4 source batches and 2 output buffers (together larger than the 126 MB L2), so every launch
reads its sources from HBM.  Achieved bandwidth counts the algorithmic bytes: every source byte once plus the packed
output written.  The end-to-end call (host job table + upload + launch, to a synchronise) is timed separately.

Host: cv2.resize(img, (size, size)) of the same batch, one thread, and one image per worker over all usable cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def usable_cores() -> int:
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return max(1, n)


def gpu_facts() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "%s (nvidia-smi unavailable: %s)" % (torch.cuda.get_device_name(0), e)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=32)
    ap.add_argument("--src", default="720x1280", help="source HxW")
    ap.add_argument("--size", type=int, default=368)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("image_prep_bench needs a CUDA device")
    from unipose_b200 import data, ops
    h, w = (int(v) for v in args.src.split("x"))
    n, s = args.n, args.size
    torch.cuda.set_device(0)
    rng = np.random.default_rng(0)
    host = [rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8) for _ in range(n)]
    batches = []
    for r in range(4):
        imgs = [torch.from_numpy(np.roll(img, r, axis=1)).cuda() for img in host]
        batches.append((imgs, data.ImageBatch(imgs)))
    outs = [ops.Act(n, s // 2, s // 8 + 1, 64, ops.mode_of("fp16"), "cuda", zero=True) for _ in range(2)]

    def launch(i):
        data.resize_into_s2d(batches[i % 4][1], outs[i % 2], s, wpad_left=2)

    for i in range(50):
        launch(i)
    torch.cuda.synchronize()
    windows = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(args.iters):
            launch(i)
        b.record()
        b.synchronize()
        windows.append(a.elapsed_time(b) * 1e3 / args.iters)
    us = float(np.median(windows))
    src_bytes = n * h * w * 3
    out_bytes = n * (s // 2) * (s // 2) * 16 * 2
    gbs = (src_bytes + out_bytes) / (us * 1e-6) / 1e9

    # end to end: job table from the image list, upload, launch, synchronise
    t_e2e = []
    for r in range(60):
        imgs = batches[r % 4][0]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        data.resize_into_s2d(data.ImageBatch(imgs), outs[r % 2], s, wpad_left=2)
        torch.cuda.synchronize()
        t_e2e.append((time.perf_counter() - t0) * 1e6)
    e2e = float(np.median(t_e2e[10:]))

    import cv2
    cores = usable_cores()
    cv2.setNumThreads(1)
    for img in host[:4]:
        cv2.resize(img, (s, s))
    t0 = time.perf_counter()
    for _ in range(3):
        for img in host:
            cv2.resize(img, (s, s))
    one = 3 * n / (time.perf_counter() - t0)
    with ThreadPoolExecutor(cores) as ex:
        list(ex.map(lambda im: cv2.resize(im, (s, s)), host))
        t0 = time.perf_counter()
        for _ in range(5):
            list(ex.map(lambda im: cv2.resize(im, (s, s)), host))
        allc = 5 * n / (time.perf_counter() - t0)

    res = {
        "gpu": gpu_facts(), "n": n, "src": [h, w], "size": s, "mode": "s2d fp16",
        "kernel_us_per_batch": round(us, 2), "kernel_us_windows": [round(x, 2) for x in windows],
        "kernel_frames_per_s": round(n / (us * 1e-6)), "bytes_per_batch": src_bytes + out_bytes,
        "achieved_GB_per_s": round(gbs, 1), "call_us_end_to_end": round(e2e, 1),
        "host_cv2_frames_per_s_1_thread": round(one, 1), "host_cores": cores,
        "host_cv2_frames_per_s_all_cores": round(allc, 1), "cv2": cv2.__version__,
    }
    lines = [
        "image_prep_bench on %s" % res["gpu"],
        "%d x %dx%d uint8 -> %d^2 fp16 space-to-depth: %.2f us per batch (median of 5 windows of %d launches: %s)"
        % (n, h, w, s, us, args.iters, ", ".join("%.2f" % x for x in windows)),
        "  %.0f frames/s; %.1f MB read + %.1f MB written -> %.0f GB/s achieved"
        % (res["kernel_frames_per_s"], src_bytes / 1e6, out_bytes / 1e6, gbs),
        "  end-to-end call (job table, upload, launch, synchronise): %.1f us" % e2e,
        "host cv2.resize %s, same batch: %.1f frames/s on 1 thread, %.1f frames/s on %d threads"
        % (cv2.__version__, one, allc, cores),
        json.dumps(res),
    ]
    text = "\n".join(lines)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
